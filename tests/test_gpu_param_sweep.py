"""Every kernel against the oracle across the numerical settings the C ABI accepts, not only those
of the decks: de Hoog M 2..31 (compile-time M = 10 and 26 in the one-inversion-per-thread de Hoog,
a runtime-M body for every other M, odd M ending on a one-stage q-d sweep, rows above lane 31 in
the warp de Hoog), Wynn-epsilon on 2..32 terms (register/shared lozenges up to 14 terms, the
column-order and blocked tables above), tanh-sinh k = 3..12 and Gauss-Lobatto orders down to one
node per interval.  Each case is a base deck with overridden M, gl_nacc, ts_k/ts_R and gl_ord; all
seven models appear.  The same points go through the 128-z kernel, the lanes<->z kernel, the point
kernel with four, two and one z per CTA, and (for three cases) the screen and gradient kernels.

The bar is helpers.check_parity at every point, flags and NaN pattern equal to the oracle's, and
at least half of the points quiet (NOISE_K * spread <= RTOL * |s|) so that the case discriminates;
at the quiet points the kernels also agree with each other (s to 1e-11, ds to 1e-10).

Also here: the cost-ordered path of large scattered point sets, bitwise against the unordered
paths, and the largest accepted settings evaluated at every grid shape."""
import numpy as np
import pytest

import unconfined_b200 as ub
from oracle import oracle
from oracle import screens as oscr
from oracle import dz as odz
from helpers import load_deck, check_parity, oracle_with_noise, RTOL, NOISE_K

pytestmark = pytest.mark.gpu

DECK_OF_MODEL = {0: "theis-input.dat", 1: "hantush-input.dat", 2: "hantush-storage-input.dat",
                 3: "cape-cod-moench.in", 4: "malama-fullpen-input.dat", 5: "malama-partpen-input.dat",
                 6: "mishra-neuman-malama.in"}

MAXSET = dict(gl_nacc=32, ts_k=12, ts_R=10, gl_ord=100)

# name: (model of the base deck, overrides, (times as fractions of the deck's time list, radii)).
# Large M amplifies rounding in the q-d table most at early times, so those cases take later times
# (at 1/3 and 2/3 of the list fewer than half of their points would be quiet).  The k = 12 cases
# keep to two columns: the oracle needs ~0.1 s per point there before its jitter samples.
MID, LATE = (1 / 3, 2 / 3), (3 / 4, 9 / 10)
R3 = [0.3, 1.0, 3.0]
CASES = {
    "min-corner": (0, dict(M=2, gl_nacc=2, ts_k=3, ts_R=1, gl_ord=3), (MID, R3)),
    "M3-nacc13": (1, dict(M=3, gl_nacc=13), (MID, R3)),
    "M16-nacc14-ord37": (2, dict(M=16, gl_nacc=14, gl_ord=37), (MID, R3)),   # 14 * 35 = 490 nodes
    "M17-nacc15-k3": (3, dict(M=17, gl_nacc=15, ts_k=3, ts_R=1), (MID, R3)),
    "M18-nacc32": (4, dict(M=18, gl_nacc=32), (LATE, R3)),
    "M27-nacc13": (5, dict(M=27, gl_nacc=13), (LATE, R3)),
    "M31-nacc16": (6, dict(M=31, gl_nacc=16), ((1 / 2,), [0.5, 1.5])),
    "M27-max-settings": (1, dict(M=27, **MAXSET), ((1 / 2,), [0.4, 2.0])),
    "max-corner": (1, dict(M=31, **MAXSET), ((1 / 2,), [0.4, 2.0])),
}
SCREEN_DZ_CASES = ["M17-nacc15-k3", "M18-nacc32", "M27-nacc13"]


@pytest.fixture(autouse=True)
def _need_gpu():
    assert ub.device_count() >= 1, "no CUDA device: the product path has no CPU fallback"
    ub.force_kernel(None)
    ub.set_carry(True)
    yield
    ub.force_kernel(None)
    ub.set_carry(True)


def z_list(pd, n=40):
    """n values in [0, 1] that include 0, 1 - lD, 1 - dD and 1."""
    z = set(np.linspace(0.0, 1.0, n - 2).tolist()) | {1.0 - pd["lD"], 1.0 - pd["dD"]}
    z = sorted(z)
    while len(z) < n:                                 # 1 - lD or 1 - dD fell on the grid
        i = int(np.argmax(np.diff(z)))
        z.insert(i + 1, 0.5 * (z[i] + z[i + 1]))
    return np.array(z)


def case_inputs(name):
    model, over, (tfrac, radii) = CASES[name]
    d, pd = load_deck(DECK_OF_MODEL[model])
    assert pd["model"] == model
    pq = dict(pd, **over)
    pq["j0z"] = oracle.j0_zeros(max(d["j0s"]) + pq["gl_nacc"] + 1)
    # away from the deck's earliest times (ill-conditioned de Hoog inversions of tiny drawdowns)
    if len(d["tD"]) > 1:
        tD = d["tD"][[int(f * len(d["tD"])) for f in tfrac]]
    else:                                             # the Theis deck has one time
        tD = d["tD"][0] * np.array([1.0, 30.0])[:len(tfrac)]
    sv = oracle.split_index(tD, d["j0s"])
    zD = z_list(pq)
    return d, pq, (tD, sv, np.array(radii, float), zD, oracle.zlay(zD, pq["lD"], pq["dD"]))


_ORACLE = {}


def case_oracle(name):
    """Fresh-mode oracle values, noise envelope and flags of a case (computed once per module)."""
    if name not in _ORACLE:
        d, pq, args = case_inputs(name)
        po = oracle.Params(pq)
        so, do, sps, spd = oracle_with_noise(po, args)
        _, _, fo = oracle.eval_grid(po, *args, carry=False)
        _ORACLE[name] = (so, do, sps, spd, fo)
    return _ORACLE[name]


def run_grid(prm, args, kernel):
    ub.force_kernel(kernel)
    try:
        return ub.eval_grid(prm, *args, want_flags=True)
    finally:
        ub.force_kernel(None)


def sub_z(args, idx):
    tD, sv, rD, zD, lay = args
    return (tD, sv, rD, zD[idx], lay[idx])


@pytest.mark.parametrize("name", list(CASES))
def test_every_kernel_against_the_oracle(name):
    d, pq, args = case_inputs(name)
    so, do, sps, spd, fo = case_oracle(name)
    prm = ub.Params(pq)
    tD, sv, rD, zD, lay = args
    nz = len(zD)
    i6 = np.array([0, 7, 15, 23, 31, 39]); i3 = np.array([0, 20, 39])
    res = {}
    # the 128-z kernel (auto would take the point kernel: this grid has fewer columns than SMs)
    res["grid8"] = run_grid(prm, args, "grid8")
    res["grid2"] = run_grid(prm, args, "grid2")          # lanes<->z: ZL = 2, ZL = 1 from M = 27
    res["point"] = run_grid(prm, args, "point")          # four z per CTA (two where four do not fit)
    for tag, idx in (("point6", i6), ("point3", i3)):    # ragged ZT = 4 and ZT = 2 tiles
        s, ds, fl = run_grid(prm, sub_z(args, idx), "point")
        full = [np.full(so.shape, np.nan), np.full(so.shape, np.nan), np.zeros(so.shape, np.int32)]
        for a, b in zip(full, (s, ds, fl)):
            a[:, :, idx] = b
        res[tag] = (tuple(full), idx)
    # one z per CTA: the flattened (t, r, z) set through unc_eval_points
    T, R, Z = np.meshgrid(np.arange(len(tD)), np.arange(len(rD)), np.arange(nz), indexing="ij")
    T, R, Z = T.ravel(), R.ravel(), Z.ravel()
    s, ds, fl = ub.eval_points(prm, tD[T], sv[T], rD[R], zD[Z], lay[Z], want_flags=True)
    res["points"] = (s.reshape(so.shape), ds.reshape(so.shape), fl.reshape(so.shape))

    quiet_s = NOISE_K * sps <= RTOL * np.abs(so)
    quiet_d = NOISE_K * spd <= RTOL * np.abs(do)
    assert quiet_s.mean() >= 0.5, f"{name}: only {quiet_s.mean():.2f} of the points are quiet"
    vals = {}
    for kernel, r in res.items():
        if kernel in ("point6", "point3"):
            (s, ds, fl), idx = r
            sel = (slice(None), slice(None), idx)
        else:
            s, ds, fl = r
            sel = (slice(None), slice(None), slice(None))
        what = f"{name}[{kernel}]"
        assert np.array_equal(fl[sel], fo[sel]), f"{what}: flags differ"
        check_parity(s[sel], ds[sel], so[sel], do[sel], sps[sel], spd[sel], what=what)
        vals[kernel] = (s, ds, sel)
    # kernels against each other where the oracle's own noise is far below the bar: s to 1e-11.
    # ds inverts p f(p), whose rounding the q-d table amplifies more; at its quiet points the
    # kernels differ by up to 3.4e-11 (M31-nacc16, lanes<->z vs 128-z, on a B200), so 1e-10.
    s8, d8, _ = vals["grid8"]
    for kernel, (s, ds, sel) in vals.items():
        for got, ref, quiet, q, tol in ((s, s8, quiet_s, "s", 1e-11), (ds, d8, quiet_d, "ds", 1e-10)):
            g, r, m = got[sel], ref[sel], quiet[sel]
            rel = np.abs(g[m] - r[m]) / np.abs(r[m])
            assert rel.size == 0 or rel.max() <= tol, f"{name}: {kernel} vs grid8 {q}: {rel.max():.3e} at a quiet point"


def screen_set(pq):
    b1, b2 = 1.0 - pq["lD"], 1.0 - pq["dD"]
    scr = [(0.0, 1.0), (0.1, 0.45), (0.6, 0.95), (max(0.0, b1 - 0.1), min(1.0, b2 + 0.002)), (0.3, 0.3 + 1e-3)]
    return [(lo, hi) for lo, hi in scr if lo < hi]


@pytest.mark.parametrize("name", SCREEN_DZ_CASES)
def test_screens_and_vertical_gradient_against_the_oracle(name):
    d, pq, (tD, sv, rD, zD, lay) = case_inputs(name)
    po, prm = oracle.Params(pq), ub.Params(pq)
    T, R = np.meshgrid(np.arange(len(tD)), np.arange(len(rD)), indexing="ij")
    T, R = T.ravel(), R.ravel()
    # screens: every screen at every (t, r)
    scr = np.array(screen_set(pq))
    st, sr = np.repeat(T, len(scr)), np.repeat(R, len(scr))
    zb, zt = np.tile(scr[:, 0], len(T)), np.tile(scr[:, 1], len(T))
    sargs = (tD[st], sv[st], rD[sr], zb, zt)
    f = lambda: oscr.eval_screens(po, *sargs)  # noqa: E731
    so, do, sps, spd = oscr.noise_envelope(f, nsamples=5)
    sl, dl, _ = oscr.eval_screens(po, *sargs, long_double=True)
    _, _, fo = f()
    sps = np.fmax(sps, np.abs(so - sl)); spd = np.fmax(spd, np.abs(do - dl))
    s, ds, fl = ub.eval_screens(prm, *sargs, want_flags=True)
    assert np.array_equal(fl, fo), f"{name} screens: flags differ"
    check_parity(s, ds, so, do, sps, spd, what=f"{name} screens")
    assert (NOISE_K * sps <= RTOL * np.abs(so)).mean() >= 0.5
    # vertical gradient at eight z of the case's list, including 0, 1 - lD, 1 - dD and 1
    zs = zD[np.array([0, 5, 11, 17, 23, 29, 35, 39])]
    zs = np.unique(np.concatenate([zs, [1.0 - pq["lD"], 1.0 - pq["dD"]]]))
    n = len(T) * len(zs)
    pt, pr = np.repeat(T, len(zs)), np.repeat(R, len(zs))
    dargs = (tD[pt], sv[pt], rD[pr], np.tile(zs, len(T)))
    f = lambda: odz.eval_points_dz(po, *dargs)  # noqa: E731
    go, gdo, spg, spgd = odz.noise_envelope(f, nsamples=5)
    gl, gdl, _ = odz.eval_points_dz(po, *dargs, long_double=True)
    _, _, fo = f()
    spg = np.fmax(spg, np.abs(go - gl)); spgd = np.fmax(spgd, np.abs(gdo - gdl))
    gz, dgz, fl = ub.eval_points_dz(prm, *dargs, want_flags=True)
    assert np.array_equal(fl, fo), f"{name} gradient: flags differ"
    check_parity(gz, dgz, go, gdo, spg, spgd, what=f"{name} gradient")
    assert (NOISE_K * spg <= RTOL * np.abs(go)).mean() >= 0.5
    assert n == len(gz)


# ---- the cost-ordered point path ------------------------------------------------------------

N_SCATTER = 3 * 2 ** 14 + 77


def scatter_set(seed=20261021):
    """3 * 2^14 + 77 scattered points of the Neuman-type deck with a water table and a partially
    penetrating well (model 5, beta > 0): rD log-uniform over 1e-3..1e3, so that both clamped ends
    of cost_bin and most bins in between are hit, and 4000 points that repeat others."""
    d, pd = load_deck("malama-partpen-input.dat")
    rng = np.random.default_rng(seed)
    n = N_SCATTER
    rD = 10 ** rng.uniform(-3, 3, n); zD = rng.uniform(0, 1, n); tD = 10 ** rng.uniform(-1, 7, n)
    dst, src = rng.choice(n, 4000, replace=False), rng.choice(n, 4000)
    rD[dst], zD[dst], tD[dst] = rD[src], zD[src], tD[src]
    sv = oracle.split_index(tD, d["j0s"])
    lay = oracle.zlay(zD, pd["lD"], pd["dD"])
    pd = dict(pd, j0z=oracle.j0_zeros(max(d["j0s"]) + pd["gl_nacc"] + 1))
    return pd, (tD, sv, rD, zD, lay)


def eval_points_prefilled(prm, args, **kw):
    """eval_points into outputs pre-filled with a value no point evaluates to, so that an output
    the kernel never writes cannot pass for a result."""
    n = len(args[0])
    out = (np.full(n, 1e300), np.full(n, 1e300))
    s, ds, fl = ub.eval_points(prm, *args, want_flags=True, out=out, **kw)
    return s, ds, fl


def test_cost_ordered_points_equal_the_unordered_paths_bitwise():
    import torch
    pd, args = scatter_set()
    prm = ub.Params(pd)
    n = N_SCATTER
    s0, d0, f0 = eval_points_prefilled(prm, args)            # >= 16384 points: cost-ordered
    assert not (s0 == 1e300).any() and not (d0 == 1e300).any()
    runs = {}
    ub.force_kernel("point")
    try:
        runs["unordered"] = eval_points_prefilled(prm, args)
    finally:
        ub.force_kernel(None)
    chunks = [np.arange(n)[i:i + 10000] for i in range(0, n, 10000)]
    parts = [eval_points_prefilled(prm, tuple(a[c] for a in args)) for c in chunks]
    runs["chunks"] = tuple(np.concatenate([p[k] for p in parts]) for k in range(3))
    runs["ngpu=0"] = eval_points_prefilled(prm, args, ngpu=0)
    dev = torch.device("cuda", 0)
    g = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dtype=dt)  # noqa: E731
    tD, sv, rD, zD, lay = args
    s_ = torch.full((n,), 1e300, dtype=torch.float64, device=dev); d_ = torch.full_like(s_, 1e300)
    f_ = torch.full((n,), -1, dtype=torch.int32, device=dev)
    ub.eval_points_device(prm, g(tD, torch.float64), g(sv, torch.int32), g(rD, torch.float64),
                          g(zD, torch.float64), g(lay, torch.int32), s_, d_, flags=f_)
    torch.cuda.synchronize()
    runs["device"] = (s_.cpu().numpy(), d_.cpu().numpy(), f_.cpu().numpy())
    for what, (s, ds, fl) in runs.items():
        assert np.array_equal(s, s0, equal_nan=True), f"{what}: s differs at {np.argwhere(~((s == s0) | (np.isnan(s) & np.isnan(s0))))[:5].ravel()}"
        assert np.array_equal(ds, d0, equal_nan=True), f"{what}: ds differs"
        assert np.array_equal(fl, f0), f"{what}: flags differ"
    # repeated points: identical results
    key = np.stack([tD, rD, zD], 1)
    _, first, inv = np.unique(key, axis=0, return_index=True, return_inverse=True)
    inv = inv.ravel()
    assert len(first) < n
    assert np.array_equal(s0, s0[first][inv], equal_nan=True)
    # a sample against the oracle, among the points with rD >= 0.01 (below that the overflowing
    # integrands leave sentinel-dominated values, compared in test_gpu_parity.test_non_finite_flow_matches)
    rng = np.random.default_rng(7)
    pick = rng.choice(np.flatnonzero(rD >= 0.01), 256, replace=False)
    sub = tuple(a[pick] for a in args)
    so, do, sps, spd = oracle_with_noise(oracle.Params(pd), sub, points=True)
    _, _, fo = oracle.eval_points(oracle.Params(pd), *sub)
    assert np.array_equal(f0[pick], fo)
    check_parity(s0[pick], d0[pick], so, do, sps, spd, what="cost-ordered sample")


# ---- the largest accepted settings evaluate at every grid shape ------------------------------

@pytest.mark.parametrize("name", ["max-corner", "M27-max-settings"])
def test_largest_settings_evaluate_at_every_grid_shape(name):
    """M = 27 and 31 with 32 Wynn terms, k = 12, R = 10 and ord = 100: four z per point-kernel CTA
    need more than 227 KB of shared memory there, so the point kernel takes two.  Every grid shape
    must evaluate, with two columns (the point kernel up to nz = 63) and with more columns than SMs
    (the lanes<->z kernel from nz = 12, the 128-z kernel from nz = 33).  The many columns repeat
    the two radii, so every result is held to the oracle of the case's two columns."""
    import torch
    d, pq, args = case_inputs(name)
    so, do, sps, spd, fo = case_oracle(name)
    prm = ub.Params(pq)
    tD, sv, rD, zD, lay = args
    rep_many = torch.cuda.get_device_properties(0).multi_processor_count // len(rD) + 8
    for nz in (1, 3, 5, 11, 12, 40):
        idx = np.unique(np.linspace(0, len(zD) - 1, nz).round().astype(int))
        assert len(idx) == nz
        for rep in (1, rep_many):
            s, ds, fl = ub.eval_grid(prm, tD, sv, np.tile(rD, rep), zD[idx], lay[idx], want_flags=True)
            w = [np.tile(a[:, :, idx], (1, rep, 1)) for a in (so, do, sps, spd, fo)]
            what = f"{name} nz={nz} ncol={len(tD) * len(rD) * rep}"
            assert np.array_equal(fl, w[4]), f"{what}: flags differ"
            check_parity(s, ds, *w[:4], what=what)

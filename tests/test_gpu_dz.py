"""Vertical drawdown gradient on the GPU (unc_eval_points_dz, lh_dz_kernel): parity with the
oracle's gradient mode on the decks of models 0-6, exact limits (Theis has no z dependence, the
Hantush aquifer has impervious bottom and top), the kinematic water-table condition of the
Neuman-type models, consistency with point drawdowns (integral and finite difference), and the
plumbing (device entry, cost-ordered large calls, sharding, determinism, command line)."""
import os
import subprocess

import numpy as np
import pytest

import unconfined_b200 as ub
from oracle import oracle
from oracle import dz as odz
from helpers import load_deck, stale_scale, ROOT

pytestmark = pytest.mark.gpu

# The parity bar of tests/helpers.py, restated for the gradient: a point passes if
#   |gpu - oracle| <= RTOL*|oracle| + NOISE_K*spread
# where spread is how far the oracle's own result moves under <= 2-ulp libm jitter or in long
# double.  NaN patterns and flags must match exactly.
RTOL = 1e-9
NOISE_K = 12.0

DECKS = [("theis-input.dat", 0), ("hantush-input.dat", 1), ("hantush-storage-input.dat", 2),
         ("cape-cod-moench.in", 3), ("malama-fullpen-input.dat", 4), ("malama-partpen-input.dat", 5),
         ("cape-cod-neuman74.in", 5), ("mishra-neuman-malama.in", 6)]


def z_values(pd):
    """zD = 0, zD = 1, the boundaries 1-lD and 1-dD inside (0, 1), and the middle of each layer."""
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    z = [0.0, 1.0]
    z += [b for b in (b1, b2) if 0.0 < b < 1.0]
    if b1 > 0.0:
        z.append(0.5 * b1)
    if b2 > b1:
        z.append(0.5 * (b1 + b2))
    if b2 < 1.0:
        z.append(0.5 * (b2 + 1.0))
    return sorted(set(z))


def point_set(d, pd, every=10):
    """Every `every`-th time of the deck times every z of z_values, at the deck's first radius."""
    it = np.arange(0, len(d["tD"]), every)
    zs = np.array(z_values(pd))
    ti, zi = np.meshgrid(it, np.arange(len(zs)), indexing="ij")
    ti, zi = ti.ravel(), zi.ravel()
    return d["tD"][ti], d["sv"][ti], np.full(len(ti), d["rD"][0]), zs[zi]


def oracle_dz_with_noise(po, args, ts_scale=None, nsamples=4):
    f = lambda: odz.eval_points_dz(po, *args, ts_scale=ts_scale)  # noqa: E731
    g0, d0, sp_g, sp_d = odz.noise_envelope(f, nsamples=nsamples)
    gl, dl, _ = odz.eval_points_dz(po, *args, ts_scale=ts_scale, long_double=True)
    with np.errstate(invalid="ignore"):
        sp_g = np.fmax(sp_g, np.abs(g0 - gl))
        sp_d = np.fmax(sp_d, np.abs(d0 - dl))
    return g0, d0, sp_g, sp_d


def check(got, want, spread, what, floor=0.0):
    nan_same = np.isnan(got) == np.isnan(want)
    assert nan_same.all(), f"{what}: NaN pattern differs at {np.argwhere(~nan_same)[:5].ravel()}"
    ok = np.isnan(want) | (np.abs(got - want) <= RTOL * np.abs(want) + NOISE_K * spread + floor) | (got == want)
    assert ok.all(), (f"{what}: {int((~ok).sum())} of {ok.size} fail ({np.argwhere(~ok)[:10].ravel()}); first: "
                      f"gpu={got[~ok][0]!r} oracle={want[~ok][0]!r} spread={spread[~ok][0]:.3e}")


def impervious_top(pd, zD):
    """The top of the aquifers without a water table (models 0, 1, 2), where the gradient vanishes
    identically: the oracle forms it as eta sinh(eta dD) - ff1 eta sinh(eta)/sinh(eta), a
    rounding residue (exactly 0 when dD = 0), the fast path as eta (cp e^eta - cm e^-eta) with
    cp e^eta = cm e^-eta, another.  Whether a residue is exactly 0 at every abscissa -- the
    stale-infint flag -- depends on that operation order, so flags are compared everywhere else.
    Values here, gz and dgz alike, are held to the bar of the Hantush limit test, 1e-9 of max|gz|
    over the points of the same time: the residues are of the size of the rounding of the
    gradient's terms, while dgz itself vanishes as the drawdown becomes steady."""
    return (zD == 1.0) & (pd["model"] <= 2)


def profile_floor(want, tD, mask):
    """1e-9 max|oracle gz| over the points of the same time, at the points of `mask`."""
    floor = np.zeros(len(want))
    for t in np.unique(tD):
        sel = tD == t
        floor[sel & mask] = 1e-9 * np.nanmax(np.abs(np.where(sel, want, 0.0)))
    return floor


@pytest.mark.parametrize("name,model", DECKS)
@pytest.mark.parametrize("stale", [False, True], ids=["fresh", "ts_scale"])
def test_dz_parity_with_oracle(name, model, stale):
    d, pd = load_deck(name)
    assert pd["model"] == model
    args = point_set(d, pd)
    ts = np.full(len(args[0]), stale_scale(d)) if stale else None
    gz, dgz, fl = ub.eval_points_dz(ub.Params(pd), *args, ts_scale=ts, want_flags=True)
    go, do, sp_g, sp_d = oracle_dz_with_noise(oracle.Params(pd), args, ts_scale=ts)
    _, _, flo = odz.eval_points_dz(oracle.Params(pd), *args, ts_scale=ts)
    imp = impervious_top(pd, args[3])
    assert np.array_equal(fl[~imp], flo[~imp])
    check(gz, go, sp_g, f"{name} gz", profile_floor(go, args[0], imp))
    check(dgz, do, sp_d, f"{name} dgz", profile_floor(go, args[0], imp))


def test_small_radius_literal_path_and_certain_nan():
    """rD = 0.075 (hantush-contours): the largest abscissae exceed the fast-path bound, so the
    literal gradient path runs, and beyond Re(eta) = 718 the certain-NaN rule (sinh(eta)
    overflows) replaces it; values and NaN pattern of the results must still be the oracle's."""
    d, pd = load_deck("hantush-contours-input.dat")
    tD = np.geomspace(1e-2, 1e4, 13)
    sv = ub.split_index(tD, (2, 2))
    zs = z_values(pd)
    n = len(tD) * len(zs)
    args = (np.repeat(tD, len(zs)), np.repeat(sv, len(zs)), np.full(n, 0.075), np.tile(zs, len(tD)))
    for model in (1, 5):
        p = dict(pd, model=model, beta=0.0, alphaD=1e4)
        gz, dgz, fl = ub.eval_points_dz(ub.Params(p), *args, want_flags=True)
        go, do, sp_g, sp_d = oracle_dz_with_noise(oracle.Params(p), args)
        _, _, flo = odz.eval_points_dz(oracle.Params(p), *args)
        print(f"model {model}: {int(np.isnan(go).sum())} NaN of {n}")
        imp = impervious_top(p, args[3])
        assert np.array_equal(fl[~imp], flo[~imp])
        check(gz, go, sp_g, f"rD=0.075 model {model} gz", profile_floor(go, args[0], imp))
        check(dgz, do, sp_d, f"rD=0.075 model {model} dgz", profile_floor(go, args[0], imp))


def test_theis_gradient_is_zero_bitwise():
    d, pd = load_deck("theis-input.dat")
    tD = np.geomspace(0.1, 1e5, 24)
    sv = ub.split_index(tD, (2, 2))
    rD = np.geomspace(0.05, 3.0, 24)
    zD = np.linspace(0.0, 1.0, 24)
    gz, dgz, fl = ub.eval_points_dz(ub.Params(pd), tD, sv, rD, zD, want_flags=True)
    assert (gz == 0.0).all() and (dgz == 0.0).all()
    assert (fl == 1).all()        # every area is 0: the infint is stale everywhere


@pytest.mark.parametrize("name", ["hantush-input.dat", "hantush-storage-input.dat"])
def test_hantush_gradient_vanishes_at_bottom_and_top(name):
    """Models 1 and 2 have an impervious bottom and top: gz(0) = 0 bit for bit (layer 1's
    derivative is 2 G eta sinh(eta z), exactly 0 at z = 0), |gz(1)| <= 1e-9 max|gz| of the
    z-profile at that time."""
    d, pd = load_deck(name)
    prm = ub.Params(pd)
    it = np.arange(0, len(d["tD"]), 5)
    zs = np.linspace(0.0, 1.0, 41)
    T = np.repeat(d["tD"][it], len(zs)); S = np.repeat(d["sv"][it], len(zs))
    Z = np.tile(zs, len(it)); R = np.full(len(T), d["rD"][0])
    gz, _ = ub.eval_points_dz(prm, T, S, R, Z)
    gz = gz.reshape(len(it), len(zs))
    assert np.isfinite(gz).all()
    assert (gz[:, 0] == 0.0).all()
    top = np.abs(gz[:, -1]) / np.abs(gz).max(axis=1)
    print(f"{name}: worst |gz(1)|/max|gz| = {top.max():.2e}")
    assert top.max() <= 1e-9


WT_DECKS = [("cape-cod-neuman74.in", None), ("malama-fullpen-input.dat", 0.0)]


@pytest.mark.parametrize("name,beta", WT_DECKS)
def test_water_table_kinematic_condition(name, beta):
    """With beta = 0: gz(1) = -ds(1)/(alphaD tD), ds from unc_eval_points with zLay = 3, to
    1e-8 |rhs| + 12 spread (the oracle's noise on both sides, as in test_dz_host.py)."""
    d, pd = load_deck(name)
    if beta is not None:
        pd = dict(pd, beta=beta)
    assert pd["beta"] == 0.0
    n = len(d["tD"])
    args = (d["tD"], d["sv"], np.full(n, d["rD"][0]))
    one, three = np.ones(n), np.full(n, 3, np.int32)
    gz, _ = ub.eval_points_dz(ub.Params(pd), *args, one)
    _, ds = ub.eval_points(ub.Params(pd), *args, one, three)
    po = oracle.Params(pd)
    _, _, sg, _ = oracle_dz_with_noise(po, args + (one,))
    _, d0, _, sd = oracle.noise_envelope(lambda **k: oracle.eval_points(po, *args, one, three, **k), nsamples=4)
    dl = oracle.eval_points(po, *args, one, three, long_double=True)[1]
    sd = np.fmax(sd, np.abs(d0 - dl))
    rhs = -ds / (pd["alphaD"] * d["tD"])
    spread = sg + sd / (pd["alphaD"] * d["tD"])
    err = np.abs(gz - rhs)
    print(f"{name}: worst |gz(1) + ds(1)/(alphaD tD)| / |rhs| = {float(np.max(err / np.abs(rhs))):.3e}")
    assert np.isfinite(gz).all()
    ok = err <= 1e-8 * np.abs(rhs) + NOISE_K * spread
    assert ok.all(), np.argwhere(~ok)[:5].ravel()


def _segments(pd):
    """(z1, z2) inside each layer at least 0.01 thick (room for the h = 1e-3 stencil), away
    from its boundaries."""
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    out = []
    for lo, hi in ((0.0, b1), (b1, b2), (b2, 1.0)):
        if hi - lo >= 0.01:
            out.append((lo + 0.15 * (hi - lo), lo + 0.85 * (hi - lo)))
    return out


def test_gradient_consistent_with_point_values():
    """Not a parity bar: at well-conditioned times, away from the layer boundaries, (a) a 16-node
    Gauss-Legendre integral of gz over a segment inside one layer matches s(z2) - s(z1) of
    unc_eval_points, and (b) a 4th-order central difference of unc_eval_points (h = 1e-3) matches
    gz at the segment's middle; both to 1e-6 of max|gz| over the z-profile at that time."""
    x, w = np.polynomial.legendre.leggauss(16)
    h = 1e-3
    worst_int = worst_fd = 0.0
    for name in ("hantush-input.dat", "cape-cod-moench.in", "cape-cod-neuman74.in", "malama-fullpen-input.dat",
                 "mishra-neuman-malama.in"):
        d, pd = load_deck(name)
        prm = ub.Params(pd)
        tD = d["tD"][40::12]
        sv = d["sv"][40::12]
        nt = len(tD)
        rD = np.full(nt, d["rD"][0])
        zprof = np.linspace(0.0, 1.0, 101)
        gp, _ = ub.eval_points_dz(prm, np.repeat(tD, len(zprof)), np.repeat(sv, len(zprof)),
                                  np.repeat(rD, len(zprof)), np.tile(zprof, nt))
        gmax = np.abs(gp.reshape(nt, len(zprof))).max(axis=1)
        for z1, z2 in _segments(pd):
            zg = 0.5 * (z2 - z1) * x + 0.5 * (z2 + z1)
            zm = 0.5 * (z1 + z2)
            zz = np.concatenate([zg, [zm]])
            gz, _ = ub.eval_points_dz(prm, np.repeat(tD, len(zz)), np.repeat(sv, len(zz)), np.repeat(rD, len(zz)),
                                      np.tile(zz, nt))
            gz = gz.reshape(nt, len(zz))
            zs = np.concatenate([[z1, z2], zm + h * np.array([-2.0, -1.0, 1.0, 2.0])])
            lay = ub.zlay(zs, pd["lD"], pd["dD"])
            assert len(set(lay.tolist())) == 1
            s, _ = ub.eval_points(prm, np.repeat(tD, len(zs)), np.repeat(sv, len(zs)), np.repeat(rD, len(zs)),
                                  np.tile(zs, nt), np.tile(lay, nt))
            s = s.reshape(nt, len(zs))
            integral = (gz[:, :16] * w).sum(axis=1) * 0.5 * (z2 - z1)
            e_int = np.abs(integral - (s[:, 1] - s[:, 0])) / (gmax * (z2 - z1))
            fd = (s[:, 2] - 8.0 * s[:, 3] + 8.0 * s[:, 4] - s[:, 5]) / (12.0 * h)
            e_fd = np.abs(fd - gz[:, 16]) / gmax
            worst_int = max(worst_int, float(e_int.max()))
            worst_fd = max(worst_fd, float(e_fd.max()))
    print(f"gz vs point values: integral identity worst {worst_int:.3e}, central difference worst {worst_fd:.3e}")
    assert worst_int < 1e-6 and worst_fd < 1e-6, (worst_int, worst_fd)


def _big_set(n, seed=11):
    d, pd = load_deck("cape-cod-moench.in")
    rng = np.random.default_rng(seed)
    tD = 10.0 ** rng.uniform(-1, 6, n)
    sv = ub.split_index(tD, (2, 2))
    rD = rng.uniform(0.05, 3.0, n)
    zD = rng.uniform(0.0, 1.0, n)
    return pd, tD, sv, rD, zD


def test_plumbing_device_entry_cost_order_sharding_determinism():
    import torch
    pd, tD, sv, rD, zD = _big_set(20000)
    prm = ub.Params(pd)
    gz, dgz, fl = ub.eval_points_dz(prm, tD, sv, rD, zD, want_flags=True)            # cost-ordered (>= 16384)
    assert np.isfinite(gz).all() and np.isfinite(dgz).all()
    parts = [ub.eval_points_dz(prm, tD[i:i + 8000], sv[i:i + 8000], rD[i:i + 8000], zD[i:i + 8000])
             for i in range(0, 20000, 8000)]
    assert np.array_equal(gz, np.concatenate([p[0] for p in parts]))
    assert np.array_equal(dgz, np.concatenate([p[1] for p in parts]))
    g2, d2 = ub.eval_points_dz(prm, tD, sv, rD, zD)
    assert np.array_equal(gz, g2) and np.array_equal(dgz, d2)                        # deterministic
    # device entry == host entry
    m = 3000
    dev = lambda a, t: torch.as_tensor(np.ascontiguousarray(a[:m]), dtype=t, device="cuda")  # noqa: E731
    out_g = torch.empty(m, dtype=torch.float64, device="cuda")
    out_d = torch.empty(m, dtype=torch.float64, device="cuda")
    out_f = torch.empty(m, dtype=torch.int32, device="cuda")
    ub.set_device(0)
    ub.eval_points_dz_device(prm, dev(tD, torch.float64), dev(sv, torch.int32), dev(rD, torch.float64),
                             dev(zD, torch.float64), out_g, out_d, flags=out_f)
    torch.cuda.synchronize()
    hg, hd, hf = ub.eval_points_dz(prm, tD[:m], sv[:m], rD[:m], zD[:m], want_flags=True)
    assert np.array_equal(out_g.cpu().numpy(), hg) and np.array_equal(out_d.cpu().numpy(), hd)
    assert np.array_equal(out_f.cpu().numpy(), hf)
    if ub.device_count() > 1:
        g0, d0 = ub.eval_points_dz(prm, tD, sv, rD, zD, ngpu=0)
        assert np.array_equal(g0, gz) and np.array_equal(d0, dgz)


def _row_values(text):
    """Numeric columns of the data rows of an output file."""
    rows = [ln for ln in text.split("\n") if ln.strip() and not ln.startswith("#")]
    return np.array([[float(c) for c in ln.split()] for ln in rows])


@pytest.mark.parametrize("name", ["cape-cod-neuman74.in", "hantush-input.dat", "hantush-contours-input.dat"])
def test_cli_vertical_gradient_rows(name):
    """The rows of --vertical-gradient are unc_eval_points_dz at every (t, r, z) of the deck, with
    the reference's stale abscissae, times Hc/Lc for a dimensional deck; headers are unchanged."""
    from oracle import deck
    cli = os.path.join(ROOT, "cli", "unconfined_cli")
    subprocess.run(["make", "-C", os.path.join(ROOT, "cli")], check=True, capture_output=True)
    cfg = os.path.join(ROOT, "configs")

    def run(*a):
        r = subprocess.run([cli, name, *a], capture_output=True, text=True, cwd=cfg)
        assert r.returncode == 0, r.stderr
        return r.stdout
    plain, vg = run("--stdout"), run("--vertical-gradient", "--stdout")
    head = lambda t: [ln for ln in t.split("\n") if ln.startswith("#")]  # noqa: E731
    assert head(plain) == head(vg)
    d = deck.read_deck(os.path.join(cfg, name))
    pd = deck.params_dict(d)
    nt, nr, nz = len(d["tD"]), len(d["rD"]), len(d["zD"])
    ti = np.repeat(np.arange(nt), nr * nz)
    ri = np.tile(np.repeat(np.arange(nr), nz), nt)
    zi = np.tile(np.arange(nz), nt * nr)
    stale = np.full(len(ti), d["j0z"][d["sv"][0] - 1] / d["rD"][0])
    gz, dgz = ub.eval_points_dz(ub.Params(pd), d["tD"][ti], d["sv"][ti], d["rD"][ri], d["zD"][zi], ts_scale=stale)
    sc = 1.0 if d["dimless"] else d["Hc"] / d["Lc"]
    got = _row_values(vg)
    assert got.shape[0] == len(gz)
    want_g = np.array([float("%.15E" % v) for v in gz * sc])
    want_d = np.array([float("%.15E" % v) for v in dgz * sc])
    assert np.array_equal(got[:, -2], want_g, equal_nan=True) and np.array_equal(got[:, -1], want_d, equal_nan=True)
    assert not np.array_equal(_row_values(plain)[:, -2], got[:, -2])

"""Screened observation wells on the GPU (unc_eval_screens, lh_column_kernel<COL_SCREEN>): parity
with the oracle's screen mode on the decks of models 0-6, limits (a thin screen is a point, Theis
has no z dependence, a fully penetrating Hantush well is Theis), consistency with Gauss-Legendre
means of point values, and the plumbing (device entry, cost-ordered large calls, sharding,
determinism, command line)."""
import os
import subprocess

import numpy as np
import pytest

import unconfined_b200 as ub
from oracle import oracle
from oracle import screens as oscreens
from helpers import load_deck, stale_scale, ROOT

pytestmark = pytest.mark.gpu

# The parity bar of tests/helpers.py, restated for screens: a screen passes if
#   |gpu - oracle| <= RTOL*|oracle| + NOISE_K*spread
# where spread is how far the oracle's own result moves under <= 2-ulp libm jitter or in long
# double.  NaN patterns and flags must match exactly.
RTOL = 1e-9
NOISE_K = 12.0

DECKS = [("theis-input.dat", 0), ("hantush-input.dat", 1), ("hantush-storage-input.dat", 2),
         ("cape-cod-moench.in", 3), ("malama-fullpen-input.dat", 4), ("malama-partpen-input.dat", 5),
         ("cape-cod-neuman74.in", 5), ("mishra-neuman-malama.in", 6)]


def screens_for(pd):
    """Screens inside each layer, across one boundary and across both (where the deck has them)."""
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    if b1 <= 0.0 and b2 >= 1.0:
        return [(0.0, 1.0), (0.2, 0.35), (0.9, 1.0)]
    sc = [(0.1 * b1, 0.6 * b1)]
    if b2 > b1:
        sc += [(b1 + 0.2 * (b2 - b1), b1 + 0.7 * (b2 - b1)), (0.5 * b1, b1 + 0.5 * (b2 - b1))]
    if b2 < 1.0:
        sc += [(b2 + 0.3 * (1 - b2), 1.0), (b1 + 0.5 * (b2 - b1), b2 + 0.5 * (1 - b2)), (0.5 * b1, 1.0)]
    return sc


def screen_set(d, pd, every=10):
    """Every `every`-th time of the deck times every screen of screens_for."""
    it = np.arange(0, len(d["tD"]), every)
    sc = screens_for(pd)
    ti, si = np.meshgrid(it, np.arange(len(sc)), indexing="ij")
    ti, si = ti.ravel(), si.ravel()
    zb = np.array([sc[k][0] for k in si]); zt = np.array([sc[k][1] for k in si])
    rD = np.full(len(ti), d["rD"][0])
    return d["tD"][ti], d["sv"][ti], rD, zb, zt


def oracle_screens_with_noise(po, args, ts_scale=None, nsamples=4):
    f = lambda **k: oscreens.eval_screens(po, *args, ts_scale=ts_scale, **k)  # noqa: E731
    s0, d0, sp_s, sp_d = oscreens.noise_envelope(f, nsamples=nsamples)
    sl, dl, _ = f(long_double=True)
    with np.errstate(invalid="ignore"):
        sp_s = np.fmax(sp_s, np.abs(s0 - sl))
        sp_d = np.fmax(sp_d, np.abs(d0 - dl))
    return s0, d0, sp_s, sp_d


def check(got, want, spread, what):
    nan_same = np.isnan(got) == np.isnan(want)
    assert nan_same.all(), f"{what}: NaN pattern differs at {np.argwhere(~nan_same)[:5].ravel()}"
    ok = np.isnan(want) | (np.abs(got - want) <= RTOL * np.abs(want) + NOISE_K * spread) | (got == want)
    assert ok.all(), (f"{what}: {int((~ok).sum())} of {ok.size} fail; first {np.argwhere(~ok)[0]}: "
                      f"gpu={got[~ok][0]!r} oracle={want[~ok][0]!r} spread={spread[~ok][0]:.3e}")


@pytest.mark.parametrize("name,model", DECKS)
@pytest.mark.parametrize("stale", [False, True], ids=["fresh", "ts_scale"])
def test_screen_parity_with_oracle(name, model, stale):
    d, pd = load_deck(name)
    assert pd["model"] == model
    args = screen_set(d, pd)
    ts = np.full(len(args[0]), stale_scale(d)) if stale else None
    s, ds, fl = ub.eval_screens(ub.Params(pd), *args, ts_scale=ts, want_flags=True)
    so, do, sp_s, sp_d = oracle_screens_with_noise(oracle.Params(pd), args, ts_scale=ts)
    _, _, flo = oscreens.eval_screens(oracle.Params(pd), *args, ts_scale=ts)
    assert np.array_equal(fl, flo)
    check(s, so, sp_s, f"{name} s")
    check(ds, do, sp_d, f"{name} ds")


def test_small_radius_screens_literal_path_and_certain_nan():
    """rD = 0.075 (hantush-contours): the largest abscissae exceed the fast-path bound, so the
    literal screen path runs, and beyond Re(eta) = 718 the certain-NaN rule (sinh(eta) overflows)
    replaces it; those NaN abscissae truncate the Wynn series, so values and NaN pattern of the
    results must still be the oracle's."""
    d, pd = load_deck("hantush-contours-input.dat")
    tD = np.geomspace(1e-2, 1e4, 13)
    sv = ub.split_index(tD, (2, 2))
    sc = screens_for(pd)
    n = len(tD) * len(sc)
    args = (np.repeat(tD, len(sc)), np.repeat(sv, len(sc)), np.full(n, 0.075),
            np.tile([z[0] for z in sc], len(tD)), np.tile([z[1] for z in sc], len(tD)))
    for model in (1, 5):
        p = dict(pd, model=model, beta=0.0, alphaD=1e4)
        s, ds, fl = ub.eval_screens(ub.Params(p), *args, want_flags=True)
        so, do, sp_s, sp_d = oracle_screens_with_noise(oracle.Params(p), args)
        print(f"model {model}: {int(np.isnan(so).sum())} NaN of {n}")
        check(s, so, sp_s, f"rD=0.075 model {model} s")
        check(ds, do, sp_d, f"rD=0.075 model {model} ds")


def test_thin_screen_is_the_point_value_at_its_midpoint():
    for name in ("hantush-input.dat", "cape-cod-moench.in", "mishra-neuman-malama.in"):
        d, pd = load_deck(name)
        b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
        mids = np.array([0.3 * max(b1, 0.5), 0.8 * max(b1, 0.5), 0.5 * (b1 + b2)])   # layers 1, 1 and 2
        tD = d["tD"][::20]
        T, Z = np.meshgrid(tD, mids, indexing="ij")
        T, Z = T.ravel(), Z.ravel()
        sv = d["sv"][::20].repeat(len(mids))
        rD = np.full(len(T), d["rD"][0])
        lay = ub.zlay(Z, pd["lD"], pd["dD"])
        sp, dp = ub.eval_points(ub.Params(pd), T, sv, rD, Z, lay)
        ss, dss = ub.eval_screens(ub.Params(pd), T, sv, rD, Z - 0.5e-7, Z + 0.5e-7)
        _, _, sp_s, sp_d = oracle.noise_envelope(
            lambda **k: oracle.eval_points(oracle.Params(pd), T, sv, rD, Z, lay, **k), nsamples=4)
        check(ss, sp, sp_s, f"{name} thin screen s")
        check(dss, dp, sp_d, f"{name} thin screen ds")


def test_theis_screen_equals_point_bitwise():
    d, pd = load_deck("theis-input.dat")
    prm = ub.Params(pd)
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    tD = np.geomspace(0.1, 1e5, 24)
    sv = ub.split_index(tD, (2, 2))
    rD = np.geomspace(0.05, 3.0, 24)
    sp, dp = ub.eval_points(prm, tD, sv, rD, np.full(24, 0.3 * b1), ub.zlay(np.full(24, 0.3 * b1), pd["lD"], pd["dD"]))
    for zb, zt in ((0.1 * b1, 0.5 * b1), (b1 + 0.1 * (b2 - b1), b1 + 0.9 * (b2 - b1)), (0.0, 1.0)):
        ss, dss = ub.eval_screens(prm, tD, sv, rD, np.full(24, zb), np.full(24, zt))
        assert np.array_equal(ss, sp) and np.array_equal(dss, dp), (zb, zt)


def test_fully_penetrating_hantush_screen_is_theis():
    _, pd = load_deck("theis-contours-input.dat")
    tD = np.repeat([1.0, 30.0, 1e3, 1e5], 16)
    sv = ub.split_index(tD, (1, 1))
    rD = np.tile(np.geomspace(0.5, 40.0, 16), 4)
    zb, zt = np.zeros(len(tD)), np.ones(len(tD))
    th, dth = ub.eval_screens(ub.Params(dict(pd, model=0)), tD, sv, rD, zb, zt)
    ha, dha, fl = ub.eval_screens(ub.Params(dict(pd, model=1, lD=1.0, dD=0.0, bD=1.0)), tD, sv, rD, zb, zt,
                                  want_flags=True)
    assert not fl.any()
    for a, b in ((ha, th), (dha, dth)):
        a, b = a.reshape(4, 16), b.reshape(4, 16)
        err = np.abs(a - b) / np.abs(b).max(axis=1, keepdims=True)
        print("Hantush(full) screen - Theis: max |diff|/max|s| per time", err.max(axis=1))
        assert err.max() < 1e-9


def test_screen_agrees_with_gauss_legendre_mean_of_point_values():
    """At well-conditioned times the screen result is close to a 16-node Gauss-Legendre mean of
    GPU point values per segment; they differ because de Hoog and Wynn are nonlinear."""
    x, w = np.polynomial.legendre.leggauss(16)
    worst = 0.0
    for name in ("hantush-input.dat", "cape-cod-moench.in", "cape-cod-neuman74.in", "mishra-neuman-malama.in"):
        d, pd = load_deck(name)
        prm = ub.Params(pd)
        tD = d["tD"][40::12]
        sv = d["sv"][40::12]
        rD = np.full(len(tD), d["rD"][0])
        for zb, zt in screens_for(pd):
            ss, _ = ub.eval_screens(prm, tD, sv, rD, np.full(len(tD), zb), np.full(len(tD), zt))
            b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
            mean = np.zeros(len(tD))
            for lo, hi in ((zb, min(zt, b1)), (max(zb, b1), min(zt, b2)), (max(zb, b2), zt)):
                if not hi > lo:
                    continue
                z = 0.5 * (hi - lo) * x + 0.5 * (hi + lo)
                Z = np.tile(z, len(tD)); T = np.repeat(tD, 16)
                sp, _ = ub.eval_points(prm, T, np.repeat(sv, 16), np.repeat(rD, 16), Z, ub.zlay(Z, pd["lD"], pd["dD"]))
                mean += (sp.reshape(len(tD), 16) * (0.5 * w)).sum(axis=1) * (hi - lo) / (zt - zb)
            rel = np.abs(ss - mean) / np.abs(mean)
            worst = max(worst, float(rel.max()))
    print(f"screen vs 16-node Gauss-Legendre mean of point values: worst rel {worst:.3e}")
    assert worst < 1e-6, worst


def _big_set(n, seed=11):
    d, pd = load_deck("cape-cod-moench.in")
    rng = np.random.default_rng(seed)
    tD = 10.0 ** rng.uniform(-1, 6, n)
    sv = ub.split_index(tD, (2, 2))
    rD = rng.uniform(0.05, 3.0, n)
    wdt = 10.0 ** rng.uniform(-2, np.log10(0.5), n)
    zb = rng.uniform(0.0, 1.0 - wdt)
    return pd, tD, sv, rD, zb, zb + wdt


def test_plumbing_device_entry_cost_order_sharding_determinism():
    import torch
    pd, tD, sv, rD, zb, zt = _big_set(20000)
    prm = ub.Params(pd)
    s, ds, fl = ub.eval_screens(prm, tD, sv, rD, zb, zt, want_flags=True)            # cost-ordered (>= 16384)
    assert np.isfinite(s).all()
    parts = [ub.eval_screens(prm, tD[i:i + 8000], sv[i:i + 8000], rD[i:i + 8000], zb[i:i + 8000], zt[i:i + 8000])
             for i in range(0, 20000, 8000)]
    assert np.array_equal(s, np.concatenate([p[0] for p in parts]))
    assert np.array_equal(ds, np.concatenate([p[1] for p in parts]))
    s2, ds2 = ub.eval_screens(prm, tD, sv, rD, zb, zt)
    assert np.array_equal(s, s2) and np.array_equal(ds, ds2)                        # deterministic
    # device entry == host entry
    m = 3000
    dev = lambda a, t: torch.as_tensor(np.ascontiguousarray(a[:m]), dtype=t, device="cuda")  # noqa: E731
    out_s = torch.empty(m, dtype=torch.float64, device="cuda")
    out_d = torch.empty(m, dtype=torch.float64, device="cuda")
    out_f = torch.empty(m, dtype=torch.int32, device="cuda")
    ub.set_device(0)
    ub.eval_screens_device(prm, dev(tD, torch.float64), dev(sv, torch.int32), dev(rD, torch.float64),
                           dev(zb, torch.float64), dev(zt, torch.float64), out_s, out_d, flags=out_f)
    torch.cuda.synchronize()
    hs, hd, hf = ub.eval_screens(prm, tD[:m], sv[:m], rD[:m], zb[:m], zt[:m], want_flags=True)
    assert np.array_equal(out_s.cpu().numpy(), hs) and np.array_equal(out_d.cpu().numpy(), hd)
    assert np.array_equal(out_f.cpu().numpy(), hf)
    if ub.device_count() > 1:
        s0, d0 = ub.eval_screens(prm, tD, sv, rD, zb, zt, ngpu=0)
        assert np.array_equal(s0, s) and np.array_equal(d0, ds)


def fmt24(x):
    if np.isnan(x):
        return "NaN".rjust(24)
    m, e = ("%.15E" % x).split("E")
    return (m + "E%s%04d" % (e[0], int(e[1:]))).rjust(24)


def test_cli_exact_screen_writes_screen_means():
    from oracle import deck
    cli = os.path.join(ROOT, "cli", "unconfined_cli")
    subprocess.run(["make", "-C", os.path.join(ROOT, "cli")], check=True, capture_output=True)
    cfg = os.path.join(ROOT, "configs")
    name = "cape-cod-moench.in"

    def run(*a):
        r = subprocess.run([cli, name, *a], capture_output=True, text=True, cwd=cfg)
        assert r.returncode == 0, r.stderr
        return r.stdout
    plain, exact = run("--stdout"), run("--exact-screen", "--stdout")
    head = lambda t: [l for l in t.split("\n") if l.startswith("#")]  # noqa: E731
    rows = lambda t: [l for l in t.split("\n") if l and not l.startswith("#")]  # noqa: E731
    assert head(plain) == head(exact)
    d = deck.read_deck(os.path.join(cfg, name))
    pd = deck.params_dict(d)
    assert not d["piezometer"] and d["zTop"] > d["zBot"]
    n = len(d["tD"])
    stale = np.full(n, d["j0z"][d["sv"][0] - 1] / d["rD"][0])
    s, ds = ub.eval_screens(ub.Params(pd), d["tD"], d["sv"], np.full(n, d["rD"][0]),
                            np.full(n, d["zBot"] / d["Lc"]), np.full(n, d["zTop"] / d["Lc"]), ts_scale=stale)
    got = rows(exact)
    assert len(got) == n
    sc = 1.0 if d["dimless"] else d["Hc"]
    for i in range(n):
        tcol = d["tD"][i] if d["dimless"] else d["t"][i]
        assert got[i] == "%14.7E %s %s " % (tcol, fmt24(s[i] * sc), fmt24(ds[i] * sc)), i
    assert rows(plain) != got     # the reference's two-point rule is a different number

"""CPU tests of the vertical drawdown gradient (unc_eval_points_dz): the oracle's derivative
integrand against the fundamental theorem of calculus on its point integrand, continuity of the
slope across the layer boundaries, the device fast path (csrc/fast.cuh compiled for the host by
tests/hostcheck) against the oracle in long double and its overflow margin, the water-table
condition f'(1) = -(p/alphaD) f(1) of the Neuman-type models, argument validation of the C ABI
and the CLI flag."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import unconfined_b200 as ub
from oracle import oracle
from oracle import dz as odz
from unconfined_b200.build import _nvcc
from helpers import load_deck, ROOT

HC_DIR = os.path.join(ROOT, "tests", "hostcheck")

# one deck per model 0..6
DECKS = [("theis-input.dat", 0), ("hantush-input.dat", 1), ("hantush-storage-input.dat", 2),
         ("cape-cod-moench.in", 3), ("malama-fullpen-input.dat", 4), ("cape-cod-neuman74.in", 5),
         ("mishra-neuman-malama.in", 6)]


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    """The gradient fast path compiled for the host (tests/hostcheck/hostcheck_dz.cu)."""
    so = str(tmp_path_factory.mktemp("hostcheck") / "hostcheck_dz.so")
    subprocess.run([_nvcc(), "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-Xcompiler", "-fPIC", "-shared", "-o", so, os.path.join(HC_DIR, "hostcheck_dz.cu")],
                   check=True, capture_output=True)
    return C.CDLL(so)


def layer_segments(pd):
    """(z1, z2, layer) inside each layer the deck has, away from the boundaries."""
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    out = []
    if b1 > 0.0:
        out.append((0.1 * b1, 0.7 * b1, 1))
    if b2 > b1:
        out.append((b1 + 0.2 * (b2 - b1), b1 + 0.8 * (b2 - b1), 2))
    if b2 < 1.0:
        out.append((b2 + 0.25 * (1 - b2), 1.0, 3))
    return out


def set_mn(lib, pd):
    beta0 = pd["mn_ak"] * pd["mn_b"]
    vartheta = beta0 * pd["mn_Sy"] / (pd["Ss"] * pd["mn_b"]) * math.exp(-beta0 * (pd["mn_psia"] - pd["mn_psik"]) / pd["mn_b"])
    lib.hc_set_mn(C.c_double(vartheta), C.c_double(beta0 / 2))


@pytest.mark.parametrize("long_double", [False, True], ids=["double", "long_double"])
@pytest.mark.parametrize("name,model", DECKS)
def test_oracle_gradient_integrates_to_the_point_difference(name, model, long_double):
    """32-node Gauss-Legendre integral of soln_dz over a segment inside one layer equals
    soln(z2) - soln(z1) of the same precision (the branch switch MAXEXP of models 3-5 differs
    between double and long double), for every layer the deck has and several (a, p)."""
    d, pd = load_deck(name)
    assert pd["model"] == model
    po = oracle.Params(pd)
    x, w = np.polynomial.legendre.leggauss(32)
    worst, n = 0.0, 0
    for z1, z2, L in layer_segments(pd):
        z = 0.5 * (z2 - z1) * x + 0.5 * (z2 + z1)
        for tD in (0.3, 1e3):
            for a in (0.01, 0.5, 3.0, 20.0):
                integral = sum(wk * odz.soln_dz(po, a, 0.3, tD, zk, L, long_double=long_double)
                               for zk, wk in zip(z, w)) * (0.5 * (z2 - z1))
                f1 = odz.soln_value(po, a, 0.3, tD, z1, L, long_double=long_double)
                f2 = odz.soln_value(po, a, 0.3, tD, z2, L, long_double=long_double)
                diff = f2 - f1
                scale = np.maximum(np.abs(f1), np.abs(f2))
                ok = np.isfinite(integral) & np.isfinite(diff) & (scale > 0)
                assert ok.sum() >= len(ok) // 2
                worst = max(worst, float((np.abs(integral[ok] - diff[ok]) / scale[ok]).max()))
                n += int(ok.sum())
    assert n > 0
    print(f"{name}: worst |GL integral - difference| / max|soln| = {worst:.2e}")
    assert worst < 1e-12, worst


def _aux(pd, p):
    """Per-p tables of the point kernel: model 3 Moench sum, model 2 A0 and p tDb + 1."""
    if pd["model"] == 3:
        return sum(1 / (1 + p / g) for g in pd["moench_gamma"]), 0j
    if pd["model"] == 2:
        CDw = pd["rDw"] ** 2 / (2 * (pd["l"] - pd["d"]) * pd["Ss"])
        tDb = math.pi * pd["rDwobs"] ** 2 / (pd["sF"] * pd["Ss"])
        xi = pd["rDw"] * np.sqrt(p)
        K0, K1, _, _ = oracle.cbesk01(complex(xi))
        return 2 / (p * CDw * K0 + xi * K1), p * tDb + 1
    return 0j, 0j


def fast_dz(hc, pd, a, p, z, lay=0, aux=0j, aux2=0j):
    out = (C.c_double * 2)(); eta = (C.c_double * 2)()
    ok = hc.hc_fast_dz(int(pd["model"]), C.c_double(pd["kappa"]), C.c_double(pd["alphaD"]), C.c_double(pd["beta"]),
                       C.c_double(pd["lD"]), C.c_double(pd["dD"]), C.c_double(pd["bD"]),
                       len(pd.get("moench_gamma", [])), C.c_double(aux.real), C.c_double(aux.imag),
                       C.c_double(aux2.real), C.c_double(aux2.imag), C.c_double(a), C.c_double(p.real),
                       C.c_double(p.imag), C.c_double(z), int(lay), out, eta)
    return ok, complex(out[0], out[1]), complex(eta[0], eta[1])


CONT_DECKS = [("hantush-input.dat", 1), ("hantush-storage-input.dat", 2), ("cape-cod-moench.in", 3),
              ("cape-cod-neuman74.in", 5), ("malama-partpen-input.dat", 5)]


@pytest.mark.parametrize("name,model", CONT_DECKS)
def test_slope_is_continuous_across_layer_boundaries(hc, name, model):
    """The formulas of the layers on either side of 1-lD and of 1-dD give the same slope there:
    the oracle's to 1e-11 relative, the host-compiled fast path's to the same bar."""
    d, pd = load_deck(name)
    assert pd["model"] == model
    po = oracle.Params(pd)
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    bounds = [(b, lo, hi) for b, lo, hi in ((b1, 1, 2), (b2, 2, 3)) if 0.0 < b < 1.0]
    assert bounds
    worst_o, worst_f, nf = 0.0, 0.0, 0
    for b, lo, hi in bounds:
        for tD in (0.3, 30.0, 1e3):
            pv = oracle.pvalues(po, 2 * tD)
            for a in (0.01, 0.5, 3.0, 20.0):
                fl = odz.soln_dz(po, a, 0.3, tD, b, lo)
                fh = odz.soln_dz(po, a, 0.3, tD, b, hi)
                ok = np.isfinite(fl) & np.isfinite(fh)
                assert ok.sum() >= len(ok) // 2
                sc = np.maximum(np.abs(fl), np.abs(fh))[ok]
                worst_o = max(worst_o, float((np.abs(fl - fh)[ok] / sc).max()))
                for k in (0, 1, len(pv) // 2, len(pv) - 1):
                    p = complex(pv[k])
                    aux, aux2 = _aux(pd, p)
                    okl, gl, _ = fast_dz(hc, pd, a, p, b, lo, aux, aux2)
                    okh, gh, _ = fast_dz(hc, pd, a, p, b, hi, aux, aux2)
                    if okl and okh:
                        worst_f = max(worst_f, abs(gl - gh) / max(abs(gl), abs(gh)))
                        nf += 1
    print(f"{name}: slope jump oracle {worst_o:.2e}, fast path {worst_f:.2e}")
    assert nf > 20
    assert worst_o < 1e-11, worst_o
    assert worst_f < 1e-11, worst_f


@pytest.mark.parametrize("name,model", DECKS)
def test_device_gradient_closed_form_matches_long_double_oracle(hc, name, model):
    """hc_fast_dz (no common factor) against the long-double oracle at rD = 0 and lapTime = 1
    (time_type 3, delay 0), where the oracle's common factor is a itself.  The natural scale of
    a z-derivative is |eta| times that of the value, |2/(p+a^2)|/bD.  No point is excluded:
    where cp ~ cm (layer 1, every layer of model 6) the fast path forms 2 G sinh(eta z) without
    cancellation (eval_dz_split).  Where the literal formulas themselves cancel (above the pumping
    screen at large eta) the long-double oracle is the less accurate side: as in
    test_screens_host.py the bar adds 0.05 |double - long double|, and the rounding of the
    long-double layer-3 terms, which reach |eta| e^(Re(eta) dD) times the value's scale (2^-64
    of that)."""
    d, pd = load_deck(name)
    pq = dict(pd, time_type=3, time_par=[0.0, 1.0])
    po = oracle.Params(pq)
    if model == 6:
        set_mn(hc, pd)
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    zs = [0.0, 1e-5, 0.3 * max(b1, 0.0), 0.9 * max(b1, 0.0), 0.5 * (b1 + b2), b1, b2, 0.5 * (b2 + 1.0), 1.0]
    zs = sorted(set(z for z in zs if 0.0 <= z <= 1.0))
    worst, nfast = 0.0, 0
    for z in zs:
        lay = 1 if z < b1 else (2 if z < b2 else 3)
        for tD in (0.05, 3.0, 1e3):
            pv = oracle.pvalues(po, 2 * tD)
            for a in (1e-3, 0.03, 0.7, 5.0, 40.0, 150.0, 400.0 * math.sqrt(pd["kappa"]),
                      680.0 * math.sqrt(pd["kappa"])):
                want_all = odz.soln_dz(po, a, 0.0, tD, z, long_double=True) / a
                dbl_all = odz.soln_dz(po, a, 0.0, tD, z) / a
                for k in (0, 1, len(pv) // 2, len(pv) - 1):
                    p = complex(pv[k])
                    aux, aux2 = _aux(pd, p)
                    ok, got, eta = fast_dz(hc, pd, a, p, z, 0, aux, aux2)
                    if not ok:
                        assert eta.real > 345.0
                        continue
                    want = want_all[k]
                    if model == 0:
                        assert got == 0 and want == 0, (got, want)   # no z dependence
                        nfast += 1
                        continue
                    if not np.isfinite(want):
                        continue
                    if model in (3, 4, 5) and 12.0 < eta.real < 14.8:
                        continue   # MAXEXP = -log(eps)/3 is 12.01 in double, 14.7 in long double: other branch
                    nfast += 1
                    k0 = abs(2 / (p + a * a)) / (1.0 if model in (0, 4, 6) else pd["bD"])
                    scale = abs(eta) * k0
                    allow = 0.05 * abs(dbl_all[k] - want) if np.isfinite(dbl_all[k]) else 0.0
                    allow = max(allow, 2.0 ** -64 * scale * math.exp(eta.real * pd["dD"]))
                    worst = max(worst, max(abs(got - want) - allow, 0.0) / max(scale, abs(want)))
    print(f"{name}: worst {worst:.2e} over {nfast} fast-path values")
    assert nfast > 100
    assert worst < 2e-12, worst


@pytest.mark.parametrize("name,model", [("cape-cod-moench.in", 3), ("cape-cod-neuman74.in", 5)])
def test_device_gradient_at_the_bottom_keeps_the_water_table_term(hc, name, model):
    """At zD = 0 the Hantush part of layer 1 has zero slope and only the water-table term is
    left: exactly 0 where Re(eta) < MAXEXP (its cosh(eta z) form), and -eta udp(1) e^-eta/D'
    beyond (the reference's exp(eta(z-1)) form), which is far below an ulp of the layer's cp and
    cm.  The fast path must give 0 bit for bit where the long-double oracle does, and the term
    itself to 1e-12 relative elsewhere.  The literal formulas form udp(1) ~ e^(-eta dD) as the
    difference cosh(eta dD) - sinh(eta dD) of terms ~ e^(eta dD), so the long-double oracle holds
    it to 2^-64 e^(2 Re(eta) dD) only: the comparison stops where that exceeds 1e-14."""
    d, pd = load_deck(name)
    po = oracle.Params(dict(pd, time_type=3, time_par=[0.0, 1.0]))
    nz = nexp = 0
    worst = 0.0
    for tD in (0.05, 3.0, 1e3):
        pv = oracle.pvalues(po, 2 * tD)
        for a in np.geomspace(1e-3, 600.0 * math.sqrt(pd["kappa"]), 25):
            want_all = odz.soln_dz(po, a, 0.0, tD, 0.0, long_double=True) / a
            for k in (0, 1, len(pv) // 2, len(pv) - 1):
                p = complex(pv[k])
                aux, aux2 = _aux(pd, p)
                ok, got, eta = fast_dz(hc, pd, a, p, 0.0, 0, aux, aux2)
                if not ok or 12.0 < eta.real < 14.8:
                    continue   # MAXEXP differs between double and long double
                if 2.0 ** -64 * math.exp(2.0 * eta.real * pd["dD"]) > 1e-14:
                    continue
                want = want_all[k]
                if eta.real < 12.0:
                    assert got == 0 and want == 0, (a, p, got, want)
                    nz += 1
                else:
                    worst = max(worst, abs(got - want) / abs(want))
                    nexp += 1
    print(f"{name}: {nz} exact zeros, {nexp} water-table terms, worst rel {worst:.2e}")
    assert nz > 20 and nexp > 20
    assert worst < 1e-12, worst


@pytest.mark.parametrize("name,model", DECKS[1:])
def test_device_gradient_coefficients_do_not_overflow(hc, name, model):
    """Up to the fast-path bound (Re(eta) m = 700) and |Im eta| = 2e5 the derivative
    coefficients (0, eta cp, -eta cm) and eval_dz_fast stay finite wherever the value's
    coefficients are."""
    d, pd = load_deck(name)
    if model == 6:
        set_mn(hc, pd)
    m = 1.03 if model == 6 else (1.0 + pd["dD"])
    nchk = 0
    for er in np.concatenate([np.geomspace(1e-3, 690.0 / m, 40), [699.9 / m]]):
        for ei in np.concatenate([[0.0], np.geomspace(1e-3, 2e5, 40)]):
            aux = complex(len(pd.get("moench_gamma", [])) or 1.0)
            bad = hc.hc_dz_overflow_check(int(model), C.c_double(pd["kappa"]), C.c_double(pd["alphaD"]),
                                          C.c_double(pd["beta"]), C.c_double(pd["lD"]), C.c_double(pd["dD"]),
                                          C.c_double(pd["bD"]), len(pd.get("moench_gamma", [])),
                                          C.c_double(aux.real), C.c_double(aux.imag), C.c_double(er),
                                          C.c_double(ei))
            if bad < 0:
                continue
            assert bad == 0, (er, ei, bad)
            nchk += 1
    assert nchk > 1000


WT_DECKS = [("cape-cod-neuman74.in", 5, None), ("malama-fullpen-input.dat", 4, 0.0)]


def _wt_params(name, beta):
    d, pd = load_deck(name)
    if beta is not None:
        pd = dict(pd, beta=beta)
    assert pd["beta"] == 0.0 and pd["alphaD"] > 0
    return d, pd


@pytest.mark.parametrize("name,model,beta", WT_DECKS)
def test_oracle_water_table_condition(name, model, beta):
    """With beta = 0 the water table is a kinematic boundary: f'(1) = -(p/alphaD) f(1) of
    layer 3, term by term in the Laplace domain.  f(1) is the difference of the deck's value
    without the water-table term, u(1) (model 1 for model 5, Theis for model 4), and a term of
    the same size, which cancel when |xi| = |eta alphaD/p| is small.  f'(1) of model 5 contains
    u'(1), which is 0 in exact arithmetic (no flux through the top of the Hantush layer 3) and is
    rounded from two terms of size |eta sinh(eta dD)| theta/bD (theta: the Theis integrand with
    the common factor).  The bar is 1e-12 relative to the larger of (p/alphaD) max(|f(1)|, |u(1)|)
    and that size: the sizes of the terms both sides are rounded from."""
    d, pd = _wt_params(name, beta)
    assert pd["model"] == model
    po = oracle.Params(pd)
    pu = oracle.Params(dict(pd, model=1 if model == 5 else 0))
    pt = oracle.Params(dict(pd, model=0))
    worst = 0.0
    for tD in (d["tD"][10], d["tD"][len(d["tD"]) // 2], d["tD"][-1]):
        pv = oracle.pvalues(po, 2 * tD)
        for a in (0.01, 0.3, 3.0, 30.0):
            g = odz.soln_dz(po, a, d["rD"][0], tD, 1.0)
            f = odz.soln_value(po, a, d["rD"][0], tD, 1.0, 3)
            u = odz.soln_value(pu, a, d["rD"][0], tD, 1.0, 3)
            rhs = -(pv / pd["alphaD"]) * f
            th = odz.soln_value(pt, a, d["rD"][0], tD, 1.0, 3)
            eta = np.sqrt((pv + a * a) / pd["kappa"])
            scale = np.maximum(np.abs(pv / pd["alphaD"]) * np.maximum(np.abs(f), np.abs(u)),
                               np.abs(eta * np.sinh(eta * pd["dD"])) * np.abs(th) / pd["bD"])
            ok = np.isfinite(g) & np.isfinite(rhs) & (scale > 0)
            assert ok.sum() >= len(ok) // 2
            worst = max(worst, float((np.abs(g - rhs)[ok] / scale[ok]).max()))
    print(f"{name}: worst |f'(1) + (p/alphaD) f(1)| / scale = {worst:.2e}")
    assert worst < 1e-12, worst


@pytest.mark.parametrize("name,model,beta", WT_DECKS)
def test_oracle_water_table_condition_end_to_end(name, model, beta):
    """Through the whole algorithm: gz(zD = 1) = -ds(zD = 1, zLay = 3)/(alphaD tD) at the deck's
    times, to 1e-8 |rhs| + 12 spread.  spread: the oracle's own noise on both sides, the larger of
    its spread under 2-ulp libm jitter and its distance to long double (as tests/helpers.py)."""
    d, pd = _wt_params(name, beta)
    po = oracle.Params(pd)
    n = len(d["tD"])
    args = (d["tD"], d["sv"], np.full(n, d["rD"][0]))
    one, three = np.ones(n), np.full(n, 3, np.int32)
    gz, _, sg, _ = odz.noise_envelope(lambda: odz.eval_points_dz(po, *args, one), nsamples=4)
    gzl, _, _ = odz.eval_points_dz(po, *args, one, long_double=True)
    _, ds, _, sd = oracle.noise_envelope(lambda **k: oracle.eval_points(po, *args, one, three, **k), nsamples=4)
    dsl = oracle.eval_points(po, *args, one, three, long_double=True)[1]
    sg = np.fmax(sg, np.abs(gz - gzl))
    sd = np.fmax(sd, np.abs(ds - dsl))
    rhs = -ds / (pd["alphaD"] * d["tD"])
    spread = sg + sd / (pd["alphaD"] * d["tD"])
    err = np.abs(gz - rhs)
    ok = err <= 1e-8 * np.abs(rhs) + 12.0 * spread
    print(f"{name}: worst |gz(1) - rhs| / |rhs| = {float(np.max(err / np.abs(rhs))):.2e}")
    assert np.isfinite(gz).all() and ok.all(), np.argwhere(~ok)[:5].ravel()


def test_dz_abi_validation():
    d, pd = load_deck("cape-cod-moench.in")
    prm = ub.Params(pd)
    n = 3
    tD, sv, rD = d["tD"][:n], d["sv"][:n], np.full(n, d["rD"][0])
    zD = np.array([0.1, 0.5, 1.0])
    lib = ub.lib()
    for name in ("unc_eval_points_dz", "unc_eval_points_dz_device"):
        assert hasattr(lib, name)
    # n = 0 succeeds without touching a device
    g, dg = ub.eval_points_dz(prm, [], [], [], [])
    assert g.size == 0 and dg.size == 0
    for bad in (np.array([0.1, -1e-12, 0.3]), np.array([0.1, 0.2, 1.0 + 1e-12]), np.array([np.nan, 0.2, 0.3]),
                np.array([0.1, np.inf, 0.3]), np.array([0.1, 0.2, -np.inf])):
        with pytest.raises(ub.UncError) as e:
            ub.eval_points_dz(prm, tD, sv, rD, bad)
        assert e.value.code == -1, (bad, e.value)      # UNC_ERR_BAD_ARG, before UNC_ERR_NO_DEVICE
    dp = C.POINTER(C.c_double)
    arr = zD.ctypes.data_as(dp)
    svp = np.ascontiguousarray(sv, np.int32).ctypes.data_as(C.POINTER(C.c_int32))
    out = np.empty(n)
    rc = lib.unc_eval_points_dz(C.byref(prm.s), C.c_int64(n), arr, svp, arr, None, None, 1,
                                out.ctypes.data_as(dp), out.ctypes.data_as(dp), None)
    assert rc == -1                                     # NULL zD
    rc = lib.unc_eval_points_dz(C.byref(prm.s), C.c_int64(n), arr, svp, arr, arr, None, 1,
                                None, out.ctypes.data_as(dp), None)
    assert rc == -1                                     # NULL gz
    rc = lib.unc_eval_points_dz_device(C.byref(prm.s), C.c_int64(n), arr, svp, None, arr, None,
                                       out.ctypes.data_as(dp), out.ctypes.data_as(dp), None, None)
    assert rc == -1                                     # NULL rD
    if ub.device_count() == 0:
        with pytest.raises(ub.UncError) as e:
            ub.eval_points_dz(prm, tD, sv, rD, zD)
        assert e.value.code == -3


CLI = os.path.join(ROOT, "cli", "unconfined_cli")


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.join(ROOT, "cli")], check=True, capture_output=True)
    return CLI


def test_cli_vertical_gradient_flag(cli):
    deck = os.path.join(ROOT, "configs", "hantush-input.dat")
    h = subprocess.run([cli, deck, "--header-only"], capture_output=True, text=True, check=True).stdout
    hx = subprocess.run([cli, deck, "--vertical-gradient", "--header-only"], capture_output=True, text=True,
                        check=True).stdout
    assert h == hx
    dmp = subprocess.run([cli, deck, "--dump"], capture_output=True, text=True, check=True).stdout
    dmpx = subprocess.run([cli, deck, "--dump", "--vertical-gradient"], capture_output=True, text=True,
                          check=True).stdout
    assert dmp == dmpx
    usage = subprocess.run([cli, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--vertical-gradient" in usage and "dz" in usage
    # a screened observation well is refused before any device work
    scr = os.path.join(ROOT, "configs", "cape-cod-moench.in")
    r = subprocess.run([cli, scr, "--vertical-gradient", "--stdout"], capture_output=True, text=True)
    assert r.returncode == 1 and "--vertical-gradient" in r.stderr and "piezometer" in r.stderr

"""CPU tests of screened observation wells (unc_eval_screens): the oracle's screen-averaged
integrand against numerical quadrature of its point integrand, the device closed form
(csrc/fast.cuh compiled for the host by tests/hostcheck) against the oracle in long double,
S(x) = sinh(x)/x against mpmath, argument validation of the C ABI and the CLI flag."""
import ctypes as C
import math
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

import unconfined_b200 as ub
from oracle import oracle
from oracle import screens as oscreens
from unconfined_b200.build import _nvcc
from helpers import load_deck, ROOT

HC_DIR = os.path.join(ROOT, "tests", "hostcheck")

# one deck per model 0..6
DECKS = [("theis-input.dat", 0), ("hantush-input.dat", 1), ("hantush-storage-input.dat", 2),
         ("cape-cod-moench.in", 3), ("malama-fullpen-input.dat", 4), ("cape-cod-neuman74.in", 5),
         ("mishra-neuman-malama.in", 6)]


def _host_build(tmp_path_factory, src):
    so = str(tmp_path_factory.mktemp("hostcheck") / (os.path.splitext(src)[0] + ".so"))
    subprocess.run([_nvcc(), "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-Xcompiler", "-fPIC", "-shared", "-o", so, os.path.join(HC_DIR, src)],
                   check=True, capture_output=True)
    return C.CDLL(so)


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    """The screen fast path compiled for the host (tests/hostcheck/hostcheck_screens.cu)."""
    return _host_build(tmp_path_factory, "hostcheck_screens.cu")


@pytest.fixture(scope="module")
def hcp(tmp_path_factory):
    """The point fast path compiled for the host (tests/hostcheck/hostcheck.cu)."""
    return _host_build(tmp_path_factory, "hostcheck.cu")


def segments(zbot, ztop, lD, dD):
    """[u, v, layer] of the definition: split at 1-lD and 1-dD, empty segments dropped."""
    b1, b2 = 1.0 - lD, 1.0 - dD
    out = []
    for L, (lo, hi) in enumerate(((zbot, min(ztop, b1)), (max(zbot, b1), min(ztop, b2)), (max(zbot, b2), ztop))):
        if hi > lo:
            out.append((lo, hi, L + 1))
    return out


def screens_for(pd):
    """Screens inside each layer, across one boundary and across both (where the deck has them)."""
    b1, b2 = 1.0 - pd["lD"], 1.0 - pd["dD"]
    sc = [(0.1 * b1, 0.6 * b1)]                                   # layer 1
    if b2 > b1:
        sc.append((b1 + 0.2 * (b2 - b1), b1 + 0.7 * (b2 - b1)))   # layer 2
        sc.append((0.5 * b1, b1 + 0.5 * (b2 - b1)))               # across 1-lD
    if b2 < 1.0:
        sc.append((b2 + 0.3 * (1 - b2), 1.0))                     # layer 3
        sc.append((0.8 * b1 if b2 == b1 else b1 + 0.5 * (b2 - b1), b2 + 0.5 * (1 - b2)))   # across 1-dD
        sc.append((0.5 * b1, 1.0))                                # across both
    if b1 <= 0.0 and b2 >= 1.0:
        sc = [(0.0, 1.0), (0.2, 0.35), (0.9, 1.0)]
    return sc


def gl_mean(po, a, rD, tD, u, v, L, panels=4, order=24):
    """Composite Gauss-Legendre mean over [u, v] of the oracle's point integrand (layer L)."""
    x, w = np.polynomial.legendre.leggauss(order)
    acc = 0.0
    edges = np.linspace(u, v, panels + 1)
    for lo, hi in zip(edges[:-1], edges[1:]):
        z = 0.5 * (hi - lo) * x + 0.5 * (hi + lo)
        f = oracle.soln(po, a, rD, tD, z, np.full(len(z), L, np.int32))
        acc = acc + (f * (0.5 * (hi - lo) * w)).sum(axis=1)
    return acc / (v - u)


@pytest.mark.parametrize("name,model", DECKS)
def test_oracle_screen_integrand_matches_quadrature(name, model):
    d, pd = load_deck(name)
    assert pd["model"] == model
    po = oracle.Params(pd)
    worst, n = 0.0, 0
    for zbot, ztop in screens_for(pd):
        for tD in (0.3, 1e3):
            for a in (0.01, 0.5, 3.0, 20.0):
                want = None
                for (u, v, L) in segments(zbot, ztop, pd["lD"], pd["dD"]):
                    part = gl_mean(po, a, 0.3, tD, u, v, L) * ((v - u) / (ztop - zbot))
                    want = part if want is None else want + part
                got = oscreens.soln_screen(po, a, 0.3, tD, zbot, ztop)
                ok = np.isfinite(want) & np.isfinite(got)
                assert ok.sum() >= len(ok) // 2
                err = np.abs(got[ok] - want[ok]) / np.abs(want[ok])
                worst = max(worst, float(err.max()))
                n += int(ok.sum())
    assert n > 0
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


def fast_screen(hc, pd, a, p, zbot, ztop, aux=0j, aux2=0j):
    out = (C.c_double * 2)(); eta = (C.c_double * 2)()
    ok = hc.hc_fast_screen(int(pd["model"]), C.c_double(pd["kappa"]), C.c_double(pd["alphaD"]),
                           C.c_double(pd["beta"]), C.c_double(pd["lD"]), C.c_double(pd["dD"]),
                           C.c_double(pd["bD"]), len(pd.get("moench_gamma", [])), C.c_double(aux.real),
                           C.c_double(aux.imag), C.c_double(aux2.real), C.c_double(aux2.imag), C.c_double(a),
                           C.c_double(p.real), C.c_double(p.imag), C.c_double(zbot), C.c_double(ztop), out, eta)
    return ok, complex(out[0], out[1]), complex(eta[0], eta[1])


@pytest.mark.parametrize("name,model", DECKS)
def test_device_screen_closed_form_matches_long_double_oracle(hc, name, model):
    """hc_fast_screen (no common factor) against the long-double oracle at rD = 0 and
    lapTime = 1 (time_type 3, delay 0), where the oracle's common factor is a itself.  Where the
    literal formulas cancel (above the pumping screen at large eta) the long-double oracle itself
    is off by up to a few percent of the double oracle's error: the bar adds 0.05 |double - long
    double| (the quadrature test below holds the closed form to 2e-12 there as well)."""
    d, pd = load_deck(name)
    pq = dict(pd, time_type=3, time_par=[0.0, 1.0])
    po = oracle.Params(pq)
    if model == 6:
        beta0 = pd["mn_ak"] * pd["mn_b"]
        vartheta = beta0 * pd["mn_Sy"] / (pd["Ss"] * pd["mn_b"]) * math.exp(-beta0 * (pd["mn_psia"] - pd["mn_psik"]) / pd["mn_b"])
        hc.hc_set_mn(C.c_double(vartheta), C.c_double(beta0 / 2))
    sc = list(screens_for(pd))
    b1 = 1.0 - pd["lD"]
    # widths from 1e-8 to the whole aquifer: both branches of S(eta h)
    sc += [(0.5 * b1, 0.5 * b1 + 1e-8), (0.3 * b1, 0.3 * b1 + 1e-4), (0.0, 1.0)]
    worst, nfast = 0.0, 0
    for zbot, ztop in sc:
        for tD in (0.05, 3.0, 1e3):
            pv = oracle.pvalues(po, 2 * tD)
            # up to the fast-path bound: Re(eta) = a/sqrt(kappa) reaches ~700/(1+dD)
            for a in (1e-3, 0.03, 0.7, 5.0, 40.0, 150.0, 400.0 * math.sqrt(pd["kappa"]),
                      680.0 * math.sqrt(pd["kappa"])):
                want_all = oscreens.soln_screen(po, a, 0.0, tD, zbot, ztop, long_double=True) / a
                dbl_all = oscreens.soln_screen(po, a, 0.0, tD, zbot, ztop) / a
                for k in (0, 1, len(pv) // 2, len(pv) - 1):
                    p = complex(pv[k])
                    aux, aux2 = _aux(pd, p)
                    ok, got, eta = fast_screen(hc, pd, a, p, zbot, ztop, aux, aux2)
                    if not ok:
                        assert eta.real > 345.0
                        continue
                    want = want_all[k]
                    if not np.isfinite(want):
                        continue
                    if model in (3, 4, 5) and 12.0 < eta.real < 14.8:
                        continue   # MAXEXP = -log(eps)/3 is 12.01 in double, 14.7 in long double: other branch
                    nfast += 1
                    scale = abs(2 / (p + a * a)) / (1.0 if model in (0, 4, 6) else pd["bD"])
                    allow = 0.05 * abs(dbl_all[k] - want) if np.isfinite(dbl_all[k]) else 0.0
                    worst = max(worst, max(abs(got - want) - allow, 0.0) / max(scale, abs(want)))
    assert nfast > 100
    assert worst < 2e-12, worst


@pytest.mark.parametrize("name,model", DECKS)
def test_device_screen_closed_form_matches_quadrature_of_the_point_closed_form(hc, hcp, name, model):
    """The screen mean of the closed form against a composite Gauss-Legendre mean of the point
    closed form (hc_fast_soln, held to 2e-13 of the 40-digit literal formulas by
    test_fast_math_host.py), per segment; independent of the oracle's cancellation."""
    d, pd = load_deck(name)
    if model == 6:
        beta0 = pd["mn_ak"] * pd["mn_b"]
        vartheta = beta0 * pd["mn_Sy"] / (pd["Ss"] * pd["mn_b"]) * math.exp(-beta0 * (pd["mn_psia"] - pd["mn_psik"]) / pd["mn_b"])
        hc.hc_set_mn(C.c_double(vartheta), C.c_double(beta0 / 2))
        hcp.hc_set_mn(C.c_double(vartheta), C.c_double(beta0 / 2))
    po = oracle.Params(pd)
    x, w = np.polynomial.legendre.leggauss(24)
    worst, n = 0.0, 0
    for zbot, ztop in screens_for(pd):
        for tD in (0.05, 1e3):
            pv = oracle.pvalues(po, 2 * tD)
            for a in (0.03, 5.0, 150.0, 400.0 * math.sqrt(pd["kappa"])):
                for k in (0, 1, len(pv) - 1):
                    p = complex(pv[k])
                    aux, aux2 = _aux(pd, p)
                    ok, got, _ = fast_screen(hc, pd, a, p, zbot, ztop, aux, aux2)
                    if not ok:
                        continue
                    want = 0j
                    for (u, v, L) in segments(zbot, ztop, pd["lD"], pd["dD"]):
                        edges = np.linspace(u, v, 9)
                        for lo, hi in zip(edges[:-1], edges[1:]):
                            z = 0.5 * (hi - lo) * x + 0.5 * (hi + lo)
                            okp, f = _fast_points(hcp, pd, a, p, z, L, aux, aux2)
                            assert okp
                            want += (f * w).sum() * 0.5 * (hi - lo) / (ztop - zbot)
                    scale = abs(2 / (p + a * a)) / (1.0 if model in (0, 4, 6) else pd["bD"])
                    worst = max(worst, abs(got - want) / max(scale, abs(want)))
                    n += 1
    assert n > 20
    assert worst < 2e-12, worst


def _fast_points(hc, pd, a, p, zD, L, aux, aux2):
    n = len(zD)
    z = (C.c_double * n)(*zD); lay = (C.c_int * n)(*([int(L)] * n))
    out = (C.c_double * (2 * n))(); eta = (C.c_double * 2)()
    ok = hc.hc_fast_soln(int(pd["model"]), C.c_double(pd["kappa"]), C.c_double(pd["alphaD"]),
                         C.c_double(pd["beta"]), C.c_double(pd["lD"]), C.c_double(pd["dD"]),
                         C.c_double(pd["bD"]), len(pd.get("moench_gamma", [])), C.c_double(aux.real),
                         C.c_double(aux.imag), C.c_double(aux2.real), C.c_double(aux2.imag),
                         C.c_double(a), C.c_double(p.real), C.c_double(p.imag), n, z, lay, out, eta)
    return ok, np.array(out[:]).view(np.complex128)


def test_sinhc_matches_mpmath(hc):
    mp.mp.dps = 40
    out = (C.c_double * 2)()
    rng = np.random.default_rng(3)
    # eta h lies in the sector |arg| < pi/4 (Re(p + a^2) > 0); both branches, up to Re x = 350
    r = np.concatenate([10.0 ** rng.uniform(-9, math.log10(350.0), 600), [0.0, 1e-300, 0.49, 0.5, 0.51]])
    th = rng.uniform(-math.pi / 4, math.pi / 4, len(r))
    worst = 0.0
    for x in r * np.exp(1j * th):
        hc.hc_sinhc(C.c_double(x.real), C.c_double(x.imag), out)
        xm = mp.mpc(x.real, x.imag)
        want = mp.sinh(xm) / xm if xm != 0 else mp.mpf(1)
        worst = max(worst, float(abs(mp.mpc(out[0], out[1]) - want) / abs(want)))
    assert worst < 1e-15, worst        # a few ulp


def test_screen_abi_validation():
    d, pd = load_deck("cape-cod-moench.in")
    prm = ub.Params(pd)
    n = 3
    tD, sv, rD = d["tD"][:n], d["sv"][:n], np.full(n, d["rD"][0])
    zb, zt = np.array([0.1, 0.2, 0.3]), np.array([0.5, 0.6, 0.9])
    lib = ub.lib()
    for name in ("unc_eval_screens", "unc_eval_screens_device"):
        assert hasattr(lib, name)
    # n = 0 succeeds without touching a device
    s, ds = ub.eval_screens(prm, [], [], [], [], [])
    assert s.size == 0 and ds.size == 0
    bad = [(np.array([0.5, 0.2, 0.3]), zt),            # zbot == ztop
           (np.array([0.6, 0.2, 0.3]), zt),            # zbot > ztop
           (np.array([-0.1, 0.2, 0.3]), zt),           # below 0
           (zb, np.array([0.5, 1.2, 0.9])),            # above 1
           (np.array([np.nan, 0.2, 0.3]), zt),         # NaN
           (zb, np.array([0.5, np.inf, 0.9]))]         # Inf
    for b, t in bad:
        with pytest.raises(ub.UncError) as e:
            ub.eval_screens(prm, tD, sv, rD, b, t)
        assert e.value.code == -1, (b, t, e.value)      # UNC_ERR_BAD_ARG, before UNC_ERR_NO_DEVICE
    dp = C.POINTER(C.c_double)
    arr = zb.ctypes.data_as(dp)
    svp = np.ascontiguousarray(sv, np.int32).ctypes.data_as(C.POINTER(C.c_int32))
    out = np.empty(n)
    rc = lib.unc_eval_screens(C.byref(prm.s), C.c_int64(n), arr, svp, arr, None, arr, None, 1,
                              out.ctypes.data_as(dp), out.ctypes.data_as(dp), None)
    assert rc == -1                                     # NULL ztop
    rc = lib.unc_eval_screens_device(C.byref(prm.s), C.c_int64(n), arr, svp, arr, arr, None, None,
                                     out.ctypes.data_as(dp), out.ctypes.data_as(dp), None, None)
    assert rc == -1
    if ub.device_count() == 0:
        with pytest.raises(ub.UncError) as e:
            ub.eval_screens(prm, tD, sv, rD, zb, zt)
        assert e.value.code == -3


CLI = os.path.join(ROOT, "cli", "unconfined_cli")


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-C", os.path.join(ROOT, "cli")], check=True, capture_output=True)
    return CLI


def test_cli_exact_screen_flag_leaves_header_and_dump_unchanged(cli):
    deck = os.path.join(ROOT, "configs", "cape-cod-moench.in")
    h = subprocess.run([cli, deck, "--header-only"], capture_output=True, text=True, check=True).stdout
    hx = subprocess.run([cli, deck, "--exact-screen", "--header-only"], capture_output=True, text=True,
                        check=True).stdout
    assert h == hx and "screened obs well" in h
    dmp = subprocess.run([cli, deck, "--dump"], capture_output=True, text=True, check=True).stdout
    dmpx = subprocess.run([cli, deck, "--dump", "--exact-screen"], capture_output=True, text=True, check=True).stdout
    assert dmp == dmpx
    usage = subprocess.run([cli, "--help"], capture_output=True, text=True, check=True).stdout
    assert "--exact-screen" in usage

"""CPU tests of the PRODUCT's fast-path algebra (csrc/fast.cuh compiled for the host by
tests/hostcheck) against the oracle's literal restatement evaluated in long double at
single (a,p,z) points, for every model and layer.  This pins the closed forms used on the
GPU (classical Hantush layer functions, folded water-table term) to the reference formulas."""
import ctypes as C
import math
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

from oracle import oracle
from unconfined_b200.build import _nvcc
from helpers import load_deck, ROOT

HC_DIR = os.path.join(ROOT, "tests", "hostcheck")


@pytest.fixture(scope="module")
def hc():
    so = os.path.join(HC_DIR, "libhostcheck.so")
    src = os.path.join(HC_DIR, "hostcheck.cu")
    deps = [os.path.join(ROOT, "unconfined_b200", "csrc", f) for f in ("fast.cuh", "wynn.cuh", "cmath.cuh", "params.cuh")]
    if not os.path.exists(so) or max([os.path.getmtime(src)] + [os.path.getmtime(f) for f in deps]) > os.path.getmtime(so):
        subprocess.run([_nvcc(), "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                        "-Xcompiler", "-fPIC", "-shared", "-o", so, src], check=True, capture_output=True)
    return C.CDLL(so)


def test_exp_pm_and_sincos_accuracy(hc):
    mp.mp.dps = 40
    out = (C.c_double * 4)()
    rng = np.random.default_rng(0)
    worst = 0.0
    for x in np.concatenate([rng.uniform(-700, 700, 400), rng.uniform(-1, 1, 200), [0.0, 1e-9, -1e-5, 0.3465, -0.3467]]):
        hc.hc_exp_pm(C.c_double(x), out)
        ex = [mp.exp(x), mp.exp(-x), mp.cosh(x), mp.sinh(x)]
        for got, want in zip(out, ex):
            err = abs(mp.mpf(got) - want) / (abs(want) if want != 0 else 1)
            worst = max(worst, float(err))
    assert worst < 4.5e-16, worst                      # <= 2 ulp, sinh accurate for small x
    o2 = (C.c_double * 2)()
    worst = 0.0
    for y in np.concatenate([rng.uniform(-3000, 3000, 600), rng.uniform(-1, 1, 100), [0.0, math.pi / 2, 1e5, -1.9e5]]):
        hc.hc_sincos(C.c_double(y), o2)
        worst = max(worst, abs(o2[0] - float(mp.sin(mp.mpf(float(y))))), abs(o2[1] - float(mp.cos(mp.mpf(float(y))))))
    assert worst < 2.3e-16, worst                      # absolute (amplitude 1)


def fast_soln(hc, pd, a, p, zD, lay, aux=0j, aux2=0j):
    n = len(zD)
    z = (C.c_double * n)(*zD); l = (C.c_int * n)(*[int(x) for x in lay])
    out = (C.c_double * (2 * n))(); eta = (C.c_double * 2)()
    ok = hc.hc_fast_soln(int(pd["model"]), C.c_double(pd["kappa"]), C.c_double(pd["alphaD"]),
                         C.c_double(pd["beta"]), C.c_double(pd["lD"]), C.c_double(pd["dD"]),
                         C.c_double(pd["bD"]), len(pd.get("moench_gamma", [])), C.c_double(aux.real),
                         C.c_double(aux.imag), C.c_double(aux2.real), C.c_double(aux2.imag),
                         C.c_double(a), C.c_double(p.real), C.c_double(p.imag), n, z, l, out, eta)
    return ok, np.array(out[:]).view(np.complex128), complex(eta[0], eta[1])


CASES = [("hantush-input.dat", 1), ("cape-cod-neuman74.in", 5), ("cape-cod-moench.in", 3),
         ("malama-fullpen-input.dat", 4), ("theis-input.dat", 0), ("malama-partpen-input.dat", 5)]


def literal_truth(pd, a, p, z, L):
    """laplace_hankel_solutions.f90:30-116 exactly as written, in 40-digit arithmetic."""
    model = pd["model"]
    p = mp.mpc(p.real, p.imag)
    th = 2 / (p + a * a)
    if model == 0:
        return complex(th)
    eta = mp.sqrt((p + a * a) / pd["kappa"])
    dD1, lD1 = 1 - mp.mpf(pd["dD"]), 1 - mp.mpf(pd["lD"])

    def udp(z, L):
        ff1, ff2, sh = mp.sinh(eta * pd["dD"]), mp.sinh(eta * lD1), mp.sinh(eta)
        g2 = (ff1 * mp.cosh(eta * z) + ff2 * mp.cosh(eta * (1 - z))) / sh
        if L == 1:
            u = (mp.exp(-eta * lD1) - (ff1 + mp.exp(-eta) * ff2) / sh) * mp.cosh(eta * z)
        elif L == 2:
            u = 1 - g2
        else:
            u = mp.cosh(eta * (dD1 - z)) - g2
        return u * th / pd["bD"]
    if model == 1:
        return complex(udp(z, L))
    xi = eta * pd["alphaD"] / p
    if model == 3:
        xi = xi * len(pd["moench_gamma"]) / sum(1 / (1 + p / g) for g in pd["moench_gamma"])
    u = th if model == 4 else udp(z, L)
    top = th if model == 4 else udp(mp.mpf(1), 3)
    if eta.real < mp.mpf("12.014551129705717"):
        f = u - top * mp.cosh(eta * z) / ((1 + pd["beta"] * eta * xi) * mp.cosh(eta) + xi * mp.sinh(eta))
    else:
        f = u - top * mp.exp(eta * (z - 1)) / (1 + pd["beta"] * eta * xi + xi)
    return complex(f)


@pytest.mark.parametrize("name,model", CASES)
def test_fast_path_matches_literal_formulas(hc, name, model):
    mp.mp.dps = 40
    d, pd = load_deck(name)
    assert pd["model"] == model
    po = oracle.Params(pd)
    zD = np.array([0.0, 0.1, 0.5 * (1 - pd["lD"]), 1 - pd["lD"] + 0.3 * pd["bD"], 1 - pd["lD"] + 0.9 * pd["bD"],
                   1 - 0.5 * pd["dD"], 1.0])
    lay = oracle.zlay(zD, pd["lD"], pd["dD"])
    worst = 0.0
    for tD in (0.05, 3.0, 1e3, 1e7):
        pv = oracle.pvalues(po, 2 * tD)
        for a in (1e-4, 0.03, 0.7, 5.0, 40.0, 150.0):
            for k in (0, 1, len(pv) // 2, len(pv) - 1):
                aux = 0j
                if model == 3:
                    aux = sum(1 / (1 + pv[k] / g) for g in pd["moench_gamma"])
                ok, got, eta = fast_soln(hc, pd, a, complex(pv[k]), zD, lay, aux)
                if not ok:
                    assert eta.real > 345.0
                    continue
                scale = abs(2 / (pv[k] + a * a)) / (1.0 if model in (0, 4) else pd["bD"])
                for i in range(len(zD)):
                    tr = literal_truth(pd, a, complex(pv[k]), mp.mpf(float(zD[i])), int(lay[i]))
                    # relative to the natural scale of the kernel (|theis|/bD) or to the value
                    # itself where a layer formula is used outside its range (zD=1 is
                    # classified "beside the screen" by driver_io.f90:579-581 and blows up)
                    worst = max(worst, abs(got[i] - tr) / max(scale, abs(tr)))
    assert worst < 2e-13, worst


def test_fast_path_is_closer_to_long_double_truth_than_the_double_literal(hc):
    """Where the reference's expressions cancel (above the screen, large eta) the closed form
    keeps its digits: compare both against the long-double evaluation of the literal formulas."""
    d, pd = load_deck("hantush-input.dat")
    pq = dict(pd, time_type=3, time_par=[0.0, 1.0])
    po = oracle.Params(pq)
    zD = np.array([0.97, 0.99]); lay = oracle.zlay(zD, pd["lD"], pd["dD"])
    assert lay.tolist() == [3, 3]
    tD, a = 1.0, 60.0
    pv = oracle.pvalues(po, 2 * tD)
    ref_d = oracle.soln(po, a, 0.0, tD, zD, lay) / a
    # long double literal via eval of the same routine is not exposed per point; use mpmath
    mp.mp.dps = 40
    k = 3
    p = mp.mpc(pv[k].real, pv[k].imag)
    eta = mp.sqrt((p + a * a) / pd["kappa"])
    dD1, lD1 = 1 - mp.mpf(pd["dD"]), 1 - mp.mpf(pd["lD"])
    truth = []
    for z in zD:
        g1 = mp.cosh(eta * (dD1 - z))
        g2 = (mp.sinh(eta * pd["dD"]) * mp.cosh(eta * z) + mp.sinh(eta * lD1) * mp.cosh(eta * (1 - z))) / mp.sinh(eta)
        truth.append(complex((g1 - g2) * 2 / (p + a * a) / pd["bD"]))
    truth = np.array(truth)
    ok, got, _ = fast_soln(hc, pd, a, complex(pv[k]), zD, lay)
    assert ok
    e_fast = np.abs(got - truth) / np.abs(truth)
    e_lit = np.abs(ref_d[k] - truth) / np.abs(truth)
    assert e_fast.max() < 1e-12
    assert e_fast.max() <= e_lit.max() * 1.01 + 1e-15


def _hc_wynn(hc, series, which):
    s = np.ascontiguousarray(series, np.complex128)
    out = (C.c_double * 2)()
    hc.hc_wynn(s.view(np.float64).ctypes.data_as(C.POINTER(C.c_double)), len(s), which, out)
    return complex(out[0], out[1])


def test_device_wynn_matches_oracle_including_edge_semantics(hc):
    """Both device implementations (local-memory column order, register 'moving lozenge')
    against the oracle's restatement of integration.f90:125-189: full table, truncation,
    sentinel, and the order-dependent |denom|<=epsilon early exit."""
    rng = np.random.default_rng(5)
    cases = []
    for n in (2, 3, 4, 5, 7, 10, 11, 12):
        for _ in range(6):
            k = np.arange(n)
            s = (-1.0) ** k / (k + 1 + rng.uniform(0, 2)) * (1 + 0.3j * rng.uniform(-1, 1, n))
            cases.append(s)
    # geometric (nearly exactly summable -> tiny denominators and 'epsilon cancel' exits)
    for n in (6, 10, 12):
        cases.append(np.array([0.5 ** i for i in range(n)], complex))
        cases.append(np.array([(-0.25) ** i * (1 + 1j) for i in range(n)], complex))
        cases.append(np.array([1.0, 0.5] + [1e-17 * 0.1 ** i for i in range(n - 2)], complex))
        cases.append(np.array([1e-20 * (-0.5) ** i for i in range(n)], complex))   # everything below epsilon
    # cancels placed at different (column,row) positions
    base = np.array([(-1.0) ** i / (i + 1.0) for i in range(12)], complex)
    for pos in range(2, 11):
        s = base.copy(); s[pos] = 0.0
        cases.append(s)
        s = base.copy(); s[pos] = 1e-18; s[pos - 1] = 1e-18
        cases.append(s)
    # non-finite terms: truncation and sentinel
    for pos in (0, 2, 3, 4, 5, 8, 11):
        s = base.copy(); s[pos] = complex(np.inf, 0)
        cases.append(s)
        s = base.copy(); s[pos] = complex(0, np.nan)
        cases.append(s)
    # random series with exact repeats (zero differences in higher columns too), tiny terms and
    # non-finite entries at random places: ill-conditioned, so only the two lozenge versions are
    # compared with each other (bitwise)
    rand_cases = []
    for _ in range(300):
        n = int(rng.integers(2, 15))
        s = rng.normal(size=n) * 10.0 ** rng.uniform(-3, 1, n) * np.exp(1j * rng.uniform(0, 6.3, n))
        r = rng.uniform()
        if r < 0.3:
            s[rng.integers(0, n)] = 0.0
        elif r < 0.5:
            i = rng.integers(1, n); s[i] = -s[i - 1]
        elif r < 0.6:
            s[rng.integers(0, n)] = complex(np.nan, 0)
        elif r < 0.7:
            s[rng.integers(1, n):] = 0.0
        rand_cases.append(s)
    n_cancel = 0
    for s in cases:
        want, info = oracle.wynn(s)
        n_cancel += info == 3
        for which in (0, 1, 2, 3, 4, 5):
            if which == 2 and len(s) > 12:      # the register version is instantiated for 12 terms
                continue
            got = _hc_wynn(hc, s, which)
            assert abs(got - want) <= 1e-12 * max(abs(want), 1e-300) + 1e-300, (which, info, s, got, want)
    # two diagonals in lockstep (the grid kernel's) = the sequential lozenge, bit for bit
    n_exit = 0
    for s in cases + rand_cases:
        g4, g5 = _hc_wynn(hc, s, 4), _hc_wynn(hc, s, 5)
        assert (g4 == g5) or (g4 != g4 and g5 != g5), (s, g4, g5)
        n_exit += oracle.wynn(s)[1] == 3
    assert n_exit >= 40
    assert n_cancel >= 5        # the early-exit branch was really exercised


def test_model6_fast_path_matches_literal_formula(hc):
    """mishraNeumanMalama (laplace_hankel_solutions.f90:404-442) closed form vs the formula
    as written, in 40-digit arithmetic.  u = u0(1 - sqrt(1 + (eta1/u0)^2)) cancels in double
    for |eta1| << u0 (in the reference too): that part of the error is bounded separately."""
    mp.mp.dps = 40
    d, pd = load_deck("mishra-neuman-malama.in")
    assert pd["model"] == 6 and pd["mn_type"] == 1
    po = oracle.Params(pd)
    beta0 = pd["mn_ak"] * pd["mn_b"]
    vartheta = beta0 * pd["mn_Sy"] / (pd["Ss"] * pd["mn_b"]) * math.exp(-beta0 * (pd["mn_psia"] - pd["mn_psik"]) / pd["mn_b"])
    u0 = beta0 / 2
    hc.hc_set_mn(C.c_double(vartheta), C.c_double(u0))
    zD = np.array([0.0, 0.2, 0.77, 1.0]); lay = np.array([1, 1, 1, 1])
    worst = 0.0
    for tD in (0.05, 3.0, 1e3, 1e7):
        pv = oracle.pvalues(po, 2 * tD)
        # a >= 360: Re(eta) > 350, where |Delta0|^2 overflows although Delta0 does not (the fast
        # path is accepted up to Re(eta) = 700/1.03; reachable for rD < 0.1 at kappa = 1)
        for a in (1e-3, 0.03, 0.7, 5.0, 40.0, 150.0, 250.0, 360.0 * math.sqrt(pd["kappa"]),
                  600.0 * math.sqrt(pd["kappa"]), 670.0 * math.sqrt(pd["kappa"])):
            for k in (0, 1, len(pv) // 2, len(pv) - 1):
                ok, got, eta = fast_soln(hc, pd, a, complex(pv[k]), zD, lay)
                assert ok
                p = mp.mpc(pv[k].real, pv[k].imag)
                eta1 = mp.sqrt((p * vartheta + a * a) / pd["kappa"])
                v = mp.sqrt(1 + (eta1 / u0) ** 2)
                u = u0 * (1 - v)
                etasq = (p + a * a) / pd["kappa"]
                et = mp.sqrt(etasq)
                D0 = et * mp.sinh(et) - u * mp.cosh(et)
                for i, z in enumerate(zD):
                    tr = 2 / (pd["kappa"] * etasq) * (1 + u / D0 * mp.cosh(et * z))
                    cancel = 4 * 2.2e-16 * u0 * abs(2 / (pd["kappa"] * etasq) * mp.cosh(et * z) / D0)
                    err = abs(got[i] - complex(tr))
                    assert err <= 2e-13 * abs(tr) + float(cancel), (tD, a, k, z, got[i], complex(tr))
                    worst = max(worst, err / abs(tr))
    assert worst < 1e-6

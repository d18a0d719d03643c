"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the CPU oracle (oracle/liboracle.so).

PARITY UNPINNED (no Fortran compiler, no reference golden outputs): see
oracle/oracle_math.hpp.  Imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs only; never by unconfined_b200/.
"""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class OrcParams(C.Structure):
    # same layout as orc::params (oracle_core.hpp)
    _fields_ = [
        ("model", C.c_int32), ("M", C.c_int32),
        ("alpha", C.c_double), ("tol", C.c_double), ("tee_mult", C.c_double),
        ("time_type", C.c_int32), ("n_time_par", C.c_int32),
        ("time_par", C.POINTER(C.c_double)),
        ("ts_k", C.c_int32), ("ts_R", C.c_int32), ("gl_nacc", C.c_int32), ("gl_ord", C.c_int32),
        ("n_j0z", C.c_int32), ("moench_M", C.c_int32),
        ("j0z", C.POINTER(C.c_double)), ("moench_gamma", C.POINTER(C.c_double)),
        ("kappa", C.c_double), ("alphaD", C.c_double), ("beta", C.c_double),
        ("lD", C.c_double), ("dD", C.c_double), ("bD", C.c_double), ("rDw", C.c_double),
        ("l", C.c_double), ("d", C.c_double), ("Ss", C.c_double), ("rDwobs", C.c_double),
        ("sF", C.c_double),
        ("mn_type", C.c_int32), ("mn_reserved", C.c_int32),
        ("mn_ak", C.c_double), ("mn_psia", C.c_double), ("mn_psik", C.c_double),
        ("mn_b", C.c_double), ("mn_Sy", C.c_double),
    ]


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("oracle_capi.cpp", "oracle_core.hpp", "oracle_math.hpp")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["make", "-C", _HERE, "liboracle.so"], check=True, capture_output=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.orc_dehoog.restype = C.c_double
    return _LIB


def use_native_build():
    """bench.py's CPU arm only: build the port ON THIS HOST with the reference's release flags
    (-O3 -march=native -flto -fopenmp, Makefile:32 of the reference) and time that build.
    It is built in a fresh temporary directory: -march=native must never reuse a build made on
    another host, and the benchmark writes nothing into the tree (which may be read-only).
    Falls back to the portable test build (x86-64-v3, no contraction) if the compile fails."""
    global _LIB
    tmp = tempfile.mkdtemp(prefix="oracle_native_")
    so = os.path.join(tmp, "liboracle_native.so")
    try:
        subprocess.run(["make", "-C", _HERE, "native", "NATIVE_SO=" + so], check=True, capture_output=True)
        _LIB = C.CDLL(so)
        _LIB.orc_dehoog.restype = C.c_double
        return "g++ -O3 -march=native -flto -fopenmp (the reference's Makefile:32 flags), built on this host"
    except Exception as e:  # noqa: BLE001
        lib()
        return f"portable test build -O3 -march=x86-64-v3 -ffp-contract=off (native build failed: {e})"
    finally:
        shutil.rmtree(tmp, ignore_errors=True)     # the loaded library stays mapped


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


class Params:
    """Owns the numpy arrays behind an OrcParams."""

    def __init__(self, d):
        self.d = dict(d)
        self._tp = np.ascontiguousarray(d.get("time_par", [0.0, 1.0]), dtype=np.float64)
        self._j0 = np.ascontiguousarray(d["j0z"], dtype=np.float64)
        self._mg = np.ascontiguousarray(d.get("moench_gamma", []), dtype=np.float64)
        s = OrcParams()
        for k in ("model", "M", "alpha", "tol", "ts_k", "ts_R", "gl_nacc", "gl_ord", "kappa",
                  "alphaD", "beta", "lD", "dD", "bD", "rDw", "l", "d", "Ss", "rDwobs", "sF"):
            setattr(s, k, d[k])
        for k in ("mn_type", "mn_ak", "mn_psia", "mn_psik", "mn_b", "mn_Sy"):
            setattr(s, k, d.get(k, 0))
        s.tee_mult = d.get("tee_mult", 2.0)
        s.time_type = d.get("time_type", 1)
        s.n_time_par = len(self._tp)
        s.time_par = _dp(self._tp)
        s.n_j0z = len(self._j0)
        s.j0z = _dp(self._j0)
        s.moench_M = len(self._mg)
        s.moench_gamma = _dp(self._mg) if len(self._mg) else None
        self.s = s

    @property
    def np_(self):
        return 2 * self.d["M"] + 1


def eval_grid(prm, tD, sv, rD, zD, zLay, ts_scale=None, carry=True, nthreads=0, long_double=False):
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zD = np.ascontiguousarray(zD, np.float64)
    sv = np.ascontiguousarray(sv, np.int32); zLay = np.ascontiguousarray(zLay, np.int32)
    nt, nr, nz = len(tD), len(rD), len(zD)
    s = np.empty((nt, nr, nz)); ds = np.empty((nt, nr, nz))
    fl = np.zeros((nt, nr, nz), np.int32)
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(np.broadcast_to(ts_scale, (nt, nr)), np.float64)
        sc = _dp(scv)
    fn = lib().orc_eval_grid_ld if long_double else lib().orc_eval_grid
    rc = fn(C.byref(prm.s), nt, _dp(tD), _ip(sv), nr, _dp(rD), nz, _dp(zD), _ip(zLay), sc,
            int(carry), int(nthreads), _dp(s), _dp(ds), _ip(fl))
    assert rc == 0
    return s, ds, fl


def eval_points(prm, tD, sv, rD, zD, zLay, ts_scale=None, nthreads=0, long_double=False):
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zD = np.ascontiguousarray(zD, np.float64)
    sv = np.ascontiguousarray(sv, np.int32); zLay = np.ascontiguousarray(zLay, np.int32)
    n = len(tD)
    s = np.empty(n); ds = np.empty(n); fl = np.zeros(n, np.int32)
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(ts_scale, np.float64)
        sc = _dp(scv)
    fn = lib().orc_eval_points_ld if long_double else lib().orc_eval_points
    rc = fn(C.byref(prm.s), C.c_int64(n), _dp(tD), _ip(sv), _dp(rD), _dp(zD), _ip(zLay), sc,
            int(nthreads), _dp(s), _dp(ds), _ip(fl))
    assert rc == 0
    return s, ds, fl


def j0_zeros(n):
    out = np.empty(n)
    lib().orc_j0_zeros(n, _dp(out))
    return out


def split_index(tD, j0s):
    tD = np.ascontiguousarray(tD, np.float64)
    sv = np.empty(len(tD), np.int32)
    lib().orc_split_index(len(tD), _dp(tD), int(j0s[0]), int(j0s[1]), _ip(sv))
    return sv


def zlay(zD, lD, dD):
    zD = np.ascontiguousarray(zD, np.float64)
    out = np.empty(len(zD), np.int32)
    lib().orc_zlay(len(zD), _dp(zD), C.c_double(lD), C.c_double(dD), _ip(out))
    return out


def tanh_sinh(k, s=1.0):
    n = 2 ** k - 1
    w = np.empty(n); a = np.empty(n)
    lib().orc_tanh_sinh(k, C.c_double(s), _dp(w), _dp(a))
    return w, a


def gauss_lobatto(ord_):
    x = np.empty(ord_ - 2); w = np.empty(ord_ - 2)
    lib().orc_gauss_lobatto(ord_, _dp(x), _dp(w))
    return x, w


def wynn(series):
    s = np.ascontiguousarray(series, np.complex128)
    out = np.empty(2)
    info = lib().orc_wynn(_dp(s.view(np.float64)), len(s), _dp(out))
    return complex(out[0], out[1]), info


def extrap(x, y):
    x = np.ascontiguousarray(x, np.float64); y = np.ascontiguousarray(y, np.complex128)
    out = np.empty(2)
    lib().orc_extrap(_dp(x), _dp(y.view(np.float64)), len(x), _dp(out))
    return complex(out[0], out[1])


def pvalues(prm, tee):
    p = np.empty(prm.np_, np.complex128)
    lib().orc_pvalues(C.byref(prm.s), C.c_double(tee), _dp(p.view(np.float64)))
    return p


def dehoog(prm, t, tee, fp):
    fp = np.ascontiguousarray(fp, np.complex128)
    assert len(fp) == prm.np_
    return lib().orc_dehoog(C.byref(prm.s), C.c_double(t), C.c_double(tee), _dp(fp.view(np.float64)))


def lap_time(prm, p):
    p = np.ascontiguousarray(p, np.complex128)
    out = np.empty(len(p), np.complex128)
    lib().orc_lap_time(C.byref(prm.s), len(p), _dp(p.view(np.float64)), _dp(out.view(np.float64)))
    return out


def cbesk01(z):
    out = np.empty(4); nz = C.c_int(0)
    ierr = lib().orc_cbesk01(C.c_double(z.real), C.c_double(z.imag), _dp(out), C.byref(nz))
    return complex(out[0], out[1]), complex(out[2], out[3]), ierr, nz.value


def soln(prm, a, rD, tD, zD, zLay):
    zD = np.ascontiguousarray(zD, np.float64); zLay = np.ascontiguousarray(zLay, np.int32)
    out = np.empty((prm.np_, len(zD)), np.complex128)
    lib().orc_soln(C.byref(prm.s), C.c_double(a), C.c_double(rD), C.c_double(tD), len(zD), _dp(zD),
                   _ip(zLay), _dp(out.view(np.float64)))
    return out


def set_jitter(ulps, seed=0):
    """Perturb every libm result by up to `ulps` units in the last place (0 = off)."""
    lib().orc_set_jitter(C.c_double(ulps), C.c_ulonglong(seed))


def noise_envelope(fn, nsamples=4, ulps=2.0):
    """Run fn() (returning (s, ds, ...)) unperturbed and `nsamples` times under jitter;
    return (s, ds, spread_s, spread_ds) with spread = max |jittered - clean|."""
    set_jitter(0.0)
    base = fn()
    s0, d0 = np.array(base[0]), np.array(base[1])
    sp_s = np.zeros_like(s0); sp_d = np.zeros_like(d0)
    try:
        for k in range(nsamples):
            set_jitter(ulps, 1000 + k)
            r = fn()
            with np.errstate(invalid="ignore"):
                sp_s = np.fmax(sp_s, np.abs(np.array(r[0]) - s0))
                sp_d = np.fmax(sp_d, np.abs(np.array(r[1]) - d0))
    finally:
        set_jitter(0.0)
    return s0, d0, sp_s, sp_d


def num_threads():
    return lib().orc_num_threads()

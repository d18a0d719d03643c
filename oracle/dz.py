"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the vertical-gradient oracle
(oracle/liboracle_dz.so, built from oracle_dz_capi.cpp + oracle_dz.hpp on top of oracle_core.hpp).

The CPU restatement of unc_eval_points_dz's definition (include/unconfined_b200.h): the point
algorithm of oracle.eval_points with the integrand replaced by its z-derivative, layers geometric
(1 below 1-lD, 2 below 1-dD, else 3).  Imported by tests/ only; never by unconfined_b200/.  The
library is compiled with the flags of oracle/Makefile's liboracle.so and keeps its own
libm-jitter state, so noise_envelope() here perturbs this library.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .oracle import _dp, _ip

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRCS = ("oracle_dz_capi.cpp", "oracle_dz.hpp", "oracle_core.hpp", "oracle_math.hpp")
_CXXFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
             "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter"]


def _cxx():
    return "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"


def build(force=False):
    """Compile liboracle_dz.so next to liboracle.so if missing or older than its sources
    (into a temporary directory if the tree is not writable); returns its path."""
    srcs = [os.path.join(_HERE, f) for f in _SRCS]
    so = os.path.join(_HERE, "liboracle_dz.so")
    if not force and os.path.exists(so) and all(os.path.getmtime(s) <= os.path.getmtime(so) for s in srcs):
        return so
    if not os.access(_HERE, os.W_OK):
        so = os.path.join(tempfile.mkdtemp(prefix="oracle_dz_"), "liboracle_dz.so")
    subprocess.run([_cxx()] + _CXXFLAGS + ["-shared", "-o", so, srcs[0], "-lm"], check=True, capture_output=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def eval_points_dz(prm, tD, sv, rD, zD, ts_scale=None, nthreads=0, long_double=False):
    """One (gz, dgz, flag) per point; prm is an oracle.Params."""
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zD = np.ascontiguousarray(zD, np.float64)
    sv = np.ascontiguousarray(sv, np.int32)
    n = len(tD)
    gz = np.empty(n); dgz = np.empty(n); fl = np.zeros(n, np.int32)
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(ts_scale, np.float64)
        sc = _dp(scv)
    fn = lib().orc_eval_points_dz_ld if long_double else lib().orc_eval_points_dz
    rc = fn(C.byref(prm.s), C.c_int64(n), _dp(tD), _ip(sv), _dp(rD), _dp(zD), sc, int(nthreads), _dp(gz),
            _dp(dgz), _ip(fl))
    assert rc == 0, "a zD is not in [0, 1]"
    return gz, dgz, fl


def soln_dz(prm, a, rD, tD, zD, lay=0, long_double=False):
    """d/dz of the integrand at one abscissa a (counterpart of oracle.soln): shape (np,).
    lay = 1..3 evaluates that layer's formula at zD; lay = 0 takes the geometric layer."""
    out = np.empty(prm.np_, np.complex128)
    fn = lib().orc_soln_dz_ld if long_double else lib().orc_soln_dz
    fn(C.byref(prm.s), C.c_double(a), C.c_double(rD), C.c_double(tD), C.c_double(zD), C.c_int(int(lay)),
       _dp(out.view(np.float64)))
    return out


def soln_value(prm, a, rD, tD, zD, lay, long_double=False):
    """The point integrand at (zD, layer lay), one abscissa a, in double or long double: shape (np,)."""
    out = np.empty(prm.np_, np.complex128)
    fn = lib().orc_soln_value_ld if long_double else lib().orc_soln_value
    fn(C.byref(prm.s), C.c_double(a), C.c_double(rD), C.c_double(tD), C.c_double(zD), C.c_int(int(lay)),
       _dp(out.view(np.float64)))
    return out


def set_jitter(ulps, seed=0):
    """Perturb every libm result of this library by up to `ulps` units in the last place (0 = off)."""
    lib().orcd_set_jitter(C.c_double(ulps), C.c_ulonglong(seed))


def noise_envelope(fn, nsamples=4, ulps=2.0):
    """oracle.noise_envelope for functions of this library: (gz, dgz, spread_gz, spread_dgz)."""
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

"""TEST INFRASTRUCTURE ONLY -- ctypes binding of the screen oracle (oracle/liboracle_screens.so,
built from oracle_screens_capi.cpp + oracle_screens.hpp on top of oracle_core.hpp).

The CPU restatement of unc_eval_screens' definition (include/unconfined_b200.h): the point
algorithm of oracle.eval_points with the integrand replaced by its mean over a screen
[zbot, ztop].  Imported by tests/ only; never by unconfined_b200/.  The library is compiled
with the flags of oracle/Makefile's liboracle.so and keeps its own libm-jitter state, so
noise_envelope() here perturbs this library (oracle.noise_envelope perturbs liboracle.so).
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .oracle import _dp, _ip

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_SRCS = ("oracle_screens_capi.cpp", "oracle_screens.hpp", "oracle_core.hpp", "oracle_math.hpp")
_CXXFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
             "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter"]


def _cxx():
    return "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"


def build(force=False):
    """Compile liboracle_screens.so next to liboracle.so if missing or older than its sources
    (into a temporary directory if the tree is not writable); returns its path."""
    srcs = [os.path.join(_HERE, f) for f in _SRCS]
    so = os.path.join(_HERE, "liboracle_screens.so")
    if not force and os.path.exists(so) and all(os.path.getmtime(s) <= os.path.getmtime(so) for s in srcs):
        return so
    if not os.access(_HERE, os.W_OK):
        so = os.path.join(tempfile.mkdtemp(prefix="oracle_screens_"), "liboracle_screens.so")
    subprocess.run([_cxx()] + _CXXFLAGS + ["-shared", "-o", so, srcs[0], "-lm"], check=True, capture_output=True)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def eval_screens(prm, tD, sv, rD, zbot, ztop, ts_scale=None, nthreads=0, long_double=False):
    """One (s, ds, flag) per screen [zbot, ztop]; prm is an oracle.Params."""
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zbot = np.ascontiguousarray(zbot, np.float64); ztop = np.ascontiguousarray(ztop, np.float64)
    sv = np.ascontiguousarray(sv, np.int32)
    n = len(tD)
    s = np.empty(n); ds = np.empty(n); fl = np.zeros(n, np.int32)
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(ts_scale, np.float64)
        sc = _dp(scv)
    fn = lib().orc_eval_screens_ld if long_double else lib().orc_eval_screens
    rc = fn(C.byref(prm.s), C.c_int64(n), _dp(tD), _ip(sv), _dp(rD), _dp(zbot), _dp(ztop), sc,
            int(nthreads), _dp(s), _dp(ds), _ip(fl))
    assert rc == 0, "a screen is not a non-empty interval in [0, 1]"
    return s, ds, fl


def soln_screen(prm, a, rD, tD, zbot, ztop, long_double=False):
    """The screen-averaged integrand at one abscissa a (screen counterpart of oracle.soln): shape (np,)."""
    out = np.empty(prm.np_, np.complex128)
    fn = lib().orc_soln_screen_ld if long_double else lib().orc_soln_screen
    fn(C.byref(prm.s), C.c_double(a), C.c_double(rD), C.c_double(tD), C.c_double(zbot), C.c_double(ztop),
       _dp(out.view(np.float64)))
    return out


def set_jitter(ulps, seed=0):
    """Perturb every libm result of this library by up to `ulps` units in the last place (0 = off)."""
    lib().orcs_set_jitter(C.c_double(ulps), C.c_ulonglong(seed))


def noise_envelope(fn, nsamples=4, ulps=2.0):
    """oracle.noise_envelope for functions of this library: (s, ds, spread_s, spread_ds)."""
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

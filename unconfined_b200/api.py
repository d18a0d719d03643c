"""ctypes binding of include/unconfined_b200.h.

Mirrors the reference-facing boundary: one call evaluates driver.f90:100-231 for a
whole (t,r,z) grid (``eval_grid``) or for a flattened list of points
(``eval_points``).  The ``*_device`` variants take torch CUDA tensors (device memory,
current stream) -- PyTorch is plumbing only.  No CPU fallback exists.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# UNC_B200_LIB: measurement tooling only (tools/variants.py times experimental builds of the same ABI)
_SO = os.environ.get("UNC_B200_LIB") or os.path.join(_HERE, "libunconfined_b200.so")
_LIB = None


class UncError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"unconfined_b200 error {code}: {msg}")
        self.code = code


class UncParams(C.Structure):
    """struct unc_params (include/unconfined_b200.h)."""
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


def lib():
    """Load the CUDA library; fails loudly if it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(_SO):
            raise UncError(-3, f"{_SO} is missing: run __graft_entry__.build() (nvcc, sm_100a); "
                               "there is no CPU fallback")
        _LIB = C.CDLL(_SO)
        _LIB.unc_last_error.restype = C.c_char_p
        _LIB.unc_version.restype = C.c_char_p
    return _LIB


def last_error():
    return lib().unc_last_error().decode()


def _ck(rc):
    if rc != 0:
        raise UncError(rc, last_error())


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


class Params:
    """Owns the small host arrays an UncParams points to."""

    def __init__(self, d):
        self.d = dict(d)
        self._tp = np.ascontiguousarray(d.get("time_par", [0.0, 1.0]), dtype=np.float64)
        self._j0 = np.ascontiguousarray(d["j0z"], dtype=np.float64)
        self._mg = np.ascontiguousarray(d.get("moench_gamma", []), dtype=np.float64)
        s = UncParams()
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

    @property
    def n_abscissae(self):
        return (2 ** self.d["ts_k"] - 1) + self.d["gl_nacc"] * (self.d["gl_ord"] - 2)


def eval_grid(prm, tD, sv, rD, zD, zLay, ts_scale=None, ngpu=1, want_flags=False):
    """unc_eval_grid_ex on host arrays.  Returns s, ds with shape (nt, nr, nz)."""
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zD = np.ascontiguousarray(zD, np.float64)
    sv = np.ascontiguousarray(sv, np.int32); zLay = np.ascontiguousarray(zLay, np.int32)
    nt, nr, nz = len(tD), len(rD), len(zD)
    s = np.empty((nt, nr, nz)); ds = np.empty((nt, nr, nz))
    fl = np.zeros((nt, nr, nz), np.int32) if want_flags else None
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(np.broadcast_to(ts_scale, (nt, nr)), np.float64)
        sc = _dp(scv)
    _ck(lib().unc_eval_grid_ex(C.byref(prm.s), nt, _dp(tD), _ip(sv), nr, _dp(rD), nz, _dp(zD),
                               _ip(zLay), sc, int(ngpu), _dp(s), _dp(ds),
                               _ip(fl) if want_flags else None))
    return (s, ds, fl) if want_flags else (s, ds)


def eval_points(prm, tD, sv, rD, zD, zLay, ts_scale=None, ngpu=1, want_flags=False, out=None):
    """unc_eval_points_ex on host arrays (n independent (r,z,t) points)."""
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zD = np.ascontiguousarray(zD, np.float64)
    sv = np.ascontiguousarray(sv, np.int32); zLay = np.ascontiguousarray(zLay, np.int32)
    n = len(tD)
    if out is None:
        s = np.empty(n); ds = np.empty(n)
    else:
        s, ds = out
    fl = np.zeros(n, np.int32) if want_flags else None
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(ts_scale, np.float64)
        sc = _dp(scv)
    _ck(lib().unc_eval_points_ex(C.byref(prm.s), C.c_int64(n), _dp(tD), _ip(sv), _dp(rD), _dp(zD),
                                 _ip(zLay), sc, int(ngpu), _dp(s), _dp(ds),
                                 _ip(fl) if want_flags else None))
    return (s, ds, fl) if want_flags else (s, ds)


def eval_screens(prm, tD, sv, rD, zbot, ztop, ts_scale=None, ngpu=1, want_flags=False):
    """unc_eval_screens on host arrays: exact drawdown averaged over n screens [zbot, ztop]
    (dimensionless, 0 <= zbot < ztop <= 1); one inversion per screen."""
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zbot = np.ascontiguousarray(zbot, np.float64); ztop = np.ascontiguousarray(ztop, np.float64)
    sv = np.ascontiguousarray(sv, np.int32)
    n = len(tD)
    s = np.empty(n); ds = np.empty(n)
    fl = np.zeros(n, np.int32) if want_flags else None
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(ts_scale, np.float64)
        sc = _dp(scv)
    _ck(lib().unc_eval_screens(C.byref(prm.s), C.c_int64(n), _dp(tD), _ip(sv), _dp(rD), _dp(zbot),
                               _dp(ztop), sc, int(ngpu), _dp(s), _dp(ds),
                               _ip(fl) if want_flags else None))
    return (s, ds, fl) if want_flags else (s, ds)


def eval_screens_device(prm, tD, sv, rD, zbot, ztop, s, ds, ts_scale=None, flags=None):
    """unc_eval_screens_device: torch CUDA tensors on the current device (float64 / int32);
    enqueued on torch's current stream, no sync."""
    n = tD.numel()
    _ck(lib().unc_eval_screens_device(C.byref(prm.s), C.c_int64(n), _tp(tD, C.c_double),
                                      _tp(sv, C.c_int32), _tp(rD, C.c_double), _tp(zbot, C.c_double),
                                      _tp(ztop, C.c_double), _tp(ts_scale, C.c_double),
                                      _tp(s, C.c_double), _tp(ds, C.c_double),
                                      _tp(flags, C.c_int32), _stream_ptr()))


def eval_points_dz(prm, tD, sv, rD, zD, ts_scale=None, ngpu=1, want_flags=False):
    """unc_eval_points_dz on host arrays: the vertical gradient gz = ds_D/dz_D at n points and its
    log-time derivative dgz (dimensionless, 0 <= zD <= 1, layers geometric); one inversion each."""
    tD = np.ascontiguousarray(tD, np.float64); rD = np.ascontiguousarray(rD, np.float64)
    zD = np.ascontiguousarray(zD, np.float64)
    sv = np.ascontiguousarray(sv, np.int32)
    n = len(tD)
    gz = np.empty(n); dgz = np.empty(n)
    fl = np.zeros(n, np.int32) if want_flags else None
    sc = None
    if ts_scale is not None:
        scv = np.ascontiguousarray(ts_scale, np.float64)
        sc = _dp(scv)
    _ck(lib().unc_eval_points_dz(C.byref(prm.s), C.c_int64(n), _dp(tD), _ip(sv), _dp(rD), _dp(zD), sc, int(ngpu),
                                 _dp(gz), _dp(dgz), _ip(fl) if want_flags else None))
    return (gz, dgz, fl) if want_flags else (gz, dgz)


def eval_points_dz_device(prm, tD, sv, rD, zD, gz, dgz, ts_scale=None, flags=None):
    """unc_eval_points_dz_device: torch CUDA tensors on the current device (float64 / int32);
    enqueued on torch's current stream, no sync."""
    n = tD.numel()
    _ck(lib().unc_eval_points_dz_device(C.byref(prm.s), C.c_int64(n), _tp(tD, C.c_double), _tp(sv, C.c_int32),
                                        _tp(rD, C.c_double), _tp(zD, C.c_double), _tp(ts_scale, C.c_double),
                                        _tp(gz, C.c_double), _tp(dgz, C.c_double), _tp(flags, C.c_int32),
                                        _stream_ptr()))


def _tp(t, typ):
    return C.cast(C.c_void_p(t.data_ptr() if t is not None else 0), C.POINTER(typ))


def _stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def eval_points_device(prm, tD, sv, rD, zD, zLay, s, ds, ts_scale=None, flags=None):
    """unc_eval_points_device: all arguments are torch CUDA tensors on the current device
    (float64 / int32); the kernel is enqueued on torch's current stream, no sync."""
    n = tD.numel()
    _ck(lib().unc_eval_points_device(C.byref(prm.s), C.c_int64(n), _tp(tD, C.c_double),
                                     _tp(sv, C.c_int32), _tp(rD, C.c_double), _tp(zD, C.c_double),
                                     _tp(zLay, C.c_int32), _tp(ts_scale, C.c_double),
                                     _tp(s, C.c_double), _tp(ds, C.c_double),
                                     _tp(flags, C.c_int32), _stream_ptr()))


def eval_grid_device(prm, tD, sv, rD, zD, zLay, s, ds, ts_scale=None, flags=None):
    """unc_eval_grid_device: torch CUDA tensors; s, ds hold nt*nr*nz doubles (z fastest)."""
    _ck(lib().unc_eval_grid_device(C.byref(prm.s), tD.numel(), _tp(tD, C.c_double),
                                   _tp(sv, C.c_int32), rD.numel(), _tp(rD, C.c_double),
                                   zD.numel(), _tp(zD, C.c_double), _tp(zLay, C.c_int32),
                                   _tp(ts_scale, C.c_double), _tp(s, C.c_double),
                                   _tp(ds, C.c_double), _tp(flags, C.c_int32), _stream_ptr()))


def j0_zeros(n):
    out = np.empty(n)
    _ck(lib().unc_j0_zeros(int(n), _dp(out)))
    return out


def split_index(tD, j0s):
    tD = np.ascontiguousarray(tD, np.float64)
    sv = np.empty(len(tD), np.int32)
    _ck(lib().unc_split_index(len(tD), _dp(tD), int(j0s[0]), int(j0s[1]), _ip(sv)))
    return sv


def zlay(zD, lD, dD):
    zD = np.ascontiguousarray(zD, np.float64)
    out = np.empty(len(zD), np.int32)
    _ck(lib().unc_zlay(len(zD), _dp(zD), C.c_double(lD), C.c_double(dD), _ip(out)))
    return out


def device_count():
    n = C.c_int32(0)
    _ck(lib().unc_device_count(C.byref(n)))
    return n.value


def set_device(dev):
    _ck(lib().unc_set_device(int(dev)))


def device_info():
    n = C.c_int32(0); f = C.c_double(0)
    _ck(lib().unc_device_info(C.byref(n), C.byref(f)))
    return n.value, f.value


def measure_fp64_peak():
    f = C.c_double(0)
    _ck(lib().unc_measure_fp64_peak(C.byref(f)))
    return f.value


def kernel_launch_count():
    n = C.c_int64(0)
    _ck(lib().unc_kernel_launch_count(C.byref(n)))
    return n.value


def shutdown():
    _ck(lib().unc_shutdown())


def set_carry(on):
    """unc_set_carry: reference-compatible grid calls inherit stale infint (default on)."""
    _ck(lib().unc_set_carry(1 if on else 0))


_KERNELS = {None: 0, "auto": 0, "point": 1, "grid": 2, "grid2": 3, "grid8": 4}


def force_kernel(which=None):
    """Test hook (unc_debug_force_kernel): None/'auto', 'point', 'grid', 'grid2', 'grid8'."""
    _ck(lib().unc_debug_force_kernel(_KERNELS[which]))


def debug_cbesk01(z):
    """Test hook (unc_debug_cbesk01): K0(z), K1(z) by the device routine for an array of complex z."""
    z = np.ascontiguousarray(z, np.complex128)
    out = np.empty((len(z), 2), np.complex128)
    _ck(lib().unc_debug_cbesk01(len(z), _dp(z.view(np.float64)), _dp(out.view(np.float64))))
    return out[:, 0], out[:, 1]

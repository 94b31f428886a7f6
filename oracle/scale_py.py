"""ctypes wrapper over the body-scale builds (oracle/scale.mk).  TEST INFRASTRUCTURE ONLY.

`ScaledOracle`: the CPU oracle with the reference's `useScale` switch on (oracle/scale_oracle.cpp), variants "default"
(portable fdlibm sin/cos, no FMA contraction: bit-compatible with the strict CUDA build) and "glibc".
`scaled_ref(variant)`: oracle_py-style `RefPath` over _ref/libref_path_scaled_<variant>.so, the reference's own source built with
`useScale` on; `set_ref_scale` gives it its getScale spec.

A spec is the svsdf_scale form used everywhere in the tests: x, y = (c, [(a, w, phi), ...]) per axis (up to 4 terms).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import ref_py

_HERE = os.path.dirname(os.path.abspath(__file__))
_VARIANTS = {"default": os.path.join(_HERE, "_build", "libsvsdf_scale_oracle.so"),
             "glibc": os.path.join(_HERE, "_build", "libsvsdf_scale_oracle_glibc.so")}
REF_VARIANTS = ("scaled_glibc", "scaled_portable")
_libs = {}
dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)


def build(force: bool = False) -> None:
    srcs = [os.path.join(_HERE, f) for f in ("scale_oracle.cpp", "svsdf_oracle.hpp", "minco_oracle.hpp", "shapes.hpp", "portable_sincos.hpp")]
    stale = any((not os.path.exists(so)) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs) for so in _VARIANTS.values())
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-s", "-f", "scale.mk", "scale"])


def build_ref() -> None:
    """make -C oracle -f scale.mk ref_scaled (needs /root/reference)."""
    subprocess.check_call(["make", "-C", _HERE, "-s", "-f", "scale.mk", "ref_scaled"], stdout=subprocess.DEVNULL)


def ref_available() -> bool:
    return all(ref_py.available(v) for v in REF_VARIANTS)


def spec_arrays(x=None, y=None):
    """(n[2] int32, c[2], a[2][4], w[2][4], phi[2][4]) of a spec; a missing axis is the constant 1."""
    n, c = np.zeros(2, np.int32), np.ones(2)
    a, w, phi = np.zeros((2, 4)), np.zeros((2, 4)), np.zeros((2, 4))
    for ax, spec in enumerate((x, y)):
        if spec is None:
            continue
        c[ax] = spec[0]
        n[ax] = len(spec[1])
        for k, (ak, wk, pk) in enumerate(spec[1]):
            a[ax, k], w[ax, k], phi[ax, k] = ak, wk, pk
    return n, c, a, w, phi


def _p(a):
    return a.ctypes.data_as(dp) if a is not None else None


def lib(variant: str = "default"):
    if variant not in _libs:
        build()
        L = C.CDLL(_VARIANTS[variant])
        L.sor_create.restype = C.c_void_p
        L.sor_create.argtypes = [C.c_char_p, dp, dp, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_int]
        L.sor_destroy.argtypes = [C.c_void_p]
        L.sor_set_threads.argtypes = [C.c_void_p, C.c_int]
        L.sor_set_scale.argtypes = [C.c_void_p, ip, dp, dp, dp, dp, C.c_int]
        L.sor_set_points.argtypes = [C.c_void_p, dp, C.c_int64, C.c_int]
        L.sor_set_traj.argtypes = [C.c_void_p, C.c_int, dp, dp]
        L.sor_query.argtypes = [C.c_void_p, C.c_int64, dp, dp, dp, dp, ip]
        L.sor_cost_grad.restype = C.c_int64
        L.sor_cost_grad.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, dp, dp]
        L.sor_set_conditions.argtypes = [C.c_void_p, dp, dp, C.c_int]
        L.sor_evaluate.restype = C.c_double
        L.sor_evaluate.argtypes = [C.c_void_p, dp, dp, C.c_int]
        _libs[variant] = L
    return _libs[variant]


class ScaledOracle:
    """The oracle's SweptVolume + TrajOptimizer with a body scale; the same calls as oracle_py.Oracle for what it covers."""

    def __init__(self, shape="star", x=None, y=None, exact_yaw_grad=False, poly_params=(0.0, 0.0, 0.0), weight_p=60.0,
                 safety_hor=0.7, rho=3.8, threads=1, variant="default", mesh=None):
        self.L = lib(variant)
        pp = np.ascontiguousarray(poly_params, dtype=np.float64)
        V = F = None
        if mesh is not None:
            V = np.ascontiguousarray(mesh[0], dtype=np.float64).reshape(-1, 3)
            F = np.ascontiguousarray(mesh[1], dtype=np.int32).reshape(-1, 3)
        self.h = self.L.sor_create((shape or "").encode(), _p(pp), _p(V), 0 if V is None else V.shape[0],
                                   None if F is None else F.ctypes.data_as(C.c_void_p), 0 if F is None else F.shape[0],
                                   weight_p, safety_hor, rho, threads)
        self.set_scale(x, y, exact_yaw_grad)

    def __del__(self):
        try:
            if self.h:
                self.L.sor_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_scale(self, x=None, y=None, exact_yaw_grad=False):
        n, c, a, w, phi = spec_arrays(x, y)
        self.L.sor_set_scale(self.h, n.ctypes.data_as(ip), _p(c), _p(a), _p(w), _p(phi), 1 if exact_yaw_grad else 0)

    def set_threads(self, n):
        self.L.sor_set_threads(self.h, int(n))

    def set_points(self, pts):
        pts = np.ascontiguousarray(pts, dtype=np.float64)
        self.L.sor_set_points(self.h, _p(pts), pts.shape[0], pts.shape[1])

    def set_traj(self, T, coeffs_colmajor):
        T = np.ascontiguousarray(T, dtype=np.float64)
        c = np.ascontiguousarray(coeffs_colmajor, dtype=np.float64).reshape(-1)
        self.L.sor_set_traj(self.h, T.shape[0], _p(T), _p(c))

    def query(self, pts):
        pts = np.ascontiguousarray(pts, dtype=np.float64).reshape(-1, 3)
        n = pts.shape[0]
        sdf, ts, g = np.empty(n), np.empty(n), np.empty((n, 3))
        rounds = np.zeros(n, dtype=np.int32)
        self.L.sor_query(self.h, n, _p(pts), _p(sdf), _p(ts), _p(g), rounds.ctypes.data_as(ip))
        return sdf, ts, g, rounds

    def cost_grad(self, T, coeffs_colmajor):
        T = np.ascontiguousarray(T, dtype=np.float64)
        c = np.ascontiguousarray(coeffs_colmajor, dtype=np.float64).reshape(-1)
        N = T.shape[0]
        cost = C.c_double(0.0)
        gT, gC = np.zeros(N), np.zeros(18 * N)
        self.L.sor_cost_grad(self.h, N, _p(T), _p(c), C.cast(C.byref(cost), dp), _p(gT), _p(gC))
        return cost.value, gT, gC

    def set_conditions(self, init_s, final_s, N):
        i_s = np.ascontiguousarray(np.asarray(init_s, dtype=np.float64).T).reshape(-1)
        f_s = np.ascontiguousarray(np.asarray(final_s, dtype=np.float64).T).reshape(-1)
        self.L.sor_set_conditions(self.h, _p(i_s), _p(f_s), N)

    def evaluate(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        g = np.empty_like(x)
        f = self.L.sor_evaluate(self.h, _p(x), _p(g), x.shape[0])
        return f, g


def scaled_ref(shape, x=None, y=None, variant="scaled_portable", **kw):
    """ref_py.RefPath over the reference built with useScale on, its getScale set to the spec."""
    L = ref_py.lib(variant)
    L.ref_set_scale.argtypes = [C.c_void_p, ip, dp, dp, dp, dp]
    ref = ref_py.RefPath(shape, variant=variant, **kw)
    n, c, a, w, phi = spec_arrays(x, y)
    L.ref_set_scale(ref.h, n.ctypes.data_as(ip), _p(c), _p(a), _p(w), _p(phi))
    return ref

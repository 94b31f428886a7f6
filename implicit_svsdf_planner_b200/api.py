"""Python binding (ctypes) over the C ABI of libsvsdf_b200.so (include/svsdf.h).

The classes mirror the reference's call surface for this path so tests read like the reference's usage:

* ``SweptVolumeManager``  — ``updateTraj``, ``getTrueSDFofSweptVolume``, ``getSDFofSweptVolume``
  (src/swept_volume/include/swept_volume/sw_manager.hpp:376-385, 844-866, 916-1018) and the shape functor
  ``getonlySDF`` / ``getonlyGrad1`` (src/utils/include/utils/Shape.hpp:266-270).
* ``TrajOptimizer`` — ``setParam`` (via the constructor), ``parallel_points``, ``costFunction`` (=
  ``costFunctionLmbmParallel``), ``addSaftyPenaOnSweptVolumeParallelTrueSDF``, ``optimize_traj``
  (src/planner_algorithm/include/planner_algorithm/back_end_optimizer.hpp:344-408, 774-869, 877-945;
  src/planner_algorithm/src/back_end_optimizer.cpp:3-97).

There is no CPU fallback: if the CUDA library is missing or no B200 is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsvsdf_b200.so")
_lib = None

dp = C.POINTER(C.c_double)


class SvsdfError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [
        ("shape", C.c_char_p),
        ("poly_params", C.c_double * 3),
        ("weight_p", C.c_double),
        ("safety_hor", C.c_double),
        ("rho", C.c_double),
        ("device", C.c_int),
        ("strict_fp", C.c_int),
        ("polygon_xy", dp),
        ("polygon_n", C.c_int),
        ("mesh_vertices", dp),
        ("mesh_nv", C.c_int),
        ("mesh_faces", C.POINTER(C.c_int32)),
        ("mesh_nf", C.c_int),
    ]


class LmbmParams(C.Structure):
    """svsdf_lmbm_params == lmbm::lmbm_parameter_t (lmbm.h:15-174)."""
    _fields_ = [("timeout", C.c_float), ("bundle_size", C.c_int), ("ini_corrections", C.c_int), ("max_corrections", C.c_int),
                ("exponent_distmeasure", C.c_int), ("max_iterations", C.c_int), ("max_evaluations", C.c_int), ("past", C.c_int),
                ("verbose", C.c_int), ("update_method", C.c_int), ("scaling_strategy", C.c_int), ("delta_past", C.c_double),
                ("f_rel_eps", C.c_double), ("f_lower_bound", C.c_double), ("terminate_param1", C.c_double), ("terminate_param2", C.c_double),
                ("distance_measure", C.c_double), ("sufficient_dec", C.c_double), ("max_stepsize", C.c_double)]


class MidConfig(C.Structure):
    """svsdf_mid_config: the yaml keys OriTraj::setParam reads (mid_end.hpp:333-359)."""
    _fields_ = [("rho_mid_end", C.c_double), ("vmax", C.c_double), ("omgmax", C.c_double), ("weight_v", C.c_double), ("weight_omg", C.c_double),
                ("weight_pr", C.c_double), ("weight_ar", C.c_double), ("smoothingEps", C.c_double), ("integralIntervs", C.c_int),
                ("vehicleMass", C.c_double), ("gravAcc", C.c_double), ("horizDrag", C.c_double), ("vertDrag", C.c_double), ("parasDrag", C.c_double),
                ("speedEps", C.c_double), ("mem_size", C.c_int), ("past", C.c_int), ("min_step", C.c_double), ("g_epsilon", C.c_double),
                ("relCostTolMidEnd", C.c_double), ("max_iterations", C.c_int), ("cancel_after", C.c_int), ("solver", C.c_int)]


class LbfgsParams(C.Structure):
    _fields_ = [
        ("mem_size", C.c_int),
        ("past", C.c_int),
        ("delta", C.c_double),
        ("g_epsilon", C.c_double),
        ("max_iterations", C.c_int),
        ("max_linesearch", C.c_int),
        ("min_step", C.c_double),
        ("max_step", C.c_double),
        ("f_dec_coeff", C.c_double),
        ("s_curv_coeff", C.c_double),
        ("cautious_factor", C.c_double),
        ("machine_prec", C.c_double),
        ("nonsmooth_restarts", C.c_int),
    ]


class ScaleSpec(C.Structure):
    """svsdf_scale: body scale S(t) = diag(s_x(t), s_y(t), 1), per axis s = c, then s = s + sin(w_k t + phi_k) a_k."""
    _fields_ = [
        ("n_terms", C.c_int * 2),
        ("c", C.c_double * 2),
        ("a", (C.c_double * 4) * 2),
        ("w", (C.c_double * 4) * 2),
        ("phi", (C.c_double * 4) * 2),
        ("exact_yaw_grad", C.c_int),
    ]


# the reference's commented getScale example (sw_manager.hpp:499-502): diag(0.8 + sin(1.5 t - 1.0) 0.6, sin(1.8 t) 0.4 + 0.8, 1)
REFERENCE_SCALE_EXAMPLE = dict(x=(0.8, [(0.6, 1.5, -1.0)]), y=(0.8, [(0.4, 1.8, 0.0)]))


def scale_spec(x=None, y=None, exact_yaw_grad=False) -> ScaleSpec:
    """ScaleSpec from per-axis (c, [(a, w, phi), ...]) tuples (up to 4 terms; None: the constant 1)."""
    s = ScaleSpec()
    for ax, spec in enumerate((x, y)):
        c, terms = (1.0, []) if spec is None else (spec[0], list(spec[1]))
        if len(terms) > 4:
            raise ValueError("at most 4 sine terms per axis")
        s.n_terms[ax] = len(terms)
        s.c[ax] = float(c)
        for k, (a, w, phi) in enumerate(terms):
            s.a[ax][k], s.w[ax][k], s.phi[ax][k] = float(a), float(w), float(phi)
    s.exact_yaw_grad = 1 if exact_yaw_grad else 0
    return s


class OptStats(C.Structure):
    _fields_ = [
        ("final_cost", C.c_double),
        ("iterations", C.c_int),
        ("evaluations", C.c_int),
        ("status", C.c_int),
        ("seconds", C.c_double),
        ("gpu_seconds", C.c_double),
    ]


PROGRESS_T = C.CFUNCTYPE(C.c_int, C.c_void_p, dp, C.c_int)
EVAL_T = C.CFUNCTYPE(C.c_double, C.c_void_p, dp, dp, C.c_int)

# every symbol include/svsdf.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = [
    "svsdf_default_config", "svsdf_create", "svsdf_destroy", "svsdf_last_error", "svsdf_shape_id", "svsdf_shape_bound_radius",
    "svsdf_set_points", "svsdf_set_points_device", "svsdf_set_traj", "svsdf_set_scale", "svsdf_query", "svsdf_cost_grad",
    "svsdf_set_boundary", "svsdf_evaluate", "svsdf_last_costs", "svsdf_get_traj", "svsdf_default_lbfgs_params",
    "svsdf_optimize", "svsdf_optimize_batch", "svsdf_cost_grad_batch", "svsdf_minco_forward", "svsdf_minco_propagate", "svsdf_forward_T", "svsdf_backward_T",
    "svsdf_shape_sdf", "svsdf_shape_grad1", "svsdf_cost_grad_device", "svsdf_kernel_launches",
    "svsdf_executed_evals", "svsdf_fp64_peak", "svsdf_device_ptr_points", "svsdf_lbfgs_minimize", "svsdf_last_kernel_ms", "svsdf_sincos", "svsdf_set_map", "svsdf_set_map_device",
    "svsdf_extract_points", "svsdf_extract_points3d", "svsdf_set_map3d", "svsdf_get_points",
    "svsdf_mid_default_config", "svsdf_mid_cost", "svsdf_mid_get_ori_traj",
    "svsdf_lmbm_default_params", "svsdf_lmbm_open", "svsdf_lmbm_close", "svsdf_lmbm_last_error", "svsdf_lmbm_minimize", "svsdf_set_lmbm_library", "svsdf_read_obj", "svsdf_free", "svsdf_mesh_fwn_host",
    "svsdf_front_init", "svsdf_front_get_kernels", "svsdf_front_cspace", "svsdf_front_check_kernel_value", "svsdf_front_expand", "svsdf_front_astar",
]


def lib():
    """Load libsvsdf_b200.so (built in-tree by ``python -m implicit_svsdf_planner_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SvsdfError(
            f"{LIB_PATH} not found: build it with `python -m implicit_svsdf_planner_b200.build` "
            "(there is no CPU fallback for the SVSDF path)"
        )
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.svsdf_default_config.argtypes = [C.POINTER(_Config)]
    L.svsdf_create.argtypes = [C.POINTER(_Config), C.POINTER(vp)]
    L.svsdf_destroy.argtypes = [vp]
    L.svsdf_last_error.restype = C.c_char_p
    L.svsdf_last_error.argtypes = [vp]
    L.svsdf_shape_id.argtypes = [C.c_char_p]
    L.svsdf_read_obj.argtypes = [C.c_char_p, C.POINTER(dp), C.POINTER(C.c_int), C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.c_int)]
    L.svsdf_free.argtypes = [vp]
    L.svsdf_front_init.argtypes = [vp, C.c_int, C.c_int, C.c_double, C.c_double]
    L.svsdf_front_get_kernels.argtypes = [vp, dp, vp, vp]
    L.svsdf_front_cspace.argtypes = [vp, vp, C.POINTER(C.c_float), C.POINTER(vp)]
    L.svsdf_front_check_kernel_value.argtypes = [vp, C.c_int64, dp, vp, vp, dp]
    L.svsdf_front_expand.argtypes = [vp, C.c_int64, vp, dp, vp, dp, vp]
    L.svsdf_front_astar.argtypes = [vp, C.c_int, dp, dp, C.c_int, dp, vp, vp, C.POINTER(C.c_int64)]
    L.svsdf_set_points.argtypes = [vp, dp, C.c_int64, C.c_int]
    L.svsdf_set_points_device.argtypes = [vp, vp, C.c_int64]
    L.svsdf_set_traj.argtypes = [vp, C.c_int, dp, dp]
    L.svsdf_set_scale.argtypes = [vp, C.POINTER(ScaleSpec)]
    L.svsdf_query.argtypes = [vp, C.c_int, dp, dp, C.c_int64, dp, dp, dp, dp, C.POINTER(C.c_int), C.c_int]
    L.svsdf_cost_grad.argtypes = [vp, C.c_int, dp, dp, dp, dp, dp]
    L.svsdf_set_boundary.argtypes = [vp, dp, dp, C.c_int]
    L.svsdf_evaluate.restype = C.c_double
    L.svsdf_evaluate.argtypes = [vp, dp, dp, C.c_int]
    L.svsdf_last_costs.argtypes = [vp, dp]
    L.svsdf_get_traj.argtypes = [vp, dp, dp]
    L.svsdf_default_lbfgs_params.argtypes = [C.POINTER(LbfgsParams)]
    L.svsdf_optimize.argtypes = [vp, dp, dp, dp, C.c_int, C.POINTER(LbfgsParams), vp, vp, dp, dp, C.POINTER(OptStats)]
    L.svsdf_lbfgs_minimize.argtypes = [EVAL_T, vp, dp, C.c_int, C.POINTER(LbfgsParams), vp, vp, C.POINTER(OptStats)]
    L.svsdf_minco_forward.argtypes = [dp, dp, C.c_int, dp, dp, dp, dp, dp, dp]
    L.svsdf_minco_propagate.argtypes = [dp, dp, C.c_int, dp, dp, dp, dp, dp, dp]
    L.svsdf_forward_T.argtypes = [C.c_int, dp, dp]
    L.svsdf_backward_T.argtypes = [C.c_int, dp, dp]
    L.svsdf_shape_sdf.argtypes = [vp, C.c_int64, dp, dp]
    L.svsdf_shape_grad1.argtypes = [vp, C.c_int64, dp, dp]
    L.svsdf_cost_grad_device.argtypes = [vp, C.c_int, dp, dp, C.c_int, C.POINTER(C.c_float), dp]
    L.svsdf_sincos.argtypes = [vp, C.c_int64, dp, dp, dp]
    L.svsdf_set_map.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double]
    L.svsdf_set_map_device.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double]
    L.svsdf_extract_points.argtypes = [vp, dp, C.c_int, C.c_double, dp, C.c_int, C.c_double, C.POINTER(C.c_int64)]
    L.svsdf_extract_points3d.argtypes = [vp, dp, C.c_int, dp, dp, C.c_int, C.c_double, C.POINTER(C.c_int64)]
    L.svsdf_set_map3d.argtypes = [vp, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, dp, C.c_double]
    L.svsdf_lmbm_default_params.argtypes = [C.POINTER(LmbmParams)]
    L.svsdf_lmbm_default_params.restype = None
    L.svsdf_lmbm_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    L.svsdf_lmbm_close.argtypes = [C.c_void_p]
    L.svsdf_lmbm_close.restype = None
    L.svsdf_lmbm_last_error.restype = C.c_char_p
    L.svsdf_lmbm_minimize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, dp, C.c_int, C.POINTER(LmbmParams), C.c_void_p, dp]
    L.svsdf_set_lmbm_library.argtypes = [vp, C.c_char_p, C.POINTER(LmbmParams)]
    L.svsdf_mid_default_config.argtypes = [C.POINTER(MidConfig)]
    L.svsdf_mid_default_config.restype = None
    L.svsdf_mid_cost.argtypes = [C.POINTER(MidConfig), C.c_int, dp, dp, dp, dp, dp, dp, dp]
    L.svsdf_mid_get_ori_traj.argtypes = [C.POINTER(MidConfig), C.c_int, dp, dp, dp, dp, dp, dp, dp, dp, dp, C.POINTER(C.c_int)]
    L.svsdf_get_points.argtypes = [vp, dp, C.c_int64, C.POINTER(C.c_int64)]
    L.svsdf_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.svsdf_kernel_launches.argtypes = [vp, C.POINTER(C.c_int64)]
    L.svsdf_executed_evals.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64)]
    L.svsdf_fp64_peak.argtypes = [vp, dp]
    L.svsdf_device_ptr_points.argtypes = [vp, C.POINTER(vp)]
    _lib = L
    return L


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(dp) if a is not None else None


def _colmajor33(m):
    return _f64(np.asarray(m, dtype=np.float64).T).reshape(-1)


def default_lbfgs_params(**kw) -> LbfgsParams:
    p = LbfgsParams()
    lib().svsdf_default_lbfgs_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def minco_forward(init_s, final_s, q, T):
    """Host MINCO_S3NU of the product. Returns b (6N x 3), energy, dE/dc (6N x 3), dE/dT (N)."""
    T = _f64(T)
    N = T.shape[0]
    qq = _f64(np.asarray(q).T).reshape(-1)
    b, gc, gt = np.empty(18 * N), np.empty(18 * N), np.empty(N)
    e = C.c_double()
    rc = lib().svsdf_minco_forward(_p(_colmajor33(init_s)), _p(_colmajor33(final_s)), N, _p(qq), _p(T), _p(b),
                                   C.cast(C.byref(e), dp), _p(gc), _p(gt))
    if rc:
        raise SvsdfError(f"svsdf_minco_forward: {rc}")
    return b.reshape(3, 6 * N).T.copy(), e.value, gc.reshape(3, 6 * N).T.copy(), gt


def minco_propagate(init_s, final_s, q, T, gdC, gdT):
    T = _f64(T)
    N = T.shape[0]
    qq = _f64(np.asarray(q).T).reshape(-1)
    gc = _f64(np.asarray(gdC).T).reshape(-1)
    gq, gT = np.empty(3 * (N - 1)), np.empty(N)
    rc = lib().svsdf_minco_propagate(_p(_colmajor33(init_s)), _p(_colmajor33(final_s)), N, _p(qq), _p(T), _p(gc),
                                     _p(_f64(gdT)), _p(gq), _p(gT))
    if rc:
        raise SvsdfError(f"svsdf_minco_propagate: {rc}")
    return gq.reshape(N - 1, 3).T.copy(), gT


def lbfgs_minimize(fun, x0, params: "LbfgsParams | None" = None):
    """Host L-BFGS of the product on a Python callable fun(x) -> (f, g).  Returns (status, x, stats)."""
    x = _f64(x0).copy()
    n = x.shape[0]

    def _cb(_inst, xp, gp, nn):
        xv = np.ctypeslib.as_array(xp, shape=(nn,))
        f, g = fun(xv.copy())
        np.ctypeslib.as_array(gp, shape=(nn,))[:] = g
        return float(f)

    cb = EVAL_T(_cb)
    st = OptStats()
    rc = lib().svsdf_lbfgs_minimize(cb, None, _p(x), n, C.byref(params) if params is not None else None, None, None,
                                    C.byref(st))
    return rc, x, dict(final_cost=st.final_cost, iterations=st.iterations, evaluations=st.evaluations, status=st.status)


def forward_T(tau):
    tau = _f64(tau)
    T = np.empty_like(tau)
    lib().svsdf_forward_T(tau.shape[0], _p(tau), _p(T))
    return T


def backward_T(T):
    T = _f64(T)
    tau = np.empty_like(T)
    lib().svsdf_backward_T(T.shape[0], _p(T), _p(tau))
    return tau


class Problem(C.Structure):
    """svsdf_problem (include/svsdf.h)."""
    _fields_ = [
        ("initS", dp), ("finalS", dp), ("opt_x", dp), ("points", dp), ("P", C.c_int64), ("stride", C.c_int),
        ("waypoints_xy", dp), ("W", C.c_int), ("half", C.c_double), ("keepout_xy", dp), ("n_keepout", C.c_int),
        ("clearance", C.c_double), ("T_out", dp), ("coeffs_out", dp),
    ]


NEXT_T = C.CFUNCTYPE(C.c_int, C.c_void_p)


def optimize_batch(ctxs, problems, N, params=None, next_index=None):
    """svsdf_optimize_batch over a pool of Contexts.  problems: list of dicts with init_s, final_s (3x3), x0 and either
    points (P x stride) or waypoints (W x 2) + half [+ keepout (K x 2), clearance].  next_index: optional callable returning
    the next problem index (< 0 or >= len(problems) stops a worker) — e.g. a counter shared by all ranks.
    Returns (rc, x [n, nvar], stats list of dicts, status [n], points [n])."""
    n = len(problems)
    nvar = N + 3 * (N - 1)
    arr = (Problem * max(n, 1))()
    keep = []
    X = np.zeros((n, nvar))
    for k, pr in enumerate(problems):
        i_s, f_s = _colmajor33(pr["init_s"]), _colmajor33(pr["final_s"])
        X[k] = _f64(pr["x0"])
        a = arr[k]
        a.initS, a.finalS, a.opt_x = _p(i_s), _p(f_s), X[k].ctypes.data_as(dp)
        keep += [i_s, f_s]
        if pr.get("points") is not None:
            pts = _f64(pr["points"])
            a.points, a.P, a.stride = _p(pts), pts.shape[0], pts.shape[1]
            keep.append(pts)
        else:
            w = _f64(pr["waypoints"]).reshape(-1, 2)
            a.points, a.waypoints_xy, a.W, a.half = None, _p(w), w.shape[0], float(pr["half"])
            keep.append(w)
            ko = pr.get("keepout")
            if ko is not None:
                ko = _f64(ko).reshape(-1, 2)
                a.keepout_xy, a.n_keepout, a.clearance = _p(ko), ko.shape[0], float(pr.get("clearance", 0.0))
                keep.append(ko)
    hs = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
    stats = (OptStats * max(n, 1))()
    status = np.zeros(n, dtype=np.int32)
    npts = np.zeros(n, dtype=np.int64)
    cb = NEXT_T(lambda _u: int(next_index())) if next_index is not None else None
    L = lib()
    L.svsdf_optimize_batch.restype = C.c_int
    rc = L.svsdf_optimize_batch(hs, len(ctxs), arr, n, int(N), C.byref(params) if params is not None else None,
                                cb if cb is not None else C.cast(None, NEXT_T), None, stats, status.ctypes.data_as(C.POINTER(C.c_int)),
                                npts.ctypes.data_as(C.POINTER(C.c_int64)))
    st = [dict(final_cost=s.final_cost, iterations=s.iterations, evaluations=s.evaluations, status=s.status, seconds=s.seconds,
               gpu_seconds=s.gpu_seconds) for s in stats[:n]]
    return rc, X, st, status, npts


def cost_grad_batch(ctxs, point_sets, T, coeffs_colmajor, N):
    """svsdf_cost_grad_batch: one cost+gradient evaluation per problem with host buffers.  point_sets: list of (P_k x stride)
    arrays (same stride); T: [n, N]; coeffs_colmajor: [n, 18 N].  Returns (rc, cost [n], gradT [n, N], gradC [n, 18 N])."""
    n = len(point_sets)
    pts = [_f64(p) for p in point_sets]
    stride = pts[0].shape[1]
    ptrs = (dp * n)(*[_p(p) for p in pts])
    P = np.array([p.shape[0] for p in pts], dtype=np.int64)
    T = _f64(T).reshape(n, N)
    co = _f64(coeffs_colmajor).reshape(n, 18 * N)
    cost, gT, gC = np.zeros(n), np.zeros((n, N)), np.zeros((n, 18 * N))
    hs = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
    rc = lib().svsdf_cost_grad_batch(hs, len(ctxs), n, int(N), ptrs, P.ctypes.data_as(C.POINTER(C.c_int64)), stride, _p(T), _p(co),
                                     _p(cost), _p(gT), _p(gC))
    return rc, cost, gT, gC


def shape_bound_radius(shape="star", poly_params=(0.0, 0.0, 0.0), polygon=None) -> float:
    """svsdf_shape_bound_radius: R with sdf(q) >= |q| - R for the configured shape functor (host-only, no GPU needed)."""
    L = lib()
    cfg = _Config()
    L.svsdf_default_config(C.byref(cfg))
    name = (shape or "").encode()
    cfg.shape = name
    cfg.poly_params = (C.c_double * 3)(*[float(v) for v in poly_params])
    poly = None
    if polygon is not None:
        poly = _f64(polygon).reshape(-1)
        cfg.polygon_xy = _p(poly)
        cfg.polygon_n = poly.size // 2
    out = C.c_double()
    rc = L.svsdf_shape_bound_radius(C.byref(cfg), C.byref(out))
    if rc != 0:
        raise SvsdfError(f"svsdf_shape_bound_radius failed with status {rc}")
    return out.value


def mesh_fwn_host(V, F, Q=None):
    """svsdf_mesh_fwn_host: (children [nn, 4] uint32, data [nn, 23, 4] float32, w [n]) of the library's own winding-number hierarchy."""
    V = _f64(V).reshape(-1, 3)
    F = np.ascontiguousarray(F, dtype=np.int32).reshape(-1, 3)
    nn = C.c_int()
    L = lib()
    i32p = C.POINTER(C.c_int32)
    rc = L.svsdf_mesh_fwn_host(_p(V), V.shape[0], F.ctypes.data_as(i32p), F.shape[0], C.byref(nn), 0, None, None, C.c_int64(0), None, None)
    if rc != 0:
        raise SvsdfError(f"svsdf_mesh_fwn_host failed with status {rc}")
    ch = np.zeros((nn.value, 4), dtype=np.uint32)
    data = np.zeros((nn.value, 23, 4), dtype=np.float32)
    Q = _f64(Q).reshape(-1, 3) if Q is not None else np.zeros((0, 3))
    w = np.zeros(Q.shape[0])
    rc = L.svsdf_mesh_fwn_host(_p(V), V.shape[0], F.ctypes.data_as(i32p), F.shape[0], C.byref(nn), nn.value, ch.ctypes.data_as(C.c_void_p),
                               data.ctypes.data_as(C.c_void_p), C.c_int64(Q.shape[0]), _p(Q), _p(w))
    if rc != 0:
        raise SvsdfError(f"svsdf_mesh_fwn_host failed with status {rc}")
    return ch, data, w


def read_obj(path: str):
    """svsdf_read_obj: (V [nv, 3] float64, F [nf, 3] int32) of a Wavefront .obj (host code only, needs no GPU)."""
    L = lib()
    v, f = dp(), C.POINTER(C.c_int32)()
    nv, nf = C.c_int(), C.c_int()
    rc = L.svsdf_read_obj(os.fsencode(path), C.byref(v), C.byref(nv), C.byref(f), C.byref(nf))
    if rc != 0:
        raise SvsdfError(f"svsdf_read_obj({path!r}) failed with status {rc}")
    try:
        V = np.ctypeslib.as_array(v, shape=(nv.value, 3)).copy()
        F = np.ctypeslib.as_array(f, shape=(nf.value, 3)).copy()
    finally:
        L.svsdf_free(C.cast(v, C.c_void_p))
        L.svsdf_free(C.cast(f, C.c_void_p))
    return V, F


class Context:
    """Owns one svsdf_ctx (one GPU, one stream)."""

    def __init__(self, shape="star", poly_params=(0.0, 0.0, 0.0), weight_p=60.0, safety_hor=0.7, rho=3.8, device=0,
                 strict_fp=True, polygon=None, mesh=None):
        L = lib()
        cfg = _Config()
        L.svsdf_default_config(C.byref(cfg))
        self._shape_b = (shape or "").encode()
        cfg.shape = self._shape_b
        cfg.poly_params = (C.c_double * 3)(*[float(v) for v in poly_params])
        cfg.weight_p, cfg.safety_hor, cfg.rho = float(weight_p), float(safety_hor), float(rho)
        cfg.device, cfg.strict_fp = int(device), int(bool(strict_fp))
        self._poly = None
        if polygon is not None:
            self._poly = _f64(polygon).reshape(-1)
            cfg.polygon_xy = _p(self._poly)
            cfg.polygon_n = self._poly.size // 2
        if mesh is not None:  # (V [nv, 3], F [nf, 3]): the triangle-mesh functor (getonlySDF_igl) replaces the registry shape
            self._mesh_v = _f64(mesh[0]).reshape(-1, 3)
            self._mesh_f = np.ascontiguousarray(mesh[1], dtype=np.int32).reshape(-1, 3)
            cfg.mesh_vertices = _p(self._mesh_v)
            cfg.mesh_nv = self._mesh_v.shape[0]
            cfg.mesh_faces = self._mesh_f.ctypes.data_as(C.POINTER(C.c_int32))
            cfg.mesh_nf = self._mesh_f.shape[0]
        h = C.c_void_p()
        rc = L.svsdf_create(C.byref(cfg), C.byref(h))
        if rc != 0 or not h:
            raise SvsdfError(f"svsdf_create failed with status {rc} (no usable sm_100 CUDA device? no CPU fallback)")
        self.h = h
        self.P = 0

    def close(self):
        if getattr(self, "h", None):
            lib().svsdf_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc != 0:
            raise SvsdfError(f"{what}: status {rc}: {lib().svsdf_last_error(self.h).decode()}")

    # ---- raw ABI wrappers ----
    def set_points(self, pts):
        pts = _f64(pts)
        if pts.ndim != 2 or pts.shape[1] < 2:
            raise ValueError("points must be P x (2|3)")
        self._ck(lib().svsdf_set_points(self.h, _p(pts), pts.shape[0], pts.shape[1]), "svsdf_set_points")
        self.P = pts.shape[0]

    def set_points_device(self, dev_ptr: int, P: int):
        self._ck(lib().svsdf_set_points_device(self.h, C.c_void_p(dev_ptr), P), "svsdf_set_points_device")
        self.P = P

    def points_device_ptr(self) -> int:
        v = C.c_void_p()
        self._ck(lib().svsdf_device_ptr_points(self.h, C.byref(v)), "svsdf_device_ptr_points")
        return v.value or 0

    def set_traj(self, T, coeffs_colmajor):
        T = _f64(T)
        c = _f64(coeffs_colmajor).reshape(-1)
        self._ck(lib().svsdf_set_traj(self.h, T.shape[0], _p(T), _p(c)), "svsdf_set_traj")

    def set_scale(self, x=None, y=None, exact_yaw_grad=False, spec: "ScaleSpec | None" = None):
        """Deformable robot: body scale S(t) = diag(s_x(t), s_y(t), 1) on this context's cost path (svsdf_set_scale).
        x, y = (c, [(a, w, phi), ...]) per axis, or a ready ScaleSpec; no arguments return to the rigid body.
        e.g. ctx.set_scale(**REFERENCE_SCALE_EXAMPLE)."""
        if spec is None and (x is not None or y is not None):
            spec = scale_spec(x, y, exact_yaw_grad)
        self._ck(lib().svsdf_set_scale(self.h, C.byref(spec) if spec is not None else None), "svsdf_set_scale")

    def query(self, T, coeffs_colmajor, pts, outer_only=False):
        T = _f64(T)
        c = _f64(coeffs_colmajor).reshape(-1)
        pts = _f64(pts).reshape(-1, 3)
        n = pts.shape[0]
        sdf, ts, g = np.empty(n), np.empty(n), np.empty((n, 3))
        rounds = np.zeros(n, dtype=np.int32)
        self._ck(lib().svsdf_query(self.h, T.shape[0], _p(T), _p(c), n, _p(pts), _p(sdf), _p(ts), _p(g),
                                   rounds.ctypes.data_as(C.POINTER(C.c_int)), int(bool(outer_only))), "svsdf_query")
        return sdf, ts, g, rounds

    def cost_grad(self, T, coeffs_colmajor, cost0=0.0, gradT0=None, gradC0=None):
        T = _f64(T)
        c = _f64(coeffs_colmajor).reshape(-1)
        N = T.shape[0]
        cost = C.c_double(cost0)
        gT = np.zeros(N) if gradT0 is None else _f64(gradT0).copy()
        gC = np.zeros(18 * N) if gradC0 is None else _f64(gradC0).reshape(-1).copy()
        self._ck(lib().svsdf_cost_grad(self.h, N, _p(T), _p(c), C.cast(C.byref(cost), dp), _p(gT), _p(gC)),
                 "svsdf_cost_grad")
        return cost.value, gT, gC

    def cost_grad_device(self, T, coeffs_colmajor, repeats=1, fetch=True):
        """Device-resident evaluation; returns (ms per evaluation, out array [cost, gradC(18N), gradT(N), n_inside])."""
        T = _f64(T)
        c = _f64(coeffs_colmajor).reshape(-1)
        N = T.shape[0]
        ms = C.c_float()
        out = np.empty(1 + 19 * N + 1) if fetch else None
        self._ck(lib().svsdf_cost_grad_device(self.h, N, _p(T), _p(c), repeats, C.byref(ms), _p(out)),
                 "svsdf_cost_grad_device")
        return ms.value, out

    def set_boundary(self, init_s, final_s, N):
        self._ck(lib().svsdf_set_boundary(self.h, _p(_colmajor33(init_s)), _p(_colmajor33(final_s)), N),
                 "svsdf_set_boundary")

    def evaluate(self, x):
        x = _f64(x)
        g = np.empty_like(x)
        f = lib().svsdf_evaluate(self.h, _p(x), _p(g), x.shape[0])
        if not np.isfinite(f):
            raise SvsdfError(f"svsdf_evaluate returned {f}: {lib().svsdf_last_error(self.h).decode()}")
        return f, g

    def last_costs(self):
        out = np.empty(3)
        lib().svsdf_last_costs(self.h, _p(out))
        return out

    def get_traj(self, N):
        T, b = np.empty(N), np.empty(18 * N)
        self._ck(lib().svsdf_get_traj(self.h, _p(T), _p(b)), "svsdf_get_traj")
        return T, b

    def optimize(self, init_s, final_s, x0, N, params: LbfgsParams | None = None, progress=None):
        x = _f64(x0).copy()
        T, b = np.empty(N), np.empty(18 * N)
        st = OptStats()
        cb = PROGRESS_T(progress) if progress is not None else None
        rc = lib().svsdf_optimize(self.h, _p(_colmajor33(init_s)), _p(_colmajor33(final_s)), _p(x), N,
                                  C.byref(params) if params is not None else None,
                                  C.cast(cb, C.c_void_p) if cb is not None else None, None, _p(T), _p(b), C.byref(st))
        stats = dict(final_cost=st.final_cost, iterations=st.iterations, evaluations=st.evaluations, status=st.status,
                     seconds=st.seconds, gpu_seconds=st.gpu_seconds)
        return rc, x, T, b, stats

    def shape_sdf(self, rel):
        rel = _f64(rel).reshape(-1, 3)
        out = np.empty(rel.shape[0])
        self._ck(lib().svsdf_shape_sdf(self.h, rel.shape[0], _p(rel), _p(out)), "svsdf_shape_sdf")
        return out

    def shape_grad1(self, rel):
        rel = _f64(rel).reshape(-1, 3)
        out = np.empty((rel.shape[0], 3))
        self._ck(lib().svsdf_shape_grad1(self.h, rel.shape[0], _p(rel), _p(out)), "svsdf_shape_grad1")
        return out

    # ---- K3: query points from the packed map (next row) ----
    def set_map(self, kernel_u8, X, Y, kernel_size, origin, res):
        k = np.ascontiguousarray(kernel_u8, dtype=np.uint8)
        self._ck(lib().svsdf_set_map(self.h, k.ctypes.data_as(C.c_void_p), X, Y, kernel_size, float(origin[0]), float(origin[1]),
                                     float(res)), "svsdf_set_map")

    def set_map_device(self, dev_ptr, X, Y, kernel_size, origin, res):
        self._ck(lib().svsdf_set_map_device(self.h, C.c_void_p(dev_ptr), X, Y, kernel_size, float(origin[0]), float(origin[1]),
                                            float(res)), "svsdf_set_map_device")

    def extract_points(self, waypoints_xy, half, keepout_xy=None, clearance=0.0):
        w = _f64(waypoints_xy).reshape(-1, 2)
        ko = _f64(keepout_xy).reshape(-1, 2) if keepout_xy is not None else None
        n = C.c_int64()
        self._ck(lib().svsdf_extract_points(self.h, _p(w), w.shape[0], float(half), _p(ko), 0 if ko is None else ko.shape[0],
                                            float(clearance), C.byref(n)), "svsdf_extract_points")
        self.P = n.value
        return n.value

    def set_map3d(self, kernel_bytes, X, Y, Z, kernel_size, origin_xyz, res):
        """The reference's 3-D packed map (generateMapKernel layout, PCSmap_manager.h:39-78)."""
        kb = np.ascontiguousarray(kernel_bytes, dtype=np.uint8)
        h = (int(kernel_size) - 1) // 2
        if kb.size != (X + 2 * h) * (Y + 2 * h) * ((Z + 2 * h + 7) // 8):
            raise ValueError("set_map3d: kernel_bytes has the wrong size for X, Y, Z, kernel_size")
        o = _f64(origin_xyz).reshape(3)
        self._ck(lib().svsdf_set_map3d(self.h, kb.ctypes.data_as(C.c_void_p), int(X), int(Y), int(Z), int(kernel_size), _p(o), float(res)),
                 "svsdf_set_map3d")

    def extract_points3d(self, waypoints_xyz, half_xyz, keepout_xy=None, clearance=0.0):
        w = _f64(waypoints_xyz).reshape(-1, 3)
        hx = _f64(half_xyz).reshape(3)
        ko = _f64(keepout_xy).reshape(-1, 2) if keepout_xy is not None else None
        n = C.c_int64()
        self._ck(lib().svsdf_extract_points3d(self.h, _p(w), w.shape[0], _p(hx), _p(ko), 0 if ko is None else ko.shape[0],
                                              float(clearance), C.byref(n)), "svsdf_extract_points3d")
        self.P = n.value
        return n.value

    def set_lmbm_library(self, path, params: "LmbmParams" = None):
        """svsdf_optimize / optimize_batch on this context run the reference's LMBM (own private instance) instead of L-BFGS; None: back."""
        self._ck(lib().svsdf_set_lmbm_library(self.h, None if path is None else str(path).encode(), C.byref(params) if params is not None else None),
                 "svsdf_set_lmbm_library")

    def get_points(self):
        n = C.c_int64()
        lib().svsdf_get_points(self.h, None, 0, C.byref(n))
        out = np.empty((n.value, 2))
        if n.value:
            self._ck(lib().svsdf_get_points(self.h, _p(out), n.value, C.byref(n)), "svsdf_get_points")
        return out

    # ---- A* front-end collision kernels (SURVEY.md 8f rank 3) ----
    def front_init(self, kernel_size, kernel_yaw_num, occupancy_resolution, front_end_safeh=0.0):
        """BasicShape::initShape on the device (Shape.hpp:386-430)."""
        self._front = (int(kernel_size), int(kernel_yaw_num))
        self._ck(lib().svsdf_front_init(self.h, int(kernel_size), int(kernel_yaw_num), float(occupancy_resolution), float(front_end_safeh)),
                 "svsdf_front_init")

    def front_kernels(self):
        """(yaw [K], bool kernels [K, ks, ks], byte kernels [K, ks, ceil(ks / 8)])."""
        ks, K = self._front
        yaw = np.empty(K)
        cells = np.zeros((K, ks, ks), dtype=np.uint8)
        byt = np.zeros((K, ks, (ks + 7) // 8), dtype=np.uint8)
        self._ck(lib().svsdf_front_get_kernels(self.h, _p(yaw), cells.ctypes.data_as(C.c_void_p), byt.ctypes.data_as(C.c_void_p)),
                 "svsdf_front_get_kernels")
        return yaw, cells.astype(bool), byt

    def front_cspace(self, X, Y, fetch=True):
        """kernelConv for every yaw kernel and cell of the map set with set_map: (free [K, X, Y] bool or None, device ms)."""
        ks, K = self._front
        W = (Y + 31) // 32
        words = np.zeros((K, X, W), dtype=np.uint32) if fetch else None
        ms = C.c_float()
        self._ck(lib().svsdf_front_cspace(self.h, words.ctypes.data_as(C.c_void_p) if fetch else None, C.byref(ms), None), "svsdf_front_cspace")
        if not fetch:
            return None, ms.value
        bits = (words[..., None] >> (31 - np.arange(32, dtype=np.uint32))) & 1
        return bits.reshape(K, X, 32 * W)[:, :, :Y].astype(bool), ms.value

    def front_check_kernel_value(self, father_yaw, ind_xy):
        """SweptVolumeManager::checkKernelValue for a batch of nodes: (ok [n] bool, child_yaw [n])."""
        fy = _f64(father_yaw).reshape(-1)
        ind = np.ascontiguousarray(ind_xy, dtype=np.int32).reshape(-1, 2)
        ok = np.zeros(fy.size, dtype=np.uint8)
        cy = np.empty(fy.size)
        self._ck(lib().svsdf_front_check_kernel_value(self.h, fy.size, _p(fy), ind.ctypes.data_as(C.c_void_p), ok.ctypes.data_as(C.c_void_p), _p(cy)),
                 "svsdf_front_check_kernel_value")
        return ok.astype(bool), cy

    def front_expand(self, node_ij, node_yaw):
        """The neighbour loop of the A* `process` step (front_end_Astar.hpp:192-240) for n nodes:
        (ok [n, 9] bool, child_yaw [n, 9], parts [n, 9])."""
        ij = np.ascontiguousarray(node_ij, dtype=np.int32).reshape(-1, 2)
        fy = _f64(node_yaw).reshape(-1)
        n = fy.size
        ok = np.zeros((n, 9), dtype=np.uint8)
        cy = np.zeros((n, 9))
        parts = np.zeros((n, 9), dtype=np.uint8)
        self._ck(lib().svsdf_front_expand(self.h, n, ij.ctypes.data_as(C.c_void_p), _p(fy), ok.ctypes.data_as(C.c_void_p), _p(cy),
                                          parts.ctypes.data_as(C.c_void_p)), "svsdf_front_expand")
        return ok.astype(bool), cy, parts

    def front_astar(self, start_xy, goal_xy, max_path=1024):
        """AstarPathSearch + getPath for n start/goal pairs in lock-step (one expand launch per iteration):
        (paths: list of [len, 3] arrays or None, expansions [n], rounds)."""
        st = _f64(start_xy).reshape(-1, 2)
        go = _f64(goal_xy).reshape(-1, 2)
        n = st.shape[0]
        path = np.zeros((n, max_path, 3))
        ln = np.zeros(n, dtype=np.int32)
        ex = np.zeros(n, dtype=np.int32)
        rounds = C.c_int64()
        self._ck(lib().svsdf_front_astar(self.h, n, _p(st), _p(go), int(max_path), _p(path), ln.ctypes.data_as(C.c_void_p),
                                         ex.ctypes.data_as(C.c_void_p), C.byref(rounds)), "svsdf_front_astar")
        return [path[q, : ln[q]].copy() if ln[q] else None for q in range(n)], ex, rounds.value

    def sincos(self, x):
        x = _f64(x).reshape(-1)
        s, c = np.empty_like(x), np.empty_like(x)
        self._ck(lib().svsdf_sincos(self.h, x.size, _p(x), _p(s), _p(c)), "svsdf_sincos")
        return s, c

    def last_kernel_ms(self):
        """Device ms of (k_pose_table, k_outer, k_compact + k_gsip, k_finalize) in the last cost_grad_device call."""
        out = (C.c_float * 4)()
        self._ck(lib().svsdf_last_kernel_ms(self.h, out), "svsdf_last_kernel_ms")
        return [float(v) for v in out]

    def kernel_launches(self) -> int:
        n = C.c_int64()
        lib().svsdf_kernel_launches(self.h, C.byref(n))
        return n.value

    def executed_evals(self, enable=True) -> int:
        n = C.c_uint64()
        self._ck(lib().svsdf_executed_evals(self.h, int(bool(enable)), C.byref(n)), "svsdf_executed_evals")
        return n.value

    def fp64_peak_tflops(self) -> float:
        v = C.c_double()
        self._ck(lib().svsdf_fp64_peak(self.h, C.cast(C.byref(v), dp)), "svsdf_fp64_peak")
        return v.value


class SweptVolumeManager:
    """Mirror of the reference's SweptVolumeManager for the SVSDF queries (sw_manager.hpp)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._T = None
        self._coeffs = None

    def updateTraj(self, T, coeffs_colmajor):  # sw_manager.hpp:376-385
        self._T, self._coeffs = _f64(T), _f64(coeffs_colmajor).reshape(-1)
        self.ctx.set_traj(self._T, self._coeffs)

    def getTrueSDFofSweptVolume(self, pos_eva):  # sw_manager.hpp:916-1018 (batched over points)
        sdf, ts, g, rounds = self.ctx.query(self._T, self._coeffs, pos_eva, outer_only=False)
        return sdf, ts, g, rounds

    def getSDFofSweptVolume(self, pos_eva):  # sw_manager.hpp:844-866 (batched)
        sdf, ts, g, _ = self.ctx.query(self._T, self._coeffs, pos_eva, outer_only=True)
        return sdf, ts, g

    def getonlySDF(self, pos_rel):  # Shape.hpp:266
        return self.ctx.shape_sdf(pos_rel)

    def getonlyGrad1(self, pos_rel):  # Shape.hpp:268
        return self.ctx.shape_grad1(pos_rel)


class TrajOptimizer:
    """Mirror of the reference's TrajOptimizer for the back-end SVSDF cost (back_end_optimizer.hpp)."""

    def __init__(self, shape="star", poly_params=(0.0, 0.0, 0.0), weight_p=60.0, safety_hor=0.7, rho=3.8, device=0,
                 strict_fp=True, polygon=None, mesh=None):
        self.ctx = Context(shape, poly_params, weight_p, safety_hor, rho, device, strict_fp, polygon, mesh)
        self.sv_manager = SweptVolumeManager(self.ctx)
        self._points = None
        self.pieceN = 0

    @property
    def parallel_points(self):
        return self._points

    @parallel_points.setter
    def parallel_points(self, pts):  # plan_manager.cpp:168-175
        self._points = _f64(pts)
        self.ctx.set_points(self._points)

    @property
    def parallel_points_num(self):
        return 0 if self._points is None else self._points.shape[0]

    def addSaftyPenaOnSweptVolumeParallelTrueSDF(self, T, coeffs_colmajor, cost=0.0, gradT=None, gradC=None):
        return self.ctx.cost_grad(T, coeffs_colmajor, cost, gradT, gradC)

    def setConditions(self, init_s, final_s, N):
        self.pieceN = N
        self.ctx.set_boundary(init_s, final_s, N)

    def costFunction(self, x):  # costFunctionLmbmParallel
        return self.ctx.evaluate(x)

    def optimize_traj(self, init_s, final_s, opt_x, N, params=None, progress=None):
        self.pieceN = N
        return self.ctx.optimize(init_s, final_s, opt_x, N, params, progress)


# ---- mid end (host only): OriTraj::costFunction / getOriTraj ----
def mid_default_config(**over) -> MidConfig:
    c = MidConfig()
    lib().svsdf_mid_default_config(C.byref(c))
    for k, v in over.items():
        setattr(c, k, v)
    return c


def _mid_args(init_s, final_s, Q, rot_list):
    i_s = np.ascontiguousarray(np.asarray(init_s, dtype=np.float64).T).reshape(-1)   # 3x3 column-major
    f_s = np.ascontiguousarray(np.asarray(final_s, dtype=np.float64).T).reshape(-1)
    Q = np.asarray(Q, dtype=np.float64).reshape(3, -1)                               # 3 x (N - 1)
    q = np.ascontiguousarray(Q.T).reshape(-1)                                        # column-major
    R = np.asarray(rot_list, dtype=np.float64).reshape(-1, 3, 3)
    r = np.ascontiguousarray(np.transpose(R, (0, 2, 1))).reshape(-1)                 # each 3x3 column-major
    return i_s, f_s, q, r, Q.shape[1] + 1


def mid_cost(init_s, final_s, Q, rot_list, x, cfg: MidConfig = None):
    """OriTraj::costFunction: (cost, gradient) at x = [tau, xi]."""
    cfg = cfg or mid_default_config()
    i_s, f_s, q, r, N = _mid_args(init_s, final_s, Q, rot_list)
    x = _f64(x).reshape(-1)
    assert x.size == N + 3 * (N - 1) and r.size == 9 * (N - 1)
    cost = C.c_double()
    g = np.zeros_like(x)
    rc = lib().svsdf_mid_cost(C.byref(cfg), N, _p(i_s), _p(f_s), _p(q), _p(r), _p(x), C.byref(cost), _p(g))
    if rc != 0:
        raise SvsdfError(f"svsdf_mid_cost failed with {rc}")
    return cost.value, g


def mid_get_ori_traj(init_s, final_s, Q, T_init, rot_list, cfg: MidConfig = None):
    """OriTraj::getOriTraj: (status, opt_x, T, coeffs [6N, 3], final_cost, iterations)."""
    cfg = cfg or mid_default_config()
    i_s, f_s, q, r, N = _mid_args(init_s, final_s, Q, rot_list)
    T0 = _f64(T_init).reshape(-1)
    assert T0.size == N
    x = np.zeros(N + 3 * (N - 1))
    T = np.zeros(N)
    co = np.zeros(18 * N)
    fc = C.c_double()
    it = C.c_int()
    rc = lib().svsdf_mid_get_ori_traj(C.byref(cfg), N, _p(i_s), _p(f_s), _p(q), _p(T0), _p(r), _p(x), _p(T), _p(co), C.byref(fc), C.byref(it))
    if rc < 0 and rc > -1000:
        raise SvsdfError(f"svsdf_mid_get_ori_traj failed with {rc}")
    return rc, x, T, co.reshape(3, 6 * N).T.copy(), fc.value, it.value


# ---- the reference's LMBM library as a plug-in ----
def lmbm_default_params(**over) -> LmbmParams:
    p = LmbmParams()
    lib().svsdf_lmbm_default_params(C.byref(p))
    for k, v in over.items():
        setattr(p, k, v)
    return p


class Lmbm:
    """One instance of the reference's lmbm.so (svsdf_lmbm_open): private_copy=True loads a private copy of the file, so that several
    instances can minimise concurrently from different threads (the library keeps its state in statics)."""

    def __init__(self, path: str, private_copy: bool = True):
        h = C.c_void_p()
        rc = lib().svsdf_lmbm_open(str(path).encode(), int(bool(private_copy)), C.byref(h))
        if rc != 0:
            raise SvsdfError(f"svsdf_lmbm_open failed ({rc}): {lib().svsdf_lmbm_last_error().decode()}")
        self.h = h

    def minimize(self, fun, x0, params: LmbmParams = None):
        """fun(x) -> (f, g).  Returns (lmbm status, x, f, evaluations)."""
        x = _f64(x0).copy()
        n_eval = [0]

        def _eval(_inst, xp, gp, n):
            xv = np.ctypeslib.as_array(xp, shape=(n,))
            f, g = fun(xv.copy())
            np.ctypeslib.as_array(gp, shape=(n,))[:] = g
            n_eval[0] += 1
            return float(f)

        cb = EVAL_T(_eval)
        fx = C.c_double()
        rc = lib().svsdf_lmbm_minimize(self.h, C.cast(cb, C.c_void_p), None, _p(x), x.size, C.byref(params) if params is not None else None, None,
                                       C.byref(fx))
        return rc, x, fx.value, n_eval[0]

    def close(self):
        if self.h:
            lib().svsdf_lmbm_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

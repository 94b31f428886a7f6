"""One plan from point cloud to optimised trajectory: the chain PlannerManager::generatePath / generateTraj drives in the reference
(src/plan_manager/src/plan_manager.cpp:96-227), on this build's entry points.

  point cloud -> occupancy grid                 PCSmapManager::rcvGlobalMapHandler      map_manager/src/PCSmap_manager.cpp:113-190
  grid -> byte-packed maps                      generateMapKernel / generateMapKernel2D  map_manager/include/map_manager/PCSmap_manager.h:39-108
  A* over (x, y, yaw) with the shape kernels    AstarPathSearcher::AstarPathSearch       -> svsdf_front_astar (GPU node tests)
  path -> waypoints, boxes -> query points      generateTraj                             plan_manager.cpp:131-175 -> svsdf_extract_points3d (GPU)
  warm start                                    OriTraj::getOriTraj                      -> svsdf_mid_get_ori_traj (host)
  SVSDF back end                                TrajOptimizer::optimize_traj_lmbm        -> svsdf_optimize (GPU cost + gradient, host solver)

Host-side glue only (numpy); every arithmetic step is behind the C ABI.  The map construction and the waypoint rule are checked against
oracle/k3_points.py by tests/test_oracle_k3.py, the chain itself by tests/test_gpu_plan.py on the reference's own star scene."""
from __future__ import annotations

import dataclasses
import math
from typing import Optional

import numpy as np

from . import api, scenes


@dataclasses.dataclass
class CloudMap:
    occ: np.ndarray            # [X, Y, Z] bool
    boundary_min: np.ndarray   # boundary_xyzmin
    boundary_max: np.ndarray   # boundary_xyzmax
    res: float


def gridmap3d_from_cloud(points_f32, res: float, sta_threshold: int = 1) -> CloudMap:
    """rcvGlobalMapHandler: boundary = min / max of the cloud (pcl::PointXYZ floats widened to double), size = ceil(extent / res)
    (Gridmap3D.cpp:25-41), a voxel is occupied when at least sta_threshold points fall into it; index = floor((p - min) / res) clamped to
    the last cell (Gridmap3D.cpp:137-174; every cloud point is inside the boundary by construction)."""
    pts = np.asarray(points_f32, dtype=np.float32).astype(np.float64).reshape(-1, 3)
    lo, hi = pts.min(axis=0), pts.max(axis=0)
    size = np.maximum(np.ceil((hi - lo) / res).astype(np.int64), 0)
    cnt = np.zeros(tuple(int(s) for s in size), dtype=np.int64)
    if cnt.size:
        idx = np.floor((pts - lo) / res).astype(np.int64)
        idx = np.minimum(np.maximum(idx, 0), size - 1)
        np.add.at(cnt, (idx[:, 0], idx[:, 1], idx[:, 2]), 1)
    return CloudMap(occ=cnt >= sta_threshold, boundary_min=lo, boundary_max=hi, res=float(res))


def pack_map_kernel3d(occ: np.ndarray, kernel_size: int) -> np.ndarray:
    """generateMapKernel (PCSmap_manager.h:39-78): [(X + 2h)][(Y + 2h)][ceil((Z + 2h) / 8)] bytes, z bits MSB first."""
    h = (kernel_size - 1) // 2
    X, Y, Z = occ.shape
    bits = np.zeros((X + 2 * h, Y + 2 * h, 8 * ((Z + 2 * h + 7) // 8)), dtype=np.uint8)
    bits[h:h + X, h:h + Y, h:h + Z] = occ
    return np.packbits(bits, axis=2)  # MSB first, as or_mask = {0x80, ..., 0x01}


def waypoints_of_path(path: np.ndarray, traj_parlength: float, res: float):
    """plan_manager.cpp:131-158: index_gap = ceil(traj_parlength / res), shrunk by 1.5 until the path has more cells than one gap; every
    index_gap-th node of the front-end path (ends excluded) becomes a waypoint.  Returns (indices, waypoints)."""
    path = np.asarray(path, dtype=np.float64)
    n = path.shape[0]
    t = float(traj_parlength)
    gap = int(math.ceil(t / res))
    while gap >= n - 1:
        t /= 1.5
        gap = int(math.ceil(t / res))
    idx = np.arange(gap, n - 1, gap)
    return idx, path[idx]


def rot_z(yaw: float) -> np.ndarray:
    c, s = math.cos(yaw), math.sin(yaw)
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


def generate_traj(ctx: "api.Context", cmap: CloudMap, start_xy, goal_xy, kernel_size: int = scenes.YAML["kernel_size"], kernel_yaw_num: int = 18,
                  front_end_safeh: float = 0.0, traj_parlength: float = 3.0, inittime: float = scenes.YAML["inittime"],
                  mid_cfg: Optional["api.MidConfig"] = None, lbfgs_params=None, max_path: int = 4096, scale: Optional[dict] = None) -> dict:
    """generatePath + generateTraj for one start / goal on the map `cmap` (the context's shape is the robot).
    scale: a deformable robot's body scale for the back end only (keyword arguments of Context.set_scale, e.g.
    api.REFERENCE_SCALE_EXAMPLE); the front and mid ends plan for the rigid body, as the reference's do.  The context is
    back to the rigid body when the call returns."""
    X, Y, Z = cmap.occ.shape
    res = cmap.res
    ctx.set_map3d(pack_map_kernel3d(cmap.occ, kernel_size), X, Y, Z, kernel_size, cmap.boundary_min, res)
    ctx.front_init(kernel_size, kernel_yaw_num, res, front_end_safeh)
    paths, expansions, rounds = ctx.front_astar(np.asarray(start_xy, dtype=np.float64).reshape(1, 2), np.asarray(goal_xy, dtype=np.float64).reshape(1, 2), max_path)
    path = paths[0]
    if path is None or len(path) < 3:
        return dict(ok=False, reason="front end found no path", expansions=int(expansions[0]))
    idx, wps = waypoints_of_path(path, traj_parlength, res)
    N = len(wps) + 1
    half = kernel_size * res / 3.0                      # bdx / 3 (plan_manager.cpp:57-59, 165)
    n_points = ctx.extract_points3d(wps, [half, half, half])  # the waypoint (x, y, yaw) is the box centre, as in the reference
    init_s, final_s = np.zeros((3, 3)), np.zeros((3, 3))
    init_s[:, 0], final_s[:, 0] = path[0], path[-1]     # plan_manager.cpp:143-147
    rots = np.stack([rot_z(p[2]) for p in wps])
    rc_mid, opt_x, T_mid, co_mid, cost_mid, it_mid = api.mid_get_ori_traj(init_s, final_s, wps.T, np.full(N, inittime), rots, mid_cfg)
    if rc_mid < 0:
        return dict(ok=False, reason=f"mid end failed ({rc_mid})", N=N, n_points=int(n_points))
    params = lbfgs_params or api.default_lbfgs_params(mem_size=16, past=3, delta=1e-6, g_epsilon=0.0, max_iterations=0, min_step=1e-32)
    if scale is not None:
        ctx.set_scale(**scale)
    try:
        f0, _ = ctx_evaluate(ctx, init_s, final_s, N, opt_x)
        rc, x, T, b, st = ctx.optimize(init_s, final_s, opt_x, N, params)  # the query points are the context's resident set (extract_points3d)
    finally:
        if scale is not None:
            ctx.set_scale()
    return dict(ok=rc >= 0, status=int(rc), N=N, n_points=int(n_points), path=path, waypoints=wps, expansions=int(expansions[0]), astar_rounds=int(rounds),
                mid=dict(status=int(rc_mid), cost=float(cost_mid), iterations=int(it_mid), T=T_mid), cost_at_warm_start=float(f0),
                final_cost=float(st["final_cost"]), iterations=int(st["iterations"]), evaluations=int(st["evaluations"]), T=T, coeffs=b, x=x,
                seconds=float(st["seconds"]))


def ctx_evaluate(ctx, init_s, final_s, N, x):
    ctx.set_boundary(init_s, final_s, N)
    return ctx.evaluate(x)

"""Trajectories and query sets at the edges of what svsdf_query / svsdf_cost_grad accept: 1 to 64 pieces, durations far
from the 2.5 s of scenes.make_scene, a total duration D just below 300 s, D on and around the layer-1 lattice, points so far
away that no layer-1 sample is below 1e9, and thousands of interior (GSIP) points.  Shared by tests/test_oracle_envelope.py
(which checks, on the CPU, that every case really reaches the edge it is named after) and tests/test_gpu_envelope.py (which
compares the CUDA path with the oracle on the same cases).

Trajectories are built the way scenes.make_scene builds them: scenes.make_trajectory, durations overridden, then
scenes.minco_dense; query points come from the same candidate machinery (occupied cell centres in the waypoint boxes, outside
a corridor around the nominal path).  The helpers that mirror the runtime (lattice, blob_layout, outer_smem_doubles,
locate_piece) restate svsdf_runtime.cpp:upload_traj, svsdf_types.h and Trajectory::locatePieceIdx in plain Python floats.
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np

from implicit_svsdf_planner_b200 import scenes

LAT_DT = 0.15          # choiceTInit layer-1 step
MAX_PIECES = 64        # svsdf_types.h kMaxPieces
MAX_DURATION = 300.0   # svsdf_types.h kMaxDuration (exclusive)
WARPS = 8              # svsdf_types.h kWarpsPerBlock


# ---------------------------------------------------------------------------------------------------------------------
# mirrors of the runtime's bookkeeping
# ---------------------------------------------------------------------------------------------------------------------
def seq_sum(T) -> float:
    """Trajectory::getTotalDuration: left-to-right IEEE sum."""
    D = 0.0
    for v in T:
        D += float(v)
    return D


def lattice(D: float) -> list:
    """upload_traj: for (t = 0; t <= D; t += 0.15) — the accumulated layer-1 times."""
    out, t = [], 0.0
    while t <= D:
        out.append(t)
        t += LAT_DT
    return out


def lattice_values(n: int) -> list:
    """The first n accumulated lattice values, independent of D."""
    out, t = [], 0.0
    for _ in range(n):
        out.append(t)
        t += LAT_DT
    return out


def blob_doubles(N: int, K1: int) -> int:
    """svsdf_types.h blob_layout(N, K1).total."""
    npad, k1pad = (N + 1) & ~1, (K1 + 1) & ~1
    total = 4 + npad + 18 * N + k1pad + 4 * k1pad
    return (total + 1) & ~1


def outer_smem_doubles(N: int, K1: int) -> int:
    """svsdf_types.h outer_smem_doubles: blob + 8 warps x (19N + 1) accumulators + 8 warps x 128 work area."""
    return blob_doubles(N, K1) + WARPS * (19 * N + 1) + WARPS * 128


def locate_piece(T, t: float):
    """Trajectory<5>::locatePieceIdx: (piece, local time, wrapped) where `wrapped` is the idx == N case (the sample is
    still greater than T[N-1] after subtracting T[0..N-2])."""
    N = len(T)
    idx = 0
    while idx < N:
        if not (t > T[idx]):
            break
        t -= float(T[idx])
        idx += 1
    if idx == N:
        return N - 1, t + float(T[N - 1]), True
    return idx, t, False


# ---------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Case:
    name: str
    init_s: np.ndarray
    final_s: np.ndarray
    q: np.ndarray
    T: np.ndarray
    coeffs: np.ndarray   # MINCO b, 6N x 3
    points: np.ndarray   # P x 3

    @property
    def N(self) -> int:
        return int(self.T.shape[0])

    @property
    def P(self) -> int:
        return int(self.points.shape[0])

    @property
    def D(self) -> float:
        return seq_sum(self.T)

    @property
    def K1(self) -> int:
        return len(lattice(self.D))

    def co(self) -> np.ndarray:
        return np.ascontiguousarray(self.coeffs.T).reshape(-1)

    def pts0(self) -> np.ndarray:
        return np.c_[self.points[:, :2], np.zeros(self.P)]

    def with_points(self, name, points) -> "Case":
        return dataclasses.replace(self, name=name, points=np.asarray(points, dtype=np.float64))


def scene_points(init_s, final_s, q, T, b, P, clearance=2.75, seed=scenes.SEED_MAP):
    """make_scene's query set for an arbitrary trajectory: P cell centres of a seeded occupancy grid inside the waypoint
    boxes, outside a corridor of half-width `clearance` around the nominal path."""
    half = scenes.YAML["kernel_size"] * scenes.YAML["occupancy_resolution"] / 3.0
    wps = np.concatenate([init_s[:2, :1], q[:2], final_s[:2, :1]], axis=1).T
    lo, hi = wps.min(axis=0) - half, wps.max(axis=0) + half
    D = seq_sum(T)
    path = scenes.eval_traj_xy(b, T, np.linspace(0.0, D, max(4001, 40 * T.shape[0] + 1)))[:, :2]

    def grid(res):
        nx, ny = int(math.ceil((hi[0] - lo[0]) / res)), int(math.ceil((hi[1] - lo[1]) / res))
        xs, ys = lo[0] + (np.arange(nx) + 0.5) * res, lo[1] + (np.arange(ny) + 0.5) * res
        return scenes._candidates(xs, ys, wps, half, path, clearance)

    res = 0.25
    cand = grid(res)
    if cand.shape[0] < 3.0 * P:
        res = 0.25 * math.sqrt(cand.shape[0] / (3.3 * P))
        cand = grid(res)
    rng = scenes._rng(seed)
    sel = np.sort(rng.choice(cand.shape[0], size=P, replace=False))
    pts = np.zeros((P, 3))
    pts[:, :2] = cand[sel]
    pts[:, 2] = rng.integers(0, 3, size=P) * scenes.YAML["occupancy_resolution"]
    return pts


def build(name, N, T, start, goal, P, clearance=2.75, q=None, seed=scenes.SEED_TRAJ):
    init_s, final_s, q0, _ = scenes.make_trajectory("star", N, seed, start, goal)
    q = q0 if q is None else q
    T = np.asarray(T, dtype=np.float64)
    b = scenes.minco_dense(init_s, final_s, q, T)
    return Case(name, init_s, final_s, q, T, b, scene_points(init_s, final_s, q, T, b, P, clearance))


def max_blob(P=20_000) -> Case:
    """64 pieces of 299.99 / 64 s: D just below 300 s, K1 = 2000, ~176 KB of k_outer shared memory per CTA."""
    return build("max_blob", MAX_PIECES, np.full(MAX_PIECES, 299.99 / MAX_PIECES), (0.0, 0.0), (240.0, 120.0), P)


def single_piece() -> Case:
    """N = 1, D = 3.05 s: K1 = 21 (< 32, the nearest-pose window is partial)."""
    return build("single_piece", 1, [3.05], (2.0, 3.0), (5.0, 4.0), 400, clearance=2.2)


TINY_D = (0.1, 4.6, 4.81)  # not 4.8: lat[32] = 4.800000000000001 > 4.8, so D = 4.8 still has K1 = 32


def tiny(D: float) -> Case:
    """N = 2, two equal pieces of D / 2: K1 = 1 (D = 0.1), 31 (4.6) and 33 (4.81), either side of the 32-sample window."""
    dist = max(0.1, D)
    return build(f"tiny_{D}", 2, [D / 2, D / 2], (1.0, 1.0), (1.0 + 0.8 * dist, 1.0 + 0.6 * dist), 300, clearance=1.8)


SHORT = 0.004


def sub_step() -> Case:
    """N = 16 with every odd piece (1, 3, ..., 13) 0.004 s long — shorter than the 0.01 s descent step, so one step crosses
    several pieces — and the other pieces 2.5 s.  Each short piece ends 3 mm from where it starts, along the path (about the
    speed the long pieces give it), so the MINCO coefficients stay moderate."""
    N = 16
    start, goal = np.array([3.0, 4.0]), np.array([40.0, 30.0])
    init_s, final_s, q, _ = scenes.make_trajectory("star", N, scenes.SEED_TRAJ, start, goal)
    T = np.full(N, 2.5)
    short = [i for i in range(1, N - 1, 2)]
    T[short] = SHORT
    u = (goal - start) / np.linalg.norm(goal - start)
    for i in short:
        q[:2, i] = q[:2, i - 1] + 0.003 * u
        q[2, i] = q[2, i - 1] + 0.002
    b = scenes.minco_dense(init_s, final_s, q, T)
    pts = scene_points(init_s, final_s, q, T, b, 900, clearance=2.0)
    # points on and beside the path where each short piece starts: their outer t* (and the ring samples' t*) settle next to
    # the short piece
    starts = np.concatenate([[0.0], np.cumsum(T)[:-1]])
    extra = []
    for i in short:
        x = scenes.eval_traj_xy(b, T, np.array([starts[i]]))[0]
        for d in (0.0, 0.05, -0.05, 0.2, -0.2, 0.5, -0.5, 1.0, -1.0):
            extra.append([x[0] - d * u[1], x[1] + d * u[0], 0.0])
    return Case("sub_step", init_s, final_s, q, T, b, np.r_[pts, np.asarray(extra)])


def on_boundaries() -> Case:
    """Piece boundaries exactly on lattice samples: the sequential subtraction of T[0..k-1] from lat[20 (k + 1)] leaves
    exactly T[k], for k = 0..4 (3 s pieces), so locatePieceIdx meets `t == dur` and the guess search its `tl == 0` case."""
    N = 6
    lat = lattice_values(20 * N + 1)
    T = []
    for k in range(N - 1):
        t = lat[20 * (k + 1)]
        for v in T:
            t -= v
        T.append(t)
    T.append(2.7)
    return build("on_boundaries", N, T, (2.0, 2.0), (14.0, 12.0), 700, clearance=2.2)


def d_lattice(where: str) -> Case:
    """Eight pieces of irregular length; T[7] nudged by ulps until the sequential sum D equals lattice value lat[m] exactly
    ("on"), or is one ulp below ("below") or above ("above") it.  On this trajectory t = D = lat[m] rounds past the last
    piece in locatePieceIdx (idx == N) — the wrap-around case."""
    N, m = 8, 133
    T = [2.5 + 0.0137 * ((5 * i) % 7) - 0.02 * (i % 3) for i in range(N)]
    target = lattice_values(m + 1)[m]
    T[-1] = target - seq_sum(T[:-1])
    for _ in range(64):
        D = seq_sum(T)
        if D == target:
            break
        T[-1] = float(np.nextafter(T[-1], np.inf if D < target else -np.inf))
    assert seq_sum(T) == target
    if where != "on":
        goal = np.nextafter(target, -np.inf if where == "below" else np.inf)
        for _ in range(64):
            D = seq_sum(T)
            if D == goal:
                break
            T[-1] = float(np.nextafter(T[-1], np.inf if D < goal else -np.inf))
        assert seq_sum(T) == goal
    start, goal = (np.asarray(v) for v in scenes.START_GOAL["star"])
    init_s, final_s, q, _ = scenes.make_trajectory("star", N, scenes.SEED_TRAJ, start, goal)
    # the robot still moves at t = D (3 m/s along the path), so the end of the trajectory is not flat: a point whose
    # layer-1 minimum is the last sample (t = D) ends elsewhere when that sample is missing
    final_s[:2, 1] = 3.0 * (goal - start) / np.linalg.norm(goal - start)
    T = np.asarray(T, dtype=np.float64)
    b = scenes.minco_dense(init_s, final_s, q, T)
    pts = scene_points(init_s, final_s, q, T, b, 1500)
    D = seq_sum(T)
    extra = []
    for back in (0.0, 0.02, 0.04, 0.06):
        x0, x1 = scenes.eval_traj_xy(b, T, np.array([D - back - 1e-3, D - back]))[:, :2]
        n = np.array([x0[1] - x1[1], x1[0] - x0[0]]) / np.linalg.norm(x1 - x0)
        for d in (-3.4, -3.0, 3.0, 3.4):
            extra.append([x1[0] + d * n[0], x1[1] + d * n[1], 0.0])
    return Case(f"d_{where}", init_s, final_s, q, T, b, np.r_[pts, np.asarray(extra)])


# ---------------------------------------------------------------------------------------------------------------------
# query sets on a config-1 trajectory
# ---------------------------------------------------------------------------------------------------------------------
def config1(P=2000) -> Case:
    sc = scenes.make_scene("star", 8, P)
    return Case("config1", sc.init_s, sc.final_s, sc.q, sc.T, sc.coeffs, sc.points)


def far_points(n=64) -> np.ndarray:
    """n points about 2e9 m from the trajectory: every layer-1 sample's SDF is >= 1e9 (the descent's degenerate F0 mode)."""
    ang = np.linspace(0.0, 2 * np.pi, n, endpoint=False)
    r = 2e9 * (1.0 + 0.01 * np.arange(n) / n)
    return np.c_[r * np.cos(ang), r * np.sin(ang), np.zeros(n)]


def interleave_far(points, far, every=7) -> tuple:
    """Insert one far point after every `every - 1` normal points; returns (points, mask of the far ones)."""
    out, mask, j = [], [], 0
    for i, p in enumerate(points):
        out.append(p)
        mask.append(False)
        if i % (every - 1) == every - 2 and j < len(far):
            out.append(far[j])
            mask.append(True)
            j += 1
    return np.asarray(out), np.asarray(mask)


def many_inside(case: Case, n=4000, seed=11) -> Case:
    """`n` trajectory poses jittered by up to 0.3 m, appended to the case's points so that P = 7 (mod 16)."""
    rng = np.random.default_rng(seed)
    D = case.D
    ts = np.sort(rng.uniform(0.0, D, n))
    xy = scenes.eval_traj_xy(case.coeffs, case.T, ts)[:, :2] + rng.uniform(-0.3, 0.3, size=(n, 2))
    pts = np.r_[case.points, np.c_[xy, np.zeros(n)]]
    drop = (pts.shape[0] - 7) % 16
    return case.with_points("many_inside", pts[: pts.shape[0] - drop])


def rest_ends(case: Case, seed=12) -> tuple:
    """The start and goal positions and 8 points within 0.3 m of each, on the side facing away from the path (the robot is
    at rest there, and t* stays at the end): returns (case with these 18 points appended, indices of the start group,
    indices of the goal group)."""
    rng = np.random.default_rng(seed)
    groups = []
    for pos, t_in in ((case.init_s[:2, 0], 0.5), (case.final_s[:2, 0], case.D - 0.5)):
        away = pos - scenes.eval_traj_xy(case.coeffs, case.T, np.array([t_in]))[0, :2]
        ang = math.atan2(away[1], away[0]) + rng.uniform(-0.6, 0.6, 8)
        rad = rng.uniform(0.05, 0.3, 8)
        groups.append(np.r_[[pos], pos + np.c_[rad * np.cos(ang), rad * np.sin(ang)]])
    P0 = case.P
    pts = np.r_[case.points, np.c_[groups[0], np.zeros(9)], np.c_[groups[1], np.zeros(9)]]
    return case.with_points("rest_ends", pts), np.arange(P0, P0 + 9), np.arange(P0 + 9, P0 + 18)


def few_inside() -> Case:
    """make_scene's 400-point narrow-corridor scene: a couple of dozen interior points (fewer than the B200's 148 SMs)."""
    sc = scenes.make_scene("star", 8, 400, clearance=2.35)
    return Case("few_inside", sc.init_s, sc.final_s, sc.q, sc.T, sc.coeffs, sc.points)

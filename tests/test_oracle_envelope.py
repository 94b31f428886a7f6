"""CPU checks that every case of tests/envelope_cases.py reaches the edge of the input envelope it is named after, so that
a later change to the scene builders cannot silently turn tests/test_gpu_envelope.py into middle-of-the-range tests.
Sizes are restated in plain Python arithmetic that mirrors upload_traj / blob_layout; per-point claims use the oracle."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import envelope_cases as ec  # noqa: E402

SMEM_LIMIT = 200 * 1024  # run_kernels refuses a k_outer shared-memory footprint above this


def test_max_blob_fills_shared_memory():
    c = ec.max_blob()
    assert c.N == ec.MAX_PIECES and 299.9 < c.D < ec.MAX_DURATION
    assert c.K1 == 2000
    smem = 8 * ec.outer_smem_doubles(c.N, c.K1)
    assert 150 * 1024 < smem <= SMEM_LIMIT, smem
    assert smem > 6 * 8 * ec.outer_smem_doubles(8, 134)  # vs config 1/2 (N = 8, D = 20 s)
    # P >= 16 x 148 SMs x 8 warps: at one CTA per SM the natural schedule is the batched one
    assert c.P >= 16 * 148 * ec.WARPS


def test_short_trajectories_have_partial_lattices():
    s = ec.single_piece()
    assert s.N == 1 and s.K1 == 21
    assert [ec.tiny(D).K1 for D in ec.TINY_D] == [1, 31, 33]
    for D in ec.TINY_D:
        c = ec.tiny(D)
        assert c.N == 2 and c.D == D


def test_sub_step_pieces_are_shorter_than_a_descent_step(oracle_mod):
    c = ec.sub_step()
    short = np.flatnonzero(c.T < 0.01)
    assert short.size >= 7 and np.all(c.T[short] == ec.SHORT)
    assert np.all(np.isfinite(c.coeffs)) and np.abs(c.coeffs).max() < 1e8
    # many points settle within one descent step of a short piece: their steps cross it
    starts = np.concatenate([[0.0], np.cumsum(c.T)[:-1]])
    orc = oracle_mod.Oracle("star", threads=oracle_mod.num_procs())
    orc.set_traj(c.T, c.co())
    _, ts, _ = orc.query_outer(c.pts0())
    near = np.zeros(c.P, dtype=bool)
    for i in short:
        near |= (ts > starts[i] - 0.01) & (ts < starts[i] + c.T[i] + 0.01)
    assert near.sum() >= 8, near.sum()


def test_piece_boundaries_sit_on_lattice_samples():
    c = ec.on_boundaries()
    lat = ec.lattice(c.D)
    for k in range(c.N - 1):
        t = lat[20 * (k + 1)]
        idx, tl, wrapped = ec.locate_piece(c.T, t)
        assert (idx, tl, wrapped) == (k, c.T[k], False)  # `!(t > dur)` at equality
        for v in c.T[:k + 1]:
            t -= v
        assert t == 0.0  # the guess search with hint k + 1 sees tl == 0


def test_duration_on_and_around_the_lattice(oracle_mod):
    on, below, above = ec.d_lattice("on"), ec.d_lattice("below"), ec.d_lattice("above")
    m = 133
    lat_m = ec.lattice_values(m + 1)[m]
    assert on.D == lat_m and below.D == np.nextafter(lat_m, -np.inf) and above.D == np.nextafter(lat_m, np.inf)
    assert on.K1 == m + 1 and below.K1 == m and above.K1 == m + 1
    # only the "on" case changes when the lattice loop's `t <= D` becomes `t < D`
    for c in (on, below, above):
        strict = sum(1 for t in ec.lattice_values(m + 2) if t < c.D)
        assert (strict != c.K1) == (c is on)
    # the trajectory does not come to rest at t = D, and some points have their layer-1 minimum at the last sample
    orc = oracle_mod.Oracle("star", threads=oracle_mod.num_procs())
    orc.set_traj(on.T, on.co())
    assert np.linalg.norm(orc.traj_vel(on.D)[:2]) > 1.0
    # the same pieces apart from T[N-1] (nudged by a few ulps)
    assert np.array_equal(on.T[:-1], below.T[:-1]) and abs(on.T[-1] - below.T[-1]) < 1e-13


def test_duration_on_the_lattice_wraps_past_the_last_piece():
    """t = D = lat[m] is still greater than T[N-1] after subtracting T[0..N-2]: locatePieceIdx reaches idx == N."""
    c = ec.d_lattice("on")
    lat = ec.lattice(c.D)
    wrapped = [t for t in lat if ec.locate_piece(c.T, t)[2]]
    assert wrapped == [c.D]
    t = c.D
    for v in c.T[:-1]:
        t -= v
    assert t > c.T[-1]


def test_far_points_are_beyond_1e9_at_every_lattice_pose(oracle_mod):
    c = ec.config1()
    far = ec.far_points()
    orc = oracle_mod.Oracle("star", threads=oracle_mod.num_procs())
    orc.set_traj(c.T, c.co())
    poses = np.array([orc.traj_pos(t) for t in ec.lattice(c.D)])
    for p in far:
        d = p[:2] - poses[:, :2]
        cy, sy = np.cos(poses[:, 2]), np.sin(poses[:, 2])
        rel = np.c_[cy * d[:, 0] + sy * d[:, 1], -sy * d[:, 0] + cy * d[:, 1], np.zeros(len(poses))]
        assert oracle_mod.shape_sdf("star", rel).min() >= 1e9
    pts, mask = ec.interleave_far(c.points, far)
    assert mask.sum() == far.shape[0] and np.array_equal(pts[~mask], c.points)
    assert np.all(np.diff(np.flatnonzero(mask)) == 7)


def test_many_inside_points_exceed_a_gsip_grid(oracle_mod):
    m = ec.many_inside(ec.config1())
    assert m.P % 16 == 7
    orc = oracle_mod.Oracle("star", threads=oracle_mod.num_procs())
    orc.set_points(m.points)
    *_, inside = orc.cost_grad(m.T, m.co())
    assert inside >= 3000, inside  # more than one pass of k_gsip's grid (148 SMs x 3 CTAs)


def test_rest_end_points_reach_both_velocity_scans(oracle_mod):
    c, g0, g1 = ec.rest_ends(ec.config1())
    orc = oracle_mod.Oracle("star", threads=oracle_mod.num_procs())
    orc.set_traj(c.T, c.co())
    _, ts, _ = orc.query_outer(c.pts0())
    _, _, _, rounds = orc.query(c.pts0())
    assert np.all(ts[g0] < 0.1) and np.all(ts[g1] > c.D - 0.1)
    assert np.all(rounds[g0] > 0) and np.all(rounds[g1] > 0)
    # the robot is at rest at those t*: k_gsip falls back to the forward / backward velocity scans
    for i in np.r_[g0, g1]:
        assert np.linalg.norm(orc.traj_vel(ts[i])) < 0.01


def test_few_inside_scene_selects_the_wide_gsip_kernel(oracle_mod):
    c = ec.few_inside()
    orc = oracle_mod.Oracle("star", threads=oracle_mod.num_procs())
    orc.set_points(c.points)
    *_, inside = orc.cost_grad(c.T, c.co())
    assert 1 <= inside <= 148


@pytest.mark.parametrize("T", [[150.0, 150.0], [299.99 / 64] * 64])
def test_duration_limit_arithmetic(T):
    """[150, 150] sums to exactly 300 (rejected); the max-blob durations sum to just below it (accepted)."""
    D = ec.seq_sum(T)
    assert (D < ec.MAX_DURATION) == (len(T) == 64)

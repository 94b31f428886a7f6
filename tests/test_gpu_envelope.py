"""GPU tests at the edges of the trajectory and point-set envelope (run with -m gpu on a B200): 64 pieces with D just below
300 s (the largest trajectory blob, ~176 KB of k_outer shared memory), one piece, D below one lattice step, pieces shorter
than a descent step, piece boundaries and D exactly on lattice samples, points so far away that choiceTInit finds nothing
below 1e9, thousands of interior points, interior points at the rest ends, and both k_gsip widths.  The cases are built in
tests/envelope_cases.py; tests/test_oracle_envelope.py checks on the CPU that each reaches its edge.

Standard (as test_gpu_parity.test_strict_query_is_bit_identical_to_oracle): the strict build against the oracle gives the same
bits per point — sdf, t*, gradient and GSIP round count, outside and inside — and the cost to 1e-12, gradC and gradT to 1e-9."""
import os
import sys

import numpy as np
import pytest

from implicit_svsdf_planner_b200 import api

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import envelope_cases as ec  # noqa: E402

pytestmark = pytest.mark.gpu


def nrel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def gT_err(gT, gT_ref, gC_ref):
    """gradT error in units of its budget ||gradT|| + 1e-3 ||gradC|| (a heavily cancelling sum; see test_gpu_parity)."""
    return np.linalg.norm(np.asarray(gT) - gT_ref) / (np.linalg.norm(gT_ref) + 1e-3 * np.linalg.norm(gC_ref))


def oracle(oracle_mod, shape="star", **kw):
    return oracle_mod.Oracle(shape, threads=oracle_mod.num_procs(), **kw)


def assert_query_bitwise(ctx, orc, case, pts=None):
    """Outer solve and true SDF of every point, bit for bit; returns the oracle's (sdf, t*, grad, rounds)."""
    p = case.pts0() if pts is None else pts
    orc.set_traj(case.T, case.co())
    s_c, t_c, g_c = orc.query_outer(p)
    s_g, t_g, g_g, _ = ctx.query(case.T, case.co(), p, outer_only=True)
    assert np.array_equal(s_g, s_c) and np.array_equal(t_g, t_c) and np.array_equal(g_g, g_c), case.name
    ref = orc.query(p)
    got = ctx.query(case.T, case.co(), p)
    assert np.array_equal(got[3], ref[3]), case.name  # GSIP round counts
    for a, b in zip(got[:3], ref[:3]):
        bad = np.flatnonzero((a != b).reshape(p.shape[0], -1).any(axis=1))
        assert bad.size == 0, (case.name, bad[:5], ref[3][bad[:5]])
    return ref


def assert_cost_matches(ctx, orc, case, points=None):
    pts = case.points if points is None else points
    orc.set_points(pts)
    c0, gT0, gC0, _, inside = orc.cost_grad(case.T, case.co())
    ctx.set_points(pts)
    c1, gT1, gC1 = ctx.cost_grad(case.T, case.co())
    assert abs(c1 - c0) <= 1e-12 * max(1.0, abs(c0)), (case.name, c1, c0)
    assert nrel(gC1, gC0) <= 1e-9 and gT_err(gT1, gT0, gC0) <= 1e-9, (case.name, nrel(gC1, gC0), gT_err(gT1, gT0, gC0))
    return (c1, gT1, gC1), inside


@pytest.fixture(scope="module")
def max_blob():
    return ec.max_blob()


@pytest.fixture(scope="module")
def config1():
    return ec.config1()


# ----------------------------------------------------------------------------------------------------------------
# 1. trajectory envelope
# ----------------------------------------------------------------------------------------------------------------
def test_max_blob_natural_and_sparse_schedules(oracle_mod, max_blob, monkeypatch):
    """64 pieces, D = 299.99 s, 20 000 points: one CTA per SM, the batched schedule chosen by P, ~90 KB TMA copy; then the
    one-point-per-warp schedule on the same input gives the same bits."""
    c = max_blob
    monkeypatch.delenv("SVSDF_FORCE_GRID_OUTER", raising=False)
    monkeypatch.delenv("SVSDF_FORCE_BATCHED", raising=False)
    ctx = api.Context("star", strict_fp=True)
    orc = oracle(oracle_mod)
    ref = assert_query_bitwise(ctx, orc, c)
    assert (ref[3] > 0).any()  # interior points: k_gsip loads the same blob
    natural, _ = assert_cost_matches(ctx, orc, c)
    ctx.close()
    monkeypatch.setenv("SVSDF_FORCE_BATCHED", "0")
    ctx = api.Context("star", strict_fp=True)
    got = ctx.query(c.T, c.co(), c.pts0())
    for a, b in zip(got, ref):
        assert np.array_equal(a, b)
    sparse, _ = assert_cost_matches(ctx, orc, c)
    ctx.close()
    assert abs(sparse[0] - natural[0]) <= 1e-13 * abs(natural[0]) and nrel(sparse[2], natural[2]) <= 1e-12
    assert gT_err(sparse[1], natural[1], natural[2]) <= 1e-12


@pytest.mark.parametrize("functor", ["sdHorseshoe", "unknown_mesh_shape", "mesh"])
def test_max_blob_other_functors(oracle_mod, max_blob, functor):
    """The concave registry shape, the Polygon fallback (sign filter over a 2000-sample lattice) and the triangle-mesh functor
    (its own launch bound) with the largest blob."""
    if functor == "mesh":
        g = np.load(os.path.join(HERE, "golden", "fwn_ref.npz"))
        mesh = (g["star_V"], g["star_F"])
        ctx = api.Context("star_obj_mesh_sdf", mesh=mesh, strict_fp=True)
        orc = oracle(oracle_mod, mesh=mesh)
        P = 200
    else:
        ctx = api.Context(functor, strict_fp=True)
        orc = oracle(oracle_mod, functor)
        P = 600
    idx = np.random.default_rng(21).choice(max_blob.P, size=P, replace=False)
    c = max_blob.with_points(f"max_blob_{functor}", max_blob.points[np.sort(idx)])
    assert_query_bitwise(ctx, orc, c)
    assert_cost_matches(ctx, orc, c)
    ctx.close()


SHORT_CASES = {
    "single_piece": ec.single_piece,
    **{f"tiny_{D}": (lambda D=D: ec.tiny(D)) for D in ec.TINY_D},
    "sub_step": ec.sub_step,
    "on_boundaries": ec.on_boundaries,
    **{f"d_{w}": (lambda w=w: ec.d_lattice(w)) for w in ("on", "below", "above")},
}


@pytest.mark.parametrize("name", list(SHORT_CASES))
def test_trajectory_envelope_case(oracle_mod, name):
    """One piece; D below one lattice step and either side of the 32-sample window; 4 ms pieces; piece boundaries on lattice
    samples; D on, one ulp below and one ulp above a lattice sample (t = D rounds past the last piece)."""
    c = SHORT_CASES[name]()
    ctx = api.Context("star", strict_fp=True)
    orc = oracle(oracle_mod)
    assert_query_bitwise(ctx, orc, c)
    assert_cost_matches(ctx, orc, c)
    ctx.close()


# ----------------------------------------------------------------------------------------------------------------
# 2. degenerate points: no layer-1 sample below 1e9
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batched", ["0", "1"])
def test_far_points_alone_and_interleaved(oracle_mod, config1, batched, monkeypatch):
    monkeypatch.setenv("SVSDF_FORCE_GRID_OUTER", "2")
    monkeypatch.setenv("SVSDF_FORCE_BATCHED", batched)
    c = config1
    far = ec.far_points()
    mixed_pts, mask = ec.interleave_far(c.points, far)
    ctx = api.Context("star", strict_fp=True)
    orc = oracle(oracle_mod)
    alone = assert_query_bitwise(ctx, orc, c.with_points("far", far))
    assert np.all(alone[0] >= 1e9)
    mixed = assert_query_bitwise(ctx, orc, c.with_points("far_mixed", mixed_pts))
    for a, b in zip(mixed, alone):
        assert np.array_equal(a[mask], b)  # a far point's result does not depend on its neighbours in the warp
    # far points add nothing to the cost or the gradients
    ctx.set_points(far)
    cf, gTf, gCf = ctx.cost_grad(c.T, c.co())
    assert cf == 0.0 and not gTf.any() and not gCf.any()
    (cm, gTm, gCm), _ = assert_cost_matches(ctx, orc, c, mixed_pts)
    (cn, gTn, gCn), _ = assert_cost_matches(ctx, orc, c)
    assert abs(cm - cn) <= 1e-13 * abs(cn) and nrel(gCm, gCn) <= 1e-12 and gT_err(gTm, gTn, gCn) <= 1e-12
    ctx.close()


# ----------------------------------------------------------------------------------------------------------------
# 3. interior branch at scale and at rest
# ----------------------------------------------------------------------------------------------------------------
def test_many_inside_points(oracle_mod, config1):
    """~4000 interior points (more than one pass of k_gsip's grid), P = 7 (mod 16): k_compact's ragged tail."""
    c = ec.many_inside(config1)
    ctx = api.Context("star", strict_fp=True)
    orc = oracle(oracle_mod)
    ref = assert_query_bitwise(ctx, orc, c)
    _, inside = assert_cost_matches(ctx, orc, c)
    assert inside >= 3000 and inside == int((ref[3] > 0).sum())
    ctx.close()
    ctx = api.Context("star", strict_fp=True)
    ctx.set_points(c.points)
    _, out = ctx.cost_grad_device(c.T, c.co())
    assert int(out[-1]) == inside
    ctx.close()


def test_interior_points_at_the_rest_ends(oracle_mod, config1):
    c, g0, g1 = ec.rest_ends(config1)
    ctx = api.Context("star", strict_fp=True)
    orc = oracle(oracle_mod)
    ref = assert_query_bitwise(ctx, orc, c)
    assert np.all(ref[3][np.r_[g0, g1]] > 0)
    assert_cost_matches(ctx, orc, c)
    ctx.close()


def test_both_gsip_widths(oracle_mod, config1):
    """run_kernels picks the 22-warp k_gsip when the previous evaluation of the same point set had 1..sm_count interior
    points, the 8-warp one otherwise (first evaluation after set_points, or more interior points)."""
    import torch

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    few, many = ec.few_inside(), ec.many_inside(config1)
    orc = oracle(oracle_mod)
    orc.set_points(few.points)
    c0, gT0, gC0, _, n_few = orc.cost_grad(few.T, few.co())
    assert 1 <= n_few <= sms  # so the second evaluation runs the 22-warp variant
    ctx = api.Context("star", strict_fp=True)
    ctx.set_points(few.points)
    r8 = ctx.cost_grad(few.T, few.co())   # 8 warps
    r22 = ctx.cost_grad(few.T, few.co())  # 22 warps
    assert r8[0] == r22[0] and np.array_equal(r8[1], r22[1]) and np.array_equal(r8[2], r22[2])
    assert abs(r8[0] - c0) <= 1e-12 * abs(c0) and nrel(r8[2], gC0) <= 1e-9 and gT_err(r8[1], gT0, gC0) <= 1e-9

    def fresh(case):
        f = api.Context("star", strict_fp=True)
        f.set_points(case.points)
        r = f.cost_grad(case.T, case.co())
        f.close()
        return r

    rm = fresh(many)
    # 22 -> 8 (many interior points) -> 22 on the same context; every result equals a fresh context's
    ctx.set_points(many.points)
    for _ in range(2):  # the second evaluation stays at 8 warps (more interior points than SMs)
        r = ctx.cost_grad(many.T, many.co())
        assert r[0] == rm[0] and np.array_equal(r[1], rm[1]) and np.array_equal(r[2], rm[2])
    ctx.set_points(few.points)
    for _ in range(2):
        r = ctx.cost_grad(few.T, few.co())
        assert r[0] == r8[0] and np.array_equal(r[1], r8[1]) and np.array_equal(r[2], r8[2])
    ctx.close()


# ----------------------------------------------------------------------------------------------------------------
# 4. fast build and error edges
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["max_blob", "tiny_0.1", "tiny_4.81", "many_inside"])
def test_fast_build_at_the_edges(oracle_mod, max_blob, config1, name):
    """strict_fp = 0 (FMA contraction in the kernels) within the reference's own noise floor at the same sizes."""
    c = {"max_blob": lambda: max_blob, "many_inside": lambda: ec.many_inside(config1)}.get(name, SHORT_CASES.get(name))()
    ctx = api.Context("star", strict_fp=False)
    orc = oracle(oracle_mod)
    orc.set_traj(c.T, c.co())
    s_c, _, _, r_c = orc.query(c.pts0())
    s_g, _, _, r_g = ctx.query(c.T, c.co(), c.pts0())
    assert np.array_equal(r_g, r_c)
    out = r_c == 0
    assert np.abs(s_g - s_c)[out].max() <= 1e-9
    if (~out).any():
        # interior values: the reference's own source compiled with FMA contraction moves a few of the ~4000 interior points
        # of many_inside by up to ~5e-7 (a ring sample's descent ends elsewhere); the fast build may not do worse
        o_fma = oracle(oracle_mod, variant="fma")
        o_fma.set_traj(c.T, c.co())
        floor = np.abs(o_fma.query(c.pts0())[0] - s_c).max()
        assert np.abs(s_g - s_c)[~out].max() <= max(1e-9, 2.0 * floor)
    orc.set_points(c.points)
    c0, gT0, gC0, _, _ = orc.cost_grad(c.T, c.co())
    ctx.set_points(c.points)
    c1, gT1, gC1 = ctx.cost_grad(c.T, c.co())
    assert abs(c1 - c0) <= 1e-9 * max(1.0, abs(c0))
    assert nrel(gC1, gC0) <= 1e-4 and gT_err(gT1, gT0, gC0) <= 1e-4, (nrel(gC1, gC0), gT_err(gT1, gT0, gC0))
    ctx.close()


def test_duration_limit(max_blob):
    c = max_blob
    idx = np.random.default_rng(22).choice(c.P, size=2000, replace=False)
    pts = c.points[np.sort(idx)]
    ctx = api.Context("star", strict_fp=True)
    ctx.set_points(pts)
    first = ctx.cost_grad(c.T, c.co())  # D = 299.99 s is accepted
    assert np.isfinite(first[0]) and first[0] > 0
    with pytest.raises(api.SvsdfError):  # no pieces
        ctx.cost_grad(np.zeros(0), np.zeros(0))
    T300 = np.array([150.0, 150.0])
    assert T300[0] + T300[1] == 300.0
    with pytest.raises(api.SvsdfError):  # D exactly 300 s
        ctx.cost_grad(T300, c.co()[: 36])
    again = ctx.cost_grad(c.T, c.co())
    assert again[0] == first[0] and np.array_equal(again[1], first[1]) and np.array_equal(again[2], first[2])
    ctx.close()

"""Deformable robot (svsdf_set_scale) on the B200 (run with -m gpu).

The strict build must reproduce the reference's own source built with `useScale` on (tests/golden/ref_scale_path.npz,
portable libm) bit for bit per point, and the identity spec or a reset must give the rigid body's bits back.
"""
import os
import sys

import numpy as np
import pytest

from implicit_svsdf_planner_b200 import api, scenes
from oracle import scale_py

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_scale_golden as MG  # noqa: E402  (fixture loader)

G = MG.load()
IDENTITY = dict(x=(1.0, [(0.0, 1.5, -1.0)]), y=(1.0, []))


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _scene(key):
    return dict(shape=str(G[f"{key}_shape"]), N=int(G[f"{key}_N"]), T=G[f"{key}_T"], coeffs=G[f"{key}_coeffs"],
                points=G[f"{key}_points"], init_s=G[f"{key}_init_s"], final_s=G[f"{key}_final_s"], x0=G[f"{key}_x0"],
                params=G[f"{key}_params"])


def _ctx(s, **kw):
    wp, sh, rho = s["params"]
    return api.Context(s["shape"], weight_p=wp, safety_hor=sh, rho=rho, **kw)


def _all_outputs(ctx, T, co, pts):
    """query (sdf, t*, grad, rounds) + cost_grad on the same points."""
    p = np.c_[pts[:, :2], np.zeros(len(pts))]
    q = ctx.query(T, co, p)
    ctx.set_points(pts)
    return (*q, *ctx.cost_grad(T, co))


@pytest.mark.parametrize("case", [MG.case_name(*c) for c in MG.CASES])
def test_kernels_equal_the_scaled_reference(case):
    scene, spec = case.split("_")
    s = _scene(scene)
    ctx = _ctx(s, strict_fp=True)
    ctx.set_scale(**G["specs"][spec])
    sdf, ts, g, rounds, cost, gT, gC = _all_outputs(ctx, s["T"], s["coeffs"], s["points"])
    v = "portable"
    assert np.array_equal(sdf, G[f"{case}_sdf_{v}"]) and np.array_equal(ts, G[f"{case}_tstar_{v}"])
    assert np.array_equal(g, G[f"{case}_grad_{v}"]) and np.array_equal(rounds, G[f"rounds_{case}"])
    assert _rel(cost, G[f"{case}_cost_{v}"]) < 1e-11 and _rel(gT, G[f"{case}_gradT_{v}"]) < 1e-11
    assert _rel(gC, G[f"{case}_gradC_{v}"]) < 1e-11
    ctx.set_boundary(s["init_s"], s["final_s"], s["N"])
    f, gg = ctx.evaluate(s["x0"])
    assert _rel(f, G[f"{case}_f_{v}"]) < 1e-11 and _rel(gg, G[f"{case}_g_{v}"]) < 1e-11
    # exact yaw gradient: same per-point values, the oracle's sums
    ctx.set_scale(**G["specs"][spec], exact_yaw_grad=True)
    ctx.set_points(s["points"])
    cost, gT, gC = ctx.cost_grad(s["T"], s["coeffs"])
    assert _rel(cost, G[f"exact_{case}_cost"]) < 1e-11 and _rel(gT, G[f"exact_{case}_gradT"]) < 1e-11
    assert _rel(gC, G[f"exact_{case}_gradC"]) < 1e-11
    ctx.set_boundary(s["init_s"], s["final_s"], s["N"])
    f, gg = ctx.evaluate(s["x0"])
    assert _rel(f, G[f"exact_{case}_f"]) < 1e-11 and _rel(gg, G[f"exact_{case}_g"]) < 1e-11
    ctx.close()


@pytest.mark.parametrize("P", [600, 200_000])
def test_identity_spec_and_reset_give_the_rigid_bits(P):
    """Config 1 (the fixture's star scene) and config 2 at full size: an identity spec equals no spec bit for bit, and
    svsdf_set_scale(ctx, NULL) after a spec returns today's bits."""
    if P == 600:
        s = _scene("star")
        T, co, pts = s["T"], s["coeffs"], s["points"]
    else:
        sc = scenes.make_scene("star", 8, P)
        T, co, pts = sc.T, sc.coeffs_colmajor(), sc.points
    ctx = api.Context("star", weight_p=60.0, safety_hor=0.7, strict_fp=True)
    rigid = _all_outputs(ctx, T, co, pts)
    ctx.set_scale(**IDENTITY)
    ident = _all_outputs(ctx, T, co, pts)
    ctx.set_scale(**MG.SPECS["ref"])
    scaled = _all_outputs(ctx, T, co, pts)
    ctx.set_scale()
    reset = _all_outputs(ctx, T, co, pts)
    for a, b, c in zip(rigid, ident, reset):
        assert np.array_equal(a, b) and np.array_equal(a, c)
    assert not np.array_equal(scaled[0], rigid[0])
    ctx.close()


def test_invalid_specs_are_rejected_and_the_context_stays_usable():
    s = _scene("star")
    ctx = _ctx(s, strict_fp=True)
    ctx.set_scale(**MG.SPECS["ref"])
    before = _all_outputs(ctx, s["T"], s["coeffs"], s["points"][:200])
    bad = [
        dict(x=(0.5, [(0.5, 1.0, 0.0)]), y=(1.0, [])),                        # c - |a| = 0
        dict(x=(1.0, []), y=(0.5, [(0.3, 1.0, 0.0), (-0.3, 2.0, 0.0)])),       # c - sum |a| < 0
        dict(x=(-1.0, []), y=(1.0, [])),                                      # negative constant
        dict(x=(float("nan"), []), y=(1.0, [])),
        dict(x=(1.0, [(0.1, float("inf"), 0.0)]), y=(1.0, [])),
    ]
    for spec in bad:
        with pytest.raises(api.SvsdfError):
            ctx.set_scale(**spec)
    for n in (-1, 5):
        raw = api.scale_spec(**MG.SPECS["ref"])
        raw.n_terms[0] = n
        with pytest.raises(api.SvsdfError):
            ctx.set_scale(spec=raw)
    after = _all_outputs(ctx, s["T"], s["coeffs"], s["points"][:200])  # the previous (valid) spec is still in force
    for a, b in zip(before, after):
        assert np.array_equal(a, b)
    ctx.close()


def test_mesh_functor_with_scale_matches_the_oracle(oracle_mod, scene_small_inside):
    m = scenes.extrude_outline(scenes.star_outline(n_per_edge=2), half_height=0.49)
    sc = scene_small_inside
    co = sc.coeffs_colmajor()
    ctx = api.Context("ignored", strict_fp=True, mesh=m)
    ctx.set_scale(**MG.SPECS["ref"])
    orc = scale_py.ScaledOracle(mesh=m, **MG.SPECS["ref"], threads=oracle_mod.num_procs())
    orc.set_traj(sc.T, co)
    p = np.c_[sc.points[:, :2], np.zeros(sc.P)]
    s_c, t_c, g_c, r_c = orc.query(p)
    s_g, t_g, g_g, r_g = ctx.query(sc.T, co, p)
    assert sc.P >= 200 and (r_c > 0).sum() >= 1
    assert np.array_equal(s_g, s_c) and np.array_equal(t_g, t_c) and np.array_equal(g_g, g_c) and np.array_equal(r_g, r_c)
    ctx.close()


def test_optimize_with_the_reference_example_is_deterministic():
    s = _scene("star")
    params = api.default_lbfgs_params(mem_size=16, past=3, delta=1e-6, g_epsilon=0.0, max_iterations=0, min_step=1e-32)
    runs = []
    for _ in range(2):
        ctx = _ctx(s, strict_fp=True)
        ctx.set_scale(**MG.SPECS["ref"])
        ctx.set_points(s["points"])
        for _ in range(2):
            rc, x, T, b, st = ctx.optimize(s["init_s"], s["final_s"], s["x0"], s["N"], params)
            assert rc >= 0, rc
            runs.append((x, T, b, st["final_cost"]))
        ctx.close()
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert np.array_equal(a, b)

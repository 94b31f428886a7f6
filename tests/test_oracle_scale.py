"""Deformable robot (body scale S(t)) on the CPU: the oracle's scaled mode (oracle/scale_oracle.cpp) against the reference's
own source built with `useScale` on (oracle/_ref/libref_path_scaled_*.so, or its committed outputs
tests/golden/ref_scale_path.npz where the libraries are absent), the identity scale against the rigid body, and the
yaw-gradient finding by finite differences."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, "golden"))
from implicit_svsdf_planner_b200 import scenes  # noqa: E402
from oracle import oracle_py as O  # noqa: E402
from oracle import ref_py as R  # noqa: E402
from oracle import scale_py as SP  # noqa: E402

import make_scale_golden as MG  # noqa: E402

G = MG.load()
ORACLE_OF = {"portable": "default", "glibc": "glibc"}  # reference build -> oracle build with the same libm


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(1.0, float(np.max(np.abs(b)))))


def _scene(key):
    return dict(shape=str(G[f"{key}_shape"]), N=int(G[f"{key}_N"]), T=G[f"{key}_T"], coeffs=G[f"{key}_coeffs"],
                points=G[f"{key}_points"], init_s=G[f"{key}_init_s"], final_s=G[f"{key}_final_s"], x0=G[f"{key}_x0"],
                params=G[f"{key}_params"])


def _reference_outputs(scene, spec, v):
    """The scaled reference's outputs for one case: computed now when its library exists, else the committed ones."""
    cn = MG.case_name(scene, spec)
    if not R.available("scaled_" + v):
        return {k: G[f"{cn}_{k}_{v}"] for k in ("sdf", "tstar", "grad", "cost", "gradT", "gradC", "f", "g")}
    s = _scene(scene)
    wp, sh, rho = s["params"]
    ref = SP.scaled_ref(s["shape"], **G["specs"][spec], weight_p=wp, safety_hor=sh, rho=rho, threads=8, variant="scaled_" + v)
    ref.set_traj(s["T"], s["coeffs"])
    out = dict(zip(("sdf", "tstar", "grad"), ref.query(np.c_[s["points"][:, :2], np.zeros(len(s["points"]))])))
    ref.set_threads(1)
    ref.set_points(s["points"])
    out["cost"], out["gradT"], out["gradC"] = ref.cost_grad(s["T"], s["coeffs"])
    ref.set_conditions(s["init_s"], s["final_s"], s["N"])
    out["f"], out["g"] = ref.evaluate(s["x0"])
    return out


def _oracle(scene, spec, variant="default", exact=False, threads=8):
    """The scaled oracle for a spec, the rigid oracle for spec None."""
    s = _scene(scene)
    wp, sh, rho = s["params"]
    if spec is None:
        orc = O.Oracle(s["shape"], weight_p=wp, safety_hor=sh, rho=rho, threads=threads, variant=variant)
    else:
        orc = SP.ScaledOracle(s["shape"], **G["specs"][spec], exact_yaw_grad=exact, weight_p=wp, safety_hor=sh, rho=rho,
                              threads=threads, variant=variant)
    orc.set_traj(s["T"], s["coeffs"])
    return orc, s


@pytest.mark.parametrize("v", ["portable", "glibc"])
@pytest.mark.parametrize("case", [MG.case_name(*c) for c in MG.CASES])
def test_oracle_equals_scaled_reference(case, v):
    """Per point bit for bit (sdf, t*, gradient; portable reference = default oracle, glibc = glibc); sums to 1e-13."""
    scene, spec = case.split("_")
    ref = _reference_outputs(scene, spec, v)
    orc, s = _oracle(scene, spec, ORACLE_OF[v])
    sdf, ts, g, rounds = orc.query(np.c_[s["points"][:, :2], np.zeros(len(s["points"]))])
    assert np.array_equal(sdf, ref["sdf"]) and np.array_equal(ts, ref["tstar"]) and np.array_equal(g, ref["grad"])
    if v == "portable":
        assert np.array_equal(rounds, G[f"rounds_{case}"])
    orc.set_threads(1)
    orc.set_points(s["points"])
    cost, gT, gC = orc.cost_grad(s["T"], s["coeffs"])
    assert _rel(cost, ref["cost"]) < 1e-13 and _rel(gT, ref["gradT"]) < 1e-13 and _rel(gC, ref["gradC"]) < 1e-13
    orc.set_conditions(s["init_s"], s["final_s"], s["N"])
    f, gg = orc.evaluate(s["x0"])
    assert _rel(f, ref["f"]) < 1e-13 and _rel(gg, ref["g"]) < 1e-13


def test_golden_cases_run_the_interior_branch_and_move_the_body():
    """The fixture exercises GSIP, and the scale changes what the rigid body would give."""
    for scene, spec in MG.CASES:
        cn = MG.case_name(scene, spec)
        if scene != "star" or spec != "iso":
            assert (G[f"rounds_{cn}"] > 0).sum() >= 2, cn
        orc, s = _oracle(scene, None)
        sdf = orc.query(np.c_[s["points"][:, :2], np.zeros(len(s["points"]))])[0]
        assert (sdf != G[f"{cn}_sdf_portable"]).mean() > 0.5, cn


@pytest.mark.parametrize("unit", [dict(x=(1.0, []), y=(1.0, [])), dict(x=(1.0, [(0.0, 1.5, -1.0)]), y=(1.0, [(0.0, 1.8, 0.0)]))])
def test_identity_scale_equals_rigid(unit):
    s = _scene("star")
    wp, sh, rho = s["params"]
    outs = []
    for spec in (None, unit):
        if spec is None:
            orc = O.Oracle(s["shape"], weight_p=wp, safety_hor=sh, rho=rho, threads=1)
        else:
            orc = SP.ScaledOracle(s["shape"], **spec, weight_p=wp, safety_hor=sh, rho=rho, threads=1)
        orc.set_traj(s["T"], s["coeffs"])
        q = orc.query(np.c_[s["points"][:, :2], np.zeros(len(s["points"]))])
        orc.set_points(s["points"])
        cg = orc.cost_grad(s["T"], s["coeffs"])
        orc.set_conditions(s["init_s"], s["final_s"], s["N"])
        outs.append((*q, cg[0], cg[1], cg[2], *orc.evaluate(s["x0"])))
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


def _fd_penalty(orc, T, co, wrt, h=1e-6):
    fd = np.zeros(len(co) if wrt == "coeffs" else len(T))
    for i in range(len(fd)):
        if wrt == "coeffs":
            cp, cm = co.copy(), co.copy()
            cp[i] += h
            cm[i] -= h
            fd[i] = (orc.cost_grad(T, cp)[0] - orc.cost_grad(T, cm)[0]) / (2 * h)
        else:
            tp, tm = T.copy(), T.copy()
            tp[i] += h
            tm[i] -= h
            fd[i] = (orc.cost_grad(tp, co)[0] - orc.cost_grad(tm, co)[0]) / (2 * h)
    return fd


def _err(fd, an):
    return np.abs(fd - an) / np.maximum(1e-3 * np.abs(an).max(), np.abs(an))


def test_yaw_gradient_by_finite_differences():
    """exact_yaw_grad = 1: the penalty's gradient with respect to every MINCO coefficient and every duration matches central
    differences.  Default (the reference's formula g^T VR^T (p - x)): the x / y coefficients still match, the yaw coefficients
    and — through gdT = -G . vel — the durations do not; the gap is pinned here so that it stays documented.
    Points with sdf > 0.05 only: the interior branch's ring search is not differentiable."""
    sc = scenes.make_scene("star", 8, 300)
    co = sc.coeffs_colmajor().reshape(-1)
    spec = G["specs"]["ref"]
    errs = {}
    for exact in (True, False):
        orc = SP.ScaledOracle("star", **spec, exact_yaw_grad=exact, weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho,
                              threads=8)
        orc.set_traj(sc.T, co)
        sdf = orc.query(np.c_[sc.points[:, :2], np.zeros(sc.P)])[0]
        orc.set_points(sc.points[sdf > 0.05])
        _, gT, gC = orc.cost_grad(sc.T, co)
        eC = _err(_fd_penalty(orc, sc.T, co, "coeffs"), gC).reshape(3, -1).max(axis=1)
        eT = _err(_fd_penalty(orc, sc.T, co, "T"), gT).max()
        errs[exact] = (eC, eT)
    (ex_c, ex_t), (ref_c, ref_t) = errs[True], errs[False]
    assert ex_c.max() < 1e-3 and ex_t < 1e-3, errs
    assert ref_c[0] < 1e-3 and ref_c[1] < 1e-3, errs
    assert ref_c[2] > 0.1 and ref_t > 0.01, errs


def test_exact_yaw_golden_matches_oracle():
    """The committed exact-yaw outputs are reproducible (they are the oracle's own)."""
    for scene, spec in MG.CASES:
        cn = MG.case_name(scene, spec)
        orc, s = _oracle(scene, spec, exact=True, threads=1)
        orc.set_points(s["points"])
        cost, gT, gC = orc.cost_grad(s["T"], s["coeffs"])
        assert _rel(cost, G[f"exact_{cn}_cost"]) < 1e-13 and _rel(gT, G[f"exact_{cn}_gradT"]) < 1e-13
        assert _rel(gC, G[f"exact_{cn}_gradC"]) < 1e-13
        # the yaw column is where the two modes differ
        assert not np.array_equal(gC.reshape(3, -1)[2], G[f"{cn}_gradC_portable"].reshape(3, -1)[2])


@pytest.mark.skipif(not os.path.isdir("/root/reference/src"), reason="needs the reference tree")
def test_scaled_fragment_leaves_out_get_scale_only():
    """The useScale build's methods are sw_methods.inc without the cut getScale block (the shim supplies it)."""
    gen = os.path.join(ROOT, "oracle", "_ref", "gen")
    if not os.path.exists(os.path.join(gen, "sw_methods_scaled.inc")):
        pytest.skip("oracle/_ref/gen not generated")
    full = open(os.path.join(gen, "sw_methods.inc"), encoding="utf-8", errors="surrogateescape").read()
    scaled = open(os.path.join(gen, "sw_methods_scaled.inc"), encoding="utf-8", errors="surrogateescape").read()
    assert "getScale(const double t)" in full and "getScale(const double t)" not in scaled
    assert "getDotScale(const double t)" in scaled
    assert len(full) - len(scaled) < 1200

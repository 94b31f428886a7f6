"""GPU parity against THE REFERENCE'S OWN CODE (run with -m gpu on a B200).

tests/golden/ref_pin_*.npz hold what the reference's source computes (compiled where it lies under /root/reference into
oracle/_ref/libref_path_*.so, tests/golden/make_ref_pin_golden.py).  The "portable" variant is the reference with only its
per-sample libm calls (sin, cos, atan2) redirected to the pinned fdlibm algorithm the kernels implement — everything else
(shape classes, Piece<5>, choiceTInit, gradientDescent, the FD gradient, the GSIP loop) is the reference's text.  The CUDA
path (strict build, through the C ABI) must reproduce every per-point output of it BIT FOR BIT; sums to rounding.
Against the "glibc" variant (the reference as it runs) the known libm noise floor applies (see test_gpu_parity.py).
"""
import os
import sys

import numpy as np
import pytest

from implicit_svsdf_planner_b200 import api

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
sys.path.insert(0, GOLD)
import make_ref_pin_golden as mk  # noqa: E402  (fixture loader; its reference calls are not used here)


def bits_differ(a, b):
    """Number of elements whose bit patterns differ; -0.0 and +0.0 count as equal (the kernels skip the body-frame
    pre-transform when it is the identity, the reference multiplies by it: x * 1 + y * 0 + z * 0 turns a -0.0 input into
    +0.0 — the only observable difference, and only for inputs that are exactly -0.0)."""
    a = np.ascontiguousarray(a, dtype=np.float64).ravel() + 0.0
    b = np.ascontiguousarray(b, dtype=np.float64).ravel() + 0.0
    assert a.shape == b.shape
    return int((a.view(np.int64) != b.view(np.int64)).sum())


@pytest.fixture(scope="module")
def gshapes():
    return mk.load_fixture("ref_pin_shapes.npz")


@pytest.fixture(scope="module")
def gpath():
    return np.load(os.path.join(GOLD, "ref_pin_path.npz"))


def test_shape_functors_are_bitwise_the_reference_classes(gshapes):
    rel = gshapes["rel"]
    rel0 = np.c_[rel[:, :2], np.zeros(len(rel))]  # the C ABI evaluates the planar functors at (x, y); z is ignored by them
    for ip, pp in enumerate(gshapes["pre"]):
        for s in gshapes["shapes"]:
            s = str(s)
            ctx = api.Context(s, poly_params=tuple(pp), strict_fp=True)
            assert bits_differ(ctx.shape_sdf(rel0), gshapes[f"sdf_portable_{ip}_{s}"]) == 0, (s, ip)
            g = ctx.shape_grad1(rel0[:400])
            gr = gshapes[f"grad1_portable_{ip}_{s}"]
            if s == "fallbackPolygon":  # Polygon::getonlyGrad1 keeps pos_rel(2) - pos_rel(2) = 0 in z; same numbers in x, y
                assert bits_differ(g[:, :2], gr[:, :2]) == 0, (s, ip)
            else:
                assert bits_differ(g, gr) == 0, (s, ip)
            ctx.close()


def test_front_end_shape_kernels_are_the_reference_initshape(gshapes):
    ks, K, res, safeh = gshapes["kernel_cfg"]
    for s in gshapes["shapes"][:16]:
        s = str(s)
        ctx = api.Context(s)
        ctx.front_init(int(ks), int(K), float(res), float(safeh))
        yaw, _, byt = ctx.front_kernels()
        assert bits_differ(yaw, gshapes[f"kyaw_portable_{s}"]) == 0
        assert np.array_equal(byt, gshapes[f"kbytes_portable_{s}"]), s
        ctx.close()


@pytest.mark.parametrize("key", ["c1", "inside", "c3s"])
def test_path_is_bitwise_the_reference_code(gpath, key):
    g = gpath
    shape, N = str(g[f"{key}_shape"]), int(g[f"{key}_N"])
    T, co, pts = g[f"{key}_T"], g[f"{key}_coeffs"], g[f"{key}_points"]
    wp, sh, rho = (float(v) for v in g[f"{key}_params"])
    ctx = api.Context(shape, weight_p=wp, safety_hor=sh, rho=rho, strict_fp=True)
    p0 = np.c_[pts[:, :2], np.zeros(len(pts))]
    # per-point query API (getTrueSDFofSweptVolume<true>): outside AND interior (GSIP) points
    sdf, tstar, grad, rounds = ctx.query(T, co, p0)
    assert bits_differ(sdf, g[f"{key}_sdf_portable"]) == 0
    assert bits_differ(tstar, g[f"{key}_tstar_portable"]) == 0
    assert bits_differ(grad, g[f"{key}_grad_portable"]) == 0
    assert np.array_equal(rounds > 0, g[f"{key}_sdf_portable"] <= 0)
    so, to, go, _ = ctx.query(T, co, p0[:200], outer_only=True)
    assert bits_differ(so, g[f"{key}_osdf_portable"]) + bits_differ(to, g[f"{key}_otstar_portable"]) + bits_differ(go, g[f"{key}_ograd_portable"]) == 0
    # the accumulating penalty loop and the whole callback: sums, to summation-order rounding
    ctx.set_points(pts)
    c, gT, gC = ctx.cost_grad(T, co)
    rc, rT, rC = float(g[f"{key}_cost_portable"]), g[f"{key}_gradT_portable"], g[f"{key}_gradC_portable"]
    assert abs(c - rc) <= 1e-12 * abs(rc)
    assert np.linalg.norm(gC - rC) <= 1e-11 * np.linalg.norm(rC)
    assert np.abs(gT - rT).max() <= 1e-11 * np.linalg.norm(rC)  # -G.vel cancels at interior minima: scale of the terms
    ctx.set_boundary(g[f"{key}_init_s"], g[f"{key}_final_s"], N)
    f, gg = ctx.evaluate(g[f"{key}_x0"])
    rf, rg = float(g[f"{key}_f_portable"]), g[f"{key}_g_portable"]
    assert abs(f - rf) <= 1e-12 * abs(rf)
    assert np.linalg.norm(gg - rg) <= 1e-10 * np.linalg.norm(rg)
    # and against the reference as it really runs (glibc libm): the north-star tolerance on the cost, the documented
    # flat-minimum noise floor on the gradient
    assert abs(c - float(g[f"{key}_cost_glibc"])) <= 1e-9 * abs(c)
    assert abs(f - float(g[f"{key}_f_glibc"])) <= 1e-9 * abs(f)
    assert np.linalg.norm(gg - g[f"{key}_g_glibc"]) <= 1e-4 * np.linalg.norm(gg)
    assert np.abs(sdf - g[f"{key}_sdf_glibc"]).max() <= 1e-9
    ctx.close()


def test_live_reference_library_on_this_box_agrees_at_20k_points():
    """A scene of 20 000 fresh seeded points, not only the committed path fixture: every point is queried, a seeded sample of
    2 000 is compared with what the reference's portable build computes there (ref_pin_sample.npz)."""
    g = mk.load_fixture("ref_pin_sample.npz")
    sc = mk.scene_20k()
    idx = g["scene20k_idx"]
    ctx = api.Context("star", weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, strict_fp=True)
    s, t, gr, _ = ctx.query(sc.T, sc.coeffs_colmajor(), np.c_[sc.points[:, :2], np.zeros(sc.P)])
    assert bits_differ(s[idx], g["scene20k_sdf"]) + bits_differ(t[idx], g["scene20k_tstar"]) + bits_differ(gr[idx], g["scene20k_grad"]) == 0
    ctx.close()

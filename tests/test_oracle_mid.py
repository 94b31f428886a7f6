"""CPU tests of the mid end (SURVEY.md §8f rank 4): the product's host code (csrc/host/mid_end.hpp, through the C ABI svsdf_mid_*)
against THE REFERENCE'S OWN CODE — OriTraj's member functions and getOriTraj cut verbatim from mid_end.hpp / mid_end.cpp, the flatness
map, MINCO and the patched L-BFGS included whole, compiled into oracle/_ref/libref_mid.so (oracle/ref_mid_shim.cpp).  Committed outputs of
that library: tests/golden/ref_mid.npz (tests/golden/make_mid_golden.py)."""
import os
import sys

import numpy as np
import pytest

from implicit_svsdf_planner_b200 import api

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_mid_golden as mk  # noqa: E402  (problem generator and the two parameter sets; its reference calls are not used here)


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(HERE, "golden", "ref_mid.npz"))


@pytest.mark.parametrize("cname", list(mk.CONFIGS))
@pytest.mark.parametrize("N", [2, 3, 6, 12])
def test_cost_and_gradient_equal_the_reference_cost_function(gold, cname, N):
    """OriTraj::costFunction: MINCO energy + cubic waypoint pull + trapezoid integral of the velocity / body-rate / attitude penalties
    through the flatness map + rho sum(T), and its gradient w.r.t. (tau, xi).  Same operations, the band solve of MINCO in another
    order: rounding-level agreement."""
    k = f"{cname}_N{N}_"
    cfg = api.mid_default_config(**mk.CONFIGS[cname])
    c, g = api.mid_cost(gold[k + "init_s"], gold[k + "final_s"], gold[k + "Q"], gold[k + "rots"], gold[k + "x"], cfg)
    assert abs(c - float(gold[k + "cost"])) <= 1e-13 * abs(c)
    assert np.linalg.norm(g - gold[k + "grad"]) <= 1e-11 * np.linalg.norm(g)


def test_gradient_is_the_derivative_of_the_cost():
    """Central differences.  (The attitude term's cost and gradient routines disagree in the reference itself — costaltitude has
    `- 2 c1 (2 w x + y z)`, gradaltitude differentiates `2 y z` — so the check runs with the yaml's weight_ar = 0 and, with the term
    on, only requires the mismatch to stay the size of that term.)"""
    init_s, final_s, Q, rots, x = mk.problem(6, 7)
    for over, tol in (({}, 1e-7), (dict(vmax=1.5, omgmax=0.8, integralIntervs=8), 1e-7), (dict(weight_ar=3.0), 5e-2)):
        cfg = api.mid_default_config(**over)
        c, g = api.mid_cost(init_s, final_s, Q, rots, x, cfg)
        fd = np.zeros_like(x)
        for i in range(x.size):
            e = np.zeros_like(x)
            e[i] = 1e-6
            fd[i] = (api.mid_cost(init_s, final_s, Q, rots, x + e, cfg)[0] - api.mid_cost(init_s, final_s, Q, rots, x - e, cfg)[0]) / 2e-6
        assert np.linalg.norm(fd - g) <= tol * np.linalg.norm(g), (over, np.linalg.norm(fd - g) / np.linalg.norm(g))


@pytest.mark.parametrize("cname", list(mk.CONFIGS))
@pytest.mark.parametrize("N", [2, 3, 6, 12])
def test_warm_start_is_the_reference_warm_start(gold, cname, N):
    """getOriTraj with solver = 0 (default): the reference's patched L-BFGS behaviour (Armijo-only line search, quasi-Newton directions
    of length >= 0.04 replaced by -g at the previous direction's length, stop after 100 iterations) restated in host/lbfgs.hpp.  Same
    function, same rules: the iterates follow the reference's for 100 iterations — opt_x agrees to 1e-8 or better in 7 of the 8 golden
    cases; in one the two runs part at a rounding-level accept / reject decision late in the run and end 2e-3 apart in x, 1.3e-5 in cost."""
    k = f"{cname}_N{N}_"
    cfg = api.mid_default_config(**mk.CONFIGS[cname])
    assert cfg.solver == 0
    args = (gold[k + "init_s"], gold[k + "final_s"], gold[k + "Q"])
    rc, x, T, co, fc, it = api.mid_get_ori_traj(*args, np.ones(N), gold[k + "rots"], cfg)
    assert rc >= 0 and it == int(gold[k + "iterations"]) == 101
    c_ref, _ = api.mid_cost(*args, gold[k + "rots"], gold[k + "opt_x"], cfg)
    dx = np.abs(x - gold[k + "opt_x"]).max()
    assert dx <= 1e-6 or abs(fc - c_ref) <= 1e-4 * abs(c_ref), (dx, fc, c_ref)
    assert abs(fc - c_ref) <= 1e-4 * abs(c_ref)
    if dx <= 1e-6:
        assert np.abs(T - gold[k + "T"]).max() <= 1e-6 and np.abs(co - gold[k + "coeffs"]).max() <= 1e-5 * np.abs(co).max()
    # the spline returned is the one of (T, inner points): boundary states and waypoints are interpolated
    assert co.shape == (6 * N, 3)
    assert np.allclose(co[0], gold[k + "init_s"][:, 0]) and np.allclose(co[1], gold[k + "init_s"][:, 1])
    P = x[N:].reshape(N - 1, 3)
    for i in range(N - 1):
        assert np.allclose(co[6 * (i + 1)], P[i], atol=1e-9)


@pytest.mark.parametrize("cname", list(mk.CONFIGS))
@pytest.mark.parametrize("N", [2, 3, 6, 12])
def test_own_solver_reaches_at_least_what_the_reference_reaches(gold, cname, N):
    """solver = 1: this build's L-BFGS (weak-Wolfe line search, restarts) under the same 100-iteration rule — never worse than the
    reference's result (evaluated by the same cost function), usually converged well before the limit."""
    k = f"{cname}_N{N}_"
    cfg = api.mid_default_config(solver=1, **mk.CONFIGS[cname])
    args = (gold[k + "init_s"], gold[k + "final_s"], gold[k + "Q"])
    rc, x, T, co, fc, it = api.mid_get_ori_traj(*args, np.ones(N), gold[k + "rots"], cfg)
    assert rc >= 0 and it <= 101 and np.all(T > 0) and np.all(np.isfinite(co))
    c_ref, _ = api.mid_cost(*args, gold[k + "rots"], gold[k + "opt_x"], cfg)
    c_own, _ = api.mid_cost(*args, gold[k + "rots"], x, cfg)
    assert abs(c_own - fc) <= 1e-12 * abs(fc) and fc <= c_ref * (1.0 + 1e-6), (fc, c_ref)


def test_live_reference_library_when_present(gold):
    """Cost and gradient away from the golden x: the reference's values at seeded perturbations of two further problems
    (tests/golden/ref_mid_perturbed.npz, make_mid_golden.perturbed_fixture)."""
    ref = np.load(os.path.join(HERE, "golden", "ref_mid_perturbed.npz"))
    for k, N, cfg, init_s, final_s, Q, rots, xx in mk.perturbed_cases():
        c, g = api.mid_cost(init_s, final_s, Q, rots, xx, cfg)
        cr, gr = float(ref[k + "cost"]), ref[k + "grad"]
        assert abs(c - cr) <= 1e-13 * abs(cr) and np.linalg.norm(g - gr) <= 1e-11 * np.linalg.norm(gr), k


def test_mid_end_argument_checks():
    init_s, final_s, Q, rots, x = mk.problem(3, 1)
    with pytest.raises(api.SvsdfError):
        api.mid_cost(init_s, final_s, Q, rots, x, api.mid_default_config(integralIntervs=0))
    with pytest.raises(api.SvsdfError):
        api.mid_get_ori_traj(init_s, final_s, Q, np.array([1.0, -1.0, 1.0]), rots)


def test_cpp_mirror_of_the_mid_end_runs_without_a_gpu(tmp_path):
    """include/svsdf.hpp: svsdf::OriTraj over the C ABI, driven by tests/cpp/mid_main.cpp like plan_manager.cpp:176-192 drives the
    original; linked against the shipped library, executed on the host (the mid end needs no GPU)."""
    import subprocess

    from implicit_svsdf_planner_b200 import build

    root = os.path.dirname(HERE)
    so = build.build()
    exe = str(tmp_path / "mid_main")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "mid_main.cpp"),
                           so, "-Wl,-rpath," + os.path.dirname(so), "-o", exe])
    N = 6
    init_s, final_s, Q, rots, _ = mk.problem(N, 42)
    i_s, f_s, q, r, _ = api._mid_args(init_s, final_s, Q, rots)
    inp = tmp_path / "problem.txt"
    inp.write_text(f"{N} 1.0\n" + " ".join(repr(float(v)) for v in np.r_[i_s, f_s, q, r]) + "\n")
    out = subprocess.run([exe, str(inp)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    lines = out.stdout.strip().split("\n")
    ok, fc, it = lines[0].split()
    x = np.array([float(v) for v in lines[1].split()])
    T = np.array([float(v) for v in lines[2].split()])
    rc, x2, T2, co2, fc2, it2 = api.mid_get_ori_traj(init_s, final_s, Q, np.ones(N), rots)
    assert ok == "1" and rc >= 0 and int(it) == it2 and float(fc) == fc2
    assert np.array_equal(x, x2) and np.array_equal(T, T2)

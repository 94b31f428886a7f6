"""Golden vectors for the mid end (OriTraj) from the REFERENCE'S OWN CODE.

Runs in the build container only (needs /root/reference):  python tests/golden/make_mid_golden.py
`make -C oracle ref_path` compiles the reference's mid end — mid_end.hpp's member functions and mid_end.cpp's getOriTraj cut verbatim by
oracle/ref_extract.py, utils/flatness.hpp / utils/lbfgs.hpp / utils/minco.hpp included whole — against the Eigen stand-in into
oracle/_ref/libref_mid.so.  This script runs it on seeded problems (two parameter sets: config/star.yaml's and one with the attitude
term switched on and tight velocity / body-rate limits so that every penalty branch is active) and stores inputs and outputs in
tests/golden/ref_mid.npz: cost and gradient of OriTraj::costFunction at a random x, and what OriTraj::getOriTraj returns with the
reference's own patched L-BFGS (opt_x, T, iterations)."""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from implicit_svsdf_planner_b200 import api  # noqa: E402  (only for the config struct and the argument packing)
from oracle import ref_py as R  # noqa: E402

CONFIGS = {"star_yaml": {}, "all_terms": dict(weight_ar=3.0, vmax=1.5, omgmax=0.8, integralIntervs=8)}


def rot(a, b):
    ca, sa, cb, sb = np.cos(a), np.sin(a), np.cos(b), np.sin(b)
    return np.array([[ca, -sa, 0], [sa, ca, 0], [0, 0, 1]]) @ np.array([[1, 0, 0], [0, cb, -sb], [0, sb, cb]])


def problem(N, seed):
    rng = np.random.Generator(np.random.MT19937(seed))
    init_s, final_s = np.zeros((3, 3)), np.zeros((3, 3))
    init_s[:, 0] = [0, 0, 1]
    final_s[:, 0] = [3 * N, 5, 2]
    init_s[:, 1] = [0.3, 0.1, 0]
    Q = np.linspace(init_s[:, 0], final_s[:, 0], N + 1)[1:-1].T + rng.normal(0, 0.5, (3, N - 1))
    rots = np.stack([rot(*rng.uniform(-0.5, 0.5, 2)) for _ in range(N - 1)])
    x = np.r_[rng.normal(0, 0.5, N), (Q + rng.normal(0, 0.3, Q.shape)).T.reshape(-1)]
    return init_s, final_s, Q, rots, x


def perturbed_cases():
    """(key, N, cfg, init_s, final_s, Q, rots, x) at seeded perturbations of two problems, both parameter sets."""
    rng = np.random.default_rng(3)
    for N in (4, 9):
        init_s, final_s, Q, rots, x = problem(N, 500 + N)
        for cname, over in CONFIGS.items():
            cfg = api.mid_default_config(**over)
            for j in range(3):
                yield f"{cname}_N{N}_{j}_", N, cfg, init_s, final_s, Q, rots, x + rng.normal(0, 0.2, x.shape)


def perturbed_fixture():
    """ref_mid_perturbed.npz: cost and gradient of the reference's OriTraj::costFunction at perturbed_cases."""
    out = {}
    for k, N, cfg, init_s, final_s, Q, rots, x in perturbed_cases():
        i_s, f_s, q, r, _ = api._mid_args(init_s, final_s, Q, rots)
        out[k + "cost"], out[k + "grad"] = R.mid_cost(cfg, N, i_s, f_s, q, r, x)
    np.savez_compressed(os.path.join(HERE, "ref_mid_perturbed.npz"), **out)


def main():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref_path"], stdout=subprocess.DEVNULL)
    perturbed_fixture()
    out = {}
    for cname, over in CONFIGS.items():
        cfg = api.mid_default_config(**over)
        for N in (2, 3, 6, 12):
            init_s, final_s, Q, rots, x = problem(N, 100 + N)
            i_s, f_s, q, r, _ = api._mid_args(init_s, final_s, Q, rots)
            c, g = R.mid_cost(cfg, N, i_s, f_s, q, r, x)
            ok, xo, T, co, it = R.mid_get_ori_traj(cfg, N, i_s, f_s, q, np.ones(N), r)
            k = f"{cname}_N{N}_"
            out.update({k + "init_s": init_s, k + "final_s": final_s, k + "Q": Q, k + "rots": rots, k + "x": x, k + "cost": c, k + "grad": g,
                        k + "ok": ok, k + "opt_x": xo, k + "T": T, k + "coeffs": co, k + "iterations": it})
            print(k, "cost", c, "getOriTraj ok", ok, "iterations", it, "sum T", T.sum())
    np.savez_compressed(os.path.join(HERE, "ref_mid.npz"), **out)


if __name__ == "__main__":
    main()

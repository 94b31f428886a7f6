"""Generate tests/golden/ref_pin_*.npz: outputs of THE REFERENCE'S OWN CODE for the analytic hot path.

    make -C oracle ref_path && python tests/golden/make_ref_pin_golden.py      (only where /root/reference exists)

The libraries oracle/_ref/libref_path_{glibc,portable}.so are the reference's source compiled where it lies
(oracle/ref_path_shim.cpp: trajectory.hpp and minco.hpp included whole; the Shape.hpp classes, the SweptVolumeManager
query methods and the TrajOptimizer penalty loop cut verbatim by oracle/ref_extract.py; Eigen = oracle/ref_shim).
"glibc" is the reference as it runs on x86-64; "portable" has its sin/cos/atan2 calls redirected to the pinned fdlibm
algorithm that the CUDA kernels implement — so the CUDA path can be compared with the reference's own code BIT FOR BIT.

Fixtures (inputs + reference outputs; the reference tree cannot travel to the GPU box, these can):
  ref_pin_shapes.npz  16 registry shapes + Circle + Polygon fallback x 2 body-frame pre-transforms: getonlySDF on 2 000
                      points, getonlyGrad1 on 400, BasicShape::initShape byte kernels (17 x 17 x 18 yaws)
  ref_pin_sample.npz  seeded samples of larger inputs (sample_fixture)
  ref_pin_path.npz    three scenes (config 1: star / N = 8 / 2 000 points; a 400-point scene with ~6 % interior points;
                      sdHorseshoe / N = 16 / 1 500 points): Trajectory<5>::getPos/getVel samples, per point
                      getTrueSDFofSweptVolume<true> (sdf, t*, gradient), the accumulating penalty loop (cost, gradT,
                      gradC), costFunctionLmbmParallel (f, g) at x0, MINCO_S3NU forward/adjoint, smoothedL1, tau<->T
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from implicit_svsdf_planner_b200 import scenes  # noqa: E402
from oracle import ref_py as R  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SHAPES = ["star", "sdHorseshoe", "sdPie", "sdPie2", "sdArc", "sdTunnel", "sdCutDisk", "sdTrapezoid", "sdRhombus", "sdHeart",
          "sdRoundedX", "bigX", "sdRoundedCross", "sdOrientedVesica", "sdMoon", "sdUnevenCapsule", "Circle", "fallbackPolygon"]
PRE = [(0.0, 0.0, 0.0), (0.3, -0.2, 25.0)]
VARIANTS = ("glibc", "portable")
SCENES = {
    "c1": dict(shape="star", N=8, P=2000),
    "inside": dict(shape="star", N=8, P=400, clearance=2.35),
    "c3s": dict(shape="sdHorseshoe", N=16, P=1500),
}


def shapes_fixture():
    rng = np.random.default_rng(20240601)
    rel = np.c_[rng.uniform(-8.0, 8.0, (2000, 2)), rng.uniform(-1.0, 1.0, 2000)]
    # points ON lattice values / axes, where branches of the closed forms switch
    rel[:64, 0] = np.round(rel[:64, 0])
    rel[64:128, 1] = np.round(rel[64:128, 1])
    rel[128:160, 0] = 0.0
    rel[160:192, 1] = 0.0
    out = dict(rel=rel, shapes=np.array(SHAPES), pre=np.array(PRE), kernel_cfg=np.array([17, 18, 1.0, 0.0]))
    for v in VARIANTS:
        for ip, pp in enumerate(PRE):
            for s in SHAPES:
                out[f"sdf_{v}_{ip}_{s}"] = R.shape_sdf(s, rel, pp, variant=v)
                out[f"grad1_{v}_{ip}_{s}"] = R.shape_grad1(s, rel[:400], pp, variant=v)
        for s in SHAPES[:16]:  # initShape is what the registry shapes run in their constructors
            yaw, cells, byt = R.shape_kernels(s, 17, 18, 1.0, 0.0, variant=v)
            out[f"kyaw_{v}_{s}"] = yaw
            out[f"kbytes_{v}_{s}"] = byt
    save_fixture("ref_pin_shapes.npz", out)
    print("ref_pin_shapes.npz", len(out), "arrays")


def save_fixture(name, out):
    """Most shapes call no libm function, so both builds agree bit for bit: such a "portable" array is stored once, as "glibc"."""
    for k in [k for k in out if "_portable_" in k]:
        a, b = out[k], out[k.replace("_portable_", "_glibc_")]
        if a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes():
            del out[k]
    np.savez_compressed(os.path.join(HERE, name), **out)


def load_fixture(name):
    """A fixture written by save_fixture, with every "portable" array present again."""
    g = dict(np.load(os.path.join(HERE, name)))
    for k in [k for k in g if "_glibc_" in k]:
        g.setdefault(k.replace("_glibc_", "_portable_"), g[k])
    return g


def shapes_1e5_points():
    """The 1e5 body-frame points of the sampled shape test, two pre-transforms, and the seeded sample stored of them."""
    rng = np.random.default_rng(77)
    n = 100_000
    rel = np.c_[rng.uniform(-9.0, 9.0, (n, 2)), rng.uniform(-1.0, 1.0, n)]
    pick = np.random.default_rng(78)
    return rel, [(0.0, 0.0, 0.0), (-0.4, 0.15, -70.0)], np.sort(pick.choice(n, 512, replace=False)), np.sort(pick.choice(5000, 128, replace=False))


def scene_20k():
    return scenes.make_scene("star", 8, 20_000, seed_map=991)


def sample_fixture():
    """ref_pin_sample.npz: the reference's outputs at a seeded sample of larger inputs (shapes_1e5_points: getonlySDF on 512 of 1e5
    points, getonlyGrad1 on 128 of 5 000; scene_20k: getTrueSDFofSweptVolume<true> of the portable build on 2 000 of 20 000 points)."""
    rel, pres, si, gi = shapes_1e5_points()
    out = {}
    for v in VARIANTS:
        for ip, pp in enumerate(pres):
            for s in SHAPES:
                out[f"sdf_{v}_{ip}_{s}"] = R.shape_sdf(s, rel[si], pp, variant=v)
        for s in SHAPES:
            out[f"grad1_{v}_{s}"] = R.shape_grad1(s, rel[:5000][gi], variant=v)
    sc = scene_20k()
    idx = np.sort(np.random.default_rng(992).choice(sc.P, 2000, replace=False))
    ref = R.RefPath("star", weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, threads=8, variant="portable")
    ref.set_traj(sc.T, sc.coeffs_colmajor())
    out["scene20k_idx"] = idx
    out["scene20k_sdf"], out["scene20k_tstar"], out["scene20k_grad"] = ref.query(np.c_[sc.points[idx, :2], np.zeros(len(idx))])
    save_fixture("ref_pin_sample.npz", out)


def path_fixture():
    out = {}
    rng = np.random.default_rng(20240602)
    xs = np.r_[np.linspace(-0.02, 0.03, 501), rng.uniform(-1.0, 2.0, 500)]
    tau = rng.uniform(-3.0, 3.0, 256)
    out["l1_x"] = xs
    out["tau"] = tau
    for v in VARIANTS:
        ret, f, df = R.smoothed_l1(xs, 0.01, variant=v)
        out[f"l1_ret_{v}"], out[f"l1_f_{v}"], out[f"l1_df_{v}"] = ret, f, df
        T = R.forward_T(tau, variant=v)
        out[f"fwdT_{v}"] = T
        out[f"bwdT_{v}"] = R.backward_T(T, variant=v)
    for key, kw in SCENES.items():
        sc = scenes.make_scene(**kw)
        co = sc.coeffs_colmajor()
        pts0 = np.c_[sc.points[:, :2], np.zeros(sc.P)]
        D = float(sc.T.sum())
        ts = np.r_[rng.uniform(-0.2, D + 0.2, 300), np.cumsum(sc.T), 0.0]
        out.update({f"{key}_shape": sc.shape, f"{key}_N": sc.N, f"{key}_T": sc.T, f"{key}_coeffs": co, f"{key}_points": sc.points,
                    f"{key}_init_s": sc.init_s, f"{key}_final_s": sc.final_s, f"{key}_q": sc.q, f"{key}_x0": sc.x0,
                    f"{key}_params": np.array([sc.weight_p, sc.safety_hor, sc.rho]), f"{key}_ts": ts})
        for v in VARIANTS:
            ref = R.RefPath(sc.shape, weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, threads=8, variant=v)
            ref.set_traj(sc.T, co)
            out[f"{key}_pos_{v}"] = np.array([ref.traj_pos(t) for t in ts])
            out[f"{key}_vel_{v}"] = np.array([ref.traj_vel(t) for t in ts])
            sdf, tstar, g = ref.query(pts0)
            out[f"{key}_sdf_{v}"], out[f"{key}_tstar_{v}"], out[f"{key}_grad_{v}"] = sdf, tstar, g
            so, to, go = ref.query_outer(pts0[:200])
            out[f"{key}_osdf_{v}"], out[f"{key}_otstar_{v}"], out[f"{key}_ograd_{v}"] = so, to, go
            ref.set_points(sc.points)
            cost, gT, gC = ref.cost_grad(sc.T, co)
            out[f"{key}_cost_{v}"], out[f"{key}_gradT_{v}"], out[f"{key}_gradC_{v}"] = cost, gT, gC
            ref.set_conditions(sc.init_s, sc.final_s, sc.N)
            f, gg = ref.evaluate(sc.x0)
            out[f"{key}_f_{v}"], out[f"{key}_g_{v}"] = f, gg
            out[f"{key}_costs3_{v}"] = ref.last_costs()
            b, e, gdC, gdT = ref.minco_forward(sc.q, sc.T)
            out[f"{key}_b_{v}"], out[f"{key}_energy_{v}"], out[f"{key}_gdC_{v}"], out[f"{key}_gdT_{v}"] = b, e, gdC, gdT
            gP, gTt = ref.minco_propagate(gdC, gdT)
            out[f"{key}_adjP_{v}"], out[f"{key}_adjT_{v}"] = gP, gTt
            print(key, v, "cost", cost, "f", f, "inside", int((sdf <= 0).sum()))
    np.savez_compressed(os.path.join(HERE, "ref_pin_path.npz"), **out)
    print("ref_pin_path.npz", len(out), "arrays")


if __name__ == "__main__":
    if not R.available("glibc"):
        R.build()
    shapes_fixture()
    path_fixture()
    sample_fixture()

"""Generate tests/golden/ref_scale_path.npz: the reference's swept-volume path with its `useScale` switch on.

    make -C oracle -f scale.mk ref_scaled && python tests/golden/make_scale_golden.py      (only where /root/reference exists)

oracle/_ref/libref_path_scaled_{glibc,portable}.so are the reference's own source (the same verbatim fragments as
libref_path_*.so) compiled with `useScale` redefined to true and getScale supplied from a spec (oracle/scale.mk);
"portable" redirects its sin/cos/atan2 to the pinned fdlibm algorithm that the CUDA kernels implement.

Cases (scene x scale spec; SPECS uses the svsdf_scale form x, y = (c, [(a, w, phi), ...])):
  star_<spec>       config-1-style star scene, N = 8, 600 points with a narrow corridor (interior points, so GSIP runs),
                    for every spec
  horseshoe_ref     sdHorseshoe, N = 8, 400 points, the reference's commented example
  polygon_ref       the Polygon fallback (unknown shape name), N = 8, 400 points, the reference's commented example
Per case and build: getTrueSDFofSweptVolume<true> per point (sdf, t*, gradient), the penalty loop (cost, gradT, gradC) and
costFunctionLmbmParallel (f, g) at x0.  The GSIP round count is not observable in the reference; it is stored from the
oracle (rounds_<case>), whose per-point outputs equal the reference's bit for bit.  The reference has no exact-yaw mode:
exact_<case>_* are the oracle's (default build) penalty and callback with exact_yaw_grad = 1.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from implicit_svsdf_planner_b200 import scenes  # noqa: E402
from oracle import scale_py as SP  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "ref_scale_path.npz")

SPECS = {
    # sw_manager.hpp:499-502 (commented): diag(0.8 + sin(1.5 t - 1.0) 0.6, sin(1.8 t) 0.4 + 0.8, 1)
    "ref": dict(x=(0.8, [(0.6, 1.5, -1.0)]), y=(0.8, [(0.4, 1.8, 0.0)])),
    "iso": dict(x=(0.7, [(0.2, 1.1, 0.3)]), y=(0.7, [(0.2, 1.1, 0.3)])),
    "aniso": dict(x=(1.3, [(0.5, 0.9, 0.2), (0.3, 2.7, -0.6)]), y=(0.45, [(0.15, 1.7, 1.0), (0.1, 3.1, 0.0)])),
}
SCENES = {
    "star": dict(shape="star", N=8, P=600, clearance=2.35),
    "horseshoe": dict(shape="sdHorseshoe", N=8, P=400, clearance=2.35),
    "polygon": dict(shape="fallbackPolygon", N=8, P=400, clearance=2.35),
}
CASES = [("star", s) for s in SPECS] + [("horseshoe", "ref"), ("polygon", "ref")]
VARIANTS = ("glibc", "portable")


def case_name(scene, spec):
    return f"{scene}_{spec}"


def spec_arrays(spec):
    """(n[2], c[2], a[2][4], w[2][4], phi[2][4]) of a spec."""
    n, c = np.zeros(2, np.int32), np.ones(2)
    a, w, phi = np.zeros((2, 4)), np.zeros((2, 4)), np.zeros((2, 4))
    for ax, key in enumerate("xy"):
        c[ax] = spec[key][0]
        n[ax] = len(spec[key][1])
        for k, (ak, wk, pk) in enumerate(spec[key][1]):
            a[ax, k], w[ax, k], phi[ax, k] = ak, wk, pk
    return n, c, a, w, phi


def spec_from_arrays(n, c, a, w, phi):
    return {key: (float(c[ax]), [(float(a[ax, k]), float(w[ax, k]), float(phi[ax, k])) for k in range(int(n[ax]))])
            for ax, key in enumerate("xy")}


def main():
    out = {"cases": np.array([case_name(*c) for c in CASES])}
    for key, kw in SCENES.items():
        sc = scenes.make_scene(**kw)
        out.update({f"{key}_shape": sc.shape, f"{key}_N": sc.N, f"{key}_T": sc.T, f"{key}_coeffs": sc.coeffs_colmajor(),
                    f"{key}_points": sc.points, f"{key}_init_s": sc.init_s, f"{key}_final_s": sc.final_s, f"{key}_x0": sc.x0,
                    f"{key}_params": np.array([sc.weight_p, sc.safety_hor, sc.rho])})
    for sname, spec in SPECS.items():
        for k, v in zip(("n", "c", "a", "w", "phi"), spec_arrays(spec)):
            out[f"spec_{sname}_{k}"] = v
    for scene, spec in CASES:
        sc = scenes.make_scene(**SCENES[scene])
        co = sc.coeffs_colmajor()
        pts0 = np.c_[sc.points[:, :2], np.zeros(sc.P)]
        cn = case_name(scene, spec)
        for v in VARIANTS:
            ref = SP.scaled_ref(sc.shape, **SPECS[spec], weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, threads=8,
                                variant="scaled_" + v)
            ref.set_traj(sc.T, co)
            sdf, tstar, g = ref.query(pts0)
            out[f"{cn}_sdf_{v}"], out[f"{cn}_tstar_{v}"], out[f"{cn}_grad_{v}"] = sdf, tstar, g
            ref.set_threads(1)  # the penalty loop accumulates in point order
            ref.set_points(sc.points)
            cost, gT, gC = ref.cost_grad(sc.T, co)
            out[f"{cn}_cost_{v}"], out[f"{cn}_gradT_{v}"], out[f"{cn}_gradC_{v}"] = cost, gT, gC
            ref.set_conditions(sc.init_s, sc.final_s, sc.N)
            f, gg = ref.evaluate(sc.x0)
            out[f"{cn}_f_{v}"], out[f"{cn}_g_{v}"] = f, gg
            print(cn, v, "cost", cost, "f", f, "inside", int((sdf <= 0).sum()))
        orc = SP.ScaledOracle(sc.shape, **SPECS[spec], weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, threads=8)
        orc.set_traj(sc.T, co)
        out[f"rounds_{cn}"] = orc.query(pts0)[3]
        orc.set_threads(1)
        orc.set_scale(**SPECS[spec], exact_yaw_grad=True)
        orc.set_points(sc.points)
        cost, gT, gC = orc.cost_grad(sc.T, co)
        out[f"exact_{cn}_cost"], out[f"exact_{cn}_gradT"], out[f"exact_{cn}_gradC"] = cost, gT, gC
        orc.set_conditions(sc.init_s, sc.final_s, sc.N)
        out[f"exact_{cn}_f"], out[f"exact_{cn}_g"] = orc.evaluate(sc.x0)
    np.savez_compressed(OUT, **out)
    print(os.path.basename(OUT), len(out), "arrays")


def load():
    """The fixture as a dict, plus `specs` = {spec name: x/y spec}."""
    g = dict(np.load(OUT))
    g["specs"] = {s: spec_from_arrays(*(g[f"spec_{s}_{k}"] for k in ("n", "c", "a", "w", "phi"))) for s in SPECS}
    return g


if __name__ == "__main__":
    if not SP.ref_available():
        SP.build_ref()
    main()

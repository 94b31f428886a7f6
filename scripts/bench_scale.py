"""Cost of the body scale S(t) (svsdf_set_scale) on config 2: star, 8-piece MINCO, 200 000 query points.

    python scripts/bench_scale.py [--steps 30] [--warmup 3] [--out profiles/r3_scale_bench.json]

Three settings, alternated step by step in one process so that clocks and neighbours affect them alike:
  rigid      no spec (the shipped kernels)
  identity   a spec with S = I (the scaled kernels, same bits as rigid)
  reference  the reference's commented getScale example
Each step is one cost + gradient evaluation (svsdf_cost_grad_device, strict build, device-resident points) timed with CUDA
events; L2 is overwritten (320 MB memset, untimed) before every step.  Reports k_outer, k_compact + k_gsip and the step:
median, min and max over the steps, with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from implicit_svsdf_planner_b200 import api, scenes  # noqa: E402

SETTINGS = {
    "rigid": None,
    "identity": dict(x=(1.0, []), y=(1.0, [])),
    "reference": api.REFERENCE_SCALE_EXAMPLE,
}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, plim, smax = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=plim, sm_max_clock=smax)
    except Exception as e:  # the numbers are still device-timed; the card is then unnamed
        return dict(error=f"nvidia-smi: {e}")


def stats(v):
    v = np.asarray(v)
    return dict(median=float(np.median(v)), min=float(v.min()), max=float(v.max()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_scale_bench.json"))
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_scale: no CUDA device")
    sc = scenes.make_scene("star", 8, 200_000)
    co = sc.coeffs_colmajor()
    ctxs = {}
    for name, spec in SETTINGS.items():
        c = api.Context("star", weight_p=sc.weight_p, safety_hor=sc.safety_hor, rho=sc.rho, strict_fp=True)
        c.set_points(sc.points)
        if spec is not None:
            c.set_scale(**spec)
        ctxs[name] = c
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.float16, device="cuda:0")  # 320 MB > 126 MB L2
    for _ in range(a.warmup):
        for c in ctxs.values():
            c.cost_grad_device(sc.T, co, repeats=1, fetch=False)
    rec = {n: dict(step=[], k_outer=[], k_gsip=[]) for n in SETTINGS}
    out = {}
    for _ in range(a.steps):
        for name, c in ctxs.items():
            flush.zero_()
            torch.cuda.synchronize()
            ms, o = c.cost_grad_device(sc.T, co, repeats=1, fetch=True)
            km = c.last_kernel_ms()
            rec[name]["step"].append(ms)
            rec[name]["k_outer"].append(km[1])
            rec[name]["k_gsip"].append(km[2])
            out[name] = o
    res = {
        "what": "config 2 (star, 8-piece MINCO, 200 000 points), strict build, one cost+gradient evaluation per step; settings "
                "alternated step by step; L2 overwritten before each step; CUDA events; ms",
        "gpu": gpu_info(),
        "steps": a.steps,
        "warmup": a.warmup,
        "settings": {n: (None if s is None else {k: [v[0], [list(t) for t in v[1]]] for k, v in s.items()}) for n, s in SETTINGS.items()},
        "results": {n: {k: stats(v) for k, v in r.items()} for n, r in rec.items()},
        "n_inside": {n: int(o[-1]) for n, o in out.items()},
        "identity_equals_rigid_bitwise": bool(np.array_equal(out["identity"], out["rigid"])),
    }
    base = res["results"]["rigid"]
    res["ratio_to_rigid_median"] = {n: {k: r[k]["median"] / base[k]["median"] for k in r} for n, r in res["results"].items()}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))
    for c in ctxs.values():
        c.close()


if __name__ == "__main__":
    main()

"""Golden vectors for the mesh functor's winding number, from the REFERENCE's own code.

Runs in the build container only (needs /root/reference):  python tests/golden/make_fwn_golden.py
  1. `make -C oracle ref` compiles the reference's fast-winding-number implementation (the HDK UT_SolidAngle<float,float>
     behind igl::fast_winding_number; src/utils/include/igl/FastWindingNumberForSoups.h) from the source where it lies
     into oracle/_ref/libref_fwn.so (git-ignored), behind the shim oracle/ref_fwn_shim.cpp.
  2. The reference's shipped meshes src/plan_manager/shapes/{star,sdHorseshoe}.obj are read, the BVH is built exactly as
     BasicShape's constructor does (order 2, Shape.hpp:312) and queried exactly as getonlySDF_igl does (accuracy_scale 2.0,
     Shape.hpp:337) at seeded points in the z = 0 plane (where the planner queries) and in 3-D.
  3. Inputs (V, F, Q) and the reference's outputs (w_ref) go to tests/golden/fwn_ref.npz.
  4. The hierarchy the reference built is dumped too (oracle/ref_fwn_shim.cpp: ref_fwn_dump): the child words of every node
     and its 23 rows of expansion coefficients (tree_children, tree_data).
tests/test_oracle_mesh.py requires the repo's own host builder (csrc/host/fwn_bvh.hpp) to reproduce tree, coefficients and
w_ref BIT FOR BIT, and compares the exact double-precision winding number with w_ref (the reference's value is a float,
order-2 approximation: the observed difference, <= 2.1e-3, is its approximation error — the exact value is an integer to
1e-15 on these closed meshes).
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from implicit_svsdf_planner_b200 import scenes  # noqa: E402

REF_SHAPES = "/root/reference/src/plan_manager/shapes"


def ref_fwn(V, F, Q, order=2, accuracy=2.0):
    dp = C.POINTER(C.c_double)
    L = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_fwn.so"))
    L.ref_fwn_create.restype = C.c_void_p
    L.ref_fwn_create.argtypes = [dp, C.c_int, C.c_void_p, C.c_int, C.c_int]
    L.ref_fwn_eval.argtypes = [C.c_void_p, C.c_float, C.c_int64, dp, dp]
    L.ref_fwn_destroy.argtypes = [C.c_void_p]
    V = np.ascontiguousarray(V, dtype=np.float64)
    F = np.ascontiguousarray(F, dtype=np.int32)
    Q = np.ascontiguousarray(Q, dtype=np.float64)
    h = L.ref_fwn_create(V.ctypes.data_as(dp), V.shape[0], F.ctypes.data_as(C.c_void_p), F.shape[0], order)
    w = np.empty(Q.shape[0])
    L.ref_fwn_eval(h, accuracy, Q.shape[0], Q.ctypes.data_as(dp), w.ctypes.data_as(dp))
    L.ref_fwn_destroy(h)
    return w


def ref_fwn_tree(V, F, order=2):
    """(children [nn, 4] uint32, data [nn, 23, 4] float32) of the hierarchy the reference builds."""
    dp = C.POINTER(C.c_double)
    L = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_fwn.so"))
    L.ref_fwn_create.restype = C.c_void_p
    L.ref_fwn_create.argtypes = [dp, C.c_int, C.c_void_p, C.c_int, C.c_int]
    L.ref_fwn_num_nodes.argtypes = [C.c_void_p]
    L.ref_fwn_dump.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.ref_fwn_destroy.argtypes = [C.c_void_p]
    V = np.ascontiguousarray(V, dtype=np.float64)
    F = np.ascontiguousarray(F, dtype=np.int32)
    h = L.ref_fwn_create(V.ctypes.data_as(dp), V.shape[0], F.ctypes.data_as(C.c_void_p), F.shape[0], order)
    nn = L.ref_fwn_num_nodes(h)
    ch = np.zeros((nn, 4), np.uint32)
    data = np.zeros((nn, 23, 4), np.float32)
    L.ref_fwn_dump(h, ch.ctypes.data_as(C.c_void_p), data.ctypes.data_as(C.c_void_p))
    L.ref_fwn_destroy(h)
    return ch, data


BRANCH_MESHES = ["synthetic_star", "two_faces", "seven_faces", "grid_900", "degenerate_duplicates"]


def branch_case(mesh):
    """(V, F, Q) of a mesh that exercises one branch of the hierarchy builder: 2 items, the exhaustive <= 6 split, the sorted
    <= 32 split, the 16-span binning, coincident centres (nthElement fallback)."""
    rng = np.random.default_rng(9)
    if mesh == "synthetic_star":
        V, F = scenes.extrude_outline(scenes.star_outline(n_per_edge=4))
    elif mesh in ("two_faces", "seven_faces"):
        nf = 2 if mesh == "two_faces" else 7
        V = rng.uniform(-2, 2, size=(3 * nf, 3))
        F = np.arange(3 * nf, dtype=np.int32).reshape(nf, 3)
    elif mesh == "grid_900":
        n = 16
        xs, ys = np.meshgrid(np.linspace(-3, 3, n), np.linspace(-2, 2, n))
        V = np.c_[xs.ravel(), ys.ravel(), 0.3 * np.sin(xs.ravel() * 2.0) * np.cos(ys.ravel())]
        F = []
        for i in range(n - 1):
            for j in range(n - 1):
                a = i * n + j
                F += [[a, a + 1, a + n + 1], [a, a + n + 1, a + n]]
        F = np.asarray(F, dtype=np.int32)
    else:  # many faces sharing one centre: the span partition cannot split them
        base = rng.uniform(-1, 1, size=(3, 3))
        V = np.concatenate([base * (1.0 + 0.0 * k) for k in range(40)] + [rng.uniform(-2, 2, size=(30, 3))])
        F = np.arange(len(V), dtype=np.int32).reshape(-1, 3)
    lo, hi = V.min(axis=0) - 1.5, V.max(axis=0) + 1.5
    Q = np.zeros((3000, 3))
    Q[:, :2] = rng.uniform(lo[:2], hi[:2], size=(3000, 2))
    Q[1500:] = rng.uniform(lo, hi, size=(1500, 3))
    return V, F, Q


def branch_fixture():
    """fwn_ref_branches.npz: the reference's winding numbers and hierarchy for the meshes of branch_case."""
    out = {}
    for mesh in BRANCH_MESHES:
        V, F, Q = branch_case(mesh)
        out[mesh + "_w_ref"] = ref_fwn(V, F, Q)
        out[mesh + "_tree_children"], out[mesh + "_tree_data"] = ref_fwn_tree(V, F)
    np.savez_compressed(os.path.join(HERE, "fwn_ref_branches.npz"), **out)


def main():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"])
    rng = np.random.Generator(np.random.MT19937(20240511))
    out = {}
    for name in ("star", "sdHorseshoe"):
        V, F = scenes.load_obj(os.path.join(REF_SHAPES, name + ".obj"))
        lo, hi = V.min(axis=0) - 1.5, V.max(axis=0) + 1.5
        Q = np.zeros((3000, 3))
        Q[:2000, :2] = rng.uniform(lo[:2], hi[:2], size=(2000, 2))  # the plane the planner queries
        Q[2000:] = rng.uniform(lo, hi, size=(1000, 3))
        out[name + "_V"], out[name + "_F"], out[name + "_Q"] = V, F, Q
        out[name + "_w_ref"] = ref_fwn(V, F, Q)
        out[name + "_tree_children"], out[name + "_tree_data"] = ref_fwn_tree(V, F)
    np.savez_compressed(os.path.join(HERE, "fwn_ref.npz"), **out)
    # a deeper hierarchy (973 nodes over 2000 faces): shapes/sdArc.obj, own file and own stream so that fwn_ref.npz stays as it was
    rng2 = np.random.Generator(np.random.MT19937(20240512))
    V, F = scenes.load_obj(os.path.join(REF_SHAPES, "sdArc.obj"))
    lo, hi = V.min(axis=0) - 1.5, V.max(axis=0) + 1.5
    Q = np.zeros((3000, 3))
    Q[:2000, :2] = rng2.uniform(lo[:2], hi[:2], size=(2000, 2))
    Q[2000:] = rng2.uniform(lo, hi, size=(1000, 3))
    np.savez_compressed(os.path.join(HERE, "fwn_ref_sdarc.npz"), sdArc_V=V, sdArc_F=F, sdArc_Q=Q, sdArc_w_ref=ref_fwn(V, F, Q),
                        sdArc_tree_children=ref_fwn_tree(V, F)[0])
    branch_fixture()
    for k, v in out.items():
        print(k, v.shape, v.dtype)


if __name__ == "__main__":
    main()

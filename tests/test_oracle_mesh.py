"""CPU tests of the triangle-mesh functor (BasicShape::getonlySDF_igl, Shape.hpp:332-340): the oracle's restatement, the host
builder of the winding-number hierarchy (csrc/host/fwn_bvh.hpp, through the C ABI) and the host-side .obj reader.  Pins:
closed-form answers on a cube, the 2-D polygon SDF of the extruded outline, and the reference's OWN fast-winding-number code
(compiled from /root/reference into oracle/_ref; tree, coefficients and outputs committed in tests/golden/fwn_ref.npz) —
hierarchy and winding numbers BIT FOR BIT."""
import os

import numpy as np
import pytest

from implicit_svsdf_planner_b200 import api, scenes

HERE = os.path.dirname(os.path.abspath(__file__))


def cube(h=1.0):
    V = np.array([[x, y, z] for x in (-h, h) for y in (-h, h) for z in (-h, h)], dtype=np.float64)
    # outward-oriented faces of the cube (vertex index = 4*ix + 2*iy + iz)
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    F = []
    for a, b, c, d in quads:
        F += [[a, b, c], [a, c, d]]
    return V, np.asarray(F, dtype=np.int32)


def test_cube_known_answers(oracle_mod):
    m = cube(1.0)
    Q = np.array([[0, 0, 0], [0.5, 0.2, 0], [2.0, 0, 0], [2.0, 2.0, 0], [0, -3.0, 0], [2.0, 2.0, 2.0], [0.25, 0, 0.9]], dtype=np.float64)
    w = oracle_mod.mesh_eval(m, Q, "winding_exact")
    assert np.allclose(w, [1, 1, 0, 0, 0, 0, 1], atol=1e-14)
    d2 = oracle_mod.mesh_eval(m, Q, "sqr_distance")
    assert np.allclose(d2, [1.0, 0.25, 1.0, 2.0, 4.0, 3.0, 0.01], atol=1e-14)
    sdf = oracle_mod.mesh_eval(m, Q, "sdf_exact")
    assert np.allclose(sdf, [-1.0, -0.5, 1.0, np.sqrt(2.0), 2.0, np.sqrt(3.0), -0.1], atol=1e-13)
    # orientation matters: the inward-oriented cube has winding number -1 inside -> (1 - 2w) = 3 (the reference's formula)
    m_in = (m[0], m[1][:, ::-1].copy())
    assert np.allclose(oracle_mod.mesh_eval(m_in, Q[:1], "winding_exact"), [-1.0], atol=1e-14)
    # what the reference computes instead: the float order-2 hierarchy — the same numbers to its approximation error
    wf = oracle_mod.mesh_eval(m, Q, "winding")
    assert np.abs(wf - w).max() < 2e-3 and np.abs(wf - w).max() > 0.0
    assert np.allclose(oracle_mod.mesh_eval(m, Q, "sdf"), (1.0 - 2.0 * wf) * np.sqrt(d2), rtol=0, atol=0)


def test_extruded_outline_matches_the_polygon_sdf_in_the_mid_plane(oracle_mod):
    outline = scenes.star_outline(n_per_edge=3)
    m = scenes.extrude_outline(outline, half_height=0.49)
    rng = np.random.default_rng(5)
    Q = np.c_[rng.uniform(-4, 4, size=(4000, 2)), np.zeros(4000)]
    sd = oracle_mod.mesh_eval(m, Q, "sdf_exact")
    poly = oracle_mod.shape_sdf("custom_poly", Q, polygon=outline)
    out = poly > 0
    assert np.abs(sd - poly)[out].max() < 1e-13           # outside: the in-plane distance
    assert (np.sign(sd) == np.sign(poly)).all()
    assert np.allclose(sd[~out], np.maximum(poly[~out], -0.49), atol=1e-13)  # inside: saturates at the caps
    w = oracle_mod.mesh_eval(m, Q, "winding_exact")
    assert np.abs(w - np.round(w)).max() < 1e-13          # closed mesh: integer winding number
    # the reference's functor (float hierarchy): same sign away from the surface, distance scaled by (1 - 2 w) with |w - w_exact| < 5e-3
    sdf = oracle_mod.mesh_eval(m, Q, "sdf")
    far = np.abs(poly) > 1e-3
    assert (np.sign(sdf) == np.sign(poly))[far].all()
    assert np.abs(sdf - sd).max() <= 1e-2 * np.abs(sd).max()
    # FD gradient (Shape.hpp:35-53): close to unit length away from creases (the float winding number adds O(1e-4 / eps) noise to
    # a central difference: this is the reference's behaviour), zero z component
    g = oracle_mod.mesh_eval(m, Q[out][:500], "grad1")
    nrm = np.linalg.norm(g[:, :2], axis=1)
    assert np.isfinite(g).all() and np.all(g[:, 2] == 0.0)
    assert (np.abs(nrm - 1.0) < 0.2).mean() > 0.9


def test_poly_params_move_the_mesh_vertices(oracle_mod):
    """BasicShape's constructor applies poly_params to the vertices (R v + trans, Shape.hpp:285-302): the level set moves
    WITH the transform (unlike the analytic functors, which transform the query)."""
    outline = scenes.star_outline()
    m = scenes.extrude_outline(outline)
    pp = (0.6, -0.3, 25.0)
    th = np.deg2rad(pp[2])
    R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    rng = np.random.default_rng(6)
    Q = np.c_[rng.uniform(-4, 4, size=(500, 2)), np.zeros(500)]
    Qb = Q.copy()
    Qb[:, :2] = (Q[:, :2] - np.array(pp[:2])) @ R  # R^T (q - trans)
    a = oracle_mod.mesh_eval(m, Q, "sdf_exact", poly_params=pp)
    b = oracle_mod.mesh_eval(m, Qb, "sdf_exact")
    assert np.abs(a - b).max() < 1e-12
    # the float hierarchy is rebuilt over the moved vertices: a different tree, the same numbers to its approximation error
    af = oracle_mod.mesh_eval(m, Q, "sdf", poly_params=pp)
    assert np.abs(af - a).max() <= 1e-2 * np.abs(a).max()


def test_portable_atan2f_is_the_c_library_atan2f(oracle_mod):
    """The winding-number leaves call atan2f; host and device use the pinned fdlibm code instead of their libraries'.  It must
    equal the C library the reference links (glibc) bit for bit, or the w parity below would be luck."""
    rng = np.random.default_rng(11)
    n = 4_000_000
    y = rng.standard_normal(n).astype(np.float32)
    x = rng.standard_normal(n).astype(np.float32)
    # wide dynamic range, exact axes, signed zeros, tiny and huge ratios
    scale = np.exp2(rng.integers(-60, 60, size=n)).astype(np.float32)
    y[: n // 2] *= scale[: n // 2]
    x[n // 4: n // 2] /= scale[n // 4: n // 2]
    sp = np.array([0.0, -0.0, 1.0, -1.0, 1e-30, -1e-30, 1e30, -1e30, 3.0e7, 3.4e7, 0.4375, 0.6875, 1.1875, 2.4375], dtype=np.float32)
    yy, xx = np.meshgrid(sp, sp)
    y = np.concatenate([y, yy.ravel()])
    x = np.concatenate([x, xx.ravel()])
    a, b = oracle_mod.atan2f_pair(y, x)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _fwn_gold(name):
    g = np.load(os.path.join(HERE, "golden", "fwn_ref_sdarc.npz" if name == "sdArc" else "fwn_ref.npz"))
    return g


def test_deep_hierarchy_sdarc_2000_faces(oracle_mod):
    """shapes/sdArc.obj: 2000 faces, 973 nodes — tree and winding numbers of the reference's compiled code, bit for bit."""
    g = _fwn_gold("sdArc")
    ch, data, w = api.mesh_fwn_host(g["sdArc_V"], g["sdArc_F"], g["sdArc_Q"])
    assert np.array_equal(ch, g["sdArc_tree_children"]) and np.array_equal(w, g["sdArc_w_ref"])
    assert np.array_equal(oracle_mod.mesh_eval((g["sdArc_V"], g["sdArc_F"]), g["sdArc_Q"][:500], "winding"), g["sdArc_w_ref"][:500])


@pytest.mark.parametrize("name", ["star", "sdHorseshoe"])
def test_winding_number_is_bitwise_the_reference_fwn_golden(oracle_mod, name):
    """w_ref, tree_children, tree_data were produced by the reference's own igl/HDK code on its own shapes/*.obj
    (tests/golden/make_fwn_golden.py).  The repo's host builder must reproduce the hierarchy node by node and coefficient by
    coefficient, and both its traversal (through the C ABI) and the oracle's functor must return w_ref BIT FOR BIT.  The exact
    double-precision sum differs from it by the reference's approximation error (2.1e-3 at worst)."""
    g = np.load(os.path.join(HERE, "golden", "fwn_ref.npz"))
    m = (g[name + "_V"], g[name + "_F"])
    Q, w_ref = g[name + "_Q"], g[name + "_w_ref"]
    ch, data, w_host = api.mesh_fwn_host(m[0], m[1], Q)
    assert np.array_equal(ch, g[name + "_tree_children"])
    assert np.array_equal(data.view(np.uint32), g[name + "_tree_data"].view(np.uint32))
    assert np.array_equal(w_host, w_ref)
    w = oracle_mod.mesh_eval(m, Q, "winding")
    assert np.array_equal(w, w_ref)
    we = oracle_mod.mesh_eval(m, Q, "winding_exact")
    assert np.abs(we - np.round(we)).max() < 1e-13
    d2 = oracle_mod.mesh_eval(m, Q, "sqr_distance")
    far = d2 > 1e-4  # on the surface the winding number jumps; float vs double vertices decide the side
    assert np.abs(we - w_ref)[far].max() < 5e-3, np.abs(we - w_ref)[far].max()
    assert np.array_equal(np.round(w_ref[far]), np.round(we[far]))
    # getonlySDF_igl = (1 - 2 w) sqrt(d2) exactly as the reference evaluates it
    sdf = oracle_mod.mesh_eval(m, Q, "sdf")
    assert np.array_equal(sdf, (1.0 - 2.0 * w_ref) * np.sqrt(d2))
    assert np.abs(sdf - oracle_mod.mesh_eval(m, Q, "sdf_exact"))[far].max() <= 1.0e-2 * np.abs(sdf[far]).max()


@pytest.mark.parametrize("mesh", ["synthetic_star", "two_faces", "seven_faces", "grid_900", "degenerate_duplicates"])
def test_reference_fwn_live_tree_coefficients_and_values(oracle_mod, mesh):
    """Against what the reference's compiled code computes (tests/golden/fwn_ref_branches.npz, make_fwn_golden.branch_fixture)
    on meshes that exercise every branch of the builder: 2 items, the exhaustive <= 6 split, the sorted <= 32 split, the
    16-span binning, coincident centres (nthElement fallback)."""
    import sys

    sys.path.insert(0, os.path.join(HERE, "golden"))
    import make_fwn_golden as mk

    V, F, Q = mk.branch_case(mesh)
    g = np.load(os.path.join(HERE, "golden", "fwn_ref_branches.npz"))
    w_ref, rc, rd = g[mesh + "_w_ref"], g[mesh + "_tree_children"], g[mesh + "_tree_data"]
    ch, data, w_host = api.mesh_fwn_host(V, F, Q)
    assert np.array_equal(ch, rc)
    assert np.array_equal(data.view(np.uint32), rd.view(np.uint32))
    assert np.array_equal(w_host, w_ref)
    assert np.array_equal(oracle_mod.mesh_eval((V, F), Q, "winding"), w_ref)


def test_obj_reader_host(tmp_path):
    p = tmp_path / "m.obj"
    p.write_text("# comment\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nv 0.5 0.5 1\n"
                 "vn 0 0 1\nf 1 2 3 4\nf 1/1/1 2/2/1 5/3/1\nf -4//1 -3//1 -1//1\n")
    V, F = api.read_obj(str(p))
    V2, F2 = scenes.load_obj(str(p))
    assert np.array_equal(V, V2) and np.array_equal(F, F2)
    assert V.shape == (5, 3) and F.tolist() == [[0, 1, 2], [0, 2, 3], [0, 1, 4], [1, 2, 4]]
    with pytest.raises(api.SvsdfError):
        api.read_obj(str(tmp_path / "missing.obj"))
    bad = tmp_path / "bad.obj"
    bad.write_text("v 0 0 0\nf 1 2 3\n")
    with pytest.raises(api.SvsdfError):
        api.read_obj(str(bad))

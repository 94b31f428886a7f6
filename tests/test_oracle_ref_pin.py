"""The oracle (oracle/*.hpp, the hand-written restatement every GPU parity test is checked against) is PINNED HERE to the
reference's own source, compiled where it lies into oracle/_ref/libref_path_*.so (oracle/ref_path_shim.cpp).

Two layers:
  * fixture tests (always run, also on machines without /root/reference): tests/golden/ref_pin_*.npz hold the outputs of
    the reference's code (tests/golden/make_ref_pin_golden.py); the oracle must reproduce every per-point quantity BIT FOR
    BIT — shape values and FD gradients for all 18 functors, initShape byte kernels, Piece<5>/Trajectory<5> samples,
    getTrueSDFofSweptVolume (sdf, t*, gradient; outside and GSIP points), smoothedL1, tau<->T — and every summed quantity
    (cost, gradC, gradT, f, g, MINCO) to summation-order rounding;
  * 1e5 random points per shape against a seeded sample of the reference's values (ref_pin_sample.npz);
  * live tests (when the .so files are present, i.e. where the reference was compiled): the fixtures are what the reference
    produces, and the proof that the one arithmetic freedom of the Eigen stand-in (association order of reductions) cannot move any pinned
    per-point output: three builds with three orders agree bit for bit.
Variant mapping: reference "glibc" <-> oracle "glibc"; reference "portable" (its libm calls redirected to the pinned
fdlibm sin/cos/atan2) <-> oracle "default" (the variant the CUDA kernels are bit-identical to).
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
sys.path.insert(0, GOLD)
import make_ref_pin_golden as mk  # noqa: E402  (fixture loader; its reference calls are not used here)
PAIRS = [("glibc", "glibc"), ("portable", "default")]  # (reference variant, oracle variant)


def bits_differ(a, b):
    a = np.ascontiguousarray(a, dtype=np.float64).ravel()
    b = np.ascontiguousarray(b, dtype=np.float64).ravel()
    assert a.shape == b.shape
    return int((a.view(np.int64) != b.view(np.int64)).sum())


@pytest.fixture(scope="module")
def gshapes():
    return mk.load_fixture("ref_pin_shapes.npz")


@pytest.fixture(scope="module")
def gpath():
    return np.load(os.path.join(GOLD, "ref_pin_path.npz"))


def _orc_shape(O, variant, name, rel, pp, what):
    import ctypes as C

    L = O.lib(variant)
    rel = np.ascontiguousarray(rel, dtype=np.float64)
    ppa = np.asarray(pp, dtype=np.float64)
    n = rel.shape[0]
    if what == "sdf":
        out = np.empty(n)
        L.orc_shape_sdf(name.encode(), O._p(ppa), None, 0, n, O._p(rel), O._p(out))
    else:
        out = np.empty((n, 3))
        L.orc_shape_grad1(name.encode(), O._p(ppa), None, 0, n, O._p(rel), O._p(out))
    return out


def _orc_kernels(O, variant, name, ks, K, res, safeh):
    import ctypes as C

    L = O.lib(variant)
    yaw = np.empty(K)
    cells = np.zeros((K, ks, ks), np.uint8)
    byt = np.zeros((K, ks, (ks + 7) // 8), np.uint8)
    pp = np.zeros(3)
    u8 = C.POINTER(C.c_uint8)
    L.orc_shape_kernels(name.encode(), O._p(pp), ks, K, res, safeh, O._p(yaw), cells.ctypes.data_as(u8), byt.ctypes.data_as(u8))
    return yaw, cells, byt


# ---------------------------------------------------------------------------------------------------------------------
# fixtures: reference outputs committed under tests/golden
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rv,ov", PAIRS)
def test_shape_functors_match_reference_code_bitwise(oracle_mod, gshapes, rv, ov):
    rel = gshapes["rel"]
    for ip, pp in enumerate(gshapes["pre"]):
        for s in gshapes["shapes"]:
            s = str(s)
            assert bits_differ(_orc_shape(oracle_mod, ov, s, rel, pp, "sdf"), gshapes[f"sdf_{rv}_{ip}_{s}"]) == 0, (s, ip)
            assert bits_differ(_orc_shape(oracle_mod, ov, s, rel[:400], pp, "grad"), gshapes[f"grad1_{rv}_{ip}_{s}"]) == 0, (s, ip)


@pytest.mark.parametrize("rv,ov", PAIRS)
def test_init_shape_kernels_match_reference_code(oracle_mod, gshapes, rv, ov):
    ks, K, res, safeh = gshapes["kernel_cfg"]
    for s in gshapes["shapes"][:16]:
        s = str(s)
        yaw, _, byt = _orc_kernels(oracle_mod, ov, s, int(ks), int(K), float(res), float(safeh))
        assert bits_differ(yaw, gshapes[f"kyaw_{rv}_{s}"]) == 0
        assert np.array_equal(byt, gshapes[f"kbytes_{rv}_{s}"]), s


@pytest.mark.parametrize("rv,ov", PAIRS)
def test_scalar_maps_match_reference_code_bitwise(oracle_mod, gpath, rv, ov):
    import ctypes as C

    L = oracle_mod.lib(ov)
    tau = np.ascontiguousarray(gpath["tau"])
    T = np.empty_like(tau)
    L.orc_forward_T(tau.size, oracle_mod._p(tau), oracle_mod._p(T))
    assert bits_differ(T, gpath[f"fwdT_{rv}"]) == 0
    back = np.empty_like(tau)
    L.orc_backward_T(T.size, oracle_mod._p(T), oracle_mod._p(back))
    assert bits_differ(back, gpath[f"bwdT_{rv}"]) == 0
    if hasattr(L, "orc_smoothed_l1"):
        x = np.ascontiguousarray(gpath["l1_x"])
        f, df = np.empty_like(x), np.empty_like(x)
        ret = np.zeros(x.size, np.uint8)
        L.orc_smoothed_l1.argtypes = [C.c_int64, oracle_mod.dp, C.c_double, oracle_mod.dp, oracle_mod.dp, C.POINTER(C.c_uint8)]
        L.orc_smoothed_l1(x.size, oracle_mod._p(x), 0.01, oracle_mod._p(f), oracle_mod._p(df), ret.ctypes.data_as(C.POINTER(C.c_uint8)))
        m = gpath[f"l1_ret_{rv}"]
        assert np.array_equal(ret.astype(bool), m)
        assert bits_differ(f[m], gpath[f"l1_f_{rv}"][m]) == 0 and bits_differ(df[m], gpath[f"l1_df_{rv}"][m]) == 0


@pytest.mark.parametrize("key", ["c1", "inside", "c3s"])
@pytest.mark.parametrize("rv,ov", PAIRS)
def test_path_matches_reference_code(oracle_mod, gpath, key, rv, ov):
    g = gpath
    shape, N = str(g[f"{key}_shape"]), int(g[f"{key}_N"])
    T, co, pts = g[f"{key}_T"], g[f"{key}_coeffs"], g[f"{key}_points"]
    wp, sh, rho = g[f"{key}_params"]
    orc = oracle_mod.Oracle(shape, weight_p=wp, safety_hor=sh, rho=rho, threads=min(8, oracle_mod.num_procs()), variant=ov)
    orc.set_traj(T, co)
    # A1: Piece<5>::getPos/getVel + locatePieceIdx (incl. t < 0, t > D, t exactly on the junctions)
    ts = g[f"{key}_ts"]
    assert bits_differ(np.array([orc.traj_pos(t) for t in ts]), g[f"{key}_pos_{rv}"]) == 0
    assert bits_differ(np.array([orc.traj_vel(t) for t in ts]), g[f"{key}_vel_{rv}"]) == 0
    # A2-A7: the per-point query API, outside and interior (GSIP) points alike
    pts0 = np.c_[pts[:, :2], np.zeros(len(pts))]
    sdf, tstar, grad, _ = orc.query(pts0)
    assert bits_differ(sdf, g[f"{key}_sdf_{rv}"]) == 0
    assert bits_differ(tstar, g[f"{key}_tstar_{rv}"]) == 0
    assert bits_differ(grad, g[f"{key}_grad_{rv}"]) == 0
    if key == "inside":
        assert int((sdf <= 0).sum()) >= 20  # the GSIP branch is really exercised
    so, to, go = orc.query_outer(pts0[:200])
    assert bits_differ(so, g[f"{key}_osdf_{rv}"]) + bits_differ(to, g[f"{key}_otstar_{rv}"]) + bits_differ(go, g[f"{key}_ograd_{rv}"]) == 0
    # A8: penalty, chain rule, reduction — sums: equal up to the association order of the additions
    orc.set_points(pts)
    cost, gT, gC, _, _ = orc.cost_grad(T, co)
    rc, rT, rC = float(g[f"{key}_cost_{rv}"]), g[f"{key}_gradT_{rv}"], g[f"{key}_gradC_{rv}"]
    assert abs(cost - rc) <= 1e-13 * abs(rc)
    assert np.linalg.norm(gC - rC) <= 1e-13 * np.linalg.norm(rC)
    # gradT sums -G.vel over points; at an interior minimum of t -> sdf that product is ~0 by optimality (heavy
    # cancellation), so it is compared on the scale of its terms, |gradC| * |vel| ~ |gradC|
    assert np.abs(gT - rT).max() <= 1e-12 * np.linalg.norm(rC)
    # A10: MINCO_S3NU + tau maps + the whole callback
    orc.set_conditions(g[f"{key}_init_s"], g[f"{key}_final_s"], N)
    f, gg = orc.evaluate(g[f"{key}_x0"])
    rf, rg = float(g[f"{key}_f_{rv}"]), g[f"{key}_g_{rv}"]
    assert abs(f - rf) <= 1e-13 * abs(rf)
    assert np.linalg.norm(gg - rg) <= 1e-12 * np.linalg.norm(rg)
    b, e, gdC, gdT = oracle_mod.minco_forward(g[f"{key}_init_s"], g[f"{key}_final_s"], g[f"{key}_q"], T)
    rb = g[f"{key}_b_{rv}"]
    assert np.linalg.norm(np.asarray(b).T.reshape(-1) - rb) <= 1e-13 * np.linalg.norm(rb)
    assert abs(e - float(g[f"{key}_energy_{rv}"])) <= 1e-13 * abs(e)
    assert np.linalg.norm(np.asarray(gdC).T.reshape(-1) - g[f"{key}_gdC_{rv}"]) <= 1e-13 * np.linalg.norm(g[f"{key}_gdC_{rv}"])
    assert np.linalg.norm(np.asarray(gdT) - g[f"{key}_gdT_{rv}"]) <= 1e-13 * np.linalg.norm(g[f"{key}_gdT_{rv}"])
    gq, gt = oracle_mod.minco_propagate(g[f"{key}_init_s"], g[f"{key}_final_s"], g[f"{key}_q"], T, g[f"{key}_gdC_{rv}"].reshape(3, 6 * N).T, g[f"{key}_gdT_{rv}"])
    assert np.linalg.norm(np.asarray(gq) - g[f"{key}_adjP_{rv}"]) <= 1e-12 * np.linalg.norm(g[f"{key}_adjP_{rv}"])
    assert np.linalg.norm(np.asarray(gt) - g[f"{key}_adjT_{rv}"]) <= 1e-12 * np.linalg.norm(g[f"{key}_adjT_{rv}"])


# ---------------------------------------------------------------------------------------------------------------------
# live: the reference libraries themselves (present in this container and, as built .so files, on the GPU box)
# ---------------------------------------------------------------------------------------------------------------------
def _ref():
    from oracle import ref_py

    if not all(ref_py.available(v) for v in ref_py.VARIANTS):
        pytest.skip("oracle/_ref/libref_path_*.so not built (needs /root/reference: make -C oracle ref_path)")
    return ref_py


@pytest.mark.parametrize("rv,ov", PAIRS)
def test_live_shapes_1e5_points_bitwise(oracle_mod, gshapes, rv, ov):
    """1e5 fresh random points per shape; a seeded sample of them is compared with the reference's values there
    (ref_pin_sample.npz)."""
    g = mk.load_fixture("ref_pin_sample.npz")
    rel, pres, si, gi = mk.shapes_1e5_points()
    for ip, pp in enumerate(pres):
        for s in gshapes["shapes"]:
            s = str(s)
            assert bits_differ(_orc_shape(oracle_mod, ov, s, rel, pp, "sdf")[si], g[f"sdf_{rv}_{ip}_{s}"]) == 0, (s, pp)
    for s in gshapes["shapes"]:
        s = str(s)
        assert bits_differ(_orc_shape(oracle_mod, ov, s, rel[:5000], (0.0, 0.0, 0.0), "grad")[gi], g[f"grad1_{rv}_{s}"]) == 0, s


def test_live_fixture_is_what_the_reference_code_produces(gpath, gshapes):
    """The committed fixtures are reproducible from the reference libraries (guards against a stale fixture)."""
    R = _ref()
    for rv in ("glibc", "portable"):
        assert bits_differ(R.shape_sdf("star", gshapes["rel"], variant=rv), gshapes[f"sdf_{rv}_0_star"]) == 0
        key = "inside"
        ref = R.RefPath(str(gpath[f"{key}_shape"]), threads=8, variant=rv, weight_p=gpath[f"{key}_params"][0],
                        safety_hor=gpath[f"{key}_params"][1], rho=gpath[f"{key}_params"][2])
        ref.set_traj(gpath[f"{key}_T"], gpath[f"{key}_coeffs"])
        pts = gpath[f"{key}_points"]
        sdf, tstar, grad = ref.query(np.c_[pts[:, :2], np.zeros(len(pts))])
        assert bits_differ(sdf, gpath[f"{key}_sdf_{rv}"]) + bits_differ(tstar, gpath[f"{key}_tstar_{rv}"]) + bits_differ(grad, gpath[f"{key}_grad_{rv}"]) == 0


def test_live_reduction_order_of_the_eigen_stand_in_does_not_move_pinned_outputs(gpath):
    """oracle/ref_shim/Eigen has ONE arithmetic freedom: how an n-term reduction is associated.  Three builds (recursive
    halving, left-to-right, two-lane) give identical per-point outputs; only the summed outputs move, by rounding."""
    R = _ref()
    key = "inside"
    pts = gpath[f"{key}_points"]
    pts0 = np.c_[pts[:, :2], np.zeros(len(pts))]
    res = {}
    for v in ("glibc", "glibc_r1", "glibc_r2"):
        ref = R.RefPath(str(gpath[f"{key}_shape"]), threads=8, variant=v, weight_p=gpath[f"{key}_params"][0],
                        safety_hor=gpath[f"{key}_params"][1], rho=gpath[f"{key}_params"][2])
        ref.set_traj(gpath[f"{key}_T"], gpath[f"{key}_coeffs"])
        q = ref.query(pts0)
        ref.set_points(pts)
        cg = ref.cost_grad(gpath[f"{key}_T"], gpath[f"{key}_coeffs"])
        ts = gpath[f"{key}_ts"]
        tr = np.array([np.r_[ref.traj_pos(t), ref.traj_vel(t)] for t in ts])
        res[v] = (q, cg, tr)
    assert [R.lib(v).ref_redux_order() for v in ("glibc", "glibc_r1", "glibc_r2")] == [0, 1, 2]
    for v in ("glibc_r1", "glibc_r2"):
        for a, b in zip(res["glibc"][0], res[v][0]):
            assert bits_differ(a, b) == 0
        assert bits_differ(res["glibc"][2], res[v][2]) == 0
        c0, t0, g0 = res["glibc"][1]
        c1, t1, g1 = res[v][1]
        assert abs(c0 - c1) <= 1e-13 * abs(c0) and np.linalg.norm(g0 - g1) <= 1e-13 * np.linalg.norm(g0)


def test_extraction_is_verbatim():
    """Every generated fragment is a byte-for-byte substring of the reference file it names (no edits on the way)."""
    import re

    gen = os.path.join(os.path.dirname(HERE), "oracle", "_ref", "gen")
    if not (os.path.isdir("/root/reference/src") and os.path.isdir(gen)):
        pytest.skip("needs /root/reference and oracle/_ref/gen")
    n = 0
    for fn in sorted(os.listdir(gen)):
        if not fn.endswith(".inc"):
            continue
        txt = open(os.path.join(gen, fn), encoding="utf-8", errors="surrogateescape").read()
        parts = re.split(r"^// ---- verbatim (\S+):(\d+)-(\d+)\n", txt, flags=re.M)
        for k in range(1, len(parts), 4):
            rel, body = parts[k], parts[k + 3]
            body = re.sub(r"^#line \d+ \"[^\"]+\"\n", "", body, count=1)
            src = open(os.path.join("/root/reference", rel), encoding="utf-8", errors="surrogateescape").read()
            assert body.rstrip("\n") in src, (fn, rel, parts[k + 1])
            n += 1
    assert n >= 45

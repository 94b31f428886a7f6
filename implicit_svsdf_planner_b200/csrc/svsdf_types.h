// svsdf_types.h — POD types shared by the host runtime and the sm_100a kernels.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define SVSDF_HD __host__ __device__
#else
#define SVSDF_HD
#endif

namespace svsdf {

// Shape registry ids. Keys mirror the reference's shapeConstructors map
// (src/swept_volume/include/swept_volume/sw_manager.hpp:187-235); unknown names fall back to the
// rectangle Polygon (sw_manager.hpp:363-372).
enum ShapeId : int {
    SH_STAR = 0,
    SH_HORSESHOE,
    SH_PIE,
    SH_PIE2,
    SH_ARC,
    SH_TUNNEL,
    SH_CUTDISK,
    SH_TRAPEZOID,
    SH_RHOMBUS,
    SH_HEART,
    SH_ROUNDEDX,
    SH_BIGX,
    SH_ROUNDEDCROSS,
    SH_VESICA,
    SH_MOON,
    SH_UNEVENCAPSULE,
    SH_CIRCLE,
    SH_POLYGON,
    SH_MESH,   // triangle-mesh functor, BasicShape::getonlySDF_igl (Shape.hpp:332-340); selected by svsdf_config.mesh_*
    SH_COUNT
};

constexpr int kMaxPolyEdges = 64;
constexpr int kMeshStride = 10;          // doubles per face record: a, b, c, rmax (see ShapeFn<SH_MESH>)
constexpr int kMaxMeshFaces = 1 << 20;  // SH_MESH: faces of the triangle soup
constexpr int kFwnMaxDepth = 24;        // SH_MESH: deepest hierarchy the device traversal's explicit stack holds (svsdf_create checks)
constexpr int kMaxPieces = 64;       // pieces per trajectory supported by the per-warp accumulators
constexpr int kWarpsPerBlock = 8;    // k_outer block = 256 threads
constexpr int kGsipWarps = 22;       // k_gsip block = 704 threads: one warp per ring sample (<= 21 per round)
constexpr double kMaxDuration = 300.0;  // sw_manager.hpp:380: durations >= 300 s are not accepted by updateTraj

// Parameters of the robot-shape SDF functor. Trigonometric constants the reference evaluates on the host
// at construction (cos(20.5), sin(43) ... radians of the literal, Shape.hpp:855,1235,1276,1320) are
// evaluated on the host here too and passed in, so host/device libm differences cannot enter.
struct ShapeParams {
    int id;
    int has_xform;      // 0: trans == 0 and Rotate == I (all shipped yamls) -> pre-transform skipped (bit-exact)
    double trans[2];    // poly_params[0..1]              (Shape.hpp:287)
    double rot[4];      // Rotate(0,0),(0,1),(1,0),(1,1)  (Shape.hpp:288-294)
    double cst[4];      // per-shape host-computed constants (see shape_registry.cpp)
    double radius;      // Circle
    double rout;        // conservative circumradius about the body origin (incl. |trans|): sdf(q) >= |q| - rout for every q.
                        // Lets choiceTInit's layer-1 scan skip lattice samples that provably cannot be the minimum
                        // (thread_choice_t_init).  >= 1e30 disables the pruning (mesh functor).
    double prune_scale, prune_rmin;  // generalisation for functors that are only approximately distances far away (mesh: the float
                        // winding number w scales the distance by 1 - 2w): sdf(q) >= (|q| - rout) / prune_scale for |q| >= prune_rmin.
                        // Analytic shapes: 1 and 0.
    int poly_n;         // Polygon edge count
    int pad_;
    double poly_sx[kMaxPolyEdges], poly_sy[kMaxPolyEdges], poly_ex[kMaxPolyEdges], poly_ey[kMaxPolyEdges];
    const double *mesh_tri;  // SH_MESH: device pointer, kMeshStride doubles per face (a, b, c, rmax), vertices already R v + trans (Shape.hpp:296-302)
    int mesh_nf;
    int fwn_nn;              // SH_MESH: nodes of the 4-way winding-number hierarchy (host/fwn_bvh.hpp), 0 = none
    float fwn_boxmag;        // SH_MESH: >= |every x / y coordinate of the child boxes| (error term of the float box bounds)
    int pad3_;
    // device copies of FwnBvh's arrays: child words [nn][4]; expansion rows [nn][23][4] float (one lane per child); child boxes
    // [nn][4][6] float: lo x, lo y, hi x, hi y rounded OUTWARDS by two ulps (they contain the double vertices), squared z gap to
    // the plane z = 0 rounded down, pad; leaf triangles in float [nf][12]
    const unsigned int *fwn_child;
    const float *fwn_data;
    const float *fwn_cbox;
    const float *fwn_trif;
};

// Trajectory blob: one contiguous, 16-byte aligned buffer that the kernels pull into shared memory with a
// single TMA bulk copy (cp.async.bulk.shared::cluster.global).  All offsets are in doubles.
//   [0]  header (4 doubles: N, K1, D, reserved)
//   [4]  T[Npad]              piece durations (Npad = N rounded up to even)
//   [..] c[N][3][6]           per piece, per dim (x,y,yaw), ascending powers (== MINCO b rows 6i..6i+5)
//   [..] lat[K1pad]           layer-1 lattice times t_k = 0.15 accumulated k times (host, IEEE adds)
//   [..] pose[4][K1pad]       SoA rows x, y, cos yaw, sin yaw at lat[k] (conflict-free lane-strided reads) —
//                             filled on device by k_pose_table
struct BlobLayout {
    int N, K1;
    int off_T, off_c, off_lat, off_pose, K1pad, total;  // in doubles; total is even (16-byte multiple)
};

SVSDF_HD inline BlobLayout blob_layout(int N, int K1) {
    BlobLayout L;
    L.N = N;
    L.K1 = K1;
    int Npad = (N + 1) & ~1;
    int K1pad = (K1 + 1) & ~1;
    L.off_T = 4;
    L.off_c = L.off_T + Npad;
    L.off_lat = L.off_c + 18 * N;
    L.off_pose = L.off_lat + K1pad;
    L.K1pad = K1pad;
    L.total = L.off_pose + 4 * K1pad;
    L.total = (L.total + 1) & ~1;
    return L;
}

// dynamic shared memory of k_outer in doubles: [ blob | 8 warps x (19N + 1) accumulators | 8 warps x 32 x 4 work area ]
SVSDF_HD inline size_t outer_smem_doubles(int blob_doubles, int N) {
    return (size_t)blob_doubles + (size_t)kWarpsPerBlock * (19 * N + 1) + (size_t)kWarpsPerBlock * 128;
}

// Penalty parameters (star.yaml: weight_p 60, safety_hor 0.7; smoothedL1 mu = 0.01 is a literal in the
// reference, back_end_optimizer.hpp:1052)
struct CostParams {
    double weight_p;
    double safety_hor;
};

// Time-varying body scale S(t) = diag(s_x(t), s_y(t), 1) (svsdf_set_scale): per axis
// s(t) = c, then s = s + sin(w_k t + phi_k) a_k for k < n, in that order; t is absolute trajectory time.
constexpr int kMaxScaleTerms = 4;
struct ScaleParams {
    int n[2];
    double c[2], a[2][kMaxScaleTerms], w[2][kMaxScaleTerms], phi[2][kMaxScaleTerms];
    int exact_yaw_grad;  // 0: the reference's yaw term g^T VR^T (p - x); 1: g^T VR^T S^-1 (p - x)
};

// Kernel argument block
struct KernelArgs {
    const double *blob;        // trajectory blob (global)
    int blob_doubles;
    const double *points_xy;   // P x 2, packed (x, y)
    int64_t P;
    CostParams cp;
    // per-point outputs (optional, may be null)
    double *out_sdf, *out_tstar, *out_grad;   // grad: P x 3
    int *out_rounds;                           // GSIP rounds per point (0 for outside points)
    // reduction outputs
    double *partials;          // [gridDim.x][19N+1] block partial sums (K1)
    int want_reduce;
    int want_gsip;             // 0: stop after the outer solve (getSDFofSweptVolume semantics)
    int batched;               // k_outer: run choiceTInit / gradient / chain rule one point per lane (large P)
    // inside-point bookkeeping
    unsigned char *inside_flag;  // P
    double *inside_tstar;        // P (sparse: written for inside points only)
    int *inside_list;            // compacted, ascending point index
    int *n_inside;               // device scalar
    double *gsip_contrib;        // [n_inside][20]: cost, 18 gdC entries ([d][q]), gdT
    int *gsip_piece;             // [n_inside]
    unsigned long long *eval_counter;  // optional: executed lane-evaluations (profiling builds)
};

// K3 (svsdf_extract.cu): query-point extraction from the packed map kernel
constexpr int kMaxWaypoints = 66;   // interior waypoints of <= 64 pieces (+ optional end points)
constexpr int kMaxMapLayers = 64;   // z layers of a 3-D map (svsdf_set_map3d)
constexpr int kMaxKeepout = 160;    // keep-out polyline samples (synthetic scenes only)
struct ExtractArgs {
    const unsigned char *map;  // (X + 2h) x row_bytes, MSB-first bits along y (PCSmap_manager.h:81-108)
    int X, Y, h, row_bytes;
    double ox, oy, res;        // boundary_xyzmin (x, y) and grid resolution
    int W;                     // number of waypoint boxes
    int bx1[kMaxWaypoints], bx2[kMaxWaypoints], by1[kMaxWaypoints], by2[kMaxWaypoints];  // clamped index boxes
    // "OutOfLastOne": the box whose cells waypoint w skips is the box of waypoint w - 1; for w = 0 it is the box around
    // tmp_pos = (999, 999, 999) (plan_manager.cpp:152), i.e. after projInMap the far corner cell of the map
    int px1, px2, py1, py2;
    // one launch handles ONE z layer of the map: act[w] = the layer lies in waypoint w's z range, excl[w] = it lies in the z range
    // of the box waypoint w skips (a skipped cell must be inside the last box in all three dimensions, PCSmap_manager.h:207-209)
    unsigned char act[kMaxWaypoints], excl[kMaxWaypoints];
    int rx1, wy1, nW;          // bounding rectangle: first row, first 32-cell word, words per row
    long long n_items;         // rows * nW
    int n_keepout;
    double clearance;
    double keepout[2 * kMaxKeepout];
};

// K5 (svsdf_frontend.cu): collision kernels of the A* front end
constexpr int kMaxYawKernels = 64;
constexpr int kMaxKernelSize = 32;  // kernel rows are held as 32-bit masks
struct FrontParams {
    int kernel_size, kernel_count;
    double res, safemargin;      // kernelresu (occupancy_resolution), max(front_end_safeh, res / 2)
    int X, Y, h, row_bytes;      // map (svsdf_set_map)
    int out_words;               // 32-cell words per output row: ceil(Y / 32)
    double ox, oy, map_res;      // boundary_xyzmin (x, y) and grid resolution of the map
};
// k_expand_nodes: sample parameters of checkSubSWCollision (kt = 0, 0.02, ... accumulated on the host, <= 1)
struct SubSwParams {
    int nkt;
    double half_box;             // kernel_size / 2 + 1 (integer division), world units (front_end_Astar.hpp:224)
    double kt[64];
};

}  // namespace svsdf

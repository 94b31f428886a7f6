// svsdf_runtime.cpp — host runtime and C ABI (include/svsdf.h) of libsvsdf_b200.so.
//
// Owns the device buffers (query points resident in HBM, trajectory blob, per-CTA partials, inside-point lists),
// the CUDA stream, pinned staging memory, the host MINCO spline and the host L-BFGS; launches the sm_100a kernels
// of svsdf_kernels.cuh.  There is deliberately no CPU implementation of the hot path in this library: if CUDA is
// unavailable svsdf_create fails.
#include <cuda_runtime.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include <atomic>
#include <chrono>
#include <thread>
#include <algorithm>
#include <cmath>
#include <dlfcn.h>
#include <unistd.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/svsdf.h"
#include "host/astar.hpp"
#include "host/fwn_bvh.hpp"
#include "host/mid_end.hpp"
#include "host/lbfgs.hpp"
#include "host/minco.hpp"
#include "svsdf_launch.h"
#include "svsdf_types.h"

using namespace svsdf;

struct svsdf_ctx {
    svsdf_config cfg;
    std::string shape_name;
    ShapeParams shape;
    CostParams cp;
    bool scaled = false;  // svsdf_set_scale: body scale S(t) on the cost path (false: rigid body)
    ScaleParams scale{};
    double rho = 3.8;
    int device = 0;
    bool strict = false;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t evk[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // per-kernel timing marks
    bool mark_kernels = false;
    float last_kernel_ms[4] = {0, 0, 0, 0};  // pose table, k_outer, k_compact + k_gsip, k_finalize
    std::string err;
    int64_t launches = 0;

    // query points
    double *d_mesh_tri = nullptr;  // SH_MESH: kMeshStride doubles per face
    unsigned int *d_fwn_child = nullptr;  // SH_MESH: the winding-number hierarchy (host/fwn_bvh.hpp)
    float *d_fwn_data = nullptr, *d_fwn_cbox = nullptr, *d_fwn_trif = nullptr;
    // K5: A* front-end collision kernels
    bool front_ready = false;
    FrontParams front{};
    std::vector<double> front_yaw;
    std::vector<unsigned char> front_cells, front_bytes;
    unsigned char *d_front_bytes = nullptr;
    unsigned *d_front_rowmask = nullptr;
    unsigned *d_cspace = nullptr;
    size_t cap_cspace = 0;
    unsigned char *d_front_scratch = nullptr;  // grow-only device scratch of the batched front-end calls
    size_t cap_front_scratch = 0;
    double *d_points = nullptr;  // packed xy
    bool own_points = true;
    int64_t P = 0;
    int64_t cap_points = 0;
    // scratch sized by P
    unsigned char *d_flag = nullptr;
    double *d_inside_tstar = nullptr;
    int *d_inside_list = nullptr;
    double *d_gsip_contrib = nullptr;
    int *d_gsip_piece = nullptr;
    int64_t cap_scratch = 0;
    int *d_n_inside = nullptr;
    unsigned long long *d_eval_counter = nullptr;
    bool count_evals = false;
    // trajectory blob
    double *d_blob = nullptr;
    int cap_blob = 0;
    double *h_blob = nullptr;  // pinned
    int cap_hblob = 0;
    BlobLayout layout{};
    int traj_N = 0;
    double traj_D = 0.0;
    int occ_N = -1, occ_blob = -1, occ_outer = 2, occ_gsip = 2;  // cached occupancy query
    int64_t last_n_inside = -1;  // interior points seen by the previous cost evaluation (picks the k_gsip variant)
    // reduction
    double *d_partials = nullptr;
    int64_t cap_partials = 0;
    double *d_out = nullptr;  // 1 + 19N + 1
    double *d_tot = nullptr;  // 19N + 1 (finalize scratch)
    unsigned int *d_ticket = nullptr;
    double *h_out = nullptr;  // pinned
    int cap_out = 0;
    // query scratch (per-point outputs)
    double *d_q_points = nullptr, *d_q_sdf = nullptr, *d_q_ts = nullptr, *d_q_grad = nullptr;
    int *d_q_rounds = nullptr;
    int64_t cap_q = 0;
    double *h_stage = nullptr;  // pinned staging for results download and the small uploads of the other entry points
    size_t cap_stage = 0;
    // svsdf_set_points has its own pinned stage and does NOT wait for its copies: the kernels that follow are ordered behind them
    // on the context's stream, and the host goes on (builds the trajectory blob) while the DMA runs.  ev_pts marks the end of the
    // last upload: the next svsdf_set_points (which overwrites the stage) and svsdf_device_ptr_points (which hands the buffer to
    // other streams) wait on it.
    svsdf_lmbm *lmbm = nullptr;          // svsdf_set_lmbm_library: this context's private instance of the reference's LMBM
    svsdf_lmbm_params lmbm_params;
    double *h_pts_stage = nullptr;
    size_t cap_pts_stage = 0;
    cudaEvent_t ev_pts = nullptr;
    bool pts_inflight = false;

    // packed map kernel (K3)
    unsigned char *d_map = nullptr;
    bool own_map = true;
    size_t cap_map = 0;
    int map_X = 0, map_Y = 0, map_h = 0, map_row_bytes = 0;
    int map_Z = 1;             // z layers held on the device (svsdf_set_map3d), each in the 2-D layout; layer 0 first
    double map_ox = 0, map_oy = 0, map_oz = 0, map_res = 0;
    int *d_block_counts = nullptr;
    int cap_block_counts = 0;
    int64_t *d_n_total = nullptr;

    // optimiser state (R3/R4)
    host::MincoS3NU minco;
    int pieceN = 0;
    bool have_boundary = false;
    std::vector<double> times, gradByTimes, partialGradByTimes, partialGradByCoeffs, gradByPoints;
    double cost_pos = 0, cost_other = 0, cost_total = 0;
    int n_evaluate = 0;
    double gpu_ms_total = 0.0;
    bool time_kernels = false;
    int last_status = 0;
    // test hooks, read ONCE at svsdf_create (SVSDF_FORCE_GRID_OUTER / SVSDF_FORCE_BATCHED): exercise the batched schedule
    // on small inputs; -1 = not set
    int force_grid_outer = -1;
    int force_batched = -1;
};

namespace {

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                        \
            return SVSDF_ERR_CUDA;                                                                 \
        }                                                                                          \
    } while (0)

const char *kShapeNames[] = {"star",      "sdHorseshoe", "sdPie",      "sdPie2", "sdArc",          "sdTunnel",
                             "sdCutDisk", "sdTrapezoid", "sdRhombus",  "sdHeart", "sdRoundedX",    "bigX",
                             "sdRoundedCross", "sdOrientedVesica", "sdMoon", "sdUnevenCapsule"};

int shape_id_from_name(const char *name) {
    if (name) {
        for (int i = 0; i < 16; ++i)
            if (std::strcmp(name, kShapeNames[i]) == 0) return i;
        if (std::strcmp(name, "Circle") == 0) return SH_CIRCLE;
    }
    return SH_POLYGON;  // sw_manager.hpp:363-372
}

// Host-side construction of the shape functor parameters (what the reference's shape constructors do:
// Shape.hpp:281-294 base transform, and the per-class constant members).
void build_shape(const svsdf_config &cfg, ShapeParams &S) {
    std::memset(&S, 0, sizeof(S));
    S.id = shape_id_from_name(cfg.shape);
    const double PI = 3.14159265358979323846;  // Shape.hpp:31
    const double yaw = (cfg.poly_params[2] * PI / 180.0);
    S.trans[0] = cfg.poly_params[0];
    S.trans[1] = cfg.poly_params[1];
    S.rot[0] = std::cos(yaw);
    S.rot[1] = -std::sin(yaw);
    S.rot[2] = std::sin(yaw);
    S.rot[3] = std::cos(yaw);
    S.has_xform = !(S.trans[0] == 0.0 && S.trans[1] == 0.0 && S.rot[0] == 1.0 && S.rot[1] == 0.0 && S.rot[2] == 0.0 &&
                    S.rot[3] == 1.0);
    S.radius = 1.0;
    S.rout = 1e300;
    S.prune_scale = 1.0;
    S.prune_rmin = 0.0;
    if (cfg.mesh_faces && cfg.mesh_nf > 0) {  // triangle-mesh functor requested: overrides the registry name
        S.id = SH_MESH;
        return;
    }
    {
        // Circumradius of each analytic shape about its own origin, rounded up with a 0.05 margin (measured: the largest
        // |q| with sdf(q) <= 0; the functors are exact distances outside the shape, so sdf(q) >= |q| - R everywhere —
        // tests/test_oracle_shapes.py::test_circumradius_bound checks every entry against the oracle, the GPU parity
        // tests check the pruned scan bit for bit).  The body-frame pre-transform shifts the origin by |trans|.
        static const double kRout[17] = {2.85, 2.36, 3.05, 3.05, 2.88, 2.97, 5.05, 3.65, 4.55, 4.63, 2.42, 3.84, 2.05, 4.52, 3.05, 6.05, 1.05};
        if (S.id >= 0 && S.id <= SH_CIRCLE) S.rout = kRout[S.id] + std::sqrt(S.trans[0] * S.trans[0] + S.trans[1] * S.trans[1]);
    }
    switch (S.id) {
        case SH_HORSESHOE: S.cst[0] = std::cos(20.5); S.cst[1] = std::sin(20.5); break;  // Shape.hpp:855
        case SH_PIE: S.cst[0] = std::cos(43.0); S.cst[1] = std::sin(43.0); break;        // :1235
        case SH_PIE2: S.cst[0] = std::cos(1.0); S.cst[1] = std::sin(1.0); break;         // :1276
        case SH_ARC: S.cst[0] = std::sin(20.0); S.cst[1] = std::cos(20.0); break;        // :1320
        case SH_CUTDISK: S.cst[0] = std::sqrt(5.0 * 5.0 - 2.0 * 2.0); break;             // :701
        case SH_HEART: S.cst[0] = std::sqrt(2.0) / 4.0; break;                           // :946
        case SH_VESICA: {                                                                // :1119-1128
            const double ax = 2, ay = 4, bx = -2, by = -4, w = 0.8;
            const double bax = bx - ax, bay = by - ay;
            const double r = 0.5 * std::sqrt(bax * bax + bay * bay);
            S.cst[0] = r;
            S.cst[1] = 0.5 * (r * r - w * w) / w;
            S.cst[2] = bax / r;
            S.cst[3] = bay / r;
            break;
        }
        case SH_MOON: {  // :1205-1206
            const double d = 0.8, ra = 3.0, rb = 2.4;
            const double a = (ra * ra - rb * rb + d * d) / (2.0 * d);
            S.cst[0] = a;
            S.cst[1] = std::sqrt(std::max(ra * ra - a * a, 0.0));
            break;
        }
        case SH_UNEVENCAPSULE: {  // :535-536
            const double b = (2.0 - 1.0) / 5.0;
            S.cst[0] = b;
            S.cst[1] = std::sqrt(1.0 - b * b);
            break;
        }
        case SH_POLYGON: {
            const double rect[8] = {6, -0.1, 6, 0.1, -6, 0.1, -6, -0.1};  // sw_manager.hpp:365-369
            const double *xy = rect;
            int n = 4;
            if (cfg.polygon_xy && cfg.polygon_n >= 3 && cfg.polygon_n <= kMaxPolyEdges) {
                xy = cfg.polygon_xy;
                n = cfg.polygon_n;
            }
            S.poly_n = n;
            for (int i = 0; i < n; ++i) {  // Polygon ctor, Shape.hpp:1429-1446
                const int j = (i + 1) % n;
                S.poly_sx[i] = xy[2 * i];
                S.poly_sy[i] = xy[2 * i + 1];
                S.poly_ex[i] = xy[2 * j];
                S.poly_ey[i] = xy[2 * j + 1];
            }
            S.has_xform = 0;
            S.rout = 0.0;  // Polygon ignores trans/Rotate: the farthest vertex bounds it
            for (int i = 0; i < n; ++i) S.rout = std::max(S.rout, std::sqrt(xy[2 * i] * xy[2 * i] + xy[2 * i + 1] * xy[2 * i + 1]));
            S.rout += 0.05;
            break;
        }
        default: break;
    }
}

int ensure_scratch(svsdf_ctx *ctx, int64_t P) {
    if (P <= ctx->cap_scratch) return SVSDF_OK;
    cudaFree(ctx->d_flag); cudaFree(ctx->d_inside_tstar); cudaFree(ctx->d_inside_list);
    cudaFree(ctx->d_gsip_contrib); cudaFree(ctx->d_gsip_piece);
    ctx->d_flag = nullptr; ctx->d_inside_tstar = nullptr; ctx->d_inside_list = nullptr;
    ctx->d_gsip_contrib = nullptr; ctx->d_gsip_piece = nullptr;
    ctx->cap_scratch = 0;
    int64_t cap = P + P / 8 + 1024;
    CK(cudaMalloc(&ctx->d_flag, cap));
    CK(cudaMalloc(&ctx->d_inside_tstar, cap * sizeof(double)));
    CK(cudaMalloc(&ctx->d_inside_list, cap * sizeof(int)));
    CK(cudaMalloc(&ctx->d_gsip_contrib, cap * 20 * sizeof(double)));
    CK(cudaMalloc(&ctx->d_gsip_piece, cap * sizeof(int)));
    ctx->cap_scratch = cap;
    return SVSDF_OK;
}

int ensure_stage(svsdf_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->cap_stage) return SVSDF_OK;
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    ctx->h_stage = nullptr;
    ctx->cap_stage = 0;
    size_t cap = bytes + bytes / 4 + 4096;
    CK(cudaMallocHost(&ctx->h_stage, cap));
    ctx->cap_stage = cap;
    return SVSDF_OK;
}

// updateTraj (sw_manager.hpp:376-385) + the layer-1 lattice of choiceTInit (:538-581): builds the blob in
// pinned memory, uploads it and launches the pose-table kernel.
int pose_table(svsdf_ctx *ctx) {
    cudaError_t e = ctx->strict ? strict::launch_pose_table(ctx->d_blob, ctx->layout.K1, ctx->stream)
                                : fast::launch_pose_table(ctx->d_blob, ctx->layout.K1, ctx->stream);
    CK(e);
    ctx->launches += 1;
    return SVSDF_OK;
}

int upload_traj(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, bool launch_pose = true) {
    if (N < 1 || N > kMaxPieces || !T || !coeffs) {
        ctx->err = "svsdf: N out of range (1..64) or null trajectory";
        return SVSDF_ERR_INVALID;
    }
    double D = 0.0;  // Trajectory::getTotalDuration (trajectory.hpp:410-419)
    for (int i = 0; i < N; ++i) {
        if (!(T[i] > 0.0) || !std::isfinite(T[i])) {
            ctx->err = "svsdf: non-positive or non-finite piece duration";
            return SVSDF_ERR_INVALID;
        }
        D += T[i];
    }
    if (!(D < kMaxDuration)) {
        // The reference silently keeps the previous duration in this case (sw_manager.hpp:380); we refuse.
        ctx->err = "svsdf: total duration >= 300 s is not supported (reference updateTraj ignores it)";
        return SVSDF_ERR_INVALID;
    }
    // layer-1 lattice: for (t = 0; t <= D; t += 0.15)
    int K1 = 0;
    for (double t = 0.0; t <= D; t += 0.15) K1++;
    BlobLayout L = blob_layout(N, K1);
    if (L.total > ctx->cap_hblob) {
        if (ctx->h_blob) cudaFreeHost(ctx->h_blob);
        ctx->h_blob = nullptr;
        ctx->cap_hblob = 0;
        CK(cudaMallocHost(&ctx->h_blob, (size_t)(L.total + 1024) * sizeof(double)));
        ctx->cap_hblob = L.total + 1024;
    }
    if (L.total > ctx->cap_blob) {
        cudaFree(ctx->d_blob);
        ctx->d_blob = nullptr;
        ctx->cap_blob = 0;
        CK(cudaMalloc(&ctx->d_blob, (size_t)(L.total + 1024) * sizeof(double)));
        ctx->cap_blob = L.total + 1024;
    }
    double *h = ctx->h_blob;
    std::memset(h, 0, (size_t)L.off_pose * sizeof(double));
    h[0] = (double)N;
    h[1] = (double)K1;
    h[2] = D;
    for (int i = 0; i < N; ++i) h[L.off_T + i] = T[i];
    // coefficients: MINCO b (col-major 6N x 3) -> [piece][dim][power]  (minco.hpp:515-528 builds the same
    // per-piece matrices, stored there highest power first)
    for (int i = 0; i < N; ++i)
        for (int d = 0; d < 3; ++d)
            for (int k = 0; k < 6; ++k) h[L.off_c + 18 * i + 6 * d + k] = coeffs[(size_t)d * 6 * N + 6 * i + k];
    {
        int k = 0;
        for (double t = 0.0; t <= D; t += 0.15) h[L.off_lat + k++] = t;
    }
    CK(cudaMemcpyAsync(ctx->d_blob, h, (size_t)L.off_pose * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    ctx->layout = L;
    ctx->traj_N = N;
    ctx->traj_D = D;
    if (launch_pose) return pose_table(ctx);
    return SVSDF_OK;
}

int refresh_occupancy(svsdf_ctx *ctx) {
    if (ctx->occ_N == ctx->traj_N && ctx->occ_blob == ctx->layout.total) return SVSDF_OK;
    int oo = 0, og = 0;
    cudaError_t e = ctx->strict ? strict::query_occupancy(ctx->shape, ctx->traj_N, ctx->layout.total, &oo, &og)
                                : fast::query_occupancy(ctx->shape, ctx->traj_N, ctx->layout.total, &oo, &og);
    CK(e);
    ctx->occ_outer = oo > 0 ? oo : 1;
    ctx->occ_gsip = og > 0 ? og : 1;
    ctx->occ_N = ctx->traj_N;
    ctx->occ_blob = ctx->layout.total;
    return SVSDF_OK;
}

int grid_for(const svsdf_ctx *ctx, int64_t P) {
    // one warp per point, 8 warps per CTA, warp-stride loop.  The grid is exactly one full wave (SMs x resident CTAs
    // per SM, from the occupancy query): a larger grid would run a partially filled second wave.
    int64_t need = (P + kWarpsPerBlock - 1) / kWarpsPerBlock;
    int64_t cap = (int64_t)ctx->sm_count * ctx->occ_outer;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

// Runs K1 (+compact, K2) (+finalize).  Inputs resident on the device.
int run_kernels(svsdf_ctx *ctx, const double *d_points, int64_t P, bool reduce, bool gsip, double *o_sdf,
                double *o_ts, double *o_grad, int *o_rounds) {
    const int N = ctx->traj_N;
    int rc = ensure_scratch(ctx, P);
    if (rc) return rc;
    rc = refresh_occupancy(ctx);
    if (rc) return rc;
    int grid = grid_for(ctx, P);
    if (ctx->force_grid_outer > 0) grid = ctx->force_grid_outer;  // test hook
    const int nacc = 19 * N + 1;
    if (reduce) {
        int64_t need = (int64_t)grid * nacc;
        if (need > ctx->cap_partials) {
            cudaFree(ctx->d_partials);
            ctx->d_partials = nullptr;
            ctx->cap_partials = 0;
            CK(cudaMalloc(&ctx->d_partials, (size_t)(need + 4096) * sizeof(double)));
            ctx->cap_partials = need + 4096;
        }
        if (nacc + 1 > ctx->cap_out) {
            cudaFree(ctx->d_out);
            if (ctx->h_out) cudaFreeHost(ctx->h_out);
            ctx->d_out = nullptr; ctx->h_out = nullptr; ctx->cap_out = 0;
            CK(cudaMalloc(&ctx->d_out, (size_t)(nacc + 64) * sizeof(double)));
            cudaFree(ctx->d_tot);
            ctx->d_tot = nullptr;
            CK(cudaMalloc(&ctx->d_tot, (size_t)(nacc + 64) * sizeof(double)));
            CK(cudaMallocHost(&ctx->h_out, (size_t)(nacc + 64) * sizeof(double)));
            ctx->cap_out = nacc + 64;
        }
    }
    KernelArgs A;
    std::memset(&A, 0, sizeof(A));
    A.blob = ctx->d_blob;
    A.blob_doubles = ctx->layout.total;
    A.points_xy = d_points;
    A.P = P;
    A.cp = ctx->cp;
    A.out_sdf = o_sdf; A.out_tstar = o_ts; A.out_grad = o_grad; A.out_rounds = o_rounds;
    A.partials = ctx->d_partials;
    A.want_reduce = reduce ? 1 : 0;
    A.want_gsip = gsip ? 1 : 0;
    // batched path pays off once every warp owns a couple of dozen points; small problems keep one point per warp
    A.batched = (P >= (int64_t)16 * grid * kWarpsPerBlock) ? 1 : 0;
    if (ctx->force_batched >= 0) A.batched = ctx->force_batched;  // test hook
    A.inside_flag = ctx->d_flag;
    A.inside_tstar = ctx->d_inside_tstar;
    A.inside_list = ctx->d_inside_list;
    A.n_inside = ctx->d_n_inside;
    A.gsip_contrib = ctx->d_gsip_contrib;
    A.gsip_piece = ctx->d_gsip_piece;
    A.eval_counter = ctx->count_evals ? ctx->d_eval_counter : nullptr;
    // previous evaluation had few interior points -> 22-warp CTAs (one warp per ring sample, lower latency)
    // (the scaled kernels exist in the 8-warp width only)
    const int gsip_wide = (!ctx->scaled && reduce && ctx->last_n_inside >= 0 && ctx->last_n_inside <= ctx->sm_count) ? 1 : 0;
    const int grid_gsip = gsip_wide ? ctx->sm_count : ctx->sm_count * ctx->occ_gsip;
    if (!gsip) CK(cudaMemsetAsync(ctx->d_n_inside, 0, sizeof(int), ctx->stream));
    size_t smem = outer_smem_doubles(A.blob_doubles, N) * sizeof(double);
    if (smem > 200 * 1024) {
        ctx->err = "svsdf: trajectory blob does not fit in shared memory";
        return SVSDF_ERR_INVALID;
    }
    const ScaleParams *Z = ctx->scaled ? &ctx->scale : nullptr;
    cudaError_t e = ctx->strict ? strict::launch_cost_kernels(A, ctx->shape, Z, N, grid, grid_gsip, ctx->stream,
                                                              ctx->mark_kernels ? ctx->evk[2] : nullptr, gsip_wide)
                                : fast::launch_cost_kernels(A, ctx->shape, Z, N, grid, grid_gsip, ctx->stream,
                                                            ctx->mark_kernels ? ctx->evk[2] : nullptr, gsip_wide);
    CK(e);
    ctx->launches += gsip ? 3 : 1;
    if (ctx->mark_kernels) CK(cudaEventRecord(ctx->evk[3], ctx->stream));
    if (reduce) {
        e = ctx->strict ? strict::launch_finalize(ctx->d_partials, grid, N, ctx->d_n_inside, ctx->d_gsip_contrib,
                                                  ctx->d_gsip_piece, ctx->d_tot, ctx->d_ticket, ctx->d_out, ctx->stream)
                        : fast::launch_finalize(ctx->d_partials, grid, N, ctx->d_n_inside, ctx->d_gsip_contrib,
                                                ctx->d_gsip_piece, ctx->d_tot, ctx->d_ticket, ctx->d_out, ctx->stream);
        CK(e);
        ctx->launches += 1;
    }
    return SVSDF_OK;
}

// R1 on the context's points; result (1 + 19N + 1 doubles) lands in ctx->h_out after the stream sync.
int cost_grad_raw(svsdf_ctx *ctx, int N, const double *T, const double *coeffs) {
    if (!ctx->d_points || ctx->P < 0) {
        ctx->err = "svsdf: query points not set";
        return SVSDF_ERR_NOT_READY;
    }
    int rc = upload_traj(ctx, N, T, coeffs);
    if (rc) return rc;
    if (ctx->time_kernels) CK(cudaEventRecord(ctx->ev0, ctx->stream));
    rc = run_kernels(ctx, ctx->d_points, ctx->P, true, true, nullptr, nullptr, nullptr, nullptr);
    if (rc) return rc;
    if (ctx->time_kernels) CK(cudaEventRecord(ctx->ev1, ctx->stream));
    const int nout = 1 + 19 * N + 1;
    CK(cudaMemcpyAsync(ctx->h_out, ctx->d_out, (size_t)nout * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->time_kernels) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        ctx->gpu_ms_total += ms;
    }
    ctx->last_n_inside = (int64_t)ctx->h_out[1 + 19 * N];
    return SVSDF_OK;
}

double evaluate_impl(svsdf_ctx *ctx, const double *x, double *g, int n) {
    const int N = ctx->pieceN;
    if (!ctx->have_boundary || n != N + 3 * (N - 1)) {
        ctx->err = "svsdf_evaluate: boundary conditions not set or wrong n";
        ctx->last_status = SVSDF_ERR_NOT_READY;
        return NAN;
    }
    ctx->n_evaluate++;
    // forwardT / forwardP (back_end_optimizer.hpp:353-354)
    for (int i = 0; i < N; ++i) ctx->times[i] = host::forwardT(x[i]);
    const double *q = x + N;
    ctx->minco.setParameters(q, ctx->times.data());
    double cost = ctx->minco.getEnergy();
    ctx->minco.getEnergyPartialGradByCoeffs(ctx->partialGradByCoeffs.data());
    ctx->minco.getEnergyPartialGradByTimes(ctx->partialGradByTimes.data());
    const double energy_cost = cost;
    int rc = cost_grad_raw(ctx, N, ctx->times.data(), ctx->minco.getCoeffs());
    if (rc) {
        ctx->last_status = rc;
        return NAN;
    }
    const double *o = ctx->h_out;
    cost += o[0];
    for (int e = 0; e < 18 * N; ++e) ctx->partialGradByCoeffs[e] += o[1 + e];
    for (int i = 0; i < N; ++i) ctx->partialGradByTimes[i] += o[1 + 18 * N + i];
    const double pos_cost = cost - energy_cost;
    ctx->minco.propogateGrad(ctx->partialGradByCoeffs.data(), ctx->partialGradByTimes.data(),
                             ctx->gradByPoints.data(), ctx->gradByTimes.data());
    double tsum = 0.0;
    for (int i = 0; i < N; ++i) tsum += ctx->times[i];
    cost += ctx->rho * tsum;
    for (int i = 0; i < N; ++i) ctx->gradByTimes[i] += ctx->rho;
    ctx->cost_pos = pos_cost;
    ctx->cost_other = cost - pos_cost;
    ctx->cost_total = cost;
    for (int i = 0; i < N; ++i) g[i] = host::backwardGradT(x[i], ctx->gradByTimes[i]);
    for (int i = 0; i < 3 * (N - 1); ++i) g[N + i] = ctx->gradByPoints[i];
    ctx->last_status = SVSDF_OK;
    return cost;
}

}  // namespace

// ---- batch variants: a pool of contexts, one worker thread each, dynamic hand-out of problem indices ------------------
namespace {
template <class Body>
int run_pool(svsdf_ctx *const *ctxs, int n_ctx, int n_problems, svsdf_next_problem_t next, void *next_user, Body body) {
    if (!ctxs || n_ctx < 1 || n_problems < 0) return SVSDF_ERR_INVALID;
    for (int c = 0; c < n_ctx; ++c)
        if (!ctxs[c]) return SVSDF_ERR_INVALID;
    std::atomic<int> counter{0};
    std::atomic<int> first_err{SVSDF_OK};
    auto worker = [&](int c) {
        for (;;) {
            const int k = next ? next(next_user) : counter.fetch_add(1);
            if (k < 0 || k >= n_problems) break;
            const int rc = body(ctxs[c], k);
            if (rc != SVSDF_OK) {
                int expected = SVSDF_OK;
                first_err.compare_exchange_strong(expected, rc);
            }
        }
    };
    if (n_ctx == 1) {
        worker(0);
    } else {
        std::vector<std::thread> th;
        th.reserve(n_ctx);
        for (int c = 0; c < n_ctx; ++c) th.emplace_back(worker, c);
        for (auto &t : th) t.join();
    }
    return first_err.load();
}
}  // namespace


extern "C" {

void svsdf_default_config(svsdf_config *cfg) {
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->shape = "star";
    cfg->weight_p = 60.0;
    cfg->safety_hor = 0.7;
    cfg->rho = 3.8;
    cfg->strict_fp = 1;  // reference-rounding build is the default
}

int svsdf_shape_id(const char *name) { return shape_id_from_name(name); }
int svsdf_shape_bound_radius(const svsdf_config *cfg, double *radius_out) {
    if (!cfg || !radius_out) return SVSDF_ERR_INVALID;
    ShapeParams S;
    build_shape(*cfg, S);
    *radius_out = S.rout;
    return SVSDF_OK;
}

// Wavefront .obj -> (V, F): `v x y z` and `f i[/..] j[/..] k[/..] ...` records (1-based or negative indices), polygons
// fan-triangulated — what igl::read_triangle_mesh yields for the reference's shapes/*.obj (Shape.hpp:285).
int svsdf_read_obj(const char *path, double **vertices_out, int *nv_out, int32_t **faces_out, int *nf_out) {
    if (!path || !vertices_out || !nv_out || !faces_out || !nf_out) return SVSDF_ERR_INVALID;
    *vertices_out = nullptr; *faces_out = nullptr; *nv_out = 0; *nf_out = 0;
    std::FILE *fp = std::fopen(path, "r");
    if (!fp) return SVSDF_ERR_INVALID;
    std::vector<double> V;
    std::vector<int32_t> F;
    char line[4096];
    bool bad = false;
    while (std::fgets(line, sizeof(line), fp)) {
        const size_t len = std::strlen(line);
        if (len + 1 == sizeof(line) && line[len - 1] != '\n') { bad = true; break; }  // record longer than the buffer
        char *p = line;
        while (*p == ' ' || *p == '\t') ++p;
        if (p[0] == 'v' && (p[1] == ' ' || p[1] == '\t')) {
            double x, y, z;
            if (std::sscanf(p + 1, "%lf %lf %lf", &x, &y, &z) != 3) { bad = true; break; }
            V.push_back(x); V.push_back(y); V.push_back(z);
        } else if (p[0] == 'f' && (p[1] == ' ' || p[1] == '\t')) {
            std::vector<int32_t> idx;
            char *q = p + 1;
            for (;;) {
                while (*q == ' ' || *q == '\t') ++q;
                if (*q == 0 || *q == '\n' || *q == '\r' || *q == '#') break;
                char *end = nullptr;
                long i = std::strtol(q, &end, 10);
                if (end == q) { bad = true; break; }
                const long nv = (long)(V.size() / 3);
                idx.push_back((int32_t)(i > 0 ? i - 1 : nv + i));
                q = end;
                while (*q && *q != ' ' && *q != '\t' && *q != '\n' && *q != '\r') ++q;  // skip /vt/vn
            }
            if (bad) break;
            for (size_t k = 1; k + 1 < idx.size(); ++k) { F.push_back(idx[0]); F.push_back(idx[k]); F.push_back(idx[k + 1]); }
        }
    }
    std::fclose(fp);
    const int nv = (int)(V.size() / 3), nf = (int)(F.size() / 3);
    for (int32_t i : F)
        if (i < 0 || i >= nv) bad = true;
    if (bad || nv == 0 || nf == 0) return SVSDF_ERR_INVALID;
    double *vo = (double *)std::malloc(V.size() * sizeof(double));
    int32_t *fo = (int32_t *)std::malloc(F.size() * sizeof(int32_t));
    if (!vo || !fo) { std::free(vo); std::free(fo); return SVSDF_ERR_INVALID; }
    std::memcpy(vo, V.data(), V.size() * sizeof(double));
    std::memcpy(fo, F.data(), F.size() * sizeof(int32_t));
    *vertices_out = vo; *faces_out = fo; *nv_out = nv; *nf_out = nf;
    return SVSDF_OK;
}
int svsdf_mesh_fwn_host(const double *vertices, int nv, const int32_t *faces, int nf, int *n_nodes_out, int node_capacity,
                        uint32_t *children_out, float *data_out, int64_t n, const double *q, double *w_out) {
    if (!vertices || !faces || nv < 3 || nf < 1 || n < 0 || (n > 0 && (!q || !w_out))) return SVSDF_ERR_INVALID;
    for (int64_t k = 0; k < 3 * (int64_t)nf; ++k)
        if (faces[k] < 0 || faces[k] >= nv) return SVSDF_ERR_INVALID;
    host::FwnBvh B;
    B.build(vertices, nv, faces, nf);
    if (n_nodes_out) *n_nodes_out = B.nn;
    if (children_out && node_capacity >= B.nn) std::memcpy(children_out, B.child.data(), B.child.size() * sizeof(uint32_t));
    if (data_out && node_capacity >= B.nn) std::memcpy(data_out, B.data.data(), B.data.size() * sizeof(float));
    for (int64_t i = 0; i < n; ++i) w_out[i] = B.winding_number(q + 3 * i);
    return SVSDF_OK;
}

void svsdf_free(void *p) { std::free(p); }

// ---------------------------------------------------------------------------------------------------------------------
// The reference's LMBM library as a plug-in (lmbm.h:214-221).  Each handle is its own dlopen of (a private copy of) the file.
// ---------------------------------------------------------------------------------------------------------------------
struct svsdf_lmbm {
    void *dl = nullptr;
    // lmbm::lmbm_optimize(int, double*, double*, lmbm_evaluate_t, void*, lmbm_progress_t, lmbm_parameter_t*)
    int (*optimize)(int, double *, double *, svsdf_eval_t, void *, svsdf_progress_t, svsdf_lmbm_params *) = nullptr;
};
static thread_local std::string g_lmbm_err;
const char *svsdf_lmbm_last_error(void) { return g_lmbm_err.c_str(); }
void svsdf_lmbm_default_params(svsdf_lmbm_params *p) {  // the member initialisers of lmbm::lmbm_parameter_t (lmbm.h:15-174)
    if (!p) return;
    p->timeout = 300.0f; p->bundle_size = 2; p->ini_corrections = 7; p->max_corrections = 15; p->exponent_distmeasure = 2;
    p->max_iterations = 10000; p->max_evaluations = 20000; p->past = 10; p->verbose = -1; p->update_method = 0; p->scaling_strategy = 0;
    p->delta_past = 1.0e-8; p->f_rel_eps = 1.0e+4; p->f_lower_bound = -1.0e+60; p->terminate_param1 = 1.0e-6; p->terminate_param2 = 1.0e-6;
    p->distance_measure = 0.5; p->sufficient_dec = 1.0e-4; p->max_stepsize = 1.5;
}
int svsdf_lmbm_open(const char *path, int private_copy, svsdf_lmbm **out) {
    if (!path || !out) return SVSDF_ERR_INVALID;
    *out = nullptr;
    std::string load = path;
    bool temp = false;
    if (private_copy) {  // a distinct file is a distinct library instance to the loader: own statics, own Fortran COMMON / SAVE data
        FILE *src = std::fopen(path, "rb");
        if (!src) { g_lmbm_err = std::string("svsdf_lmbm_open: cannot read ") + path; return SVSDF_ERR_INVALID; }
        char tmpl[] = "/tmp/svsdf_lmbm_XXXXXX";
        const int fd = mkstemp(tmpl);
        if (fd < 0) { std::fclose(src); g_lmbm_err = "svsdf_lmbm_open: mkstemp failed"; return SVSDF_ERR_INVALID; }
        char buf[1 << 16];
        size_t nrd;
        bool ok = true;
        while ((nrd = std::fread(buf, 1, sizeof(buf), src)) > 0) ok = ok && (write(fd, buf, nrd) == (ssize_t)nrd);
        std::fclose(src);
        close(fd);
        if (!ok) { unlink(tmpl); g_lmbm_err = "svsdf_lmbm_open: copy failed"; return SVSDF_ERR_INVALID; }
        load = tmpl;
        temp = true;
    }
    void *dl = dlopen(load.c_str(), RTLD_NOW | RTLD_LOCAL);
    if (temp) unlink(load.c_str());  // the mapping stays valid
    if (!dl) { g_lmbm_err = std::string("svsdf_lmbm_open: dlopen: ") + (dlerror() ? dlerror() : "?"); return SVSDF_ERR_INVALID; }
    void *sym = dlsym(dl, "_ZN4lmbm13lmbm_optimizeEiPdS0_PFdPvPKdS0_iES1_PFiS1_S3_iEPNS_16lmbm_parameter_tE");
    if (!sym) { dlclose(dl); g_lmbm_err = "svsdf_lmbm_open: lmbm::lmbm_optimize not found in the library"; return SVSDF_ERR_INVALID; }
    svsdf_lmbm *h = new svsdf_lmbm();
    h->dl = dl;
    h->optimize = reinterpret_cast<decltype(h->optimize)>(sym);
    *out = h;
    return SVSDF_OK;
}
void svsdf_lmbm_close(svsdf_lmbm *h) {
    if (!h) return;
    if (h->dl) dlclose(h->dl);
    delete h;
}
int svsdf_lmbm_minimize(svsdf_lmbm *h, svsdf_eval_t eval, void *instance, double *x, int n, const svsdf_lmbm_params *params,
                        svsdf_progress_t progress, double *f_out) {
    if (!h || !h->optimize || !eval || !x || n < 1) return SVSDF_ERR_INVALID;
    svsdf_lmbm_params p;
    if (params) p = *params; else svsdf_lmbm_default_params(&p);
    double fx = 0.0;
    // lmbm.cpp calls the progress function unconditionally (earlyexit_): never hand it a null pointer
    const int ret = h->optimize(n, x, &fx, eval, instance, progress ? progress : +[](void *, const double *, const int) { return 0; }, &p);
    if (f_out) *f_out = fx;
    return ret;
}
int svsdf_set_lmbm_library(svsdf_ctx *ctx, const char *path, const svsdf_lmbm_params *params) {
    if (!ctx) return SVSDF_ERR_INVALID;
    if (ctx->lmbm) { svsdf_lmbm_close(ctx->lmbm); ctx->lmbm = nullptr; }
    if (!path) return SVSDF_OK;
    if (params) ctx->lmbm_params = *params; else svsdf_lmbm_default_params(&ctx->lmbm_params);
    const int rc = svsdf_lmbm_open(path, 1, &ctx->lmbm);
    if (rc) ctx->err = g_lmbm_err;
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// mid end (host/mid_end.hpp): OriTraj's cost function and warm-start optimisation, host only
// ---------------------------------------------------------------------------------------------------------------------
void svsdf_mid_default_config(svsdf_mid_config *c) {
    if (!c) return;
    const host::MidEndConfig d;
    c->rho_mid_end = d.rho_mid_end; c->vmax = d.vmax; c->omgmax = d.omgmax; c->weight_v = d.weight_v; c->weight_omg = d.weight_omg;
    c->weight_pr = d.weight_pr; c->weight_ar = d.weight_ar; c->smoothingEps = d.smoothingEps; c->integralIntervs = d.integralIntervs;
    c->vehicleMass = d.vehicleMass; c->gravAcc = d.gravAcc; c->horizDrag = d.horizDrag; c->vertDrag = d.vertDrag; c->parasDrag = d.parasDrag;
    c->speedEps = d.speedEps; c->mem_size = d.mem_size; c->past = d.past; c->min_step = d.min_step; c->g_epsilon = d.g_epsilon;
    c->relCostTolMidEnd = d.relCostTolMidEnd; c->max_iterations = d.max_iterations; c->cancel_after = d.cancel_after; c->solver = d.solver;
}
static host::MidEndConfig mid_cfg(const svsdf_mid_config *c) {
    host::MidEndConfig d;
    if (!c) return d;
    d.rho_mid_end = c->rho_mid_end; d.vmax = c->vmax; d.omgmax = c->omgmax; d.weight_v = c->weight_v; d.weight_omg = c->weight_omg;
    d.weight_pr = c->weight_pr; d.weight_ar = c->weight_ar; d.smoothingEps = c->smoothingEps; d.integralIntervs = c->integralIntervs;
    d.vehicleMass = c->vehicleMass; d.gravAcc = c->gravAcc; d.horizDrag = c->horizDrag; d.vertDrag = c->vertDrag; d.parasDrag = c->parasDrag;
    d.speedEps = c->speedEps; d.mem_size = c->mem_size; d.past = c->past; d.min_step = c->min_step; d.g_epsilon = c->g_epsilon;
    d.relCostTolMidEnd = c->relCostTolMidEnd; d.max_iterations = c->max_iterations; d.cancel_after = c->cancel_after; d.solver = c->solver;
    return d;
}
static bool mid_args_ok(const svsdf_mid_config *c, int N, const double *initS, const double *finalS, const double *Q, const double *rot) {
    return N >= 2 && N <= kMaxPieces && initS && finalS && Q && rot && (!c || (c->integralIntervs >= 1 && c->smoothingEps > 0.0 && c->vehicleMass > 0.0));
}
int svsdf_mid_cost(const svsdf_mid_config *cfg, int N, const double *initS, const double *finalS, const double *Q, const double *rot_list,
                   const double *x, double *cost_out, double *grad_out) {
    if (!mid_args_ok(cfg, N, initS, finalS, Q, rot_list) || !x || !cost_out || !grad_out) return SVSDF_ERR_INVALID;
    host::MidEnd M(mid_cfg(cfg));
    M.setup(initS, finalS, N, Q, rot_list);
    *cost_out = M.cost(x, grad_out);
    return SVSDF_OK;
}
int svsdf_mid_get_ori_traj(const svsdf_mid_config *cfg, int N, const double *initS, const double *finalS, const double *Q,
                           const double *T_init, const double *rot_list, double *opt_x_out, double *T_out, double *coeffs_out,
                           double *final_cost_out, int *iterations_out) {
    if (!mid_args_ok(cfg, N, initS, finalS, Q, rot_list) || !T_init || !opt_x_out) return SVSDF_ERR_INVALID;
    for (int i = 0; i < N; ++i)
        if (!(T_init[i] > 0.0)) return SVSDF_ERR_INVALID;
    host::MidEnd M(mid_cfg(cfg));
    M.setup(initS, finalS, N, Q, rot_list);
    return M.optimize(T_init, opt_x_out, T_out, coeffs_out, final_cost_out, iterations_out);
}

// ---------------------------------------------------------------------------------------------------------------------
// K5: collision kernels of the A* front end (csrc/svsdf_frontend.cu)
// ---------------------------------------------------------------------------------------------------------------------
int svsdf_front_init(svsdf_ctx *ctx, int kernel_size, int kernel_yaw_num, double occupancy_resolution, double front_end_safeh) {
    if (!ctx) return SVSDF_ERR_INVALID;
    if (kernel_size < 1 || kernel_size > kMaxKernelSize || (kernel_size % 2) == 0 || kernel_yaw_num < 1 || kernel_yaw_num > kMaxYawKernels ||
        !(occupancy_resolution > 0.0)) {
        ctx->err = "svsdf_front_init: kernel_size must be odd and <= 32, 1 <= kernel_yaw_num <= 64, resolution > 0";
        return SVSDF_ERR_INVALID;
    }
    if (ctx->shape.id == SH_POLYGON || ctx->shape.id == SH_MESH) {
        ctx->err = "svsdf_front_init: the reference defines no rotated kernels for the Polygon / mesh functors (Shape.hpp:1477 vs :267)";
        return SVSDF_ERR_INVALID;
    }
    CK(cudaSetDevice(ctx->device));
    ctx->front_ready = false;
    FrontParams F{};
    F.kernel_size = kernel_size;
    F.kernel_count = kernel_yaw_num;
    F.res = occupancy_resolution;
    F.safemargin = std::max(front_end_safeh, occupancy_resolution / 2);  // Shape.hpp:399
    const double PI = 3.14159265358979323846;                             // Shape.hpp:31
    const double yaw_res = 2 * PI / kernel_yaw_num;
    ctx->front_yaw.assign(kernel_yaw_num, 0.0);
    int ind = 0;
    for (double yaw = -PI; yaw < PI && ind < kernel_yaw_num; yaw += yaw_res, ind++) ctx->front_yaw[ind] = yaw;  // :401
    const int K = kernel_yaw_num, ks = kernel_size, bpr = (ks + 7) / 8;
    double *d_yaw = nullptr;
    unsigned char *d_cells = nullptr;
    CK(cudaMalloc(&d_yaw, K * sizeof(double)));
    cudaError_t e = cudaMalloc(&d_cells, (size_t)K * ks * ks);
    if (e != cudaSuccess) { cudaFree(d_yaw); ctx->err = cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
    ctx->front_cells.assign((size_t)K * ks * ks, 0);
    e = cudaMemcpyAsync(d_yaw, ctx->front_yaw.data(), K * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_front_cells(ctx->shape, F, d_yaw, d_cells, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->front_cells.data(), d_cells, ctx->front_cells.size(), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_yaw); cudaFree(d_cells);
    if (e != cudaSuccess) { ctx->err = std::string("svsdf_front_init: ") + cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
    ctx->launches += 1;
    // generateByteKernel (Shape.hpp:194-216) + the same rows as 32-bit masks (bit 31 - b <-> column b)
    static const unsigned char or_mask[8] = {0x80, 0x40, 0x20, 0x10, 0x08, 0x04, 0x02, 0x01};
    ctx->front_bytes.assign((size_t)K * ks * bpr, 0);
    std::vector<unsigned> rowmask((size_t)K * ks, 0u);
    for (int k = 0; k < K; ++k)
        for (int a = 0; a < ks; ++a)
            for (int b = 0; b < ks; ++b)
                if (ctx->front_cells[((size_t)k * ks + a) * ks + b]) {
                    ctx->front_bytes[((size_t)k * ks + a) * bpr + b / 8] |= or_mask[b % 8];
                    rowmask[(size_t)k * ks + a] |= 0x80000000u >> b;
                }
    cudaFree(ctx->d_front_bytes); cudaFree(ctx->d_front_rowmask);
    ctx->d_front_bytes = nullptr; ctx->d_front_rowmask = nullptr;
    CK(cudaMalloc(&ctx->d_front_bytes, ctx->front_bytes.size()));
    CK(cudaMalloc(&ctx->d_front_rowmask, rowmask.size() * sizeof(unsigned)));
    CK(cudaMemcpy(ctx->d_front_bytes, ctx->front_bytes.data(), ctx->front_bytes.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->d_front_rowmask, rowmask.data(), rowmask.size() * sizeof(unsigned), cudaMemcpyHostToDevice));
    ctx->front = F;
    ctx->front_ready = true;
    return SVSDF_OK;
}

int svsdf_front_get_kernels(svsdf_ctx *ctx, double *yaw_out, unsigned char *cells_out, unsigned char *bytes_out) {
    if (!ctx) return SVSDF_ERR_INVALID;
    if (!ctx->front_ready) { ctx->err = "svsdf_front_get_kernels: call svsdf_front_init first"; return SVSDF_ERR_NOT_READY; }
    if (yaw_out) std::memcpy(yaw_out, ctx->front_yaw.data(), ctx->front_yaw.size() * sizeof(double));
    if (cells_out) std::memcpy(cells_out, ctx->front_cells.data(), ctx->front_cells.size());
    if (bytes_out) std::memcpy(bytes_out, ctx->front_bytes.data(), ctx->front_bytes.size());
    return SVSDF_OK;
}

static int front_scratch(svsdf_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->cap_front_scratch) return SVSDF_OK;
    cudaFree(ctx->d_front_scratch);
    ctx->d_front_scratch = nullptr;
    ctx->cap_front_scratch = 0;
    const size_t cap = bytes + bytes / 2 + 4096;
    CK(cudaMalloc(&ctx->d_front_scratch, cap));
    ctx->cap_front_scratch = cap;
    return SVSDF_OK;
}

static int front_params_with_map(svsdf_ctx *ctx, FrontParams &F, const char *who) {
    if (!ctx->front_ready) { ctx->err = std::string(who) + ": call svsdf_front_init first"; return SVSDF_ERR_NOT_READY; }
    if (!ctx->d_map) { ctx->err = std::string(who) + ": map not set (svsdf_set_map)"; return SVSDF_ERR_NOT_READY; }
    F = ctx->front;
    F.X = ctx->map_X; F.Y = ctx->map_Y; F.h = ctx->map_h; F.row_bytes = ctx->map_row_bytes;
    F.out_words = (ctx->map_Y + 31) / 32;
    F.ox = ctx->map_ox; F.oy = ctx->map_oy; F.map_res = ctx->map_res;
    if (F.h != (F.kernel_size - 1) / 2) {
        ctx->err = std::string(who) + ": the map was packed for another kernel_size (its inflation must be (kernel_size - 1) / 2)";
        return SVSDF_ERR_INVALID;
    }
    if (F.res != F.map_res) {  // the reference has ONE conf.occupancy_resolution for the map and the shape kernels
        ctx->err = std::string(who) + ": svsdf_front_init's occupancy_resolution differs from the map resolution";
        return SVSDF_ERR_INVALID;
    }
    return SVSDF_OK;
}

int svsdf_front_cspace(svsdf_ctx *ctx, uint32_t *words_out, float *ms_out, const uint32_t **dev_words_out) {
    if (!ctx) return SVSDF_ERR_INVALID;
    FrontParams F;
    int rc = front_params_with_map(ctx, F, "svsdf_front_cspace");
    if (rc != SVSDF_OK) return rc;
    CK(cudaSetDevice(ctx->device));
    const size_t n = (size_t)F.kernel_count * F.X * F.out_words;
    if (n > ctx->cap_cspace) {
        cudaFree(ctx->d_cspace);
        ctx->d_cspace = nullptr;
        ctx->cap_cspace = 0;
        CK(cudaMalloc(&ctx->d_cspace, n * sizeof(unsigned)));
        ctx->cap_cspace = n;
    }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(launch_front_cspace(F, ctx->d_map, ctx->d_front_rowmask, ctx->d_cspace, ctx->stream));
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->launches += 1;
    if (words_out) CK(cudaMemcpyAsync(words_out, ctx->d_cspace, n * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ms_out) CK(cudaEventElapsedTime(ms_out, ctx->ev0, ctx->ev1));
    if (dev_words_out) *dev_words_out = ctx->d_cspace;
    return SVSDF_OK;
}

int svsdf_front_expand(svsdf_ctx *ctx, int64_t n, const int32_t *node_ij, const double *node_yaw, unsigned char *ok_out, double *child_yaw_out,
                       unsigned char *parts_out) {
    if (!ctx || n < 0 || (n > 0 && (!node_ij || !node_yaw || !ok_out || !child_yaw_out))) return SVSDF_ERR_INVALID;
    FrontParams F;
    int rc = front_params_with_map(ctx, F, "svsdf_front_expand");
    if (rc != SVSDF_OK) return rc;
    if (n == 0) return SVSDF_OK;
    for (int64_t i = 0; i < n; ++i)
        if (node_ij[2 * i] < 0 || node_ij[2 * i] >= F.X || node_ij[2 * i + 1] < 0 || node_ij[2 * i + 1] >= F.Y) {
            ctx->err = "svsdf_front_expand: node index outside the map";
            return SVSDF_ERR_INVALID;
        }
    SubSwParams P{};
    P.half_box = (double)(F.kernel_size / 2 + 1);
    for (double kt = 0.0; kt <= 1.0 && P.nkt < 64; kt += 0.02) P.kt[P.nkt++] = kt;  // sw_manager.hpp:1190
    CK(cudaSetDevice(ctx->device));
    // One device scratch block and a pinned mirror of it: outputs first (child yaws [9n] f64 | ok [9n] | parts [9n], padded to
    // 8 bytes), then inputs (father yaws [n] f64 | node indices [2n] i32) — one copy in, one launch, one copy out.
    const size_t un = (size_t)n;
    const size_t out_bytes = (9 * un * 8 + 18 * un + 7) & ~(size_t)7, in_bytes = un * 8 + 2 * un * 4;
    rc = front_scratch(ctx, out_bytes + in_bytes + 64);
    if (rc != SVSDF_OK) return rc;
    rc = ensure_stage(ctx, out_bytes + in_bytes + 64);
    if (rc != SVSDF_OK) return rc;
    unsigned char *hb = reinterpret_cast<unsigned char *>(ctx->h_stage), *db = ctx->d_front_scratch;
    double *d_cy = reinterpret_cast<double *>(db);
    unsigned char *d_ok = db + 9 * un * 8, *d_parts = d_ok + 9 * un;
    double *d_fy = reinterpret_cast<double *>(db + out_bytes);
    int *d_ij = reinterpret_cast<int *>(db + out_bytes + un * 8);
    std::memcpy(hb + out_bytes, node_yaw, un * 8);
    std::memcpy(hb + out_bytes + un * 8, node_ij, 2 * un * 4);
    cudaError_t e = cudaMemcpyAsync(db + out_bytes, hb + out_bytes, in_bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_front_expand(ctx->shape, F, P, ctx->d_map, ctx->d_front_bytes, n, d_ij, d_fy, d_ok, d_cy, d_parts, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hb, db, out_bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) {
        std::memcpy(child_yaw_out, hb, 9 * un * 8);
        std::memcpy(ok_out, hb + 9 * un * 8, 9 * un);
        if (parts_out) std::memcpy(parts_out, hb + 9 * un * 8 + 9 * un, 9 * un);
    }
    if (e != cudaSuccess) { ctx->err = std::string("svsdf_front_expand: ") + cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
    ctx->launches += 1;
    return SVSDF_OK;
}

int svsdf_front_astar(svsdf_ctx *ctx, int n, const double *start_xy, const double *goal_xy, int max_path, double *paths_out, int32_t *len_out,
                      int32_t *expansions_out, int64_t *rounds_out) {
    if (!ctx || n < 0 || max_path < 1 || (n > 0 && (!start_xy || !goal_xy || !paths_out || !len_out))) return SVSDF_ERR_INVALID;
    FrontParams F;
    int rc = front_params_with_map(ctx, F, "svsdf_front_astar");
    if (rc != SVSDF_OK) return rc;
    host::AstarGrid G;
    G.X = F.X; G.Y = F.Y; G.ox = F.ox; G.oy = F.oy; G.res = F.map_res;
    host::AstarStats stats;
    auto expand = [&](int m, const int32_t *ij, const double *yaw, unsigned char *ok, double *cyaw) {
        return svsdf_front_expand(ctx, m, ij, yaw, ok, cyaw, nullptr);
    };
    rc = host::astar_batch(G, n, start_xy, goal_xy, max_path, paths_out, len_out, expansions_out, (int64_t)1 << 40, expand, &stats);
    if (rounds_out) *rounds_out = stats.rounds;
    return rc;
}

int svsdf_front_check_kernel_value(svsdf_ctx *ctx, int64_t n, const double *father_yaw, const int32_t *ind_xy, unsigned char *ok_out,
                                   double *child_yaw_out) {
    if (!ctx || n < 0 || (n > 0 && (!father_yaw || !ind_xy || !ok_out || !child_yaw_out))) return SVSDF_ERR_INVALID;
    FrontParams F;
    int rc = front_params_with_map(ctx, F, "svsdf_front_check_kernel_value");
    if (rc != SVSDF_OK) return rc;
    if (n == 0) return SVSDF_OK;
    for (int64_t i = 0; i < n; ++i)
        if (ind_xy[2 * i] < 0 || ind_xy[2 * i] >= F.X || ind_xy[2 * i + 1] < 0 || ind_xy[2 * i + 1] >= F.Y) {
            ctx->err = "svsdf_front_check_kernel_value: cell index outside the map";
            return SVSDF_ERR_INVALID;
        }
    CK(cudaSetDevice(ctx->device));
    const size_t un = (size_t)n;
    rc = front_scratch(ctx, un * 8 + un * 8 + 2 * un * 4 + un + 64);
    if (rc != SVSDF_OK) return rc;
    double *d_fy = reinterpret_cast<double *>(ctx->d_front_scratch);
    double *d_cy = d_fy + un;
    int *d_ind = reinterpret_cast<int *>(d_cy + un);
    unsigned char *d_ok = reinterpret_cast<unsigned char *>(d_ind + 2 * un);
    cudaError_t e = cudaMemcpyAsync(d_fy, father_yaw, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ind, ind_xy, 2 * n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_front_check(F, ctx->d_map, ctx->d_front_bytes, n, d_fy, d_ind, d_ok, d_cy, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ok_out, d_ok, n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(child_yaw_out, d_cy, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->err = std::string("svsdf_front_check_kernel_value: ") + cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
    ctx->launches += 1;
    return SVSDF_OK;
}

int svsdf_create(const svsdf_config *cfg, svsdf_ctx **out) {
    if (!cfg || !out) return SVSDF_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SVSDF_ERR_CUDA;  // no CPU fallback
    if (cfg->device < 0 || cfg->device >= ndev) return SVSDF_ERR_INVALID;
    if (cfg->polygon_xy && (cfg->polygon_n < 3 || cfg->polygon_n > kMaxPolyEdges)) return SVSDF_ERR_INVALID;
    if (cfg->mesh_nf < 0 || cfg->mesh_nv < 0 || cfg->mesh_nf > kMaxMeshFaces) return SVSDF_ERR_INVALID;
    if (cfg->mesh_nf > 0) {
        if (!cfg->mesh_faces || !cfg->mesh_vertices || cfg->mesh_nv < 3) return SVSDF_ERR_INVALID;
        for (int64_t k = 0; k < 3 * (int64_t)cfg->mesh_nf; ++k)
            if (cfg->mesh_faces[k] < 0 || cfg->mesh_faces[k] >= cfg->mesh_nv) return SVSDF_ERR_INVALID;
    }
    svsdf_ctx *ctx = new svsdf_ctx();
    ctx->cfg = *cfg;
    ctx->shape_name = cfg->shape ? cfg->shape : "";
    ctx->cfg.shape = ctx->shape_name.c_str();
    build_shape(*cfg, ctx->shape);
    ctx->cp.weight_p = cfg->weight_p;
    ctx->cp.safety_hor = cfg->safety_hor;
    ctx->rho = cfg->rho;
    ctx->device = cfg->device;
    ctx->strict = cfg->strict_fp != 0;
    if (const char *fg = std::getenv("SVSDF_FORCE_GRID_OUTER")) ctx->force_grid_outer = std::atoi(fg);
    if (const char *fb = std::getenv("SVSDF_FORCE_BATCHED")) ctx->force_batched = std::atoi(fb);
    auto fail = [&](cudaError_t e) {
        std::fprintf(stderr, "svsdf_create: %s\n", cudaGetErrorString(e));
        svsdf_destroy(ctx);
        return SVSDF_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(ctx->device)) != cudaSuccess) return fail(e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, ctx->device)) != cudaSuccess) return fail(e);
    if (prop.major < 10) {
        std::fprintf(stderr, "svsdf_create: device sm_%d%d is not Blackwell (kernels are built for sm_100a only)\n",
                     prop.major, prop.minor);
        svsdf_destroy(ctx);
        return SVSDF_ERR_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(e);
    if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return fail(e);
    if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return fail(e);
    for (int k = 0; k < 5; ++k)
        if ((e = cudaEventCreate(&ctx->evk[k])) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&ctx->d_n_inside, sizeof(int))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&ctx->d_eval_counter, sizeof(unsigned long long))) != cudaSuccess) return fail(e);
    if ((e = cudaMalloc(&ctx->d_ticket, sizeof(unsigned int))) != cudaSuccess) return fail(e);
    cudaMemset(ctx->d_ticket, 0, sizeof(unsigned int));
    cudaMemset(ctx->d_n_inside, 0, sizeof(int));
    cudaMemset(ctx->d_eval_counter, 0, sizeof(unsigned long long));
    ctx->cfg.mesh_vertices = nullptr;  // caller's arrays are not kept
    ctx->cfg.mesh_faces = nullptr;
    ctx->cfg.polygon_xy = nullptr;
    if (ctx->shape.id == SH_MESH) {
        // BasicShape ctor (Shape.hpp:285-309): every vertex becomes R v + trans, then the per-face soup
        const ShapeParams &S = ctx->shape;
        const double R[3][3] = {{S.rot[0], S.rot[1], 0.0}, {S.rot[2], S.rot[3], 0.0}, {0.0, 0.0, 1.0}};
        const double tr[3] = {S.trans[0], S.trans[1], 0.0};
        std::vector<double> tri((size_t)cfg->mesh_nf * kMeshStride);
        for (int f = 0; f < cfg->mesh_nf; ++f) {
            double *rec = &tri[(size_t)f * kMeshStride];
            for (int k = 0; k < 3; ++k) {
                const double *v = cfg->mesh_vertices + 3 * (size_t)cfg->mesh_faces[3 * f + k];
                for (int j = 0; j < 3; ++j)
                    rec[3 * k + j] = ((v[0] * R[j][0] + v[1] * R[j][1]) + v[2] * R[j][2]) + tr[j];
            }
            // rmax: farthest point of the face from vertex a (one of the other two vertices), padded upwards
            const double ab = std::sqrt((rec[3] - rec[0]) * (rec[3] - rec[0]) + (rec[4] - rec[1]) * (rec[4] - rec[1]) + (rec[5] - rec[2]) * (rec[5] - rec[2]));
            const double ac = std::sqrt((rec[6] - rec[0]) * (rec[6] - rec[0]) + (rec[7] - rec[1]) * (rec[7] - rec[1]) + (rec[8] - rec[2]) * (rec[8] - rec[2]));
            rec[9] = std::max(ab, ac) * (1.0 + 1e-12) + 1e-300;
        }
        if ((e = cudaMalloc(&ctx->d_mesh_tri, tri.size() * sizeof(double))) != cudaSuccess) return fail(e);
        if ((e = cudaMemcpy(ctx->d_mesh_tri, tri.data(), tri.size() * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess) return fail(e);
        ctx->shape.mesh_tri = ctx->d_mesh_tri;
        ctx->shape.mesh_nf = cfg->mesh_nf;
        ctx->shape.has_xform = 0;
        // the winding-number hierarchy over the SAME transformed vertices (fast_winding_number.cpp:380-408 is handed V after
        // the ctor's transform, Shape.hpp:303-309), built on the host and uploaded as four flat arrays
        std::vector<double> Vt((size_t)cfg->mesh_nv * 3);
        for (int i = 0; i < cfg->mesh_nv; ++i) {
            const double *v = cfg->mesh_vertices + 3 * (size_t)i;
            for (int j = 0; j < 3; ++j) Vt[3 * (size_t)i + j] = ((v[0] * R[j][0] + v[1] * R[j][1]) + v[2] * R[j][2]) + tr[j];
        }
        host::FwnBvh B;
        B.build(Vt.data(), cfg->mesh_nv, cfg->mesh_faces, cfg->mesh_nf);
        if (B.nn < 1 || B.depth() > kFwnMaxDepth) {
            ctx->err = "svsdf_create: mesh hierarchy deeper than kFwnMaxDepth";
            svsdf_destroy(ctx);
            return SVSDF_ERR_INVALID;
        }
        // child boxes for the closest-triangle descent: lo x, lo y, hi x, hi y two ulps outwards (the float boxes then contain
        // the double vertices), squared z gap to the query plane z = 0 rounded down, pad
        std::vector<float> cb(B.cbox.size(), 0.0f);
        float boxmag = 0.0f;
        {
            const float ninf = -std::numeric_limits<float>::infinity(), pinf = std::numeric_limits<float>::infinity();
            auto out = [&](float v, float dir) { return std::isfinite(v) ? std::nextafter(std::nextafter(v, dir), dir) : v; };
            for (size_t k = 0; k + 5 < cb.size(); k += 6) {
                const float *b = &B.cbox[k];  // min xyz, max xyz
                const float lox = out(b[0], ninf), loy = out(b[1], ninf), loz = out(b[2], ninf), hix = out(b[3], pinf), hiy = out(b[4], pinf),
                            hiz = out(b[5], pinf);
                cb[k] = lox; cb[k + 1] = loy; cb[k + 2] = hix; cb[k + 3] = hiy;
                const double gz = std::max(std::max((double)loz, -(double)hiz), 0.0);
                float dz2 = (float)(gz * gz);
                if ((double)dz2 > gz * gz) dz2 = std::nextafter(dz2, 0.0f);
                cb[k + 4] = std::isfinite(dz2) ? dz2 : 0.0f;
                for (int j = 0; j < 4; ++j)
                    if (std::isfinite(cb[k + j])) boxmag = std::max(boxmag, std::fabs(cb[k + j]));
            }
        }
        ctx->shape.fwn_boxmag = boxmag;
        std::vector<float> tf((size_t)cfg->mesh_nf * 12, 0.0f);
        for (int f = 0; f < cfg->mesh_nf; ++f)
            for (int k = 0; k < 3; ++k)
                for (int j = 0; j < 3; ++j) tf[12 * (size_t)f + 3 * k + j] = B.U[3 * (size_t)B.F[3 * f + k] + j];
        const size_t b_child = B.child.size() * sizeof(uint32_t), b_data = B.data.size() * sizeof(float), b_box = cb.size() * sizeof(float),
                     b_tri = tf.size() * sizeof(float);
        auto up = [&](void **dst, const void *src, size_t bytes) -> cudaError_t {
            cudaError_t e2 = cudaMalloc(dst, bytes);
            if (e2 != cudaSuccess) return e2;
            return cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
        };
        if ((e = up((void **)&ctx->d_fwn_child, B.child.data(), b_child)) != cudaSuccess) return fail(e);
        if ((e = up((void **)&ctx->d_fwn_data, B.data.data(), b_data)) != cudaSuccess) return fail(e);
        if ((e = up((void **)&ctx->d_fwn_cbox, cb.data(), b_box)) != cudaSuccess) return fail(e);
        if ((e = up((void **)&ctx->d_fwn_trif, tf.data(), b_tri)) != cudaSuccess) return fail(e);
        // Far-field bound for choiceTInit's layer-1 pruning (thread_choice_t_init): sdf = (1 - 2 w) d with d >= |q| - Rv (Rv: the
        // largest vertex norm; the query has z = 0, the origin is the body origin).  Beyond rho0 = max_i(|P_i| + 2 sqrt(maxPDist2_i))
        // none of the root's children is entered, w is the sum of their four expansions / (4 pi), and each expansion is bounded
        // term by term through the magnitudes of its coefficients (|q^| <= 1 componentwise) and |q - P_i| >= rho0 - |P_i|:
        //   |order 0| <= |N|_1 m^2,  |order 1| <= (|tr| + 3 (sum of |Nij| rows)) m^3,  |order 2| <= (1.5 A + 7.5 B) m^4,  m = 1 / (rho0 - |P_i|).
        // With omega that bound (padded 2 % for the float rounding of the evaluation), sdf >= (1 - 2 omega)(|q| - Rv) for |q| >= rho0.
        {
            double Rv = 0.0;
            for (int i = 0; i < cfg->mesh_nv; ++i)
                Rv = std::max(Rv, std::sqrt(Vt[3 * (size_t)i] * Vt[3 * (size_t)i] + Vt[3 * (size_t)i + 1] * Vt[3 * (size_t)i + 1] + Vt[3 * (size_t)i + 2] * Vt[3 * (size_t)i + 2]));
            double rho0 = 0.0;
            int nchild = 0;
            for (int i = 0; i < 4; ++i) {
                if (B.child[i] == host::FwnBvh::EMPTY) break;
                ++nchild;
                const double Pn = std::sqrt((double)B.row(0, 1)[i] * B.row(0, 1)[i] + (double)B.row(0, 2)[i] * B.row(0, 2)[i] + (double)B.row(0, 3)[i] * B.row(0, 3)[i]);
                rho0 = std::max(rho0, Pn + 2.0 * std::sqrt(std::max(0.0, (double)B.row(0, 0)[i])));
            }
            rho0 = std::max(rho0, Rv) * (1.0 + 1e-4) + 1e-6;
            double omega = 0.0;
            bool finite = std::isfinite(rho0);
            for (int i = 0; i < nchild && finite; ++i) {
                auto a = [&](int r) { return std::fabs((double)B.row(0, r)[i]); };
                const double Pn = std::sqrt((double)B.row(0, 1)[i] * B.row(0, 1)[i] + (double)B.row(0, 2)[i] * B.row(0, 2)[i] + (double)B.row(0, 3)[i] * B.row(0, 3)[i]);
                const double m = 1.0 / (rho0 - Pn);
                const double A0 = a(4) + a(5) + a(6);
                const double A1 = std::fabs((double)B.row(0, 7)[i] + B.row(0, 8)[i] + B.row(0, 9)[i]) + 3.0 * (a(7) + a(8) + a(9) + a(10) + a(11) + a(12));
                const double t0 = std::fabs((double)B.row(0, 20)[i] + B.row(0, 21)[i]) + std::fabs((double)B.row(0, 22)[i] + B.row(0, 17)[i]) +
                                  std::fabs((double)B.row(0, 18)[i] + B.row(0, 19)[i]);
                const double t1 = a(17) + a(18) + a(19) + a(20) + a(21) + a(22);
                const double A2 = 1.5 * (3.0 * (a(13) + a(14) + a(15)) + t0) + 7.5 * (a(13) + a(14) + a(15) + a(16) + t1);
                omega += A0 * m * m + A1 * m * m * m + A2 * m * m * m * m;
                finite = finite && std::isfinite(omega);
            }
            omega = omega / (4.0 * 3.14159265358979323846) * 1.02 + 1e-6;
            if (finite && omega < 0.45) {
                ctx->shape.rout = Rv * (1.0 + 1e-9) + 1e-9;
                ctx->shape.prune_scale = 1.0 / (1.0 - 2.0 * omega);
                ctx->shape.prune_rmin = rho0;
            }
        }
        ctx->shape.fwn_nn = B.nn;
        ctx->shape.fwn_child = ctx->d_fwn_child;
        ctx->shape.fwn_data = ctx->d_fwn_data;
        ctx->shape.fwn_cbox = ctx->d_fwn_cbox;
        ctx->shape.fwn_trif = ctx->d_fwn_trif;
    }
    *out = ctx;
    return SVSDF_OK;
}

void svsdf_destroy(svsdf_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->own_points) cudaFree(ctx->d_points);
    cudaFree(ctx->d_mesh_tri); cudaFree(ctx->d_fwn_child); cudaFree(ctx->d_fwn_data); cudaFree(ctx->d_fwn_cbox); cudaFree(ctx->d_fwn_trif);
    cudaFree(ctx->d_front_bytes); cudaFree(ctx->d_front_rowmask); cudaFree(ctx->d_cspace); cudaFree(ctx->d_front_scratch);
    cudaFree(ctx->d_flag); cudaFree(ctx->d_inside_tstar); cudaFree(ctx->d_inside_list);
    cudaFree(ctx->d_gsip_contrib); cudaFree(ctx->d_gsip_piece); cudaFree(ctx->d_n_inside);
    cudaFree(ctx->d_eval_counter); cudaFree(ctx->d_tot); cudaFree(ctx->d_ticket); cudaFree(ctx->d_blob); cudaFree(ctx->d_partials); cudaFree(ctx->d_out);
    cudaFree(ctx->d_q_points); cudaFree(ctx->d_q_sdf); cudaFree(ctx->d_q_ts); cudaFree(ctx->d_q_grad);
    cudaFree(ctx->d_q_rounds);
    if (ctx->own_map) cudaFree(ctx->d_map);
    cudaFree(ctx->d_block_counts); cudaFree(ctx->d_n_total);
    if (ctx->h_blob) cudaFreeHost(ctx->h_blob);
    if (ctx->h_out) cudaFreeHost(ctx->h_out);
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    if (ctx->h_pts_stage) cudaFreeHost(ctx->h_pts_stage);
    if (ctx->ev_pts) cudaEventDestroy(ctx->ev_pts);
    if (ctx->lmbm) svsdf_lmbm_close(ctx->lmbm);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (int k = 0; k < 5; ++k)
        if (ctx->evk[k]) cudaEventDestroy(ctx->evk[k]);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *svsdf_last_error(const svsdf_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int svsdf_set_points(svsdf_ctx *ctx, const double *pts, int64_t P, int stride) {
    if (!ctx || P < 0 || stride < 2 || (P > 0 && !pts)) return SVSDF_ERR_INVALID;
    if (P > 2000000000LL) { ctx->err = "svsdf: too many points"; return SVSDF_ERR_INVALID; }
    CK(cudaSetDevice(ctx->device));
    if (!ctx->own_points) { ctx->d_points = nullptr; ctx->own_points = true; ctx->cap_points = 0; }
    if (P > ctx->cap_points) {
        cudaFree(ctx->d_points);
        ctx->d_points = nullptr;
        ctx->cap_points = 0;
        CK(cudaMalloc(&ctx->d_points, (size_t)(P + 1024) * 2 * sizeof(double)));
        ctx->cap_points = P + 1024;
    }
    if (!ctx->d_points) {  // P == 0 and nothing allocated yet
        CK(cudaMalloc(&ctx->d_points, 1024 * 2 * sizeof(double)));
        ctx->cap_points = 1024;
    }
    if (ctx->pts_inflight) {  // the previous upload still reads the stage
        CK(cudaEventSynchronize(ctx->ev_pts));
        ctx->pts_inflight = false;
    }
    if (!ctx->ev_pts) CK(cudaEventCreateWithFlags(&ctx->ev_pts, cudaEventDisableTiming));
    const size_t need = (size_t)P * 2 * sizeof(double);
    if (need > ctx->cap_pts_stage) {
        if (ctx->h_pts_stage) cudaFreeHost(ctx->h_pts_stage);
        ctx->h_pts_stage = nullptr;
        ctx->cap_pts_stage = 0;
        const size_t cap = need + need / 4 + 4096;
        CK(cudaMallocHost(&ctx->h_pts_stage, cap));
        ctx->cap_pts_stage = cap;
    }
    int rc = SVSDF_OK;
    double *h = ctx->h_pts_stage;
    // pos_eva(2) = 0 (back_end_optimizer.hpp:791): only x, y are kept.  Packed into the pinned stage chunk by chunk by a few
    // host threads; every chunk is handed to the copy engine as soon as it is packed (packing of the next chunks overlaps the
    // DMA of the finished ones).  One thread for small inputs.
    const int64_t chunk = 16384;
    const int64_t nchunks = (P + chunk - 1) / chunk;
    int nth = (int)std::min<int64_t>(nchunks, 4);
#ifdef _OPENMP
    nth = std::max(1, std::min(nth, omp_get_num_procs()));  // not omp_get_max_threads(): launchers set OMP_NUM_THREADS = 1 per rank
#else
    nth = 1;
#endif
    int first_err = (int)cudaSuccess;
    const int dev = ctx->device;
    double *d_points = ctx->d_points;
    cudaStream_t stream = ctx->stream;
#pragma omp parallel num_threads(nth) if (nth > 1)
    {
        if (nth > 1) cudaSetDevice(dev);  // the worker threads' current device
#pragma omp for schedule(dynamic, 1)
        for (int64_t c = 0; c < nchunks; ++c) {
            const int64_t b = c * chunk, e = std::min(P, b + chunk);
            if (stride == 2) {
                std::memcpy(h + 2 * b, pts + 2 * b, (size_t)(e - b) * 2 * sizeof(double));
            } else {
                for (int64_t i = b; i < e; ++i) {
                    h[2 * i] = pts[i * stride];
                    h[2 * i + 1] = pts[i * stride + 1];
                }
            }
            cudaError_t ce = cudaMemcpyAsync(d_points + 2 * b, h + 2 * b, (size_t)(e - b) * 2 * sizeof(double), cudaMemcpyHostToDevice, stream);
            if (ce != cudaSuccess) {
#pragma omp atomic write
                first_err = (int)ce;
            }
        }
    }
    if (first_err != (int)cudaSuccess) {
        ctx->err = std::string("svsdf_set_points: cudaMemcpyAsync: ") + cudaGetErrorString((cudaError_t)first_err);
        return SVSDF_ERR_CUDA;
    }
    CK(cudaEventRecord(ctx->ev_pts, ctx->stream));  // no wait here: see ev_pts
    ctx->pts_inflight = true;
    ctx->P = P;
    ctx->last_n_inside = -1;
    (void)rc;
    return ensure_scratch(ctx, P);
}

int svsdf_set_points_device(svsdf_ctx *ctx, const double *dev_xy, int64_t P) {
    if (!ctx || P < 0 || (P > 0 && !dev_xy)) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (ctx->own_points) cudaFree(ctx->d_points);
    ctx->d_points = const_cast<double *>(dev_xy);
    ctx->own_points = false;
    ctx->cap_points = 0;
    ctx->P = P;
    return ensure_scratch(ctx, P);
}

int svsdf_device_ptr_points(svsdf_ctx *ctx, const double **dev_xy) {
    if (!ctx || !dev_xy) return SVSDF_ERR_INVALID;
    if (ctx->pts_inflight) {  // the pointer may be used on other streams: the upload has to be complete
        CK(cudaSetDevice(ctx->device));
        CK(cudaEventSynchronize(ctx->ev_pts));
        ctx->pts_inflight = false;
    }
    *dev_xy = ctx->d_points;
    return SVSDF_OK;
}

int svsdf_set_scale(svsdf_ctx *ctx, const svsdf_scale *spec) {
    if (!ctx) return SVSDF_ERR_INVALID;
    if (!spec) {
        ctx->scaled = false;
        return SVSDF_OK;
    }
    ScaleParams Z{};
    for (int ax = 0; ax < 2; ++ax) {
        const int n = spec->n_terms[ax];
        if (n < 0 || n > kMaxScaleTerms) {
            ctx->err = "svsdf_set_scale: n_terms must be in [0, 4]";
            return SVSDF_ERR_INVALID;
        }
        double amp = 0.0;
        bool finite = std::isfinite(spec->c[ax]);
        for (int k = 0; k < n; ++k)
            finite = finite && std::isfinite(spec->a[ax][k]) && std::isfinite(spec->w[ax][k]) && std::isfinite(spec->phi[ax][k]);
        if (!finite) {
            ctx->err = "svsdf_set_scale: non-finite entry";
            return SVSDF_ERR_INVALID;
        }
        for (int k = 0; k < n; ++k) amp += std::fabs(spec->a[ax][k]);
        // the scale must stay positive at every t: S^-1 is singular where an axis reaches 0
        if (!(spec->c[ax] - amp > 0.0)) {
            ctx->err = "svsdf_set_scale: c - sum |a_k| must be > 0 on both axes";
            return SVSDF_ERR_INVALID;
        }
        Z.n[ax] = n;
        Z.c[ax] = spec->c[ax];
        for (int k = 0; k < n; ++k) {
            Z.a[ax][k] = spec->a[ax][k];
            Z.w[ax][k] = spec->w[ax][k];
            Z.phi[ax][k] = spec->phi[ax][k];
        }
    }
    if (spec->exact_yaw_grad != 0 && spec->exact_yaw_grad != 1) {
        ctx->err = "svsdf_set_scale: exact_yaw_grad must be 0 or 1";
        return SVSDF_ERR_INVALID;
    }
    Z.exact_yaw_grad = spec->exact_yaw_grad;
    ctx->scale = Z;
    ctx->scaled = true;
    return SVSDF_OK;
}

int svsdf_set_traj(svsdf_ctx *ctx, int N, const double *T, const double *coeffs) {
    if (!ctx) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = upload_traj(ctx, N, T, coeffs);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    return SVSDF_OK;
}

int svsdf_query(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, int64_t P, const double *pts,
                double *sdf, double *tstar, double *grad3, int *rounds, int outer_only) {
    if (!ctx || P < 0 || (P > 0 && !pts)) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = upload_traj(ctx, N, T, coeffs);
    if (rc) return rc;
    if (P == 0) { CK(cudaStreamSynchronize(ctx->stream)); return SVSDF_OK; }
    if (P > ctx->cap_q) {
        cudaFree(ctx->d_q_points); cudaFree(ctx->d_q_sdf); cudaFree(ctx->d_q_ts); cudaFree(ctx->d_q_grad);
        cudaFree(ctx->d_q_rounds);
        ctx->d_q_points = ctx->d_q_sdf = ctx->d_q_ts = ctx->d_q_grad = nullptr;
        ctx->d_q_rounds = nullptr;
        ctx->cap_q = 0;
        int64_t cap = P + 1024;
        CK(cudaMalloc(&ctx->d_q_points, cap * 2 * sizeof(double)));
        CK(cudaMalloc(&ctx->d_q_sdf, cap * sizeof(double)));
        CK(cudaMalloc(&ctx->d_q_ts, cap * sizeof(double)));
        CK(cudaMalloc(&ctx->d_q_grad, cap * 3 * sizeof(double)));
        CK(cudaMalloc(&ctx->d_q_rounds, cap * sizeof(int)));
        ctx->cap_q = cap;
    }
    rc = ensure_stage(ctx, (size_t)P * 5 * sizeof(double) + (size_t)P * sizeof(int));
    if (rc) return rc;
    double *h = ctx->h_stage;
    for (int64_t i = 0; i < P; ++i) { h[2 * i] = pts[3 * i]; h[2 * i + 1] = pts[3 * i + 1]; }
    CK(cudaMemcpyAsync(ctx->d_q_points, h, (size_t)P * 2 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    rc = run_kernels(ctx, ctx->d_q_points, P, false, outer_only == 0, ctx->d_q_sdf, ctx->d_q_ts, ctx->d_q_grad,
                     ctx->d_q_rounds);
    if (rc) return rc;
    double *h_sdf = h, *h_ts = h + P, *h_grad = h + 2 * P;
    int *h_rounds = reinterpret_cast<int *>(h + 5 * P);
    CK(cudaMemcpyAsync(h_sdf, ctx->d_q_sdf, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_ts, ctx->d_q_ts, (size_t)P * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_grad, ctx->d_q_grad, (size_t)P * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(h_rounds, ctx->d_q_rounds, (size_t)P * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (sdf) std::memcpy(sdf, h_sdf, (size_t)P * sizeof(double));
    if (tstar) std::memcpy(tstar, h_ts, (size_t)P * sizeof(double));
    if (grad3) std::memcpy(grad3, h_grad, (size_t)P * 3 * sizeof(double));
    if (rounds) std::memcpy(rounds, h_rounds, (size_t)P * sizeof(int));
    return SVSDF_OK;
}

int svsdf_cost_grad(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, double *cost_io,
                    double *gradT_io, double *gradC_io) {
    if (!ctx || !cost_io || !gradT_io || !gradC_io) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = cost_grad_raw(ctx, N, T, coeffs);
    if (rc) return rc;
    const double *o = ctx->h_out;
    *cost_io += o[0];
    for (int e = 0; e < 18 * N; ++e) gradC_io[e] += o[1 + e];
    for (int i = 0; i < N; ++i) gradT_io[i] += o[1 + 18 * N + i];
    if (!std::isfinite(o[0])) return SVSDF_ERR_NONFINITE;
    return SVSDF_OK;
}

int svsdf_cost_grad_device(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, int repeats,
                           float *ms_per_eval, double *out_host) {
    if (!ctx || repeats < 1) return SVSDF_ERR_INVALID;
    if (!ctx->d_points) { ctx->err = "svsdf: query points not set"; return SVSDF_ERR_NOT_READY; }
    CK(cudaSetDevice(ctx->device));
    int rc = upload_traj(ctx, N, T, coeffs, false);
    if (rc) return rc;
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    for (int r = 0; r < repeats; ++r) {
        ctx->mark_kernels = (r == repeats - 1);
        if (ctx->mark_kernels) CK(cudaEventRecord(ctx->evk[0], ctx->stream));
        rc = pose_table(ctx);
        if (rc) return rc;
        if (ctx->mark_kernels) CK(cudaEventRecord(ctx->evk[1], ctx->stream));
        rc = run_kernels(ctx, ctx->d_points, ctx->P, true, true, nullptr, nullptr, nullptr, nullptr);
        if (ctx->mark_kernels) cudaEventRecord(ctx->evk[4], ctx->stream);
        ctx->mark_kernels = false;
        if (rc) return rc;
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    for (int k = 0; k < 4; ++k) CK(cudaEventElapsedTime(&ctx->last_kernel_ms[k], ctx->evk[k], ctx->evk[k + 1]));
    if (ms_per_eval) *ms_per_eval = ms / repeats;
    {
        const int nout = 1 + 19 * N + 1;
        CK(cudaMemcpy(ctx->h_out, ctx->d_out, (size_t)nout * sizeof(double), cudaMemcpyDeviceToHost));
        ctx->last_n_inside = (int64_t)ctx->h_out[1 + 19 * N];
        if (out_host) std::memcpy(out_host, ctx->h_out, (size_t)nout * sizeof(double));
    }
    return SVSDF_OK;
}

int svsdf_set_boundary(svsdf_ctx *ctx, const double *initS, const double *finalS, int N) {
    if (!ctx || !initS || !finalS || N < 2 || N > kMaxPieces) return SVSDF_ERR_INVALID;
    ctx->pieceN = N;
    ctx->minco.setConditions(initS, finalS, N);
    ctx->times.assign(N, 0.0);
    ctx->gradByTimes.assign(N, 0.0);
    ctx->partialGradByTimes.assign(N, 0.0);
    ctx->partialGradByCoeffs.assign((size_t)18 * N, 0.0);
    ctx->gradByPoints.assign((size_t)3 * (N - 1), 0.0);
    ctx->have_boundary = true;
    return SVSDF_OK;
}

double svsdf_evaluate(void *instance, const double *x, double *g, const int n) {
    svsdf_ctx *ctx = static_cast<svsdf_ctx *>(instance);
    if (!ctx || !x || !g) return NAN;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return NAN;
    return evaluate_impl(ctx, x, g, n);
}

int svsdf_last_costs(const svsdf_ctx *ctx, double *out3) {
    if (!ctx || !out3) return SVSDF_ERR_INVALID;
    out3[0] = ctx->cost_pos; out3[1] = ctx->cost_other; out3[2] = ctx->cost_total;
    return SVSDF_OK;
}

int svsdf_get_traj(const svsdf_ctx *ctx, double *T_out, double *coeffs_out) {
    if (!ctx || !ctx->have_boundary) return SVSDF_ERR_NOT_READY;
    if (T_out) std::memcpy(T_out, ctx->times.data(), sizeof(double) * ctx->pieceN);
    if (coeffs_out) std::memcpy(coeffs_out, ctx->minco.getCoeffs(), sizeof(double) * 18 * ctx->pieceN);
    return SVSDF_OK;
}

void svsdf_default_lbfgs_params(svsdf_lbfgs_params *p) {
    host::LbfgsParams d;
    p->mem_size = d.mem_size; p->past = d.past; p->delta = d.delta; p->g_epsilon = d.g_epsilon;
    p->max_iterations = d.max_iterations; p->max_linesearch = d.max_linesearch; p->min_step = d.min_step;
    p->max_step = d.max_step; p->f_dec_coeff = d.f_dec_coeff; p->s_curv_coeff = d.s_curv_coeff;
    p->cautious_factor = d.cautious_factor; p->machine_prec = d.machine_prec;
    p->nonsmooth_restarts = 8;  // the SVSDF cost is non-smooth: restart across kinks, end with status 3 at a kink (svsdf.h)
}

static host::LbfgsParams to_host_params(const svsdf_lbfgs_params *params) {
    svsdf_lbfgs_params dp;
    svsdf_default_lbfgs_params(&dp);
    if (!params) params = &dp;
    host::LbfgsParams hp;
    hp.mem_size = params->mem_size; hp.past = params->past; hp.delta = params->delta; hp.g_epsilon = params->g_epsilon;
    hp.max_iterations = params->max_iterations; hp.max_linesearch = params->max_linesearch;
    hp.min_step = params->min_step; hp.max_step = params->max_step; hp.f_dec_coeff = params->f_dec_coeff;
    hp.s_curv_coeff = params->s_curv_coeff; hp.cautious_factor = params->cautious_factor;
    hp.machine_prec = params->machine_prec;
    hp.nonsmooth_restarts = params->nonsmooth_restarts;
    return hp;
}

int svsdf_lbfgs_minimize(svsdf_eval_t eval, void *instance, double *x, int n, const svsdf_lbfgs_params *params,
                         svsdf_progress_t progress, void *user, svsdf_opt_stats *stats) {
    if (!eval || !x || n <= 0) return host::LBFGSERR_INVALID_N;
    host::Lbfgs solver(to_host_params(params));
    auto t0 = std::chrono::steady_clock::now();
    host::LbfgsResult R = solver.minimize(x, n, eval, instance, progress, user);
    auto t1 = std::chrono::steady_clock::now();
    if (stats) {
        stats->final_cost = R.f; stats->iterations = R.iterations; stats->evaluations = R.evaluations;
        stats->status = R.status; stats->seconds = std::chrono::duration<double>(t1 - t0).count();
        stats->gpu_seconds = 0.0;
    }
    return R.status;
}

int svsdf_optimize(svsdf_ctx *ctx, const double *initS, const double *finalS, double *opt_x, int N,
                   const svsdf_lbfgs_params *params, svsdf_progress_t progress, void *user, double *T_out,
                   double *coeffs_out, svsdf_opt_stats *stats) {
    if (!ctx || !opt_x) return SVSDF_ERR_INVALID;
    int rc = svsdf_set_boundary(ctx, initS, finalS, N);
    if (rc) return rc;
    host::LbfgsParams hp = to_host_params(params);
    const int n = N + 3 * (N - 1);
    ctx->gpu_ms_total = 0.0;
    ctx->time_kernels = true;
    auto t0 = std::chrono::steady_clock::now();
    host::LbfgsResult R;
    if (ctx->lmbm) {  // the reference's own LMBM drives the callback (back_end_optimizer.cpp:29-36); this context's private instance
        struct Count { svsdf_ctx *ctx; int evals; svsdf_progress_t progress; void *user; int iters; } cnt{ctx, 0, progress, user, 0};
        double fx = 0.0;
        R.status = ctx->lmbm->optimize(
            n, opt_x, &fx,
            [](void *u, const double *xx, double *gg, const int nn) { Count *c = static_cast<Count *>(u); ++c->evals; return svsdf_evaluate(c->ctx, xx, gg, nn); }, &cnt,
            [](void *u, const double *xx, const int k) { Count *c = static_cast<Count *>(u); c->iters = k; return c->progress ? c->progress(c->user, xx, k) : 0; },
            &ctx->lmbm_params);
        R.f = fx;
        R.evaluations = cnt.evals;
        R.iterations = cnt.iters;
    } else {
        host::Lbfgs solver(hp);
        R = solver.minimize(opt_x, n, svsdf_evaluate, ctx, progress, user);
    }
    auto t1 = std::chrono::steady_clock::now();
    ctx->time_kernels = false;
    // final trajectory from the returned iterate (optimize_traj_lmbm does the same on success and failure,
    // back_end_optimizer.cpp:44-94)
    for (int i = 0; i < N; ++i) ctx->times[i] = host::forwardT(opt_x[i]);
    ctx->minco.setParameters(opt_x + N, ctx->times.data());
    if (T_out) std::memcpy(T_out, ctx->times.data(), sizeof(double) * N);
    if (coeffs_out) std::memcpy(coeffs_out, ctx->minco.getCoeffs(), sizeof(double) * 18 * N);
    if (stats) {
        stats->final_cost = R.f;
        stats->iterations = R.iterations;
        stats->evaluations = R.evaluations;
        stats->status = R.status;
        stats->seconds = std::chrono::duration<double>(t1 - t0).count();
        stats->gpu_seconds = ctx->gpu_ms_total * 1e-3;
    }
    // an evaluation that failed (points not set, CUDA error, duration >= 300 s) is an error of the run, whatever the
    // solver made of the NaN it was handed
    if (ctx->last_status != SVSDF_OK) return ctx->last_status;
    int ret = R.status;
    if (ret == 0) ret = 1;  // back_end_optimizer.cpp:66-69
    return ret;
}

int svsdf_optimize_batch(svsdf_ctx *const *ctxs, int n_ctx, const svsdf_problem *problems, int n_problems, int N,
                         const svsdf_lbfgs_params *params, svsdf_next_problem_t next, void *next_user,
                         svsdf_opt_stats *stats_out, int *status_out, int64_t *points_out) {
    if (!problems && n_problems > 0) return SVSDF_ERR_INVALID;
    return run_pool(ctxs, n_ctx, n_problems, next, next_user, [&](svsdf_ctx *ctx, int k) -> int {
        const svsdf_problem &pr = problems[k];
        if (!pr.initS || !pr.finalS || !pr.opt_x) return SVSDF_ERR_INVALID;
        int rc;
        int64_t np = 0;
        if (pr.points) {
            rc = svsdf_set_points(ctx, pr.points, pr.P, pr.stride);
            np = pr.P;
        } else {
            rc = svsdf_extract_points(ctx, pr.waypoints_xy, pr.W, pr.half, pr.keepout_xy, pr.n_keepout, pr.clearance, &np);
        }
        if (rc != SVSDF_OK) {
            if (status_out) status_out[k] = rc;
            return rc;
        }
        if (points_out) points_out[k] = np;
        svsdf_opt_stats st;
        std::memset(&st, 0, sizeof(st));
        const int ret = svsdf_optimize(ctx, pr.initS, pr.finalS, pr.opt_x, N, params, nullptr, nullptr, pr.T_out, pr.coeffs_out, &st);
        if (stats_out) stats_out[k] = st;
        if (status_out) status_out[k] = ret;
        // solver codes (incl. negative line-search codes) are per-problem results; API / CUDA errors abort the call's status
        return (ret <= SVSDF_ERR_INVALID && ret > -1000) ? ret : SVSDF_OK;
    });
}

int svsdf_cost_grad_batch(svsdf_ctx *const *ctxs, int n_ctx, int n_problems, int N, const double *const *pts, const int64_t *P,
                          int stride, const double *T, const double *coeffs, double *cost_io, double *gradT_io, double *gradC_io) {
    if (n_problems > 0 && (!pts || !P || !T || !coeffs || !cost_io || !gradT_io || !gradC_io)) return SVSDF_ERR_INVALID;
    return run_pool(ctxs, n_ctx, n_problems, nullptr, nullptr, [&](svsdf_ctx *ctx, int k) -> int {
        int rc = svsdf_set_points(ctx, pts[k], P[k], stride);
        if (rc != SVSDF_OK) return rc;
        return svsdf_cost_grad(ctx, N, T + (size_t)k * N, coeffs + (size_t)k * 18 * N, cost_io + k, gradT_io + (size_t)k * N,
                               gradC_io + (size_t)k * 18 * N);
    });
}

int svsdf_minco_forward(const double *initS, const double *finalS, int N, const double *q, const double *T,
                        double *coeffs_out, double *energy, double *gradC_out, double *gradT_out) {
    if (!initS || !finalS || !q || !T || N < 2) return SVSDF_ERR_INVALID;
    host::MincoS3NU m;
    m.setConditions(initS, finalS, N);
    m.setParameters(q, T);
    if (coeffs_out) std::memcpy(coeffs_out, m.getCoeffs(), sizeof(double) * 18 * N);
    if (energy) *energy = m.getEnergy();
    if (gradC_out) m.getEnergyPartialGradByCoeffs(gradC_out);
    if (gradT_out) m.getEnergyPartialGradByTimes(gradT_out);
    return SVSDF_OK;
}

int svsdf_minco_propagate(const double *initS, const double *finalS, int N, const double *q, const double *T,
                          const double *gradC, const double *gradT, double *gradQ_out, double *gradT_out) {
    if (!initS || !finalS || !q || !T || !gradC || !gradT || !gradQ_out || !gradT_out || N < 2) return SVSDF_ERR_INVALID;
    host::MincoS3NU m;
    m.setConditions(initS, finalS, N);
    m.setParameters(q, T);
    m.propogateGrad(gradC, gradT, gradQ_out, gradT_out);
    return SVSDF_OK;
}

void svsdf_forward_T(int n, const double *tau, double *T) { for (int i = 0; i < n; ++i) T[i] = host::forwardT(tau[i]); }
void svsdf_backward_T(int n, const double *T, double *tau) { for (int i = 0; i < n; ++i) tau[i] = host::backwardT(T[i]); }

static int shape_eval(svsdf_ctx *ctx, int64_t n, const double *rel, double *out, int grad) {
    if (!ctx || n < 0 || (n > 0 && (!rel || !out))) return SVSDF_ERR_INVALID;
    if (n == 0) return SVSDF_OK;
    CK(cudaSetDevice(ctx->device));
    const int ow = grad ? 3 : 1;
    int rc = ensure_stage(ctx, (size_t)n * (2 + ow) * sizeof(double));
    if (rc) return rc;
    double *d_in = nullptr, *d_out = nullptr;
    CK(cudaMalloc(&d_in, (size_t)n * 2 * sizeof(double)));
    if (cudaMalloc(&d_out, (size_t)n * ow * sizeof(double)) != cudaSuccess) { cudaFree(d_in); ctx->err = "cudaMalloc"; return SVSDF_ERR_CUDA; }
    double *h = ctx->h_stage;
    for (int64_t i = 0; i < n; ++i) { h[2 * i] = rel[3 * i]; h[2 * i + 1] = rel[3 * i + 1]; }
    cudaError_t e = cudaMemcpyAsync(d_in, h, (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = ctx->strict ? strict::launch_shape_eval(ctx->shape, d_in, n, d_out, grad, ctx->stream)
                        : fast::launch_shape_eval(ctx->shape, d_in, n, d_out, grad, ctx->stream);
    ctx->launches += 1;
    double *ho = h + 2 * n;
    if (e == cudaSuccess) e = cudaMemcpyAsync(ho, d_out, (size_t)n * ow * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_in);
    cudaFree(d_out);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
    std::memcpy(out, ho, (size_t)n * ow * sizeof(double));
    return SVSDF_OK;
}
int svsdf_shape_sdf(svsdf_ctx *ctx, int64_t n, const double *rel, double *sdf_out) { return shape_eval(ctx, n, rel, sdf_out, 0); }
int svsdf_shape_grad1(svsdf_ctx *ctx, int64_t n, const double *rel, double *grad3_out) { return shape_eval(ctx, n, rel, grad3_out, 1); }

static int set_map_meta(svsdf_ctx *ctx, int X, int Y, int kernel_size, double ox, double oy, double res) {
    if (X <= 0 || Y <= 0 || kernel_size < 1 || (kernel_size & 1) == 0 || !(res > 0.0)) {
        ctx->err = "svsdf_set_map: bad map geometry (kernel_size must be odd, res > 0)";
        return SVSDF_ERR_INVALID;
    }
    ctx->map_X = X; ctx->map_Y = Y; ctx->map_h = (kernel_size - 1) / 2;
    ctx->map_row_bytes = (Y + 2 * ctx->map_h + 7) / 8;
    ctx->map_ox = ox; ctx->map_oy = oy; ctx->map_oz = 0.0; ctx->map_res = res;
    ctx->map_Z = 1;
    return SVSDF_OK;
}

int svsdf_set_map(svsdf_ctx *ctx, const unsigned char *kernel_bytes, int X, int Y, int kernel_size, double origin_x,
                  double origin_y, double res) {
    if (!ctx || !kernel_bytes) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = set_map_meta(ctx, X, Y, kernel_size, origin_x, origin_y, res);
    if (rc) return rc;
    const size_t bytes = (size_t)(X + 2 * ctx->map_h) * ctx->map_row_bytes;
    if (!ctx->own_map) { ctx->d_map = nullptr; ctx->own_map = true; ctx->cap_map = 0; }
    if (bytes > ctx->cap_map) {
        cudaFree(ctx->d_map);
        ctx->d_map = nullptr;
        ctx->cap_map = 0;
        CK(cudaMalloc(&ctx->d_map, bytes + 64));
        ctx->cap_map = bytes + 64;
    }
    CK(cudaMemcpyAsync(ctx->d_map, kernel_bytes, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SVSDF_OK;
}

int svsdf_set_map_device(svsdf_ctx *ctx, const unsigned char *dev_kernel_bytes, int X, int Y, int kernel_size,
                         double origin_x, double origin_y, double res) {
    if (!ctx || !dev_kernel_bytes) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = set_map_meta(ctx, X, Y, kernel_size, origin_x, origin_y, res);
    if (rc) return rc;
    if (ctx->own_map) cudaFree(ctx->d_map);
    ctx->d_map = const_cast<unsigned char *>(dev_kernel_bytes);
    ctx->own_map = false;
    ctx->cap_map = 0;
    return SVSDF_OK;
}

// generateMapKernel's layout (PCSmap_manager.h:39-78: [(X + 2h)][(Y + 2h)][ceil((Z + 2h) / 8)] bytes, z bits MSB first) is re-packed on
// the host, once per map, into Z layers of the 2-D layout the kernels read ([(X + 2h)][ceil((Y + 2h) / 8)], y bits MSB first); layer 0 is
// what generateMapKernel2D would have produced, so the front-end kernels see the same map as with svsdf_set_map.
int svsdf_set_map3d(svsdf_ctx *ctx, const unsigned char *kernel_bytes, int X, int Y, int Z, int kernel_size, const double *origin_xyz,
                    double res) {
    if (!ctx || !kernel_bytes || !origin_xyz || Z < 1 || Z > kMaxMapLayers) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    int rc = set_map_meta(ctx, X, Y, kernel_size, origin_xyz[0], origin_xyz[1], res);
    if (rc) return rc;
    const int h = ctx->map_h;
    const size_t layer = (size_t)(X + 2 * h) * ctx->map_row_bytes;
    const int zb = (Z + 2 * h + 7) / 8;
    std::vector<unsigned char> L(layer * (size_t)Z, 0);
    for (int x = 0; x < X; ++x)
        for (int y = 0; y < Y; ++y) {
            const unsigned char *col = kernel_bytes + ((size_t)(x + h) * (Y + 2 * h) + (size_t)(y + h)) * zb;
            for (int z = 0; z < Z; ++z) {
                const int fz = z + h;
                if (col[fz / 8] & (0x80u >> (fz % 8))) {
                    const int fy = y + h;
                    L[(size_t)z * layer + (size_t)(x + h) * ctx->map_row_bytes + fy / 8] |= (unsigned char)(0x80u >> (fy % 8));
                }
            }
        }
    const size_t bytes = L.size();
    if (!ctx->own_map) { ctx->d_map = nullptr; ctx->own_map = true; ctx->cap_map = 0; }
    if (bytes > ctx->cap_map) {
        cudaFree(ctx->d_map);
        ctx->d_map = nullptr;
        ctx->cap_map = 0;
        CK(cudaMalloc(&ctx->d_map, bytes + 64));
        ctx->cap_map = bytes + 64;
    }
    CK(cudaMemcpyAsync(ctx->d_map, L.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->map_Z = Z;
    ctx->map_oz = origin_xyz[2];
    return SVSDF_OK;
}

// Shared by the flat and the 3-D entry points.  wp: W x 3 waypoint centres, half: box half sizes (x, y, z).
static int extract_impl(svsdf_ctx *ctx, const char *who, const double *wp, int W, const double *half, const double *keepout_xy,
                        int n_keepout, double clearance, int64_t *n_points) {
    if (!ctx->d_map) { ctx->err = std::string(who) + ": map not set"; return SVSDF_ERR_NOT_READY; }
    CK(cudaSetDevice(ctx->device));
    ExtractArgs E;
    std::memset(&E, 0, sizeof(E));
    E.X = ctx->map_X; E.Y = ctx->map_Y; E.h = ctx->map_h; E.row_bytes = ctx->map_row_bytes;
    E.ox = ctx->map_ox; E.oy = ctx->map_oy; E.res = ctx->map_res;
    E.W = W;
    const int Z = ctx->map_Z;
    const double lo[3] = {E.ox, E.oy, ctx->map_oz};
    const double hi[3] = {E.ox + (double)E.X * E.res, E.oy + (double)E.Y * E.res, ctx->map_oz + (double)Z * E.res};  // boundary_xyzmax
    const int size[3] = {E.X, E.Y, Z};
    // clamped index box around a centre: corner = centre -+ half -> projInMap (PCSmap_manager.h:128-135) -> getGridIndex
    // (Gridmap3D.cpp:137-174: floor, clamped to the last cell)
    auto box = [&](const double *c, int idx[3][2]) {
        for (int a = 0; a < 3; ++a)
            for (int side = 0; side < 2; ++side) {
                double v = c[a] + (side ? half[a] : -half[a]);
                v = v < lo[a] ? lo[a] : v;
                v = v > hi[a] ? hi[a] : v;
                int i = (int)std::floor((v - lo[a]) / E.res);
                i = i < 0 ? 0 : i;
                i = i >= size[a] ? size[a] - 1 : i;
                idx[a][side] = i;
            }
    };
    int bz1[kMaxWaypoints + 1], bz2[kMaxWaypoints + 1];  // slot 0: the box around tmp_pos, slot w + 1: waypoint w
    {
        const double tmp_pos[3] = {999.0, 999.0, 999.0};  // plan_manager.cpp:152
        int idx[3][2];
        box(tmp_pos, idx);
        E.px1 = idx[0][0]; E.px2 = idx[0][1]; E.py1 = idx[1][0]; E.py2 = idx[1][1];
        bz1[0] = idx[2][0]; bz2[0] = idx[2][1];
    }
    int rxmin = E.X, rxmax = -1, rymin = E.Y, rymax = -1;
    for (int w = 0; w < W; ++w) {
        int idx[3][2];
        box(wp + 3 * w, idx);
        E.bx1[w] = idx[0][0]; E.bx2[w] = idx[0][1]; E.by1[w] = idx[1][0]; E.by2[w] = idx[1][1];
        bz1[w + 1] = idx[2][0]; bz2[w + 1] = idx[2][1];
        rxmin = std::min(rxmin, E.bx1[w]); rxmax = std::max(rxmax, E.bx2[w]);
        rymin = std::min(rymin, E.by1[w]); rymax = std::max(rymax, E.by2[w]);
    }
    E.rx1 = rxmin;
    E.wy1 = (rymin + E.h) / 32;
    const int wy2 = (rymax + E.h) / 32;
    E.nW = wy2 - E.wy1 + 1;
    E.n_items = (long long)(rxmax - rxmin + 1) * E.nW;
    E.n_keepout = n_keepout;
    E.clearance = clearance;
    for (int q = 0; q < 2 * n_keepout; ++q) E.keepout[q] = keepout_xy[q];
    const int n_blocks = (int)((E.n_items + 255) / 256);
    const size_t need_counts = (size_t)(n_blocks + 1) * (size_t)Z;
    if (need_counts > (size_t)ctx->cap_block_counts) {
        cudaFree(ctx->d_block_counts);
        ctx->d_block_counts = nullptr;
        ctx->cap_block_counts = 0;
        CK(cudaMalloc(&ctx->d_block_counts, (need_counts + 1024) * sizeof(int)));
        ctx->cap_block_counts = (int)(need_counts + 1024);
    }
    if (!ctx->d_n_total) CK(cudaMalloc(&ctx->d_n_total, kMaxMapLayers * sizeof(int64_t)));
    const size_t layer = (size_t)(E.X + 2 * E.h) * E.row_bytes;
    auto layer_args = [&](int k) {
        ExtractArgs Ek = E;
        Ek.map = ctx->d_map + (size_t)k * layer;
        for (int w = 0; w < W; ++w) {
            Ek.act[w] = (k >= bz1[w + 1] && k <= bz2[w + 1]) ? 1 : 0;
            Ek.excl[w] = (k >= bz1[w] && k <= bz2[w]) ? 1 : 0;
        }
        return Ek;
    };
    for (int k = 0; k < Z; ++k) {
        CK(launch_extract_count(layer_args(k), ctx->d_block_counts + (size_t)k * (n_blocks + 1), n_blocks, ctx->d_n_total + k, ctx->stream));
        ctx->launches += 2;
    }
    int64_t totals[kMaxMapLayers];
    CK(cudaMemcpyAsync(totals, ctx->d_n_total, (size_t)Z * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int64_t total = 0;
    for (int k = 0; k < Z; ++k) total += totals[k];
    if (total > 2000000000LL) { ctx->err = std::string(who) + ": too many points"; return SVSDF_ERR_INVALID; }
    if (!ctx->own_points) { ctx->d_points = nullptr; ctx->own_points = true; ctx->cap_points = 0; }
    if (total > ctx->cap_points || !ctx->d_points) {
        cudaFree(ctx->d_points);
        ctx->d_points = nullptr;
        ctx->cap_points = 0;
        CK(cudaMalloc(&ctx->d_points, (size_t)(total + 1024) * 2 * sizeof(double)));
        ctx->cap_points = total + 1024;
    }
    int64_t base = 0;
    for (int k = 0; k < Z; ++k) {  // layer-major output: layer 0's cells in ascending (i * Y + j) order, then layer 1's, ...
        CK(launch_extract_write(layer_args(k), ctx->d_block_counts + (size_t)k * (n_blocks + 1), n_blocks, ctx->d_points + 2 * base, totals[k], ctx->stream));
        ctx->launches += 1;
        base += totals[k];
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->P = total;
    ctx->last_n_inside = -1;
    if (n_points) *n_points = total;
    return ensure_scratch(ctx, total);
}

int svsdf_extract_points(svsdf_ctx *ctx, const double *waypoints_xy, int W, double half, const double *keepout_xy,
                         int n_keepout, double clearance, int64_t *n_points) {
    if (!ctx || !waypoints_xy || W < 1 || W > kMaxWaypoints || n_keepout < 0 || n_keepout > kMaxKeepout ||
        (n_keepout > 0 && !keepout_xy) || !(half >= 0.0))
        return SVSDF_ERR_INVALID;
    if (ctx->map_Z != 1) { ctx->err = "svsdf_extract_points: the map has several z layers, use svsdf_extract_points3d"; return SVSDF_ERR_INVALID; }
    // the flat case: one layer, every box spans it (centre z in the middle of the layer)
    std::vector<double> wp((size_t)W * 3);
    for (int w = 0; w < W; ++w) {
        wp[3 * (size_t)w] = waypoints_xy[2 * w];
        wp[3 * (size_t)w + 1] = waypoints_xy[2 * w + 1];
        wp[3 * (size_t)w + 2] = ctx->map_oz + 0.5 * ctx->map_res;
    }
    const double h3[3] = {half, half, half};
    return extract_impl(ctx, "svsdf_extract_points", wp.data(), W, h3, keepout_xy, n_keepout, clearance, n_points);
}

int svsdf_extract_points3d(svsdf_ctx *ctx, const double *waypoints_xyz, int W, const double *half_xyz, const double *keepout_xy,
                           int n_keepout, double clearance, int64_t *n_points) {
    if (!ctx || !waypoints_xyz || !half_xyz || W < 1 || W > kMaxWaypoints || n_keepout < 0 || n_keepout > kMaxKeepout ||
        (n_keepout > 0 && !keepout_xy) || !(half_xyz[0] >= 0.0) || !(half_xyz[1] >= 0.0) || !(half_xyz[2] >= 0.0))
        return SVSDF_ERR_INVALID;
    return extract_impl(ctx, "svsdf_extract_points3d", waypoints_xyz, W, half_xyz, keepout_xy, n_keepout, clearance, n_points);
}

int svsdf_get_points(svsdf_ctx *ctx, double *xy_out, int64_t capacity, int64_t *n_points) {
    if (!ctx) return SVSDF_ERR_INVALID;
    if (n_points) *n_points = ctx->P;
    if (!xy_out || capacity <= 0 || ctx->P == 0) return SVSDF_OK;
    CK(cudaSetDevice(ctx->device));
    const int64_t n = ctx->P < capacity ? ctx->P : capacity;
    CK(cudaMemcpy(xy_out, ctx->d_points, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost));
    return SVSDF_OK;
}

int svsdf_sincos(svsdf_ctx *ctx, int64_t n, const double *x, double *sin_out, double *cos_out) {
    if (!ctx || n < 0 || (n > 0 && (!x || !sin_out || !cos_out))) return SVSDF_ERR_INVALID;
    if (n == 0) return SVSDF_OK;
    CK(cudaSetDevice(ctx->device));
    double *d = nullptr;
    CK(cudaMalloc(&d, (size_t)n * 3 * sizeof(double)));
    cudaError_t e = cudaMemcpyAsync(d, x, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
        e = ctx->strict ? strict::launch_sincos(d, n, d + n, d + 2 * n, ctx->stream)
                        : fast::launch_sincos(d, n, d + n, d + 2 * n, ctx->stream);
    ctx->launches += 1;
    if (e == cudaSuccess) e = cudaMemcpyAsync(sin_out, d + n, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(cos_out, d + 2 * n, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
    return SVSDF_OK;
}

int svsdf_last_kernel_ms(const svsdf_ctx *ctx, float *out4) {
    if (!ctx || !out4) return SVSDF_ERR_INVALID;
    for (int k = 0; k < 4; ++k) out4[k] = ctx->last_kernel_ms[k];
    return SVSDF_OK;
}

int svsdf_kernel_launches(const svsdf_ctx *ctx, int64_t *count) {
    if (!ctx || !count) return SVSDF_ERR_INVALID;
    *count = ctx->launches;
    return SVSDF_OK;
}

int svsdf_executed_evals(svsdf_ctx *ctx, int enable, uint64_t *count) {
    if (!ctx) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    if (count) {
        unsigned long long v = 0;
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaMemcpy(&v, ctx->d_eval_counter, sizeof(v), cudaMemcpyDeviceToHost));
        *count = v;
    }
    ctx->count_evals = enable != 0;
    CK(cudaMemset(ctx->d_eval_counter, 0, sizeof(unsigned long long)));
    return SVSDF_OK;
}

int svsdf_fp64_peak(svsdf_ctx *ctx, double *tflops) {
    if (!ctx || !tflops) return SVSDF_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int grid = ctx->sm_count * 8, iters = 1 << 16;
    double *d = nullptr;
    CK(cudaMalloc(&d, (size_t)grid * 256 * sizeof(double)));
    float best = 1e30f;
    for (int r = 0; r < 5; ++r) {
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        cudaError_t e = fast::launch_fp64_peak(d, grid, iters, ctx->stream);
        if (e != cudaSuccess) { cudaFree(d); ctx->err = cudaGetErrorString(e); return SVSDF_ERR_CUDA; }
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        if (r > 0 && ms < best) best = ms;
        ctx->launches += 1;
    }
    cudaFree(d);
    const double flops = 2.0 * 8.0 * (double)iters * (double)grid * 256.0;
    *tflops = flops / (best * 1e-3) / 1e12;
    return SVSDF_OK;
}

}  // extern "C"

// svsdf_kernels.cuh — sm_100a kernels for the SVSDF collision cost + gradient hot path.
//
// Replaces the OpenMP loop  TrajOptimizer::addSaftyPenaOnSweptVolumeParallelTrueSDF
// (src/planner_algorithm/include/planner_algorithm/back_end_optimizer.hpp:774-869) and everything it calls in
// SweptVolumeManager (src/swept_volume/include/swept_volume/sw_manager.hpp:465-474, 521-526, 538-581, 741-757,
// 779-806, 844-866, 916-1018, 1249-1325).
//
// Mapping (one warp per query point):
//   * the trajectory blob (durations, quintic coefficients, layer-1 time lattice and its pose table) is pulled
//     into shared memory once per CTA with a TMA bulk copy (cp.async.bulk + mbarrier);
//   * choiceTInit's four scan layers are evaluated 32 samples per round, one sample per lane, and reduced with
//     a shuffle arg-min that keeps the reference's "first strict minimum wins" rule;
//   * gradientDescent's inner loop (29 step halvings, each needing 3 SDF evaluations) is evaluated
//     speculatively in parallel: lanes 30/31 compute the finite-difference slope, lanes 0-29 the candidates for
//     both signs, and the first accepted halving is picked with a ballot — decisions are identical to the
//     sequential loop given identical SDF values;
//   * the FD gradient uses 4 lanes; the smoothed-L1 penalty and the chain rule to the 6x3 coefficient block are
//     accumulated in per-warp shared-memory accumulators (no atomics), reduced per CTA in a fixed order and
//     written as one partial per CTA; a tiny finalize kernel sums the partials in a fixed order, so results are
//     bit-reproducible run to run.
//   * points found inside the swept volume (sdf <= 0) are compacted in index order and handled by k_gsip, one
//     CTA per point, ring samples spread over the CTA's warps.
//
// This file is compiled twice (see svsdf_kernels_fast.cu / svsdf_kernels_strict.cu): with FMA contraction
// (default) and with -fmad=false ("strict": same rounding sequence as the CPU, used to debug parity).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "svsdf_shapes.cuh"
#include "svsdf_sincos.cuh"
#include "svsdf_types.h"

#ifndef SVSDF_NS
#error "define SVSDF_NS (fast|strict) before including svsdf_kernels.cuh"
#endif

namespace svsdf {
namespace SVSDF_NS {

constexpr unsigned FULL = 0xffffffffu;
using dev::smaxd;
using dev::smind;

// ------------------------------------------------------------------------------------------------
// Trajectory view over the shared-memory copy of the blob
// ------------------------------------------------------------------------------------------------
struct TrajView {
    int N, K1;
    double D;
    const double *T;     // [N]
    const double *c;     // [N][3][6] ascending powers
    const double *lat;   // [K1]
    const double *pose;  // [4][K1pad] SoA: x, y, cos, sin
    int K1pad;
    // the same arrays as 32-bit shared-window addresses (valid when the view is on the shared-memory copy of the blob):
    // the hot loops read through these with ld.shared so the address is one register + immediate instead of a
    // generic pointer whose shared-window base the compiler re-derives (S2R SR_CgaCtaId + LEA) at every use
    uint32_t sT, sc, slat, spose;
};

__device__ __forceinline__ double lds_f64(uint32_t a) {
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void lds_v2(uint32_t a, double &v0, double &v1) {
    asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v0), "=d"(v1) : "r"(a));
}

__device__ __forceinline__ TrajView make_view(const double *blob) {
    TrajView tv;
    tv.N = (int)blob[0];
    tv.K1 = (int)blob[1];
    tv.D = blob[2];
    BlobLayout L = blob_layout(tv.N, tv.K1);
    tv.T = blob + L.off_T;
    tv.c = blob + L.off_c;
    tv.lat = blob + L.off_lat;
    tv.pose = blob + L.off_pose;
    tv.K1pad = L.K1pad;
    // (meaningless for a view on global memory, k_pose_table).  The blob is read-only once the TMA copy has landed; the
    // empty volatile asm orders every ld.shared that derives its address from `sb` after the mbarrier wait.
    uint32_t sb = (uint32_t)__cvta_generic_to_shared(blob);
    asm volatile("" : "+r"(sb) : : "memory");
    tv.sT = sb + 8u * (uint32_t)L.off_T;
    tv.sc = sb + 8u * (uint32_t)L.off_c;
    tv.slat = sb + 8u * (uint32_t)L.off_lat;
    tv.spose = sb + 8u * (uint32_t)L.off_pose;
    return tv;
}

// Trajectory<5>::locatePieceIdx (trajectory.hpp:498-516): subtract durations while t > dur (strict).
__device__ __forceinline__ int locate_piece(const TrajView &tv, double &t) {
    int idx = 0;
#pragma unroll 1
    for (; idx < tv.N; ++idx) {
        double dur = tv.T[idx];
        if (!(t > dur)) break;
        t -= dur;
    }
    if (idx == tv.N) {
        idx--;
        t += tv.T[idx];
    }
    return idx;
}

// locatePieceIdx with a guess.  The reference's loop yields piece h and local time t_h = ((t - T_0) - T_1) ... - T_{h-1}
// (one rounding per subtraction) iff every test before h passed and the test at h failed.  fl(a - b) > 0 <=> a > b, so
// "all earlier tests passed" is equivalent to t_h > 0 (induction: t_h > 0 => t_{h-1} > T_{h-1} > 0 => ...).  With the
// guess taken from the caller's previous sample (consecutive samples of a scan or of a descent almost always fall into
// the same piece) the search is the bare subtraction chain plus two compares; a wrong guess (or NaN, or the idx == N
// wrap-around case) falls back to the reference loop.  Same result bit for bit.
__device__ __forceinline__ int locate_piece(const TrajView &tv, double &t, int &hint) {
    const int h = hint;
    double tl = t;
    uint32_t a = tv.sT;  // 16-byte aligned
    int i = 0;
#pragma unroll 1
    for (; i + 2 <= h; i += 2, a += 16) {
        double d0, d1;
        lds_v2(a, d0, d1);
        tl -= d0;
        tl -= d1;
    }
    if (i < h) {
        tl -= lds_f64(a);
        a += 8;
    }
    const double Th = lds_f64(a);  // T[h]
    if ((h == 0 || tl > 0.0) && !(tl > Th)) {
        t = tl;
        return h;
    }
    hint = locate_piece(tv, t);
    return hint;
}

// Piece<5>::getPos (trajectory.hpp:104-114): ascending powers with tn *= t (not Horner).
__device__ __forceinline__ void traj_pos_at(const TrajView &tv, int i, double t, double &x, double &y, double &yaw) {
    const uint32_t a = tv.sc + 144u * (uint32_t)i;  // 18 doubles per piece, 16-byte aligned
    double c[18];
#pragma unroll
    for (int k = 0; k < 9; ++k) lds_v2(a + 16u * k, c[2 * k], c[2 * k + 1]);
    x = 0.0; y = 0.0; yaw = 0.0;
    double tn = 1.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        x += tn * c[k];
        y += tn * c[6 + k];
        yaw += tn * c[12 + k];
        tn *= t;
    }
}
__device__ __forceinline__ void traj_pos(const TrajView &tv, double t, double &x, double &y, double &yaw) {
    int i = locate_piece(tv, t);
    const double *c = tv.c + 18 * i;
    x = 0.0; y = 0.0; yaw = 0.0;
    double tn = 1.0;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        x += tn * c[k];
        y += tn * c[6 + k];
        yaw += tn * c[12 + k];
        tn *= t;
    }
}

// Piece<5>::getVel (trajectory.hpp:116-128)
__device__ __forceinline__ void traj_vel(const TrajView &tv, double t, double &vx, double &vy, double &vw) {
    int i = locate_piece(tv, t);
    const double *c = tv.c + 18 * i;
    vx = 0.0; vy = 0.0; vw = 0.0;
    double tn = 1.0;
#pragma unroll
    for (int k = 1; k < 6; ++k) {
        double f = (double)k * tn;
        vx += f * c[k];
        vy += f * c[6 + k];
        vw += f * c[12 + k];
        tn *= t;
    }
}

// getStateOnTrajStamp (sw_manager.hpp:465-474) + posEva2Rel (:521-526): rel = Rz(yaw)^T (p - x)
__device__ __forceinline__ void rel_from_pose(double px, double py, double x, double y, double cy, double sy,
                                              double &rx, double &ry) {
    double d0 = px - x, d1 = py - y;
    rx = cy * d0 + sy * d1;
    ry = -sy * d0 + cy * d1;
}

// getSDFAtTimeStamp<false> (sw_manager.hpp:741-757)
template <int SHAPE, bool XFORM>
__device__ __forceinline__ double eval_sdf(const TrajView &tv, const ShapeParams &S, double px, double py, double t) {
    double x, y, yaw, sy, cy, rx, ry;
    traj_pos(tv, t, x, y, yaw);
    dev::sincos_portable(yaw, sy, cy);
    rel_from_pose(px, py, x, y, cy, sy, rx, ry);
    return dev::shape_sdf<SHAPE, XFORM>(S, rx, ry);
}
// same with a piece-index guess carried by the caller from its previous sample
template <int SHAPE, bool XFORM>
__device__ __forceinline__ double eval_sdf(const TrajView &tv, const ShapeParams &S, double px, double py, double t, int &hint) {
    double x, y, yaw, sy, cy, rx, ry;
    const int i = locate_piece(tv, t, hint);
    traj_pos_at(tv, i, t, x, y, yaw);
    dev::sincos_portable(yaw, sy, cy);
    rel_from_pose(px, py, x, y, cy, sy, rx, ry);
    return dev::shape_sdf<SHAPE, XFORM>(S, rx, ry);
}

// getScale (sw_manager.hpp:495-507, the reference's edit point) as svsdf_set_scale specifies it: S(t) = diag(sx, sy, 1),
// per axis s = c, then s = s + sin(w_k t + phi_k) a_k, at ABSOLUTE time t.  Returns the two diagonal entries of S^-1 as the
// reference's 3x3 inverse forms them (cofactors times 1/det, Eigen's formula): det = sy sx, S^-1 = diag(sy inv, sx inv, .)
// with inv = 1 / det — not 1 / sx.  Every other term of the cofactor expansion is a product with an exact zero.
__device__ __forceinline__ void scale_inv(const ScaleParams &Z, double t, double &i00, double &i11) {
    double s[2];
#pragma unroll
    for (int ax = 0; ax < 2; ++ax) {
        double v = Z.c[ax];
#pragma unroll 1
        for (int k = 0; k < Z.n[ax]; ++k) {
            double sn, cs;
            dev::sincos_portable(Z.w[ax][k] * t + Z.phi[ax][k], sn, cs);
            v = v + sn * Z.a[ax][k];
        }
        s[ax] = v;
    }
    const double inv = 1.0 / (s[1] * s[0]);
    i00 = s[1] * inv;
    i11 = s[0] * inv;
}
// posEva2Rel(p, x, R, S) (sw_manager.hpp:528-535): rel = (R^T S^-1) (p - x), the 3x3 product formed first; its zero terms
// dropped.  With S = I (i00 = i11 = 1 exactly) this is rel_from_pose bit for bit.
__device__ __forceinline__ void rel_from_pose_scaled(double px, double py, double x, double y, double cy, double sy, double i00,
                                                     double i11, double &rx, double &ry) {
    double d0 = px - x, d1 = py - y;
    rx = (cy * i00) * d0 + (sy * i11) * d1;
    ry = (-(sy * i00)) * d0 + (cy * i11) * d1;
}
// the body-frame point of the scaled body at t (getStateOnTrajStamp(t, xt, Rt, St) + posEva2Rel(p, x, R, S): the rel of
// getSDFAtTimeStamp<true>, getSDFAtTimeStamp_igl<true> and getGradPrelAtTimeStamp<true>, sw_manager.hpp:741-795).  t is
// absolute trajectory time.
__device__ __forceinline__ void rel_at_scaled(const TrajView &tv, const ScaleParams &Z, double px, double py, double t, int &hint,
                                              double &rx, double &ry) {
    double x, y, yaw, sy, cy, i00, i11;
    const double ta = t;
    const int i = locate_piece(tv, t, hint);
    traj_pos_at(tv, i, t, x, y, yaw);
    dev::sincos_portable(yaw, sy, cy);
    scale_inv(Z, ta, i00, i11);
    rel_from_pose_scaled(px, py, x, y, cy, sy, i00, i11, rx, ry);
}
// the descent's samples: getSDFAtTimeStamp<useScale> (gradientDescent, sw_manager.hpp:1289-1304)
template <int SHAPE, bool XFORM, bool SCALED>
__device__ __forceinline__ double eval_sdf(const TrajView &tv, const ShapeParams &S, const ScaleParams &Z, double px, double py,
                                           double t, int &hint) {
    if (!SCALED) return eval_sdf<SHAPE, XFORM>(tv, S, px, py, t, hint);
    double rx, ry;
    rel_at_scaled(tv, Z, px, py, t, hint, rx, ry);
    return dev::shape_sdf<SHAPE, XFORM>(S, rx, ry);
}

// Warp arg-min with the sequential loop's semantics: the FIRST lane holding the minimum value wins; NaN never wins
// (callers map NaN to +inf; the reference's test is `dis < min_dis`).  Two 32-bit REDUX.MIN over an order-preserving
// integer image of the double, then a ballot for the first lane.  Returns the winning lane; f becomes the minimum.
__device__ __forceinline__ int warp_argmin_lane(double &f) {
    f = f + 0.0;  // -0.0 -> +0.0 so that equal values have equal keys
    unsigned long long b = (unsigned long long)__double_as_longlong(f);
    b ^= (b >> 63) ? 0xffffffffffffffffull : 0x8000000000000000ull;  // monotone map double -> uint64
    const unsigned hi = (unsigned)(b >> 32), lo = (unsigned)b;
    const unsigned mh = __reduce_min_sync(FULL, hi);
    const unsigned ml = __reduce_min_sync(FULL, hi == mh ? lo : 0xffffffffu);
    const unsigned win = __ballot_sync(FULL, hi == mh && lo == ml);
    const int src = __ffs(win) - 1;
    f = __shfl_sync(FULL, f, src);
    return src;
}

struct OuterResult {
    double sdf, tstar;
    int evals;  // lane-evaluations executed (active lanes), for E_executed accounting
};

// getSDFofSweptVolume<false,*> (sw_manager.hpp:844-866) = choiceTInit (:538-581) + gradientDescent (:1249-1325),
// executed cooperatively by one warp. All lanes return the same values.
//
// After the table-driven layer 1 and the three 21-sample layers of choiceTInit, the descent is organised as ROUNDS of one
// SDF evaluation per lane, driven by a small warp-uniform state machine with a single eval_sdf call site:
//   M_F0   f(x0) when no sample was below the initial 1e9 (degenerate input; the reference evaluates it at iter == 0)
//   M_A    first descent step: lanes 0-14 x - tau_j (slope sign +1), 15-29 x + tau_j (sign -1), j = 0..14; 30/31 slope
//   M_B    halvings j = 15..28 in the known direction (only if M_A found no decreasing candidate)
//   M_P    29 halvings in the PREDICTED direction + slope on lanes 30/31
//   M_M    29 halvings in the actual direction after a misprediction
// Decisions are the sequential loop's: the slope's sign always comes from the finite difference on lanes 30/31, and the
// accepted halving is the first (largest step) whose candidate decreases f.
// SCALED: choiceTInit stays rigid whatever useScale says (its four layers call the rigid posEva2Rel, :569-570); the
// descent evaluates the scaled body, so f(x0) is not choiceTInit's minimum and is evaluated first (M_F0), as the reference
// does at iter == 0.
template <int SHAPE, bool XFORM, bool SCALED>
__device__ __forceinline__ OuterResult solve_outer(const TrajView &tv, const ShapeParams &S, const ScaleParams &Z, double px,
                                                   double py, bool have_seed = false, double seed_in = 0.0,
                                                   double min_in = 1e9) {
    const int lane = threadIdx.x & 31;
    const double D = tv.D;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    int evals = 0;

    // ---- choiceTInit layer 1: shared lattice t_k (accumulated 0.15 adds) with the pose table ----
    // Exact pruning as in thread_choice_t_init: the result is the lexicographic minimum of (f_k, k) over the samples with
    // f_k < 1e9, and f_k >= |p - x_k| - S.rout.  The 32 lattice poses around the one nearest to p are evaluated first (one
    // round: this already contains the minimum almost always), then every block of 32 is revisited and only samples with
    // |p - x_k| <= min + rout are evaluated (usually none).  (Skipped when the caller ran choiceTInit thread-per-point.)
    double min_dis = have_seed ? min_in : 1e9, seed = have_seed ? seed_in : 0.0;
    if (!have_seed) {
        const uint32_t row = 8u * (uint32_t)tv.K1pad;
        const int K1 = tv.K1;
        // nearest lattice pose
        double bd2 = INF;
        int k0 = 0;
        for (int k = lane; k < K1; k += 32) {
            const uint32_t ps = tv.spose + 8u * (uint32_t)k;
            const double ax = px - lds_f64(ps), ay = py - lds_f64(ps + row);
            const double d2 = ax * ax + ay * ay;
            if (d2 < bd2) { bd2 = d2; k0 = k; }
        }
        {
            double v = bd2;
            const int src = warp_argmin_lane(v);
            k0 = __shfl_sync(FULL, k0, src);
        }
        const int w0 = max(0, min(k0 - 16, K1 - 32));   // window [w0, w0 + 32) (whole lattice when K1 <= 32)
        int kb = -1;
        double thr2 = INF;
        // it = -1: the window; it >= 0: block it (samples of the window are not evaluated twice)
        for (int it = -1; 32 * it < K1; ++it) {
            const int k = (it < 0) ? w0 + lane : 32 * it + lane;
            bool need = k >= 0 && k < K1;
            double rx = 0.0, ry = 0.0;
            if (need) {
                const uint32_t ps = tv.spose + 8u * (uint32_t)k;
                const double xk = lds_f64(ps), yk = lds_f64(ps + row);
                const double ax = px - xk, ay = py - yk;
                need = (it < 0) || ((ax * ax + ay * ay <= thr2) && !(k >= w0 && k < w0 + 32));
                if (need) rel_from_pose(px, py, xk, yk, lds_f64(ps + 2 * row), lds_f64(ps + 3 * row), rx, ry);
            }
            const unsigned mneed = __ballot_sync(FULL, need);
            if (mneed == 0u) continue;
            double f = INF;
            if (need) {
                f = dev::shape_sdf<SHAPE, XFORM>(S, rx, ry);
                if (!(f == f)) f = INF;
            }
            evals += __popc(mneed);
            const int kl = k - lane + warp_argmin_lane(f);   // first lane holding the block minimum; f := that minimum
            if (__any_sync(FULL, f < min_dis || (f == min_dis && f < 1e9 && kl < kb))) {
                min_dis = f;
                kb = kl;
                const double thr0 = f * S.prune_scale + S.rout, thr = fmax(thr0, S.prune_rmin);  // analytic shapes: f * 1 + rout, max with 0
                thr2 = (thr0 >= 0.0) ? thr * thr : INF;
            }
        }
        seed = (kb >= 0) ? lds_f64(tv.slat + 8u * (uint32_t)kb) : 0.0;
    }

    // ---- choiceTInit layers 2..4: 21-sample window around the seed, dt *= 0.1 per layer, one sample per lane ----
    if (!have_seed) {
        double dt = 0.15;
        int hint = 0;
#pragma unroll 1
        for (int layer = 2; layer <= 4; ++layer) {
            dt *= 0.1;
            double t = smaxd(0.0, seed - 10 * dt);
            const double term = smind(D, seed + 10 * dt);
#pragma unroll
            for (int i = 0; i < 20; ++i)
                if (i < lane) t += dt;  // lane k (<= 20) holds t0 + dt added k times (same rounding as the loop)
            const double fq = eval_sdf<SHAPE, XFORM>(tv, S, px, py, t, hint);
            const bool lat_valid = (lane <= 20) && (t <= term);
            double fl = (lat_valid && (fq == fq)) ? fq : INF;
            evals += __popc(__ballot_sync(FULL, lat_valid));
            const int kb = warp_argmin_lane(fl);  // fl := warp minimum
            const double tb = __shfl_sync(FULL, t, kb);
            if (__any_sync(FULL, fl < min_dis)) {
                min_dis = fl;
                seed = tb;
            }
        }
    }

    // ---- gradientDescent (:1249-1325) from x0 = seed, bounds [ts-3.4, ts+3.4] ∩ [0, D] (:856-857) ----
    // ROUNDS of one evaluation per lane.  Per-lane round constants: tau (step of this lane's candidate), sbit (sign bit
    // of the offset: candidates move against the slope direction the round assumes) and the clamp interval — the
    // descent interval for candidates, [0, +inf) / (-inf, D] for the two finite-difference samples on lanes 30 / 31
    // (smaxd(0, x - 1e-6), smind(D, x + 1e-6): :798-806).  They change only when the round type changes.
    enum { M_F0 = 0, M_A, M_B, M_P, M_M };
    const double t_min = smaxd(0.0, seed - 3.4), t_max = smind(seed + 3.4, D);
    const bool slope_lane = lane >= 30;
    const double lo_l = slope_lane ? (lane == 30 ? 0.0 : -INF) : t_min;
    const double hi_l = slope_lane ? (lane == 30 ? INF : D) : t_max;
    const int hi001 = __double2hiint(0.01), lo001 = __double2loint(0.01);
    // alpha = 0.01 halved j times: exact, so subtract j from the exponent field (0.01 * 2^-46 is still normal)
    const int tauP_hi = slope_lane ? __double2hiint(0.000001) : hi001 - (lane << 20);
    const int tau_lo = slope_lane ? __double2loint(0.000001) : lo001;
    const unsigned sbit_fix = (lane == 30) ? 0x80000000u : 0u;  // lane 30: x - 1e-6, lane 31: x + 1e-6
    double x = seed, fx = min_dis, prev_x = 10000000.0;
    int iter = 0, pred = 0, sgn = 0, hint = 0;
    int mode;
    int tau_hi;        // this lane's step, high word
    unsigned sbit;     // this lane's offset sign bit
    if (SCALED || __any_sync(FULL, min_dis >= 1e9)) {
        // nothing below the initial 1e9 (degenerate input), or a scaled body: the reference evaluates f(x0) at iter == 0
        mode = M_F0;
        tau_hi = 0; sbit = 0;   // offset +0.0: the sample is x itself
    } else {
        mode = M_A;
        prev_x = x;             // `prev_x = x` after the (true) first loop test
        tau_hi = slope_lane ? tauP_hi : hi001 - (((lane < 15) ? lane : lane - 15) << 20);
        sbit = slope_lane ? sbit_fix : ((lane < 15) ? 0x80000000u : 0u);
    }
    bool running = true;
#pragma unroll 1
    while (running) {
        const double off = __hiloint2double(tau_hi ^ (int)sbit, (mode == M_F0) ? 0 : tau_lo);
        const double tq = smaxd(smind(x + off, hi_l), lo_l);
        const double fq = eval_sdf<SHAPE, XFORM, SCALED>(tv, S, Z, px, py, tq, hint);
        const unsigned m_dec = __ballot_sync(FULL, (fq - fx) < 0);  // candidates that decrease f
        int jacc = -1, src = 0;
        bool failed = false, step_end = true;
        if (mode == M_P) {
            // 29 halvings in the predicted direction + the slope: the common round
            evals += 31;
            const double g = (__shfl_sync(FULL, fq, 31) - __shfl_sync(FULL, fq, 30)) * 500000;
            sgn = (int)__any_sync(FULL, g > 0) - (int)__any_sync(FULL, g < 0);  // (int)(g > 0) - (g < 0)
            const unsigned m = m_dec & 0x1fffffffu;
            if (sgn != 0 && sgn != pred) {  // mispredicted: redo the halvings in the actual direction
                mode = M_M;
                sbit = (sgn > 0) ? 0x80000000u : 0u;
                step_end = false;
            } else if (sgn != 0 && m) {
                jacc = __ffs(m) - 1; src = jacc;
            } else failed = true;
        } else if (mode == M_M) {
            evals += 29;
            const unsigned m = m_dec & 0x1fffffffu;
            if (m) { jacc = __ffs(m) - 1; src = jacc; }
            else failed = true;
        } else if (mode == M_A) {
            // first step: lanes 0-14 x - tau_j (slope sign +1), 15-29 x + tau_j (sign -1), j = 0..14; 30/31 slope
            evals += 32;
            const double g = (__shfl_sync(FULL, fq, 31) - __shfl_sync(FULL, fq, 30)) * 500000;
            sgn = (int)__any_sync(FULL, g > 0) - (int)__any_sync(FULL, g < 0);
            const unsigned grp = (sgn > 0) ? (m_dec & 0x7fffu) : ((m_dec >> 15) & 0x7fffu);
            if (sgn == 0) failed = true;
            else if (grp) { jacc = __ffs(grp) - 1; src = (sgn > 0) ? jacc : jacc + 15; }
            else {  // halvings j = 15..28 in the known direction
                mode = M_B;
                tau_hi = hi001 - ((15 + lane) << 20);
                sbit = (sgn > 0) ? 0x80000000u : 0u;
                step_end = false;
            }
        } else if (mode == M_B) {
            evals += 14;
            const unsigned mb = m_dec & 0x3fffu;
            if (mb) { src = __ffs(mb) - 1; jacc = 15 + src; }
            else failed = true;
        } else {  // M_F0
            fx = __shfl_sync(FULL, fq, 0);
            evals += 1;
        }
        if (jacc >= 0) {
            const double xacc = __shfl_sync(FULL, tq, src), facc = __shfl_sync(FULL, fq, src);
            // a full, unclamped stride means we are still walking downhill: same slope sign next; otherwise the step
            // overshot the minimiser (tau_j is the largest decreasing step) and the slope flips
            const bool walking = (jacc == 0) && __all_sync(FULL, xacc == x + (-0.01 * (double)sgn));
            pred = walking ? sgn : -sgn;
            x = xacc;
            fx = facc;
            iter += jacc + 1;
        } else if (failed) {
            iter += 29;
        }
        if (step_end) {
            // while (iter < max_iter && !stop && abs(x - prev_x) > tol)   (:1288)
            running = (iter < 1000) && !failed && __all_sync(FULL, fabs(x - prev_x) > 1e-16);
            prev_x = x;
            if (pred == 0) {  // only after M_F0: first descent step
                mode = M_A;
                tau_hi = slope_lane ? tauP_hi : hi001 - (((lane < 15) ? lane : lane - 15) << 20);
                sbit = slope_lane ? sbit_fix : ((lane < 15) ? 0x80000000u : 0u);
            } else {
                mode = M_P;
                tau_hi = tauP_hi;
                sbit = slope_lane ? sbit_fix : ((pred > 0) ? 0x80000000u : 0u);
            }
        }
    }
    OuterResult R;
    R.sdf = fx;
    R.tstar = x;
    R.evals = evals;
    return R;
}

// getGradPrelAtTimeStamp (sw_manager.hpp:779-795) -> getonlyGrad1: central FD, dx = 1e-6 in the body frame
// (Shape.hpp:35-53), or the Polygon's analytic override (Shape.hpp:1508-1534). 4 lanes do the 4 evaluations.
template <int SHAPE, bool XFORM, bool SCALED>
__device__ __forceinline__ void grad_prel(const TrajView &tv, const ShapeParams &S, const ScaleParams &Z, double px, double py,
                                          double t, double &gx, double &gy) {
    const int lane = threadIdx.x & 31;
    double rx, ry;
    if (SCALED) {
        int hint = 0;
        rel_at_scaled(tv, Z, px, py, t, hint, rx, ry);
    } else {
        double x, y, yaw, sy, cy;
        traj_pos(tv, t, x, y, yaw);
        dev::sincos_portable(yaw, sy, cy);
        rel_from_pose(px, py, x, y, cy, sy, rx, ry);
    }
    if (SHAPE == SH_POLYGON) {
        dev::PolyHit H = dev::polygon_scan(S, rx, ry);
        double vx = rx - H.cx, vy = ry - H.cy;
        double z = vx * vx + vy * vy;
        if (z > 0.0) {
            double n = sqrt(z);
            vx /= n; vy /= n;
        }
        if (H.rs % 2 != 0) { vx = -vx; vy = -vy; }
        gx = vx; gy = vy;
        return;
    }
    if (SHAPE == SH_CIRCLE) {
        dev::circle_grad1<XFORM>(S, rx, ry, gx, gy);
        return;
    }
    const double dx = 0.000001;
    double qx = rx, qy = ry;
    if (lane == 0) { qx -= dx; }
    if (lane == 1) { qx -= dx; qx += 2 * dx; }
    if (lane == 2) { qy -= dx; }
    if (lane == 3) { qy -= dx; qy += 2 * dx; }
    double f = dev::shape_sdf<SHAPE, XFORM>(S, qx, qy);
    double f0 = __shfl_sync(FULL, f, 0), f1 = __shfl_sync(FULL, f, 1);
    double f2 = __shfl_sync(FULL, f, 2), f3 = __shfl_sync(FULL, f, 3);
    gx = (f1 - f0) / (2 * dx);
    gy = (f3 - f2) / (2 * dx);
}

// smoothedL1 (back_end_optimizer.hpp:316-340), mu = 0.01
__device__ __forceinline__ bool smoothed_l1(double x, double mu, double &f, double &df) {
    if (x < 0.0) return false;
    if (x > mu) {
        f = x - 0.5 * mu;
        df = 1.0;
        return true;
    }
    const double xdmu = x / mu;
    const double sqrxdmu = xdmu * xdmu;
    const double mumxd2 = mu - 0.5 * x;
    f = mumxd2 * sqrxdmu * xdmu;
    df = sqrxdmu * ((-0.5) * xdmu + 3.0 * mumxd2 / mu);
    return true;
}

// Per-point penalty and chain rule: the loop body of addSaftyPenaOnSweptVolumeParallelTrueSDF after the SDF
// query (back_end_optimizer.hpp:797-854) with grad_cost_p_sw (:1031-1066).
// In: world point p, sdf, t*, gradient g (body frame for sdf > 0; world-frame GSIP direction otherwise).
// Out (uniform across the warp): piece index, beta0[6], G[3] = w_p * (d/dx, d/dy, d/dyaw), gdT, pena.
struct Contribution {
    int piece;
    double s1;
    double G[3];
    double gdT, pena;
    bool active;
};
// SCALED (St = getScale(t*), :827): the xy part is -L' (-S^-T R g); the yaw part keeps the reference's g^T VR^T (p - x),
// which misses the S^-1 of the true derivative, unless Z.exact_yaw_grad asks for g^T VR^T S^-1 (p - x).
template <bool SCALED>
__device__ __forceinline__ Contribution point_contribution(const TrajView &tv, const CostParams &cp, const ScaleParams &Z,
                                                           double px, double py, double sdf, double tstar, double gx,
                                                           double gy) {
    Contribution C;
    double tl = tstar;
    int i = locate_piece(tv, tl);
    const double *c = tv.c + 18 * i;
    double s1 = tl, s2 = s1 * s1, s3 = s2 * s1, s4 = s2 * s2, s5 = s4 * s1;
    double b0[6] = {1.0, s1, s2, s3, s4, s5};
    double b1[6] = {0.0, 1.0, 2.0 * s1, 3.0 * s2, 4.0 * s3, 5.0 * s4};
    double pos[3], vel[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int q = 0; q < 6; ++q) {
            a += c[6 * d + q] * b0[q];
            b += c[6 * d + q] * b1[q];
        }
        pos[d] = a;
        vel[d] = b;
    }
    double yaw = pos[2], sy, cy;
    dev::sincos_portable(yaw, sy, cy);
    if (sdf < 0) {  // :832 world -> body
        double g0 = cy * gx + sy * gy;
        double g1 = -sy * gx + cy * gy;
        gx = g0; gy = g1;
    }
    double sdf_cost = -1.0, sdf_out_grad = 0.0;
    smoothed_l1(cp.safety_hor - sdf, 0.01, sdf_cost, sdf_out_grad);
    C.piece = i;
    C.s1 = s1;
    C.G[0] = C.G[1] = C.G[2] = 0.0;
    C.gdT = 0.0;
    C.pena = 0.0;
    C.active = false;
    if (sdf_cost > 0) {
        double i00 = 1.0, i11 = 1.0;
        if (SCALED) scale_inv(Z, tstar, i00, i11);
        // (-S^-T R) g: rows -(i00 c, -i00 s), -(i11 s, i11 c)
        double rg0 = SCALED ? -((i00 * cy) * gx + (-(i00 * sy)) * gy) : -(cy * gx + (-sy) * gy);
        double rg1 = SCALED ? -((i11 * sy) * gx + (i11 * cy) * gy) : -(sy * gx + cy * gy);
        double sg0 = -sdf_out_grad * rg0, sg1 = -sdf_out_grad * rg1;
        double d0 = px - pos[0], d1 = py - pos[1];
        if (SCALED && Z.exact_yaw_grad) { d0 = i00 * d0; d1 = i11 * d1; }
        double w0 = -sy * d0 + cy * d1;
        double w1 = -cy * d0 + -sy * d1;
        double gyaw = (-sdf_out_grad * gx) * w0 + (-sdf_out_grad * gy) * w1;
        C.G[0] = cp.weight_p * sg0;
        C.G[1] = cp.weight_p * sg1;
        C.G[2] = cp.weight_p * gyaw;
        C.pena = cp.weight_p * sdf_cost;
        C.gdT = -(C.G[0] * vel[0] + C.G[1] * vel[1] + C.G[2] * vel[2]);
        C.active = true;
    }
    return C;
}

// ------------------------------------------------------------------------------------------------
// Thread-per-point pieces used by the batched path of k_outer (32 points per warp at a time): the parts of the
// per-point work that have no intra-point parallelism worth a warp are run one point per LANE, literally as the
// reference's loops, and only gradientDescent (29-way speculative) stays one point per WARP.
// ------------------------------------------------------------------------------------------------
// choiceTInit<false>(p, 0.15) (sw_manager.hpp:538-581); layer 1 reads the shared pose table.
//
// Layer 1 (the 0.15 s lattice over the whole trajectory, K1 = 134 samples at D = 20 s) is an arg-min with the rule
// "first strict minimum wins, nothing >= 1e9 wins".  That result is the lexicographic minimum of (f_k, k) over the samples
// with f_k < 1e9, whatever the order of evaluation — so samples that PROVABLY cannot attain the minimum need not be
// evaluated.  The shape functors are distances outside the shape: f_k = sdf(R_k^T (p - x_k)) >= |p - x_k| - rout
// (S.rout: circumradius + margin, checked against the oracle for every shape).  Pass 1 finds the lattice pose nearest to p
// (5 flops per sample) and evaluates it: m; pass 2 walks k upwards and evaluates only samples with
// |p - x_k| <= m + rout, tightening m as it goes.  A skipped sample has f_k > m >= the final minimum.  Typically ~15 of
// the 134 samples survive; bits identical to the full scan (GPU parity tests, strict build).
template <int SHAPE, bool XFORM>
__device__ __forceinline__ void thread_choice_t_init(const TrajView &tv, const ShapeParams &S, double px, double py,
                                                     double &seed, double &min_dis, int &evals) {
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    const uint32_t row = 8u * (uint32_t)tv.K1pad;
    const int K1 = tv.K1;
    // pass 1: nearest lattice pose (rows are 16-byte aligned and K1pad is even: two samples per load)
    double bd2 = INF;
    int k0 = 0;
    {
        uint32_t ps = tv.spose;
#pragma unroll 1
        for (int k = 0; k < K1; k += 2, ps += 16) {
            double x0, x1, y0, y1;
            lds_v2(ps, x0, x1);
            lds_v2(ps + row, y0, y1);
            const double ax = px - x0, ay = py - y0, bx = px - x1, by = py - y1;
            const double d0 = ax * ax + ay * ay, d1 = bx * bx + by * by;
            if (d0 < bd2) { bd2 = d0; k0 = k; }
            if (k + 1 < K1 && d1 < bd2) { bd2 = d1; k0 = k + 1; }
        }
    }
    // pass 2: the nearest pose first (it = -1), then every sample that can still reach the minimum, k ascending; ties are
    // resolved towards the smaller k, so the visiting order does not matter.  One functor call site.
    min_dis = 1e9;
    int kb = -1, ne = 0;
    double thr2 = INF;  // squared pruning radius: |p - x_k| > min_dis + rout  =>  f_k > min_dis
#pragma unroll 1
    for (int it = -1; it < K1; ++it) {
        const int k = (it < 0) ? k0 : it;
        const uint32_t ps = tv.spose + 8u * (uint32_t)k;
        const double xk = lds_f64(ps), yk = lds_f64(ps + row);
        const double ax = px - xk, ay = py - yk;
        const double d2 = ax * ax + ay * ay;
        if (it >= 0 && (!(d2 <= thr2) || k == k0)) continue;
        double rx, ry;
        rel_from_pose(px, py, xk, yk, lds_f64(ps + 2 * row), lds_f64(ps + 3 * row), rx, ry);
        const double f = dev::shape_sdf<SHAPE, XFORM>(S, rx, ry);
        ++ne;
        if (f < min_dis || (f == min_dis && k < kb)) {
            min_dis = f;
            kb = k;
            const double thr0 = f * S.prune_scale + S.rout, thr = fmax(thr0, S.prune_rmin);  // analytic shapes: f * 1 + rout, max with 0
            thr2 = (thr0 >= 0.0) ? thr * thr : INF;      // < 0 cannot happen for a distance function; then no pruning
        }
    }
    seed = (kb >= 0) ? lds_f64(tv.slat + 8u * (uint32_t)kb) : 0.0;
    evals += ne;
    double dt = 0.15;
    int hint = 0;  // piece of the previous sample (the windows are <= 0.3 s wide)
#pragma unroll 1
    for (int layer = 2; layer <= 4; ++layer) {
        dt *= 0.1;
        double t = smaxd(0.0, seed - 10 * dt);
        const double term = smind(tv.D, seed + 10 * dt);
#pragma unroll 1
        for (; t <= term; t += dt) {
            const double f = eval_sdf<SHAPE, XFORM>(tv, S, px, py, t, hint);
            ++evals;
            if (f < min_dis) {
                seed = t;
                min_dis = f;
            }
        }
    }
}

// getGradPrelAtTimeStamp (sw_manager.hpp:779-795) -> getonlyGrad1 (Shape.hpp:35-53), one point per thread
template <int SHAPE, bool XFORM, bool SCALED>
__device__ __forceinline__ void thread_grad_prel(const TrajView &tv, const ShapeParams &S, const ScaleParams &Z, double px,
                                                 double py, double t, double &gx, double &gy) {
    double rx, ry;
    if (SCALED) {
        int hint = 0;
        rel_at_scaled(tv, Z, px, py, t, hint, rx, ry);
    } else {
        double x, y, yaw, sy, cy;
        traj_pos(tv, t, x, y, yaw);
        dev::sincos_portable(yaw, sy, cy);
        rel_from_pose(px, py, x, y, cy, sy, rx, ry);
    }
    if (SHAPE == SH_POLYGON) {
        dev::PolyHit H = dev::polygon_scan(S, rx, ry);
        double vx = rx - H.cx, vy = ry - H.cy;
        double z = vx * vx + vy * vy;
        if (z > 0.0) {
            double n = sqrt(z);
            vx /= n; vy /= n;
        }
        if (H.rs % 2 != 0) { vx = -vx; vy = -vy; }
        gx = vx; gy = vy;
        return;
    }
    if (SHAPE == SH_CIRCLE) {
        dev::circle_grad1<XFORM>(S, rx, ry, gx, gy);
        return;
    }
    const double dx = 0.000001;
    double f[4];
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {  // (x-dx), (x-dx)+2dx, (y-dx), (y-dx)+2dx — one evaluation site
        double qx = rx, qy = ry;
        if (q < 2) { qx -= dx; if (q == 1) qx += 2 * dx; }
        else { qy -= dx; if (q == 3) qy += 2 * dx; }
        f[q] = dev::shape_sdf<SHAPE, XFORM>(S, qx, qy);
    }
    gx = (f[1] - f[0]) / (2 * dx);
    gy = (f[3] - f[2]) / (2 * dx);
}

// ------------------------------------------------------------------------------------------------
// gradientDescent (sw_manager.hpp:1249-1325) for a BATCH of points, a quarter warp (8 lanes) per point, four points in
// flight per warp — the batched path of k_outer and the interior-branch kernel.
//
// The reference's loop, per descent step: slope sign from the finite difference at x (2 evaluations, recomputed for every
// halving in the reference but always at the same x, hence the same bits), then candidates x - sign * 0.01 * 2^-j for
// j = 0, 1, ... until the first one that decreases f (29 failures end the descent).  Measured on configs 1-3 (oracle,
// orc_descent_stats): ~8 steps per point, accepted j spread evenly over 7..20 (never 1..6), so a full warp per step
// (29 candidates + slope, the round-1 design) spends most of its lanes on candidates beyond the accepted one, and one lane per
// point (sequential, 155 +- 65 evaluations) leaves the warp waiting for its slowest lane.  Eight lanes per point in
// rounds of one evaluation per lane:
//   R1   lanes 0/1 of the quarter: the two finite-difference samples; lanes 2..7: candidates j = 0..5 in the PREDICTED
//        direction (the slope flips after every non-full step because the accepted step is the largest decreasing one)
//   RN   candidates j = jbase .. jbase + 7 in the known direction (jbase = 6, 14, 22 after R1; 0, 8, 16, 24 after a
//        misprediction)
//   F0   f(x0) when choiceTInit found nothing below 1e9 (degenerate input; the reference evaluates it at iter == 0)
// => ~21 lane-evaluations per step instead of 31.  A quarter that finishes its point stores (sdf, t*) and takes the next
// point of the batch (warp-uniform cursor), so the four quarters stay busy until the batch runs dry.  Every decision is
// the sequential loop's decision given the same SDF values: the accepted halving is the FIRST j whose candidate
// decreases f, the sign comes from the finite difference — bit-identical results (GPU parity tests, strict build).
// In: lane i (< nb) holds point i of the batch (px, py, choiceTInit seed and minimum).  Out: res[2 i] = sdf, res[2 i + 1] = t*.
// ------------------------------------------------------------------------------------------------
template <int SHAPE, bool XFORM, bool SCALED>
__device__ __forceinline__ void descent_engine(const TrajView &tv, const ShapeParams &S, const ScaleParams &Z, int nb, double mpx, double mpy,
                                               double mseed, double mmin, double *res, unsigned &evals) {
    enum { E_F0 = 0, E_R1 = 1, E_RN = 2 };
    const int lane = threadIdx.x & 31, q = lane & 7, qbase = lane & 24;
    const double D = tv.D;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    const int hi001 = __double2hiint(0.01), lo001 = __double2loint(0.01);
    // state of this lane's quarter (identical in its 8 lanes)
    int pt = -1, mode = E_R1, iter = 0, pred = 1, sgn = 1, jbase = 0, hint = 0;
    double px = 0.0, py = 0.0, x = 0.0, fx = 0.0, prev_x = 0.0, t_min = 0.0, t_max = 0.0;
    bool need = true;   // the quarter wants a point
    int next_i = 0;     // warp-uniform cursor into the batch
#pragma unroll 1
    for (;;) {
        // ---- hand the next points of the batch to the quarters that are free ----
        const unsigned want = __ballot_sync(FULL, need && q == 0);
        if (want) {
            const int cand = next_i + __popc(want & ((1u << qbase) - 1u));
            next_i += __popc(want);
            const bool take = need && cand < nb;
            const int src = take ? cand : lane;
            const double npx = __shfl_sync(FULL, mpx, src), npy = __shfl_sync(FULL, mpy, src);
            const double nsd = __shfl_sync(FULL, mseed, src), nmn = __shfl_sync(FULL, mmin, src);
            if (need) {
                need = false;
                pt = -1;
                if (take) {
                    pt = cand;
                    px = npx; py = npy;
                    x = nsd; fx = nmn; prev_x = nsd;   // `prev_x = x` after the (true) first loop test
                    t_min = smaxd(0.0, nsd - 3.4);      // :856-857
                    t_max = smind(nsd + 3.4, D);
                    iter = 0; pred = 1; sgn = 1; jbase = 0; hint = 0;
                    mode = (SCALED || nmn >= 1e9) ? E_F0 : E_R1;
                }
            }
        }
        if (!__any_sync(FULL, pt >= 0)) break;

        // ---- this lane's sample (straight-line code: the four quarters are in different modes) ----
        const bool isR1 = mode == E_R1, isF0 = mode == E_F0;
        const bool slope = isR1 && q < 2;
        const int j = isR1 ? q - 2 : jbase + q;
        const bool cand = !isF0 && !slope && j <= 28;
        evals += (pt >= 0 && (cand || slope || (isF0 && q == 0))) ? 1u : 0u;
        // candidate: tau = 0.01 halved j times (exact: subtract j from the exponent field); change = -tau * sign
        const int dir = isR1 ? pred : sgn;
        const int tau_hi = (hi001 - ((j & 31) << 20)) ^ ((dir > 0) ? (int)0x80000000 : 0);
        // slope samples: t1 = max(0, x - 1e-6), t2 = min(D, x + 1e-6)   (:798-806)
        const double off = slope ? ((q == 0) ? -0.000001 : 0.000001) : __hiloint2double(tau_hi, lo001);
        const double lo_l = slope ? ((q == 0) ? 0.0 : -INF) : t_min;
        const double hi_l = slope ? ((q == 0) ? INF : D) : t_max;
        const double tc = smaxd(smind(x + off, hi_l), lo_l);
        const double tq = (cand || slope) ? tc : x;
        const double fq = eval_sdf<SHAPE, XFORM, SCALED>(tv, S, Z, px, py, tq, hint);

        // ---- collectives (all lanes), then each quarter's decision, again without branches ----
        const unsigned m8 = (__ballot_sync(FULL, (fq - fx) < 0) >> qbase) & 0xffu;
        const double f0 = __shfl_sync(FULL, fq, qbase), f1 = __shfl_sync(FULL, fq, qbase + 1);
        const double g = (f1 - f0) * 500000;
        const int s_new = (int)(g > 0) - (int)(g < 0);
        sgn = isR1 ? s_new : sgn;
        const bool zero = isR1 && sgn == 0;              // all 29 candidates equal x: none decreases f
        const bool mispred = isR1 && sgn != 0 && sgn != pred;
        const int nvalid = max(0, min(8, 29 - jbase));   // (idle quarters keep counting jbase up)
        const unsigned mc = isR1 ? (m8 >> 2) : (m8 & ((1u << nvalid) - 1u));
        const bool hit = (pt >= 0) && !isF0 && !zero && !mispred && mc != 0u;   // first decreasing candidate found
        const int k = __ffs(mc) - 1;
        const int jacc = isR1 ? k : jbase + k;
        const int src = hit ? qbase + (isR1 ? k + 2 : k) : lane;
        const double xacc = __shfl_sync(FULL, tq, src), facc = __shfl_sync(FULL, fq, src);
        // no decreasing candidate in this round: next chunk of halvings (R1: j = 6.., or j = 0.. after a misprediction)
        const int jb_next = isR1 ? (mispred ? 0 : 6) : jbase + 8;
        const bool failed = (pt >= 0) && !isF0 && (zero || (!hit && !mispred && jb_next > 28));
        // a full, unclamped stride means we are still walking downhill: same slope sign next; otherwise the step overshot
        // the minimiser (tau_j is the largest decreasing step) and the slope flips
        const bool walking = (jacc == 0) && (xacc == x + (-0.01 * (double)sgn));
        pred = hit ? (walking ? sgn : -sgn) : pred;
        iter += hit ? jacc + 1 : (failed ? 29 : 0);
        x = hit ? xacc : x;
        fx = hit ? facc : (isF0 ? f0 : fx);
        const bool step_end = hit || failed;
        // while (iter < max_iter && !stop && abs(x - prev_x) > tol)   (:1288)
        const bool running = (iter < 1000) && !failed && (fabs(x - prev_x) > 1e-16);
        prev_x = step_end ? x : prev_x;
        mode = (step_end || isF0) ? E_R1 : E_RN;
        jbase = jb_next;
        if (step_end && !running) {
            if (q == 0) { res[2 * pt] = fx; res[2 * pt + 1] = x; }
            pt = -1;
            need = true;
        }
    }
    __syncwarp();
}

// descent_engine with TWO samples per lane: a group of 4 lanes per point (8 points in flight per warp), each lane evaluates
// samples s = q and s = q + 4 of its group's round (same rounds as above: R1 = 2 slope samples + candidates j = 0..5,
// RN = candidates jbase..jbase + 7).  The two evaluations are independent instruction streams (latency hiding inside the
// thread, on top of the resident warps) and the per-round bookkeeping is paid once per two evaluations.
// wk: per-warp shared work area, 4 doubles per point in (px, py, seed, min), 2 doubles per point out (sdf, t*) at wk[4 i].
// The queue of prepared points is shared by the CTA's 8 warps (wk: 8 x 32 entries of 4 doubles, entry (w, i) at
// wk[4 (32 w + i)], valid for i < nbw[w]; served in the order i-major, w-minor through the shared cursor): a group that
// finishes its point takes the next one of the whole CTA, so the warps of a CTA finish together whatever the lengths of
// their own descents.  Which group solves a point does not change its result; the reductions stay per warp, fixed order.
template <int SHAPE, bool XFORM, bool SCALED>
__device__ __forceinline__ void descent_engine2(const TrajView &tv, const ShapeParams &S, const ScaleParams &Z, double *wk, const int *nbw, int *cursor,
                                                int limit, unsigned &evals) {
    enum { E_F0 = 0, E_R1 = 1, E_RN = 2 };
    const int lane = threadIdx.x & 31, q = lane & 3, gbase = lane & 28;
    const double D = tv.D;
    const double INF = __longlong_as_double(0x7ff0000000000000LL);
    const int hi001 = __double2hiint(0.01), lo001 = __double2loint(0.01);
    int pt = -1, mode = E_R1, iter = 0, pred = 1, sgn = 1, jbase = 0, hintA = 0, hintB = 0;
    double px = 0.0, py = 0.0, x = 0.0, fx = 0.0, prev_x = 0.0, t_min = 0.0, t_max = 0.0;
    bool need = true;
#pragma unroll 1
    for (;;) {
        const unsigned want = __ballot_sync(FULL, need && q == 0);
        if (want) {
            int base = 0;
            if (lane == 0) base = atomicAdd(cursor, __popc(want));
            base = __shfl_sync(FULL, base, 0);
            const int c = base + __popc(want & ((1u << gbase) - 1u));
            if (need) {
                pt = -1;
                const int cw = c & (kWarpsPerBlock - 1), ci = c >> 3;     // entry (warp cw, point ci)
                need = c < limit;                                          // a hole (ci >= nbw[cw]): ask again
                if (c < limit && ci < nbw[cw]) {
                    need = false;
                    pt = 32 * cw + ci;
                    const double *w = wk + 4 * pt;
                    px = w[0]; py = w[1];
                    const double nsd = w[2], nmn = w[3];
                    x = nsd; fx = nmn; prev_x = nsd;
                    t_min = smaxd(0.0, nsd - 3.4);
                    t_max = smind(nsd + 3.4, D);
                    iter = 0; pred = 1; sgn = 1; jbase = 0; hintA = 0; hintB = 0;
                    mode = (SCALED || nmn >= 1e9) ? E_F0 : E_R1;   // scaled: f(x0) is not choiceTInit's minimum
                }
            }
        }
        if (!__any_sync(FULL, pt >= 0)) {
            if (__any_sync(FULL, need)) continue;   // drew only holes: ask again (the queue is not exhausted yet)
            break;
        }

        const bool isR1 = mode == E_R1, isF0 = mode == E_F0;
        const int dir = isR1 ? pred : sgn;
        const int sbit = (dir > 0) ? (int)0x80000000 : 0;
        // slot A: sample s = q (R1: s = 0, 1 are the slope samples, s = 2, 3 candidates j = 0, 1); slot B: s = q + 4
        const bool slopeA = isR1 && q < 2;
        const int jA = isR1 ? q - 2 : jbase + q;
        const int jB = isR1 ? q + 2 : jbase + q + 4;
        const bool candA = !isF0 && !slopeA && jA <= 28, candB = !isF0 && jB <= 28;
        evals += (pt >= 0) ? ((candA || slopeA || (isF0 && q == 0)) ? 1u : 0u) + (candB ? 1u : 0u) : 0u;
        const double offA = slopeA ? ((q == 0) ? -0.000001 : 0.000001) : __hiloint2double((hi001 - ((jA & 31) << 20)) ^ sbit, lo001);
        const double offB = __hiloint2double((hi001 - ((jB & 31) << 20)) ^ sbit, lo001);
        const double loA = slopeA ? ((q == 0) ? 0.0 : -INF) : t_min, hiA = slopeA ? ((q == 0) ? INF : D) : t_max;
        const double tcA = smaxd(smind(x + offA, hiA), loA), tcB = smaxd(smind(x + offB, t_max), t_min);
        const double tA = (candA || slopeA) ? tcA : x, tB = candB ? tcB : x;
        const double fA = eval_sdf<SHAPE, XFORM, SCALED>(tv, S, Z, px, py, tA, hintA);
        const double fB = eval_sdf<SHAPE, XFORM, SCALED>(tv, S, Z, px, py, tB, hintB);

        const unsigned balA = __ballot_sync(FULL, (fA - fx) < 0), balB = __ballot_sync(FULL, (fB - fx) < 0);
        const unsigned m8 = ((balA >> gbase) & 0xfu) | (((balB >> gbase) & 0xfu) << 4);
        const double f0 = __shfl_sync(FULL, fA, gbase), f1 = __shfl_sync(FULL, fA, gbase + 1);
        const double g = (f1 - f0) * 500000;
        const int s_new = (int)(g > 0) - (int)(g < 0);
        sgn = isR1 ? s_new : sgn;
        const bool zero = isR1 && sgn == 0;
        const bool mispred = isR1 && sgn != 0 && sgn != pred;
        const int nvalid = max(0, min(8, 29 - jbase));
        const unsigned mc = isR1 ? (m8 >> 2) : (m8 & ((1u << nvalid) - 1u));
        const bool hit = (pt >= 0) && !isF0 && !zero && !mispred && mc != 0u;
        const int k = __ffs(mc) - 1;
        const int jacc = isR1 ? k : jbase + k;
        const int sidx = isR1 ? k + 2 : k;                       // accepted sample index within the round
        const int src = hit ? gbase + (sidx & 3) : lane;
        const bool fromB = (sidx & 4) != 0;
        const double tsel = fromB ? tB : tA, fsel = fromB ? fB : fA;
        const double xacc = __shfl_sync(FULL, tsel, src), facc = __shfl_sync(FULL, fsel, src);
        const int jb_next = isR1 ? (mispred ? 0 : 6) : jbase + 8;
        const bool failed = (pt >= 0) && !isF0 && (zero || (!hit && !mispred && jb_next > 28));
        const bool walking = (jacc == 0) && (xacc == x + (-0.01 * (double)sgn));
        pred = hit ? (walking ? sgn : -sgn) : pred;
        iter += hit ? jacc + 1 : (failed ? 29 : 0);
        x = hit ? xacc : x;
        fx = hit ? facc : (isF0 ? f0 : fx);
        const bool step_end = hit || failed;
        const bool running = (iter < 1000) && !failed && (fabs(x - prev_x) > 1e-16);
        prev_x = step_end ? x : prev_x;
        mode = (step_end || isF0) ? E_R1 : E_RN;
        jbase = jb_next;
        if (step_end && !running) {
            if (q == 0) { wk[4 * pt] = fx; wk[4 * pt + 1] = x; }
            pt = -1;
            need = true;
        }
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// TMA bulk copy of the trajectory blob into shared memory (cp.async.bulk + mbarrier)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void tma_load_blob(double *smem_blob, const double *gmem_blob, int n_doubles,
                                              uint64_t *bar) {
    const uint32_t bar_a = smem_u32(bar);
    const uint32_t bytes = (uint32_t)n_doubles * 8u;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_a), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                smem_u32(smem_blob)),
            "l"(gmem_blob), "r"(bytes), "r"(bar_a)
            : "memory");
    }
    // all threads wait on phase 0
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(bar_a), "r"(0)
            : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// k_pose_table: (x, y, cos yaw, sin yaw) at the layer-1 lattice times, written into the blob in place.
// The lattice and its poses are shared by every query point (choiceTInit layer 1 always scans 0..D in 0.15 s
// steps), so they are computed once per evaluation instead of once per point.
// ------------------------------------------------------------------------------------------------
__global__ void k_pose_table(double *blob) {
    TrajView tv = make_view(blob);
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= tv.K1) return;
    double x, y, yaw, sy, cy;
    traj_pos(tv, tv.lat[k], x, y, yaw);
    dev::sincos_portable(yaw, sy, cy);
    const BlobLayout L = blob_layout(tv.N, tv.K1);
    double *ps = blob + L.off_pose + k;
    ps[0] = x; ps[L.K1pad] = y; ps[2 * L.K1pad] = cy; ps[3 * L.K1pad] = sy;
}

// ------------------------------------------------------------------------------------------------
// K1: outer solve for every point (+ penalty, chain rule and CTA reduction for outside points)
// dynamic smem: [ blob | 8 warps x (19N + 1) accumulators ]
// ------------------------------------------------------------------------------------------------
#ifndef SVSDF_ENGINE_ILP
#define SVSDF_ENGINE_ILP 2   // samples per lane and round in the batched descent (1: descent_engine, 2: descent_engine2)
#endif
#ifndef SVSDF_MESH_MIN_CTAS
#define SVSDF_MESH_MIN_CTAS 4  // measured on config 4m: 2 -> 245 ms, 3 -> 206 ms, 4 -> 198 ms (the traversal is latency bound; spills stay in L1)
#endif
#ifndef SVSDF_OUTER_MIN_CTAS
#define SVSDF_OUTER_MIN_CTAS 3
#endif
#ifndef SVSDF_GSIP_MIN_CTAS
#define SVSDF_GSIP_MIN_CTAS 3
#endif
// BATCHED selects the schedule at compile time (two kernels: each carries only its own evaluation sites)
// SCALED: the body scale S(t) of svsdf_set_scale (Z) on every evaluation after choiceTInit (only the batched schedule is
// instantiated scaled)
template <int SHAPE, bool XFORM, bool BATCHED, bool SCALED>
__global__ void __launch_bounds__(kWarpsPerBlock * 32, (SHAPE == SH_MESH) ? SVSDF_MESH_MIN_CTAS : SVSDF_OUTER_MIN_CTAS)
    k_outer(const __grid_constant__ KernelArgs A, const __grid_constant__ ShapeParams S, const __grid_constant__ ScaleParams Z) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ int s_nb[kWarpsPerBlock];
    __shared__ int s_cursor;
    double *sblob = smem;
    tma_load_blob(sblob, A.blob, A.blob_doubles, &bar);
    const TrajView tv = make_view(sblob);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nacc = 19 * tv.N + 1;
    double *acc = smem + A.blob_doubles + warp * nacc;  // [N][18] gdC, then [N] gdT-by-piece, then cost
    if (A.want_reduce)
        for (int e = lane; e < nacc; e += 32) acc[e] = 0.0;
    __syncwarp();

    const int64_t wstride = (int64_t)gridDim.x * kWarpsPerBlock;
    const int64_t first = (int64_t)blockIdx.x * kWarpsPerBlock + warp;
    unsigned long long my_evals = 0;
    double *res = smem + A.blob_doubles + kWarpsPerBlock * nacc + warp * 128;  // per-warp work area of the descent engine
    // The warp walks its points in batches of up to 32 (lane i <-> i-th point of the batch).
    //  * Batched schedule (large P): the points are cut into nB = W * ceil(P / 32 W) CONTIGUOUS batches of equal size
    //    (+-1; neighbouring map cells: the lanes of a warp then prune the same layer-1 samples and run descents of similar
    //    length), warp w owns batches w, w + W, ... (strided: a warp's batches come from different regions of the map, so
    //    hard regions are spread over the warps; static, hence deterministic).  choiceTInit and the FD gradient /
    //    penalty / chain rule run one point per lane, gradientDescent one point per quarter warp (descent_engine).
    //  * Sparse schedule (few points per warp, i.e. small problems): the warp owns points w, w + W, ...; everything one
    //    point per warp, as solve_outer / grad_prel do (lowest latency).
    constexpr bool chunked = BATCHED;
    const int64_t lstride = chunked ? 1 : wstride;  // distance between the points of neighbouring lanes
    const int64_t nB = wstride * ((A.P + 32 * wstride - 1) / (32 * wstride));   // batches (batched schedule)
    for (int64_t bi = first; chunked ? (bi < nB) : (bi < A.P); bi += chunked ? wstride : 32 * wstride) {
        // batched: batch bi covers [bi P / nB, (bi + 1) P / nB); sparse: points bi, bi + W, ...
        const int64_t bfirst = chunked ? (bi * A.P) / nB : bi;
        const int64_t bend = chunked ? ((bi + 1) * A.P) / nB : A.P;
        const int64_t my_pt = bfirst + (int64_t)lane * lstride;
        const int nb = (int)min((int64_t)32, (bend - bfirst + lstride - 1) / lstride);  // batch size (warp-uniform)
        const bool my_valid = lane < nb;
        const int64_t ld_pt = my_valid ? my_pt : bfirst;
        const double mpx = __ldg(A.points_xy + 2 * ld_pt), mpy = __ldg(A.points_xy + 2 * ld_pt + 1);
        const bool batched = chunked;   // CTA-uniform: the batched schedule synchronises the CTA around its shared queue
        double m_seed = 0.0, m_min = 1e9, m_sdf = 0.0, m_ts = 0.0, m_gx = 0.0, m_gy = 0.0;
        if (BATCHED && batched) {
            int ev = 0;
            if (my_valid) thread_choice_t_init<SHAPE, XFORM>(tv, S, mpx, mpy, m_seed, m_min, ev);
            __syncwarp();
            unsigned ev2 = 0;
#if SVSDF_ENGINE_ILP == 2
            if (my_valid) { res[4 * lane] = mpx; res[4 * lane + 1] = mpy; res[4 * lane + 2] = m_seed; res[4 * lane + 3] = m_min; }
            if (lane == 0) s_nb[warp] = nb;
            if (threadIdx.x == 0) s_cursor = 0;
            __syncthreads();   // every warp has the same number of batches (nB is a multiple of the warp count)
            descent_engine2<SHAPE, XFORM, SCALED>(tv, S, Z, res - 128 * warp, s_nb, &s_cursor, kWarpsPerBlock * 32, ev2);
            __syncthreads();
            if (my_valid) { m_sdf = res[4 * lane]; m_ts = res[4 * lane + 1]; }
#else
            descent_engine<SHAPE, XFORM, SCALED>(tv, S, Z, nb, mpx, mpy, m_seed, m_min, res, ev2);
            if (my_valid) { m_sdf = res[2 * lane]; m_ts = res[2 * lane + 1]; }
#endif
            my_evals += (unsigned long long)__reduce_add_sync(FULL, (unsigned)ev + ev2);
            __syncwarp();
        } else {
#pragma unroll 1
            for (int i = 0; i < nb; ++i) {
                const double px = __shfl_sync(FULL, mpx, i), py = __shfl_sync(FULL, mpy, i);
                const OuterResult R = solve_outer<SHAPE, XFORM, SCALED>(tv, S, Z, px, py);
                my_evals += (unsigned long long)R.evals;
                if (lane == i) { m_sdf = R.sdf; m_ts = R.tstar; }
                double gx, gy;
                grad_prel<SHAPE, XFORM, SCALED>(tv, S, Z, px, py, R.tstar, gx, gy);
                if (lane == i) { m_gx = gx; m_gy = gy; }
            }
        }
        my_evals += 4ull * (unsigned long long)nb;
        if (BATCHED && batched && my_valid) thread_grad_prel<SHAPE, XFORM, SCALED>(tv, S, Z, mpx, mpy, m_ts, m_gx, m_gy);
        // ---- per-lane epilogue: outputs, interior flag, penalty + chain rule (one point per lane) ----
        const bool inside = my_valid && A.want_gsip && !(m_sdf > 0);  // getTrueSDFofSweptVolume: `if (argmin_dis > 0) return`
        if (my_valid) {
            if (A.out_sdf) A.out_sdf[my_pt] = m_sdf;
            if (A.out_tstar) A.out_tstar[my_pt] = m_ts;
            if (A.out_grad) { A.out_grad[3 * my_pt] = m_gx; A.out_grad[3 * my_pt + 1] = m_gy; A.out_grad[3 * my_pt + 2] = 0.0; }
            if (A.out_rounds) A.out_rounds[my_pt] = 0;
            if (A.inside_flag) A.inside_flag[my_pt] = inside ? 1 : 0;
            if (inside && A.inside_tstar) A.inside_tstar[my_pt] = m_ts;
        }
        if (A.want_reduce) {
            Contribution C;
            C.active = false;
            if (my_valid && !inside) C = point_contribution<SCALED>(tv, A.cp, Z, mpx, mpy, m_sdf, m_ts, m_gx, m_gy);
            // accumulate the active lanes' contributions in batch order (deterministic)
            unsigned m = __ballot_sync(FULL, C.active);
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const int piece = __shfl_sync(FULL, C.piece, src);
                const double s1 = __shfl_sync(FULL, C.s1, src);
                const double g0 = __shfl_sync(FULL, C.G[0], src), g1 = __shfl_sync(FULL, C.G[1], src),
                             g2 = __shfl_sync(FULL, C.G[2], src);
                const double gdT = __shfl_sync(FULL, C.gdT, src), pena = __shfl_sync(FULL, C.pena, src);
                if (lane < 18) {
                    const int d = lane / 6, q = lane - 6 * d;
                    const double s2 = s1 * s1, s3 = s2 * s1, s4 = s2 * s2, s5 = s4 * s1;
                    const double beta = (q == 0) ? 1.0 : (q == 1) ? s1 : (q == 2) ? s2 : (q == 3) ? s3 : (q == 4) ? s4 : s5;
                    const double gd = (d == 0) ? g0 : (d == 1) ? g1 : g2;
                    acc[piece * 18 + lane] += beta * gd;
                } else if (lane == 18) {
                    acc[18 * tv.N + piece] += gdT;
                } else if (lane == 19) {
                    acc[19 * tv.N] += pena;
                }
                __syncwarp();
            }
        }
    }
    if (A.eval_counter && lane == 0) atomicAdd(A.eval_counter, my_evals);
    if (A.want_reduce) {
        __syncthreads();
        const double *acc0 = smem + A.blob_doubles;
        for (int e = threadIdx.x; e < nacc; e += blockDim.x) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kWarpsPerBlock; ++w) s += acc0[w * nacc + e];
            A.partials[(int64_t)blockIdx.x * nacc + e] = s;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// k_compact: ordered compaction of the inside flags (single CTA, 1024 threads) -> inside_list, n_inside.
// Flags are 0/1 bytes; every thread owns a contiguous run of 16-byte words (coalesced uint4 loads, popcount).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_compact(const unsigned char *flag, int64_t P, int *list, int *n_out) {
    __shared__ int wsum[32];
    __shared__ int total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t nwords = (P + 15) / 16;              // flag buffer is allocated with >= 16 bytes of slack
    const int64_t per = (nwords + 1023) / 1024;        // words per thread
    const int64_t w0 = (int64_t)tid * per, w1 = (w0 + per < nwords) ? w0 + per : nwords;
    const uint4 *f4 = reinterpret_cast<const uint4 *>(flag);
    int cnt = 0;
    for (int64_t w = w0; w < w1; ++w) {
        uint4 v = f4[w];
        if (16 * w + 16 > P) {  // mask the tail beyond P
            unsigned char *b = reinterpret_cast<unsigned char *>(&v);
            for (int q = 0; q < 16; ++q)
                if (16 * w + q >= P) b[q] = 0;
        }
        cnt += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
    }
    int inc = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int v = __shfl_up_sync(FULL, inc, off);
        if (lane >= off) inc += v;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int v = wsum[lane];
        int vi = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            int u = __shfl_up_sync(FULL, vi, off);
            if (lane >= off) vi += u;
        }
        wsum[lane] = vi - v;  // exclusive
        if (lane == 31) total = vi;
    }
    __syncthreads();
    int pos = wsum[warp] + inc - cnt;
    if (cnt > 0) {
        for (int64_t w = w0; w < w1; ++w) {
            const uint4 v = f4[w];
            if ((v.x | v.y | v.z | v.w) == 0u) continue;
            const unsigned char *b = reinterpret_cast<const unsigned char *>(&v);
            for (int q = 0; q < 16; ++q) {
                const int64_t i = 16 * w + q;
                if (i < P && b[q]) list[pos++] = (int)i;
            }
        }
    }
    if (tid == 0) *n_out = total;
}

// ------------------------------------------------------------------------------------------------
// K2: interior branch of getTrueSDFofSweptVolume<true> (sw_manager.hpp:926-1017, SampleSet2D :41-124).
// One CTA per inside point; the ring samples of a round are distributed over the CTA's warps, each warp
// running a full outer solve on its sample.
// dynamic smem: [ blob ]
// ------------------------------------------------------------------------------------------------
// SCALED: the ring samples' outer solves and the chain rule use S(t) (only the 8-warp width is instantiated scaled)
template <int SHAPE, bool XFORM, int WARPS, bool SCALED>
__global__ void __launch_bounds__(WARPS * 32, (WARPS == kWarpsPerBlock && SHAPE != SH_MESH) ? SVSDF_GSIP_MIN_CTAS : 1)
    k_gsip(const __grid_constant__ KernelArgs A, const __grid_constant__ ShapeParams S, const __grid_constant__ ScaleParams Z) {
    extern __shared__ __align__(16) double smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ double s_theta[24], s_val[24], s_ts[24];
    double *sblob = smem;
    tma_load_blob(sblob, A.blob, A.blob_doubles, &bar);
    const TrajView tv = make_view(sblob);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double PI = 3.14159265358979323846;  // Shape.hpp:31
    const int n_in = *A.n_inside;
    unsigned long long my_evals = 0;

    for (int slot = blockIdx.x; slot < n_in; slot += gridDim.x) {
        const int pt = A.inside_list[slot];
        const double px = __ldg(A.points_xy + 2 * (int64_t)pt), py = __ldg(A.points_xy + 2 * (int64_t)pt + 1);
        const double ts0 = A.inside_tstar[pt];
        // velocity at t* with the reference's fallback scan (:928-954); all threads redundantly
        double vx, vy, vw;
        traj_vel(tv, ts0, vx, vy, vw);
        if (sqrt(vx * vx + vy * vy + vw * vw) < 0.01) {
            if (ts0 < 0.1) {
                for (double t_scan = ts0; t_scan <= tv.D; t_scan += 0.1) {
                    traj_vel(tv, t_scan, vx, vy, vw);
                    if (sqrt(vx * vx + vy * vy + vw * vw) >= 0.01) break;
                }
            } else if (ts0 > tv.D - 0.1) {
                for (double t_scan = ts0; t_scan >= 0; t_scan -= 0.1) {
                    traj_vel(tv, t_scan, vx, vy, vw);
                    if (sqrt(vx * vx + vy * vy + vw * vw) >= 0.01) break;
                }
            }
        }
        // SampleSet2D::initSet (:74-103)
        double r = 10.0;
        double theta0 = dev::atan2_portable(vx, -vy);
        if (theta0 < 0) theta0 += 2 * PI;
        double theta_res = PI + 0.1;
        double r_star = 0.0, real_t_star = 0.0, star_theta = 0.0;
        int iter = 1, rounds = 0;
        while (true) {
            // getElements (:59-71): one ring (rk = 1.0), theta accumulated from theta0 while < theta0 + 2 PI
            int ns = 0;
            for (double th = theta0; th < theta0 + 2 * PI; th += theta_res) {
                if (threadIdx.x == 0 && ns < 24) s_theta[ns] = th;
                ns++;
            }
            if (ns > 24) ns = 24;  // cannot happen: theta_res >= 0.3 -> at most 21 samples
            __syncthreads();
            for (int k = warp; k < ns; k += WARPS) {
                double th = s_theta[k];
                double sn, cs;
                dev::sincos_portable(th, sn, cs);
                double yx = px + 1.0 * r * cs, yy = py + 1.0 * r * sn;  // CircleCoord2D::getPosition (:36-39)
                OuterResult R = solve_outer<SHAPE, XFORM, SCALED>(tv, S, Z, yx, yy);
                my_evals += (unsigned long long)R.evals;
                if (lane == 0) { s_val[k] = R.sdf; s_ts[k] = R.tstar; }
            }
            __syncthreads();
            double max_g = -100000;
            for (int k = 0; k < ns; ++k) {
                double cur = s_val[k];
                if (cur > max_g) {
                    max_g = cur;
                    real_t_star = s_ts[k];
                    star_theta = s_theta[k];
                }
            }
            __syncthreads();  // everyone has read s_* before the next round overwrites them
            r_star = r - max_g;
            r = r_star;
            rounds++;
            if (iter > 8) break;
            if (fabs(max_g) < 0.1) break;
            theta_res /= (2 + 1);  // expandSet(2, theta*) (:105-123)
            theta_res = smaxd(0.3, theta_res);
            theta0 = star_theta;
            iter++;
        }
        double sn, cs;
        dev::sincos_portable(star_theta, sn, cs);
        double corx = px + 1.0 * r_star * cs, cory = py + 1.0 * r_star * sn;
        double gx = corx - px, gy = cory - py;
        double z = gx * gx + gy * gy;
        if (z > 0) {
            double n = sqrt(z);
            gx /= n; gy /= n;
        }
        const double sdf = -r_star;
        if (threadIdx.x == 0) {
            if (A.out_sdf) A.out_sdf[pt] = sdf;
            if (A.out_tstar) A.out_tstar[pt] = real_t_star;
            if (A.out_grad) { A.out_grad[3 * pt] = gx; A.out_grad[3 * pt + 1] = gy; A.out_grad[3 * pt + 2] = 0.0; }
            if (A.out_rounds) A.out_rounds[pt] = rounds;
        }
        if (A.want_reduce && warp == 0) {
            Contribution C = point_contribution<SCALED>(tv, A.cp, Z, px, py, sdf, real_t_star, gx, gy);
            double *o = A.gsip_contrib + 20 * (int64_t)slot;
            if (lane < 18) {
                int d = lane / 6, q = lane - 6 * d;
                double s1 = C.s1, s2 = s1 * s1, s3 = s2 * s1, s4 = s2 * s2, s5 = s4 * s1;
                double beta = (q == 0) ? 1.0 : (q == 1) ? s1 : (q == 2) ? s2 : (q == 3) ? s3 : (q == 4) ? s4 : s5;
                o[1 + lane] = C.active ? beta * C.G[d] : 0.0;
            } else if (lane == 18) {
                o[19] = C.active ? C.gdT : 0.0;
            } else if (lane == 19) {
                o[0] = C.active ? C.pena : 0.0;
                A.gsip_piece[slot] = C.piece;
            }
        }
    }
    if (A.eval_counter && lane == 0) atomicAdd(A.eval_counter, my_evals);
}

// ------------------------------------------------------------------------------------------------
// k_finalize: fixed-order sum of the K1 CTA partials and the K2 per-point contributions.  One warp per accumulator
// entry: lane l adds partials l, l+32, ... in order, the 32 lane sums are combined by a fixed shuffle tree, so the
// result is bit-reproducible.  The last CTA to finish (ticket counter) writes the output record:
// out: [0] cost, [1 .. 18N] gradC in Eigen column-major order (d*6N + 6i + q), [1+18N .. 1+19N) gradT with the
// reference's rule gradT(j) += gdT for all j < piece (back_end_optimizer.hpp:859-862), [1+19N] n_inside.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum_fixed(double v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(FULL, v, off);
    return __shfl_sync(FULL, v, 0);
}

__global__ void __launch_bounds__(256) k_finalize(const double *partials, int n_blocks, int N, const int *n_inside,
                                                  const double *gsip_contrib, const int *gsip_piece, double *tot,
                                                  unsigned int *ticket, double *out) {
    const int nacc = 19 * N + 1;
    const int n_in = n_inside ? *n_inside : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int e = blockIdx.x * 8 + warp;
    if (e < nacc) {
        double s = 0.0;
        for (int b = lane; b < n_blocks; b += 32) s += partials[(int64_t)b * nacc + e];
        s = warp_sum_fixed(s);
        // K2 contributions, ascending point order (inside_list is sorted)
        double s2 = 0.0;
        if (e < 18 * N) {
            const int piece = e / 18, within = e - 18 * piece;
            for (int k = lane; k < n_in; k += 32)
                if (gsip_piece[k] == piece) s2 += gsip_contrib[20 * (int64_t)k + 1 + within];
        } else if (e < 19 * N) {
            const int piece = e - 18 * N;
            for (int k = lane; k < n_in; k += 32)
                if (gsip_piece[k] == piece) s2 += gsip_contrib[20 * (int64_t)k + 19];
        } else {
            for (int k = lane; k < n_in; k += 32) s2 += gsip_contrib[20 * (int64_t)k];
        }
        s2 = warp_sum_fixed(s2);
        if (lane == 0) tot[e] = s + s2;
    }
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    for (int q = threadIdx.x; q < nacc; q += blockDim.x) {
        if (q < 18 * N) {
            const int piece = q / 18, within = q - 18 * piece;
            const int d = within / 6, pw = within - 6 * d;
            out[1 + d * 6 * N + 6 * piece + pw] = __ldcg(tot + q);
        } else if (q < 19 * N) {
            const int j = q - 18 * N;
            double sfx = 0.0;
            for (int i = j + 1; i < N; ++i) sfx += __ldcg(tot + 18 * N + i);
            out[1 + 18 * N + j] = sfx;
        } else {
            out[0] = __ldcg(tot + q);
        }
    }
    if (threadIdx.x == 0) {
        out[1 + 19 * N] = (double)n_in;
        *ticket = 0u;  // re-arm for the next evaluation
    }
}

// ------------------------------------------------------------------------------------------------
// Shape-functor batch kernels (BasicShape::getonlySDF / getonlyGrad1 over arrays of body-frame points)
// ------------------------------------------------------------------------------------------------
template <int SHAPE, bool XFORM>
__global__ void k_shape_sdf(const __grid_constant__ ShapeParams S, const double *rel_xy, int64_t n, double *out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = dev::shape_sdf<SHAPE, XFORM>(S, rel_xy[2 * i], rel_xy[2 * i + 1]);
}
template <int SHAPE, bool XFORM>
__global__ void k_shape_grad(const __grid_constant__ ShapeParams S, const double *rel_xy, int64_t n, double *out3) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double rx = rel_xy[2 * i], ry = rel_xy[2 * i + 1];
    double gx, gy;
    if (SHAPE == SH_POLYGON) {
        dev::PolyHit H = dev::polygon_scan(S, rx, ry);
        double vx = rx - H.cx, vy = ry - H.cy;
        double z = vx * vx + vy * vy;
        if (z > 0.0) { double nn = sqrt(z); vx /= nn; vy /= nn; }
        if (H.rs % 2 != 0) { vx = -vx; vy = -vy; }
        gx = vx; gy = vy;
    } else if (SHAPE == SH_CIRCLE) {
        dev::circle_grad1<XFORM>(S, rx, ry, gx, gy);
    } else {
        const double dx = 0.000001;
        double t0 = rx, t1 = ry;
        t0 -= dx;
        double sdfold = dev::shape_sdf<SHAPE, XFORM>(S, t0, t1);
        t0 += 2 * dx;
        double gradx = dev::shape_sdf<SHAPE, XFORM>(S, t0, t1) - sdfold;
        t0 = rx;
        t1 -= dx;
        sdfold = dev::shape_sdf<SHAPE, XFORM>(S, t0, t1);
        t1 += 2 * dx;
        double grady = dev::shape_sdf<SHAPE, XFORM>(S, t0, t1) - sdfold;
        gx = gradx / (2 * dx);
        gy = grady / (2 * dx);
    }
    out3[3 * i] = gx; out3[3 * i + 1] = gy; out3[3 * i + 2] = 0.0;
}

__global__ void k_sincos(const double *x, int64_t n, double *s, double *c) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double sv, cv;
    dev::sincos_portable(x[i], sv, cv);
    s[i] = sv;
    c[i] = cv;
}

// FP64 FMA peak micro-benchmark (roofline denominator; MEASURED_PEAKS.json has no FP64 figure)
__global__ void __launch_bounds__(256) k_fp64_peak(double *out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-6;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[(int64_t)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------------------------
// Host-side launchers (shape dispatch)
// ------------------------------------------------------------------------------------------------
struct LaunchCfg {
    int grid_outer, grid_gsip;
    size_t smem_outer, smem_gsip;
    cudaStream_t stream;
    cudaEvent_t after_outer;  // optional timing mark recorded right after k_outer
    bool gsip_wide;           // use the 22-warp k_gsip variant
    const ScaleParams *scale; // body scale S(t) (null: rigid body)
};

// Scaled body: one k_outer schedule (batched: correct for every P) and one k_gsip width, so that the scale adds two
// instantiations per shape instead of four.
template <int SHAPE, bool XFORM>
static cudaError_t launch_shape_scaled(const KernelArgs &A, const ShapeParams &S, const LaunchCfg &cfg) {
    cudaError_t e;
    static bool attr_set_dev[64] = {};
    int dev_ord = 0;
    cudaGetDevice(&dev_ord);
    bool &attr_set = attr_set_dev[dev_ord & 63];
    if (!attr_set) {
        e = cudaFuncSetAttribute(k_outer<SHAPE, XFORM, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_gsip<SHAPE, XFORM, kWarpsPerBlock, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    KernelArgs B = A;
    B.batched = 1;
    k_outer<SHAPE, XFORM, true, true><<<cfg.grid_outer, kWarpsPerBlock * 32, cfg.smem_outer, cfg.stream>>>(B, S, *cfg.scale);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (cfg.after_outer) cudaEventRecord(cfg.after_outer, cfg.stream);
    if (A.want_gsip) {
        k_compact<<<1, 1024, 0, cfg.stream>>>(A.inside_flag, A.P, A.inside_list, A.n_inside);
        k_gsip<SHAPE, XFORM, kWarpsPerBlock, true><<<cfg.grid_gsip, kWarpsPerBlock * 32, cfg.smem_gsip, cfg.stream>>>(B, S, *cfg.scale);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

template <int SHAPE, bool XFORM>
static cudaError_t launch_shape(const KernelArgs &A, const ShapeParams &S, const LaunchCfg &cfg, int N) {
    if (cfg.scale) return launch_shape_scaled<SHAPE, XFORM>(A, S, cfg);
    cudaError_t e;
    const ScaleParams Z{};
    // the attribute is per device (a process may hold contexts on several GPUs): one flag per device ordinal
    static bool attr_set_dev[64] = {};
    int dev_ord = 0;
    cudaGetDevice(&dev_ord);
    bool &attr_set = attr_set_dev[dev_ord & 63];
    if (!attr_set) {
        e = cudaFuncSetAttribute(k_outer<SHAPE, XFORM, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_outer<SHAPE, XFORM, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_gsip<SHAPE, XFORM, kWarpsPerBlock, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_gsip<SHAPE, XFORM, kGsipWarps, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (e != cudaSuccess) return e;
        attr_set = true;
    }
    if (A.batched) k_outer<SHAPE, XFORM, true, false><<<cfg.grid_outer, kWarpsPerBlock * 32, cfg.smem_outer, cfg.stream>>>(A, S, Z);
    else k_outer<SHAPE, XFORM, false, false><<<cfg.grid_outer, kWarpsPerBlock * 32, cfg.smem_outer, cfg.stream>>>(A, S, Z);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (cfg.after_outer) cudaEventRecord(cfg.after_outer, cfg.stream);
    if (A.want_gsip) {
        k_compact<<<1, 1024, 0, cfg.stream>>>(A.inside_flag, A.P, A.inside_list, A.n_inside);
        // few inside points: one warp per ring sample (latency); many: 8-warp CTAs, two per SM (throughput)
        if (cfg.gsip_wide) k_gsip<SHAPE, XFORM, kGsipWarps, false><<<cfg.grid_gsip, kGsipWarps * 32, cfg.smem_gsip, cfg.stream>>>(A, S, Z);
        else k_gsip<SHAPE, XFORM, kWarpsPerBlock, false><<<cfg.grid_gsip, kWarpsPerBlock * 32, cfg.smem_gsip, cfg.stream>>>(A, S, Z);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    (void)N;
    return cudaSuccess;
}

template <bool XFORM>
static cudaError_t dispatch(const KernelArgs &A, const ShapeParams &S, const LaunchCfg &cfg, int N) {
    switch (S.id) {
#define SVSDF_CASE(ID) \
    case ID: return launch_shape<ID, XFORM>(A, S, cfg, N);
        SVSDF_CASE(SH_STAR)
        SVSDF_CASE(SH_HORSESHOE)
        SVSDF_CASE(SH_PIE)
        SVSDF_CASE(SH_PIE2)
        SVSDF_CASE(SH_ARC)
        SVSDF_CASE(SH_TUNNEL)
        SVSDF_CASE(SH_CUTDISK)
        SVSDF_CASE(SH_TRAPEZOID)
        SVSDF_CASE(SH_RHOMBUS)
        SVSDF_CASE(SH_HEART)
        SVSDF_CASE(SH_ROUNDEDX)
        SVSDF_CASE(SH_BIGX)
        SVSDF_CASE(SH_ROUNDEDCROSS)
        SVSDF_CASE(SH_VESICA)
        SVSDF_CASE(SH_MOON)
        SVSDF_CASE(SH_UNEVENCAPSULE)
        SVSDF_CASE(SH_CIRCLE)
#undef SVSDF_CASE
        case SH_POLYGON: return launch_shape<SH_POLYGON, false>(A, S, cfg, N);
        case SH_MESH: return launch_shape<SH_MESH, false>(A, S, cfg, N);
        default: return cudaErrorInvalidValue;
    }
}

template <int SHAPE, bool XFORM>
static cudaError_t occ_shape(size_t smem_outer, size_t smem_gsip, int *occ_outer, int *occ_gsip) {
    cudaError_t e = cudaFuncSetAttribute(k_outer<SHAPE, XFORM, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_outer<SHAPE, XFORM, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_gsip<SHAPE, XFORM, kWarpsPerBlock, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    // the two schedules are compiled to the same register cap (launch bounds); the batched kernel sizes the full wave.  The
    // scaled instantiations have the same launch bounds and shared memory, so the rigid figures size their grids too.
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ_outer, k_outer<SHAPE, XFORM, true, false>, kWarpsPerBlock * 32, smem_outer);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ_gsip, k_gsip<SHAPE, XFORM, kWarpsPerBlock, false>, kWarpsPerBlock * 32, smem_gsip);
}

// Resident CTAs per SM of k_outer / k_gsip for this shape and trajectory size: the host sizes the grids as
// SMs x occupancy so that the warp-stride loops run as exactly one full wave (no partial second wave).
cudaError_t query_occupancy(const ShapeParams &S, int N, int blob_doubles, int *occ_outer, int *occ_gsip) {
    const size_t so = outer_smem_doubles(blob_doubles, N) * sizeof(double);
    const size_t sg = (size_t)blob_doubles * sizeof(double);
    const bool xf = S.has_xform != 0;
    switch (S.id) {
#define SVSDF_CASE(ID) \
    case ID: return xf ? occ_shape<ID, true>(so, sg, occ_outer, occ_gsip) : occ_shape<ID, false>(so, sg, occ_outer, occ_gsip);
        SVSDF_CASE(SH_STAR)
        SVSDF_CASE(SH_HORSESHOE)
        SVSDF_CASE(SH_PIE)
        SVSDF_CASE(SH_PIE2)
        SVSDF_CASE(SH_ARC)
        SVSDF_CASE(SH_TUNNEL)
        SVSDF_CASE(SH_CUTDISK)
        SVSDF_CASE(SH_TRAPEZOID)
        SVSDF_CASE(SH_RHOMBUS)
        SVSDF_CASE(SH_HEART)
        SVSDF_CASE(SH_ROUNDEDX)
        SVSDF_CASE(SH_BIGX)
        SVSDF_CASE(SH_ROUNDEDCROSS)
        SVSDF_CASE(SH_VESICA)
        SVSDF_CASE(SH_MOON)
        SVSDF_CASE(SH_UNEVENCAPSULE)
        SVSDF_CASE(SH_CIRCLE)
#undef SVSDF_CASE
        case SH_POLYGON: return occ_shape<SH_POLYGON, false>(so, sg, occ_outer, occ_gsip);
        case SH_MESH: return occ_shape<SH_MESH, false>(so, sg, occ_outer, occ_gsip);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_pose_table(double *blob, int K1, cudaStream_t stream) {
    k_pose_table<<<(K1 + 127) / 128, 128, 0, stream>>>(blob);
    return cudaGetLastError();
}

cudaError_t launch_cost_kernels(const KernelArgs &A, const ShapeParams &S, const ScaleParams *scale, int N, int grid_outer,
                                int grid_gsip, cudaStream_t stream, cudaEvent_t after_outer, int gsip_wide) {
    LaunchCfg cfg;
    cfg.scale = scale;
    cfg.after_outer = after_outer;
    cfg.gsip_wide = gsip_wide != 0;
    cfg.grid_outer = grid_outer;
    cfg.grid_gsip = grid_gsip;
    cfg.smem_outer = outer_smem_doubles(A.blob_doubles, N) * sizeof(double);
    cfg.smem_gsip = (size_t)A.blob_doubles * sizeof(double);
    cfg.stream = stream;
    return S.has_xform ? dispatch<true>(A, S, cfg, N) : dispatch<false>(A, S, cfg, N);
}

cudaError_t launch_finalize(const double *partials, int n_blocks, int N, const int *n_inside,
                            const double *gsip_contrib, const int *gsip_piece, double *tot, unsigned int *ticket,
                            double *out, cudaStream_t stream) {
    const int nacc = 19 * N + 1;
    k_finalize<<<(nacc + 7) / 8, 256, 0, stream>>>(partials, n_blocks, N, n_inside, gsip_contrib, gsip_piece, tot,
                                                   ticket, out);
    return cudaGetLastError();
}

template <int SHAPE, bool XFORM>
static cudaError_t launch_shape_fn(const ShapeParams &S, const double *rel_xy, int64_t n, double *out, int grad,
                                   cudaStream_t stream) {
    int grid = (int)((n + 255) / 256);
    if (grad) k_shape_grad<SHAPE, XFORM><<<grid, 256, 0, stream>>>(S, rel_xy, n, out);
    else k_shape_sdf<SHAPE, XFORM><<<grid, 256, 0, stream>>>(S, rel_xy, n, out);
    return cudaGetLastError();
}

cudaError_t launch_shape_eval(const ShapeParams &S, const double *rel_xy, int64_t n, double *out, int grad,
                              cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    switch (S.id) {
#define SVSDF_CASE(ID)                                                                              \
    case ID:                                                                                        \
        return S.has_xform ? launch_shape_fn<ID, true>(S, rel_xy, n, out, grad, stream)             \
                           : launch_shape_fn<ID, false>(S, rel_xy, n, out, grad, stream);
        SVSDF_CASE(SH_STAR)
        SVSDF_CASE(SH_HORSESHOE)
        SVSDF_CASE(SH_PIE)
        SVSDF_CASE(SH_PIE2)
        SVSDF_CASE(SH_ARC)
        SVSDF_CASE(SH_TUNNEL)
        SVSDF_CASE(SH_CUTDISK)
        SVSDF_CASE(SH_TRAPEZOID)
        SVSDF_CASE(SH_RHOMBUS)
        SVSDF_CASE(SH_HEART)
        SVSDF_CASE(SH_ROUNDEDX)
        SVSDF_CASE(SH_BIGX)
        SVSDF_CASE(SH_ROUNDEDCROSS)
        SVSDF_CASE(SH_VESICA)
        SVSDF_CASE(SH_MOON)
        SVSDF_CASE(SH_UNEVENCAPSULE)
        SVSDF_CASE(SH_CIRCLE)
#undef SVSDF_CASE
        case SH_POLYGON: return launch_shape_fn<SH_POLYGON, false>(S, rel_xy, n, out, grad, stream);
        case SH_MESH: return launch_shape_fn<SH_MESH, false>(S, rel_xy, n, out, grad, stream);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_sincos(const double *x, int64_t n, double *s, double *c, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    k_sincos<<<(int)((n + 255) / 256), 256, 0, stream>>>(x, n, s, c);
    return cudaGetLastError();
}

cudaError_t launch_fp64_peak(double *out, int grid, int iters, cudaStream_t stream) {
    k_fp64_peak<<<grid, 256, 0, stream>>>(out, iters);
    return cudaGetLastError();
}

// occupancy query used by the host to size the grids (CTAs per SM for k_outer of this shape is not needed to be
// exact: we size for 2 resident CTAs per SM and let the hardware queue the rest)

}  // namespace SVSDF_NS
}  // namespace svsdf

// oracle/scale_oracle.cpp — TEST INFRASTRUCTURE ONLY: the CPU oracle with the reference's `useScale` switch on.
//
// A deformable robot (include/svsdf.h, svsdf_set_scale): body scale S(t) = diag(sx(t), sy(t), 1), per axis s = c, then
// s = s + sin(w_k t + phi_k) a_k (k < n), at absolute trajectory time.  This file restates what `#define useScale true`
// (sw_manager.hpp:17) changes on the path, with getScale (:495-507, the reference's edit point) given by the spec; everything
// else is svsdf_oracle.hpp / minco_oracle.hpp, used as they are:
//   * choiceTInit stays rigid (its loop calls the rigid posEva2Rel, :569-570): SweptVolume::choiceTInit;
//   * gradientDescent (:1249-1325) evaluates getSDFAtTimeStamp<true> for its values and its finite-difference slope;
//   * getGradPrelAtTimeStamp<true> (:779-795) differentiates the shape at the scaled rel;
//   * the interior branch (:916-1018) runs the same scaled outer solve on its ring samples;
//   * grad_cost_p_sw (back_end_optimizer.hpp:1031-1066) with St = getScale(t*) (:827).
// Built into oracle/_build/libsvsdf_scale_oracle{,_glibc}.so by oracle/scale.mk (oracle/scale_py.py loads it).
#include <omp.h>

#include <cstring>

#include "minco_oracle.hpp"

namespace oracle {

struct ScaleSpec {
    int n[2] = {0, 0};
    double c[2] = {1.0, 1.0}, a[2][4] = {}, w[2][4] = {}, phi[2][4] = {};
    int exact_yaw_grad = 0;
    double axis(int ax, double t) const {
        double v = c[ax];
        for (int k = 0; k < n[ax]; ++k) {
            double sn, cs;
            psc::sincos(w[ax][k] * t + phi[ax][k], sn, cs);
            v = v + sn * a[ax][k];
        }
        return v;
    }
    // diagonal of S^-1 as Eigen's 3x3 cofactor inverse forms it: cof(0,0) = sy, cof(1,1) = sx, det = sy * sx (the other
    // cofactor-expansion terms are products with exact zeros), entry = cofactor * (1 / det) — not 1 / sx
    void inv(double t, double &i00, double &i11) const {
        const double sx = axis(0, t), sy = axis(1, t);
        const double invdet = 1.0 / (sy * sx);
        i00 = sy * invdet;
        i11 = sx * invdet;
    }
};

struct ScaledSweptVolume : SweptVolume {
    ScaleSpec scale;

    // getStateOnTrajStamp(t, xt, Rt, St) :476-488 + posEva2Rel(p, x, R, S) :528-535: rel = (R^T S^-1) (p - xt), the matrix
    // product formed first: (R^T S^-1) = [[c i00, s i11, 0], [-s i00, c i11, 0], [0, 0, i22]] (zero terms dropped)
    void relAtS(const double p[3], double t, double rel[3]) const {
        double xt[3];
        traj.getPos(t, xt);
        double s, c;
        psc::sincos(xt[2], s, c);
        double i00, i11;
        scale.inv(t, i00, i11);
        const double d0 = p[0] - xt[0], d1 = p[1] - xt[1];
        rel[0] = (c * i00) * d0 + (s * i11) * d1;
        rel[1] = (-(s * i00)) * d0 + (c * i11) * d1;
        rel[2] = 0.0;  // i22 * d2 in the reference: the analytic functors ignore z; the mesh path zeroes xt(2) (:767), so d2 = 0
    }
    // getSDFAtTimeStamp<true> :741-757 (and getSDFAtTimeStamp_igl<true> :759-777 for the mesh functor)
    double sdfAtS(const double p[3], double t) const {
        double rel[3];
        relAtS(p, t, rel);
        return shape_sdf(shape, rel[0], rel[1], rel[2]);
    }
    // getSDF_DOTAtTimeStamp<true> :798-806 (the analytic branch below the early return is dead)
    double sdfDotAtS(const double p[3], double t) const {
        double t1 = std::max(0.0, t - 0.000001);
        double t2 = std::min(traj_duration, t + 0.000001);
        return (sdfAtS(p, t2) - sdfAtS(p, t1)) * 500000;
    }
    // gradientDescent :1249-1325, same loop as SweptVolume::gradientDescent with the scaled samples
    void gradientDescentS(double t_min, double t_max, const double x0, double &fx, double &x, const double p[3]) const {
        int max_iter = 1000;
        double alpha = 0.01, tau = alpha, g = 0.0, tol = 1e-16;
        x = x0;
        double change = 0;
        double prev_x = 10000000.0;
        int iter = 0;
        bool stop = false;
        double x_candidate, fx_candidate;
        g = 100.0;
        while (iter < max_iter && !stop && std::abs(x - prev_x) > tol) {
            if (iter == 0) fx = sdfAtS(p, x);
            g = sdfDotAtS(p, x);
            tau = alpha;
            prev_x = x;
            for (int div = 1; div < 30; div++) {
                iter = iter + 1;
                g = sdfDotAtS(p, x);
                change = -tau * ((int)(g > 0) - (g < 0));
                x_candidate = x + change;
                x_candidate = std::max(std::min(x_candidate, t_max), t_min);
                fx_candidate = sdfAtS(p, x_candidate);
                if ((fx_candidate - fx) < 0) {
                    x = x_candidate;
                    fx = fx_candidate;
                    break;
                }
                tau = 0.5 * tau;
                if (div == 29) stop = true;
            }
        }
    }
    // getSDFofSweptVolume<false,true> :844-866 with useScale = true
    double getSDFofSweptVolumeS(const double p[3], double &time_seed_f, double grad_prel[3]) const {
        double t_star = 0.0, sdf_star = 0.0;
        const double ts = choiceTInit(p, 0.15);  // rigid
        gradientDescentS(std::max(0.0, ts - 3.4), std::min(ts + 3.4, traj_duration), ts, sdf_star, t_star, p);
        double rel[3];
        relAtS(p, t_star, rel);
        shape_grad1(shape, rel[0], rel[1], rel[2], grad_prel);
        time_seed_f = t_star;
        return sdf_star;
    }
    // getTrueSDFofSweptVolume<true> :916-1018, the loop of SweptVolume::getTrueSDFofSweptVolume with the scaled outer solve
    double getTrueSDFofSweptVolumeS(const double p[3], double &time_seed_f, double grad_prel[3], int *gsip_rounds) const {
        const double PI = 3.14159265358979323846;
        if (gsip_rounds) *gsip_rounds = 0;
        double argmin_dis = getSDFofSweptVolumeS(p, time_seed_f, grad_prel);
        if (argmin_dis > 0) return argmin_dis;
        double vel[3];
        traj.getVel(time_seed_f, vel);
        auto norm3 = [](const double v[3]) { return std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]); };
        if (norm3(vel) < 0.01) {
            if (time_seed_f < 0.1) {
                for (double t_scan = time_seed_f; t_scan <= traj_duration; t_scan += 0.1) {
                    traj.getVel(t_scan, vel);
                    if (norm3(vel) >= 0.01) break;
                }
            } else if (time_seed_f > traj_duration - 0.1) {
                for (double t_scan = time_seed_f; t_scan >= 0; t_scan -= 0.1) {
                    traj.getVel(t_scan, vel);
                    if (norm3(vel) >= 0.01) break;
                }
            }
        }
        double cx = p[0], cy = p[1];
        double r = 10;
        double theta0 = psc::atan2(vel[0], -vel[1]);
        if (theta0 < 0) theta0 += 2 * PI;
        double theta_res = PI + 0.1;
        const double rk_res = 1.5, rk0 = 1.0;
        double r_star = 0, max_g, cur_g, real_t_star = 0, star_rk = 0, star_theta = 0;
        int iter = 1;
        double yk3[3], gtmp[3];
        while (true) {
            max_g = -100000;
            for (double rk = rk0; rk > 0; rk -= rk_res) {
                for (double theta = theta0; theta < theta0 + 2 * PI; theta += theta_res) {
                    double sth, cth;
                    psc::sincos(theta, sth, cth);
                    yk3[0] = cx + rk * r * cth;
                    yk3[1] = cy + rk * r * sth;
                    yk3[2] = 0.0;
                    cur_g = getSDFofSweptVolumeS(yk3, time_seed_f, gtmp);
                    if (cur_g > max_g) {
                        max_g = cur_g;
                        real_t_star = time_seed_f;
                        star_rk = rk;
                        star_theta = theta;
                    }
                }
            }
            r_star = r - max_g;
            r = r_star;
            if (gsip_rounds) (*gsip_rounds)++;
            if (iter > 8) break;
            if (std::abs(max_g) < 0.1) break;
            theta_res /= (2 + 1);
            theta_res = std::max(0.3, theta_res);
            theta0 = star_theta;
            iter++;
        }
        double sst, cst;
        psc::sincos(star_theta, sst, cst);
        double gx = (cx + star_rk * r_star * cst) - p[0], gy = (cy + star_rk * r_star * sst) - p[1], gz = 0.0;
        double z = gx * gx + gy * gy + gz * gz;
        if (z > 0) {
            double nn = std::sqrt(z);
            gx /= nn; gy /= nn; gz /= nn;
        }
        grad_prel[0] = gx; grad_prel[1] = gy; grad_prel[2] = gz;
        time_seed_f = real_t_star;
        return -r_star;
    }
};

// addSaftyPenaOnSweptVolumeParallelTrueSDF :774-869 with St = getScale(t*) (:827) in grad_cost_p_sw :1031-1066:
// xy part -L' (-S^-T R g); yaw part the reference's g^T VR^T (p - x), or with exact_yaw_grad g^T VR^T S^-1 (p - x)
inline void addSafetyPenaltyScaled(const ScaledSweptVolume &sv, const CostParams &cp, int N, const double *coeffs,
                                   const double *points, int64_t P, double &cost, double *gradT, double *gradC,
                                   int64_t *n_inside) {
    int64_t inside = 0;
#pragma omp parallel for num_threads(cp.threads) schedule(dynamic) reduction(+ : inside)
    for (int64_t k = 0; k < P; ++k) {
        double pos_eva[3] = {points[3 * k], points[3 * k + 1], 0.0};
        double gradp_rel[3] = {0, 0, 0};
        double time_star = 0.0;
        double sdf_value = sv.getTrueSDFofSweptVolumeS(pos_eva, time_star, gradp_rel, nullptr);
        if (!(sdf_value > 0)) inside++;
        double time_local = time_star;
        int i = sv.traj.locatePieceIdx(time_local);
        double s1 = time_local, s2 = s1 * s1, s3 = s2 * s1, s4 = s2 * s2, s5 = s4 * s1;
        double beta0[6] = {1.0, s1, s2, s3, s4, s5};
        double beta1[6] = {0.0, 1.0, 2.0 * s1, 3.0 * s2, 4.0 * s3, 5.0 * s4};
        double pos[3], vel[3];
        for (int d = 0; d < 3; ++d) {
            const double *c = coeffs + d * 6 * N + 6 * i;
            double a = 0, b = 0;
            for (int q = 0; q < 6; ++q) { a += c[q] * beta0[q]; b += c[q] * beta1[q]; }
            pos[d] = a; vel[d] = b;
        }
        double sy, cy;
        psc::sincos(pos[2], sy, cy);
        if (sdf_value < 0) {  // :832
            double g0 = cy * gradp_rel[0] + sy * gradp_rel[1];
            double g1 = -sy * gradp_rel[0] + cy * gradp_rel[1];
            gradp_rel[0] = g0; gradp_rel[1] = g1;
        }
        double sdf_cost = -1.0, sdf_out_grad = 0.0;
        smoothedL1(cp.safety_hor - sdf_value, 0.01, sdf_cost, sdf_out_grad);
        double G[3] = {0, 0, 0}, pena = 0.0;
        if (sdf_cost > 0) {
            double i00, i11;
            sv.scale.inv(time_star, i00, i11);
            // rows of -(S^-T R): -(i00 c, -i00 s), -(i11 s, i11 c)
            double rg0 = -((i00 * cy) * gradp_rel[0] + (-(i00 * sy)) * gradp_rel[1]);
            double rg1 = -((i11 * sy) * gradp_rel[0] + (i11 * cy) * gradp_rel[1]);
            double d0 = pos_eva[0] - pos[0], d1 = pos_eva[1] - pos[1];
            if (sv.scale.exact_yaw_grad) { d0 = i00 * d0; d1 = i11 * d1; }
            double w0 = -sy * d0 + cy * d1;
            double w1 = -cy * d0 + -sy * d1;
            G[0] = cp.weight_p * (-sdf_out_grad * rg0);
            G[1] = cp.weight_p * (-sdf_out_grad * rg1);
            G[2] = cp.weight_p * ((-sdf_out_grad * gradp_rel[0]) * w0 + (-sdf_out_grad * gradp_rel[1]) * w1);
            pena = cp.weight_p * sdf_cost;
        }
        double gdT = -(G[0] * vel[0] + G[1] * vel[1] + G[2] * vel[2]);
#pragma omp critical
        {
            cost += pena;
            for (int d = 0; d < 3; ++d)
                for (int q = 0; q < 6; ++q) gradC[d * 6 * N + 6 * i + q] += beta0[q] * G[d];
            for (int j = 0; j < i; ++j) gradT[j] += gdT;
        }
    }
    if (n_inside) *n_inside = inside;
}

// TrajOptimizerOracle with the scaled body: costFunctionLmbmParallel :344-408 as TrajOptimizerOracle::evaluate, with the
// scaled penalty
struct ScaledOptimizer : TrajOptimizerOracle {
    ScaledSweptVolume ssv;
    double evaluate(const double *x, double *g) {
        const int N = pieceN;
        for (int i = 0; i < N; ++i) times[i] = forwardT1(x[i]);
        minco.setParameters(x + N, times.data());
        double cost = minco.getEnergy();
        minco.getEnergyPartialGradByCoeffs(partialGradByCoeffs.data());
        minco.getEnergyPartialGradByTimes(partialGradByTimes.data());
        Trajectory tr;
        trajectory_from_coeffs(N, times.data(), minco.b.data(), tr);
        ssv.updateTraj(tr);
        addSafetyPenaltyScaled(ssv, cp, N, minco.b.data(), points.data(), P, cost, partialGradByTimes.data(),
                               partialGradByCoeffs.data(), nullptr);
        minco.propogateGrad(partialGradByCoeffs.data(), partialGradByTimes.data(), gradByPoints.data(), gradByTimes.data());
        double tsum = 0.0;
        for (int i = 0; i < N; ++i) tsum += times[i];
        cost += rho * tsum;
        for (int i = 0; i < N; ++i) gradByTimes[i] += rho;
        for (int i = 0; i < N; ++i) g[i] = backwardGradT1(x[i], gradByTimes[i]);
        for (int i = 0; i < 3 * (N - 1); ++i) g[N + i] = gradByPoints[i];
        return cost;
    }
};

}  // namespace oracle

using namespace oracle;

extern "C" {

// shape by registry name (unknown names: the rectangle Polygon fallback), or the mesh functor when nf > 0
void *sor_create(const char *name, const double *poly_params, const double *V, int nv, const int *F, int nf, double weight_p,
                 double safety_hor, double rho, int threads) {
    ScaledOptimizer *o = new ScaledOptimizer();
    Shape &S = o->ssv.shape;
    S.id = nf > 0 ? SH_MESH : shape_id_from_name(name ? name : "");
    if (poly_params) S.set_poly_params(poly_params[0], poly_params[1], poly_params[2]);
    if (S.id == SH_MESH) S.set_mesh(V, nv, F, nf);
    else if (S.id == SH_POLYGON) S.set_default_rect();
    o->cp.weight_p = weight_p;
    o->cp.safety_hor = safety_hor;
    o->cp.threads = threads > 0 ? threads : 1;
    o->rho = rho;
    return o;
}
void sor_destroy(void *h) { delete (ScaledOptimizer *)h; }
void sor_set_threads(void *h, int threads) { ((ScaledOptimizer *)h)->cp.threads = threads > 0 ? threads : 1; }
// n[2], c[2], a/w/phi[2][4] row-major
void sor_set_scale(void *h, const int *n, const double *c, const double *a, const double *w, const double *phi, int exact_yaw_grad) {
    ScaleSpec &S = ((ScaledOptimizer *)h)->ssv.scale;
    for (int ax = 0; ax < 2; ++ax) {
        S.n[ax] = n[ax];
        S.c[ax] = c[ax];
        for (int k = 0; k < 4; ++k) {
            S.a[ax][k] = a[4 * ax + k];
            S.w[ax][k] = w[4 * ax + k];
            S.phi[ax][k] = phi[4 * ax + k];
        }
    }
    S.exact_yaw_grad = exact_yaw_grad;
}
void sor_set_points(void *h, const double *pts, int64_t P, int stride) {
    ScaledOptimizer *o = (ScaledOptimizer *)h;
    o->points.resize((size_t)P * 3);
    for (int64_t i = 0; i < P; ++i) {
        o->points[3 * i] = pts[i * stride];
        o->points[3 * i + 1] = pts[i * stride + 1];
        o->points[3 * i + 2] = stride > 2 ? pts[i * stride + 2] : 0.0;
    }
    o->P = P;
}
void sor_set_traj(void *h, int N, const double *T, const double *coeffs) {
    Trajectory tr;
    trajectory_from_coeffs(N, T, coeffs, tr);
    ((ScaledOptimizer *)h)->ssv.updateTraj(tr);
}
// getTrueSDFofSweptVolume<true> per point, stride 3
void sor_query(void *h, int64_t P, const double *pts, double *sdf, double *tstar, double *grad3, int *rounds) {
    ScaledOptimizer *o = (ScaledOptimizer *)h;
#pragma omp parallel for num_threads(o->cp.threads) schedule(dynamic)
    for (int64_t i = 0; i < P; ++i) {
        double p[3] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
        double g[3], ts = 0;
        int r = 0;
        sdf[i] = o->ssv.getTrueSDFofSweptVolumeS(p, ts, g, &r);
        tstar[i] = ts;
        grad3[3 * i] = g[0]; grad3[3 * i + 1] = g[1]; grad3[3 * i + 2] = g[2];
        rounds[i] = r;
    }
}
// the penalty loop, accumulating; returns the number of points that took the interior branch
int64_t sor_cost_grad(void *h, int N, const double *T, const double *coeffs, double *cost_io, double *gradT_io, double *gradC_io) {
    ScaledOptimizer *o = (ScaledOptimizer *)h;
    sor_set_traj(h, N, T, coeffs);
    int64_t inside = 0;
    addSafetyPenaltyScaled(o->ssv, o->cp, N, coeffs, o->points.data(), o->P, *cost_io, gradT_io, gradC_io, &inside);
    return inside;
}
void sor_set_conditions(void *h, const double *initS, const double *finalS, int N) { ((ScaledOptimizer *)h)->setConditions(initS, finalS, N); }
double sor_evaluate(void *h, const double *x, double *g, int n) {
    (void)n;
    return ((ScaledOptimizer *)h)->evaluate(x, g);
}

}  // extern "C"

// svsdf.hpp — header-only C++ mirror of the reference's call surface for the SVSDF path, on top of the C ABI (svsdf.h).
//
// Same class / method names, argument meaning and error behaviour as the reference, minus Eigen and ROS (plain
// std::vector / pointers in the reference's own memory layouts), so reference-side code ports almost verbatim:
//   svsdf::Config                      <- struct Config            (src/utils/include/utils/config.hpp:96-165, hot-path subset)
//   svsdf::shape::BasicShape           <- shape::BasicShape        (src/utils/include/utils/Shape.hpp:96-431) getonlySDF / getonlyGrad1 /
//                                         getSDFwithGrad1; shapeConstructors registry keys (sw_manager.hpp:187-235)
//   svsdf::SweptVolumeManager          <- SweptVolumeManager       (src/swept_volume/include/swept_volume/sw_manager.hpp) updateTraj :376-385,
//                                         getSDFofSweptVolume :844-866, getTrueSDFofSweptVolume :916-1018
//   svsdf::TrajOptimizer               <- TrajOptimizer            (src/planner_algorithm/include/planner_algorithm/back_end_optimizer.hpp)
//                                         setParam :877-932, setEnvironment :935, parallel_points(_num), costFunctionLmbmParallel :344-408,
//                                         addSaftyPenaOnSweptVolumeParallelTrueSDF :774-869, optimize_traj_lmbm (back_end_optimizer.cpp:3-97)
// Errors: like the reference there are no exceptions on the hot path; methods return the solver / status code and
// last_error() gives the text.  Construction throws std::runtime_error when no sm_100 GPU is usable (no CPU fallback).
#pragma once
#include <array>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

extern "C" {
#include "svsdf.h"
}

namespace svsdf {

struct Config {                       // yaml keys of src/plan_manager/config/<shape>.yaml read by the hot path
    std::string inputdata = "shapes/star.obj";
    std::vector<double> poly_params{0.0, 0.0, 0.0};
    double weight_p = 60.0, safety_hor = 0.7, rho = 3.8, inittime = 2.5;
    int threads_num = 12;            // ignored (the GPU replaces the OpenMP team)
    int kernel_size = 17;
    double occupancy_resolution = 1.0, momentum = 0.0;
    int mem_size = 16, past = 3;     // outer L-BFGS (mid-end yaml keys of the reference)
    double min_step = 1.0e-32, g_epsilon = 0.0, relCostTol = 1.0e-6;
    int device = 0;
    bool strict_fp = true;
    std::vector<double> polygon_xy;  // vertices for the Polygon fallback (empty -> the reference's 12 x 0.2 rectangle)
    // Triangle-mesh functor (BasicShape::getonlySDF_igl, Shape.hpp:332-340) instead of a registry shape: either give the mesh
    // directly, or set mesh_sdf = true and let the constructor read `inputdata` as a .obj file path (Shape.hpp:284-285).
    bool mesh_sdf = false;
    std::vector<double> mesh_vertices;  // nv x 3
    std::vector<int32_t> mesh_faces;    // nf x 3, 0-based

    // registry key = basename of inputdata without extension (sw_manager.hpp:350-354)
    std::string shapetype() const {
        size_t s = inputdata.find_last_of('/');
        s = (s == std::string::npos) ? 0 : s + 1;
        size_t e = inputdata.find_last_of('.');
        if (e == std::string::npos || e < s) e = inputdata.size();
        return inputdata.substr(s, e - s);
    }
};

namespace detail {
struct Ctx {
    svsdf_ctx *h = nullptr;
    std::string key;
    explicit Ctx(const Config &c) : key(c.shapetype()) {
        svsdf_config cfg;
        svsdf_default_config(&cfg);
        cfg.shape = key.c_str();
        for (int i = 0; i < 3; ++i) cfg.poly_params[i] = i < (int)c.poly_params.size() ? c.poly_params[i] : 0.0;
        cfg.weight_p = c.weight_p; cfg.safety_hor = c.safety_hor; cfg.rho = c.rho;
        cfg.device = c.device; cfg.strict_fp = c.strict_fp ? 1 : 0;
        if (c.polygon_xy.size() >= 6) { cfg.polygon_xy = c.polygon_xy.data(); cfg.polygon_n = (int)(c.polygon_xy.size() / 2); }
        double *fv = nullptr; int32_t *ff = nullptr;
        if (!c.mesh_faces.empty()) {
            cfg.mesh_vertices = c.mesh_vertices.data(); cfg.mesh_nv = (int)(c.mesh_vertices.size() / 3);
            cfg.mesh_faces = c.mesh_faces.data(); cfg.mesh_nf = (int)(c.mesh_faces.size() / 3);
        } else if (c.mesh_sdf) {
            int nv = 0, nf = 0;
            if (svsdf_read_obj(c.inputdata.c_str(), &fv, &nv, &ff, &nf) != SVSDF_OK) throw std::runtime_error("cannot read mesh " + c.inputdata);
            cfg.mesh_vertices = fv; cfg.mesh_nv = nv; cfg.mesh_faces = ff; cfg.mesh_nf = nf;
        }
        const int rc_create = svsdf_create(&cfg, &h);
        svsdf_free(fv); svsdf_free(ff);
        if (rc_create != SVSDF_OK) h = nullptr;
        if (!h) throw std::runtime_error("svsdf_create failed (no sm_100 CUDA device? there is no CPU fallback)");
    }
    ~Ctx() { svsdf_destroy(h); }
    Ctx(const Ctx &) = delete;
    Ctx &operator=(const Ctx &) = delete;
};
}  // namespace detail

namespace shape {
// The functor API of shape::BasicShape (Shape.hpp:266-270).  pos_rel: body-frame point (x, y, z); z is ignored by the 2-D shapes.
class BasicShape {
   public:
    explicit BasicShape(std::shared_ptr<detail::Ctx> c) : ctx_(std::move(c)) {}
    double getonlySDF(const double pos_rel[3]) const {
        double out = 0.0;
        svsdf_shape_sdf(ctx_->h, 1, pos_rel, &out);
        return out;
    }
    std::array<double, 3> getonlyGrad1(const double pos_rel[3]) const {
        std::array<double, 3> g{0, 0, 0};
        svsdf_shape_grad1(ctx_->h, 1, pos_rel, g.data());
        return g;
    }
    double getSDFwithGrad1(const double pos_rel[3], double grad[3]) const {
        svsdf_shape_grad1(ctx_->h, 1, pos_rel, grad);
        return getonlySDF(pos_rel);
    }
    // batched forms (n rows of 3 doubles): one kernel launch instead of n
    int getonlySDF(int64_t n, const double *pos_rel, double *sdf_out) const { return svsdf_shape_sdf(ctx_->h, n, pos_rel, sdf_out); }
    int getonlyGrad1(int64_t n, const double *pos_rel, double *grad3_out) const { return svsdf_shape_grad1(ctx_->h, n, pos_rel, grad3_out); }

   private:
    std::shared_ptr<detail::Ctx> ctx_;
};
// registry lookup: id of a key of shapeConstructors; unknown names -> the Polygon fallback id (sw_manager.hpp:363-372)
inline int registry_id(const std::string &name) { return svsdf_shape_id(name.c_str()); }
}  // namespace shape

class SweptVolumeManager {
   public:
    typedef std::shared_ptr<SweptVolumeManager> Ptr;
    explicit SweptVolumeManager(const Config &conf) : ctx_(std::make_shared<detail::Ctx>(conf)), current_robot_shape(new shape::BasicShape(ctx_)) {}

    // updateTraj (:376-385).  T: N durations, coeffs: MINCO b (6N x 3, column-major).  Returns 0 or a negative svsdf_status
    // (the reference silently ignores durations >= 300 s; this reports SVSDF_ERR_INVALID).
    int updateTraj(int N, const double *T, const double *coeffs) {
        N_ = N; T_.assign(T, T + N); c_.assign(coeffs, coeffs + 18 * (size_t)N);
        return svsdf_set_traj(ctx_->h, N, T, coeffs);
    }
    // `#define useScale true` plus an edited getScale (:17, :495-507): the body scale S(t) as an svsdf_scale spec (see
    // svsdf.h); nullptr returns to the rigid body.  Returns 0 or SVSDF_ERR_INVALID.
    int setScale(const svsdf_scale *spec) { return svsdf_set_scale(ctx_->h, spec); }
    // getTrueSDFofSweptVolume<true>(pos_eva, time_seed_f, grad_prel, set_ts) (:916-1018); set_ts is ignored like the reference's
    // call sites pass false (the scan always runs).
    double getTrueSDFofSweptVolume(const double pos_eva[3], double &time_seed_f, double grad_prel[3], bool /*set_ts*/ = false) {
        double sdf = 0.0;
        svsdf_query(ctx_->h, N_, T_.data(), c_.data(), 1, pos_eva, &sdf, &time_seed_f, grad_prel, nullptr, 0);
        return sdf;
    }
    // getSDFofSweptVolume<false, true> (:844-866)
    double getSDFofSweptVolume(const double pos_eva[3], double &time_seed_f, double grad_prel[3]) {
        double sdf = 0.0;
        svsdf_query(ctx_->h, N_, T_.data(), c_.data(), 1, pos_eva, &sdf, &time_seed_f, grad_prel, nullptr, 1);
        return sdf;
    }
    // batched query (P rows of 3 doubles): what a caller with many points should use
    int getTrueSDFofSweptVolume(int64_t P, const double *pos_eva, double *sdf, double *tstar, double *grad3, int *rounds = nullptr) {
        return svsdf_query(ctx_->h, N_, T_.data(), c_.data(), P, pos_eva, sdf, tstar, grad3, rounds, 0);
    }
    // ---- A* front end: BasicShape::initShape (Shape.hpp:386-430) + checkKernelValue (:1158-1169), kernelConv (:1033-1096) ----
    // setMap: the byte-packed map kernel of PCSmapManager::generateMapKernel2D (PCSmap_manager.h:81-108)
    int initShape(int kernel_size, int kernel_yaw_num, double occupancy_resolution, double front_end_safeh) {
        return svsdf_front_init(ctx_->h, kernel_size, kernel_yaw_num, occupancy_resolution, front_end_safeh);
    }
    int setMap(const unsigned char *map_kernel, int X, int Y, int kernel_size, double xmin, double ymin, double res) {
        return svsdf_set_map(ctx_->h, map_kernel, X, Y, kernel_size, xmin, ymin, res);
    }
    bool checkKernelValue(double father_yaw, double &child_yaw, const int ind[2]) {
        unsigned char ok = 0;
        int32_t ij[2] = {ind[0], ind[1]};
        double cy = father_yaw;
        if (svsdf_front_check_kernel_value(ctx_->h, 1, &father_yaw, ij, &ok, &cy) != SVSDF_OK) return false;
        if (ok) child_yaw = cy;
        return ok != 0;
    }
    // all nodes of a batch at once / the whole configuration space (free[k][x][w] words, see svsdf.h)
    int checkKernelValue(int64_t n, const double *father_yaw, const int32_t *ind_xy, unsigned char *ok, double *child_yaw) {
        return svsdf_front_check_kernel_value(ctx_->h, n, father_yaw, ind_xy, ok, child_yaw);
    }
    int configurationSpace(uint32_t *free_words, float *ms = nullptr) { return svsdf_front_cspace(ctx_->h, free_words, ms, nullptr); }
    const char *last_error() const { return svsdf_last_error(ctx_->h); }
    svsdf_ctx *handle() const { return ctx_->h; }

   private:
    std::shared_ptr<detail::Ctx> ctx_;
    int N_ = 0;
    std::vector<double> T_, c_;

   public:
    std::unique_ptr<shape::BasicShape> current_robot_shape;
};

class TrajOptimizer {
   public:
    typedef std::shared_ptr<TrajOptimizer> Ptr;
    // reference members kept public on purpose (plan_manager.cpp:168-175 fills them directly)
    std::vector<std::array<double, 3>> parallel_points;
    int parallel_points_num = 0;
    double cost_pos = 0, cost_other = 0, cost_total = 0;
    int pieceN = 0, temporalDim = 0, spatialDim = 0;

    void setParam(const Config &config) { conf = config; }                       // :877-932
    void setEnvironment(SweptVolumeManager::Ptr sv) { sv_manager = std::move(sv); }  // :935

    // call after parallel_points / parallel_points_num have been filled
    int uploadPoints() {
        if (!sv_manager) return SVSDF_ERR_NOT_READY;
        return svsdf_set_points(sv_manager->handle(), parallel_points_num ? parallel_points[0].data() : nullptr, parallel_points_num, 3);
    }

    // addSaftyPenaOnSweptVolumeParallelTrueSDF(ptr, T, coeffs, cost, gradT, gradC) (:774-869): accumulates
    static int addSaftyPenaOnSweptVolumeParallelTrueSDF(void *ptr, int N, const double *T, const double *coeffs, double &cost,
                                                        double *gradT, double *gradC) {
        TrajOptimizer &obj = *static_cast<TrajOptimizer *>(ptr);
        return svsdf_cost_grad(obj.sv_manager->handle(), N, T, coeffs, &cost, gradT, gradC);
    }
    // costFunctionLmbmParallel(ptr, x, g, n) (:344-408): lmbm_evaluate_t compatible
    static double costFunctionLmbmParallel(void *ptr, const double *x_variable, double *g, const int n) {
        TrajOptimizer &obj = *static_cast<TrajOptimizer *>(ptr);
        const double f = svsdf_evaluate(obj.sv_manager->handle(), x_variable, g, n);
        double c3[3];
        if (svsdf_last_costs(obj.sv_manager->handle(), c3) == SVSDF_OK) { obj.cost_pos = c3[0]; obj.cost_other = c3[1]; obj.cost_total = c3[2]; }
        return f;
    }
    int setConditions(const double *initS, const double *finalS, int N) {
        pieceN = N; temporalDim = N; spatialDim = 3 * (N - 1);
        return svsdf_set_boundary(sv_manager->handle(), initS, finalS, N);
    }
    // optimize_traj_lmbm(initS, finalS, opt_x, N, traj) (back_end_optimizer.cpp:3-97): returns >= 0 on success (0 remapped to 1),
    // the negative solver code otherwise; opt_x and the trajectory (T, coeffs) are written either way.  The outer solver is
    // this build's host L-BFGS (lbfgs_ref.hpp semantics); LMBM can drive costFunctionLmbmParallel instead (INTEGRATION.md §2).
    int optimize_traj_lmbm(const double *initS, const double *finalS, std::vector<double> &opt_x, const int N,
                           std::vector<double> &traj_T, std::vector<double> &traj_coeffs, svsdf_opt_stats *stats = nullptr) {
        pieceN = N; temporalDim = N; spatialDim = 3 * (N - 1);
        if ((int)opt_x.size() != temporalDim + spatialDim) return SVSDF_ERR_INVALID;
        svsdf_lbfgs_params p;
        svsdf_default_lbfgs_params(&p);
        p.mem_size = conf.mem_size; p.past = conf.past; p.min_step = conf.min_step; p.g_epsilon = conf.g_epsilon; p.delta = conf.relCostTol;
        traj_T.assign(N, 0.0);
        traj_coeffs.assign(18 * (size_t)N, 0.0);
        return svsdf_optimize(sv_manager->handle(), initS, finalS, opt_x.data(), N, &p, nullptr, nullptr, traj_T.data(), traj_coeffs.data(), stats);
    }

    Config conf;
    SweptVolumeManager::Ptr sv_manager;
};

// Mid end (planner_algorithm/mid_end.hpp, src/mid_end.cpp): host only, no context.
class OriTraj {
   public:
    typedef std::shared_ptr<OriTraj> Ptr;
    svsdf_mid_config conf;  // the yaml keys OriTraj::setParam reads (mid_end.hpp:333-359); defaults = config/star.yaml
    double final_cost = 0.0;
    int iter = 0;

    OriTraj() { svsdf_mid_default_config(&conf); }
    void setParam(const svsdf_mid_config &config) { conf = config; }

    // getOriTraj(initS, finalS, Q, T, acc_list, rot_list, N, traj, opt_x) (mid_end.cpp:3-92).  Q: N - 1 waypoints; rot_list: N - 1
    // rotation matrices, 3x3 column-major each; acc_list is unused by the reference's cost and not taken.  Returns true on
    // success like the reference (solver status >= 0); opt_x, traj_T and traj_coeffs are written either way.
    bool getOriTraj(const double *initS, const double *finalS, const std::vector<std::array<double, 3>> &Q, const std::vector<double> &T,
                    const std::vector<std::array<double, 9>> &rot_list, const int N, std::vector<double> &traj_T, std::vector<double> &traj_coeffs,
                    std::vector<double> &opt_x) {
        if ((int)Q.size() != N - 1 || (int)rot_list.size() != N - 1 || (int)T.size() != N) return false;
        opt_x.assign(N + 3 * (size_t)(N - 1), 0.0);
        traj_T.assign(N, 0.0);
        traj_coeffs.assign(18 * (size_t)N, 0.0);
        const int ret = svsdf_mid_get_ori_traj(&conf, N, initS, finalS, N > 1 ? Q[0].data() : nullptr, T.data(), N > 1 ? rot_list[0].data() : nullptr,
                                               opt_x.data(), traj_T.data(), traj_coeffs.data(), &final_cost, &iter);
        return ret >= 0;
    }
    // costFunction(ptr, x, g, p_cost) (mid_end.hpp:277-325) for callers that bring their own solver
    double costFunction(const double *initS, const double *finalS, const std::vector<std::array<double, 3>> &Q,
                        const std::vector<std::array<double, 9>> &rot_list, const int N, const double *x, double *g) const {
        double c = 0.0;
        svsdf_mid_cost(&conf, N, initS, finalS, Q[0].data(), rot_list[0].data(), x, &c, g);
        return c;
    }
};

}  // namespace svsdf

/* svsdf.h — C ABI of libsvsdf_b200.so: the B200-native drop-in for the SVSDF collision cost + gradient path of
 * ZJU-FAST-Lab/Implicit-SVSDF-Planner.  Plain pointers and sizes only; no C++/torch types cross this boundary.
 * All matrices use the reference's memory layouts (Eigen default column-major) so a maintainer can pass
 * `.data()` of the existing Eigen objects (see INTEGRATION.md for the binding stubs).
 *
 * Reference interfaces replaced (paths relative to /root/reference/src):
 *   R1  TrajOptimizer::addSaftyPenaOnSweptVolumeParallelTrueSDF(void*, const VectorXd& T, const MatrixX3d& coeffs,
 *         double& cost, VectorXd& gradT, MatrixX3d& gradC)
 *         planner_algorithm/include/planner_algorithm/back_end_optimizer.hpp:774-869      -> svsdf_cost_grad
 *   R2  SweptVolumeManager::getTrueSDFofSweptVolume<true>(pos_eva, time_seed_f, grad_prel, set_ts)
 *         swept_volume/include/swept_volume/sw_manager.hpp:916-1018                        -> svsdf_query
 *       SweptVolumeManager::getSDFofSweptVolume<false,true>  sw_manager.hpp:844-866         -> svsdf_query (outer_only=1)
 *       SweptVolumeManager::updateTraj                      sw_manager.hpp:376-385         -> svsdf_set_traj
 *   R3  TrajOptimizer::costFunctionLmbmParallel(void*, const double* x, double* g, int n)
 *         back_end_optimizer.hpp:344-408; callback type lmbm_evaluate_t utils/include/utils/lmbm.h:206-209
 *                                                                                          -> svsdf_evaluate
 *   R4  TrajOptimizer::optimize_traj_lmbm(initS, finalS, opt_x, N, traj)
 *         planner_algorithm/src/back_end_optimizer.cpp:3-97 (outer solver on the host)     -> svsdf_optimize
 *   R5  shape::BasicShape::getonlySDF / getonlyGrad1 and the shapeConstructors registry
 *         utils/include/utils/Shape.hpp:266-270, sw_manager.hpp:187-235,350-373            -> svsdf_shape_sdf/_grad1
 *   R6  TrajOptimizer::setParam / parallel_points / parallel_points_num
 *         back_end_optimizer.hpp:877-932, plan_manager/src/plan_manager.cpp:168-175         -> svsdf_create/_set_points
 *   R7  MINCO_S3NU::setConditions, setParameters, getEnergy..., propogateGrad utils/include/utils/minco.hpp:397-655
 *                                                                                          -> svsdf_minco_*
 *
 * Threading: a context is not thread-safe; use one context per CUDA stream / GPU (the reference has the same
 * restriction: one optimisation per TrajOptimizer instance, back_end_optimizer.hpp:344-408 mutates members).
 * Errors: every int-returning function returns SVSDF_OK (0) or a negative svsdf_status; no exceptions cross
 * the ABI.  The library has no CPU fallback: without a usable CUDA device svsdf_create fails with
 * SVSDF_ERR_CUDA.
 */
#ifndef SVSDF_H_
#define SVSDF_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct svsdf_ctx svsdf_ctx;

typedef enum {
    SVSDF_OK = 0,
    SVSDF_ERR_INVALID = -1,   /* bad argument (null pointer, N out of range, duration >= 300 s, ...) */
    SVSDF_ERR_CUDA = -2,      /* CUDA runtime error or no device; see svsdf_last_error */
    SVSDF_ERR_NOT_READY = -3, /* points / boundary conditions not set */
    SVSDF_ERR_NONFINITE = -4  /* cost or gradient became NaN/Inf */
} svsdf_status;

/* Mirrors the subset of `struct Config` (utils/include/utils/config.hpp) the hot path reads. */
typedef struct {
    const char *shape;        /* registry key = basename of yaml `inputdata` ("star", "sdHorseshoe", ...);
                                 unknown / NULL -> Polygon fallback (rectangle 12 x 0.2 unless polygon_xy given) */
    double poly_params[3];    /* yaml poly_params: body-frame offset x, y and yaw (degrees) of the shape */
    double weight_p;          /* yaml weight_p   (star.yaml: 60.0) */
    double safety_hor;        /* yaml safety_hor (star.yaml: 0.7)  */
    double rho;               /* yaml rho        (star.yaml: 3.8)  */
    int device;               /* CUDA device ordinal */
    int strict_fp;            /* 1 (default): kernels compiled with -fmad=false, bit-compatible with the un-fused
                                 x86-64 arithmetic of the reference; 0: FMA-contracted build (~5-10 % faster, gradient
                                 only within the reference's ~1e-5 contraction noise floor) */
    const double *polygon_xy; /* optional polygon vertices (x0,y0,x1,y1,...) for the fallback shape */
    int polygon_n;            /* number of vertices (<= 64) */
    /* Optional triangle mesh.  When mesh_nf > 0 the robot shape is the reference's mesh functor
       BasicShape::getonlySDF_igl (utils/Shape.hpp:332-340: (1 - 2 * winding number) * distance to the mesh, gradient by
       the same central differences, :35-53) instead of a registry shape; `shape` is then ignored.  poly_params are
       applied to the vertices (R v + trans, Shape.hpp:285-302) at creation; the arrays are copied. */
    const double *mesh_vertices; /* mesh_nv x 3, row-major (x, y, z) */
    int mesh_nv;
    const int32_t *mesh_faces;   /* mesh_nf x 3, 0-based vertex indices */
    int mesh_nf;
} svsdf_config;

/* Fill a config with the reference's star.yaml defaults. */
void svsdf_default_config(svsdf_config *cfg);

int svsdf_create(const svsdf_config *cfg, svsdf_ctx **out);
void svsdf_destroy(svsdf_ctx *ctx);
const char *svsdf_last_error(const svsdf_ctx *ctx);
/* Shape registry lookup: returns the internal id (>= 0); unknown names map to the Polygon fallback id. */
int svsdf_shape_id(const char *name);
/* Radius R (about the body origin, pre-transform included) such that the configured shape functor satisfies
   sdf(q) >= |q| - R for every body-frame point q.  The kernels use it to skip lattice samples of choiceTInit's first layer
   (sw_manager.hpp:538-581) that provably cannot be the minimum; exposed so that the bound can be tested against the oracle
   without a GPU.  Writes a value >= 1e300 when no bound is used (mesh functor).  Host-only, no context needed. */
int svsdf_shape_bound_radius(const svsdf_config *cfg, double *radius_out);
/* Read a Wavefront .obj (what igl::read_triangle_mesh does for yaml `inputdata`, utils/Shape.hpp:284-285): vertices
   (nv x 3 doubles) and fan-triangulated faces (nf x 3, 0-based), malloc'ed; release both with svsdf_free. */
int svsdf_read_obj(const char *path, double **vertices_out, int *nv_out, int32_t **faces_out, int *nf_out);
/* Host-side view of the mesh functor's winding-number hierarchy (csrc/host/fwn_bvh.hpp: the 4-way BVH with order-2
   expansions that igl::fast_winding_number builds, fast_winding_number.cpp:380-457) — for tests and diagnostics, no GPU
   needed.  vertices: nv x 3 doubles as they enter the BVH (shape frame), faces: nf x 3.  Outputs (any may be NULL):
   n_nodes_out; children_out [n_nodes][4] (triangle index | 0x80000000 + node index | 0xffffffff empty; capacity in nodes given by
   node_capacity); data_out [n_nodes][23][4] floats; w_out[n] = winding number at q (n x 3 doubles, float query, accuracy 2.0). */
int svsdf_mesh_fwn_host(const double *vertices, int nv, const int32_t *faces, int nf, int *n_nodes_out, int node_capacity,
                        uint32_t *children_out, float *data_out, int64_t n, const double *q, double *w_out);
void svsdf_free(void *p);

/* R6: parallel_points.  pts: P rows of `stride` doubles (x, y, [z ...]); z is ignored like the reference
 * does (back_end_optimizer.hpp:791).  `pts` is consumed before the call returns (packed into pinned memory by a few host threads, chunk
 * by chunk, each chunk handed to the copy engine at once); the call does not wait for the host -> device transfer itself: whatever is
 * called next on this context runs behind it on the context's stream. */
int svsdf_set_points(svsdf_ctx *ctx, const double *pts, int64_t P, int stride);
/* Same, but the points already live on the device as packed (x, y) pairs; no copy is made of host data. */
int svsdf_set_points_device(svsdf_ctx *ctx, const double *dev_xy, int64_t P);

/* R2: updateTraj.  T: N durations; coeffs: MINCO `b`, 6N x 3 column-major. */
int svsdf_set_traj(svsdf_ctx *ctx, int N, const double *T, const double *coeffs);

/* Deformable robot (the reference's useScale switch with its getScale hook, sw_manager.hpp:17, 495-507): the body maps to
 * the world as p = S(t) R(yaw) q + x, with S(t) = diag(s_x(t), s_y(t), 1) acting along WORLD axes after the rotation (for
 * s_x = s_y the distinction disappears) and t absolute trajectory time.  Per axis ax (0 = x, 1 = y):
 *     s = c[ax];  for (k = 0; k < n_terms[ax]; ++k) s = s + sin(w[ax][k] * t + phi[ax][k]) * a[ax][k];
 * evaluated in exactly that order with the pinned fdlibm sin.  The reference's commented example is n_terms = {1, 1},
 * (c, a, w, phi) = (0.8, 0.6, 1.5, -1.0) for x and (0.8, 0.4, 1.8, 0.0) for y.
 * As in the reference, choiceTInit stays rigid; the descent, the body-frame gradient, the interior branch's ring solves and
 * the chain rule use S(t).  exact_yaw_grad = 0 keeps the reference's yaw term g^T VR^T (p - x) (not the derivative once
 * S != I); 1 uses the true derivative g^T VR^T S^-1 (p - x). */
typedef struct {
    int n_terms[2];   /* 0..4 */
    double c[2], a[2][4], w[2][4], phi[2][4];
    int exact_yaw_grad;
} svsdf_scale;
/* Applies to this context's svsdf_query, svsdf_cost_grad[_device], svsdf_evaluate, svsdf_optimize and batch entries (each
 * context of a pool uses its own spec: give every context of a pool the same one).  The front end (svsdf_front_*), the mid end
 * and svsdf_shape_sdf / _grad1 (body frame) stay rigid, like the reference's.  spec = NULL returns to the rigid body (the
 * default).  SVSDF_ERR_INVALID (the previous setting is kept) when n_terms is outside [0, 4], an entry in use is not
 * finite, or c - sum_k |a_k| <= 0 on either axis (the scale must stay positive for S^-1 to exist). */
int svsdf_set_scale(svsdf_ctx *ctx, const svsdf_scale *spec);

/* R2: per-point swept-volume SDF query on the trajectory given by (N, T, coeffs).
 * pts: P x 3 (x, y, z) host doubles (z ignored).  Outputs (host, may be NULL): sdf[P], tstar[P], grad3[3P]
 * (body-frame FD gradient for sdf > 0; world-frame unit direction for the interior branch, exactly what the
 * reference returns), rounds[P] (GSIP rounds, 0 for outside points).  outer_only = 1 stops after
 * getSDFofSweptVolume (no interior branch). */
int svsdf_query(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, int64_t P, const double *pts,
                double *sdf, double *tstar, double *grad3, int *rounds, int outer_only);

/* R1: accumulate the swept-volume penalty over the context's query points into cost / gradT[N] / gradC[6N x 3
 * column-major] (they already hold the energy terms, as in the reference). */
int svsdf_cost_grad(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, double *cost_io,
                    double *gradT_io, double *gradC_io);

/* R3: boundary conditions (3x3 column-major: column k = k-th derivative of (x, y, yaw)) and piece count. */
int svsdf_set_boundary(svsdf_ctx *ctx, const double *initS, const double *finalS, int N);
/* R3: LMBM / L-BFGS compatible callback: x = [tau (N), xi (3(N-1))] -> cost, g.  `instance` is a svsdf_ctx*. */
double svsdf_evaluate(void *instance, const double *x, double *g, const int n);
/* Cost split of the last svsdf_evaluate: out3 = (cost_pos, cost_other, cost_total)  (back_end_optimizer.hpp:396-398) */
int svsdf_last_costs(const svsdf_ctx *ctx, double *out3);
/* Durations and MINCO coefficients of the last svsdf_evaluate (T_out[N], coeffs_out[18N] column-major). */
int svsdf_get_traj(const svsdf_ctx *ctx, double *T_out, double *coeffs_out);

/* Host L-BFGS parameters (utils/include/utils/lbfgs_ref.hpp:20-130; yaml: mem_size, past, min_step, g_epsilon). */
typedef struct {
    int mem_size;
    int past;
    double delta;
    double g_epsilon;
    int max_iterations;
    int max_linesearch;
    double min_step, max_step;
    double f_dec_coeff, s_curv_coeff, cautious_factor, machine_prec;
    /* Non-smooth handling (the SVSDF cost has kinks and finite-difference gradients; the reference drives it with LMBM for
       that reason, back_end_optimizer.cpp:29-36).  When the line search fails on a quasi-Newton direction the memory is
       dropped and the search restarts along -g, at most this many times in a row without an accepted step; when it fails on
       -g itself the run ends with status 3 (no decrease along the steepest-descent direction to line-search precision:
       the counterpart of LMBM_NOMOREPROGRESS, lmbm.h:182).  0 = plain lbfgs_ref.hpp behaviour (negative line-search code). */
    int nonsmooth_restarts;
} svsdf_lbfgs_params;
void svsdf_default_lbfgs_params(svsdf_lbfgs_params *p);

typedef struct {
    double final_cost;
    int iterations;     /* accepted line-search steps */
    int evaluations;    /* cost+gradient evaluations */
    int status;         /* lbfgs_ref.hpp return code (0 convergence, 1 stop, 3 no more progress at a kink, <0 error) */
    double seconds;     /* wall-clock of the whole optimisation */
    double gpu_seconds; /* sum of device time of the cost kernels (CUDA events) */
} svsdf_opt_stats;

/* Progress / cancel hook, same contract as lmbm_progress_t (lmbm.h:211-213): non-zero return cancels. */
typedef int (*svsdf_progress_t)(void *user, const double *x, const int k);

/* R4: optimise opt_x in place from the given start (opt_x has N + 3(N-1) entries).  Returns >= 0 on success
 * (0 is remapped to 1 like optimize_traj_lmbm does), negative solver code otherwise; the last iterate is
 * returned either way.  T_out / coeffs_out (may be NULL) receive the final trajectory. */
int svsdf_optimize(svsdf_ctx *ctx, const double *initS, const double *finalS, double *opt_x, int N,
                   const svsdf_lbfgs_params *params, svsdf_progress_t progress, void *user, double *T_out,
                   double *coeffs_out, svsdf_opt_stats *stats);

/* Host L-BFGS on an arbitrary callback (same role as lbfgs::lbfgs_optimize, utils/include/utils/lbfgs_ref.hpp:434):
 * minimises eval(instance, x, g, n) from x (in/out).  Re-entrant.  Returns the lbfgs_ref.hpp status code. */
typedef double (*svsdf_eval_t)(void *instance, const double *x, double *g, const int n);
int svsdf_lbfgs_minimize(svsdf_eval_t eval, void *instance, double *x, int n, const svsdf_lbfgs_params *params,
                         svsdf_progress_t progress, void *user, svsdf_opt_stats *stats);

/* R7: host MINCO_S3NU. q: 3 x (N-1) column-major. Outputs may be NULL. */
int svsdf_minco_forward(const double *initS, const double *finalS, int N, const double *q, const double *T,
                        double *coeffs_out, double *energy, double *gradC_out, double *gradT_out);
int svsdf_minco_propagate(const double *initS, const double *finalS, int N, const double *q, const double *T,
                          const double *gradC, const double *gradT, double *gradQ_out, double *gradT_out);
/* tau <-> T maps (back_end_optimizer.hpp:199-289) */
void svsdf_forward_T(int n, const double *tau, double *T);
void svsdf_backward_T(int n, const double *T, double *tau);

/* R5: shape functor over n body-frame points (rel: n x 3, z ignored by the 2-D shapes). */
int svsdf_shape_sdf(svsdf_ctx *ctx, int64_t n, const double *rel, double *sdf_out);
int svsdf_shape_grad1(svsdf_ctx *ctx, int64_t n, const double *rel, double *grad3_out);

/* Device-resident evaluation for benchmarking and batch mode: runs R1 on the given trajectory with every input
 * already in HBM, leaves the result on the device, and returns the device time of the kernels in milliseconds
 * (CUDA events on the context's stream).  out_host (1 + 19N + 1 doubles: cost, gradC[18N] col-major, gradT[N],
 * n_inside) may be NULL. */
int svsdf_cost_grad_device(svsdf_ctx *ctx, int N, const double *T, const double *coeffs, int repeats,
                           float *ms_per_eval, double *out_host);

/* ---- The reference's own outer solver as a plug-in (SURVEY.md §8f rank 4) ------------------------------------------------------------
 * The back end of the reference is driven by LMBM, shipped as a prebuilt Fortran library (src/utils/include/utils/lmbm.so behind
 * lmbm.h / lmbm.cpp).  It is not redistributed here, but a deployment that has it can plug it in: svsdf_lmbm_open loads the library from
 * `path` — by default a PRIVATE COPY of the file, so that every handle has its own instance of the library's static state (lmbm.cpp:4-6
 * keeps the callback in file-scope statics and the Fortran code keeps COMMON / SAVE data): handles can then run concurrently from
 * different threads, which one shared instance cannot.  svsdf_lmbm_params mirrors lmbm::lmbm_parameter_t (lmbm.h:15-174);
 * svsdf_lmbm_default_params fills the struct's member initialisers (what back_end_optimizer.cpp:29 uses). */
typedef struct svsdf_lmbm svsdf_lmbm;
typedef struct {
    float timeout;
    int bundle_size, ini_corrections, max_corrections, exponent_distmeasure, max_iterations, max_evaluations, past, verbose, update_method,
        scaling_strategy;
    double delta_past, f_rel_eps, f_lower_bound, terminate_param1, terminate_param2, distance_measure, sufficient_dec, max_stepsize;
} svsdf_lmbm_params;
void svsdf_lmbm_default_params(svsdf_lmbm_params *p);
int svsdf_lmbm_open(const char *path, int private_copy, svsdf_lmbm **out);
void svsdf_lmbm_close(svsdf_lmbm *h);
const char *svsdf_lmbm_last_error(void);
/* lmbm::lmbm_optimize(n, x, &fx, eval, instance, progress, &param) (lmbm.h:214-221); returns LMBM's code (>= 0 success). */
int svsdf_lmbm_minimize(svsdf_lmbm *h, svsdf_eval_t eval, void *instance, double *x, int n, const svsdf_lmbm_params *params,
                        svsdf_progress_t progress, double *f_out);
/* Makes svsdf_optimize (and svsdf_optimize_batch for this context) run LMBM instead of the built-in L-BFGS: the context takes its own
 * private instance of the library at `path` (NULL: back to L-BFGS).  params NULL = defaults. */
int svsdf_set_lmbm_library(svsdf_ctx *ctx, const char *path, const svsdf_lmbm_params *params);

/* ---- Mid end (SURVEY.md §8f rank 4; host only, no GPU and no context) ---------------------------------------------------------
 * OriTraj (src/planner_algorithm/include/planner_algorithm/mid_end.hpp, src/mid_end.cpp): the warm-start optimisation between the A*
 * front end and the SVSDF back end — MINCO energy + cubic pull of the inner waypoints towards their A* cells + trapezoid integral of
 * the velocity / body-rate / attitude penalties through the multicopter flatness map (utils/flatness.hpp) + rho * sum(T).
 * svsdf_mid_config mirrors the yaml keys OriTraj::setParam reads; svsdf_mid_default_config fills config/star.yaml's values.
 * Layouts: initS / finalS 3x3 column-major; Q 3 x (N - 1) column-major (inner waypoints); rot_list (N - 1) rotation matrices, 3x3
 * column-major each (recent_se3_path[ind].getRotMatrix(), plan_manager.cpp:159); x = [tau (N), xi (3 (N - 1))]. */
typedef struct {
    double rho_mid_end, vmax, omgmax, weight_v, weight_omg, weight_pr, weight_ar, smoothingEps;
    int integralIntervs;
    double vehicleMass, gravAcc, horizDrag, vertDrag, parasDrag, speedEps;
    int mem_size, past;
    double min_step, g_epsilon, relCostTolMidEnd;
    int max_iterations, cancel_after; /* mid_end.cpp:51 (10000) and earlyExit's `k > 1e2` (mid_end.hpp:626) */
    int solver;                       /* 0: the reference's patched L-BFGS behaviour (utils/lbfgs.hpp:375, 759-779) — the same warm start as
                                         the reference; 1: this build's L-BFGS (Lewis-Overton line search, restarts) — converges further */
} svsdf_mid_config;
void svsdf_mid_default_config(svsdf_mid_config *cfg);
/* OriTraj::costFunction (mid_end.hpp:277-325): cost and gradient at x. */
int svsdf_mid_cost(const svsdf_mid_config *cfg, int N, const double *initS, const double *finalS, const double *Q, const double *rot_list,
                   const double *x, double *cost_out, double *grad_out);
/* OriTraj::getOriTraj (mid_end.cpp:3-92): T_init = config.inittime * ones(N) in the reference.  Returns the solver status (>= 0 success,
 * 2 = stopped by the `k > cancel_after` rule); opt_x_out [N + 3 (N - 1)] is what the back end starts from (plan_manager.cpp:192-199),
 * T_out [N], coeffs_out [18 N] (column-major 6N x 3) the resulting spline. */
int svsdf_mid_get_ori_traj(const svsdf_mid_config *cfg, int N, const double *initS, const double *finalS, const double *Q,
                           const double *T_init, const double *rot_list, double *opt_x_out, double *T_out, double *coeffs_out,
                           double *final_cost_out, int *iterations_out);

/* ---- Batch variants (leading problem dimension; BASELINE config 5, SURVEY.md §8b / §8e) -----------------------------------
 * Independent problems are spread over a POOL of contexts (one worker thread per context; several contexts may sit on the
 * same GPU — each has its own stream, so the host side of one problem (MINCO, line search) and the latency-bound tail of its
 * kernels overlap the kernels of another — or on different GPUs of the process).  Problems are handed out dynamically: a
 * worker takes the next index when it finishes one (`next`: optional source of indices shared with other processes, e.g. a
 * counter in the torch.distributed store; return < 0 or >= n_problems to stop; NULL = internal counter 0, 1, 2, ...).
 * Results do not depend on which context solved a problem (bit-reproducible kernels).
 *
 * svsdf_problem: one optimisation.  Query points are either given (points != NULL: P rows of `stride` doubles) or built on
 * the device from the context's map around the waypoints (svsdf_extract_points semantics; the map must have been set on every
 * context of the pool). */
typedef struct {
    const double *initS, *finalS;   /* 3x3 column-major boundary states */
    double *opt_x;                  /* in: start, out: result; N + 3 (N - 1) entries */
    const double *points;           /* explicit query points or NULL */
    int64_t P;
    int stride;
    const double *waypoints_xy;     /* W x 2 (used when points == NULL) */
    int W;
    double half;
    const double *keepout_xy;       /* optional keep-out samples (synthetic scenes), n_keepout x 2 */
    int n_keepout;
    double clearance;
    double *T_out, *coeffs_out;     /* optional: final durations [N] and MINCO coefficients [18 N] */
} svsdf_problem;
typedef int (*svsdf_next_problem_t)(void *user);
/* stats_out[n_problems] (optional), status_out[n_problems] (svsdf_optimize return values), points_out[n_problems] (optional:
 * number of query points of each problem).  Returns SVSDF_OK when every problem ran (individual solver codes are in
 * status_out), the first API error otherwise. */
int svsdf_optimize_batch(svsdf_ctx *const *ctxs, int n_ctx, const svsdf_problem *problems, int n_problems, int N,
                         const svsdf_lbfgs_params *params, svsdf_next_problem_t next, void *next_user,
                         svsdf_opt_stats *stats_out, int *status_out, int64_t *points_out);
/* One cost + gradient evaluation per problem with HOST buffers (the batch form of svsdf_set_points + svsdf_cost_grad):
 * pts[k]: P[k] rows of `stride` doubles; T: [n][N]; coeffs: [n][18 N] column-major per problem; cost_io [n], gradT_io [n][N],
 * gradC_io [n][18 N] accumulate like svsdf_cost_grad. */
int svsdf_cost_grad_batch(svsdf_ctx *const *ctxs, int n_ctx, int n_problems, int N, const double *const *pts, const int64_t *P,
                          int stride, const double *T, const double *coeffs, double *cost_io, double *gradT_io, double *gradC_io);

/* ---- "next" row (SURVEY.md §8f rank 1): query-point construction on the device --------------------------------------
 * R8  PlannerManager::generateTraj point collection  plan_manager/src/plan_manager.cpp:156-175
 *     PCSmapManager::getPointsInAABBOutOfLastOne       map_manager/include/map_manager/PCSmap_manager.h:184-219
 *     on the byte-packed map kernel of PCSmapManager::generateMapKernel2D (PCSmap_manager.h:81-108), z = 0 layer.
 * svsdf_set_map copies the packed map ((X + 2h) rows of ceil((Y + 2h)/8) bytes, h = (kernel_size-1)/2, MSB first) to the
 * device; svsdf_set_map_device adopts a device buffer (e.g. the NCCL-broadcast one) without copying.  origin = the
 * map's boundary_xyzmin (x, y), res = grid resolution. */
int svsdf_set_map(svsdf_ctx *ctx, const unsigned char *kernel_bytes, int X, int Y, int kernel_size, double origin_x,
                  double origin_y, double res);
int svsdf_set_map_device(svsdf_ctx *ctx, const unsigned char *dev_kernel_bytes, int X, int Y, int kernel_size,
                         double origin_x, double origin_y, double res);
/* The reference's 3-D map: generateMapKernel's layout (PCSmap_manager.h:39-78: (X + 2h) x (Y + 2h) x ceil((Z + 2h)/8) bytes, z bits
 * MSB first), origin = boundary_xyzmin (x, y, z).  Re-packed into Z layers of the 2-D layout on upload; layer 0 is what
 * svsdf_set_map would have been given (generateMapKernel2D), so the front-end entry points work on it unchanged.  Z <= 64. */
int svsdf_set_map3d(svsdf_ctx *ctx, const unsigned char *kernel_bytes, int X, int Y, int Z, int kernel_size,
                    const double *origin_xyz, double res);
/* svsdf_extract_points on a 3-D map: waypoints_xyz W x 3, half_xyz = the box half sizes (bdx/3, bdy/3, bdz/3 in
 * plan_manager.cpp:165).  Every occupied voxel of every layer inside a box (and outside the last box in at least one dimension)
 * is a query point; voxels stacked above the same (x, y) give several points with that (x, y) — the cost loop zeroes z
 * (back_end_optimizer.hpp:791).  Output order: layer by layer, ascending (i*Y + j) within a layer. */
int svsdf_extract_points3d(svsdf_ctx *ctx, const double *waypoints_xyz, int W, const double *half_xyz, const double *keepout_xy,
                           int n_keepout, double clearance, int64_t *n_points);
/* Builds the context's resident query-point set from the map: occupied cells inside the AABB (half-size `half` in x and
 * y) of waypoint w and outside the AABB of waypoint w-1 (for w = 0: outside the box around tmp_pos = (999, 999, 999),
 * plan_manager.cpp:152, i.e. the map's far corner cell), de-duplicated, in ascending (i*Y + j) order.
 * waypoints_xy: W x 2.  keepout_xy / clearance (optional, n_keepout = 0 to disable; not part of the reference): drop
 * cells closer than `clearance` to any keep-out sample.  n_points receives the count. */
int svsdf_extract_points(svsdf_ctx *ctx, const double *waypoints_xy, int W, double half, const double *keepout_xy,
                         int n_keepout, double clearance, int64_t *n_points);
/* Copies the context's resident points (packed x, y) back to the host (tests). */
int svsdf_get_points(svsdf_ctx *ctx, double *xy_out, int64_t capacity, int64_t *n_points);

/* ---- Next row (SURVEY.md 8f rank 3): collision kernels of the A* front end -----------------------------------------------
 *   R9  BasicShape::initShape (yaw-indexed occupancy kernels of the shape)      utils/include/utils/Shape.hpp:386-430, 194-216
 *       SweptVolumeManager::kernelConv<true> / visit_kernels_by_distance / checkKernelValue
 *                                                                                swept_volume/include/swept_volume/sw_manager.hpp:1033-1169
 * svsdf_front_init builds the kernel_yaw_num kernels (kernel_size x kernel_size cells of size occupancy_resolution, cell set
 * iff getonlySDF(cell centre, Rz(yaw_k)) <= max(front_end_safeh, occupancy_resolution / 2)) on the device with the context's
 * shape functor; yaml keys kernel_size (odd, <= 32), kernel_yaw_num (<= 64), occupancy_resolution, front_end_safeh.
 * Not available for the Polygon / mesh functors (the reference defines no rotated kernels for them).
 * svsdf_front_get_kernels: yaw_out [K], cells_out [K][ks][ks] (0/1), bytes_out [K][ks][(ks+7)/8] (MSB first) — any may be NULL.
 * svsdf_front_cspace: with the map of svsdf_set_map (packed for the same kernel_size), free[k][x][y] = kernelConv(k, (x, y)) for
 *   every yaw kernel and cell, as 32-cell words: word [k][x][w], bit (31 - t) <-> y = 32 w + t, 1 = no collision; cells beyond
 *   Y read 0.  words_out (host, K * X * ceil(Y/32) words) may be NULL; ms_out = device time of the kernel; dev_words_out = the
 *   device copy (valid until the next call).
 * svsdf_front_check_kernel_value: checkKernelValue(father_yaw, child_yaw, ind) for n nodes: ok_out[i] = a free yaw kernel was
 *   found within the reference's breadth-first search (at most 11 kernels around the father's), child_yaw_out[i] = its yaw
 *   (father_yaw when none). */
/* svsdf_front_expand: the neighbour loop of AstarPathSearcher::process (planner_algorithm/include/planner_algorithm/
 *   front_end_Astar.hpp:192-240) for n nodes at once (e.g. the current node of each problem of a batch): for node i (cell index
 *   node_ij[2i..], yaw node_yaw[i]) and each of its 9 cells (di, dj in -1..1, di-major): ok_out[9i + m] =
 *   isIndexValid && !occupied && checkKernelValue(fy, cy, vi) && checkSubSWCollision((father centre, fy), (child centre, cy),
 *   occupied cell centres within kernel_size/2 + 1 of the child) (sw_manager.hpp:1171-1210, PCSmap_manager.h:137-158);
 *   child_yaw_out[9i + m] = cy.  parts_out (optional): bit 0 valid and free, bit 1 kernel test, bit 2 sub-swept-volume test. */
int svsdf_front_expand(svsdf_ctx *ctx, int64_t n, const int32_t *node_ij, const double *node_yaw, unsigned char *ok_out,
                       double *child_yaw_out, unsigned char *parts_out);
/* svsdf_front_astar: AstarPathSearcher::AstarPathSearch + getPath (front_end_Astar.hpp:243-390; z = 0 layer) for n start/goal
 *   pairs on the map of svsdf_set_map, all searches advancing in lock-step so that every iteration is ONE svsdf_front_expand
 *   launch over the current node of every unfinished search (host logic: csrc/host/astar.hpp; per search it is the
 *   reference's: multimap open list, no re-keying of improved open nodes, re-opening of closed ones, yaw fixed at first
 *   visit).  paths_out [n][max_path][3] = (x, y, yaw) per node, start first; len_out[n] = nodes on the path (0: no path or
 *   longer than max_path); expansions_out[n] / rounds_out (optional): expansions per search / number of lock-step rounds. */
int svsdf_front_astar(svsdf_ctx *ctx, int n, const double *start_xy, const double *goal_xy, int max_path, double *paths_out,
                      int32_t *len_out, int32_t *expansions_out, int64_t *rounds_out);
int svsdf_front_init(svsdf_ctx *ctx, int kernel_size, int kernel_yaw_num, double occupancy_resolution, double front_end_safeh);
int svsdf_front_get_kernels(svsdf_ctx *ctx, double *yaw_out, unsigned char *cells_out, unsigned char *bytes_out);
int svsdf_front_cspace(svsdf_ctx *ctx, uint32_t *words_out, float *ms_out, const uint32_t **dev_words_out);
int svsdf_front_check_kernel_value(svsdf_ctx *ctx, int64_t n, const double *father_yaw, const int32_t *ind_xy,
                                   unsigned char *ok_out, double *child_yaw_out);

/* The device sin/cos used on the path (fdlibm restatement, csrc/svsdf_sincos.cuh), exposed for parity tests. */
int svsdf_sincos(svsdf_ctx *ctx, int64_t n, const double *x, double *sin_out, double *cos_out);

/* Measurement helpers */
/* Device time (ms, CUDA events on the context's stream) of the kernels of the last svsdf_cost_grad_device
 * evaluation: out4 = { k_pose_table, k_outer, k_compact + k_gsip, k_finalize }. */
int svsdf_last_kernel_ms(const svsdf_ctx *ctx, float *out4);
int svsdf_kernel_launches(const svsdf_ctx *ctx, int64_t *count);       /* kernels launched by this ctx so far */
int svsdf_executed_evals(svsdf_ctx *ctx, int enable, uint64_t *count); /* lane-level SDF evaluations counter */
int svsdf_fp64_peak(svsdf_ctx *ctx, double *tflops);                   /* measured DFMA peak (2 flop/FMA) */
int svsdf_device_ptr_points(svsdf_ctx *ctx, const double **dev_xy);    /* device pointer of the packed points */

#ifdef __cplusplus
}
#endif
#endif /* SVSDF_H_ */

// svsdf_launch.h — host-callable launchers exported by the two kernel translation units
// (svsdf_kernels_fast.cu: FMA contraction on; svsdf_kernels_strict.cu: -fmad=false).
#pragma once
#include <cuda_runtime.h>

#include "svsdf_types.h"

namespace svsdf {
#define SVSDF_DECLARE_LAUNCHERS(NS)                                                                              \
    namespace NS {                                                                                               \
    cudaError_t launch_pose_table(double *blob, int K1, cudaStream_t stream);                                    \
    cudaError_t query_occupancy(const ShapeParams &S, int N, int blob_doubles, int *occ_outer, int *occ_gsip);   \
    cudaError_t launch_cost_kernels(const KernelArgs &A, const ShapeParams &S, const ScaleParams *scale, int N,  \
                                    int grid_outer, int grid_gsip, cudaStream_t stream, cudaEvent_t after_outer, \
                                    int gsip_wide);                                                              \
    cudaError_t launch_finalize(const double *partials, int n_blocks, int N, const int *n_inside,                \
                                const double *gsip_contrib, const int *gsip_piece, double *tot,                  \
                                unsigned int *ticket, double *out, cudaStream_t stream);                         \
    cudaError_t launch_shape_eval(const ShapeParams &S, const double *rel_xy, int64_t n, double *out, int grad,  \
                                  cudaStream_t stream);                                                          \
    cudaError_t launch_fp64_peak(double *out, int grid, int iters, cudaStream_t stream);                         \
    cudaError_t launch_sincos(const double *x, int64_t n, double *s, double *c, cudaStream_t stream);            \
    }
SVSDF_DECLARE_LAUNCHERS(fast)
SVSDF_DECLARE_LAUNCHERS(strict)
#undef SVSDF_DECLARE_LAUNCHERS
cudaError_t launch_extract_count(const ExtractArgs &E, int *block_counts, int n_blocks, int64_t *n_total,
                                 cudaStream_t stream);
cudaError_t launch_extract_write(const ExtractArgs &E, const int *block_offsets, int n_blocks, double *out_xy,
                                 int64_t cap, cudaStream_t stream);
// K5 (svsdf_frontend.cu)
cudaError_t launch_front_cells(const ShapeParams &S, const FrontParams &F, const double *yaws, unsigned char *cells, cudaStream_t st);
cudaError_t launch_front_expand(const ShapeParams &S, const FrontParams &F, const SubSwParams &P, const unsigned char *map,
                                const unsigned char *kbytes, int64_t n, const int *node_ij, const double *node_yaw, unsigned char *ok_out,
                                double *child_yaw_out, unsigned char *parts_out, cudaStream_t st);
cudaError_t launch_front_cspace(const FrontParams &F, const unsigned char *map, const unsigned *rowmask, unsigned *out, cudaStream_t st);
cudaError_t launch_front_check(const FrontParams &F, const unsigned char *map, const unsigned char *kbytes, int64_t n, const double *father_yaw,
                               const int *ind_xy, unsigned char *ok_out, double *child_yaw_out, cudaStream_t st);
}  // namespace svsdf

// TEST INFRASTRUCTURE ONLY -- C-ABI shim over the reference's own CUDA launchers.
// oracle/Makefile compiles the reference .cu files UNMODIFIED, from where they lie under
// $PCREID_REFERENCE_ROOT/mmdet3d/ops/*/src/, together with this file into oracle/_ref/libref_ops.so.
// (The reference's pybind .cpp wrappers include the removed THC/THC.h and do not build against
// torch 2.11, so the launchers are bound directly.)  Gives a bit-level GPU oracle and the
// "reference kernel recompiled for sm_100a" speed bar on the GPU box.
#include <cuda_runtime.h>

void furthest_point_sampling_kernel_launcher(int b, int n, int m, const float *dataset, float *temp, int *idxs, cudaStream_t stream);
void furthest_point_sampling_with_dist_kernel_launcher(int b, int n, int m, const float *dataset, float *temp, int *idxs, cudaStream_t stream);
void knn_kernel_launcher(int b, int n, int m, int nsample, const float *xyz, const float *new_xyz, int *idx, float *dist2, cudaStream_t stream);
void ball_query_kernel_launcher(int b, int n, int m, float min_radius, float max_radius, int nsample, const float *new_xyz, const float *xyz, int *idx, cudaStream_t stream);
void group_points_kernel_launcher(int b, int c, int n, int npoints, int nsample, const float *points, const int *idx, float *out, cudaStream_t stream);
void gather_points_kernel_launcher(int b, int c, int n, int npoints, const float *points, const int *idx, float *out, cudaStream_t stream);

void three_nn_kernel_launcher(int b, int n, int m, const float *unknown, const float *known, float *dist2, int *idx, cudaStream_t stream);
void three_interpolate_kernel_launcher(int b, int c, int m, int n, const float *points, const int *idx, const float *weight, float *out, cudaStream_t stream);

extern "C" {
void ref_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2, int *idx, void *stream) {
  three_nn_kernel_launcher(b, n, m, unknown, known, dist2, idx, (cudaStream_t)stream);
}
void ref_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx, const float *weight, float *out, void *stream) {
  three_interpolate_kernel_launcher(b, c, m, n, points, idx, weight, out, (cudaStream_t)stream);
}
void ref_fps(int b, int n, int m, const float *xyz, float *temp, int *idx, void *stream) {
  furthest_point_sampling_kernel_launcher(b, n, m, xyz, temp, idx, (cudaStream_t)stream);
}
void ref_fps_with_dist(int b, int n, int m, const float *dist, float *temp, int *idx, void *stream) {
  furthest_point_sampling_with_dist_kernel_launcher(b, n, m, dist, temp, idx, (cudaStream_t)stream);
}
void ref_knn(int b, int n, int m, int k, const float *xyz, const float *new_xyz, int *idx, float *dist2, void *stream) {
  knn_kernel_launcher(b, n, m, k, xyz, new_xyz, idx, dist2, (cudaStream_t)stream);
}
void ref_ball_query(int b, int n, int m, float rmin, float rmax, int k, const float *new_xyz, const float *xyz, int *idx, void *stream) {
  ball_query_kernel_launcher(b, n, m, rmin, rmax, k, new_xyz, xyz, idx, (cudaStream_t)stream);
}
void ref_group_points(int b, int c, int n, int s, int k, const float *points, const int *idx, float *out, void *stream) {
  group_points_kernel_launcher(b, c, n, s, k, points, idx, out, (cudaStream_t)stream);
}
void ref_gather_points(int b, int c, int n, int m, const float *points, const int *idx, float *out, void *stream) {
  gather_points_kernel_launcher(b, c, n, m, points, idx, out, (cudaStream_t)stream);
}
}

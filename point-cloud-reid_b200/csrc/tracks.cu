// Device-resident track table (include/pcreid.h, pcreid_track_*): S scenes x C slots, every scene updated in one launch.
//
// Slot arrays are flat over S * C (global row s * C + slot); scene s's active list (its alive slots in ascending order, as
// global rows) sits at active[s * C ..] with active_count[s] entries.  A step passes int64 offsets [3][S + 1], exclusive
// prefix sums over the scenes of [0] A_s (active tracks entering the step), [1] D_s (detections), [2] A_s * D_s (gate
// elements); a scene without a frame has A_s = D_s = 0 and is left exactly as it is.
//
// pcreid_track_gate_blocks: the class gate (+ optional ground-plane centre distance) of every scene's (A_s, D_s) block.
// pcreid_track_update:      one CTA per scene: matched tracks, ageing / retirement, new tracks in the lowest free slots,
//                           then the next active list.  Ranks come from block-wide scans over contiguous per-thread ranges,
//                           so they are in slot / detection order whatever the thread count.
// pcreid_track_scatter:     the stored detections' xyz / feature rows (opaque bytes) into their table rows.
//
// Motion (constant-velocity Kalman filter per slot, the compact covariance of include/pcreid.h), one thread per track or
// detection, f32 without contraction so that the CPU restatement reproduces it bit for bit:
// pcreid_track_predict:            every active track of a scene with a frame, by that scene's dt.
// pcreid_track_correct:            after pcreid_track_update: matched tracks take their detection, newborn slots start.
// pcreid_track_gate_motion_blocks: pcreid_track_gate_blocks' gate on the predicted boxes, plus a Mahalanobis bound.
#include "../../include/pcreid.h"
#include "common.cuh"

#include <cmath>
#include <cstdint>

namespace {

constexpr int TRACK_MAX = 4096;          // C and D_s: the lsap limit, so every scene's active tracks can be solved
constexpr int MAX_SCENES = 65535;
constexpr int UPDATE_THREADS = 512;
constexpr int GATE_THREADS = 256;
constexpr int SCATTER_THREADS = 256;
constexpr long long SCATTER_CHUNK = SCATTER_THREADS * 16 * 4;   // bytes of one row one CTA copies

constexpr int MOTION_THREADS = 256;
constexpr int COV = 13;                  // the compact covariance of one slot (include/pcreid.h)
constexpr float TWO_PI = 6.28318548f;    // fl(2 pi) = 2 fl(pi)
constexpr float PI_F = 3.14159274f;      // fl(pi)
constexpr float HALF_PI = 1.57079637f;   // fl(pi / 2)

// the gate of table row r and detection j.  cov == nullptr: class rule and radius only (pcreid_track_gate_blocks); else the
// ground-plane Mahalanobis bound as well.  No contraction: the CPU restatement reproduces this bit for bit.
__device__ __forceinline__ bool gate_pair(long long r, long long j, const int* __restrict__ label,
                                          const int* __restrict__ length, const float* __restrict__ box,
                                          const int* __restrict__ det_label, const int* __restrict__ det_length,
                                          const float* __restrict__ det_box, int num_classes, int min_points, int use_lengths,
                                          const float* __restrict__ r2, const float* __restrict__ cov, float meas_var,
                                          float chi2) {
  const int lt = label[r];
  bool ok = lt == det_label[j] && lt >= 0 && lt < num_classes;
  if (use_lengths) ok = ok && length[r] >= min_points && det_length[j] >= min_points;
  if (ok && (r2 || cov)) {
    const float dx = __fsub_rn(box[r * 7], det_box[j * 7]), dy = __fsub_rn(box[r * 7 + 1], det_box[j * 7 + 1]);
    if (r2) ok = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) <= r2[lt];
    if (ok && cov) {
      const float sx = __fadd_rn(cov[r * COV], meas_var), sy = __fadd_rn(cov[r * COV + 3], meas_var);
      ok = __fadd_rn(__fdiv_rn(__fmul_rn(dx, dx), sx), __fdiv_rn(__fmul_rn(dy, dy), sy)) <= chi2;
    }
  }
  return ok;
}

// the packed gate of scene blockIdx.y's (A_s, D_s) block, grid-stride over its elements; both gate kernels are this loop
__device__ __forceinline__ void gate_blocks(int S, int C, const long long* __restrict__ off, const int* __restrict__ active,
                                            const int* __restrict__ label, const int* __restrict__ length,
                                            const float* __restrict__ box, const int* __restrict__ det_label,
                                            const int* __restrict__ det_length, const float* __restrict__ det_box,
                                            int num_classes, int min_points, int use_lengths, const float* __restrict__ r2,
                                            const float* __restrict__ cov, float meas_var, float chi2,
                                            unsigned char* __restrict__ gate) {
  const int s = blockIdx.y;
  const int A = (int)(off[s + 1] - off[s]);
  const int D = (int)(off[(S + 1) + s + 1] - off[(S + 1) + s]);
  const long long d0 = off[(S + 1) + s], e0 = off[2 * (S + 1) + s];
  const long long n = (long long)A * D;
  const int* act = active + (long long)s * C;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / D);
    const long long j = d0 + (e - (long long)i * D);
    gate[e0 + e] = gate_pair(act[i], j, label, length, box, det_label, det_length, det_box, num_classes, min_points, use_lengths,
                             r2, cov, meas_var, chi2) ? 1 : 0;
  }
}

__global__ void __launch_bounds__(GATE_THREADS) track_gate_kernel(int S, int C, const long long* __restrict__ off,
                                                                   const int* __restrict__ active,
                                                                   const int* __restrict__ label,
                                                                   const int* __restrict__ length,
                                                                   const float* __restrict__ box,
                                                                   const int* __restrict__ det_label,
                                                                   const int* __restrict__ det_length,
                                                                   const float* __restrict__ det_box, int num_classes,
                                                                   int min_points, int use_lengths,
                                                                   const float* __restrict__ r2,
                                                                   unsigned char* __restrict__ gate) {
  gate_blocks(S, C, off, active, label, length, box, det_label, det_length, det_box, num_classes, min_points, use_lengths, r2,
              nullptr, 0.f, 0.f, gate);
}

// pcreid_track_gate_motion_blocks: track_gate_kernel on the predicted boxes, plus the Mahalanobis bound when cov != nullptr
__global__ void __launch_bounds__(GATE_THREADS) track_gate_motion_kernel(
    int S, int C, const long long* __restrict__ off, const int* __restrict__ active, const int* __restrict__ label,
    const int* __restrict__ length, const float* __restrict__ box, const int* __restrict__ det_label,
    const int* __restrict__ det_length, const float* __restrict__ det_box, int num_classes, int min_points, int use_lengths,
    const float* __restrict__ r2, const float* __restrict__ cov, float meas_var, float chi2, unsigned char* __restrict__ gate) {
  gate_blocks(S, C, off, active, label, length, box, det_label, det_length, det_box, num_classes, min_points, use_lengths, r2,
              cov, meas_var, chi2, gate);
}

__device__ __forceinline__ float wrap_angle(float a) {
  return __fsub_rn(a, __fmul_rn(TWO_PI, rintf(__fdiv_rn(a, TWO_PI))));
}

// thread (x, s): track i of scene s (row active[s * C + i]) moves by dt[s] * velocity; its covariance grows
__global__ void __launch_bounds__(MOTION_THREADS) track_predict_kernel(int S, int C, const long long* __restrict__ off,
                                                                        const int* __restrict__ active,
                                                                        const float* __restrict__ dt_s, float* __restrict__ kf_box,
                                                                        float* __restrict__ kf_vel, float* __restrict__ kf_cov,
                                                                        float q, float q_vel) {
  const int s = blockIdx.y;
  const int A = (int)(off[s + 1] - off[s]);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A) return;
  const long long r = active[(long long)s * C + i];
  const float dt = dt_s[s];
  float* b = kf_box + r * 7;
  float* P = kf_cov + r * COV;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float v = kf_vel[r * 3 + a];
    const float pp = P[3 * a], pv = P[3 * a + 1], vv = P[3 * a + 2];
    b[a] = __fadd_rn(b[a], __fmul_rn(dt, v));
    const float t = __fadd_rn(pv, __fmul_rn(dt, vv));
    P[3 * a] = __fadd_rn(__fadd_rn(pp, __fmul_rn(dt, __fadd_rn(pv, t))), q);
    P[3 * a + 1] = t;
    P[3 * a + 2] = __fadd_rn(vv, q_vel);
  }
#pragma unroll
  for (int k = 9; k < COV; ++k) P[k] = __fadd_rn(P[k], q);
}

// thread (x, s): detection d of scene s corrects its matched track, or initialises the slot it was born into
__global__ void __launch_bounds__(MOTION_THREADS) track_correct_kernel(
    int S, const long long* __restrict__ off, const long long* __restrict__ track_rows, const long long* __restrict__ track_for_det,
    const float* __restrict__ det_box, const int* __restrict__ det_row, float* __restrict__ kf_box, float* __restrict__ kf_vel,
    float* __restrict__ kf_cov, float init_var, float init_vel_var, float meas_var) {
  const int s = blockIdx.y;
  const int D = (int)(off[(S + 1) + s + 1] - off[(S + 1) + s]);
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  const long long j = off[(S + 1) + s] + d;
  const long long t = track_for_det[j];
  const float* z = det_box + j * 7;
  if (t < 0) {
    const long long r = det_row[j];
    if (r < 0) return;                                   // dropped: no slot
#pragma unroll
    for (int k = 0; k < 6; ++k) kf_box[r * 7 + k] = z[k];
    kf_box[r * 7 + 6] = wrap_angle(z[6]);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      kf_vel[r * 3 + a] = 0.f;
      kf_cov[r * COV + 3 * a] = init_var;
      kf_cov[r * COV + 3 * a + 1] = 0.f;
      kf_cov[r * COV + 3 * a + 2] = init_vel_var;
    }
#pragma unroll
    for (int k = 9; k < COV; ++k) kf_cov[r * COV + k] = init_var;
    return;
  }
  const long long r = track_rows[off[s] + t];
  float* b = kf_box + r * 7;
  float* P = kf_cov + r * COV;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float pp = P[3 * a], pv = P[3 * a + 1], vv = P[3 * a + 2];
    const float sa = __fadd_rn(pp, meas_var);
    const float kp = __fdiv_rn(pp, sa), kv = __fdiv_rn(pv, sa);
    const float y = __fsub_rn(z[a], b[a]);
    b[a] = __fadd_rn(b[a], __fmul_rn(kp, y));
    kf_vel[r * 3 + a] = __fadd_rn(kf_vel[r * 3 + a], __fmul_rn(kv, y));
    P[3 * a + 2] = __fsub_rn(vv, __fmul_rn(kv, pv));
    P[3 * a + 1] = __fmul_rn(kv, meas_var);
    P[3 * a] = __fmul_rn(kp, meas_var);
  }
#pragma unroll
  for (int a = 3; a < 6; ++a) {
    const float k = __fdiv_rn(P[6 + a], __fadd_rn(P[6 + a], meas_var));
    b[a] = __fadd_rn(b[a], __fmul_rn(k, __fsub_rn(z[a], b[a])));
    P[6 + a] = __fmul_rn(k, meas_var);
  }
  // yaw: the innovation wrapped to (-pi, pi], and turned by pi when the detection's heading is flipped (AB3DMOT)
  const float k = __fdiv_rn(P[12], __fadd_rn(P[12], meas_var));
  float y = wrap_angle(__fsub_rn(z[6], b[6]));
  if (fabsf(y) > HALF_PI) y = wrap_angle(__fadd_rn(y, PI_F));
  b[6] = wrap_angle(__fadd_rn(b[6], __fmul_rn(k, y)));
  P[12] = __fmul_rn(k, meas_var);
}

// exclusive prefix of v over the CTA in thread order; *total = the sum.  Every thread calls it; sh holds 32 ints.
__device__ int block_scan(int v, int* total, int* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(FULL_MASK, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = lane < nw ? sh[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(FULL_MASK, w, o);
      if (lane >= o) w += y;
    }
    sh[lane] = w;
  }
  __syncthreads();
  const int before = (warp ? sh[warp - 1] : 0) + x - v;
  *total = sh[nw - 1];
  __syncthreads();
  return before;
}

__global__ void __launch_bounds__(UPDATE_THREADS) track_update_kernel(
    int S, int C, const long long* __restrict__ off, const long long* __restrict__ track_for_det,
    const int* __restrict__ det_label, const int* __restrict__ det_length, const float* __restrict__ det_box, int max_age,
    int replace_all, unsigned char* __restrict__ alive, long long* __restrict__ track_id, int* __restrict__ label,
    int* __restrict__ length, int* __restrict__ age, int* __restrict__ hits, float* __restrict__ box,
    long long* __restrict__ next_id, long long* __restrict__ dropped, int* __restrict__ active, int* __restrict__ active_count,
    long long* __restrict__ det_track_id, int* __restrict__ det_row) {
  __shared__ unsigned char matched[TRACK_MAX];   // per position of the active list
  __shared__ short free_slot[TRACK_MAX];         // k-th free slot after ageing
  __shared__ int sh[32];
  const int s = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const int A = (int)(off[s + 1] - off[s]);
  const int D = (int)(off[(S + 1) + s + 1] - off[(S + 1) + s]);
  if (A == 0 && D == 0) return;                  // no frame, or nothing to age or store: the scene is unchanged
  const long long d0 = off[(S + 1) + s];
  const long long base = (long long)s * C;
  int* act = active + base;
  const long long* tfd = track_for_det + d0;

  // 1. matched track t <- detection d
  for (int i = tid; i < A; i += nthr) matched[i] = 0;
  __syncthreads();
  for (int d = tid; d < D; d += nthr) {
    const long long t = tfd[d];
    if (t < 0) continue;
    matched[t] = 1;
    const long long r = act[t];
    const long long j = d0 + d;
    age[r] = 0;
    hits[r] += 1;
#pragma unroll
    for (int k = 0; k < 7; ++k) box[r * 7 + k] = det_box[j * 7 + k];
    const int ld = det_length[j];
    int row = -1;
    if (replace_all || length[r] <= ld) {
      length[r] = ld;
      row = (int)r;
    }
    det_track_id[j] = track_id[r];
    det_row[j] = row;
  }
  __syncthreads();

  // 2. unmatched active tracks age; past max_age (>= 0) the slot is freed
  for (int i = tid; i < A; i += nthr) {
    if (matched[i]) continue;
    const long long r = act[i];
    const int a = age[r] + 1;
    age[r] = a;
    if (max_age >= 0 && a > max_age) alive[r] = 0;
  }
  __syncthreads();

  // 3. the k-th unmatched detection (ascending d) takes the k-th lowest free slot
  const int cper = (C + nthr - 1) / nthr, c_lo = min(C, tid * cper), c_hi = min(C, c_lo + cper);
  int n = 0;
  for (int j = c_lo; j < c_hi; ++j) n += alive[base + j] ? 0 : 1;
  int nfree;
  int k = block_scan(n, &nfree, sh);
  for (int j = c_lo; j < c_hi; ++j)
    if (!alive[base + j]) free_slot[k++] = (short)j;
  const int dper = (D + nthr - 1) / nthr, d_lo = min(D, tid * dper), d_hi = min(D, d_lo + dper);
  n = 0;
  for (int d = d_lo; d < d_hi; ++d) n += tfd[d] < 0 ? 1 : 0;
  int unmatched;
  k = block_scan(n, &unmatched, sh);             // its barriers also publish free_slot
  const long long first_id = next_id[s];
  for (int d = d_lo; d < d_hi; ++d) {
    if (tfd[d] >= 0) continue;
    const long long j = d0 + d;
    if (k < nfree) {
      const long long r = base + free_slot[k];
      alive[r] = 1;
      track_id[r] = first_id + k;
      label[r] = det_label[j];
      length[r] = det_length[j];
      age[r] = 0;
      hits[r] = 1;
#pragma unroll
      for (int q = 0; q < 7; ++q) box[r * 7 + q] = det_box[j * 7 + q];
      det_track_id[j] = first_id + k;
      det_row[j] = (int)r;
    } else {
      det_track_id[j] = -1;
      det_row[j] = -1;
    }
    ++k;
  }
  __syncthreads();
  if (tid == 0) {
    const int stored = min(unmatched, nfree);
    next_id[s] = first_id + stored;
    dropped[s] += unmatched - stored;
  }

  // 4. the next active list: alive slots in ascending order
  n = 0;
  for (int j = c_lo; j < c_hi; ++j) n += alive[base + j] ? 1 : 0;
  int total;
  k = block_scan(n, &total, sh);
  for (int j = c_lo; j < c_hi; ++j)
    if (alive[base + j]) act[k++] = (int)(base + j);
  if (tid == 0) active_count[s] = total;
}

__device__ __forceinline__ void copy_chunk(const unsigned char* __restrict__ src, unsigned char* __restrict__ dst,
                                           long long bytes, long long chunk) {
  const long long lo = chunk * SCATTER_CHUNK, hi = min(bytes, lo + SCATTER_CHUNK);
  if (lo >= hi) return;
  if ((((uintptr_t)src | (uintptr_t)dst | (uintptr_t)bytes) & 15) == 0) {
    for (long long b = lo + threadIdx.x * 16; b < hi; b += SCATTER_THREADS * 16)
      *reinterpret_cast<uint4*>(dst + b) = __ldg(reinterpret_cast<const uint4*>(src + b));
  } else if ((((uintptr_t)src | (uintptr_t)dst | (uintptr_t)bytes) & 3) == 0) {
    for (long long b = lo + threadIdx.x * 4; b < hi; b += SCATTER_THREADS * 4)
      *reinterpret_cast<unsigned*>(dst + b) = __ldg(reinterpret_cast<const unsigned*>(src + b));
  } else {
    for (long long b = lo + threadIdx.x; b < hi; b += SCATTER_THREADS) dst[b] = src[b];
  }
}

// CTA (d, c): chunk c of detection d's two rows, when det_row[d] >= 0
__global__ void __launch_bounds__(SCATTER_THREADS) track_scatter_kernel(const int* __restrict__ det_row, long long bytes_a,
                                                                         const unsigned char* __restrict__ src_a,
                                                                         unsigned char* __restrict__ dst_a, long long bytes_b,
                                                                         const unsigned char* __restrict__ src_b,
                                                                         unsigned char* __restrict__ dst_b) {
  const long long d = blockIdx.x;
  const int r = det_row[d];
  if (r < 0) return;
  if (bytes_a) copy_chunk(src_a + d * bytes_a, dst_a + (long long)r * bytes_a, bytes_a, blockIdx.y);
  if (bytes_b) copy_chunk(src_b + d * bytes_b, dst_b + (long long)r * bytes_b, bytes_b, blockIdx.y);
}

}  // namespace

extern "C" {

int pcreid_track_gate_blocks(int S, int C, int max_A, int max_D, const long long* offsets, const int* active, const int* label,
                             const int* length, const float* box, const int* det_label, const int* det_length,
                             const float* det_box, int num_classes, int min_points, int use_lengths, const float* r2,
                             unsigned char* gate, void* stream) {
  if (S < 0 || C < 1 || max_A < 0 || max_D < 0 || max_A > C || num_classes < 0) return PCREID_ERR_ARG;
  if (S > MAX_SCENES || C > TRACK_MAX || max_D > TRACK_MAX) return PCREID_ERR_UNSUPPORTED;
  if (S == 0 || max_A == 0 || max_D == 0) return PCREID_OK;
  if (!offsets || !active || !label || !det_label || !gate || (use_lengths && (!length || !det_length)) ||
      (r2 && (!box || !det_box)))
    return PCREID_ERR_ARG;
  const long long per_scene = (long long)max_A * max_D;
  const int gx = (int)min((per_scene + GATE_THREADS - 1) / GATE_THREADS, 1024LL);
  track_gate_kernel<<<dim3(gx, S), GATE_THREADS, 0, (cudaStream_t)stream>>>(S, C, offsets, active, label, length, box, det_label,
                                                                            det_length, det_box, num_classes, min_points,
                                                                            use_lengths, r2, gate);
  return pcreid_launch_status();
}

int pcreid_track_gate_motion_blocks(int S, int C, int max_A, int max_D, const long long* offsets, const int* active,
                                    const int* label, const int* length, const float* box, const int* det_label,
                                    const int* det_length, const float* det_box, int num_classes, int min_points, int use_lengths,
                                    const float* r2, const float* kf_cov, float r, float gate_chi2, unsigned char* gate,
                                    void* stream) {
  if (S < 0 || C < 1 || max_A < 0 || max_D < 0 || max_A > C || num_classes < 0) return PCREID_ERR_ARG;
  if (!(isfinite(gate_chi2) && isfinite(r))) return PCREID_ERR_ARG;
  const bool chi2 = gate_chi2 > 0.f;
  if (chi2 && !(r > 0.f)) return PCREID_ERR_ARG;
  if (S > MAX_SCENES || C > TRACK_MAX || max_D > TRACK_MAX) return PCREID_ERR_UNSUPPORTED;
  if (S == 0 || max_A == 0 || max_D == 0) return PCREID_OK;
  if (!offsets || !active || !label || !det_label || !gate || (use_lengths && (!length || !det_length)) ||
      ((r2 || chi2) && (!box || !det_box)) || (chi2 && !kf_cov))
    return PCREID_ERR_ARG;
  const long long per_scene = (long long)max_A * max_D;
  const int gx = (int)min((per_scene + GATE_THREADS - 1) / GATE_THREADS, 1024LL);
  track_gate_motion_kernel<<<dim3(gx, S), GATE_THREADS, 0, (cudaStream_t)stream>>>(
      S, C, offsets, active, label, length, box, det_label, det_length, det_box, num_classes, min_points, use_lengths, r2,
      chi2 ? kf_cov : nullptr, r, gate_chi2, gate);
  return pcreid_launch_status();
}

int pcreid_track_predict(int S, int C, int max_A, const long long* offsets, const int* active, const float* dt, float* kf_box,
                         float* kf_vel, float* kf_cov, float q, float q_vel, void* stream) {
  if (S < 0 || C < 1 || max_A < 0 || max_A > C) return PCREID_ERR_ARG;
  if (!(isfinite(q) && q >= 0.f && isfinite(q_vel) && q_vel >= 0.f)) return PCREID_ERR_ARG;
  if (S > MAX_SCENES || C > TRACK_MAX) return PCREID_ERR_UNSUPPORTED;
  if (S == 0 || max_A == 0) return PCREID_OK;
  if (!offsets || !active || !dt || !kf_box || !kf_vel || !kf_cov) return PCREID_ERR_ARG;
  track_predict_kernel<<<dim3((max_A + MOTION_THREADS - 1) / MOTION_THREADS, S), MOTION_THREADS, 0, (cudaStream_t)stream>>>(
      S, C, offsets, active, dt, kf_box, kf_vel, kf_cov, q, q_vel);
  return pcreid_launch_status();
}

int pcreid_track_correct(int S, int C, int max_D, const long long* offsets, const long long* track_rows,
                         const long long* track_for_det, const float* det_box, const int* det_row, float* kf_box, float* kf_vel,
                         float* kf_cov, float init_var, float init_vel_var, float r, void* stream) {
  if (S < 0 || C < 1 || max_D < 0) return PCREID_ERR_ARG;
  if (!(isfinite(init_var) && init_var > 0.f && isfinite(init_vel_var) && init_vel_var > 0.f && isfinite(r) && r > 0.f))
    return PCREID_ERR_ARG;
  if (S > MAX_SCENES || C > TRACK_MAX || max_D > TRACK_MAX) return PCREID_ERR_UNSUPPORTED;
  if (S == 0 || max_D == 0) return PCREID_OK;
  if (!offsets || !track_for_det || !det_box || !det_row || !kf_box || !kf_vel || !kf_cov) return PCREID_ERR_ARG;
  track_correct_kernel<<<dim3((max_D + MOTION_THREADS - 1) / MOTION_THREADS, S), MOTION_THREADS, 0, (cudaStream_t)stream>>>(
      S, offsets, track_rows, track_for_det, det_box, det_row, kf_box, kf_vel, kf_cov, init_var, init_vel_var, r);
  return pcreid_launch_status();
}

int pcreid_track_update(int S, int C, int max_D, const long long* offsets, const long long* track_for_det, const int* det_label,
                        const int* det_length, const float* det_box, int max_age, int replace_all, unsigned char* alive,
                        long long* track_id, int* label, int* length, int* age, int* hits, float* box, long long* next_id,
                        long long* dropped, int* active, int* active_count, long long* det_track_id, int* det_row,
                        void* stream) {
  if (S < 0 || C < 1 || max_D < 0 || max_age < -1) return PCREID_ERR_ARG;
  if (S > MAX_SCENES || C > TRACK_MAX || max_D > TRACK_MAX) return PCREID_ERR_UNSUPPORTED;
  if (S == 0) return PCREID_OK;
  if (!offsets || !alive || !track_id || !label || !length || !age || !hits || !box || !next_id || !dropped || !active ||
      !active_count || (max_D > 0 && (!track_for_det || !det_label || !det_length || !det_box || !det_track_id || !det_row)))
    return PCREID_ERR_ARG;
  track_update_kernel<<<S, UPDATE_THREADS, 0, (cudaStream_t)stream>>>(
      S, C, offsets, track_for_det, det_label, det_length, det_box, max_age, replace_all, alive, track_id, label, length, age,
      hits, box, next_id, dropped, active, active_count, det_track_id, det_row);
  return pcreid_launch_status();
}

int pcreid_track_scatter(int n_det, const int* det_row, long long xyz_bytes, const void* det_xyz, void* xyz,
                         long long feat_bytes, const void* det_feat, void* feat, void* stream) {
  if (n_det < 0 || xyz_bytes < 0 || feat_bytes < 0) return PCREID_ERR_ARG;
  const long long chunks = ((xyz_bytes > feat_bytes ? xyz_bytes : feat_bytes) + SCATTER_CHUNK - 1) / SCATTER_CHUNK;
  if (chunks > 65535) return PCREID_ERR_UNSUPPORTED;
  if (n_det == 0 || chunks == 0) return PCREID_OK;
  if (!det_row || (xyz_bytes && (!det_xyz || !xyz)) || (feat_bytes && (!det_feat || !feat))) return PCREID_ERR_ARG;
  track_scatter_kernel<<<dim3(n_det, (unsigned)chunks), SCATTER_THREADS, 0, (cudaStream_t)stream>>>(
      det_row, xyz_bytes, (const unsigned char*)det_xyz, (unsigned char*)xyz, feat_bytes, (const unsigned char*)det_feat,
      (unsigned char*)feat);
  return pcreid_launch_status();
}

}  // extern "C"

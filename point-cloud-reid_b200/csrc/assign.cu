// Gated linear assignment of tracks to detections (include/pcreid.h, pcreid_lsap): one CTA per problem, a
// shortest-augmenting-path solver (Jonker-Volgenant as restated by Crouse, the family of scipy's linear_sum_assignment)
// with float64 dual potentials and reduced costs.
//
// Problem b: rows t < T (tracks), real columns d < D (detections) with cost c = tau - S[t, d] where the pair is admissible
// (mask != 0, S finite, S > tau) and +inf otherwise, plus one dummy column per row ("leave t unmatched") of cost 0 that no
// other row reaches.  The minimum-cost row-complete assignment of that T x (D + T) matrix is the maximum-weight matching
// of admissible pairs.  The dummies are implicit: a row that ends on its dummy is never reached again (no real column
// leads to it), so a dummy only ever enters a Dijkstra as a sink candidate of a row scanned in that same Dijkstra, with
// v = 0 and distance = (distance at which its row was reached) - u[row].  One running best over those replaces the
// T dummy columns.
//
// Rows are augmented in order t = 0 .. T-1.  Each Dijkstra step relaxes the current row over the remaining real columns
// (thread j % blockDim owns column j: its distance, predecessor, dual and visited flag live in shared memory and are
// touched by no other thread during a Dijkstra), then the CTA selects the next column by the lexicographic minimum of
//   (reduced distance, unassigned before assigned, column index; dummies index D + t)
// -- a total order, so the result does not depend on the thread count or on other problems in the launch.
// Row state (u, the column of each row, the columns selected in the current Dijkstra) lives in the per-problem workspace.
#include "../../include/pcreid.h"
#include "common.cuh"

#include <math_constants.h>

#include <cmath>

namespace {

constexpr int LSAP_MAX = 4096;         // T, D <= LSAP_MAX: column keys below fit in 14 bits
constexpr int KEY_ASSIGNED = 1 << 14;  // selection key = column index (+ KEY_ASSIGNED for an assigned real column)
constexpr int MAX_THREADS = 512;

struct Cand {
  double d;
  int key;
};

__device__ __forceinline__ bool before(double d, int key, const Cand& b) { return d < b.d || (d == b.d && key < b.key); }

__device__ __forceinline__ Cand warp_argmin(Cand c) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_xor_sync(FULL_MASK, c.d, o);
    const int ok = __shfl_xor_sync(FULL_MASK, c.key, o);
    if (before(od, ok, c)) { c.d = od; c.key = ok; }
  }
  return c;
}

// per-problem workspace: u (T doubles) | sel_d (min(T, D) + 1 doubles) | col4row (T ints) | sel_col (min(T, D) + 1 ints)
__host__ __device__ inline size_t lsap_work_bytes(int T, int D) {
  const size_t steps = (size_t)(T < D ? T : D) + 1;
  return (((size_t)T + steps) * 12 + 15) / 16 * 16;
}

__global__ void __launch_bounds__(MAX_THREADS) lsap_kernel(int T, int D, const float* __restrict__ score,
                                                            const unsigned char* __restrict__ mask, float tau,
                                                            int* __restrict__ det_for_track, int* __restrict__ track_for_det,
                                                            unsigned char* __restrict__ work) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int nthr = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
  const size_t b = blockIdx.x;
  Cand* red = reinterpret_cast<Cand*>(smem);                    // [2][32] per-warp candidates, double-buffered
  double* spc = reinterpret_cast<double*>(red + 64);            // [D] shortest reduced distance in this Dijkstra
  double* v = spc + D;                                          // [D] column duals
  int* path = reinterpret_cast<int*>(v + D);                    // [D] row that last lowered spc
  int* row4col = path + D;                                      // [D] row assigned to the column, -1 if none
  unsigned char* done = reinterpret_cast<unsigned char*>(row4col + D);   // [D] column selected in this Dijkstra

  const int steps = (T < D ? T : D) + 1;
  unsigned char* wb = work + b * lsap_work_bytes(T, D);
  double* u = reinterpret_cast<double*>(wb);
  double* sel_d = u + T;
  int* col4row = reinterpret_cast<int*>(sel_d + steps);         // real column, D + t for the dummy, -1 before row t is done
  int* sel_col = col4row + T;

  const float* S = score + b * (size_t)T * D;
  const unsigned char* M = mask ? mask + b * (size_t)T * D : nullptr;
  const double dtau = (double)tau;

  for (int j = tid; j < D; j += nthr) { v[j] = 0.0; row4col[j] = -1; }
  for (int t = tid; t < T; t += nthr) { u[t] = 0.0; col4row[t] = -1; }
  __syncthreads();

  int buf = 0;
  for (int cur = 0; cur < T; ++cur) {
    for (int j = tid; j < D; j += nthr) { spc[j] = CUDART_INF; done[j] = 0; }
    double min_val = 0.0;
    int i = cur, nsel = 0, sink;
    Cand dummy = {CUDART_INF, 0x7fffffff};                      // best dummy column of the rows scanned so far
    while (true) {
      const double ui = u[i];
      const float* srow = S + (size_t)i * D;
      const unsigned char* mrow = M ? M + (size_t)i * D : nullptr;
      Cand best = {CUDART_INF, 0x7fffffff};
      for (int j = tid; j < D; j += nthr) {
        if (done[j]) continue;
        const float s = __ldg(srow + j);
        const bool adm = (!mrow || __ldg(mrow + j)) && isfinite(s) && s > tau;
        double dj = spc[j];
        if (adm) {
          const double r = min_val + (dtau - (double)s) - ui - v[j];
          if (r < dj) { dj = r; spc[j] = r; path[j] = i; }
        }
        const int key = j + (row4col[j] >= 0 ? KEY_ASSIGNED : 0);
        if (before(dj, key, best)) { best.d = dj; best.key = key; }
      }
      const double dd = min_val - ui;                           // row i's own dummy column D + i
      if (before(dd, D + i, dummy)) { dummy.d = dd; dummy.key = D + i; }
      best = warp_argmin(best);
      if (lane == 0) red[buf * 32 + warp] = best;
      __syncthreads();
      best = dummy;
      for (int w = 0; w < nwarps; ++w) {
        const Cand c = red[buf * 32 + w];
        if (before(c.d, c.key, best)) best = c;
      }
      buf ^= 1;
      min_val = best.d;                                         // finite: row cur's dummy is always a candidate
      const int j = best.key & (KEY_ASSIGNED - 1);
      if (tid == 0) { sel_col[nsel] = j; sel_d[nsel] = best.d; }
      ++nsel;
      if (best.key < KEY_ASSIGNED) { sink = j; break; }         // unassigned real column or a dummy: augment
      if (tid == j % nthr) done[j] = 1;
      i = row4col[j];
    }
    // dual update: u[cur] += min_val; u[r] += min_val - spc[col4row[r]] for the other scanned rows;
    // v[j] -= min_val - spc[j] for the selected real columns (the sink's change is 0)
    for (int j = tid; j < D; j += nthr)
      if (done[j]) v[j] -= min_val - spc[j];
    if (tid == 0) {
      u[cur] += min_val;
      for (int k = 0; k + 1 < nsel; ++k) u[row4col[sel_col[k]]] += min_val - sel_d[k];
      // augment along the predecessor chain: sink .. cur
      int j = sink;
      while (true) {
        const int r = j >= D ? j - D : path[j];
        if (j < D) row4col[j] = r;
        const int prev = col4row[r];
        col4row[r] = j;
        j = prev;
        if (r == cur) break;
      }
    }
    __syncthreads();
  }

  for (int t = tid; t < T; t += nthr) det_for_track[b * T + t] = col4row[t] < D ? col4row[t] : -1;
  for (int j = tid; j < D; j += nthr) track_for_det[b * D + j] = row4col[j];
}

}  // namespace

extern "C" {

int pcreid_lsap_workspace_bytes(int T, int D) {
  if (T < 0 || D < 0 || T > LSAP_MAX || D > LSAP_MAX) return -1;
  return T == 0 ? 0 : (int)lsap_work_bytes(T, D);
}

int pcreid_lsap(int B, int T, int D, const float* score, const unsigned char* mask, float min_score, int* det_for_track,
                int* track_for_det, void* work, void* stream) {
  if (B < 0 || T < 0 || D < 0 || !std::isfinite(min_score)) return PCREID_ERR_ARG;
  if (B > 65535 || T > LSAP_MAX || D > LSAP_MAX) return PCREID_ERR_UNSUPPORTED;
  if (B == 0 || (T == 0 && D == 0)) return PCREID_OK;
  if ((T > 0 && D > 0 && !score) || (T > 0 && (!det_for_track || !work)) || (D > 0 && !track_for_det)) return PCREID_ERR_ARG;
  const int nthr = D >= MAX_THREADS ? MAX_THREADS : (D > 32 ? (D + 31) / 32 * 32 : 32);
  const size_t smem = 64 * sizeof(Cand) + (size_t)D * (2 * sizeof(double) + 2 * sizeof(int) + 1);
  if (smem > 48 * 1024) cudaFuncSetAttribute(lsap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  lsap_kernel<<<B, nthr, smem, (cudaStream_t)stream>>>(T, D, score, mask, min_score, det_for_track, track_for_det,
                                                       (unsigned char*)work);
  return pcreid_launch_status();
}

}  // extern "C"

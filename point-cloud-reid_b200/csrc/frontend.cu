// Crop -> centre -> resample front-end of the ReID encoder (SURVEY.md 8f row 2): from one LiDAR sweep and a set of boxes
// straight to the (B, N, 3) encoder input.
//
// Reference (mmdet3d/models/trackers/deprecated/pc_utils.py:31-96):
//   interpolate_per_frame: DepthInstance3DBoxes(bboxes, origin=(.5,.5,.5)).points_in_boxes(points)  -> per-box crops in
//     point order (core/bbox/structures/depth_box3d.py:256-282 -> ops/roiaware_pool3d/src/points_in_boxes_cuda.cu:24-105),
//     padded to the longest crop, times inverse(affine(Rz(-(-yaw)), centre))   -> box-frame coordinates;
//   get_input_batch: torch.randint(high=length) per box -> gather with replacement to N points, zeros for empty boxes.
// The reference materialises a (P, B) int mask, a python list of B crops, a (B, Lmax, 3) padded batch and a
// (B, Lmax, 4) homogeneous copy.  Here: one pass writes a bit mask (1 bit per (box, point)) and per-tile counts; after
// an exclusive scan of the counts the second pass turns every requested sample rank directly into a point (binary
// search over the tile prefix, select-the-r-th-set-bit inside the tile) and writes it centred.  Nothing of size
// B x Lmax exists.
//
// In-box test, arithmetic of the reference kernel after the Depth -> LiDAR change of frame that
// DepthInstance3DBoxes.points_in_boxes applies (SASS of the reference file compiled for sm_100a):
//   point (y, -x, z); box centre (by, -bx, fl(bz - dz/2)), w = dy, l = dx, h = dz
//   cz = float(double(z') + double(h) * 0.5);  reject if double(|pz - cz|) > double(h) * 0.5
//   a = float(double(yaw) + pi/2); c = cosf(a), s = sinf(a);  sx = py - by, sy = (-px) - (-bx)
//   lx = fma(sx, c, -(sy * s)), ly = fma(sy, c, sx * s);  inside iff -l/2 < lx < l/2 and -w/2 < ly < w/2  (doubles)
#include "../../include/pcreid.h"
#include "common.cuh"

namespace {

constexpr int CT = 1024;          // points per tile = 32 mask words
constexpr int BB = 32;            // boxes per CTA of the mask pass

struct BoxC {                     // per-box constants of the in-box test
  float cx, cy, cz, c, s;
  double hl, hw, hh;
};

__device__ __forceinline__ BoxC box_consts(const float* __restrict__ b) {
  BoxC k;
  const float bx = b[0], by = b[1], bz = b[2], dx = b[3], dy = b[4], dz = b[5], yaw = b[6];
  const float zb = __fadd_rn(bz, __fmul_rn(dz, -0.5f));            // centre origin -> bottom centre (base_box3d.py:61-64)
  k.cx = by;
  k.cy = -bx;
  k.hh = (double)dz * 0.5;
  k.cz = (float)((double)zb + k.hh);
  const float a = (float)((double)yaw + 1.57079632679489661923);
  k.c = cosf(a);
  k.s = sinf(a);
  k.hl = (double)dx * 0.5;
  k.hw = (double)dy * 0.5;
  return k;
}

__device__ __forceinline__ bool in_box(const BoxC& k, float px, float py, float pz) {
  const float xl = py, yl = -px;
  if ((double)fabsf(__fsub_rn(pz, k.cz)) > k.hh) return false;
  const float sx = __fsub_rn(xl, k.cx), sy = __fsub_rn(yl, k.cy);
  const float lx = __fmaf_rn(sx, k.c, -__fmul_rn(sy, k.s));
  const float ly = __fmaf_rn(sy, k.c, __fmul_rn(sx, k.s));
  return ((double)lx > -k.hl) & ((double)lx < k.hl) & ((double)ly > -k.hw) & ((double)ly < k.hw);
}

// pass 1 for one tile of one sweep and up to BB boxes b0 .. b0 + nb - 1 of that sweep:
//   mask[b][tile][32] (bit i of word w <-> point tile*1024 + 32 w + i), counts[b][tile]
__device__ __forceinline__ void crop_mask_tile(int P, int nb, int ntiles, int tile, const float* __restrict__ pts, int ps,
                                               const float* __restrict__ boxes, uint32_t* __restrict__ mask,
                                               int* __restrict__ counts) {
  __shared__ BoxC bc[BB];
  __shared__ int cnt[BB];
  if (threadIdx.x < nb) { bc[threadIdx.x] = box_consts(boxes + (size_t)threadIdx.x * 7); cnt[threadIdx.x] = 0; }
  float px[4], py[4], pz[4];
  bool live[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int p = tile * CT + j * 256 + threadIdx.x;
    live[j] = p < P;
    const float* q = pts + (size_t)(live[j] ? p : 0) * ps;
    px[j] = q[0]; py[j] = q[1]; pz[j] = q[2];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = 0; i < nb; ++i) {
    const BoxC k = bc[i];
    int c = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t w = __ballot_sync(FULL_MASK, live[j] && in_box(k, px[j], py[j], pz[j]));
      if (lane == 0) {
        mask[((size_t)i * ntiles + tile) * 32 + j * 8 + warp] = w;
        c += __popc(w);
      }
    }
    if (lane == 0 && c) atomicAdd(&cnt[i], c);
  }
  __syncthreads();
  if (threadIdx.x < nb) counts[(size_t)threadIdx.x * ntiles + tile] = cnt[threadIdx.x];
}

__global__ void __launch_bounds__(256) crop_mask_kernel(int P, int B, int ntiles, const float* __restrict__ pts, int ps,
                                                        const float* __restrict__ boxes, uint32_t* __restrict__ mask,
                                                        int* __restrict__ counts) {
  const int b0 = blockIdx.y * BB;
  crop_mask_tile(P, min(BB, B - b0), ntiles, blockIdx.x, pts, ps, boxes + (size_t)b0 * 7, mask + (size_t)b0 * ntiles * 32,
                 counts + (size_t)b0 * ntiles);
}

// segment of a prefix array holding x: the largest s with off[s] <= x (off nondecreasing, off[0] <= x < off[S])
__device__ __forceinline__ int segment_of(const int* __restrict__ off, int S, int x) {
  int lo = 0, hi = S;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= x) lo = mid; else hi = mid;
  }
  return lo;
}

// offsets of the segmented front-end (pcreid_crop_mask_scenes): off = [points | boxes | tiles | count words], each (S + 1)
struct SceneOff {
  const int *pt, *box, *tile, *cnt;
  __device__ SceneOff(const int* off, int S) : pt(off), box(off + (S + 1)), tile(off + 2 * (S + 1)), cnt(off + 3 * (S + 1)) {}
};

// one CTA per (tile of scene s, box group y of scene s): scene s's block of mask / counts is laid out as pcreid_crop_mask's for
// that sweep alone
__global__ void __launch_bounds__(256) crop_mask_scenes_kernel(int S, const float* __restrict__ pts, int ps,
                                                               const float* __restrict__ boxes, const int* __restrict__ off,
                                                               uint32_t* __restrict__ mask, int* __restrict__ counts) {
  const SceneOff o(off, S);
  const int s = segment_of(o.tile, S, blockIdx.x);
  const int B = o.box[s + 1] - o.box[s], b0 = blockIdx.y * BB;
  if (b0 >= B) return;
  const int ntiles = o.tile[s + 1] - o.tile[s];
  const size_t c0 = (size_t)o.cnt[s] + (size_t)b0 * ntiles;
  crop_mask_tile(o.pt[s + 1] - o.pt[s], min(BB, B - b0), ntiles, blockIdx.x - o.tile[s], pts + (size_t)o.pt[s] * ps, ps,
                 boxes + (size_t)(o.box[s] + b0) * 7, mask + c0 * 32, counts + c0);
}

// pass 2 for one output slot: o = Rz(yaw)-frame coordinates of the r-th in-box point of the box (zeros for an empty box)
//   pf[0..ntiles]: exclusive scan of the box's counts, mw: the box's mask words
__device__ __forceinline__ void crop_gather_one(int ntiles, const float* __restrict__ pts, int ps, const float* __restrict__ bx,
                                                const uint32_t* __restrict__ mw, const int* __restrict__ pf, long long r,
                                                float* __restrict__ o) {
  const int len = pf[ntiles];
  if (len <= 0) { o[0] = 0.f; o[1] = 0.f; o[2] = 0.f; return; }
  r = r < 0 ? 0 : (r >= len ? len - 1 : r);
  const int lo = segment_of(pf, ntiles, (int)r);  // largest tile with prefix[tile] <= r
  int rem = (int)r - pf[lo];
  mw += (size_t)lo * 32;
  int word = 0;
  uint32_t w = mw[0];
  while (rem >= __popc(w)) { rem -= __popc(w); w = mw[++word]; }     // mask words are stored as [pass j][warp]: word = 8 j + warp
  for (int i = 0; i < rem; ++i) w &= w - 1;                          // drop the rem lowest set bits
  const int bit = __ffs(w) - 1;
  const int p = lo * CT + (word >> 3) * 256 + (word & 7) * 32 + bit;
  const float* q = pts + (size_t)p * ps;
  float s, c;
  sincosf(bx[6], &s, &c);
  const float dx = q[0] - bx[0], dy = q[1] - bx[1];
  o[0] = c * dx - s * dy;                        // inverse of [Rz(-yaw) | centre] applied to the point (pc_utils.py:62-76)
  o[1] = s * dx + c * dy;
  o[2] = q[2] - bx[2];
}

// out[b][n] for rank[b][n]; prefix[b][0..ntiles] exclusive scan of counts
__global__ void __launch_bounds__(128) crop_gather_kernel(int P, int N, int ntiles, const float* __restrict__ pts, int ps,
                                                          const float* __restrict__ boxes, const uint32_t* __restrict__ mask,
                                                          const int* __restrict__ prefix, const long long* __restrict__ rank,
                                                          float* __restrict__ out) {
  const int b = blockIdx.y, n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  crop_gather_one(ntiles, pts, ps, boxes + (size_t)b * 7, mask + (size_t)b * ntiles * 32, prefix + (size_t)b * (ntiles + 1),
                  rank[(size_t)b * N + n], out + ((size_t)b * N + n) * 3);
}

// global box g of scene s (local index i): mask / counts at cnt[s] + i * ntiles_s, prefix at cnt[s] + i * ntiles_s + g
__global__ void __launch_bounds__(128) crop_gather_scenes_kernel(int S, int N, const float* __restrict__ pts, int ps,
                                                                 const float* __restrict__ boxes, const int* __restrict__ off,
                                                                 const uint32_t* __restrict__ mask,
                                                                 const int* __restrict__ prefix,
                                                                 const long long* __restrict__ rank, float* __restrict__ out) {
  const int g = blockIdx.y, n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const SceneOff o(off, S);
  const int s = segment_of(o.box, S, g);
  const int ntiles = o.tile[s + 1] - o.tile[s];
  const size_t c0 = (size_t)o.cnt[s] + (size_t)(g - o.box[s]) * ntiles;
  crop_gather_one(ntiles, pts + (size_t)o.pt[s] * ps, ps, boxes + (size_t)g * 7, mask + c0 * 32, prefix + c0 + g,
                  rank[(size_t)g * N + n], out + ((size_t)g * N + n) * 3);
}

}  // namespace

extern "C" {

int pcreid_crop_tiles(int P) { return (P + CT - 1) / CT; }

int pcreid_crop_mask(int P, int B, const float* pts, int pts_stride, const float* boxes, void* mask, int* counts, void* stream) {
  if (B <= 0 || P <= 0) return PCREID_OK;
  if (!pts || !boxes || !mask || !counts || pts_stride < 3) return PCREID_ERR_ARG;
  const int ntiles = (P + CT - 1) / CT;
  if ((B + BB - 1) / BB > 65535) return PCREID_ERR_UNSUPPORTED;
  crop_mask_kernel<<<dim3(ntiles, (B + BB - 1) / BB), 256, 0, (cudaStream_t)stream>>>(P, B, ntiles, pts, pts_stride, boxes,
                                                                                     (uint32_t*)mask, counts);
  return pcreid_launch_status();
}

int pcreid_crop_gather(int P, int B, int N, const float* pts, int pts_stride, const float* boxes, const void* mask,
                       const int* prefix, const long long* rank, float* out, void* stream) {
  if (B <= 0 || N <= 0) return PCREID_OK;
  if (!pts || !boxes || !mask || !prefix || !rank || !out || pts_stride < 3 || P <= 0) return PCREID_ERR_ARG;
  if (B > 65535) return PCREID_ERR_UNSUPPORTED;
  const int ntiles = (P + CT - 1) / CT;
  crop_gather_kernel<<<dim3((N + 127) / 128, B), 128, 0, (cudaStream_t)stream>>>(P, N, ntiles, pts, pts_stride, boxes,
                                                                                 (const uint32_t*)mask, prefix, rank, out);
  return pcreid_launch_status();
}

int pcreid_crop_mask_scenes(int S, int total_tiles, int max_boxes, const float* pts, int pts_stride, const float* boxes,
                            const int* offsets, void* mask, int* counts, void* stream) {
  if (S < 0 || total_tiles < 0 || max_boxes < 0) return PCREID_ERR_ARG;
  if (S == 0 || total_tiles == 0 || max_boxes == 0) return PCREID_OK;
  if (!pts || !boxes || !offsets || !mask || !counts || pts_stride < 3) return PCREID_ERR_ARG;
  if ((max_boxes + BB - 1) / BB > 65535) return PCREID_ERR_UNSUPPORTED;
  crop_mask_scenes_kernel<<<dim3(total_tiles, (max_boxes + BB - 1) / BB), 256, 0, (cudaStream_t)stream>>>(
      S, pts, pts_stride, boxes, offsets, (uint32_t*)mask, counts);
  return pcreid_launch_status();
}

int pcreid_crop_gather_scenes(int S, int total_boxes, int N, const float* pts, int pts_stride, const float* boxes,
                              const int* offsets, const void* mask, const int* prefix, const long long* rank, float* out,
                              void* stream) {
  if (S < 0 || total_boxes < 0 || N < 0) return PCREID_ERR_ARG;
  if (S == 0 || total_boxes == 0 || N == 0) return PCREID_OK;
  if (!boxes || !offsets || !prefix || !rank || !out || pts_stride < 3) return PCREID_ERR_ARG;
  if (total_boxes > 65535) return PCREID_ERR_UNSUPPORTED;
  crop_gather_scenes_kernel<<<dim3((N + 127) / 128, total_boxes), 128, 0, (cudaStream_t)stream>>>(
      S, N, pts, pts_stride, boxes, offsets, (const uint32_t*)mask, prefix, rank, out);
  return pcreid_launch_status();
}

}  // extern "C"

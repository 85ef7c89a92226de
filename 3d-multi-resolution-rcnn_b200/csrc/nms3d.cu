// 3D IoU NMS for B200 (sm_100a), batched over independent segments, entirely on the device.
//
// Replaces (reference, /root/reference): nms_cuda_3d + nms_kernel_3d + devIoU3d,
//   mmdet/ops/nms/src/nms_kernel.cu:196-257, :81-129, :23-33, reached through
//   mmdet/ops/nms/nms_wrapper.py:42-44 from rpn_head_3d.py:134 and bbox_nms.py:89.
//
// The reference sorts with ATen, computes the FULL N x N/64 bit matrix with 64-thread blocks, copies it
// to the host with a blocking cudaMemcpy, sweeps it on the CPU and copies the result back.  Here:
//   1. rank kernel     -- stable descending order by counting (score desc, index asc; O(n^2) compares,
//                         embarrassingly parallel, n <= a few thousand) and gather of the boxes into
//                         sorted 32-byte records that also carry the per-box volume factors;
//   2. mask kernel     -- upper-triangular 64x64 tiles only, column boxes staged in shared memory,
//                         one uint64 word per (row, column-tile);
//   3. sweep kernel    -- one CTA per segment walks the 64-box diagonal tiles as a pipeline: warp 0 resolves
//                         tile b with a warp-parallel fixed-point iteration (lanes hold the diagonal rows; K <- cand &
//                         ~OR{row_j : j in K} until K repeats: exactly the sequential sweep's set) and updates the
//                         next tile's `removed` word itself, while warps 1..7 apply tile b-1 to the later words and
//                         stage the mask rows of the tiles ahead through registers (coalesced loads, four tiles
//                         deep); the kept set is then compacted position-parallel twice (descending score, and
//                         ascending original index).
// No host synchronisation, no D2H copy; many (volume, level, class) segments share the three launches.
//
// Bit-exactness: IoU uses explicit _rn intrinsics in exactly the operation order of the compiled
// reference (SASS: interS and Sa plain FMULs, union = FFMA(bw*bh, bd, Sa) - interS, IEEE division,
// strict '>' against the threshold).
#include "common.cuh"

namespace roi3d {

struct __align__(16) SortedBox {
  float x1, y1, x2, y2, z1, z2;
  float sxy;  // (x2-x1+1)*(y2-y1+1)
  float sz;   // (z2-z1+1)
};

__device__ __forceinline__ unsigned score_key(float s) {
  s = s + 0.0f;  // -0 -> +0 so that +-0 tie like torch's comparison does
  unsigned u = __float_as_uint(s);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// devIoU3d(a = row box, b = column box) > thr, compiled-reference arithmetic.
__device__ __forceinline__ bool iou3d_gt(const SortedBox &a, float Sa, const SortedBox &b, float thr) {
  const float left = fmaxf(a.x1, b.x1), right = fminf(a.x2, b.x2);
  const float top = fmaxf(a.y1, b.y1), bottom = fminf(a.y2, b.y2);
  const float front = fmaxf(a.z1, b.z1), back = fminf(a.z2, b.z2);
  const float w = fmaxf(__fadd_rn(__fsub_rn(right, left), 1.0f), 0.0f);
  const float h = fmaxf(__fadd_rn(__fsub_rn(bottom, top), 1.0f), 0.0f);
  const float d = fmaxf(__fadd_rn(__fsub_rn(back, front), 1.0f), 0.0f);
  const float inter = __fmul_rn(__fmul_rn(w, h), d);
  const float uni = __fsub_rn(__fmaf_rn(b.sxy, b.sz, Sa), inter);
  // disjoint boxes (most pairs): 0 / positive union = +0, no need for the IEEE division
  if (inter == 0.0f && uni > 0.0f) return 0.0f > thr;
  return __fdiv_rn(inter, uni) > thr;
}

// ------------------------------------------------------------------------------------------------
// Coarse rejection for the bit-matrix kernels.  Most pairs of a proposal set are far apart, yet a lane spends ~25
// instructions to find inter == 0.  Every CTA therefore lays a 32 x 32 x 32 grid over the bounding range of ITS row and
// column boxes and gives each box three 32-bit masks (the cells its [lo - 1, hi + 1] interval covers per axis); a pair
// whose masks miss each other on any axis has inter == 0 exactly as the reference computes it, and for thr >= 0 the
// reference's answer to inter == 0 is "no" whatever the union is (0 / u is +-0 or NaN):
//   * the cell of a coordinate is a non-decreasing function of it (float subtract / multiply by a non-negative
//     constant / float -> int conversion, clamped), so disjoint cell ranges mean fl(a.hi + 1) < fl(b.lo - 1), hence
//     a.hi + 1 < b.lo - 1, hence min(hi) - max(lo) < -2, hence fl(fl(min(hi) - max(lo)) + 1) <= -1: the reference's
//     clamped extent is 0 on that axis (a box stored inverted by more than the margin gets an empty mask: it
//     intersects nothing in the reference either);
//   * a box with a NaN / infinite coordinate, a degenerate range, or thr < 0 (where inter == 0 can still suppress)
//     gets all-ones masks and the pair is evaluated in full.
// Pairs that pass are evaluated exactly as before, so the bit matrix is unchanged.
// ------------------------------------------------------------------------------------------------
struct CellMap {
  float lo[3], inv[3];
  int on;
};

__device__ __forceinline__ unsigned cell_range(float lo, float hi, float origin, float inv) {
  const int c0 = min(max(__float2int_rd(__fmul_rn(__fsub_rn(__fsub_rn(lo, 1.0f), origin), inv)), 0), 31);
  const int c1 = min(max(__float2int_rd(__fmul_rn(__fsub_rn(__fadd_rn(hi, 1.0f), origin), inv)), 0), 31);
  return ((2u << c1) - 1u) & ~((1u << c0) - 1u);
}

__device__ __forceinline__ uint4 box_cells(const SortedBox &b, const CellMap &m) {
  const float s = b.x1 + b.y1 + b.x2 + b.y2 + b.z1 + b.z2;
  if (!m.on || !(fabsf(s) <= 3.0e38f)) return make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u);
  return make_uint4(cell_range(b.x1, b.x2, m.lo[0], m.inv[0]), cell_range(b.y1, b.y2, m.lo[1], m.inv[1]),
                    cell_range(b.z1, b.z2, m.lo[2], m.inv[2]), 0u);
}

__device__ __forceinline__ bool cells_meet(const uint4 &a, const uint4 &b) {
  return ((a.x & b.x) != 0u) & ((a.y & b.y) != 0u) & ((a.z & b.z) != 0u);
}

// Bounding range of the boxes the CTA's threads hold (has_box: this thread contributes `b`), 256 threads.  Ends with
// a barrier; the result is in shared memory.
__device__ __forceinline__ void cta_cell_map(const SortedBox &b, bool has_box, bool enabled, CellMap *out) {
  __shared__ float red[8][6];
  const float inf = __int_as_float(0x7f800000);
  float v[6] = {inf, inf, inf, -inf, -inf, -inf};
  if (has_box) {
    v[0] = fminf(b.x1, b.x2), v[1] = fminf(b.y1, b.y2), v[2] = fminf(b.z1, b.z2);
    v[3] = fmaxf(b.x1, b.x2), v[4] = fmaxf(b.y1, b.y2), v[5] = fmaxf(b.z1, b.z2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      v[c] = fminf(v[c], __shfl_xor_sync(0xffffffffu, v[c], o));
      v[c + 3] = fmaxf(v[c + 3], __shfl_xor_sync(0xffffffffu, v[c + 3], o));
    }
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int c = 0; c < 6; ++c) red[threadIdx.x >> 5][c] = v[c];
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    const int c = threadIdx.x;
    float lo = red[0][c], hi = red[0][c + 3];
#pragma unroll
    for (int w = 1; w < 8; ++w) lo = fminf(lo, red[w][c]), hi = fmaxf(hi, red[w][c + 3]);
    lo -= 1.0f, hi += 1.0f;   // the masks cover [lo - 1, hi + 1] of every box
    const float range = hi - lo;
    const bool ok = range > 0.0f && range <= 3.0e38f && fabsf(lo) <= 3.0e38f;
    out->lo[c] = ok ? lo : 0.0f;
    out->inv[c] = ok ? 32.0f / range : 0.0f;
    if (c == 0) out->on = enabled ? 1 : 0;
  }
  __syncthreads();
}

// Evaluation-time flavour (N1): the reference's numpy nms_3d_python (mmdet/core/evaluation/coco_utils.py:245-282)
// works in float64 on the json boxes (fp32 values widened), volume = ((x2-x1+1)*(y2-y1+1))*(z2-z1+1), iou =
// inter / ((vol_i + vol_j) - inter), and KEEPS iou <= thr -- so a NaN iou suppresses.  Same operation order,
// no contraction (explicit _rn double intrinsics).
__device__ __forceinline__ bool iou3d_f64_suppresses(const SortedBox &a, const SortedBox &b, double thr) {
  const double ax1 = a.x1, ay1 = a.y1, ax2 = a.x2, ay2 = a.y2, az1 = a.z1, az2 = a.z2;
  const double bx1 = b.x1, by1 = b.y1, bx2 = b.x2, by2 = b.y2, bz1 = b.z1, bz2 = b.z2;
  const double va = __dmul_rn(__dmul_rn(__dadd_rn(__dsub_rn(ax2, ax1), 1.0), __dadd_rn(__dsub_rn(ay2, ay1), 1.0)),
                              __dadd_rn(__dsub_rn(az2, az1), 1.0));
  const double vb = __dmul_rn(__dmul_rn(__dadd_rn(__dsub_rn(bx2, bx1), 1.0), __dadd_rn(__dsub_rn(by2, by1), 1.0)),
                              __dadd_rn(__dsub_rn(bz2, bz1), 1.0));
  // np.maximum / np.minimum propagate NaN; fmax / fmin do not -- a NaN coordinate must poison the iou
  const bool nan_in = !(ax1 == ax1 && ay1 == ay1 && ax2 == ax2 && ay2 == ay2 && az1 == az1 && az2 == az2 && bx1 == bx1 &&
                        by1 == by1 && bx2 == bx2 && by2 == by2 && bz1 == bz1 && bz2 == bz2);
  const double w = fmax(0.0, __dadd_rn(__dsub_rn(fmin(ax2, bx2), fmax(ax1, bx1)), 1.0));
  const double h = fmax(0.0, __dadd_rn(__dsub_rn(fmin(ay2, by2), fmax(ay1, by1)), 1.0));
  const double d = fmax(0.0, __dadd_rn(__dsub_rn(fmin(az2, bz2), fmax(az1, bz1)), 1.0));
  const double inter = __dmul_rn(__dmul_rn(w, h), d);
  const double uni = __dsub_rn(__dadd_rn(va, vb), inter);
  if (inter == 0.0 && uni > 0.0) return nan_in || !(0.0 <= thr);  // disjoint: iou is +0, skip the division
  const double iou = __ddiv_rn(inter, uni);
  return nan_in || !(iou <= thr);
}

// ------------------------------------------------------------------------------------------------
// 1. rank + gather.  grid (ceil(n_max/32), nseg), block 256 = 32 boxes x 8 slices of the j range
//    (each warp scans one slice with warp-uniform loads; partial ranks are summed through smem).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nms3d_rank_kernel(const float *__restrict__ dets, const int32_t *seg_counts,
                                                         const unsigned char *__restrict__ presorted, int n_max,
                                                         SortedBox *__restrict__ sorted, int32_t *__restrict__ order) {
  const int seg = blockIdx.y;
  const int n = seg_counts ? min(max(seg_counts[seg], 0), n_max) : n_max;
  if ((int)(blockIdx.x * 32) >= n) return;
  // the caller vouches that this segment's rows already are in (score descending, index ascending) order -- e.g.
  // rows straight out of the segmented top-k: rank = row, only the sorted records are built
  const bool identity = presorted != nullptr && presorted[seg] != 0;
  const float *d = dets + (long long)seg * n_max * 7;
  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  const unsigned ki = i < n ? score_key(__ldg(d + (long long)i * 7 + 6)) : 0u;
  // keys are staged through shared memory in tiles: one coalesced-ish gather with every load in flight at once
  // (the scores sit 28 bytes apart), then warp-uniform broadcast reads; slice s of each tile is scanned by warp s.
  constexpr int kTile = 2048;
  __shared__ unsigned keys[kTile];
  int rank = 0;
  for (int t0 = 0; t0 < (identity ? 0 : n); t0 += kTile) {
    const int tn = min(kTile, n - t0);
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kTile / 256; ++q) {
      const int j = q * 256 + threadIdx.x;
      if (j < tn) keys[j] = score_key(__ldg(d + (long long)(t0 + j) * 7 + 6));
    }
    __syncthreads();
    const int per = (tn + 7) >> 3;
    const int j0 = slice * per, j1 = min(tn, j0 + per);
#pragma unroll 8
    for (int j = j0; j < j1; ++j) {
      const unsigned kj = keys[j];
      rank += (kj > ki) || (kj == ki && (t0 + j) < i);
    }
  }
  __shared__ int part[8][32];
  part[slice][lane] = rank;
  __syncthreads();
  if (slice == 0 && i < n) {
    rank = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) rank += part[q][lane];
    if (identity) rank = i;
    const float *b = d + (long long)i * 7;
    SortedBox sb;
    sb.x1 = b[0], sb.y1 = b[1], sb.x2 = b[2], sb.y2 = b[3], sb.z1 = b[4], sb.z2 = b[5];
    sb.sxy = __fmul_rn(__fadd_rn(__fsub_rn(sb.x2, sb.x1), 1.0f), __fadd_rn(__fsub_rn(sb.y2, sb.y1), 1.0f));
    sb.sz = __fadd_rn(__fsub_rn(sb.z2, sb.z1), 1.0f);
    sorted[(long long)seg * n_max + rank] = sb;
    order[(long long)seg * n_max + rank] = i;
  }
}

// ------------------------------------------------------------------------------------------------
// 2. suppression bit matrix, upper triangle.  grid (ceil(cb/4), cb, nseg), block 256 =
//    64 rows x 4 column tiles.  mask[seg][row][cbm] (cbm = ceil(n_max/64)).
// ------------------------------------------------------------------------------------------------
template <bool F64>
__global__ void __launch_bounds__(256) nms3d_mask_kernel(const SortedBox *__restrict__ sorted,
                                                         const int32_t *seg_counts, int n_max, float thr, double thr64,
                                                         unsigned long long *__restrict__ mask) {
  const int seg = blockIdx.z;
  const int n = seg_counts ? min(max(seg_counts[seg], 0), n_max) : n_max;
  const int cb = (n + 63) >> 6, cbm = (n_max + 63) >> 6;
  const int rb = blockIdx.y;
  const int c0 = blockIdx.x * 4;
  if (rb >= cb || c0 >= cb || c0 + 3 < rb) return;
  const SortedBox *sb = sorted + (long long)seg * n_max;
  __shared__ SortedBox cols[4][64];
  __shared__ uint4 colm[4][64];
  __shared__ CellMap cmap;
  const int rl = threadIdx.x & 63, cq = threadIdx.x >> 6;
  const int cblk = c0 + cq;
  const int row = rb * 64 + rl;
  SortedBox a = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, cbox = a;
  const int jc = cblk * 64 + rl;
  if (jc < n) cbox = sb[jc], cols[cq][rl] = cbox;
  if (row < n) a = sb[row];
  {
    // bounding range over the CTA's 64 rows and up to 256 columns: a thread folds its column and (cq == 0) its row
    SortedBox u = cbox;
    const bool hc = jc < n, hr = cq == 0 && row < n;
    if (hc && hr) {
      u.x1 = fminf(fminf(cbox.x1, cbox.x2), fminf(a.x1, a.x2)), u.x2 = fmaxf(fmaxf(cbox.x1, cbox.x2), fmaxf(a.x1, a.x2));
      u.y1 = fminf(fminf(cbox.y1, cbox.y2), fminf(a.y1, a.y2)), u.y2 = fmaxf(fmaxf(cbox.y1, cbox.y2), fmaxf(a.y1, a.y2));
      u.z1 = fminf(fminf(cbox.z1, cbox.z2), fminf(a.z1, a.z2)), u.z2 = fmaxf(fmaxf(cbox.z1, cbox.z2), fmaxf(a.z1, a.z2));
    } else if (hr) {
      u = a;
    }
    cta_cell_map(u, hc || hr, F64 ? (0.0 <= thr64) : (thr >= 0.0f), &cmap);
  }
  if (jc < n) colm[cq][rl] = box_cells(cbox, cmap);
  __syncthreads();
  if (cblk < rb || cblk >= cb || row >= n) return;
  const uint4 am = box_cells(a, cmap);
  const float Sa = __fmul_rn(a.sxy, a.sz);
  const int csize = min(64, n - cblk * 64);
  const int start = (cblk == rb) ? rl + 1 : 0;
  // coarse pass over the tile's 64 columns at compile-time bit positions (a handful of logic instructions per pair),
  // then the full test only for this lane's own survivors: a warp pays for the longest survivor list among its lanes,
  // not for every column that ANY lane cannot rule out
  unsigned plo = 0, phi = 0;
#pragma unroll
  for (int u = 0; u < 32; ++u) {
    if (cells_meet(am, colm[cq][u])) plo |= 1u << u;
    if (cells_meet(am, colm[cq][32 + u])) phi |= 1u << u;
  }
  unsigned long long pm = ((unsigned long long)phi << 32) | plo;
  if (start > 0) pm = start < 64 ? pm & ~((1ULL << start) - 1ULL) : 0ULL;
  if (csize < 64) pm &= (1ULL << csize) - 1ULL;
  unsigned long long t = 0;
  while (pm) {
    const int j = __ffsll((long long)pm) - 1;
    pm &= pm - 1ULL;
    if (F64 ? iou3d_f64_suppresses(a, cols[cq][j], thr64) : iou3d_gt(a, Sa, cols[cq][j], thr)) t |= 1ULL << j;
  }
  mask[((long long)seg * n_max + row) * cbm + cblk] = t;
}

// Same bit matrix with four times the parallelism, for few / small segments (n = 2000 alone fills only an eighth
// of the GPU with the kernel above): one CTA per 64 x 64 tile, thread = (row, quarter of the tile's columns), the
// four 16-bit partial words of a row are merged through shared memory.  grid (cb, cb, nseg).
template <bool F64>
__global__ void __launch_bounds__(256) nms3d_mask_q_kernel(const SortedBox *__restrict__ sorted,
                                                           const int32_t *seg_counts, int n_max, float thr, double thr64,
                                                           unsigned long long *__restrict__ mask) {
  const int seg = blockIdx.z;
  const int n = seg_counts ? min(max(seg_counts[seg], 0), n_max) : n_max;
  const int cb = (n + 63) >> 6, cbm = (n_max + 63) >> 6;
  const int rb = blockIdx.y, cblk = blockIdx.x;
  if (rb >= cb || cblk >= cb || cblk < rb) return;
  const SortedBox *sb = sorted + (long long)seg * n_max;
  __shared__ SortedBox cols[64];
  __shared__ uint4 colm[64];
  __shared__ CellMap cmap;
  __shared__ unsigned part[4][64];
  const int rl = threadIdx.x & 63, q = threadIdx.x >> 6;
  const int row = rb * 64 + rl;
  SortedBox a = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, cbox = a;
  const int jc = cblk * 64 + rl;
  const bool hc = q == 0 && jc < n, hr = q == 1 && row < n;   // quarter 0 folds the columns, quarter 1 the rows
  if (q == 0 && jc < n) cbox = sb[jc], cols[rl] = cbox;
  if (row < n) a = sb[row];
  cta_cell_map(hc ? cbox : a, hc || hr, F64 ? (0.0 <= thr64) : (thr >= 0.0f), &cmap);
  if (hc) colm[rl] = box_cells(cbox, cmap);
  __syncthreads();
  unsigned t = 0;
  if (row < n) {
    const uint4 am = box_cells(a, cmap);
    const float Sa = __fmul_rn(a.sxy, a.sz);
    const int csize = min(64, n - cblk * 64);
    const int j0 = max(q * 16, (cblk == rb) ? rl + 1 : 0), j1 = min(q * 16 + 16, csize);
    const uint4 *mq16 = colm + q * 16;   // coarse pass at compile-time bit positions, full test for the survivors
    unsigned pm = 0;                     // (see nms3d_mask_kernel)
#pragma unroll
    for (int u = 0; u < 16; ++u)
      if (cells_meet(am, mq16[u])) pm |= 1u << u;
    const int l0 = j0 - q * 16, l1 = j1 - q * 16;   // valid local columns [l0, l1)
    pm = l1 > l0 ? pm & ((1u << l1) - 1u) & ~((1u << l0) - 1u) : 0u;
    while (pm) {
      const int u = __ffs(pm) - 1;
      pm &= pm - 1u;
      if (F64 ? iou3d_f64_suppresses(a, cols[q * 16 + u], thr64) : iou3d_gt(a, Sa, cols[q * 16 + u], thr)) t |= 1u << u;
    }
  }
  part[q][rl] = t;
  __syncthreads();
  if (q == 0 && row < n) {
    const unsigned long long w = (unsigned long long)part[0][rl] | ((unsigned long long)part[1][rl] << 16) |
                                 ((unsigned long long)part[2][rl] << 32) | ((unsigned long long)part[3][rl] << 48);
    mask[((long long)seg * n_max + row) * cbm + cblk] = w;
  }
}

// ------------------------------------------------------------------------------------------------
// 3. greedy sweep + compaction.  One CTA (256 threads) per segment.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxColBlocks = 512;   // n_max <= 32768 (static shared memory budget)
constexpr int kPanelW = 32;           // words of each mask row held in shared memory per diagonal tile
constexpr int kPanelBufs = 4;         // tile b-1 (apply), b (resolve), b+1 (landed), b+2 (in flight)

__global__ void __launch_bounds__(256) nms3d_sweep_kernel(const unsigned long long *__restrict__ mask,
                                                          const int32_t *__restrict__ order,
                                                          const int32_t *seg_counts, int n_max,
                                                          unsigned char *__restrict__ flags,
                                                          int64_t *__restrict__ keep,
                                                          int64_t *__restrict__ keep_by_score,
                                                          int32_t *__restrict__ num_keep,
                                                          const unsigned char *__restrict__ limited, int max_keep) {
  const int seg = blockIdx.x;
  // optional early stop (the proposal path only uses the first nms_post kept boxes of a score-sorted level): once
  // `limit` boxes are kept the remaining tiles are not swept; the lists then hold a prefix of the full result
  const int limit = (max_keep > 0 && limited != nullptr && limited[seg] != 0) ? max_keep : 0x7fffffff;
  __shared__ int s_kept[2];   // running kept count after tile b, in entry b & 1 (the resolver is a tile ahead of the readers)
  int kept_total = 0;
  const int n = seg_counts ? min(max(seg_counts[seg], 0), n_max) : n_max;
  const int cb = (n + 63) >> 6, cbm = (n_max + 63) >> 6;
  const unsigned long long *m = mask + (long long)seg * n_max * cbm;
  const int32_t *ord = order + (long long)seg * n_max;
  int64_t *kp = keep + (long long)seg * n_max;
  int64_t *kps = keep_by_score ? keep_by_score + (long long)seg * n_max : nullptr;
  const int tid = threadIdx.x;

  __shared__ unsigned long long remv[kMaxColBlocks];
  __shared__ unsigned long long keptw[kMaxColBlocks];
  extern __shared__ __align__(16) unsigned long long panel_dyn[];  // [kPanelBufs][64][kPanelW]
  // row stride kPanelW + 1 words: lanes = words (helpers' stores) and lanes = rows (resolver, apply) are both conflict-free
  auto panel = [&](int buf, int row, int w) -> unsigned long long & {
    return panel_dyn[((size_t)buf * 64 + row) * (kPanelW + 1) + w];
  };
  __shared__ int s_warp[8];

  for (int i = tid; i < cb; i += 256) remv[i] = 0ULL;
  for (int i = tid; i < cb; i += 256) keptw[i] = 0ULL;

  // Pipeline over the 64-box diagonal tiles, one __syncthreads per tile:
  //   warp 0 (resolver)   resolves tile b from panel[b%4]: lane l holds diagonal rows l and l + 32 (the bits above the
  //                       row's own index) and the warp iterates  K <- cand & ~OR{row_j : j in K}  from K = cand (the
  //                       boxes not yet removed) until K repeats.  Bit i of K is final after i rounds (it depends on
  //                       the bits below it only) and a repeated K satisfies the greedy recurrence, whose solution is
  //                       unique -- so the result is exactly the sequential sweep's, in about twice the depth of the
  //                       longest suppression chain (a few rounds of two warp-wide ORs) instead of 64 dependent steps.
  //                       The warp then ORs the kept rows into word b+1 itself, so the next tile's state is complete
  //                       without waiting for anyone;
  //   warps 1..7 (helpers) meanwhile apply tile b-1's kept rows (panel[(b-1)%4]) to the words >= b+1 and move the mask
  //                       rows of the tiles ahead (words [t, t+kPanelW) of tile t's 64 rows; they do not depend on the
  //                       sweep state) through registers: loaded in iteration t-6 (coalesced 8-byte loads, a row per
  //                       warp instruction; four register sets take turns), stored to panel[t%4] in iteration t-2.  (8-byte cp.async was the helpers'
  //                       critical path: the LSU retires about one cp.async lane per clock.)
  const int warp = tid >> 5, lane = tid & 31;
  // helper warp g moves rows g, g + 7, ... of a tile (lane = word of the panel: one coalesced 256-byte row per load)
  constexpr int kHelperLoads = (64 + 6) / 7;
  static_assert(kPanelW == 32, "helper lanes are the panel's words");
  const int hg = warp - 1;
  const long long tile_step = 64LL * cbm + 1;                      // words from a tile's panel origin to the next tile's
  const unsigned long long *hbase = m + (long long)hg * cbm + lane;   // row hg of tile 0, word `lane`
  unsigned long long stage0[kHelperLoads], stage1[kHelperLoads], stage2[kHelperLoads], stage3[kHelperLoads];   // tiles blk+2 .. blk+5 on their way to the panel
  auto load_tile = [&](int blk, unsigned long long (&stage)[kHelperLoads]) {   // helpers only
    const bool on = blk < cb && lane < cb - blk;
    const unsigned long long *src = hbase + blk * tile_step;
    const int row_lim = min(64, n - blk * 64) - hg;   // rows hg + 7 q below this exist
#pragma unroll
    for (int q = 0; q < kHelperLoads; ++q) {
      stage[q] = (on && 7 * q < row_lim) ? __ldcg(src) : 0ULL;
      src += 7 * cbm;
    }
  };
  auto store_tile = [&](int blk, const unsigned long long (&stage)[kHelperLoads]) {
    unsigned long long *dst = &panel(blk % kPanelBufs, hg, lane);
#pragma unroll
    for (int q = 0; q < kHelperLoads; ++q)
      if (hg + 7 * q < 64) dst[q * 7 * (kPanelW + 1)] = stage[q];
  };
  if (warp > 0) {
    load_tile(0, stage0), load_tile(1, stage1);
    store_tile(0, stage0), store_tile(1, stage1);
    load_tile(2, stage0), load_tile(3, stage1), load_tile(4, stage2), load_tile(5, stage3);   // stored in iterations 0..3
  }
  __syncthreads();

  unsigned long long nd0 = 0ULL, nd1 = 0ULL;
  if (warp == 0) nd0 = panel(0, lane, 0), nd1 = panel(0, lane + 32, 0);
  auto sweep_tile = [&](int blk, unsigned long long (&stage)[kHelperLoads]) {
    if (warp == 0) {
      const int buf = blk % kPanelBufs;
      const int bs = min(64, n - blk * 64);
      // this tile's diagonal rows were fetched at the end of the previous iteration
      const unsigned long long d0 = nd0 & ~((2ULL << lane) - 1ULL);                               // bits above the row's own index
      const unsigned long long d1 = lane == 31 ? 0ULL : nd1 & ~((2ULL << (lane + 32)) - 1ULL);
      unsigned long long r0 = remv[blk];
      if (bs < 64) r0 |= ~0ULL << bs;  // rows past n never count as kept
      const unsigned long long cand = ~r0;
      unsigned long long kept = cand;
#pragma unroll 1
      for (int it = 0; it < 64; ++it) {
        unsigned long long v = 0ULL;
        if ((kept >> lane) & 1ULL) v |= d0;
        if ((kept >> (lane + 32)) & 1ULL) v |= d1;
        v &= cand;
        unsigned long long next = cand;
        if (__any_sync(0xffffffffu, v != 0ULL)) {   // (a vote is much cheaper than the two warp-wide ORs)
          const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v);
          const unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
          next = cand & ~(((unsigned long long)hi << 32) | lo);
        }
        if (next == kept) break;
        kept = next;
      }
      kept_total += __popcll(kept);
      if (lane == 0) keptw[blk] = kept, s_kept[blk & 1] = kept_total;
      if (blk + 1 < cb) {
        // word blk+1: lanes take rows lane and lane+32, OR-reduce across the warp
        unsigned long long v = 0ULL;
        if ((kept >> lane) & 1ULL) v |= panel(buf, lane, 1);
        if ((kept >> (lane + 32)) & 1ULL) v |= panel(buf, lane + 32, 1);
        const int nbuf = (blk + 1) % kPanelBufs;   // the next tile's diagonal rows (landed an iteration ago)
        nd0 = panel(nbuf, lane, 0), nd1 = panel(nbuf, lane + 32, 0);
        if (__any_sync(0xffffffffu, v != 0ULL)) {
          const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v);
          const unsigned hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
          if (lane == 0) {
            unsigned *dst = reinterpret_cast<unsigned *>(&remv[blk + 1]);
            if (lo) atomicOr(dst, lo);
            if (hi) atomicOr(dst + 1, hi);
          }
        }
      }
    } else {
      // helpers: park the rows loaded last iteration, request the next tile's, then finish tile blk-1 (words >= blk+1)
      store_tile(blk + 2, stage);
      load_tile(blk + 6, stage);
      if (blk >= 1) {
        const int pb = blk - 1, buf = pb % kPanelBufs;
        const unsigned long long kept = keptw[pb];
        const int nw = cb - pb - 1;              // words after the diagonal of tile pb
        const int nwp = min(kPanelW - 1, nw);    // of which the panel holds nwp (w = 1..nwp)
        // panel words w = 2..nwp (w = 1 was applied by the resolver): lane = word, helper warp g ORs the kept rows among
        // its rows g * 10 .. g * 10 + 9 (the row test is warp-uniform) and merges with native 32-bit shared atomics
        const int ht = tid - 32;                 // 0..223
        const int w = 2 + lane;
        if (w <= nwp) {
          unsigned long long v = 0ULL;
          const int r0 = hg * 10;
          const unsigned rows = (unsigned)(kept >> r0) & (r0 + 10 <= 64 ? 0x3ffu : 0xfu);
          const unsigned long long *pp = &panel(buf, r0, w);
#pragma unroll
          for (int r = 0; r < 10; ++r)
            if (rows & (1u << r)) v |= pp[r * (kPanelW + 1)];
          unsigned *dst = reinterpret_cast<unsigned *>(&remv[pb + w]);
          if ((unsigned)v) atomicOr(dst, (unsigned)v);
          if ((unsigned)(v >> 32)) atomicOr(dst + 1, (unsigned)(v >> 32));
        }
        // words beyond the panel (only when n > 64*kPanelW): straight from global memory
        for (int idx = ht; idx < (nw - nwp) * 64; idx += 224) {
          const int i = idx / (nw - nwp), ww = pb + 1 + nwp + idx % (nw - nwp);
          if ((kept >> i) & 1ULL) {
            const unsigned long long v = m[((long long)pb * 64 + i) * cbm + ww];
            if (v) atomicOr(&remv[ww], v);
          }
        }
      }
    }
    __syncthreads();
  };
  for (int blk = 0; blk < cb; blk += 4) {   // four register sets take turns: a tile's rows have four iterations to arrive
    sweep_tile(blk, stage0);                 // (two were not enough: an L2 round trip is longer than two iterations)
    if (s_kept[blk & 1] >= limit) break;     // (read behind the tile's barrier; uniform over the CTA)
    if (blk + 1 < cb) {
      sweep_tile(blk + 1, stage1);
      if (s_kept[(blk + 1) & 1] >= limit) break;
    }
    if (blk + 2 < cb) {
      sweep_tile(blk + 2, stage2);
      if (s_kept[(blk + 2) & 1] >= limit) break;
    }
    if (blk + 3 < cb) {
      sweep_tile(blk + 3, stage3);
      if (s_kept[(blk + 3) & 1] >= limit) break;
    }
  }
  // the last tile's kept rows have no later words to update; nothing left to apply

  // ---- kept set -> (a) descending-score list, (b) ascending original index ----
  // Everything below is position-parallel: no per-thread serial chains of dependent global loads.
  __shared__ int excl[kMaxColBlocks];           // exclusive prefix of popc(keptw)
  __shared__ unsigned bitmap[kMaxColBlocks * 2];  // kept flags by ORIGINAL index
  __shared__ int excl_idx[kMaxColBlocks * 2];     // exclusive prefix of popc(bitmap)
  __shared__ int s_total;
  // (1) block scan of the per-word kept counts (cb <= 512: two words per thread)
  {
    const int w0 = tid * 2;
    const int c0 = w0 < cb ? __popcll(keptw[w0]) : 0;
    const int c1 = w0 + 1 < cb ? __popcll(keptw[w0 + 1]) : 0;
    int incl = c0 + c1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int woff = 0, tot = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (q < warp) woff += s_warp[q];
      tot += s_warp[q];
    }
    const int base = woff + incl - (c0 + c1);
    if (w0 < cb) excl[w0] = base;
    if (w0 + 1 < cb) excl[w0 + 1] = base + c0;
    if (tid == 0) s_total = tot;
    for (int i = tid; i < ((n + 31) >> 5); i += 256) bitmap[i] = 0u;
    __syncthreads();
  }
  const int total = s_total;
  // (2) every sorted position in parallel: rank among the kept, original index (coalesced loads, eight in flight per
  //     thread: one global round trip per 2048 positions)
  for (int pos0 = 0; pos0 < n; pos0 += 256 * 8) {
    int orig[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int pos = pos0 + q * 256 + tid;
      orig[q] = pos < n ? __ldg(ord + pos) : 0;
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int pos = pos0 + q * 256 + tid;
      if (pos < n) {
        const unsigned long long kw = keptw[pos >> 6];
        const int b = pos & 63;
        if ((kw >> b) & 1ULL) {
          const int rank = excl[pos >> 6] + __popcll(kw & ((1ULL << b) - 1ULL));
          if (kps) kps[rank] = orig[q];
          atomicOr(&bitmap[orig[q] >> 5], 1u << (orig[q] & 31));
        }
      }
    }
  }
  __syncthreads();
  // (3) ascending original index: exclusive scan of the bitmap words' counts (<= 1024 words: four per thread), then every
  //     original index in parallel
  {
    const int nbw = (n + 31) >> 5;
    int c[4], cnt = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int w = tid * 4 + q;
      c[q] = w < nbw ? __popc(bitmap[w]) : 0;
      cnt += c[q];
    }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int woff = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q)
      if (q < warp) woff += s_warp[q];
    int run = woff + incl - cnt;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int w = tid * 4 + q;
      if (w < nbw) excl_idx[w] = run;
      run += c[q];
    }
    __syncthreads();
    for (int i = tid; i < n; i += 256) {
      const unsigned bits = bitmap[i >> 5];
      const int bb = i & 31;
      if ((bits >> bb) & 1u) kp[excl_idx[i >> 5] + __popc(bits & ((1u << bb) - 1u))] = i;
    }
  }
  if (tid == 0) num_keep[seg] = total;
  (void)flags;  // per-box flag workspace of an earlier sweep design; kept in the workspace layout
}

struct NmsWorkspace {
  SortedBox *sorted;
  int32_t *order;
  unsigned long long *mask;
  unsigned char *flags;
  size_t bytes;
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static NmsWorkspace carve(void *base, int nseg, int n_max) {
  NmsWorkspace w;
  const size_t cbm = (size_t)(n_max + 63) / 64;
  size_t off = 0;
  char *b = static_cast<char *>(base);
  w.sorted = reinterpret_cast<SortedBox *>(b + off);
  off = align_up(off + sizeof(SortedBox) * (size_t)nseg * n_max, 256);
  w.order = reinterpret_cast<int32_t *>(b + off);
  off = align_up(off + sizeof(int32_t) * (size_t)nseg * n_max, 256);
  w.mask = reinterpret_cast<unsigned long long *>(b + off);
  off = align_up(off + sizeof(unsigned long long) * (size_t)nseg * n_max * cbm, 256);
  w.flags = reinterpret_cast<unsigned char *>(b + off);
  off = align_up(off + (size_t)nseg * n_max, 256);
  w.bytes = off;
  return w;
}

}  // namespace roi3d

using namespace roi3d;

extern "C" {

size_t roi3d_nms3d_workspace_bytes(int nseg, int n_max) {
  if (nseg <= 0 || n_max <= 0) return 256;
  return carve(nullptr, nseg, n_max).bytes;
}

static int nms3d_launch(const float *dets_dev, const int32_t *seg_counts_dev, const uint8_t *presorted_dev, int nseg,
                        int n_max, float iou_thr, int max_keep_presorted,
                        double iou_thr64, bool f64, int64_t *keep_dev, int64_t *keep_by_score_dev, int32_t *num_keep_dev,
                        void *workspace_dev, size_t workspace_bytes, void *stream) {
  ROI3D_CHECK_ARG(nseg >= 0 && n_max >= 0, "bad sizes nseg=%d n_max=%d", nseg, n_max);
  if (nseg == 0) return ROI3D_OK;
  cudaStream_t st = (cudaStream_t)stream;
  ROI3D_CHECK_ARG(num_keep_dev != nullptr, "num_keep is NULL");
  if (n_max == 0) {
    ROI3D_CUDA(cudaMemsetAsync(num_keep_dev, 0, sizeof(int32_t) * nseg, st));
    return ROI3D_OK;
  }
  ROI3D_CHECK_ARG(dets_dev && keep_dev && workspace_dev, "NULL pointer");
  ROI3D_CHECK_ARG(n_max <= kMaxColBlocks * 64, "n_max=%d exceeds %d", n_max, kMaxColBlocks * 64);
  ROI3D_CHECK_ARG(nseg <= 65535, "nseg=%d exceeds 65535", nseg);
  ROI3D_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace_dev) & 255) == 0, "workspace must be 256-byte aligned");
  NmsWorkspace w = carve(workspace_dev, nseg, n_max);
  if (workspace_bytes < w.bytes) {
    set_error("nms3d workspace too small: %zu < %zu", workspace_bytes, w.bytes);
    return ROI3D_ENOMEM;
  }
  const int cbm = (n_max + 63) / 64;
  nms3d_rank_kernel<<<dim3(ceil_div(n_max, 32), nseg), 256, 0, st>>>(dets_dev, seg_counts_dev, presorted_dev, n_max,
                                                                      w.sorted, w.order);
  ROI3D_LAUNCH_CHECK();
  // tiles of the upper triangle: with few of them, one tile per CTA (4x the threads) fills the GPU better
  const long long tiles = (long long)nseg * cbm * (cbm + 1) / 2;
  if (tiles <= 4096) {
    if (f64)
      nms3d_mask_q_kernel<true><<<dim3(cbm, cbm, nseg), 256, 0, st>>>(w.sorted, seg_counts_dev, n_max, iou_thr, iou_thr64,
                                                                      w.mask);
    else
      nms3d_mask_q_kernel<false><<<dim3(cbm, cbm, nseg), 256, 0, st>>>(w.sorted, seg_counts_dev, n_max, iou_thr, iou_thr64,
                                                                       w.mask);
  } else if (f64)
    nms3d_mask_kernel<true><<<dim3(ceil_div(cbm, 4), cbm, nseg), 256, 0, st>>>(w.sorted, seg_counts_dev, n_max, iou_thr,
                                                                               iou_thr64, w.mask);
  else
    nms3d_mask_kernel<false><<<dim3(ceil_div(cbm, 4), cbm, nseg), 256, 0, st>>>(w.sorted, seg_counts_dev, n_max, iou_thr,
                                                                                iou_thr64, w.mask);
  ROI3D_LAUNCH_CHECK();
  {
    const size_t panel_bytes = (size_t)kPanelBufs * 64 * (kPanelW + 1) * sizeof(unsigned long long);  // 66 KiB
    ROI3D_CUDA(cudaFuncSetAttribute(nms3d_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)panel_bytes));
    nms3d_sweep_kernel<<<nseg, 256, panel_bytes, st>>>(w.mask, w.order, seg_counts_dev, n_max, w.flags, keep_dev,
                                                      keep_by_score_dev, num_keep_dev, presorted_dev, max_keep_presorted);
  }
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

int roi3d_nms3d_batched(const float *dets_dev, const int32_t *seg_counts_dev, int nseg, int n_max, float iou_thr,
                        int64_t *keep_dev, int64_t *keep_by_score_dev, int32_t *num_keep_dev, void *workspace_dev,
                        size_t workspace_bytes, void *stream) {
  return nms3d_launch(dets_dev, seg_counts_dev, nullptr, nseg, n_max, iou_thr, 0, 0.0, false, keep_dev, keep_by_score_dev,
                      num_keep_dev, workspace_dev, workspace_bytes, stream);
}

int roi3d_nms3d_batched_presorted(const float *dets_dev, const int32_t *seg_counts_dev, const uint8_t *presorted_dev,
                                  int nseg, int n_max, float iou_thr, int64_t *keep_dev, int64_t *keep_by_score_dev,
                                  int32_t *num_keep_dev, void *workspace_dev, size_t workspace_bytes, void *stream) {
  return nms3d_launch(dets_dev, seg_counts_dev, presorted_dev, nseg, n_max, iou_thr, 0, 0.0, false, keep_dev,
                      keep_by_score_dev, num_keep_dev, workspace_dev, workspace_bytes, stream);
}

int roi3d_nms3d_batched_limited(const float *dets_dev, const int32_t *seg_counts_dev, const uint8_t *presorted_dev,
                                int nseg, int n_max, float iou_thr, int max_keep_presorted, int64_t *keep_dev,
                                int64_t *keep_by_score_dev, int32_t *num_keep_dev, void *workspace_dev,
                                size_t workspace_bytes, void *stream) {
  return nms3d_launch(dets_dev, seg_counts_dev, presorted_dev, nseg, n_max, iou_thr, max_keep_presorted, 0.0, false,
                      keep_dev, keep_by_score_dev, num_keep_dev, workspace_dev, workspace_bytes, stream);
}

int roi3d_nms3d_eval_batched(const float *dets_dev, const int32_t *seg_counts_dev, int nseg, int n_max, double iou_thr,
                             int64_t *keep_dev, int64_t *keep_by_score_dev, int32_t *num_keep_dev, void *workspace_dev,
                             size_t workspace_bytes, void *stream) {
  return nms3d_launch(dets_dev, seg_counts_dev, nullptr, nseg, n_max, 0.0f, 0, iou_thr, true, keep_dev, keep_by_score_dev,
                      num_keep_dev, workspace_dev, workspace_bytes, stream);
}

}  // extern "C"

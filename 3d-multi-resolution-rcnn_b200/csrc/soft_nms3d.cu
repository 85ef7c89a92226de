// 3D soft-NMS for B200 (sm_100a), batched over independent segments, entirely on the device.
//
// Restates (reference, /root/reference): soft_nms_cpu, mmdet/ops/nms/src/soft_nms_cpu.pyx (mmdet v0.6.0; Bodla et al.),
//   reached through soft_nms, mmdet/ops/nms/nms_wrapper.py:55-81, and multiclass_nms_3d with nms_cfg type 'soft_nms'
//   (mmdet/core/post_processing/bbox_nms.py:75-77).  The reference's loop is 2-D, on the CPU, and stops in a debugger on
//   entry (nms_wrapper.py:56); this is its 3-D form on [n, 7] = (x1,y1,x2,y2,z1,z2,score) rows.
//
// The sequential loop (step i of at most n): select the highest score among positions i..N-1 (first position wins a
// tie; a NaN at position i is selected, a NaN elsewhere never), swap it into position i, then decay every later row that
// overlaps it and move the last row into the place of each row whose score falls below min_score (N -= 1, redo).
//
// Here one CTA runs one segment; rows never move.  Thread t owns rows t, t + blockDim, ... (R of them): x1, x2, the
// score and a 16-bit current position live in registers, the boxes and volumes in shared memory (read when a row
// overlaps the selected box in x, and for the selected box itself).  A step is:
//   1. argmax: a block reduction of the key (ordered score, -position, row) -- each thread keeps the best key of its
//      rows and recomputes it only when one of them changed (or holds a NaN score, whose key depends on i); one
//      __syncthreads, then every warp reduces the 32 warp maxima itself, so no second barrier;
//   2. the selected row leaves, the row at position i takes its old position, the owner writes output row i;
//   3. decay: every live row tests the selected box with the reference's arithmetic; a row that falls below min_score
//      sets its position's bit in a drop bitmap;
//   4. renumbering, only in a step after one with drops (detected behind the next step's barrier, so a step without
//      drops costs one barrier): the sequential tail moves have a closed form.  With N' = N - D rows left, the holes are
//      the dropped positions below N', ascending, and they receive the surviving rows at positions >= N', taken in
//      descending position: hole k gets mover k.  (Each row the loop pulls from the end is processed once, at its hole;
//      rows below N' never move.)  A mover finds its rank from the bitmap's prefix counts and its hole by a binary search
//      over them; then the argmax of the step is redone with the new positions (two more barriers).
//
// Bit-exactness: every operation is one IEEE fp32 operation in the reference's order, no contraction (explicit _rn
// intrinsics): area = ((x2-x1+1)*(y2-y1+1))*(z2-z1+1); iw = min(tx2,x2) - max(tx1,x1) + 1 with min / max as
// `a <= b ? a : b` / `a >= b ? a : b`, guards iw > 0, ih > 0, id > 0 nested; inter = (iw*ih)*id; ua = (tarea + area) -
// inter; ov = inter / ua; linear: weight = ov > iou_thr ? 1 - ov : 1; gaussian: weight = (float)exp((double)(-(ov*ov) /
// sigma)) (the reference's np.exp on a Python float).  A NaN score stays the same NaN (quieted), as the x86 multiply
// leaves it.  CUDA's double exp and the host libm's can differ by one double ulp, which changes the fp32 weight only
// when the value sits on an fp32 rounding boundary.  Coordinates are taken to be finite.
#include "common.cuh"

namespace roi3d {

constexpr int kSoftNmsMaxRows = 4096;              // positions are 16-bit, the drop bitmap is 128 words
constexpr int kSoftNmsWords = kSoftNmsMaxRows / 32;

struct __align__(16) SoftBox {
  float x1, y1, x2, y2, z1, z2, area, pad;
};

__device__ __forceinline__ float ref_min(float a, float b) { return a <= b ? a : b; }
__device__ __forceinline__ float ref_max(float a, float b) { return a >= b ? a : b; }

// ordered key of a non-NaN score: larger score -> larger key, -0 == +0, -inf -> 0x007FFFFF > 0
__device__ __forceinline__ unsigned soft_score_key(float s) {
  if (s == 0.0f) s = 0.0f;
  const unsigned u = __float_as_uint(s);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

template <int R>
__global__ void __launch_bounds__(1024) soft_nms3d_kernel(const float *__restrict__ dets, const int32_t *seg_counts,
                                                          int n_max, int method, float iou_thr, float sigma,
                                                          float min_score, float *__restrict__ out_dets,
                                                          int64_t *__restrict__ out_inds, int32_t *__restrict__ num_keep) {
  extern __shared__ __align__(16) SoftBox sbox[];          // [n_max]
  __shared__ uint2 red[2][32];                             // warp maxima, by step parity
  __shared__ unsigned drop_bits[2][kSoftNmsWords + 1];     // dropped positions of a step, by parity (+1 zero word)
  __shared__ int drop_count[2];
  __shared__ int drop_prefix[kSoftNmsWords + 1];           // exclusive prefix of popc(drop_bits) per word, then total

  const int seg = blockIdx.x;
  const int n = seg_counts ? min(max(seg_counts[seg], 0), n_max) : n_max;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const float *d = dets + (long long)seg * n_max * 7;
  float *od = out_dets + (long long)seg * n_max * 7;
  int64_t *oi = out_inds + (long long)seg * n_max;

  // per owned row: x1, x2, score, position (0xFFFF = gone)
  float rx1[R], rx2[R], rs[R];
  unsigned rpos[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int row = tid + r * blockDim.x;
    rpos[r] = 0xFFFFu;
    rx1[r] = rx2[r] = rs[r] = 0.0f;
    if (row < n) {
      const float *b = d + (long long)row * 7;
      SoftBox sb;
      sb.x1 = b[0], sb.y1 = b[1], sb.x2 = b[2], sb.y2 = b[3], sb.z1 = b[4], sb.z2 = b[5];
      sb.area = __fmul_rn(__fmul_rn(__fadd_rn(__fsub_rn(sb.x2, sb.x1), 1.0f), __fadd_rn(__fsub_rn(sb.y2, sb.y1), 1.0f)),
                          __fadd_rn(__fsub_rn(sb.z2, sb.z1), 1.0f));
      sb.pad = 0.0f;
      sbox[row] = sb;
      rx1[r] = sb.x1, rx2[r] = sb.x2, rs[r] = b[6];
      rpos[r] = (unsigned)row;
    }
  }
  for (int w = tid; w < 2 * (kSoftNmsWords + 1); w += blockDim.x) (&drop_bits[0][0])[w] = 0u;
  if (tid < 2) drop_count[tid] = 0;
  __syncthreads();

  // best key of this thread's rows: .x = ordered score (NaN: 0, or all ones at position i), .y = (0xFFFF - pos) << 16 | row
  bool dirty = true;
  uint2 best = make_uint2(0u, 0u);
  auto local_best = [&](int i) {
    bool has_nan = false;
    uint2 b = make_uint2(0u, 0u);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (rpos[r] == 0xFFFFu) continue;
      const bool nan = rs[r] != rs[r];
      has_nan |= nan;
      const unsigned k = nan ? (rpos[r] == (unsigned)i ? 0xFFFFFFFFu : 0u) : soft_score_key(rs[r]);
      const unsigned t = ((0xFFFFu - rpos[r]) << 16) | (unsigned)(tid + r * blockDim.x);
      if (k > b.x || (k == b.x && t > b.y)) b = make_uint2(k, t);
    }
    best = b;
    dirty = has_nan;   // a NaN row's key depends on the step
  };
  auto post_warp_max = [&](int par) {
    const unsigned k = __reduce_max_sync(0xffffffffu, best.x);
    const unsigned t = __reduce_max_sync(0xffffffffu, best.x == k ? best.y : 0u);
    if (lane == 0) red[par][warp] = make_uint2(k, t);
  };

  int N = n;
  for (int i = 0;; ++i) {
    const int par = i & 1;
    if (dirty) local_best(i);
    post_warp_max(par);
    __syncthreads();
    const int D = drop_count[par ^ 1];   // rows the previous step dropped
    N -= D;
    if (i >= N) break;
    if (D > 0) {
      // renumber: prefix counts of the previous step's drop bitmap (warp 0), then each mover takes its hole
      const unsigned *bits = drop_bits[par ^ 1];
      if (warp == 0) {
        unsigned c[4];
        int sum = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) c[q] = __popc(bits[lane * 4 + q]), sum += c[q];
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int v = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += v;
        }
        int run = incl - sum;
#pragma unroll
        for (int q = 0; q < 4; ++q) drop_prefix[lane * 4 + q] = run, run += c[q];
        if (lane == 31) drop_prefix[kSoftNmsWords] = incl;
      }
      __syncthreads();
      const int n_old = N + D;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const unsigned p = rpos[r];
        if (p == 0xFFFFu || p < (unsigned)N) continue;
        // survivors at positions (p, n_old) = rows there minus drops there; drops below p + 1 from the prefix counts
        const int x = (int)p + 1;
        const int below = drop_prefix[x >> 5] + __popc(bits[x >> 5] & ((1u << (x & 31)) - 1u));
        const int rank = (n_old - 1 - (int)p) - (D - below);
        // the rank-th dropped position (ascending): last word whose prefix is <= rank, then the bit inside it
        int lo = 0, hi = kSoftNmsWords;
        while (lo < hi) {
          const int mid = (lo + hi + 1) >> 1;
          if (drop_prefix[mid] <= rank) lo = mid; else hi = mid - 1;
        }
        rpos[r] = (unsigned)(lo * 32) + __fns(bits[lo], 0, rank - drop_prefix[lo] + 1);
        dirty = true;
      }
      if (dirty) local_best(i);
      post_warp_max(par);   // (every read of red[par] above happened before the last barrier)
      __syncthreads();
      if (warp == 0) {      // the bitmap is written again two steps from now
#pragma unroll
        for (int q = 0; q < 4; ++q) drop_bits[par ^ 1][lane * 4 + q] = 0u;
        if (lane == 0) drop_count[par ^ 1] = 0;
      }
    }

    // the winner: every warp reduces the warp maxima itself
    const uint2 v = lane < nwarps ? red[par][lane] : make_uint2(0u, 0u);
    const unsigned wk = __reduce_max_sync(0xffffffffu, v.x);
    const unsigned wt = __reduce_max_sync(0xffffffffu, v.x == wk ? v.y : 0u);
    const int w = (int)(wt & 0xFFFFu);
    const unsigned pw = 0xFFFFu - (wt >> 16);
    const SoftBox t = sbox[w];

    int ndrop = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int row = tid + r * blockDim.x;
      if (rpos[r] == 0xFFFFu) continue;
      if (row == w) {   // selected: output row i, with the score it has now
        float *o = od + (long long)i * 7;
        o[0] = t.x1, o[1] = t.y1, o[2] = t.x2, o[3] = t.y2, o[4] = t.z1, o[5] = t.z2, o[6] = rs[r];
        oi[i] = w;
        rpos[r] = 0xFFFFu;
        dirty = true;
        continue;
      }
      if (rpos[r] == (unsigned)i) rpos[r] = pw, dirty = true;   // the swap
      const float iw = __fadd_rn(__fsub_rn(ref_min(t.x2, rx2[r]), ref_max(t.x1, rx1[r])), 1.0f);
      if (!(iw > 0.0f)) continue;
      const SoftBox b = sbox[row];
      const float ih = __fadd_rn(__fsub_rn(ref_min(t.y2, b.y2), ref_max(t.y1, b.y1)), 1.0f);
      if (!(ih > 0.0f)) continue;
      const float id = __fadd_rn(__fsub_rn(ref_min(t.z2, b.z2), ref_max(t.z1, b.z1)), 1.0f);
      if (!(id > 0.0f)) continue;
      const float inter = __fmul_rn(__fmul_rn(iw, ih), id);
      const float ua = __fsub_rn(__fadd_rn(t.area, b.area), inter);
      const float ov = __fdiv_rn(inter, ua);
      float weight;
      if (method == 1) {
        weight = ov > iou_thr ? __fsub_rn(1.0f, ov) : 1.0f;
      } else {
        weight = (float)exp((double)__fdiv_rn(-__fmul_rn(ov, ov), sigma));
      }
      const float s = rs[r];
      rs[r] = s != s ? __uint_as_float(__float_as_uint(s) | 0x00400000u) : __fmul_rn(weight, s);
      dirty = true;
      if (rs[r] < min_score) {
        const unsigned p = rpos[r];
        atomicOr(&drop_bits[par][p >> 5], 1u << (p & 31));
        rpos[r] = 0xFFFFu;
        ++ndrop;
      }
    }
    const int wdrop = __reduce_add_sync(0xffffffffu, ndrop);
    if (lane == 0 && wdrop) atomicAdd(&drop_count[par], wdrop);
  }
  if (tid == 0) num_keep[seg] = N;
}

template <int R>
static int soft_nms3d_launch_r(const float *dets_dev, const int32_t *seg_counts_dev, int nseg, int n_max, int method,
                               float iou_thr, float sigma, float min_score, float *out_dets_dev, int64_t *inds_dev,
                               int32_t *num_keep_dev, cudaStream_t st) {
  const int threads = min(1024, ceil_div(ceil_div(n_max, R), 32) * 32);
  const size_t smem = sizeof(SoftBox) * (size_t)n_max;
  static PerDeviceSmemOptIn opt_in;
  if (opt_in.need(smem)) {
    ROI3D_CUDA(cudaFuncSetAttribute(soft_nms3d_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(sizeof(SoftBox) * kSoftNmsMaxRows)));
    opt_in.mark(sizeof(SoftBox) * kSoftNmsMaxRows);
  }
  soft_nms3d_kernel<R><<<nseg, threads, smem, st>>>(dets_dev, seg_counts_dev, n_max, method, iou_thr, sigma, min_score,
                                                   out_dets_dev, inds_dev, num_keep_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

}  // namespace roi3d

using namespace roi3d;

extern "C" {

int roi3d_soft_nms3d_batched(const float *dets_dev, const int32_t *seg_counts_dev, int nseg, int n_max, int method,
                             float iou_thr, float sigma, float min_score, float *out_dets_dev, int64_t *inds_dev,
                             int32_t *num_keep_dev, void *stream) {
  ROI3D_CHECK_ARG(nseg >= 0 && n_max >= 0, "bad sizes nseg=%d n_max=%d", nseg, n_max);
  ROI3D_CHECK_ARG(method == 1 || method == 2, "soft_nms3d: method=%d must be 1 (linear) or 2 (gaussian)", method);
  ROI3D_CHECK_ARG(n_max <= kSoftNmsMaxRows, "soft_nms3d: n_max=%d exceeds %d", n_max, kSoftNmsMaxRows);
  if (nseg == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(num_keep_dev != nullptr, "soft_nms3d: num_keep is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_max == 0) {
    ROI3D_CUDA(cudaMemsetAsync(num_keep_dev, 0, sizeof(int32_t) * nseg, st));
    return ROI3D_OK;
  }
  ROI3D_CHECK_ARG(dets_dev && out_dets_dev && inds_dev, "soft_nms3d: NULL pointer");
  if (n_max <= 1024)
    return soft_nms3d_launch_r<1>(dets_dev, seg_counts_dev, nseg, n_max, method, iou_thr, sigma, min_score, out_dets_dev,
                                  inds_dev, num_keep_dev, st);
  if (n_max <= 2048)
    return soft_nms3d_launch_r<2>(dets_dev, seg_counts_dev, nseg, n_max, method, iou_thr, sigma, min_score, out_dets_dev,
                                  inds_dev, num_keep_dev, st);
  return soft_nms3d_launch_r<4>(dets_dev, seg_counts_dev, nseg, n_max, method, iou_thr, sigma, min_score, out_dets_dev,
                                inds_dev, num_keep_dev, st);
}

}  // extern "C"

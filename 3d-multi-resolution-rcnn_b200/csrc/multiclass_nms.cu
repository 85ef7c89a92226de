// Batched multiclass 3D NMS for B200 (sm_100a): the whole test-time post-processing of B images in one call on the
// caller's stream, with fixed-shape outputs and no host synchronisation, so that it can be captured in a CUDA graph.
//
// Restates (reference, /root/reference): multiclass_nms_3d, mmdet/core/post_processing/bbox_nms.py:57-106, for B images
// at once.  Per image the reference loops over the classes (score threshold, NMS per class), concatenates the kept rows
// class by class and, when more than max_num remain, keeps the first max_num of a stable descending sort by score.
//
// Steps, each over every image:
//   1. multiclass_select_kernel: one CTA per (image b, class c >= 1) segment compacts the rows r < counts[b] with
//      scores[b, r, c] > score_thr (fp32 compare: a NaN score never passes) to the front of the segment, stably, as
//      (x1, y1, x2, y2, z1, z2, score) rows, and writes the segment's count.  Rows at or past counts[b] are not read.
//   2. NMS over the B * (C - 1) segments: roi3d_nms3d_batched (kept rows in ascending index, the order the reference's
//      nms returns them in) or roi3d_soft_nms3d_batched (rows in selection order with their decayed scores).
//   3. multiclass_collect_kernel: per image, the kept rows of classes 1..C-1 in that order, with label c - 1, into a
//      [B, (C - 1) * n] row buffer, and a validity mask (position < the image's kept total).
//   4. The max_num cut: roi3d_topk_segmented_masked over the masked buffers, one segment per image.
//   5. multiclass_gather_kernel: det [B, M, 7], labels [B, M] and det_counts [B]; rows past the count are zeros with
//      label -1.
#include <vector>

#include "common.cuh"

namespace roi3d {

constexpr int kMcThreads = 256;
constexpr int kMcWarps = kMcThreads / 32;
constexpr int kMcSoftMaxRows = 4096;    // roi3d_soft_nms3d_batched's n_max limit
constexpr int kMcHardMaxRows = 32768;   // roi3d_nms3d_batched's n_max limit
constexpr int kMcMaxSegments = 65535;   // roi3d_nms3d_batched's nseg limit

// rows of the cut: M = max_num > 0 ? max_num : (C - 1) * n
static long long mc_rows_out(int n, int num_classes, int max_num) {
  return max_num > 0 ? (long long)max_num : (long long)(num_classes - 1) * n;
}

static size_t mc_align(size_t x) { return (x + 255) / 256 * 256; }

struct McWorkspace {
  float *sel;           // [S, n, 7] selected rows per (image, class) segment
  int32_t *sel_count;   // [S]
  int32_t *num_keep;    // [S]
  int64_t *keep;        // hard NMS: [S, n] kept row indices, ascending
  void *nms_ws;         // hard NMS workspace
  size_t nms_ws_bytes;
  float *soft_out;      // soft NMS: [S, n, 7] rows in selection order
  int64_t *soft_inds;   // soft NMS: [S, n]
  float *cat;           // [B, T, 7] kept rows per image, class-major
  float *cat_scores;    // [B, T]
  int32_t *cat_labels;  // [B, T]
  uint8_t *cat_valid;   // [B, T]
  int64_t *tk_idx;      // [B, M]
  float *tk_val;        // [B, M]
  int32_t *tk_count;    // [B]
  void *tk_ws;
  size_t tk_ws_bytes;
  size_t bytes;
};

// Layout of the workspace; base == nullptr computes the size only.  Every buffer starts on a 256-byte boundary.
static McWorkspace mc_carve(void *base, int B, int n, int num_classes, int max_num, bool soft) {
  McWorkspace w{};
  const size_t S = (size_t)B * (num_classes - 1), T = (size_t)(num_classes - 1) * n;
  const size_t M = (size_t)mc_rows_out(n, num_classes, max_num);
  char *b = static_cast<char *>(base);
  size_t off = 0;
  auto take = [&](size_t nbytes) {
    char *p = b ? b + off : nullptr;
    off = mc_align(off + nbytes);
    return p;
  };
  w.sel = reinterpret_cast<float *>(take(sizeof(float) * S * n * 7));
  w.sel_count = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * S));
  w.num_keep = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * S));
  if (soft) {
    w.soft_out = reinterpret_cast<float *>(take(sizeof(float) * S * n * 7));
    w.soft_inds = reinterpret_cast<int64_t *>(take(sizeof(int64_t) * S * n));
  } else {
    w.keep = reinterpret_cast<int64_t *>(take(sizeof(int64_t) * S * n));
    w.nms_ws_bytes = roi3d_nms3d_workspace_bytes((int)S, n);
    w.nms_ws = take(w.nms_ws_bytes);
  }
  w.cat = reinterpret_cast<float *>(take(sizeof(float) * B * T * 7));
  w.cat_scores = reinterpret_cast<float *>(take(sizeof(float) * B * T));
  w.cat_labels = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * B * T));
  w.cat_valid = reinterpret_cast<uint8_t *>(take(B * T));
  w.tk_idx = reinterpret_cast<int64_t *>(take(sizeof(int64_t) * B * M));
  w.tk_val = reinterpret_cast<float *>(take(sizeof(float) * B * M));
  w.tk_count = reinterpret_cast<int32_t *>(take(sizeof(int32_t) * B));
  w.tk_ws_bytes = roi3d_topk_workspace_bytes(B, (int)M);
  w.tk_ws = take(w.tk_ws_bytes);
  w.bytes = off;
  return w;
}

// One CTA per (image, class) segment s = b * (C - 1) + (c - 1): stable compaction of the passing rows, 256 rows per
// round (a ballot per warp, the eight warp counts scanned by every thread).
__global__ void __launch_bounds__(kMcThreads) multiclass_select_kernel(const float *__restrict__ bboxes, int box_cols,
                                                                       const float *__restrict__ scores,
                                                                       const int32_t *__restrict__ counts, int n,
                                                                       int num_classes, float score_thr,
                                                                       float *__restrict__ sel, int32_t *__restrict__ sel_count) {
  __shared__ int warp_cnt[2][kMcWarps];
  const int s = blockIdx.x, ncls = num_classes - 1;
  const int b = s / ncls, c = s - b * ncls + 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rows = min(max(counts[b], 0), n);
  const int col0 = box_cols == 6 ? 0 : 6 * c;
  float *out = sel + (size_t)s * n * 7;
  int kept = 0;
  for (int base = 0, round = 0; base < rows; base += kMcThreads, round ^= 1) {
    const int r = base + threadIdx.x;
    float score = 0.0f;
    bool pass = false;
    if (r < rows) {
      score = scores[((size_t)b * n + r) * num_classes + c];
      pass = score > score_thr;
    }
    const unsigned ball = __ballot_sync(0xffffffffu, pass);
    if (lane == 0) warp_cnt[round][warp] = __popc(ball);
    __syncthreads();   // (double-buffered by round: the next round's counts go to the other half)
    int before = 0, total = 0;
#pragma unroll
    for (int q = 0; q < kMcWarps; ++q) {
      const int v = warp_cnt[round][q];
      before += q < warp ? v : 0;
      total += v;
    }
    if (pass) {
      const float *src = bboxes + ((size_t)b * n + r) * box_cols + col0;
      float *dst = out + (size_t)(kept + before + __popc(ball & ((1u << lane) - 1u))) * 7;
#pragma unroll
      for (int q = 0; q < 6; ++q) dst[q] = src[q];
      dst[6] = score;
    }
    kept += total;
  }
  if (threadIdx.x == 0) sel_count[s] = kept;
}

// grid (ceil(n / 256), S).  Row i of segment s = (b, c) goes to position (kept rows of classes < c) + i of image b.
// Every position p = (c - 1) * n + i of the image's buffer also gets its validity byte here (p < the image's total);
// the score of an invalid position is set to 0 so that nothing undefined is ever read.
__global__ void __launch_bounds__(kMcThreads) multiclass_collect_kernel(const float *__restrict__ sel,
                                                                        const int64_t *__restrict__ keep,
                                                                        const float *__restrict__ soft_out,
                                                                        const int32_t *__restrict__ num_keep, int n,
                                                                        int num_classes, float *__restrict__ cat,
                                                                        float *__restrict__ cat_scores,
                                                                        int32_t *__restrict__ cat_labels,
                                                                        uint8_t *__restrict__ cat_valid) {
  const int s = blockIdx.y, ncls = num_classes - 1;
  const int b = s / ncls, ci = s - b * ncls;
  const int i = blockIdx.x * kMcThreads + threadIdx.x;
  if (i >= n) return;
  int before = 0, total = 0, mine = 0;
  for (int q = 0; q < ncls; ++q) {
    const int v = min(max(num_keep[b * ncls + q], 0), n);
    before += q < ci ? v : 0;
    mine = q == ci ? v : mine;
    total += v;
  }
  const size_t T = (size_t)ncls * n, img = (size_t)b * T;
  if (i < mine) {
    const float *src;
    if (soft_out != nullptr) {
      src = soft_out + ((size_t)s * n + i) * 7;
    } else {
      long long r = keep[(size_t)s * n + i];
      r = r < 0 ? 0 : (r >= n ? n - 1 : r);
      src = sel + ((size_t)s * n + r) * 7;
    }
    const size_t p = img + before + i;
    float *dst = cat + p * 7;
#pragma unroll
    for (int q = 0; q < 7; ++q) dst[q] = src[q];
    cat_scores[p] = src[6];
    cat_labels[p] = ci;
  }
  const int pos = ci * n + i;
  cat_valid[img + pos] = pos < total ? 1 : 0;
  if (pos >= total) cat_scores[img + pos] = 0.0f;
}

// grid (max(ceil(M / 256), 1), B).  The reference's cut `if len > max_num: sort(desc, stable)[:max_num]`, read with
// Python's slice rule: max_num > 0 keeps min(len, max_num) rows (the top-k returned them); max_num == 0 keeps none;
// max_num < 0 keeps the first len + max_num rows of the full descending sort.
__global__ void __launch_bounds__(kMcThreads) multiclass_gather_kernel(const float *__restrict__ cat,
                                                                       const int32_t *__restrict__ cat_labels, int T,
                                                                       const int64_t *__restrict__ tk_idx,
                                                                       const int32_t *__restrict__ tk_count, int M,
                                                                       int max_num, float *__restrict__ det,
                                                                       int64_t *__restrict__ labels,
                                                                       int32_t *__restrict__ det_counts) {
  const int b = blockIdx.y, j = blockIdx.x * kMcThreads + threadIdx.x;
  int cnt = tk_count != nullptr ? min(max(tk_count[b], 0), M) : 0;
  if (max_num < 0) cnt = max(cnt + max_num, 0);
  if (blockIdx.x == 0 && threadIdx.x == 0) det_counts[b] = cnt;
  if (j >= M) return;
  float *dst = det + ((size_t)b * M + j) * 7;
  if (j < cnt) {
    long long p = tk_idx[(size_t)b * M + j];
    p = p < 0 ? 0 : (p >= T ? T - 1 : p);
    const float *src = cat + ((size_t)b * T + p) * 7;
#pragma unroll
    for (int q = 0; q < 7; ++q) dst[q] = src[q];
    labels[(size_t)b * M + j] = cat_labels[(size_t)b * T + p];
  } else {
#pragma unroll
    for (int q = 0; q < 7; ++q) dst[q] = 0.0f;
    labels[(size_t)b * M + j] = -1;
  }
}

}  // namespace roi3d

using namespace roi3d;

extern "C" {

size_t roi3d_multiclass_nms3d_workspace_bytes(int B, int n, int num_classes, int max_num, int soft) {
  if (B <= 0 || n < 0 || num_classes < 2) return 256;
  return mc_carve(nullptr, B, n, num_classes, max_num, soft != 0).bytes;
}

int roi3d_multiclass_nms3d_batched(const float *bboxes_dev, int box_cols, const float *scores_dev,
                                   const int32_t *counts_dev, int B, int n, int num_classes, float score_thr,
                                   int nms_type, float iou_thr, int soft_method, float sigma, float min_score,
                                   int max_num, float *det_dev, int64_t *labels_dev, int32_t *det_counts_dev,
                                   void *workspace_dev, size_t workspace_bytes, void *stream) {
  ROI3D_CHECK_ARG(B >= 0 && n >= 0, "multiclass_nms3d: bad sizes B=%d n=%d", B, n);
  ROI3D_CHECK_ARG(num_classes >= 2, "multiclass_nms3d: num_classes=%d must be >= 2 (class 0 is the background)",
                  num_classes);
  ROI3D_CHECK_ARG(box_cols == 6 || box_cols == 6 * num_classes,
                  "multiclass_nms3d: box_cols=%d must be 6 or 6 * num_classes = %d", box_cols, 6 * num_classes);
  ROI3D_CHECK_ARG(nms_type == 0 || nms_type == 1, "multiclass_nms3d: nms_type=%d must be 0 (nms) or 1 (soft_nms)",
                  nms_type);
  const bool soft = nms_type == 1;
  ROI3D_CHECK_ARG(!soft || soft_method == 1 || soft_method == 2,
                  "multiclass_nms3d: soft_method=%d must be 1 (linear) or 2 (gaussian)", soft_method);
  ROI3D_CHECK_ARG(!soft || n <= kMcSoftMaxRows, "multiclass_nms3d: n=%d exceeds soft-NMS's %d rows per class", n,
                  kMcSoftMaxRows);
  ROI3D_CHECK_ARG(soft || n <= kMcHardMaxRows, "multiclass_nms3d: n=%d exceeds NMS's %d rows per class", n,
                  kMcHardMaxRows);
  const long long M = mc_rows_out(n, num_classes, max_num);
  const long long T = (long long)(num_classes - 1) * n;
  ROI3D_CHECK_ARG((long long)B * (num_classes - 1) <= kMcMaxSegments, "multiclass_nms3d: B * (num_classes - 1) = %lld "
                  "exceeds %d", (long long)B * (num_classes - 1), kMcMaxSegments);
  ROI3D_CHECK_ARG(M <= 0x7FFFFFFFLL && T <= 0x7FFFFFFFLL, "multiclass_nms3d: output rows M=%lld exceed 2^31 - 1", M);
  if (B == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(det_counts_dev && (M == 0 || (det_dev && labels_dev)), "multiclass_nms3d: NULL output pointer");
  ROI3D_CHECK_ARG(n == 0 || (bboxes_dev && scores_dev && counts_dev), "multiclass_nms3d: NULL input pointer");
  ROI3D_CHECK_ARG(workspace_dev != nullptr, "multiclass_nms3d: NULL workspace");
  ROI3D_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace_dev) & 255) == 0,
                  "multiclass_nms3d: workspace must be 256-byte aligned");
  McWorkspace w = mc_carve(workspace_dev, B, n, num_classes, max_num, soft);
  if (workspace_bytes < w.bytes) {
    set_error("multiclass_nms3d: workspace too small: %zu < %zu", workspace_bytes, w.bytes);
    return ROI3D_ENOMEM;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int S = B * (num_classes - 1);
  const bool any_rows = n > 0 && max_num != 0;   // max_num == 0 keeps nothing (`[:0]`)
  if (any_rows) {
    multiclass_select_kernel<<<S, kMcThreads, 0, st>>>(bboxes_dev, box_cols, scores_dev, counts_dev, n, num_classes,
                                                      score_thr, w.sel, w.sel_count);
    ROI3D_LAUNCH_CHECK();
    int rc = soft ? roi3d_soft_nms3d_batched(w.sel, w.sel_count, S, n, soft_method, iou_thr, sigma, min_score, w.soft_out,
                                             w.soft_inds, w.num_keep, stream)
                  : roi3d_nms3d_batched(w.sel, w.sel_count, S, n, iou_thr, w.keep, nullptr, w.num_keep, w.nms_ws,
                                        w.nms_ws_bytes, stream);
    if (rc != ROI3D_OK) return rc;
    multiclass_collect_kernel<<<dim3(ceil_div(n, kMcThreads), S), kMcThreads, 0, st>>>(
        w.sel, w.keep, w.soft_out, w.num_keep, n, num_classes, w.cat, w.cat_scores, w.cat_labels, w.cat_valid);
    ROI3D_LAUNCH_CHECK();
    // one top-k segment per image over its T positions; only the valid ones take part.  max_num > 0: an image with at
    // most M rows comes back whole in concatenation order, a longer one as its top M (descending, ties to the lower
    // position).  max_num < 0: every image comes back whole in score order.
    std::vector<int64_t> seg_off(B), seg_len(B, T);
    std::vector<const uint8_t *> seg_mask(B);
    for (int b = 0; b < B; ++b) seg_off[b] = (int64_t)b * T, seg_mask[b] = w.cat_valid + (size_t)b * T;
    rc = roi3d_topk_segmented_masked(w.cat_scores, seg_off.data(), seg_len.data(), nullptr, seg_mask.data(), B, (int)M, 0,
                                     max_num > 0 ? 1 : 0, w.tk_idx, w.tk_val, w.tk_count, nullptr, w.tk_ws,
                                     w.tk_ws_bytes, stream);
    if (rc != ROI3D_OK) return rc;
  }
  multiclass_gather_kernel<<<dim3(M > 0 ? ceil_div((int)M, kMcThreads) : 1, B), kMcThreads, 0, st>>>(
      w.cat, w.cat_labels, (int)T, w.tk_idx, any_rows ? w.tk_count : nullptr, (int)M, max_num, det_dev, labels_dev,
      det_counts_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

}  // extern "C"

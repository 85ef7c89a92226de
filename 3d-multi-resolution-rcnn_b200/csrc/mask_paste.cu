// Mask paste (SURVEY section 8f, row N4): the per-detection resize + threshold of FCNMaskHead3D.get_seg_masks on
// the device, for B200 (sm_100a).
//
// Replaces (reference, /root/reference): mmdet/models/mask_heads/fcn_mask_head_3d.py:144-187 -- per detection on the
// host: sigmoid -> numpy, `skimage.transform.resize(mask, (d, h, w))`, `> mask_thr_binary`, paste into a full-volume
// uint8 array.  `resize` is third-party (scikit-image==0.18.0 over scipy==1.5.4, requirements.txt:24-25; neither is
// under /root/reference).  Its n-dimensional branch is restated here from the published algorithm:
//   factors = in / out (float64);  anti-aliasing (default for float input): sigma = max(0, (factors - 1) / 2),
//   scipy.ndimage.gaussian_filter(mode='mirror', truncate 4.0) = per axis (z, y, x) a symmetric correlate1d in float64
//   accumulators with the result rounded to the image dtype (float32) after every axis;
//   coordinates c = factors * (o + 0.5) - 0.5;  scipy.ndimage.map_coordinates(order=1, mode='mirror'): the coordinate
//   is folded into [0, n-1] by reflection, weights (1 - t, 1 - (1 - t)), the 8 corners accumulated z-outer / x-inner in float64,
//   rounded to float32;  clip to the filtered image's [min, max];  `> thr` in float32.
// Parity status: unpinned by the reference (no test exercises it) -- checked against the same restatement running on
// the scipy.ndimage that is installed in this image.
//
// Work layout: the CTA (detection, split) computes the whole filtered mask in shared memory -- the clip needs its min
// and max -- and resamples one contiguous chunk of the detection's output voxels.  A detection with few output voxels
// (the box smaller than the mask: heavy filtering, little resampling) takes one CTA; a large box (little or no
// filtering, up to hundreds of thousands of output voxels) is spread over up to `splits` CTAs.  Every axis is filtered
// in place: a warp owns a whole line, copies it with its mirror extension into a per-warp float64 buffer and writes
// the filtered line back, so one float32 image of the mask is all the CTA keeps.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace roi3d {

constexpr int kMaskMaxTaps = 257;   // mask targets: gaussian half width up to 128

constexpr int kPasteThreads = 256;
constexpr int kPasteWarps = kPasteThreads / 32;
constexpr int kPasteMaxAxis = 64;                                       // longest mask axis
constexpr int kPasteMaxHalf = 126;                                      // int(4 sigma + 0.5) at sigma = (64 / 1 - 1) / 2
constexpr int kPasteMaxTaps = 2 * kPasteMaxHalf + 1;
constexpr int kPasteLineLen = kPasteMaxAxis + 2 * kPasteMaxHalf;        // a line with its mirror extension
constexpr int kPasteFixedSmem = (kPasteMaxTaps + kPasteWarps * kPasteLineLen) * 8 + 2 * kPasteWarps * 4;  // 22,312 B
constexpr int kPasteSmemBudget = 227 * 1024;                            // shared memory of one block on sm_100
constexpr int kPasteMaxVol = (kPasteSmemBudget - kPasteFixedSmem) / 4;  // 52,534 voxels of float32 mask
constexpr long long kPasteMinChunk = 8192;  // output voxels below which a detection is not split further
constexpr int kPasteMaxSplits = 16;
constexpr int kPasteGridCtas = 4096;        // splits = clamp(kPasteGridCtas / n, 1, kPasteMaxSplits)

__device__ __forceinline__ int mirror_index(int i, int n) {
  if (n == 1) return 0;
  const int p = 2 * n - 2;
  i %= p;
  if (i < 0) i += p;
  return i < n ? i : p - i;
}

// scipy's coordinate fold for mode 'mirror' (ni_interpolation.c, map_coordinate)
__device__ __forceinline__ double mirror_coord(double c, int n) {
  if (n <= 1) return 0.0;
  const double len = (double)n - 1.0;
  if (c < 0.0) {
    const double sz2 = 2.0 * len;
    c = __dadd_rn(sz2 * (double)(long long)__ddiv_rn(-c, sz2), c);
    c = c <= -len ? __dadd_rn(c, sz2) : -c;
  } else if (c > len) {
    const double sz2 = 2.0 * len;
    c = __dsub_rn(c, sz2 * (double)(long long)__ddiv_rn(c, sz2));
    if (c > len) c = __dsub_rn(sz2, c);
  }
  return c;
}

// numpy's pairwise_sum (np.sum of a contiguous float64 array), as `phi_x / phi_x.sum()` normalises the gaussian
__device__ double np_pairwise_sum(const double *a, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r = __dadd_rn(r, a[i]);
    return r;
  }
  if (n <= 128) {
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
      for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], a[i + j]);
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, a[i]);
    return res;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  return __dadd_rn(np_pairwise_sum(a, n2), np_pairwise_sum(a + n2, n - n2));
}

// logits [n, num_channels, Dm, Hm, Wm]; detection i reads channel `channel[i]` (channel == nullptr: channel 0).
// Grid (n, splits), dynamic shared memory kPasteFixedSmem + 4 * Dm * Hm * Wm bytes.
__global__ void __launch_bounds__(kPasteThreads) mask_paste_kernel(const float *__restrict__ logits, int num_channels,
                                                                   const int64_t *__restrict__ channel, int Dm, int Hm,
                                                                   int Wm, const int32_t *__restrict__ boxes,
                                                                   const int64_t *__restrict__ offsets, float thr,
                                                                   unsigned char *__restrict__ out) {
  extern __shared__ double smem_d[];
  double *wts = smem_d;                                   // kPasteMaxTaps
  double *line = wts + kPasteMaxTaps + (threadIdx.x >> 5) * kPasteLineLen;   // this warp's line buffer
  float *red = reinterpret_cast<float *>(smem_d + kPasteMaxTaps + kPasteWarps * kPasteLineLen);  // 2 * kPasteWarps
  float *M = red + 2 * kPasteWarps;                       // the mask, Dm * Hm * Wm
  __shared__ double wsum;
  const int det = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int32_t *bx = boxes + (long long)det * 6;
  const int ow = max(bx[2] - bx[0] + 1, 1), oh = max(bx[3] - bx[1] + 1, 1), od = max(bx[5] - bx[4] + 1, 1);
  const long long total = (long long)od * oh * ow;
  const long long active = min((long long)gridDim.y, max(1LL, (total + kPasteMinChunk - 1) / kPasteMinChunk));
  if ((long long)blockIdx.y >= active) return;
  const long long chunk = (total + active - 1) / active;
  const long long lo = chunk * blockIdx.y, hi = min(total, lo + chunk);
  unsigned char *dst = out + offsets[det];
  const long long ch = channel ? channel[det] : 0;
  if (ch < 0 || ch >= num_channels) {   // documented: an out-of-range channel gives an all-zero mask
    for (long long o = lo + tid; o < hi; o += kPasteThreads) dst[o] = 0;
    return;
  }
  const int vol = Dm * Hm * Wm;
  const float *src = logits + ((long long)det * num_channels + ch) * vol;
  for (int i = tid; i < vol; i += kPasteThreads) M[i] = __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-src[i])));  // torch sigmoid
  __syncthreads();
  const int dims[3] = {Dm, Hm, Wm};
  const int outs[3] = {od, oh, ow};
  const int strides[3] = {Hm * Wm, Wm, 1};
  // ---- anti-aliasing gaussian, axis by axis, each line filtered in place by one warp ----
  for (int ax = 0; ax < 3; ++ax) {
    const double factor = __ddiv_rn((double)dims[ax], (double)outs[ax]);
    const double sigma = fmax(0.0, __dmul_rn(__dsub_rn(factor, 1.0), 0.5));   // (factors - 1) / 2
    if (!(sigma > 1e-15)) continue;
    const int lw = (int)__dadd_rn(__dmul_rn(4.0, sigma), 0.5);               // <= kPasteMaxHalf for axes <= 64
    const double k = __ddiv_rn(-0.5, __dmul_rn(sigma, sigma));
    for (int i = tid; i <= 2 * lw; i += kPasteThreads) {
      const double x = (double)(i - lw);
      wts[i] = exp(__dmul_rn(k, __dmul_rn(x, x)));
    }
    __syncthreads();
    if (tid == 0) wsum = np_pairwise_sum(wts, 2 * lw + 1);
    __syncthreads();
    for (int i = tid; i <= 2 * lw; i += kPasteThreads) wts[i] = __ddiv_rn(wts[i], wsum);
    __syncthreads();
    const int n = dims[ax], st = strides[ax], ext = n + 2 * lw;
    const int lines = vol / n;
    for (int l = warp; l < lines; l += kPasteWarps) {
      float *base = M + (l / st) * (st * n) + l % st;
      for (int j = lane; j < ext; j += 32) line[j] = (double)base[mirror_index(j - lw, n) * st];
      __syncwarp();
      for (int p = lane; p < n; p += 32) {
        const double *c = line + p + lw;
        double tmp = __dmul_rn(c[0], wts[lw]);   // scipy's symmetric correlate1d: separate multiplies and adds
        for (int ll = -lw; ll < 0; ++ll) tmp = __dadd_rn(tmp, __dmul_rn(__dadd_rn(c[ll], c[-ll]), wts[ll + lw]));
        base[p * st] = (float)tmp;
      }
      __syncwarp();
    }
    __syncthreads();
  }
  // ---- min / max of the filtered image (clip=True) ----
  float mn = INFINITY, mx = -INFINITY;
  for (int i = tid; i < vol; i += kPasteThreads) mn = fminf(mn, M[i]), mx = fmaxf(mx, M[i]);
  for (int o = 16; o > 0; o >>= 1)
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o)), mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red[warp] = mn, red[kPasteWarps + warp] = mx;
  __syncthreads();
  mn = red[0], mx = red[kPasteWarps];
  for (int w = 1; w < kPasteWarps; ++w) mn = fminf(mn, red[w]), mx = fmaxf(mx, red[kPasteWarps + w]);
  // ---- trilinear resample of this CTA's chunk at the box resolution, threshold ----
  const double fz = __ddiv_rn((double)Dm, (double)od), fy = __ddiv_rn((double)Hm, (double)oh),
               fx = __ddiv_rn((double)Wm, (double)ow);
  for (long long o = lo + tid; o < hi; o += kPasteThreads) {
    const int x = (int)(o % ow);
    const long long t1 = o / ow;
    const int y = (int)(t1 % oh), z = (int)(t1 / oh);
    // c = factors * (o + 0.5) - 0.5, folded; weights (1 - t, 1 - (1 - t)) as scipy's spline weights for order 1
    const double cz = mirror_coord(__dsub_rn(__dmul_rn(fz, __dadd_rn((double)z, 0.5)), 0.5), Dm);
    const double cy = mirror_coord(__dsub_rn(__dmul_rn(fy, __dadd_rn((double)y, 0.5)), 0.5), Hm);
    const double cx = mirror_coord(__dsub_rn(__dmul_rn(fx, __dadd_rn((double)x, 0.5)), 0.5), Wm);
    const int z0 = (int)floor(cz), y0 = (int)floor(cy), x0 = (int)floor(cx);
    const double wz0 = __dsub_rn(1.0, __dsub_rn(cz, (double)z0)), wy0 = __dsub_rn(1.0, __dsub_rn(cy, (double)y0)),
                 wx0 = __dsub_rn(1.0, __dsub_rn(cx, (double)x0));
    const double wz[2] = {wz0, __dsub_rn(1.0, wz0)}, wy[2] = {wy0, __dsub_rn(1.0, wy0)}, wx[2] = {wx0, __dsub_rn(1.0, wx0)};
    const int zi[2] = {mirror_index(z0, Dm), mirror_index(z0 + 1, Dm)};
    const int yi[2] = {mirror_index(y0, Hm), mirror_index(y0 + 1, Hm)};
    const int xi[2] = {mirror_index(x0, Wm), mirror_index(x0 + 1, Wm)};
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          double coeff = (double)M[(zi[a] * Hm + yi[b]) * Wm + xi[c]];
          coeff = __dmul_rn(coeff, wz[a]);
          coeff = __dmul_rn(coeff, wy[b]);
          coeff = __dmul_rn(coeff, wx[c]);
          acc = __dadd_rn(acc, coeff);
        }
    float v = (float)acc;
    v = fminf(fmaxf(v, mn), mx);
    dst[o] = v > thr ? 1 : 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Mask targets (SURVEY 8f, row N4, training half): mask_target_single, mmdet/core/mask/mask_target.py:17-50.
// Per positive proposal on the host the reference crops the assigned ground-truth mask to the proposal's int32 box,
// runs `255 * skimage.transform.resize(crop, (mask_size_depth, mask_size, mask_size))`, casts to uint8 (truncation)
// and sets every non-zero voxel to 1.  The crop is a uint8 array, so `resize` first maps it to float64 with
// v * (1 / 255) (skimage.util.img_as_float) and everything after that -- gaussian anti-aliasing, order-1
// map_coordinates, clip -- runs in float64.  Same restatement of the two scipy.ndimage primitives as mask_paste_kernel
// (operation order included: with {0,1} masks the reference's result hinges on the last bit of 255 * (sum w_i / 255)).
// One CTA per proposal; the filtered crop lives in a global float64 workspace (two buffers of the crop's volume).
// ---------------------------------------------------------------------------------------------------------------
struct MaskTargetJob {
  long long ws_off;   // doubles from the workspace base: two buffers of vol doubles each
  int gt;             // ground-truth mask index
  int x1, y1, z1;     // crop origin (>= 0)
  int w, h, d;        // crop size after numpy's slice clipping; any <= 0 -> all-zero target
};

__global__ void __launch_bounds__(256) mask_target_kernel(const unsigned char *__restrict__ gt_masks, int D, int H, int W,
                                                          const MaskTargetJob *__restrict__ jobs, int Md, int Mh, int Mw,
                                                          double *__restrict__ ws, float *__restrict__ out) {
  __shared__ double wts[kMaskMaxTaps];
  __shared__ double red_min[256], red_max[256];
  const int job = blockIdx.x, tid = threadIdx.x;
  const MaskTargetJob j = jobs[job];
  float *dst = out + (long long)job * Md * Mh * Mw;
  const int ovol = Md * Mh * Mw;
  if (j.w <= 0 || j.h <= 0 || j.d <= 0) {
    for (int i = tid; i < ovol; i += 256) dst[i] = 0.0f;
    return;
  }
  const long long vol = (long long)j.d * j.h * j.w;
  double *cur = ws + j.ws_off, *nxt = cur + vol;
  const unsigned char *src = gt_masks + (long long)j.gt * D * H * W;
  for (long long e = tid; e < vol; e += 256) {
    const int x = (int)(e % j.w);
    const long long t = e / j.w;
    const int y = (int)(t % j.h), z = (int)(t / j.h);
    cur[e] = (double)src[((long long)(j.z1 + z) * H + (j.y1 + y)) * W + (j.x1 + x)] * (1.0 / 255.0);  // img_as_float
  }
  __syncthreads();
  const int dims[3] = {j.d, j.h, j.w};
  const int outs[3] = {Md, Mh, Mw};
  const long long strides[3] = {(long long)j.h * j.w, (long long)j.w, 1};
  for (int ax = 0; ax < 3; ++ax) {
    const double factor = (double)dims[ax] / (double)outs[ax];
    const double sigma = fmax(0.0, (factor - 1.0) / 2.0);
    if (!(sigma > 1e-15)) continue;   // scipy's gaussian_filter skips axes with sigma <= 1e-15
    int lw = (int)(4.0 * sigma + 0.5);
    if (lw > (kMaskMaxTaps - 1) / 2) lw = (kMaskMaxTaps - 1) / 2;
    for (int i = tid; i <= 2 * lw; i += 256) {
      const double x = (double)(i - lw);
      wts[i] = exp(-0.5 / (sigma * sigma) * (x * x));
    }
    __syncthreads();
    if (tid == 0) {
      double sum = 0.0;
      for (int i = 0; i <= 2 * lw; ++i) sum += wts[i];
      for (int i = 0; i <= 2 * lw; ++i) wts[i] = wts[i] / sum;
    }
    __syncthreads();
    const int n = dims[ax];
    const long long st = strides[ax];
    for (long long e = tid; e < vol; e += 256) {
      const int pos = (int)((e / st) % n);
      const long long base = e - (long long)pos * st;
      double tmp = __dmul_rn(cur[e], wts[lw]);   // scipy's correlate1d: separate multiplies and adds, no contraction
      for (int ll = -lw; ll < 0; ++ll) {
        const double l = cur[base + (long long)mirror_index(pos + ll, n) * st];
        const double r = cur[base + (long long)mirror_index(pos - ll, n) * st];
        tmp = __dadd_rn(tmp, __dmul_rn(__dadd_rn(l, r), wts[ll + lw]));
      }
      nxt[e] = tmp;
    }
    __syncthreads();
    double *t = cur;
    cur = nxt, nxt = t;
  }
  double mn = INFINITY, mx = -INFINITY;
  for (long long i = tid; i < vol; i += 256) mn = fmin(mn, cur[i]), mx = fmax(mx, cur[i]);
  red_min[tid] = mn, red_max[tid] = mx;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) red_min[tid] = fmin(red_min[tid], red_min[tid + o]), red_max[tid] = fmax(red_max[tid], red_max[tid + o]);
    __syncthreads();
  }
  mn = red_min[0], mx = red_max[0];
  const double fz = (double)j.d / (double)Md, fy = (double)j.h / (double)Mh, fx = (double)j.w / (double)Mw;
  for (int o = tid; o < ovol; o += 256) {
    const int x = o % Mw;
    const int t1 = o / Mw;
    const int y = t1 % Mh, z = t1 / Mh;
    const double cz = mirror_coord(fz * ((double)z + 0.5) - 0.5, j.d);
    const double cy = mirror_coord(fy * ((double)y + 0.5) - 0.5, j.h);
    const double cx = mirror_coord(fx * ((double)x + 0.5) - 0.5, j.w);
    const int z0 = (int)floor(cz), y0 = (int)floor(cy), x0 = (int)floor(cx);
    const double tz = cz - (double)z0, ty = cy - (double)y0, tx = cx - (double)x0;
    const double wz[2] = {1.0 - tz, tz}, wy[2] = {1.0 - ty, ty}, wx[2] = {1.0 - tx, tx};
    const int zi[2] = {mirror_index(z0, j.d), mirror_index(z0 + 1, j.d)};
    const int yi[2] = {mirror_index(y0, j.h), mirror_index(y0 + 1, j.h)};
    const int xi[2] = {mirror_index(x0, j.w), mirror_index(x0 + 1, j.w)};
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          double coeff = cur[((long long)zi[a] * j.h + yi[b]) * j.w + xi[c]];
          coeff = __dmul_rn(coeff, wz[a]);
          coeff = __dmul_rn(coeff, wy[b]);
          coeff = __dmul_rn(coeff, wx[c]);
          acc = __dadd_rn(acc, coeff);
        }
    acc = fmin(fmax(acc, mn), mx);                       // clip=True
    const double scaled = __dmul_rn(255.0, acc);         // `255 * resize(...)`
    const unsigned char u = (unsigned char)(int)scaled;  // .astype(np.uint8): truncation (values are in [0, 255])
    dst[o] = u > 0 ? 1.0f : 0.0f;                        // target[target > 0] = 1, then .float()
  }
}

}  // namespace roi3d

using namespace roi3d;

extern "C" {

}  // extern "C"

namespace {

int mask_paste_launch(const float *logits_dev, int n, int num_channels, int Dm, int Hm, int Wm,
                      const int64_t *channel_dev, const int32_t *boxes_dev, const int64_t *offsets_dev, float thr,
                      uint8_t *out_dev, void *stream) {
  ROI3D_CHECK_ARG(n >= 0, "n = %d is negative", n);
  ROI3D_CHECK_ARG(num_channels >= 1, "num_channels = %d must be at least 1", num_channels);
  ROI3D_CHECK_ARG(Dm > 0 && Hm > 0 && Wm > 0, "mask size %dx%dx%d (Dm x Hm x Wm) must be positive", Dm, Hm, Wm);
  ROI3D_CHECK_ARG((long long)Dm * Hm * Wm <= kPasteMaxVol, "mask of %dx%dx%d (Dm x Hm x Wm) exceeds %d voxels", Dm, Hm,
                  Wm, kPasteMaxVol);
  ROI3D_CHECK_ARG(Dm <= kPasteMaxAxis && Hm <= kPasteMaxAxis && Wm <= kPasteMaxAxis,
                  "mask axes Dm, Hm, Wm = %d, %d, %d: longer than %d is not supported", Dm, Hm, Wm, kPasteMaxAxis);
  if (n == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(logits_dev, "mask logits pointer is NULL");
  ROI3D_CHECK_ARG(boxes_dev, "boxes_dev is NULL");
  ROI3D_CHECK_ARG(offsets_dev, "offsets_dev is NULL");
  ROI3D_CHECK_ARG(out_dev, "out_dev is NULL");
  const int smem = kPasteFixedSmem + 4 * Dm * Hm * Wm;
  ROI3D_CUDA(cudaFuncSetAttribute(mask_paste_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const int splits = std::min(kPasteMaxSplits, std::max(1, kPasteGridCtas / n));
  mask_paste_kernel<<<dim3((unsigned)n, (unsigned)splits), kPasteThreads, smem, (cudaStream_t)stream>>>(
      logits_dev, num_channels, channel_dev, Dm, Hm, Wm, boxes_dev, offsets_dev, thr, out_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

}  // namespace

extern "C" {

int roi3d_mask_paste(const float *mask_logits_dev, int n, int Dm, int Hm, int Wm, const int32_t *boxes_dev,
                     const int64_t *offsets_dev, float thr, uint8_t *out_dev, void *stream) {
  return mask_paste_launch(mask_logits_dev, n, 1, Dm, Hm, Wm, nullptr, boxes_dev, offsets_dev, thr, out_dev, stream);
}

int roi3d_mask_paste_select(const float *mask_pred_dev, int n, int num_channels, int Dm, int Hm, int Wm,
                            const int64_t *channel_dev, const int32_t *boxes_dev, const int64_t *offsets_dev, float thr,
                            uint8_t *out_dev, void *stream) {
  return mask_paste_launch(mask_pred_dev, n, num_channels, Dm, Hm, Wm, channel_dev, boxes_dev, offsets_dev, thr, out_dev,
                           stream);
}

size_t roi3d_mask_target_workspace_bytes(const int32_t *crop_dhw_host, int n) {
  size_t doubles = 0;
  for (int i = 0; i < n; ++i) {
    const long long d = crop_dhw_host[i * 3], h = crop_dhw_host[i * 3 + 1], w = crop_dhw_host[i * 3 + 2];
    if (d > 0 && h > 0 && w > 0) doubles += 2 * (size_t)(d * h * w);
  }
  return doubles * sizeof(double) + 256 + (size_t)n * sizeof(MaskTargetJob);
}

int roi3d_mask_target(const uint8_t *gt_masks_dev, int G, int D, int H, int W, const int32_t *boxes_host,
                      const int64_t *gt_inds_host, int n, int Md, int Mh, int Mw, float *out_dev, void *workspace_dev,
                      size_t workspace_bytes, void *stream) {
  ROI3D_CHECK_ARG(n >= 0 && G >= 0 && D > 0 && H > 0 && W > 0 && Md > 0 && Mh > 0 && Mw > 0, "bad sizes");
  if (n == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(gt_masks_dev && boxes_host && gt_inds_host && out_dev && workspace_dev, "NULL pointer");
  ROI3D_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace_dev) & 255) == 0, "workspace must be 256-byte aligned");
  std::vector<MaskTargetJob> jobs((size_t)n);
  std::vector<int32_t> crops((size_t)n * 3);
  long long off = 0;
  for (int i = 0; i < n; ++i) {
    const int32_t *b = boxes_host + (size_t)i * 6;  // x1, y1, x2, y2, z1, z2 after `.astype(np.int32)`
    ROI3D_CHECK_ARG(gt_inds_host[i] >= 0 && gt_inds_host[i] < G, "proposal %d: gt index %lld out of [0,%d)", i,
                    (long long)gt_inds_host[i], G);
    ROI3D_CHECK_ARG(b[0] >= 0 && b[1] >= 0 && b[4] >= 0, "proposal %d starts at a negative coordinate", i);
    const int w = std::max(b[2] - b[0] + 1, 1), h = std::max(b[3] - b[1] + 1, 1), d = std::max(b[5] - b[4] + 1, 1);
    MaskTargetJob &j = jobs[(size_t)i];
    j.gt = (int)gt_inds_host[i], j.x1 = b[0], j.y1 = b[1], j.z1 = b[4];
    j.w = std::min(b[0] + w, W) - b[0], j.h = std::min(b[1] + h, H) - b[1], j.d = std::min(b[4] + d, D) - b[4];  // slice clipping
    j.ws_off = off;
    crops[(size_t)i * 3] = j.d, crops[(size_t)i * 3 + 1] = j.h, crops[(size_t)i * 3 + 2] = j.w;
    if (j.w > 0 && j.h > 0 && j.d > 0) off += 2LL * j.d * j.h * j.w;
  }
  const size_t need = roi3d_mask_target_workspace_bytes(crops.data(), n);
  if (workspace_bytes < need) {
    set_error("mask_target workspace too small: %zu < %zu", workspace_bytes, need);
    return ROI3D_ENOMEM;
  }
  cudaStream_t st = (cudaStream_t)stream;
  double *ws = static_cast<double *>(workspace_dev);
  MaskTargetJob *jobs_dev = reinterpret_cast<MaskTargetJob *>(static_cast<char *>(workspace_dev) + ((size_t)off * sizeof(double) + 255) / 256 * 256);
  ROI3D_CUDA(cudaMemcpyAsync(jobs_dev, jobs.data(), jobs.size() * sizeof(MaskTargetJob), cudaMemcpyHostToDevice, st));
  ROI3D_CUDA(cudaStreamSynchronize(st));  // `jobs` is a stack-owned pageable buffer
  mask_target_kernel<<<n, 256, 0, st>>>(gt_masks_dev, D, H, W, jobs_dev, Md, Mh, Mw, ws, out_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

}  // extern "C"

// Shared device-side pieces of the RoIAlign3D kernels (roi_align3d.cu, roi_align3d_stream.cu): launch parameters,
// per-item RoI decode, and the literal (reference-order) evaluation of one output bin.
#pragma once
#include <limits.h>

#include "common.cuh"

namespace roi3d {

struct LevelDev {
  const float *feats;
  float *grad;
  int D, H, W;
  float scale, scale_d;
};

struct RoiParams {
  LevelDev lv[ROI3D_MAX_LEVELS];
  int num_levels;
  float inv_finest;
  int B, C;
  const float *rois;
  int K;
  int PD, PH, PW;
  int sample_num;
  float *out;             // forward
  const float *grad_out;  // backward
  int64_t *lvls_out;
  const int *out_rows;    // forward: output row of RoI k (nullptr = k)
  int nchunk, nphg;
  long long total_items;
  int items_per_roi, ctas_per_roi;  // ring2 kernels: CTA -> (RoI, group of kWarps * items_per_warp sub-items)
  int items_per_warp;
  int bug_compat;
  int layout;             // ROI3D_NCDHW or ROI3D_NDHWC, the same for every level
};

constexpr int kWarps = 4;
constexpr int RXMAX = 40, RYMAX = 40, RZMAX = 32;
constexpr unsigned FULL = 0xffffffffu;

template <int CV>
__device__ __forceinline__ void ldv(const float *p, float (&v)[CV]) {
  if constexpr (CV == 4) {
    float4 t = __ldg(reinterpret_cast<const float4 *>(p));
    v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  } else if constexpr (CV == 2) {
    float2 t = __ldg(reinterpret_cast<const float2 *>(p));
    v[0] = t.x, v[1] = t.y;
  } else {
    v[0] = __ldg(p);
  }
}

template <int CV>
__device__ __forceinline__ void redv(float *p, const float (&v)[CV]) {
  if constexpr (CV == 4) {
    atomicAdd(reinterpret_cast<float4 *>(p), make_float4(v[0], v[1], v[2], v[3]));
  } else if constexpr (CV == 2) {
    atomicAdd(reinterpret_cast<float2 *>(p), make_float2(v[0], v[1]));
  } else {
    atomicAdd(p, v[0]);
  }
}

// Per-warp decode of one work item + RoI geometry.
struct Item {
  int k, krow, chunk, pd, ph0, rows, lvl, b;
  bool ok;
  Axis axw, axh, axd;
  LevelDev L;
};

// RoI k's geometry: reads its row of p.rois and fills it.k, lvl, L, b, ok and the three axes.
__device__ __forceinline__ void roi_geometry(const RoiParams &p, int k, Item &it) {
  it.k = k;
  const float *roi = p.rois + (long long)k * 7;
  float r[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) r[i] = __ldg(roi + i);
  it.lvl = p.num_levels > 1 ? roi_level(r, p.num_levels, p.inv_finest) : 0;
  it.L = p.lv[it.lvl];
  it.b = (int)r[0];
  it.ok = it.b >= 0 && it.b < p.B;
  it.axw = axis_setup(r[1], r[3], it.L.scale, p.PW, p.sample_num);
  it.axh = axis_setup(r[2], r[4], it.L.scale, p.PH, p.sample_num);
  it.axd = axis_setup(r[5], r[6], it.L.scale_d, p.PD, p.sample_num);
}

__device__ __forceinline__ Item decode_item(const RoiParams &p, long long item64, int ROWS) {
  Item it;
  unsigned item = (unsigned)item64;  // launchers guarantee total_items < 2^31: 32-bit div/mod only
  const unsigned phg = item % (unsigned)p.nphg;
  item /= (unsigned)p.nphg;
  it.pd = (int)(item % (unsigned)p.PD);
  item /= (unsigned)p.PD;
  it.chunk = (int)(item % (unsigned)p.nchunk);
  const int k = (int)(item / (unsigned)p.nchunk);
  it.krow = p.out_rows != nullptr ? __ldg(p.out_rows + k) : k;
  it.ph0 = (int)phg * ROWS;
  it.rows = min(ROWS, p.PH - it.ph0);
  roi_geometry(p, k, it);
  return it;
}

// Literal evaluation of one output bin for one channel, any layout (element strides sc / sz / sy / sx): the
// reference's sample loops with its corner-weight / FFMA-chain arithmetic (roi_align_kernel.cu:134-146 + SASS).
static __device__ float literal_bin_strided(const Axis &axw, const Axis &axh, const Axis &axd, int D, int H, int W,
                                     const float *fc, long long sz, long long sy, long long sx, int pd, int ph, int pw) {
  float acc = 0.0f;
  for (int iz = 0; iz < axd.S; ++iz) {
    const Tap tz = axis_tap(axis_coord(axd, pd, iz), D);
    for (int iy = 0; iy < axh.S; ++iy) {
      const Tap ty = axis_tap(axis_coord(axh, ph, iy), H);
      for (int ix = 0; ix < axw.S; ++ix) {
        const Tap tx = axis_tap(axis_coord(axw, pw, ix), W);
        if (!(tz.valid && ty.valid && tx.valid)) continue;  // contributes 0, still counted
        const float hxhy = __fmul_rn(tx.h, ty.h), lxhy = __fmul_rn(tx.l, ty.h);
        const float hxly = __fmul_rn(tx.h, ty.l), lxly = __fmul_rn(tx.l, ty.l);
        const float w1 = __fmul_rn(hxhy, tz.h), w2 = __fmul_rn(lxhy, tz.h), w3 = __fmul_rn(hxly, tz.h),
                    w4 = __fmul_rn(lxly, tz.h), w5 = __fmul_rn(hxhy, tz.l), w6 = __fmul_rn(lxhy, tz.l),
                    w7 = __fmul_rn(hxly, tz.l), w8 = __fmul_rn(lxly, tz.l);
        const long long zl = tz.low * sz, zh = tz.high * sz, yl = ty.low * sy, yh = ty.high * sy;
        const long long xl = tx.low * sx, xh = tx.high * sx;
        float t = __fmul_rn(w2, __ldg(fc + zl + yl + xh));
        t = __fmaf_rn(w1, __ldg(fc + zl + yl + xl), t);
        t = __fmaf_rn(w3, __ldg(fc + zl + yh + xl), t);
        t = __fmaf_rn(w4, __ldg(fc + zl + yh + xh), t);
        t = __fmaf_rn(w5, __ldg(fc + zh + yl + xl), t);
        t = __fmaf_rn(w6, __ldg(fc + zh + yl + xh), t);
        t = __fmaf_rn(w7, __ldg(fc + zh + yh + xl), t);
        t = __fmaf_rn(w8, __ldg(fc + zh + yh + xh), t);
        acc = __fadd_rn(acc, t);
      }
    }
  }
  return __fdiv_rn(acc, (float)(axd.S * axh.S * axw.S));
}


// ---------------------------------------------------------------------------------------------
// Generic (literal) evaluation of one output bin for CV channels per lane: the reference's sample
// loops and its exact corner-weight / FFMA-chain arithmetic (roi_align_kernel.cu:134-146 + SASS).
// ---------------------------------------------------------------------------------------------
template <int CV>
__device__ __forceinline__ void literal_bin_fwd(const Item &it, const float *fb, int C, int pd, int ph, int pw,
                                                float (&out)[CV]) {
  const int D = it.L.D, H = it.L.H, W = it.L.W;
  float acc[CV];
#pragma unroll
  for (int c = 0; c < CV; ++c) acc[c] = 0.0f;
  for (int iz = 0; iz < it.axd.S; ++iz) {
    Tap tz = axis_tap(axis_coord(it.axd, pd, iz), D);
    for (int iy = 0; iy < it.axh.S; ++iy) {
      Tap ty = axis_tap(axis_coord(it.axh, ph, iy), H);
      for (int ix = 0; ix < it.axw.S; ++ix) {
        Tap tx = axis_tap(axis_coord(it.axw, pw, ix), W);
        if (!(tz.valid && ty.valid && tx.valid)) continue;  // contributes 0, still counted
        const float hxhy = __fmul_rn(tx.h, ty.h), lxhy = __fmul_rn(tx.l, ty.h);
        const float hxly = __fmul_rn(tx.h, ty.l), lxly = __fmul_rn(tx.l, ty.l);
        const float w1 = __fmul_rn(hxhy, tz.h), w2 = __fmul_rn(lxhy, tz.h), w3 = __fmul_rn(hxly, tz.h),
                    w4 = __fmul_rn(lxly, tz.h), w5 = __fmul_rn(hxhy, tz.l), w6 = __fmul_rn(lxhy, tz.l),
                    w7 = __fmul_rn(hxly, tz.l), w8 = __fmul_rn(lxly, tz.l);
        const long long zl = (long long)tz.low * H, zh = (long long)tz.high * H;
        float f1[CV], f2[CV], f3[CV], f4[CV], f5[CV], f6[CV], f7[CV], f8[CV];
        ldv<CV>(fb + ((zl + ty.low) * W + tx.low) * C, f1);
        ldv<CV>(fb + ((zl + ty.low) * W + tx.high) * C, f2);
        ldv<CV>(fb + ((zl + ty.high) * W + tx.low) * C, f3);
        ldv<CV>(fb + ((zl + ty.high) * W + tx.high) * C, f4);
        ldv<CV>(fb + ((zh + ty.low) * W + tx.low) * C, f5);
        ldv<CV>(fb + ((zh + ty.low) * W + tx.high) * C, f6);
        ldv<CV>(fb + ((zh + ty.high) * W + tx.low) * C, f7);
        ldv<CV>(fb + ((zh + ty.high) * W + tx.high) * C, f8);
#pragma unroll
        for (int c = 0; c < CV; ++c) {
          float t = __fmul_rn(w2, f2[c]);
          t = __fmaf_rn(w1, f1[c], t);
          t = __fmaf_rn(w3, f3[c], t);
          t = __fmaf_rn(w4, f4[c], t);
          t = __fmaf_rn(w5, f5[c], t);
          t = __fmaf_rn(w6, f6[c], t);
          t = __fmaf_rn(w7, f7[c], t);
          t = __fmaf_rn(w8, f8[c], t);
          acc[c] = __fadd_rn(acc[c], t);
        }
      }
    }
  }
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);
#pragma unroll
  for (int c = 0; c < CV; ++c) out[c] = __fdiv_rn(acc[c], count);
}

template <int CV>
__device__ __forceinline__ void literal_bin_bwd(const Item &it, float *gb, int C, int pd, int ph, int pw,
                                                const float (&top)[CV]) {
  const int D = it.L.D, H = it.L.H, W = it.L.W;
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);
  for (int iz = 0; iz < it.axd.S; ++iz) {
    Tap tz = axis_tap(axis_coord(it.axd, pd, iz), D);
    for (int iy = 0; iy < it.axh.S; ++iy) {
      Tap ty = axis_tap(axis_coord(it.axh, ph, iy), H);
      for (int ix = 0; ix < it.axw.S; ++ix) {
        Tap tx = axis_tap(axis_coord(it.axw, pw, ix), W);
        if (!(tz.valid && ty.valid && tx.valid)) continue;
        const float hxhy = __fmul_rn(tx.h, ty.h), lxhy = __fmul_rn(tx.l, ty.h);
        const float hxly = __fmul_rn(tx.h, ty.l), lxly = __fmul_rn(tx.l, ty.l);
        const float w[8] = {__fmul_rn(hxhy, tz.h), __fmul_rn(lxhy, tz.h), __fmul_rn(hxly, tz.h),
                            __fmul_rn(lxly, tz.h), __fmul_rn(hxhy, tz.l), __fmul_rn(lxhy, tz.l),
                            __fmul_rn(hxly, tz.l), __fmul_rn(lxly, tz.l)};
        const long long zl = (long long)tz.low * H, zh = (long long)tz.high * H;
        const long long off[8] = {((zl + ty.low) * W + tx.low) * C,  ((zl + ty.low) * W + tx.high) * C,
                                  ((zl + ty.high) * W + tx.low) * C, ((zl + ty.high) * W + tx.high) * C,
                                  ((zh + ty.low) * W + tx.low) * C,  ((zh + ty.low) * W + tx.high) * C,
                                  ((zh + ty.high) * W + tx.low) * C, ((zh + ty.high) * W + tx.high) * C};
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float g[CV];
#pragma unroll
          for (int c = 0; c < CV; ++c) g[c] = __fdiv_rn(__fmul_rn(top[c], w[q]), count);
          redv<CV>(gb + off[q], g);
        }
      }
    }
  }
}

// Literal evaluation of a warp's whole (pd, ph-group) tile, kept out of line so that its register
// footprint does not inflate the fast kernels that only call it for oversized footprints.
template <int CV>
__device__ __noinline__ void literal_tile_fwd(const Item &it, const float *fb, int C, int PD, int PH, int PW,
                                              int c_base, bool active, float *out) {
  for (int r = 0; r < it.rows; ++r)
    for (int pw = 0; pw < PW; ++pw) {
      float v[CV];
      literal_bin_fwd<CV>(it, fb, C, it.pd, it.ph0 + r, pw, v);
      if (active) {
#pragma unroll
        for (int c = 0; c < CV; ++c)
          out[((((long long)it.krow * C + c_base + c) * PD + it.pd) * PH + it.ph0 + r) * PW + pw] = v[c];
      }
    }
}

// Persistent TMA-fed forward kernel (roi_align3d_stream.cu): applies to 7x7xPD outputs (PD <= 7) of channels-last
// levels with C % 64 == 0; RoIs it cannot take (footprint wider than its tiles, bins with more than four taps) are
// evaluated literally inside the same launch.
// Planar forward kernel (roi_align3d_planar.cu): lanes = output elements, one shared-memory plane per channel; reads
// NCDHW levels natively (and channels-last ones), 7- or 14-wide outputs.
// Private stream-ordered memory pool of the current device (per-call device scratch: no host sync, re-entrant across
// streams, pages stay with the pool between calls).
int stream_pool(cudaMemPool_t *out);

bool fwd_planar_ok(const RoiParams &p, int layout);
int launch_fwd_planar(RoiParams &p, int layout, cudaStream_t st);

// Planar backward (14-wide outputs, channels-last gradients): transposed stages, one vector red per (voxel, 4 channels).
bool bwd_planar_ok(const RoiParams &p);
int launch_bwd_planar(RoiParams &p, cudaStream_t st);

// Streamed backward (7 x 7 x PD outputs, channels-last gradients, C % 64 == 0): one vector red per voxel, RoI and channel.
bool bwd_stream_ok(const RoiParams &p);
int launch_bwd_stream(RoiParams &p, cudaStream_t st);

bool fwd_stream_ok(const RoiParams &p);
int launch_fwd_stream(RoiParams &p, cudaStream_t st);

// Deterministic backward (roi_align3d_det.cu; any output size, channels-last gradients): one CTA per gradient tile
// gathers the RoIs that meet it in ascending index and writes each voxel once -- overwriting it (accumulate = 0,
// every voxel of every level, no zero-fill needed) or adding its finished sum to the old value (accumulate = 1).
int launch_bwd_det(RoiParams &p, int accumulate, cudaStream_t st);

}  // namespace roi3d

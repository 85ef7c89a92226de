// RoIAlign3D forward / backward and the fused multi-level RoI extractor for B200 (sm_100a).
//
// Replaces (reference, /root/reference):
//   ROIAlignForward3D / bilinear_interpolate_3d          mmdet/ops/roi_align/src/roi_align_kernel.cu:214-291, :64-149
//   ROIAlignBackward3D / bilinear_interpolate_gradient_3d roi_align_kernel.cu:519-636, :383-442
//   SingleRoIExtractor.forward / map_roi_levels           mmdet/models/roi_extractors/single_level.py:58-104
//
// Design (see DESIGN.md section 3).  The reference evaluates every output bin independently: S^3
// trilinear samples x 8 scattered 4-byte loads (64 loads / 64 atomics per output element at S=2).
// Trilinear sampling, bin averaging, the out-of-range rule and the border clamp are all separable
// per axis, so here each RoI axis is reduced once to a small dense weight table
//     A_axis[p][v] = sum over the S samples i of bin p of ( h(p,i)*[v==low] + l(p,i)*[v==high] ),
// and the output is the tensor contraction  out[pd,ph,pw] = 1/count * sum_z A_d[pd][z] sum_y A_h[ph][y]
// sum_x A_w[pw][x] F[z,y,x].  One warp owns (RoI, 32*CV channels, pd, a group of ROWS ph-rows): lanes
// run over CHANNELS of the channels-last feature map, so every feature access is one coalesced
// 128*CV-byte line, all table lookups are warp-uniform shared-memory broadcasts, and there is no
// divergence.  Each feature row is contracted along x once (PW partial sums in registers), then
// folded into the ROWS x PW register accumulators with the combined z*y weight.  Results are
// transposed through a padded per-warp shared-memory tile so the [K,C,PD,PH,PW] output is written
// in contiguous runs with streaming stores.  The sample coordinates use exactly the rounding
// sequence of the compiled reference (common.cuh), so the tables -- and therefore which voxels are
// touched and with what weights -- are bit-identical; only the summation order differs (fp32, a few
// ulp; tolerance 1e-5 forward / 1e-4 backward per BASELINE.json).
//
// RoIs whose footprint exceeds the table capacity, and output widths other than 7/14, take the
// "generic" path: the same warp-per-(RoI, channel-vector) mapping evaluating the reference's sample
// loops literally (bit-exact against the oracle with contract=1).
#include <cuda.h>
#include <limits.h>

#include "common.cuh"

#include "roi_align3d_shared.cuh"

namespace roi3d {


// Per-warp weight tables in shared memory.
//   Dx[(x - xmin) * PWP + pw], Dy[(y - ymin) * 8 + r], Dz[z - zmin]; xlo/xhi[pw] relative to xmin.
template <int PW>
struct Tables {
  static constexpr int PWP = (PW + 3) / 4 * 4;
  static constexpr int FLOATS = RXMAX * PWP + RYMAX * 8 + RZMAX + 32 + RXMAX;
  float *Dx, *Dy, *Dz;
  int *xlo, *xhi;
  int *xany;
  int xmin, xmax, ymin, ymax, zmin, zmax;
  bool empty, fits;
  __device__ __forceinline__ void bind(float *sm) {
    Dx = sm;
    Dy = Dx + RXMAX * PWP;
    Dz = Dy + RYMAX * 8;
    xlo = reinterpret_cast<int *>(Dz + RZMAX);
    xhi = xlo + 16;
    xany = xhi + 16;
  }
};

template <int PW>
__device__ __forceinline__ void build_tables(Tables<PW> &T, const Item &it, int lane) {
  constexpr int PWP = Tables<PW>::PWP;
  // lanes [0,PW): x axis; lanes [16,16+rows): y axis; lane 31: z axis.
  int role = -1, pidx = 0, size = 1;
  Axis ax = it.axw;
  if (lane < PW) {
    role = 0, pidx = lane, size = it.L.W, ax = it.axw;
  } else if (lane >= 16 && lane < 16 + it.rows) {
    role = 1, pidx = it.ph0 + lane - 16, size = it.L.H, ax = it.axh;
  } else if (lane == 31) {
    role = 2, pidx = it.pd, size = it.L.D, ax = it.axd;
  }
  int lo = INT_MAX, hi = -1;
  if (role >= 0) {
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, pidx, i), size);
      if (t.valid) lo = min(lo, t.low), hi = max(hi, t.high);
    }
  }
  T.xmin = __reduce_min_sync(FULL, role == 0 ? lo : INT_MAX);
  T.xmax = __reduce_max_sync(FULL, role == 0 ? hi : -1);
  T.ymin = __reduce_min_sync(FULL, role == 1 ? lo : INT_MAX);
  T.ymax = __reduce_max_sync(FULL, role == 1 ? hi : -1);
  T.zmin = __reduce_min_sync(FULL, role == 2 ? lo : INT_MAX);
  T.zmax = __reduce_max_sync(FULL, role == 2 ? hi : -1);
  T.empty = T.xmax < T.xmin || T.ymax < T.ymin || T.zmax < T.zmin;
  T.fits = T.empty || ((T.xmax - T.xmin < RXMAX) && (T.ymax - T.ymin < RYMAX) && (T.zmax - T.zmin < RZMAX));
  if (T.empty || !T.fits) return;
  const int RX = T.xmax - T.xmin + 1, RY = T.ymax - T.ymin + 1, RZ = T.zmax - T.zmin + 1;
  for (int i = lane; i < RX * PWP; i += 32) T.Dx[i] = 0.0f;
  for (int i = lane; i < RY * 8; i += 32) T.Dy[i] = 0.0f;
  for (int i = lane; i < RZ; i += 32) T.Dz[i] = 0.0f;
  for (int i = lane; i < RX; i += 32) T.xany[i] = 0;
  __syncwarp();
  if (role >= 0) {
    float *tab = role == 0 ? T.Dx : role == 1 ? T.Dy : T.Dz;
    const int stride = role == 0 ? PWP : role == 1 ? 8 : 1;
    const int col = role == 0 ? lane : role == 1 ? lane - 16 : 0;
    const int mn = role == 0 ? T.xmin : role == 1 ? T.ymin : T.zmin;
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, pidx, i), size);
      if (t.valid) {
        tab[(t.low - mn) * stride + col] += t.h;
        tab[(t.high - mn) * stride + col] += t.l;
        if (role == 0) T.xany[t.low - mn] = 1, T.xany[t.high - mn] = 1;
      }
    }
    if (role == 0) {
      T.xlo[lane] = hi >= lo ? lo - T.xmin : 0;
      T.xhi[lane] = hi >= lo ? hi - T.xmin : -1;
    }
  }
  __syncwarp();
}


// Epilogue shared by the forward kernels: acc / count -> padded smem tile [bin][33] (lane = channel, no bank
// conflicts) -> global [channel][bin] in contiguous runs.  The flattened (channel, bin) walk advances by
// 32 elements per step with incremental offsets only (no division, no inner loop when NB >= 32).
template <int ROWS, int PW, int CV>
__device__ __forceinline__ void copy_out_tile(const float (&acc)[ROWS][PW][CV], float count, float *stage, int lane,
                                              int NB, int chunk, int C, float *out_tile, long long ch_stride) {
  // The reference divides by the sample count (roi_align_kernel.cu:288).  1/count is exact for the
  // power-of-two counts of fixed sample_num (2^3 = 8) and within one ulp otherwise; count == 0
  // (adaptive sampling of an empty RoI) still yields NaN (0 * inf) like the reference's 0/0.
  const float inv = __frcp_rn(count);
  const int col_stride = CV * (int)ch_stride;  // global distance between consecutive smem columns (< 2^31: checked)
#pragma unroll
  for (int c = 0; c < CV; ++c) {
    __syncwarp();
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int pw = 0; pw < PW; ++pw) stage[(r * PW + pw) * 33 + lane] = acc[r][pw][c] * inv;
    __syncwarp();
    const int cols = min(32, (C - chunk * 32 * CV - c + CV - 1) / CV);  // columns whose channel is < C
    float *dst = out_tile + ((long long)chunk * 32 * CV + c) * ch_stride;
    // one column (= one channel's contiguous run of NB floats) at a time, lanes along the run:
    // ceil(NB/32) predicated stores per column, no index arithmetic beyond two pointer bumps
    const float *sp = stage + lane * 33;
    float *gp = dst + lane;
#pragma unroll 4
    for (int cl = 0; cl < cols; ++cl) {
      if (lane < NB) __stcs(gp, sp[0]);
      if (lane + 32 < NB) __stcs(gp + 32, sp[32 * 33]);
      for (int bin = lane + 64; bin < NB; bin += 32) __stcs(gp + (bin - lane), sp[(bin - lane) * 33]);
      sp += 1;
      gp += col_stride;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Forward, channels-last, separable.  One warp per (k, chunk, pd, ph-group).
// ---------------------------------------------------------------------------------------------
template <int PW, int ROWS, int CV, int NXU>
__global__ void __launch_bounds__(kWarps * 32) roi_align3d_fwd_cl_kernel(const RoiParams p) {
  using TB = Tables<PW>;
  constexpr int PWP = TB::PWP;
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int WARP_FLOATS = ((STAGE > TB::FLOATS ? STAGE : TB::FLOATS) + 3) / 4 * 4;  // 16-byte aligned per warp
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *sm = smem_all + warp * WARP_FLOATS;
  const long long item = (long long)blockIdx.x * kWarps + warp;
  if (item >= p.total_items) return;  // warp-uniform; no block-level barrier is used below

  const Item it = decode_item(p, item, ROWS);
  const int C = p.C;
  if (p.lvls_out != nullptr && it.chunk == 0 && it.pd == 0 && it.ph0 == 0 && lane == 0) p.lvls_out[it.k] = it.lvl;

  int c_base = (it.chunk * 32 + lane) * CV;
  const bool active = c_base < C;
  if (!active) c_base = 0;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  const float *fb = it.L.feats + (long long)(it.ok ? it.b : 0) * vox * C + c_base;

  float acc[ROWS][PW][CV];
#pragma unroll
  for (int r = 0; r < ROWS; ++r)
#pragma unroll
    for (int w = 0; w < PW; ++w)
#pragma unroll
      for (int c = 0; c < CV; ++c) acc[r][w][c] = 0.0f;

  TB T;
  T.bind(sm);
  T.empty = true, T.fits = true;
  if (it.ok) build_tables<PW>(T, it, lane);
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);

  if (it.ok && !T.fits) {
    // footprint larger than the tables: literal evaluation, uncoalesced stores (rare path)
    literal_tile_fwd<CV>(it, fb, C, p.PD, p.PH, PW, c_base, active, p.out);
    return;
  }

  if (!T.empty) {
    const int RY = T.ymax - T.ymin + 1;
    // Per-warp constants of the x-contraction: for every bin pw its first NXU taps as (element
    // offset from the row start, weight); the index is clamped into the bin's support and the weight
    // forced to 0 past it, so the row loop below is branch-free.
    bool long_bins = false;
    int toff[PW][NXU];
    float tw[PW][NXU];
#pragma unroll
    for (int pw = 0; pw < PW; ++pw) {
      const int lo = T.xlo[pw];
      const int n = T.xhi[pw] - lo + 1;
      const int last = n > 0 ? n - 1 : 0;
      long_bins |= n > NXU;
#pragma unroll
      for (int j = 0; j < NXU; ++j) {
        const int jj = j < last ? j : last;
        toff[pw][j] = (lo + jj) * C;
        tw[pw][j] = j < n ? T.Dx[(lo + jj) * PWP + pw] : 0.0f;
      }
    }
    for (int z = T.zmin; z <= T.zmax; ++z) {
      const float wz = T.Dz[z - T.zmin];
      if (wz == 0.0f) continue;
      for (int yy = 0; yy < RY; ++yy) {
        float wr[ROWS];
        bool any = false;
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
          wr[r] = wz * T.Dy[yy * 8 + r];
          any |= wr[r] != 0.0f;
        }
        if (!any) continue;
        const float *rowp = fb + (((long long)z * it.L.H + (T.ymin + yy)) * it.L.W + T.xmin) * C;
        // x-contraction of this feature row.  Phase 1: all PW*NXU loads are issued before any is
        // consumed (independent, branch-free, in flight together); phase 2 (bins wider than NXU
        // taps; one warp-uniform test) finishes the long bins.
        float fr[PW][NXU][CV];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw)
#pragma unroll
          for (int j = 0; j < NXU; ++j) ldv<CV>(rowp + toff[pw][j], fr[pw][j]);
        float t1[PW][CV];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
#pragma unroll
          for (int c = 0; c < CV; ++c) t1[pw][c] = tw[pw][0] * fr[pw][0][c];
#pragma unroll
          for (int j = 1; j < NXU; ++j)
#pragma unroll
            for (int c = 0; c < CV; ++c) t1[pw][c] = fmaf(tw[pw][j], fr[pw][j][c], t1[pw][c]);
        }
        if (long_bins) {
#pragma unroll
          for (int pw = 0; pw < PW; ++pw) {
            const int lo = T.xlo[pw];
            const int n = T.xhi[pw] - lo + 1;
            const float *q = rowp + (long long)lo * C;
            const float *wq = T.Dx + lo * PWP + pw;
#pragma unroll 1
            for (int j = NXU; j < n; ++j) {
              float f[CV];
              ldv<CV>(q + (long long)j * C, f);
              const float w = wq[j * PWP];
#pragma unroll
              for (int c = 0; c < CV; ++c) t1[pw][c] = fmaf(w, f[c], t1[pw][c]);
            }
          }
        }
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
          if (wr[r] != 0.0f) {
#pragma unroll
            for (int pw = 0; pw < PW; ++pw)
#pragma unroll
              for (int c = 0; c < CV; ++c) acc[r][pw][c] = fmaf(wr[r], t1[pw][c], acc[r][pw][c]);
          }
        }
      }
    }
  }

  // ---- epilogue: divide by the sample count, transpose through smem, stream out ----
  const int NB = it.rows * PW;
  float *stage = sm;  // aliases the tables: all table reads are done
  const long long out_base = (((long long)it.krow * C) * p.PD + it.pd) * p.PH * PW + (long long)it.ph0 * PW;
  const long long ch_stride = (long long)p.PD * p.PH * PW;
  copy_out_tile<ROWS, PW, CV>(acc, count, stage, lane, NB, it.chunk, C, p.out + out_base, ch_stride);
}

// ---------------------------------------------------------------------------------------------
// Forward, channels-last, separable, rows staged through a per-warp cp.async ring.
//
// Same work split and arithmetic as roi_align3d_fwd_cl_kernel, but the feature rows a warp needs
// ([xmin..xmax] x 32*CV channels of one (z,y) row) are copied global->shared with 16-byte cp.async
// (LDGSTS, no register staging) NS-1 rows ahead of the row being contracted.  The loads of the next
// rows are in flight while the current row is reduced, each voxel of the row is fetched once instead
// of once per tap, and the register file no longer holds the taps, which raises occupancy.
// Ring capacity per warp is RXR voxels per row; wider footprints take the literal path.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB>
__global__ void __launch_bounds__(kWarps * 32, MINB) roi_align3d_fwd_ring_kernel(const RoiParams p) {
  using TB = Tables<PW>;
  constexpr int PWP = TB::PWP;
  constexpr int VOX = 32 * CV;                 // floats per voxel-chunk
  constexpr int LPV = VOX / 4;                 // lanes (16 B each) per voxel-chunk
  constexpr int VPI = 32 / LPV;                // voxel-chunks copied per warp instruction
  constexpr int STRIDE = (RXR + 2) * VOX;      // floats per ring stage (two zero pad voxels)
  constexpr int RING = NS * STRIDE;            // floats
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int LISTS = 384;                   // ylist[40] + zlist[32] bytes (pad to 80) + yoff[40] + zoff[32] ints
  constexpr int RING_OR_STAGE = RING > STAGE ? RING : STAGE;
  constexpr int WARP_FLOATS = (TB::FLOATS + LISTS / 4 + RING_OR_STAGE + 3) / 4 * 4;
  static_assert(LPV <= 32 && VPI >= 1, "voxel chunk wider than a warp copy");
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *sm = smem_all + warp * WARP_FLOATS;
  const long long item = (long long)blockIdx.x * kWarps + warp;
  if (item >= p.total_items) return;  // warp-uniform; no block-level barrier is used below

  const Item it = decode_item(p, item, ROWS);
  const int C = p.C;
  if (p.lvls_out != nullptr && it.chunk == 0 && it.pd == 0 && it.ph0 == 0 && lane == 0) p.lvls_out[it.k] = it.lvl;

  int c_base = (it.chunk * 32 + lane) * CV;
  const bool active = c_base < C;
  if (!active) c_base = 0;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  const float *fb_roi = it.L.feats + (long long)(it.ok ? it.b : 0) * vox * C;
  const float *fb = fb_roi + c_base;

  TB T;
  T.bind(sm);
  unsigned char *ylist = reinterpret_cast<unsigned char *>(sm + ((TB::FLOATS + 3) / 4 * 4));
  unsigned char *zlist = ylist + 40;
  int *yoff = reinterpret_cast<int *>(ylist + 80);
  int *zoff = yoff + 40;
  float *ring = sm + ((TB::FLOATS + 3) / 4 * 4) + LISTS / 4;
  T.empty = true, T.fits = true;
  if (it.ok) build_tables<PW>(T, it, lane);
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);
  const int RX = T.xmax - T.xmin + 1;
  // the 16-byte copies need the chunk to lie inside C and be 16-byte aligned: C % 4 == 0 is checked by
  // the dispatcher; a partial last chunk (C not a multiple of 32*CV) copies only the lanes inside C.

  if (it.ok && !T.empty && (!T.fits || RX > RXR)) {
    // footprint larger than the tables / the ring: literal evaluation, uncoalesced stores (rare path)
    literal_tile_fwd<CV>(it, fb, C, p.PD, p.PH, PW, c_base, active, p.out);
    return;
  }

  float acc[ROWS][PW][CV];
#pragma unroll
  for (int r = 0; r < ROWS; ++r)
#pragma unroll
    for (int w = 0; w < PW; ++w)
#pragma unroll
      for (int c = 0; c < CV; ++c) acc[r][w][c] = 0.0f;

  if (!T.empty) {
    // ---- compact lists of the z slices / y rows that carry weight for this (pd, ph-group) ----
    const int RY = T.ymax - T.ymin + 1, RZ = T.zmax - T.zmin + 1;
    int ny = 0, nz = 0;
    for (int y0 = 0; y0 < RY; y0 += 32) {
      const int yy = y0 + lane;
      bool a = false;
      if (yy < RY) {
#pragma unroll
        for (int r = 0; r < ROWS; ++r) a |= T.Dy[yy * 8 + r] != 0.0f;
      }
      const unsigned bal = __ballot_sync(FULL, a);
      if (a) ylist[ny + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)yy;
      ny += __popc(bal);
    }
    {
      const bool a = lane < RZ && T.Dz[lane] != 0.0f;
      const unsigned bal = __ballot_sync(FULL, a);
      if (a) zlist[__popc(bal & ((1u << lane) - 1u))] = (unsigned char)lane;
      nz = __popc(bal);
    }
    __syncwarp();
    const int nrows = ny * nz;

    // per-warp constants of the x-contraction: for every bin pw its first NXU taps (weight forced to 0
    // past the bin's support).  Ring rows carry two zero-filled pad voxels after the RX real ones, so a
    // zero-weight tap always reads initialised shared memory and tap offsets are compile-time constants.
    bool long_bins = false;
    int soff[PW];
    float tw[PW][NXU];
#pragma unroll
    for (int pw = 0; pw < PW; ++pw) {
      const int lo = T.xlo[pw];
      const int n = T.xhi[pw] - lo + 1;
      long_bins |= n > NXU;
      soff[pw] = lo * VOX + lane * CV;
#pragma unroll
      for (int j = 0; j < NXU; ++j) tw[pw][j] = j < n ? T.Dx[(lo + j) * PWP + pw] : 0.0f;
    }
    static_assert(NXU <= 3, "pad voxels cover taps lo+1, lo+2 only");
    for (int sidx = 0; sidx < NS; ++sidx) {
      float *padp = ring + sidx * STRIDE + RX * VOX;
      for (int i = lane; i < 2 * VOX; i += 32) padp[i] = 0.0f;
    }
    __syncwarp();

    // copy geometry: lane -> (voxel within the instruction, 16-byte piece of the voxel chunk)
    const int cv_v = lane / LPV, cv_p = lane % LPV;
    const int ch_piece = it.chunk * VOX + cv_p * 4;          // first channel of this lane's 16 bytes
    const bool piece_ok = ch_piece + 4 <= C;
    // producer cursor (row to prefetch next): rows are visited y-major, z-minor, so that all z slices of
    // one y row are contracted along x back to back and the y-stage runs once per y row.
    const long long row_elems = (long long)it.L.W * C;
    const long long slice_elems = (long long)it.L.H * row_elems;
    const float *src0 = fb_roi + ((long long)T.zmin * it.L.H + T.ymin) * row_elems + (long long)T.xmin * C + ch_piece +
                        (long long)cv_v * C;
    float *dst0 = ring + cv_p * 4 + cv_v * VOX;
    // row offsets in units of 4 floats (16 B; C % 4 == 0), < 2^31 for any level the dispatcher accepts
    for (int i = lane; i < nz; i += 32) zoff[i] = (int)(((long long)zlist[i] * slice_elems) >> 2);
    for (int i = lane; i < ny; i += 32) yoff[i] = (int)(((long long)ylist[i] * row_elems) >> 2);
    __syncwarp();
    int pz = 0, py = 0, pstage = 0;
    auto issue = [&]() {
      const float *src = src0 + ((long long)(zoff[pz] + yoff[py]) << 2);
      float *dst = dst0 + pstage * STRIDE;
      if (piece_ok) {
#pragma unroll 2
        for (int v = cv_v; v < RX; v += VPI) {
          cp_async16(dst, src);
          dst += VPI * VOX, src += (long long)VPI * C;
        }
      }
      cp_async_commit();
      if (++pz == nz) pz = 0, ++py;
      if (++pstage == NS) pstage = 0;
    };
#pragma unroll
    for (int r = 0; r < NS - 1; ++r) {
      if (r < nrows) issue();
      else cp_async_commit();
    }
    int cstage = 0, r = 0;
    for (int yi = 0; yi < ny; ++yi) {
      float t1[PW][CV];
#pragma unroll
      for (int pw = 0; pw < PW; ++pw)
#pragma unroll
        for (int c = 0; c < CV; ++c) t1[pw][c] = 0.0f;
      for (int zi = 0; zi < nz; ++zi, ++r) {
        cp_async_wait<NS - 2>();
        __syncwarp();
        const float wz = T.Dz[zlist[zi]];
        const float *row = ring + cstage * STRIDE;
        if (++cstage == NS) cstage = 0;
        float tz[PW][CV];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          const float *q = row + soff[pw];
#pragma unroll
          for (int j = 0; j < NXU; ++j) {
            float f[CV];
            if constexpr (CV == 4) {
              const float4 t = *reinterpret_cast<const float4 *>(q + j * VOX);
              f[0] = t.x, f[1] = t.y, f[2] = t.z, f[3] = t.w;
            } else if constexpr (CV == 2) {
              const float2 t = *reinterpret_cast<const float2 *>(q + j * VOX);
              f[0] = t.x, f[1] = t.y;
            } else {
              f[0] = q[j * VOX];
            }
#pragma unroll
            for (int c = 0; c < CV; ++c) tz[pw][c] = j == 0 ? tw[pw][0] * f[c] : fmaf(tw[pw][j], f[c], tz[pw][c]);
          }
        }
        if (long_bins) {  // one warp-uniform test per row; bins wider than NXU taps are rare
#pragma unroll
          for (int pw = 0; pw < PW; ++pw) {
            const int lo = T.xlo[pw];
            const int n = T.xhi[pw] - lo + 1;
            const float *q = row + soff[pw];
            const float *wq = T.Dx + lo * PWP + pw;
#pragma unroll 1
            for (int j = NXU; j < n; ++j) {
              const float w = wq[j * PWP];
#pragma unroll
              for (int c = 0; c < CV; ++c) tz[pw][c] = fmaf(w, q[j * VOX + c], tz[pw][c]);
            }
          }
        }
#pragma unroll
        for (int pw = 0; pw < PW; ++pw)
#pragma unroll
          for (int c = 0; c < CV; ++c) t1[pw][c] = fmaf(wz, tz[pw][c], t1[pw][c]);
        __syncwarp();
        if (r + NS - 1 < nrows) issue();
        else cp_async_commit();
      }
      // y-stage, once per feature row index y
      const int yy = ylist[yi];
      float wy[8];
      {
        const float4 a = *reinterpret_cast<const float4 *>(T.Dy + yy * 8);
        const float4 b4 = *reinterpret_cast<const float4 *>(T.Dy + yy * 8 + 4);
        wy[0] = a.x, wy[1] = a.y, wy[2] = a.z, wy[3] = a.w, wy[4] = b4.x, wy[5] = b4.y, wy[6] = b4.z, wy[7] = b4.w;
      }
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) {
        if (wy[rr] != 0.0f) {
#pragma unroll
          for (int pw = 0; pw < PW; ++pw)
#pragma unroll
            for (int c = 0; c < CV; ++c) acc[rr][pw][c] = fmaf(wy[rr], t1[pw][c], acc[rr][pw][c]);
        }
      }
    }
    cp_async_wait<0>();
  }

  // ---- epilogue: divide by the sample count, transpose through smem, stream out ----
  const int NB = it.rows * PW;
  float *stage = ring;  // the ring is drained
  const long long out_base = (((long long)it.krow * C) * p.PD + it.pd) * p.PH * PW + (long long)it.ph0 * PW;
  const long long ch_stride = (long long)p.PD * p.PH * PW;
  copy_out_tile<ROWS, PW, CV>(acc, count, stage, lane, NB, it.chunk, C, p.out + out_base, ch_stride);
}

// ---- TMA bulk-copy (cp.async.bulk, SASS UBLKCP) + mbarrier helpers for the per-warp row ring ----
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned mbar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(mbar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
  unsigned ok = 0;
  for (int spin = 0; spin < (1 << 24); ++spin) {  // bounded: a byte-count mismatch traps instead of hanging the GPU
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok)
        : "r"(mbar), "r"(parity)
        : "memory");
    if (ok) return;
  }
  __trap();
}

// One TMA descriptor per pyramid level: the channels-last level seen as a 2-D tensor [voxel][channel], box =
// (RXR voxels) x (one warp's channel chunk).  A whole feature row of the RoI footprint is then ONE
// cp.async.bulk.tensor instruction issued by one lane (SASS UTMALDG) instead of RX/2 LDGSTS per warp.
struct alignas(64) TmapSet {
  CUtensorMap m[ROI3D_MAX_LEVELS];
};
__device__ __forceinline__ void tma_load_2d(unsigned dst, const void *tmap, int c0, int c1, unsigned mbar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
      "l"(tmap), "r"(c0), "r"(c1), "r"(mbar)
      : "memory");
}

// Shared-memory layout of the ring2 kernel, shared by the kernel and its launcher.
template <int PW, int ROWS, int CV, int NS, int RXR, int BULK>
struct Ring2Layout {
  static constexpr int VOX = 32 * CV;
  static constexpr int STRIDE = (RXR + 2) * VOX;
  static constexpr int RING = NS * STRIDE;
  static constexpr int STAGE = ROWS * PW * 33;
  static constexpr int LISTS = BULK == 2 ? 512 : 480;  // bytes; TMA destinations must be 128-byte aligned
  static constexpr int ALIGN = BULK == 2 ? 32 : 4;     // floats
  static constexpr int RING_OR_STAGE = RING > STAGE ? RING : STAGE;
  static constexpr int WARP_FLOATS = (LISTS / 4 + RING_OR_STAGE + ALIGN - 1) / ALIGN * ALIGN;
  static constexpr int SH_FLOATS = RXMAX * Tables<PW>::PWP + RYMAX * 16 + 40 * 16 + 32 + 3 * 32 * 2 + 16;
  static constexpr int SH_PAD = (SH_FLOATS + ALIGN - 1) / ALIGN * ALIGN;
  static constexpr size_t BYTES = ((size_t)SH_PAD + (size_t)kWarps * WARP_FLOATS) * sizeof(float);
};

// ---------------------------------------------------------------------------------------------
// Forward ring kernel with CTA-shared per-RoI tables: the four warps of a CTA always work on the same
// RoI (grid = K x ceil(items per RoI / 4)), so the axis tables are built once per CTA by three warps in
// parallel (x, y and z bins) instead of once per warp, and sit once in shared memory.  Everything after
// the table build is the per-warp pipeline of roi_align3d_fwd_ring_kernel.
// ---------------------------------------------------------------------------------------------
constexpr int RZMAX2 = 40;
template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB, int BULK, bool F2 = false, bool MULTI = false>
__global__ void __launch_bounds__(kWarps * 32, MINB)
    roi_align3d_fwd_ring2_kernel(const RoiParams p, const __grid_constant__ TmapSet tm) {
  static_assert(!F2 || CV == 2, "packed f32x2 arithmetic pairs the two channels of a lane");
  using TB = Tables<PW>;
  using LY = Ring2Layout<PW, ROWS, CV, NS, RXR, BULK>;
  constexpr int PWP = TB::PWP;
  constexpr int VOX = 32 * CV;                 // floats per voxel-chunk
  constexpr int LPV = VOX / 4;                 // lanes (16 B each) per voxel-chunk
  constexpr int VPI = 32 / LPV;                // voxel-chunks copied per warp instruction
  constexpr int STRIDE = LY::STRIDE;           // floats per ring stage (two zero pad voxels)
  constexpr int LISTS = LY::LISTS;             // ylist[40] + zlist[40] bytes + yoff[40] + zoff[40] ints + 8 mbarriers
  constexpr int WARP_FLOATS = LY::WARP_FLOATS;
  constexpr int PP = 16;                       // padded row length of the shared y / z tables (PH, PD <= 16)
  static_assert(LPV <= 32 && VPI >= 1, "voxel chunk wider than a warp copy");
  extern __shared__ __align__(128) float smem_r2[];
  float *smem_all = smem_r2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  // ---- CTA-shared per-RoI tables (all warps of a CTA work on the same RoI) ----
  float *SDx = smem_all;                       // [x - xmin][PWP]
  float *SDy = SDx + RXMAX * PWP;              // [y - ymin][PP], all PH rows
  float *SDz = SDy + RYMAX * PP;               // [z - zmin][PP], all PD slices
  int *Sxlo = reinterpret_cast<int *>(SDz + RZMAX2 * PP);
  int *Sxhi = Sxlo + 16;
  int *Srng = Sxhi + 16;                       // [3 axes][32 roles][lo, hi]
  int *Sbox = Srng + 3 * 32 * 2;               // xmin, xmax, ymin, ymax, zmin, zmax
  float *sm = smem_all + LY::SH_PAD + warp * WARP_FLOATS;

  // CTA -> (RoI k, group of kWarps * p.items_per_warp consecutive sub-items); warp w takes sub-items
  // first + w, first + w + kWarps, ...  Sub-item order: channel chunk fastest, then pd, then ph-group, so with
  // nchunk == kWarps a warp keeps its channel chunk and walks the pd slices of one RoI.
  const int k = blockIdx.x / p.ctas_per_roi;
  const int items_per_warp = MULTI ? p.items_per_warp : 1;
  const int first = (blockIdx.x - k * p.ctas_per_roi) * kWarps * items_per_warp;
  Item it;
  {
    it.k = k;
    it.krow = p.out_rows != nullptr ? __ldg(p.out_rows + k) : k;
    it.pd = 0, it.chunk = 0, it.ph0 = 0, it.rows = 0;
    float r[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)k * 7 + i);
    it.lvl = p.num_levels > 1 ? roi_level(r, p.num_levels, p.inv_finest) : 0;
    it.L = p.lv[it.lvl];
    it.b = (int)r[0];
    it.ok = it.b >= 0 && it.b < p.B;
    it.axw = axis_setup(r[1], r[3], it.L.scale, p.PW, p.sample_num);
    it.axh = axis_setup(r[2], r[4], it.L.scale, p.PH, p.sample_num);
    it.axd = axis_setup(r[5], r[6], it.L.scale_d, p.PD, p.sample_num);
  }
  const int C = p.C;
  if (p.lvls_out != nullptr && blockIdx.x == k * p.ctas_per_roi && tid == 0) p.lvls_out[k] = it.lvl;

  // role threads: warp 0 lanes [0,PW) -> x bins, warp 1 lanes [0,PH) -> y bins, warp 2 lanes [0,PD) -> z bins
  const int role = (warp == 0 && lane < PW) ? 0 : (warp == 1 && lane < p.PH) ? 1 : (warp == 2 && lane < p.PD) ? 2 : -1;
  const Axis ax = role == 1 ? it.axh : role == 2 ? it.axd : it.axw;
  const int asize = role == 1 ? it.L.H : role == 2 ? it.L.D : it.L.W;
  int lo = INT_MAX, hi = -1;
  if (role >= 0 && it.ok) {
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, lane, i), asize);
      if (t.valid) lo = min(lo, t.low), hi = max(hi, t.high);
    }
  }
  if (warp < 3) {
    const int mn = __reduce_min_sync(FULL, role >= 0 ? lo : INT_MAX);
    const int mx = __reduce_max_sync(FULL, role >= 0 ? hi : -1);
    if (lane == 0) Sbox[warp * 2] = mn, Sbox[warp * 2 + 1] = mx;
  }
  __syncthreads();
  TB T;
  T.Dx = SDx, T.xlo = Sxlo, T.xhi = Sxhi;
  T.xmin = Sbox[0], T.xmax = Sbox[1], T.ymin = Sbox[2], T.ymax = Sbox[3], T.zmin = Sbox[4], T.zmax = Sbox[5];
  T.empty = !it.ok || T.xmax < T.xmin || T.ymax < T.ymin || T.zmax < T.zmin;
  T.fits = T.empty || ((T.xmax - T.xmin < RXMAX) && (T.ymax - T.ymin < RYMAX) && (T.zmax - T.zmin < RZMAX2));
  const int RX = T.xmax - T.xmin + 1;
  if (!T.empty && T.fits) {
    const int RY = T.ymax - T.ymin + 1, RZ = T.zmax - T.zmin + 1;
    for (int i = tid; i < RX * PWP; i += kWarps * 32) SDx[i] = 0.0f;
    for (int i = tid; i < RY * PP; i += kWarps * 32) SDy[i] = 0.0f;
    for (int i = tid; i < RZ * PP; i += kWarps * 32) SDz[i] = 0.0f;
  }
  __syncthreads();
  if (!T.empty && T.fits && role >= 0) {
    float *tab = role == 0 ? SDx : role == 1 ? SDy : SDz;
    const int stride = role == 0 ? PWP : PP;
    const int mn = role == 0 ? T.xmin : role == 1 ? T.ymin : T.zmin;
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, lane, i), asize);
      if (t.valid) {
        tab[(t.low - mn) * stride + lane] += t.h;
        tab[(t.high - mn) * stride + lane] += t.l;
      }
    }
    if (role == 0) {
      Sxlo[lane] = hi >= lo ? lo - T.xmin : 0;
      Sxhi[lane] = hi >= lo ? hi - T.xmin : -1;
    }
  }
  __syncthreads();
  // no block-level barriers below: warps run their sub-items independently

  unsigned char *ylist = reinterpret_cast<unsigned char *>(sm);
  unsigned char *zlist = ylist + 40;
  int *yoff = reinterpret_cast<int *>(ylist + 80);
  int *zoff = yoff + 40;
  float *ring = sm + LISTS / 4;
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);
  const bool use_ring = !T.empty && T.fits && RX <= RXR;

  // per-warp constants of the x-contraction (RoI-level, shared by all sub-items of the warp): for every bin pw
  // its first NXU taps (weight forced to 0 past the bin's support).  Ring rows carry two zero-filled pad voxels
  // after the RX real ones, so a zero-weight tap always reads initialised shared memory and tap offsets are
  // compile-time constants.
  bool long_bins = false;
  int soff[PW];
  float tw[PW][NXU];
  static_assert(NXU <= 3, "pad voxels cover taps lo+1, lo+2 only");
#pragma unroll
  for (int pw = 0; pw < PW; ++pw) {
    const int lo = use_ring ? T.xlo[pw] : 0;
    const int n = use_ring ? T.xhi[pw] - lo + 1 : 0;
    long_bins |= n > NXU;
    soff[pw] = lo * VOX + lane * CV;
#pragma unroll
    for (int j = 0; j < NXU; ++j) tw[pw][j] = j < n ? T.Dx[(lo + j) * PWP + pw] : 0.0f;
  }
  const unsigned mbar0 = (unsigned)__cvta_generic_to_shared(ylist + 416);
  const unsigned ring_s = (unsigned)__cvta_generic_to_shared(ring);
  if constexpr (BULK) {
    static_assert(NS <= 8, "eight mbarriers per warp");
    if (lane == 0) {
      for (int sidx = 0; sidx < NS; ++sidx) mbar_init(mbar0 + sidx * 8, 1);
      mbar_fence_init();
    }
    __syncwarp();
  }
  int pstage = 0, cstage = 0;  // ring cursors persist across sub-items (every issued row is consumed)
  unsigned cpar = 0;

  for (int g = 0; g < items_per_warp; ++g) {
  const int sub = first + g * kWarps + warp;
  if (sub >= p.items_per_roi) break;
  {
    unsigned item = (unsigned)sub;
    it.chunk = (int)(item % (unsigned)p.nchunk);
    item /= (unsigned)p.nchunk;
    it.pd = (int)(item % (unsigned)p.PD);
    const unsigned phg = item / (unsigned)p.PD;
    it.ph0 = (int)phg * ROWS;
    it.rows = min(ROWS, p.PH - it.ph0);
  }
  int c_base = (it.chunk * 32 + lane) * CV;
  const bool active = c_base < C;
  if (!active) c_base = 0;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  const float *fb_roi = it.L.feats + (long long)(it.ok ? it.b : 0) * vox * C;
  const float *fb = fb_roi + c_base;
  // the 16-byte copies need the chunk to lie inside C and be 16-byte aligned: C % 4 == 0 is checked by
  // the dispatcher; a partial last chunk (C not a multiple of 32*CV) copies only the lanes inside C.

  if (!T.empty && (!T.fits || RX > RXR)) {
    // footprint larger than the tables / the ring: literal evaluation, uncoalesced stores (rare path)
    literal_tile_fwd<CV>(it, fb, C, p.PD, p.PH, PW, c_base, active, p.out);
    continue;
  }

  float acc[ROWS][PW][CV];
#pragma unroll
  for (int r = 0; r < ROWS; ++r)
#pragma unroll
    for (int w = 0; w < PW; ++w)
#pragma unroll
      for (int c = 0; c < CV; ++c) acc[r][w][c] = 0.0f;

  if (!T.empty) {
    // ---- compact lists of the z slices / y rows that carry weight for this (pd, ph-group) ----
    const int RY = T.ymax - T.ymin + 1, RZ = T.zmax - T.zmin + 1;
    int ny = 0, nz = 0;
    for (int y0 = 0; y0 < RY; y0 += 32) {
      const int yy = y0 + lane;
      bool a = false;
      if (yy < RY) {
#pragma unroll
        for (int r = 0; r < ROWS; ++r) a |= (r < it.rows) && SDy[yy * PP + it.ph0 + r] != 0.0f;
      }
      const unsigned bal = __ballot_sync(FULL, a);
      if (a) ylist[ny + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)yy;
      ny += __popc(bal);
    }
    for (int z0 = 0; z0 < RZ; z0 += 32) {
      const int zz = z0 + lane;
      const bool a = zz < RZ && SDz[zz * PP + it.pd] != 0.0f;
      const unsigned bal = __ballot_sync(FULL, a);
      if (a) zlist[nz + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)zz;
      nz += __popc(bal);
    }
    __syncwarp();
    const int nrows = ny * nz;

    for (int sidx = 0; sidx < NS; ++sidx) {
      // (TMA mode: the box always fills slots [0, RXR); taps past RX then read neighbouring voxels with weight 0)
      float *padp = ring + sidx * STRIDE + (BULK == 2 ? RXR : RX) * VOX;
      for (int i = lane; i < 2 * VOX; i += 32) padp[i] = 0.0f;
    }
    __syncwarp();

    // copy geometry: lane -> (voxel within the instruction, 16-byte piece of the voxel chunk)
    const int cv_v = lane / LPV, cv_p = lane % LPV;
    const int ch_piece = it.chunk * VOX + cv_p * 4;          // first channel of this lane's 16 bytes
    const bool piece_ok = ch_piece + 4 <= C;
    // producer cursor (row to prefetch next): rows are visited y-major, z-minor, so that all z slices of
    // one y row are contracted along x back to back and the y-stage runs once per y row.
    const long long row_elems = (long long)it.L.W * C;
    const long long slice_elems = (long long)it.L.H * row_elems;
    const float *src0 = fb_roi + ((long long)T.zmin * it.L.H + T.ymin) * row_elems + (long long)T.xmin * C + ch_piece +
                        (long long)cv_v * C;
    float *dst0 = ring + cv_p * 4 + cv_v * VOX;
    // row offsets in units of 4 floats (16 B; C % 4 == 0), < 2^31 for any level the dispatcher accepts
    if constexpr (BULK == 2) {  // TMA coordinates are voxel indices
      for (int i = lane; i < nz; i += 32) zoff[i] = (int)zlist[i] * it.L.H * it.L.W;
      for (int i = lane; i < ny; i += 32) yoff[i] = (int)ylist[i] * it.L.W;
    } else {
      for (int i = lane; i < nz; i += 32) zoff[i] = (int)(((long long)zlist[i] * slice_elems) >> 2);
      for (int i = lane; i < ny; i += 32) yoff[i] = (int)(((long long)ylist[i] * row_elems) >> 2);
    }
    __syncwarp();
    const int vbase = (((it.ok ? it.b : 0) * it.L.D + T.zmin) * it.L.H + T.ymin) * it.L.W + T.xmin;
    const void *tmap = &tm.m[it.lvl];
    int pz = 0, py = 0;
    // BULK == 1: lane v issues one cp.async.bulk of this warp's channel chunk of voxel v (<= 128*CV bytes,
    // contiguous); BULK == 2: one tensor copy per row; completion is counted in bytes on the stage's mbarrier.
    const unsigned chunk_bytes = (unsigned)min(VOX, C - it.chunk * VOX) * 4u;
    const float *srcb = fb_roi + ((long long)T.zmin * it.L.H + T.ymin) * row_elems + (long long)T.xmin * C +
                        (long long)it.chunk * VOX;
    auto issue = [&]() {
      if constexpr (BULK == 2) {
        if (lane == 0) {
          const unsigned mb = mbar0 + pstage * 8;
          mbar_expect_tx(mb, (unsigned)(RXR * VOX * 4));
          tma_load_2d(ring_s + (unsigned)(pstage * STRIDE) * 4u, tmap, it.chunk * VOX, vbase + zoff[pz] + yoff[py], mb);
        }
      } else if constexpr (BULK == 1) {
        const float *src = srcb + ((long long)(zoff[pz] + yoff[py]) << 2);
        const unsigned mb = mbar0 + pstage * 8;
        if (lane == 0) mbar_expect_tx(mb, (unsigned)RX * chunk_bytes);
        __syncwarp();
        for (int v = lane; v < RX; v += 32)
          bulk_g2s(ring_s + (unsigned)(pstage * STRIDE + v * VOX) * 4u, src + (long long)v * C, chunk_bytes, mb);
      } else {
        const float *src = src0 + ((long long)(zoff[pz] + yoff[py]) << 2);
        float *dst = dst0 + pstage * STRIDE;
        if (piece_ok) {
#pragma unroll 2
          for (int v = cv_v; v < RX; v += VPI) {
            cp_async16(dst, src);
            dst += VPI * VOX, src += (long long)VPI * C;
          }
        }
        cp_async_commit();
      }
      if (++pz == nz) pz = 0, ++py;
      if (++pstage == NS) pstage = 0;
    };
#pragma unroll
    for (int r = 0; r < NS - 1; ++r) {
      if (r < nrows) issue();
      else if constexpr (!BULK) cp_async_commit();
    }
    int r = 0;
    for (int yi = 0; yi < ny; ++yi) {
      float t1[PW][CV];
#pragma unroll
      for (int pw = 0; pw < PW; ++pw)
#pragma unroll
        for (int c = 0; c < CV; ++c) t1[pw][c] = 0.0f;
      for (int zi = 0; zi < nz; ++zi, ++r) {
        if constexpr (BULK) {
          mbar_wait(mbar0 + cstage * 8, cpar);
        } else {
          cp_async_wait<NS - 2>();
          __syncwarp();
        }
        const float wz = SDz[zlist[zi] * PP + it.pd];
        const float *row = ring + cstage * STRIDE;
        if (++cstage == NS) cstage = 0, cpar ^= 1u;
        float tz[PW][CV];
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          const float *q = row + soff[pw];
          if constexpr (F2) {
            // sm_100 packed fp32 (FFMA2 / FMUL2): both channels of the lane in one issue slot; each half is
            // rounded exactly like the scalar fmul / fma, so the pinned arithmetic is unchanged
            float2 z2;
#pragma unroll
            for (int j = 0; j < NXU; ++j) {
              const float2 t = *reinterpret_cast<const float2 *>(q + j * VOX);
              const float2 w2 = make_float2(tw[pw][j], tw[pw][j]);
              z2 = j == 0 ? __fmul2_rn(w2, t) : __ffma2_rn(w2, t, z2);
            }
            tz[pw][0] = z2.x, tz[pw][1] = z2.y;
          } else {
#pragma unroll
          for (int j = 0; j < NXU; ++j) {
            float f[CV];
            if constexpr (CV == 4) {
              const float4 t = *reinterpret_cast<const float4 *>(q + j * VOX);
              f[0] = t.x, f[1] = t.y, f[2] = t.z, f[3] = t.w;
            } else if constexpr (CV == 2) {
              const float2 t = *reinterpret_cast<const float2 *>(q + j * VOX);
              f[0] = t.x, f[1] = t.y;
            } else {
              f[0] = q[j * VOX];
            }
#pragma unroll
            for (int c = 0; c < CV; ++c) tz[pw][c] = j == 0 ? tw[pw][0] * f[c] : fmaf(tw[pw][j], f[c], tz[pw][c]);
          }
          }
        }
        if (long_bins) {  // one warp-uniform test per row; bins wider than NXU taps are rare
#pragma unroll
          for (int pw = 0; pw < PW; ++pw) {
            const int lo = T.xlo[pw];
            const int n = T.xhi[pw] - lo + 1;
            const float *q = row + soff[pw];
            const float *wq = T.Dx + lo * PWP + pw;
#pragma unroll 1
            for (int j = NXU; j < n; ++j) {
              const float w = wq[j * PWP];
#pragma unroll
              for (int c = 0; c < CV; ++c) tz[pw][c] = fmaf(w, q[j * VOX + c], tz[pw][c]);
            }
          }
        }
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          if constexpr (F2) {
            const float2 o = __ffma2_rn(make_float2(wz, wz), make_float2(tz[pw][0], tz[pw][1]),
                                        make_float2(t1[pw][0], t1[pw][1]));
            t1[pw][0] = o.x, t1[pw][1] = o.y;
          } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) t1[pw][c] = fmaf(wz, tz[pw][c], t1[pw][c]);
          }
        }
        __syncwarp();
        if (r + NS - 1 < nrows) issue();
        else if constexpr (!BULK) cp_async_commit();
      }
      // y-stage, once per feature row index y
      const int yy = ylist[yi];
      float wy[ROWS];
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) wy[rr] = rr < it.rows ? SDy[yy * PP + it.ph0 + rr] : 0.0f;
#pragma unroll
      for (int rr = 0; rr < ROWS; ++rr) {
        if (wy[rr] != 0.0f) {
#pragma unroll
          for (int pw = 0; pw < PW; ++pw) {
            if constexpr (F2) {
              const float2 o = __ffma2_rn(make_float2(wy[rr], wy[rr]), make_float2(t1[pw][0], t1[pw][1]),
                                          make_float2(acc[rr][pw][0], acc[rr][pw][1]));
              acc[rr][pw][0] = o.x, acc[rr][pw][1] = o.y;
            } else {
#pragma unroll
              for (int c = 0; c < CV; ++c) acc[rr][pw][c] = fmaf(wy[rr], t1[pw][c], acc[rr][pw][c]);
            }
          }
        }
      }
    }
    if constexpr (!BULK) cp_async_wait<0>();
  }

  // ---- epilogue: divide by the sample count, transpose through smem, stream out ----
  const int NB = it.rows * PW;
  float *stage = ring;  // the ring is drained
  const long long out_base = (((long long)it.krow * C) * p.PD + it.pd) * p.PH * PW + (long long)it.ph0 * PW;
  const long long ch_stride = (long long)p.PD * p.PH * PW;
  copy_out_tile<ROWS, PW, CV>(acc, count, stage, lane, NB, it.chunk, C, p.out + out_base, ch_stride);
  __syncwarp();  // the staging tile aliases the ring the next sub-item prefetches into
  }  // sub-item loop
}

// ---------------------------------------------------------------------------------------------
// Backward, channels-last, separable (transposed contraction).  Same work split as the forward.
// One vector red per (row voxel, lane) instead of 64 scalar atomics per output element.
// ---------------------------------------------------------------------------------------------
// Literal backward of a warp's whole (pd, ph-group) tile, out of line (see literal_tile_fwd).
template <int CV>
__device__ __noinline__ void literal_tile_bwd(const Item &it, float *gb, int C, int PW, const float *stage, int lane,
                                              bool active, float inv_unused) {
  (void)inv_unused;
  for (int r = 0; r < it.rows; ++r)
    for (int pw = 0; pw < PW; ++pw) {
      float top[CV];
#pragma unroll
      for (int c = 0; c < CV; ++c) top[c] = stage[(c * it.rows * PW + r * PW + pw) * 33 + lane];
      if (active) literal_bin_bwd<CV>(it, gb, C, it.pd, it.ph0 + r, pw, top);
    }
}

template <int PW, int ROWS, int CV, int RXR, bool F2 = false>
__global__ void __launch_bounds__(kWarps * 32) roi_align3d_bwd_cl_kernel(const RoiParams p) {
  static_assert(!F2 || CV == 2, "packed f32x2 arithmetic pairs the two channels of a lane");
  using TB = Tables<PW>;
  constexpr int PWP = TB::PWP;
  constexpr int VOX = 32 * CV;
  constexpr int STAGE = CV * ROWS * PW * 33;     // all CV slots of the grad tile at once
  constexpr int UX = RXR * VOX;                  // x-expanded row, [xx][lane*CV + c]
  constexpr int LISTS = 80;
  constexpr int WARP_FLOATS = (TB::FLOATS + LISTS / 4 + (STAGE > UX ? STAGE : UX) + 3) / 4 * 4;
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *sm = smem_all + warp * WARP_FLOATS;
  const long long item = (long long)blockIdx.x * kWarps + warp;
  if (item >= p.total_items) return;

  const Item it = decode_item(p, item, ROWS);
  if (!it.ok) return;
  const int C = p.C;
  int c_base = (it.chunk * 32 + lane) * CV;
  const bool active = c_base < C;
  if (!active) c_base = 0;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  float *gb = it.L.grad + (long long)it.b * vox * C + c_base;
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);

  TB T;
  T.bind(sm);
  unsigned char *ylist = reinterpret_cast<unsigned char *>(sm + ((TB::FLOATS + 3) / 4 * 4));
  unsigned char *zlist = ylist + 40;
  float *stage = sm + ((TB::FLOATS + 3) / 4 * 4) + LISTS / 4;
  float *ux = stage;  // aliases the stage-in tile once the gradients are in registers

  // ---- stage-in of this warp's grad_out tile: 4-byte cp.async copies that transpose on the fly
  //      (coalesced global reads -> [bin][33] padded smem), all in flight together ----
  const int NB = it.rows * PW;
  const long long ch_stride = (long long)p.PD * p.PH * PW;
  // reference index (roi_align_kernel.cu:554-555): pd*PD*PW + ph*PW + pw when bug_compat
  const long long row_base = p.bug_compat ? ((long long)it.pd * p.PD + it.ph0) * PW
                                          : ((long long)it.pd * p.PH + it.ph0) * PW;
  const long long top_total = (long long)p.K * C * ch_stride;
  {
    const int col_stride = CV * (int)ch_stride;
#pragma unroll
    for (int c = 0; c < CV; ++c) {
      const int cols = min(32, (C - it.chunk * 32 * CV - c + CV - 1) / CV);
      float *st = stage + c * (NB * 33);
      const long long g0 = ((long long)it.k * C + (long long)it.chunk * 32 * CV + c) * ch_stride + row_base;
      // elements past the end of grad_out can only be addressed with bug_compat's wrong row base
      long long lim = top_total - g0;
      int total = cols * NB;
      if (lim < (long long)(cols - 1) * col_stride + NB) {
        total = 0;  // rare (last RoI / channel with bug_compat): zero the tile, copy nothing out of range
      }
      if (total < 32 * NB) {
        for (int i = lane; i < NB * 33; i += 32) st[i] = 0.0f;
        __syncwarp();
      }
      // one column (channel run of NB floats) at a time, lanes along the run (cf. copy_out_tile)
      const int ncol = total / NB;
      unsigned sp = (unsigned)__cvta_generic_to_shared(st + lane * 33);
      const float *gp = p.grad_out + g0 + lane;
#pragma unroll 4
      for (int cl = 0; cl < ncol; ++cl) {
        if (lane < NB) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp), "l"(gp) : "memory");
        if (lane + 32 < NB)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp + 32 * 33 * 4), "l"(gp + 32) : "memory");
        for (int bin = lane + 64; bin < NB; bin += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp + (bin - lane) * 33 * 4), "l"(gp + (bin - lane))
                       : "memory");
        sp += 4;
        gp += col_stride;
      }
    }
    cp_async_commit();
  }
  build_tables<PW>(T, it, lane);  // overlaps the copies
  cp_async_wait<0>();
  __syncwarp();
  if (T.empty) return;
  const int RX = T.xmax - T.xmin + 1;
  if (!T.fits || RX > RXR) {
    literal_tile_bwd<CV>(it, gb, C, PW, stage, lane, active, 0.0f);
    return;
  }
  // gradients to registers, scaled once by 1/count (reference: top*w/count per corner, :600-608)
  const float inv = __frcp_rn(count);
  float g[ROWS][PW][CV];
#pragma unroll
  for (int c = 0; c < CV; ++c)
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int pw = 0; pw < PW; ++pw)
        g[r][pw][c] = r < it.rows ? stage[(c * NB + r * PW + pw) * 33 + lane] * inv : 0.0f;

  // compact lists of the y rows / z slices that carry weight (as in the forward)
  const int RY = T.ymax - T.ymin + 1, RZ = T.zmax - T.zmin + 1;
  int ny = 0, nz = 0;
  for (int y0 = 0; y0 < RY; y0 += 32) {
    const int yy = y0 + lane;
    bool a = false;
    if (yy < RY) {
#pragma unroll
      for (int r = 0; r < ROWS; ++r) a |= T.Dy[yy * 8 + r] != 0.0f;
    }
    const unsigned bal = __ballot_sync(FULL, a);
    if (a) ylist[ny + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)yy;
    ny += __popc(bal);
  }
  {
    const bool a = lane < RZ && T.Dz[lane] != 0.0f;
    const unsigned bal = __ballot_sync(FULL, a);
    if (a) zlist[__popc(bal & ((1u << lane) - 1u))] = (unsigned char)lane;
    nz = __popc(bal);
  }
  __syncwarp();

  const long long row_elems = (long long)it.L.W * C;
  const long long slice_elems = (long long)it.L.H * row_elems;
  float *gbase = gb + ((long long)T.zmin * it.L.H + T.ymin) * row_elems + (long long)T.xmin * C;
  bool has_gaps = false;
  for (int x0 = 0; x0 < RX; x0 += 32) has_gaps |= __any_sync(FULL, x0 + lane < RX && !T.xany[x0 + lane]);
  float zw[4];
  long long zo[4];
#pragma unroll
  for (int zi = 0; zi < 4; ++zi) {
    const int zrel = zi < nz ? zlist[zi] : 0;
    zw[zi] = zi < nz ? T.Dz[zrel] : 0.0f;
    zo[zi] = (long long)zrel * slice_elems;
  }
  for (int yi = 0; yi < ny; ++yi) {
    const int yy = ylist[yi];
    float wy[8];
    {
      const float4 a = *reinterpret_cast<const float4 *>(T.Dy + yy * 8);
      const float4 b4 = *reinterpret_cast<const float4 *>(T.Dy + yy * 8 + 4);
      wy[0] = a.x, wy[1] = a.y, wy[2] = a.z, wy[3] = a.w, wy[4] = b4.x, wy[5] = b4.y, wy[6] = b4.z, wy[7] = b4.w;
    }
    // u[pw] = sum over the ph rows of this group of wy * g  (once per y)
    float u[PW][CV];
#pragma unroll
    for (int pw = 0; pw < PW; ++pw)
#pragma unroll
      for (int c = 0; c < CV; ++c) u[pw][c] = 0.0f;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      if (wy[r] != 0.0f) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          if constexpr (F2) {  // FFMA2: both channels in one issue slot, each half rounded like fmaf
            const float2 o = __ffma2_rn(make_float2(wy[r], wy[r]), make_float2(g[r][pw][0], g[r][pw][1]),
                                        make_float2(u[pw][0], u[pw][1]));
            u[pw][0] = o.x, u[pw][1] = o.y;
          } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) u[pw][c] = fmaf(wy[r], g[r][pw][c], u[pw][c]);
          }
        }
      }
    }
    // x-expansion, once per y: ux[xx] = sum_pw Dx[xx][pw] * u[pw]   (kept per lane in shared memory)
    __syncwarp();
    for (int xx = 0; xx < RX; ++xx) {
      float wx[PWP];
#pragma unroll
      for (int q = 0; q < PWP / 4; ++q) {
        const float4 t = *reinterpret_cast<const float4 *>(T.Dx + xx * PWP + q * 4);
        wx[q * 4 + 0] = t.x, wx[q * 4 + 1] = t.y, wx[q * 4 + 2] = t.z, wx[q * 4 + 3] = t.w;
      }
      float v[CV];
#pragma unroll
      for (int c = 0; c < CV; ++c) v[c] = 0.0f;
#pragma unroll
      for (int pw = 0; pw < PW; ++pw) {
        if constexpr (F2) {
          const float2 o = __ffma2_rn(make_float2(wx[pw], wx[pw]), make_float2(u[pw][0], u[pw][1]), make_float2(v[0], v[1]));
          v[0] = o.x, v[1] = o.y;
        } else {
#pragma unroll
          for (int c = 0; c < CV; ++c) v[c] = fmaf(wx[pw], u[pw][c], v[c]);
        }
      }
#pragma unroll
      for (int c = 0; c < CV; ++c) ux[xx * VOX + lane * CV + c] = v[c];
    }
    __syncwarp();
    // scatter: one vector red per (z, x) voxel of this y row.  x is the outer loop so each ux value is read
    // once; the (typically 2-3) z slices are handled by a predicated unrolled inner loop whose weights and
    // slice offsets live in registers.
    float *q = gbase + (long long)yy * row_elems;
    const float *uxl = ux + lane * CV;
    for (int xx = 0; xx < RX; ++xx, q += C) {
      if (has_gaps && !T.xany[xx]) continue;
      float uv[CV];
#pragma unroll
      for (int c = 0; c < CV; ++c) uv[c] = uxl[xx * VOX + c];
      // No per-lane `active` test here: lanes past the last channel hold zero gradients (their stage-in columns
      // were zero-filled) and point at channel 0, so their reds add +0.0 to a valid address.  Keeping the loop
      // free of lane-dependent branches lets the warp-uniform `zi < nz` tests compile to plain predication.
#pragma unroll
      for (int zi = 0; zi < 4; ++zi) {
        if (zi < nz) {
          float v[CV];
          if constexpr (F2) {
            const float2 o = __fmul2_rn(make_float2(zw[zi], zw[zi]), make_float2(uv[0], uv[1]));
            v[0] = o.x, v[1] = o.y;
          } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) v[c] = zw[zi] * uv[c];
          }
          redv<CV>(q + zo[zi], v);
        }
      }
      for (int zi = 4; zi < nz; ++zi) {
        const int zrel = zlist[zi];
        const float wz = T.Dz[zrel];
        float v[CV];
#pragma unroll
        for (int c = 0; c < CV; ++c) v[c] = wz * uv[c];
        redv<CV>(q + (long long)zrel * slice_elems, v);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Backward with CTA-shared per-RoI tables (the backward twin of roi_align3d_fwd_ring2_kernel): the four
// warps of a CTA work on the same RoI, its axis tables are built once per CTA by three warps in parallel
// while every warp's grad_out tile is already in flight (cp.async), and the x-expansion is fused with the
// scatter -- each expanded voxel value goes from registers straight into its (typically 2-3) vector reds,
// two voxels per iteration for instruction-level parallelism, with no shared-memory round trip.
// ---------------------------------------------------------------------------------------------
template <int PW, int ROWS, int CV, bool F2, int MINB, int PP>
__global__ void __launch_bounds__(kWarps * 32, MINB) roi_align3d_bwd2_kernel(const RoiParams p) {
  static_assert(!F2 || CV == 2, "packed f32x2 arithmetic pairs the two channels of a lane");
  using TB = Tables<PW>;
  constexpr int PWP = TB::PWP;
  constexpr int STAGE = CV * ROWS * PW * 33;     // all CV slots of the grad tile at once
  constexpr int LISTS = 80;
  constexpr int WARP_FLOATS = (LISTS / 4 + STAGE + 3) / 4 * 4;
  constexpr int SH_FLOATS = (RXMAX + 1) * PWP + RYMAX * PP + RZMAX2 * PP + RXMAX + 8;
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  float *SDx = smem_all;                         // [x - xmin][PWP] (+1 row: the paired x loop may read one past RX)
  float *SDy = SDx + (RXMAX + 1) * PWP;          // [y - ymin][PP]
  float *SDz = SDy + RYMAX * PP;                 // [z - zmin][PP]
  int *Sxany = reinterpret_cast<int *>(SDz + RZMAX2 * PP);
  int *Sbox = Sxany + RXMAX;
  float *sm = smem_all + ((SH_FLOATS + 3) / 4 * 4) + warp * WARP_FLOATS;

  const int k = blockIdx.x / p.ctas_per_roi;
  const int sub = (blockIdx.x - k * p.ctas_per_roi) * kWarps + warp;
  const bool valid = sub < p.items_per_roi;
  Item it;
  {
    unsigned item = (unsigned)(valid ? sub : 0);
    const unsigned phg = item % (unsigned)p.nphg;
    item /= (unsigned)p.nphg;
    it.pd = (int)(item % (unsigned)p.PD);
    it.chunk = (int)(item / (unsigned)p.PD);
    it.k = k;
    it.ph0 = (int)phg * ROWS;
    it.rows = min(ROWS, p.PH - it.ph0);
    float r[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)k * 7 + i);
    it.lvl = p.num_levels > 1 ? roi_level(r, p.num_levels, p.inv_finest) : 0;
    it.L = p.lv[it.lvl];
    it.b = (int)r[0];
    it.ok = it.b >= 0 && it.b < p.B;
    it.axw = axis_setup(r[1], r[3], it.L.scale, p.PW, p.sample_num);
    it.axh = axis_setup(r[2], r[4], it.L.scale, p.PH, p.sample_num);
    it.axd = axis_setup(r[5], r[6], it.L.scale_d, p.PD, p.sample_num);
  }
  if (!it.ok) return;  // same RoI for the whole CTA: uniform exit before any barrier
  const int C = p.C;
  int c_base = (it.chunk * 32 + lane) * CV;
  const bool active = c_base < C;
  if (!active) c_base = 0;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  float *gb = it.L.grad + (long long)it.b * vox * C + c_base;
  unsigned char *ylist = reinterpret_cast<unsigned char *>(sm);
  unsigned char *zlist = ylist + 40;
  float *stage = sm + LISTS / 4;

  // ---- stage-in of this warp's grad_out tile (see roi_align3d_bwd_cl_kernel), issued before the table build ----
  const int NB = it.rows * PW;
  if (valid) {
    const long long ch_stride = (long long)p.PD * p.PH * PW;
    // reference index (roi_align_kernel.cu:554-555): pd*PD*PW + ph*PW + pw when bug_compat
    const long long row_base = p.bug_compat ? ((long long)it.pd * p.PD + it.ph0) * PW
                                            : ((long long)it.pd * p.PH + it.ph0) * PW;
    const long long top_total = (long long)p.K * C * ch_stride;
    const int col_stride = CV * (int)ch_stride;
#pragma unroll
    for (int c = 0; c < CV; ++c) {
      const int cols = min(32, (C - it.chunk * 32 * CV - c + CV - 1) / CV);
      float *st = stage + c * (NB * 33);
      const long long g0 = ((long long)it.k * C + (long long)it.chunk * 32 * CV + c) * ch_stride + row_base;
      long long lim = top_total - g0;  // elements past the end of grad_out: only reachable with bug_compat's row base
      int total = cols * NB;
      if (lim < (long long)(cols - 1) * col_stride + NB) total = 0;
      if (total < 32 * NB) {
        for (int i = lane; i < NB * 33; i += 32) st[i] = 0.0f;
        __syncwarp();
      }
      const int ncol = total / NB;
      unsigned sp = (unsigned)__cvta_generic_to_shared(st + lane * 33);
      const float *gp = p.grad_out + g0 + lane;
      // four columns per iteration through four address registers and immediate shared offsets: a copy still
      // queued in the memory pipeline does not hold up the address update of the next one
      int cl = 0;
      for (; cl + 4 <= ncol; cl += 4) {
        const float *g0p = gp, *g1p = gp + col_stride, *g2p = gp + 2 * col_stride, *g3p = gp + 3 * col_stride;
        if (lane < NB) {
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp), "l"(g0p) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+4], [%1], 4;\n" ::"r"(sp), "l"(g1p) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+8], [%1], 4;\n" ::"r"(sp), "l"(g2p) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+12], [%1], 4;\n" ::"r"(sp), "l"(g3p) : "memory");
        }
        if (lane + 32 < NB) {
          asm volatile("cp.async.ca.shared.global [%0+4224], [%1+128], 4;\n" ::"r"(sp), "l"(g0p) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+4228], [%1+128], 4;\n" ::"r"(sp), "l"(g1p) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+4232], [%1+128], 4;\n" ::"r"(sp), "l"(g2p) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+4236], [%1+128], 4;\n" ::"r"(sp), "l"(g3p) : "memory");
        }
        for (int bin = lane + 64; bin < NB; bin += 32) {
          const unsigned so = sp + (bin - lane) * 33 * 4;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(so), "l"(g0p + (bin - lane)) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+4], [%1], 4;\n" ::"r"(so), "l"(g1p + (bin - lane)) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+8], [%1], 4;\n" ::"r"(so), "l"(g2p + (bin - lane)) : "memory");
          asm volatile("cp.async.ca.shared.global [%0+12], [%1], 4;\n" ::"r"(so), "l"(g3p + (bin - lane)) : "memory");
        }
        sp += 16;
        gp += 4 * col_stride;
      }
      for (; cl < ncol; ++cl) {
        if (lane < NB) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp), "l"(gp) : "memory");
        if (lane + 32 < NB)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp + 32 * 33 * 4), "l"(gp + 32) : "memory");
        for (int bin = lane + 64; bin < NB; bin += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(sp + (bin - lane) * 33 * 4), "l"(gp + (bin - lane))
                       : "memory");
        sp += 4;
        gp += col_stride;
      }
    }
    cp_async_commit();
  }

  // ---- CTA-shared tables: warp 0 lanes [0,PW) -> x bins, warp 1 lanes [0,PH) -> y bins, warp 2 lanes [0,PD) -> z bins
  const int role = (warp == 0 && lane < PW) ? 0 : (warp == 1 && lane < p.PH) ? 1 : (warp == 2 && lane < p.PD) ? 2 : -1;
  const Axis ax = role == 1 ? it.axh : role == 2 ? it.axd : it.axw;
  const int asize = role == 1 ? it.L.H : role == 2 ? it.L.D : it.L.W;
  int lo = INT_MAX, hi = -1;
  if (role >= 0) {
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, lane, i), asize);
      if (t.valid) lo = min(lo, t.low), hi = max(hi, t.high);
    }
  }
  if (warp < 3) {
    const int mn = __reduce_min_sync(FULL, role >= 0 ? lo : INT_MAX);
    const int mx = __reduce_max_sync(FULL, role >= 0 ? hi : -1);
    if (lane == 0) Sbox[warp * 2] = mn, Sbox[warp * 2 + 1] = mx;
  }
  __syncthreads();
  const int xmin = Sbox[0], xmax = Sbox[1], ymin = Sbox[2], ymax = Sbox[3], zmin = Sbox[4], zmax = Sbox[5];
  const bool empty = xmax < xmin || ymax < ymin || zmax < zmin;
  const bool fits = empty || ((xmax - xmin < RXMAX) && (ymax - ymin < RYMAX) && (zmax - zmin < RZMAX2));
  const int RX = xmax - xmin + 1, RY = ymax - ymin + 1, RZ = zmax - zmin + 1;
  if (!empty && fits) {
    for (int i = tid; i < (RX + 1) * PWP; i += kWarps * 32) SDx[i] = 0.0f;
    for (int i = tid; i < RY * PP; i += kWarps * 32) SDy[i] = 0.0f;
    for (int i = tid; i < RZ * PP; i += kWarps * 32) SDz[i] = 0.0f;
    for (int i = tid; i < RX; i += kWarps * 32) Sxany[i] = 0;
  }
  __syncthreads();
  if (!empty && fits && role >= 0) {
    float *tab = role == 0 ? SDx : role == 1 ? SDy : SDz;
    const int stride = role == 0 ? PWP : PP;
    const int mn = role == 0 ? xmin : role == 1 ? ymin : zmin;
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, lane, i), asize);
      if (t.valid) {
        tab[(t.low - mn) * stride + lane] += t.h;
        tab[(t.high - mn) * stride + lane] += t.l;
        if (role == 0) Sxany[t.low - mn] = 1, Sxany[t.high - mn] = 1;
      }
    }
  }
  __syncthreads();
  if (!valid) return;  // padding warp of the last CTA of this RoI: no block-level barriers below
  cp_async_wait<0>();
  __syncwarp();
  if (empty) return;
  if (!fits) {
    literal_tile_bwd<CV>(it, gb, C, PW, stage, lane, active, 0.0f);
    return;
  }
  // gradients to registers, scaled once by 1/count (reference: top*w/count per corner, :600-608)
  const float inv = __frcp_rn((float)(it.axd.S * it.axh.S * it.axw.S));
  float g[ROWS][PW][CV];
#pragma unroll
  for (int c = 0; c < CV; ++c)
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int pw = 0; pw < PW; ++pw)
        g[r][pw][c] = r < it.rows ? stage[(c * NB + r * PW + pw) * 33 + lane] * inv : 0.0f;

  // compact lists of the y rows / z slices that carry weight for this (pd, ph-group)
  int ny = 0, nz = 0;
  for (int y0 = 0; y0 < RY; y0 += 32) {
    const int yy = y0 + lane;
    bool a = false;
    if (yy < RY) {
#pragma unroll
      for (int r = 0; r < ROWS; ++r) a |= (r < it.rows) && SDy[yy * PP + it.ph0 + r] != 0.0f;
    }
    const unsigned bal = __ballot_sync(FULL, a);
    if (a) ylist[ny + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)yy;
    ny += __popc(bal);
  }
  for (int z0 = 0; z0 < RZ; z0 += 32) {
    const int zz = z0 + lane;
    const bool a = zz < RZ && SDz[zz * PP + it.pd] != 0.0f;
    const unsigned bal = __ballot_sync(FULL, a);
    if (a) zlist[nz + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)zz;
    nz += __popc(bal);
  }
  __syncwarp();

  const long long row_elems = (long long)it.L.W * C;
  const long long slice_elems = (long long)it.L.H * row_elems;
  float *gbase = gb + ((long long)zmin * it.L.H + ymin) * row_elems + (long long)xmin * C;
  bool has_gaps = false;
  for (int x0 = 0; x0 < RX; x0 += 32) has_gaps |= __any_sync(FULL, x0 + lane < RX && !Sxany[x0 + lane]);
  float zw[4];
  long long zo[4];
#pragma unroll
  for (int zi = 0; zi < 4; ++zi) {
    const int zrel = zi < nz ? zlist[zi] : 0;
    zw[zi] = zi < nz ? SDz[zrel * PP + it.pd] : 0.0f;
    zo[zi] = (long long)zrel * slice_elems;
  }
  for (int yi = 0; yi < ny; ++yi) {
    const int yy = ylist[yi];
    // u[pw] = sum over the ph rows of this group of wy * g  (once per y)
    float u[PW][CV];
#pragma unroll
    for (int pw = 0; pw < PW; ++pw)
#pragma unroll
      for (int c = 0; c < CV; ++c) u[pw][c] = 0.0f;
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      const float wy = r < it.rows ? SDy[yy * PP + it.ph0 + r] : 0.0f;
      if (wy != 0.0f) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          if constexpr (F2) {
            const float2 o = __ffma2_rn(make_float2(wy, wy), make_float2(g[r][pw][0], g[r][pw][1]),
                                        make_float2(u[pw][0], u[pw][1]));
            u[pw][0] = o.x, u[pw][1] = o.y;
          } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) u[pw][c] = fmaf(wy, g[r][pw][c], u[pw][c]);
          }
        }
      }
    }
    // fused x-expansion + scatter, two voxels per iteration: v[x] = sum_pw Dx[x][pw] * u[pw], then one vector
    // red per (z, x).  Lanes past the last channel hold zero gradients and point at channel 0 (+0.0 adds), so
    // the loop has no lane-dependent branch.
    float *q = gbase + (long long)yy * row_elems;
    for (int xx = 0; xx < RX; xx += 2, q += 2 * (long long)C) {
      float wx[2][PWP];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int t4 = 0; t4 < PWP / 4; ++t4) {
          const float4 t = *reinterpret_cast<const float4 *>(SDx + (xx + h) * PWP + t4 * 4);
          wx[h][t4 * 4 + 0] = t.x, wx[h][t4 * 4 + 1] = t.y, wx[h][t4 * 4 + 2] = t.z, wx[h][t4 * 4 + 3] = t.w;
        }
      float v[2][CV];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int c = 0; c < CV; ++c) v[h][c] = 0.0f;
#pragma unroll
      for (int pw = 0; pw < PW; ++pw)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if constexpr (F2) {
            const float2 o = __ffma2_rn(make_float2(wx[h][pw], wx[h][pw]), make_float2(u[pw][0], u[pw][1]),
                                        make_float2(v[h][0], v[h][1]));
            v[h][0] = o.x, v[h][1] = o.y;
          } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) v[h][c] = fmaf(wx[h][pw], u[pw][c], v[h][c]);
          }
        }
      // all products and addresses first, then the reds back to back: distinct registers per red, so a red still
      // waiting in the memory pipeline does not stall the next one on a register it has yet to read
      float o[2][4][CV];
      float *ad[2][4];
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int zi = 0; zi < 4; ++zi) {
          ad[h][zi] = q + h * (long long)C + zo[zi];
          if constexpr (F2) {
            const float2 t = __fmul2_rn(make_float2(zw[zi], zw[zi]), make_float2(v[h][0], v[h][1]));
            o[h][zi][0] = t.x, o[h][zi][1] = t.y;
          } else {
#pragma unroll
            for (int c = 0; c < CV; ++c) o[h][zi][c] = zw[zi] * v[h][c];
          }
        }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (xx + h >= RX || (has_gaps && !Sxany[xx + h])) continue;  // warp-uniform
#pragma unroll
        for (int zi = 0; zi < 4; ++zi)
          if (zi < nz) redv<CV>(ad[h][zi], o[h][zi]);
        for (int zi = 4; zi < nz; ++zi) {
          const int zrel = zlist[zi];
          const float wz = SDz[zrel * PP + it.pd];
          float t[CV];
#pragma unroll
          for (int c = 0; c < CV; ++c) t[c] = wz * v[h][c];
          redv<CV>(q + h * (long long)C + (long long)zrel * slice_elems, t);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Generic kernels (any PD/PH/PW): one warp per (k, chunk, pd, ph), literal evaluation.
// ---------------------------------------------------------------------------------------------
template <int CV>
__global__ void __launch_bounds__(kWarps * 32) roi_align3d_fwd_generic_kernel(const RoiParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long item = (long long)blockIdx.x * kWarps + warp;
  if (item >= p.total_items) return;
  const Item it = decode_item(p, item, 1);
  const int C = p.C;
  if (p.lvls_out != nullptr && it.chunk == 0 && it.pd == 0 && it.ph0 == 0 && lane == 0) p.lvls_out[it.k] = it.lvl;
  int c_base = (it.chunk * 32 + lane) * CV;
  const bool active = c_base < C;
  if (!active) c_base = 0;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  const float *fb = it.L.feats + (long long)(it.ok ? it.b : 0) * vox * C + c_base;
  for (int pw = 0; pw < p.PW; ++pw) {
    float v[CV];
    if (it.ok) {
      literal_bin_fwd<CV>(it, fb, C, it.pd, it.ph0, pw, v);
    } else {
#pragma unroll
      for (int c = 0; c < CV; ++c) v[c] = 0.0f;
    }
    if (active) {
#pragma unroll
      for (int c = 0; c < CV; ++c)
        p.out[((((long long)it.krow * C + c_base + c) * p.PD + it.pd) * p.PH + it.ph0) * p.PW + pw] = v[c];
    }
  }
}

template <int CV>
__global__ void __launch_bounds__(kWarps * 32) roi_align3d_bwd_generic_kernel(const RoiParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long item = (long long)blockIdx.x * kWarps + warp;
  if (item >= p.total_items) return;
  const Item it = decode_item(p, item, 1);
  if (!it.ok) return;
  const int C = p.C;
  int c_base = (it.chunk * 32 + lane) * CV;
  if (c_base >= C) return;
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  float *gb = it.L.grad + (long long)it.b * vox * C + c_base;
  const long long bins = (long long)p.PD * p.PH * p.PW;
  const long long total = (long long)p.K * C * bins;
  for (int pw = 0; pw < p.PW; ++pw) {
    float top[CV];
#pragma unroll
    for (int c = 0; c < CV; ++c) {
      const long long off = p.bug_compat ? ((long long)it.pd * p.PD * p.PW + (long long)it.ph0 * p.PW + pw)
                                         : (((long long)it.pd * p.PH + it.ph0) * p.PW + pw);
      const long long o = ((long long)it.k * C + c_base + c) * bins + off;
      top[c] = o < total ? __ldg(p.grad_out + o) : 0.0f;
    }
    literal_bin_bwd<CV>(it, gb, C, it.pd, it.ph0, pw, top);
  }
}

__global__ void map_roi_levels_kernel(const float *rois, int K, int num_levels, float inv_finest, int64_t *lvls) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  float r[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) r[i] = rois[(long long)k * 7 + i];
  lvls[k] = roi_level(r, num_levels, inv_finest);
}

// ---------------------------------------------------------------------------------------------
// Layout conversion: per batch a [C][S] <-> [S][C] transpose (S = D*H*W).
// Fast path (C % 4 == 0, S % 4 == 0, 16-byte aligned): 32 x 128 tiles, 16-byte global accesses on both
// sides (float4 along the contiguous dimension of the source when reading, of the destination when
// writing), padded shared tile so both phases are bank-conflict free.  Generic path: 32 x 32 tiles.
// ---------------------------------------------------------------------------------------------
// src [rows][cols] -> dst [cols][rows].  Tile = 32 rows x 128 cols.  256 threads.
__global__ void __launch_bounds__(256) transpose_r32c128_kernel(const float *__restrict__ src, float *__restrict__ dst,
                                                                 int rows, int cols, int tiles_c) {
  __shared__ float tile[32][129];
  const long long boff = (long long)blockIdx.y * rows * cols;
  const int c0 = (blockIdx.x % tiles_c) * 128, r0 = (blockIdx.x / tiles_c) * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // read: one warp = one source row segment of 128 floats (32 lanes x float4)
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = r0 + warp + i * 8, c = c0 + lane * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows && c < cols) v = __ldcs(reinterpret_cast<const float4 *>(src + boff + (long long)r * cols + c));
    tile[warp + i * 8][lane * 4 + 0] = v.x, tile[warp + i * 8][lane * 4 + 1] = v.y;
    tile[warp + i * 8][lane * 4 + 2] = v.z, tile[warp + i * 8][lane * 4 + 3] = v.w;
  }
  __syncthreads();
  // write: 8 lanes x float4 cover the 32 rows (contiguous in dst) of one column; a warp covers 4 columns
  const int rq = (lane & 7) * 4, cs = lane >> 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cl = warp * 16 + i * 4 + cs;  // 8 warps x 16 columns = 128
    const int c = c0 + cl, r = r0 + rq;
    if (c < cols && r < rows) {
      const float4 v = make_float4(tile[rq + 0][cl], tile[rq + 1][cl], tile[rq + 2][cl], tile[rq + 3][cl]);
      *reinterpret_cast<float4 *>(dst + boff + (long long)c * rows + r) = v;
    }
  }
}

// src [rows][cols] -> dst [cols][rows].  Tile = 128 rows x 32 cols (the mirror image, for [S][C] -> [C][S]).
__global__ void __launch_bounds__(256) transpose_r128c32_kernel(const float *__restrict__ src, float *__restrict__ dst,
                                                                 int rows, int cols, int tiles_c) {
  __shared__ float tile[32][129];  // tile[col][row]
  const long long boff = (long long)blockIdx.y * rows * cols;
  const int c0 = (blockIdx.x % tiles_c) * 32, r0 = (blockIdx.x / tiles_c) * 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // read: 8 lanes x float4 cover the 32 columns (contiguous in src) of one row; a warp covers 4 rows
  const int cq = (lane & 7) * 4, rs = lane >> 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int rl = warp * 16 + i * 4 + rs;
    const int r = r0 + rl, c = c0 + cq;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < rows && c < cols) v = __ldcs(reinterpret_cast<const float4 *>(src + boff + (long long)r * cols + c));
    tile[cq + 0][rl] = v.x, tile[cq + 1][rl] = v.y, tile[cq + 2][rl] = v.z, tile[cq + 3][rl] = v.w;
  }
  __syncthreads();
  // write: one warp = one destination row segment of 128 floats
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = c0 + warp + i * 8, r = r0 + lane * 4;
    if (c < cols && r < rows) {
      const float4 v = make_float4(tile[warp + i * 8][lane * 4 + 0], tile[warp + i * 8][lane * 4 + 1],
                                   tile[warp + i * 8][lane * 4 + 2], tile[warp + i * 8][lane * 4 + 3]);
      *reinterpret_cast<float4 *>(dst + boff + (long long)c * rows + r) = v;
    }
  }
}

__global__ void transpose_kernel(const float *__restrict__ src, float *__restrict__ dst, int rows, int cols,
                                 int tiles_c) {
  // generic: src [rows][cols] -> dst [cols][rows]; blockIdx.y = batch; blockIdx.x = linear tile index
  __shared__ float tile[32][33];
  const long long boff = (long long)blockIdx.y * rows * cols;
  const int c0 = (blockIdx.x % tiles_c) * 32, r0 = (blockIdx.x / tiles_c) * 32;
  const int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int r = r0 + ty + i, c = c0 + tx;
    if (r < rows && c < cols) tile[ty + i][tx] = __ldcs(src + boff + (long long)r * cols + c);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int c = c0 + ty + i, r = r0 + tx;
    if (r < rows && c < cols) dst[boff + (long long)c * rows + r] = tile[tx][ty + i];
  }
}

// long_dim: 0 = rows is the short (channel) dimension [C][S] -> [S][C]; 1 = rows is the long dimension.
static int transpose_launch(const float *src, float *dst, int B, int rows, int cols, cudaStream_t st) {
  const bool vec_ok = rows % 4 == 0 && cols % 4 == 0 && (reinterpret_cast<uintptr_t>(src) % 16) == 0 &&
                      (reinterpret_cast<uintptr_t>(dst) % 16) == 0;
  ROI3D_CHECK_ARG(B <= 65535, "transpose: batch too large");
  if (vec_ok && cols >= rows) {  // [C][S] -> [S][C]
    const long long tc = ceil_div_ll(cols, 128), tr = ceil_div_ll(rows, 32);
    ROI3D_CHECK_ARG(tc * tr < 2147483647LL, "transpose: tensor too large for one launch");
    transpose_r32c128_kernel<<<dim3((unsigned)(tc * tr), (unsigned)B), 256, 0, st>>>(src, dst, rows, cols, (int)tc);
  } else if (vec_ok) {           // [S][C] -> [C][S]
    const long long tc = ceil_div_ll(cols, 32), tr = ceil_div_ll(rows, 128);
    ROI3D_CHECK_ARG(tc * tr < 2147483647LL, "transpose: tensor too large for one launch");
    transpose_r128c32_kernel<<<dim3((unsigned)(tc * tr), (unsigned)B), 256, 0, st>>>(src, dst, rows, cols, (int)tc);
  } else {
    dim3 block(32, 8);
    const long long tc = ceil_div_ll(cols, 32), tr = ceil_div_ll(rows, 32);
    ROI3D_CHECK_ARG(tc * tr < 2147483647LL, "transpose: tensor too large for one launch");
    transpose_kernel<<<dim3((unsigned)(tc * tr), (unsigned)B), block, 0, st>>>(src, dst, rows, cols, (int)tc);
  }
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

// ---------------------------------------------------------------------------------------------
// Dispatch
// ---------------------------------------------------------------------------------------------
static int g_fwd_variant = 0;  // 0 = auto; see roi3d_set_tuning
static int g_fwd_items_per_warp = 0;  // 0 = auto
extern int g_host_pipeline_kb;        // host_api.cu
extern int g_fwd_stream_cfg, g_fwd_stream_debug;  // roi_align3d_stream.cu  // roi_align3d_stream.cu
extern int g_nms_mask_variant;        // nms3d.cu
extern int g_planar_smem_floats;      // roi_align3d_planar.cu
extern int g_topk_sieve;              // proposal.cu
extern thread_local cudaEvent_t g_timing_ev[2];  // roi_align3d_stream.cu
static int g_bwd_variant = 0;

template <int PW, int ROWS, int CV, int NXU>
static int launch_fwd(RoiParams &p, cudaStream_t st) {
  using TB = Tables<PW>;
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int WARP_FLOATS = ((STAGE > TB::FLOATS ? STAGE : TB::FLOATS) + 3) / 4 * 4;  // 16-byte aligned per warp
  const size_t smem = (size_t)kWarps * WARP_FLOATS * sizeof(float);
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.total_items = (long long)p.K * p.nchunk * p.PD * p.nphg;
  auto kern = roi_align3d_fwd_cl_kernel<PW, ROWS, CV, NXU>;
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = ceil_div_ll(p.total_items, kWarps);
  ROI3D_CHECK_ARG(p.total_items < 2147483647LL, "roi_align3d forward: too many work items");
  kern<<<(unsigned)blocks, kWarps * 32, smem, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB = 0>
static int launch_fwd_ring(RoiParams &p, cudaStream_t st) {
  using TB = Tables<PW>;
  constexpr int VOX = 32 * CV;
  constexpr int RING = NS * (RXR + 2) * VOX;
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int RING_OR_STAGE = RING > STAGE ? RING : STAGE;
  constexpr int WARP_FLOATS = (TB::FLOATS + 384 / 4 + RING_OR_STAGE + 3) / 4 * 4;
  const size_t smem = (size_t)kWarps * WARP_FLOATS * sizeof(float);
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.total_items = (long long)p.K * p.nchunk * p.PD * p.nphg;
  auto kern = roi_align3d_fwd_ring_kernel<PW, ROWS, CV, NXU, NS, RXR, MINB>;
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = ceil_div_ll(p.total_items, kWarps);
  ROI3D_CHECK_ARG(p.total_items < 2147483647LL, "roi_align3d forward: too many work items");
  kern<<<(unsigned)blocks, kWarps * 32, smem, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB = 0, int BULK = 0, bool F2 = false, bool MULTI = false, int ITEMS = 1>
static int launch_fwd_ring2(RoiParams &p, cudaStream_t st) {
  using LY = Ring2Layout<PW, ROWS, CV, NS, RXR, BULK>;
  const size_t smem = LY::BYTES;
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.items_per_roi = p.nchunk * p.PD * p.nphg;
  p.items_per_warp = !MULTI ? 1 : g_fwd_items_per_warp > 0 ? g_fwd_items_per_warp : ITEMS;
  p.ctas_per_roi = ceil_div(p.items_per_roi, kWarps * p.items_per_warp);
  p.total_items = (long long)p.K * p.items_per_roi;
  const long long blocks = (long long)p.K * p.ctas_per_roi;
  ROI3D_CHECK_ARG(blocks < 2147483647LL, "roi_align3d forward: too many work items");
  static_assert(BULK == 0, "the bulk-copy / TMA row rings were measured slower and are not instantiated");
  static TmapSet tm;  // kernel argument of the (uninstantiated) TMA row ring
  auto kern = roi_align3d_fwd_ring2_kernel<PW, ROWS, CV, NXU, NS, RXR, MINB, BULK, F2, MULTI>;
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)blocks, kWarps * 32, smem, st>>>(p, tm);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

template <int PW, int ROWS, int CV, int RXR, bool F2 = false>
static int launch_bwd(RoiParams &p, cudaStream_t st) {
  using TB = Tables<PW>;
  constexpr int VOX = 32 * CV;
  constexpr int STAGE = CV * ROWS * PW * 33;
  constexpr int UX = RXR * VOX;
  constexpr int WARP_FLOATS = (TB::FLOATS + 80 / 4 + (STAGE > UX ? STAGE : UX) + 3) / 4 * 4;
  const size_t smem = (size_t)kWarps * WARP_FLOATS * sizeof(float);
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.total_items = (long long)p.K * p.nchunk * p.PD * p.nphg;
  auto kern = roi_align3d_bwd_cl_kernel<PW, ROWS, CV, RXR, F2>;
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = ceil_div_ll(p.total_items, kWarps);
  ROI3D_CHECK_ARG(p.total_items < 2147483647LL, "roi_align3d backward: too many work items");
  kern<<<(unsigned)blocks, kWarps * 32, smem, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

template <int PW, int ROWS, int CV, bool F2 = false, int MINB = 0, int PP = 16>
static int launch_bwd2(RoiParams &p, cudaStream_t st) {
  ROI3D_CHECK_ARG(p.PH <= PP && p.PD <= PP, "roi_align3d backward: table rows narrower than PH / PD");
  using TB = Tables<PW>;
  constexpr int STAGE = CV * ROWS * PW * 33;
  constexpr int WARP_FLOATS = (80 / 4 + STAGE + 3) / 4 * 4;
  constexpr int SH_FLOATS = (RXMAX + 1) * TB::PWP + RYMAX * PP + RZMAX2 * PP + RXMAX + 8;
  const size_t smem = ((size_t)((SH_FLOATS + 3) / 4 * 4) + (size_t)kWarps * WARP_FLOATS) * sizeof(float);
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.items_per_roi = p.nchunk * p.PD * p.nphg;
  p.ctas_per_roi = ceil_div(p.items_per_roi, kWarps);
  p.total_items = (long long)p.K * p.items_per_roi;
  const long long blocks = (long long)p.K * p.ctas_per_roi;
  ROI3D_CHECK_ARG(blocks < 2147483647LL, "roi_align3d backward: too many work items");
  auto kern = roi_align3d_bwd2_kernel<PW, ROWS, CV, F2, MINB, PP>;
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)blocks, kWarps * 32, smem, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

template <int CV>
static int launch_generic(RoiParams &p, bool fwd, cudaStream_t st) {
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = p.PH;
  p.total_items = (long long)p.K * p.nchunk * p.PD * p.nphg;
  const long long blocks = ceil_div_ll(p.total_items, kWarps);
  ROI3D_CHECK_ARG(p.total_items < 2147483647LL, "roi_align3d: too many work items");
  if (fwd)
    roi_align3d_fwd_generic_kernel<CV><<<(unsigned)blocks, kWarps * 32, 0, st>>>(p);
  else
    roi_align3d_bwd_generic_kernel<CV><<<(unsigned)blocks, kWarps * 32, 0, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

static bool aligned(const void *ptr, size_t a) { return (reinterpret_cast<uintptr_t>(ptr) % a) == 0; }

static int pick_cv(const RoiParams &p, bool bwd) {
  int cv = 4;
  for (int l = 0; l < p.num_levels; ++l) {
    const void *ptr = bwd ? (const void *)p.lv[l].grad : (const void *)p.lv[l].feats;
    while (cv > 1 && (p.C % cv != 0 || !aligned(ptr, cv * sizeof(float)))) cv >>= 1;
  }
  return cv;
}

// Forward kernel selection.  g_fwd_variant (roi3d_set_tuning key 0): 0 = auto, 1 = one channel per lane (the
// fallback for C % 2 != 0), 50 = the per-warp ring kernel even where the streamed kernel applies (A/B), 99 = literal.
static int dispatch_fwd(RoiParams &p, cudaStream_t st) {
  if (p.K == 0) return ROI3D_OK;
  const int cvmax = pick_cv(p, false);
  const int v = g_fwd_variant;
  if (v == 99) {  // force the literal path (tests)
    if (cvmax >= 2) return launch_generic<2>(p, true, st);
    return launch_generic<1>(p, true, st);
  }
  if (p.layout == ROI3D_NCDHW) {  // the reference's layout: the streamed kernel's NCDHW twin (bbox branch) or the planar kernel
    if (v == 0 && fwd_stream_ok(p)) return launch_fwd_stream(p, st);
    ROI3D_CHECK_ARG(fwd_planar_ok(p, ROI3D_NCDHW),
                    "NCDHW levels need a 7- or 14-wide square output, 16-byte aligned levels and W %% 4 == 0; convert "
                    "with roi3d_ncdhw_to_ndhwc otherwise");
    return launch_fwd_planar(p, ROI3D_NCDHW, st);
  }
  if (v == 0 && fwd_stream_ok(p)) return launch_fwd_stream(p, st);  // persistent TMA-fed kernel (roi_align3d_stream.cu)
  if ((v == 60 || (v == 0 && p.PW == 14)) && fwd_planar_ok(p, ROI3D_NDHWC)) return launch_fwd_planar(p, ROI3D_NDHWC, st);
  bool ring_ok = p.C % 4 == 0;
  for (int l = 0; l < p.num_levels; ++l) ring_ok = ring_ok && aligned(p.lv[l].feats, 16);
  if (p.PW == 7) {
    if (ring_ok && cvmax >= 2 && v != 1) {
      if (p.PH <= 16 && p.PD <= 16) return launch_fwd_ring2<7, 7, 2, 3, 5, 18, 2, 0, true>(p, st);
      return launch_fwd_ring<7, 7, 2, 3, 4, 18, 2>(p, st);  // per-warp tables (PH or PD > 16)
    }
    if (v == 1 || cvmax == 1) return launch_fwd<7, 7, 1, 3>(p, st);
    return launch_fwd<7, 7, 2, 3>(p, st);
  }
  if (p.PW == 14) {
    if (ring_ok && cvmax >= 2 && v != 1) {
      if (p.PH <= 16 && p.PD <= 16) return launch_fwd_ring2<14, 4, 2, 3, 3, 18, 0, 0, true, true, 7>(p, st);
      return launch_fwd_ring<14, 4, 2, 3, 3, 18>(p, st);  // per-warp tables (PH or PD > 16)
    }
    if (v == 1 || cvmax == 1) return launch_fwd<14, 7, 1, 3>(p, st);
    return launch_fwd<14, 4, 2, 3>(p, st);
  }
  if (cvmax >= 2) return launch_generic<2>(p, true, st);
  return launch_generic<1>(p, true, st);
}

// Backward kernel selection.  g_bwd_variant (key 1): 0 = auto, 1 = one channel per lane, 3 = per-warp tables, 99 = literal.
static int dispatch_bwd(RoiParams &p, cudaStream_t st) {
  if (p.K == 0) return ROI3D_OK;
  const int cvmax = pick_cv(p, true);
  const int v = g_bwd_variant;
  if (v == 99) {
    if (cvmax >= 2) return launch_generic<2>(p, false, st);
    return launch_generic<1>(p, false, st);
  }
  if (p.PW == 7) {
    if (v == 60 && bwd_planar_ok(p)) return launch_bwd_planar(p, st);   // (A/B: the planar backward on 7-wide outputs)
    if (v == 0 && bwd_stream_ok(p)) return launch_bwd_stream(p, st);    // one red per voxel (roi_align3d_stream.cu)
    if (v == 1 || cvmax == 1) return launch_bwd<7, 7, 1, 40>(p, st);
    if ((v == 0 || v == 50) && p.PH <= 16 && p.PD <= 16 && cvmax >= 2) return launch_bwd2<7, 7, 2, true>(p, st);
    return launch_bwd<7, 7, 2, 26>(p, st);  // per-warp tables (v == 3, or PH / PD > 16)
  }
  if (p.PW == 14) {
    if ((v == 0 || v == 60) && bwd_planar_ok(p)) return launch_bwd_planar(p, st);   // transposed planar stages (roi_align3d_planar.cu)
    if (v == 1 || cvmax == 1) return launch_bwd<14, 7, 1, 40>(p, st);
    if ((v == 0 || v == 50) && p.PH <= 16 && p.PD <= 16 && cvmax >= 2) return launch_bwd2<14, 2, 2, true, 4>(p, st);  // 2 ph rows per warp
    return launch_bwd<14, 4, 2, 30>(p, st);  // per-warp tables (v == 3, or PH / PD > 16)
  }
  if (cvmax >= 2) return launch_generic<2>(p, false, st);
  return launch_generic<1>(p, false, st);
}

static int fill_params(RoiParams &p, const roi3d_level_t *levels, int num_levels, int B, int C, const float *rois,
                       int K, int PD, int PH, int PW, int sample_num, float finest_scale, bool bwd) {
  ROI3D_CHECK_ARG(num_levels >= 1 && num_levels <= ROI3D_MAX_LEVELS, "num_levels=%d out of [1,%d]", num_levels,
                  ROI3D_MAX_LEVELS);
  ROI3D_CHECK_ARG(B > 0 && C > 0 && K >= 0, "bad sizes B=%d C=%d K=%d", B, C, K);
  ROI3D_CHECK_ARG(PD > 0 && PH > 0 && PW > 0, "bad output size %dx%dx%d", PD, PH, PW);
  ROI3D_CHECK_ARG(K == 0 || rois != nullptr, "rois is NULL");
  ROI3D_CHECK_ARG(finest_scale > 0.0f || num_levels == 1, "finest_scale must be > 0");
  for (int l = 0; l < num_levels; ++l) {
    ROI3D_CHECK_ARG(levels[l].layout == ROI3D_NDHWC || (!bwd && levels[l].layout == ROI3D_NCDHW),
                    "level %d: bad layout %d (forward: ROI3D_NCDHW or ROI3D_NDHWC; the backward kernels read "
                    "channels-last ROI3D_NDHWC memory, convert with roi3d_ncdhw_to_ndhwc first)",
                    l, levels[l].layout);
    ROI3D_CHECK_ARG(levels[l].layout == levels[0].layout, "level %d: all levels must share one layout", l);
    ROI3D_CHECK_ARG(levels[l].D > 0 && levels[l].H > 0 && levels[l].W > 0, "level %d: bad dims", l);
    ROI3D_CHECK_ARG(bwd ? levels[l].grad_dev != nullptr : levels[l].feats_dev != nullptr, "level %d: NULL pointer", l);
    ROI3D_CHECK_ARG((long long)levels[l].D * levels[l].H * levels[l].W < (1LL << 31), "level %d too large", l);
    ROI3D_CHECK_ARG((long long)levels[l].D * levels[l].H * levels[l].W * C < (1LL << 33), "level %d too large", l);
    p.lv[l].feats = levels[l].feats_dev;
    p.lv[l].grad = levels[l].grad_dev;
    p.lv[l].D = levels[l].D, p.lv[l].H = levels[l].H, p.lv[l].W = levels[l].W;
    p.lv[l].scale = levels[l].spatial_scale, p.lv[l].scale_d = levels[l].spatial_scale_depth;
  }
  p.num_levels = num_levels;
  p.inv_finest = num_levels > 1 ? 1.0f / finest_scale : 0.0f;
  p.B = B, p.C = C, p.rois = rois, p.K = K, p.PD = PD, p.PH = PH, p.PW = PW, p.sample_num = sample_num;
  p.out = nullptr, p.grad_out = nullptr, p.lvls_out = nullptr, p.out_rows = nullptr, p.bug_compat = 0;
  p.layout = levels[0].layout;
  return ROI3D_OK;
}

}  // namespace roi3d

using namespace roi3d;

extern "C" {

int roi3d_set_kernel_timing_events(void *start_event, void *stop_event) {
  g_timing_ev[0] = static_cast<cudaEvent_t>(start_event);
  g_timing_ev[1] = static_cast<cudaEvent_t>(stop_event);
  return ROI3D_OK;
}

int roi3d_set_tuning(int key, int value) {
  if (key == 0) g_fwd_variant = value;
  else if (key == 1) g_bwd_variant = value;
  else if (key == 2) g_fwd_items_per_warp = value;
  else if (key == 4) g_host_pipeline_kb = value;
  else if (key == 6) g_nms_mask_variant = value;
  else if (key == 7) g_fwd_stream_cfg = value;
  else if (key == 9) g_fwd_stream_debug = value;
  else if (key == 10) g_planar_smem_floats = value;
  else if (key == 11) g_topk_sieve = value;
  else return ROI3D_EINVAL;
  return ROI3D_OK;
}

int roi3d_extract_forward(const roi3d_level_t *levels, int num_levels, int B, int C, const float *rois_dev, int K,
                          int PD, int PH, int PW, int sample_num, float finest_scale, float *out_dev,
                          int64_t *lvls_out_dev, void *stream) {
  RoiParams p;
  int rc = fill_params(p, levels, num_levels, B, C, rois_dev, K, PD, PH, PW, sample_num, finest_scale, false);
  if (rc) return rc;
  ROI3D_CHECK_ARG(K == 0 || out_dev != nullptr, "out is NULL");
  p.out = out_dev;
  p.lvls_out = lvls_out_dev;
  return dispatch_fwd(p, (cudaStream_t)stream);
}

int roi3d_extract_backward(const roi3d_level_t *levels, int num_levels, int B, int C, const float *rois_dev, int K,
                           int PD, int PH, int PW, int sample_num, float finest_scale, const float *grad_out_dev,
                           int zero_fill, int bug_compat, void *stream) {
  RoiParams p;
  int rc = fill_params(p, levels, num_levels, B, C, rois_dev, K, PD, PH, PW, sample_num, finest_scale, true);
  if (rc) return rc;
  ROI3D_CHECK_ARG(K == 0 || grad_out_dev != nullptr, "grad_out is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (zero_fill) {
    for (int l = 0; l < num_levels; ++l) {
      const size_t bytes = (size_t)B * C * levels[l].D * levels[l].H * levels[l].W * sizeof(float);
      ROI3D_CUDA(cudaMemsetAsync(levels[l].grad_dev, 0, bytes, st));
    }
  }
  p.grad_out = grad_out_dev;
  p.bug_compat = bug_compat;
  return dispatch_bwd(p, st);
}

int roi3d_extract_backward_deterministic(const roi3d_level_t *levels, int num_levels, int B, int C, const float *rois_dev,
                                         int K, int PD, int PH, int PW, int sample_num, float finest_scale,
                                         const float *grad_out_dev, int accumulate, void *stream) {
  RoiParams p;
  int rc = fill_params(p, levels, num_levels, B, C, rois_dev, K, PD, PH, PW, sample_num, finest_scale, true);
  if (rc) return rc;
  ROI3D_CHECK_ARG(K == 0 || grad_out_dev != nullptr, "grad_out is NULL");
  p.grad_out = grad_out_dev;
  return launch_bwd_det(p, accumulate, (cudaStream_t)stream);
}

int roi3d_roi_align3d_forward(const float *feats_dev, int layout, int B, int C, int D, int H, int W,
                              const float *rois_dev, int K, int PD, int PH, int PW, float spatial_scale,
                              float spatial_scale_depth, int sample_num, float *out_dev, void *stream) {
  roi3d_level_t lv;
  lv.feats_dev = feats_dev, lv.grad_dev = nullptr, lv.layout = layout, lv.D = D, lv.H = H, lv.W = W;
  lv.spatial_scale = spatial_scale, lv.spatial_scale_depth = spatial_scale_depth;
  return roi3d_extract_forward(&lv, 1, B, C, rois_dev, K, PD, PH, PW, sample_num, 56.0f, out_dev, nullptr, stream);
}

int roi3d_roi_align3d_forward_rows(const float *feats_dev, int layout, int B, int C, int D, int H, int W,
                                   const float *rois_dev, int K, int PD, int PH, int PW, float spatial_scale,
                                   float spatial_scale_depth, int sample_num, float *out_dev, const int32_t *out_rows_dev,
                                   void *stream) {
  roi3d_level_t lv;
  lv.feats_dev = feats_dev, lv.grad_dev = nullptr, lv.layout = layout, lv.D = D, lv.H = H, lv.W = W;
  lv.spatial_scale = spatial_scale, lv.spatial_scale_depth = spatial_scale_depth;
  RoiParams p;
  int rc = fill_params(p, &lv, 1, B, C, rois_dev, K, PD, PH, PW, sample_num, 56.0f, false);
  if (rc) return rc;
  ROI3D_CHECK_ARG(K == 0 || out_dev != nullptr, "out is NULL");
  p.out = out_dev;
  p.out_rows = out_rows_dev;
  return dispatch_fwd(p, (cudaStream_t)stream);
}

int roi3d_roi_align3d_backward(const float *grad_out_dev, const float *rois_dev, int K, int PD, int PH, int PW,
                               float spatial_scale, float spatial_scale_depth, int sample_num, float *grad_in_dev,
                               int layout, int B, int C, int D, int H, int W, int zero_fill, int bug_compat,
                               void *stream) {
  roi3d_level_t lv;
  lv.feats_dev = nullptr, lv.grad_dev = grad_in_dev, lv.layout = layout, lv.D = D, lv.H = H, lv.W = W;
  lv.spatial_scale = spatial_scale, lv.spatial_scale_depth = spatial_scale_depth;
  return roi3d_extract_backward(&lv, 1, B, C, rois_dev, K, PD, PH, PW, sample_num, 56.0f, grad_out_dev, zero_fill,
                                bug_compat, stream);
}

int roi3d_map_roi_levels(const float *rois_dev, int K, int num_levels, float finest_scale, int64_t *lvls_dev,
                         void *stream) {
  ROI3D_CHECK_ARG(K >= 0 && num_levels >= 1 && finest_scale > 0.0f, "bad arguments");
  if (K == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(rois_dev && lvls_dev, "NULL pointer");
  map_roi_levels_kernel<<<ceil_div(K, 256), 256, 0, (cudaStream_t)stream>>>(rois_dev, K, num_levels,
                                                                           1.0f / finest_scale, lvls_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

int roi3d_ncdhw_to_ndhwc(const float *src_dev, float *dst_dev, int B, int C, int D, int H, int W, void *stream) {
  ROI3D_CHECK_ARG(src_dev && dst_dev && B > 0 && C > 0 && D > 0 && H > 0 && W > 0, "bad arguments");
  // [C][S] -> [S][C]: rows = C, cols = S
  const long long S = (long long)D * H * W;
  ROI3D_CHECK_ARG(S < (1LL << 31), "level too large");
  return transpose_launch(src_dev, dst_dev, B, C, (int)S, (cudaStream_t)stream);
}

int roi3d_ndhwc_to_ncdhw(const float *src_dev, float *dst_dev, int B, int C, int D, int H, int W, void *stream) {
  ROI3D_CHECK_ARG(src_dev && dst_dev && B > 0 && C > 0 && D > 0 && H > 0 && W > 0, "bad arguments");
  const long long S = (long long)D * H * W;
  ROI3D_CHECK_ARG(S < (1LL << 31), "level too large");
  // [S][C] -> [C][S]: rows = S, cols = C
  return transpose_launch(src_dev, dst_dev, B, (int)S, C, (cudaStream_t)stream);
}

}  // extern "C"

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

// CTA-shared per-RoI tables of the ring2 and bwd2 kernels, whose warps all work on one RoI.
//   Dx[(x - xmin) * PWP + pw], Dy[(y - ymin) * PP2 + ph] (all PH rows), Dz[(z - zmin) * PP2 + pd] (all PD slices);
//   box = xmin, xmax, ymin, ymax, zmin, zmax.  The x extras are each kernel's own: the forward (XANY = false) keeps
//   xlo / xhi[pw] relative to xmin, the backward (XANY = true) keeps xany[x - xmin] and one more zero row of Dx,
//   which its paired x loop may read one past RX.
constexpr int RZMAX2 = 40;
constexpr int PP2 = 16;  // padded row length of the CTA-shared y / z tables (PH, PD <= 16)
template <int PW, bool XANY>
struct CtaTables {
  static constexpr int PWP = Tables<PW>::PWP;
  static constexpr int DX_ROWS = XANY ? RXMAX + 1 : RXMAX;
  static constexpr int XTRA = XANY ? RXMAX : 32;  // xany[RXMAX] or xlo[16] + xhi[16]
  // 200 spare floats keep the forward's shared-memory footprint, and with it the occupancy, as measured
  static constexpr int SPARE = XANY ? 0 : 200;
  static constexpr int FLOATS = (DX_ROWS * PWP + (RYMAX + RZMAX2) * PP2 + XTRA + 8 + SPARE + 3) / 4 * 4;
  float *Dx, *Dy, *Dz;
  int *xlo, *xhi, *xany, *box;
  int xmin, xmax, ymin, ymax, zmin, zmax;
  bool empty, fits;
  __device__ __forceinline__ void bind(float *sm) {
    Dx = sm;
    Dy = Dx + DX_ROWS * PWP;
    Dz = Dy + RYMAX * PP2;
    xlo = xany = reinterpret_cast<int *>(Dz + RZMAX2 * PP2);
    xhi = xlo + 16;
    box = xlo + XTRA;
  }
};

// Builds T for RoI `it`; every thread of the CTA calls it, and it ends with a barrier.  Warp 0 lanes [0,PW) take the
// x bins, warp 1 lanes [0,PH) the y bins, warp 2 lanes [0,PD) the z bins.  A RoI outside the batch is empty.
template <int PW, bool XANY>
__device__ __forceinline__ void build_cta_tables(CtaTables<PW, XANY> &T, const Item &it, int PH, int PD, int warp,
                                                 int lane) {
  constexpr int PWP = CtaTables<PW, XANY>::PWP;
  const int tid = threadIdx.x;
  const int role = (warp == 0 && lane < PW) ? 0 : (warp == 1 && lane < PH) ? 1 : (warp == 2 && lane < PD) ? 2 : -1;
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
    if (lane == 0) T.box[warp * 2] = mn, T.box[warp * 2 + 1] = mx;
  }
  __syncthreads();
  T.xmin = T.box[0], T.xmax = T.box[1], T.ymin = T.box[2], T.ymax = T.box[3], T.zmin = T.box[4], T.zmax = T.box[5];
  T.empty = !it.ok || T.xmax < T.xmin || T.ymax < T.ymin || T.zmax < T.zmin;
  T.fits = T.empty || ((T.xmax - T.xmin < RXMAX) && (T.ymax - T.ymin < RYMAX) && (T.zmax - T.zmin < RZMAX2));
  if (!T.empty && T.fits) {
    const int RX = T.xmax - T.xmin + 1, RY = T.ymax - T.ymin + 1, RZ = T.zmax - T.zmin + 1;
    for (int i = tid; i < (RX + (XANY ? 1 : 0)) * PWP; i += kWarps * 32) T.Dx[i] = 0.0f;
    for (int i = tid; i < RY * PP2; i += kWarps * 32) T.Dy[i] = 0.0f;
    for (int i = tid; i < RZ * PP2; i += kWarps * 32) T.Dz[i] = 0.0f;
    if constexpr (XANY)
      for (int i = tid; i < RX; i += kWarps * 32) T.xany[i] = 0;
  }
  __syncthreads();
  if (!T.empty && T.fits && role >= 0) {
    float *tab = role == 0 ? T.Dx : role == 1 ? T.Dy : T.Dz;
    const int stride = role == 0 ? PWP : PP2;
    const int mn = role == 0 ? T.xmin : role == 1 ? T.ymin : T.zmin;
    for (int i = 0; i < ax.S; ++i) {
      Tap t = axis_tap(axis_coord(ax, lane, i), asize);
      if (t.valid) {
        tab[(t.low - mn) * stride + lane] += t.h;
        tab[(t.high - mn) * stride + lane] += t.l;
        if constexpr (XANY)
          if (role == 0) T.xany[t.low - mn] = 1, T.xany[t.high - mn] = 1;
      }
    }
    if constexpr (!XANY) {
      if (role == 0) {
        T.xlo[lane] = hi >= lo ? lo - T.xmin : 0;
        T.xhi[lane] = hi >= lo ? hi - T.xmin : -1;
      }
    }
  }
  __syncthreads();
}

// A work item's view of a y or z table: its entry j of table row i is t[i * stride + col + j].  Per-warp tables:
// y = (Dy, 8, 0), z = (Dz, 1, 0).  CTA-shared tables: y = (Dy, PP2, ph0), z = (Dz, PP2, pd).
struct TabView {
  const float *t;
  int stride, col;
  __device__ __forceinline__ float at(int i, int j) const { return t[i * stride + col + j]; }
};

// Compact lists of the y rows (of RY, weights in columns [0, rows) of y) and the z slices (of RZ) that carry weight
// for a work item, built with one ballot per 32 rows / slices.  Returns (ny, nz).
template <int ROWS>
__device__ __forceinline__ int2 weighted_rows(TabView y, int rows, int RY, TabView z, int RZ, unsigned char *ylist,
                                              unsigned char *zlist, int lane) {
  int ny = 0, nz = 0;
  for (int y0 = 0; y0 < RY; y0 += 32) {
    const int yy = y0 + lane;
    bool a = false;
    if (yy < RY) {
#pragma unroll
      for (int r = 0; r < ROWS; ++r) a |= (r < rows) && y.at(yy, r) != 0.0f;
    }
    const unsigned bal = __ballot_sync(FULL, a);
    if (a) ylist[ny + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)yy;
    ny += __popc(bal);
  }
#pragma unroll 1  // RZ <= 40: one or two passes; unrolled, this loop lengthens bwd2 by 2-3%
  for (int z0 = 0; z0 < RZ; z0 += 32) {
    const int zz = z0 + lane;
    const bool a = zz < RZ && z.at(zz, 0) != 0.0f;
    const unsigned bal = __ballot_sync(FULL, a);
    if (a) zlist[nz + __popc(bal & ((1u << lane) - 1u))] = (unsigned char)zz;
    nz += __popc(bal);
  }
  __syncwarp();
  return make_int2(ny, nz);
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// Per-warp constants of the forward ring's x-contraction: for every bin pw its first NXU tap weights (0 past the bin's
// support, and everywhere when !use) and the offset of its first tap in a ring row.  Ring rows carry two zero-filled
// pad voxels after the RX real ones, so a zero-weight tap always reads initialised shared memory and tap offsets are
// compile-time constants.  Returns whether a bin has more than NXU taps.
template <int PW, int CV, int NXU>
__device__ __forceinline__ bool x_taps(const float *Dx, const int *xlo, const int *xhi, bool use, int lane,
                                       int (&soff)[PW], float (&tw)[PW][NXU]) {
  constexpr int PWP = Tables<PW>::PWP;
  static_assert(NXU <= 3, "pad voxels cover taps lo+1, lo+2 only");
  bool long_bins = false;
#pragma unroll
  for (int pw = 0; pw < PW; ++pw) {
    const int lo = use ? xlo[pw] : 0;
    const int n = use ? xhi[pw] - lo + 1 : 0;
    long_bins |= n > NXU;
    soff[pw] = lo * 32 * CV + lane * CV;
#pragma unroll
    for (int j = 0; j < NXU; ++j) tw[pw][j] = j < n ? Dx[(lo + j) * PWP + pw] : 0.0f;
  }
  return long_bins;
}

// The cp.async row pipeline of one (pd, ph-group) work item of the forward ring kernels, accumulated into acc.
// The feature rows the item needs ([xmin..xmax] x 32*CV channels of one (z,y) row) are copied global->shared with
// 16-byte cp.async (LDGSTS, no register staging) NS-1 rows ahead of the row being contracted.  Rows are visited
// y-major, z-minor, so that all z slices of one y row are contracted along x back to back and the y-stage runs once
// per y row.  lists: ylist[40] + zlist[40] bytes, then yoff[40] and zoff[] ints.  pstage / cstage are the ring's
// producer and consumer slots; every row issued here is consumed here, so a caller may keep them across items.
// The 16-byte copies need the chunk to lie inside C and be 16-byte aligned: C % 4 == 0 is checked by the
// dispatcher; a partial last chunk (C not a multiple of 32*CV) copies only the lanes inside C.
template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, class TB>
__device__ __forceinline__ void ring_rows(float (&acc)[ROWS][PW][CV], const TB &T, TabView ty, int rows, TabView tz,
                                          const int (&soff)[PW], const float (&tw)[PW][NXU], bool long_bins,
                                          const float *fb_roi, int chunk, int C, int H, int W, unsigned char *lists,
                                          float *ring, int &pstage, int &cstage, int lane) {
  static_assert(CV == 2, "packed f32x2 arithmetic pairs the two channels of a lane");
  constexpr int PWP = Tables<PW>::PWP;
  constexpr int VOX = 32 * CV;                 // floats per voxel-chunk
  constexpr int LPV = VOX / 4;                 // lanes (16 B each) per voxel-chunk
  constexpr int VPI = 32 / LPV;                // voxel-chunks copied per warp instruction
  constexpr int STRIDE = (RXR + 2) * VOX;      // floats per ring stage (two zero pad voxels)
  static_assert(LPV <= 32 && VPI >= 1, "voxel chunk wider than a warp copy");
  unsigned char *ylist = lists, *zlist = lists + 40;
  int *yoff = reinterpret_cast<int *>(lists + 80);
  int *zoff = yoff + 40;
  const int RX = T.xmax - T.xmin + 1;
  const int2 n = weighted_rows<ROWS>(ty, rows, T.ymax - T.ymin + 1, tz, T.zmax - T.zmin + 1, ylist, zlist, lane);
  const int ny = n.x, nz = n.y, nrows = ny * nz;

  for (int sidx = 0; sidx < NS; ++sidx) {
    float *padp = ring + sidx * STRIDE + RX * VOX;
    for (int i = lane; i < 2 * VOX; i += 32) padp[i] = 0.0f;
  }
  __syncwarp();

  // copy geometry: lane -> (voxel within the instruction, 16-byte piece of the voxel chunk)
  const int cv_v = lane / LPV, cv_p = lane % LPV;
  const int ch_piece = chunk * VOX + cv_p * 4;             // first channel of this lane's 16 bytes
  const bool piece_ok = ch_piece + 4 <= C;
  const long long row_elems = (long long)W * C;
  const long long slice_elems = (long long)H * row_elems;
  const float *src0 = fb_roi + ((long long)T.zmin * H + T.ymin) * row_elems + (long long)T.xmin * C + ch_piece +
                      (long long)cv_v * C;
  float *dst0 = ring + cv_p * 4 + cv_v * VOX;
  // row offsets in units of 4 floats (16 B; C % 4 == 0), < 2^31 for any level the dispatcher accepts
  for (int i = lane; i < nz; i += 32) zoff[i] = (int)(((long long)zlist[i] * slice_elems) >> 2);
  for (int i = lane; i < ny; i += 32) yoff[i] = (int)(((long long)ylist[i] * row_elems) >> 2);
  __syncwarp();
  int pz = 0, py = 0;  // producer cursor: the row to prefetch next
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
  int r = 0;
  for (int yi = 0; yi < ny; ++yi) {
    float t1[PW][CV];
#pragma unroll
    for (int pw = 0; pw < PW; ++pw)
#pragma unroll
      for (int c = 0; c < CV; ++c) t1[pw][c] = 0.0f;
    for (int zi = 0; zi < nz; ++zi, ++r) {
      cp_async_wait<NS - 2>();
      __syncwarp();
      const float wz = tz.at(zlist[zi], 0);
      const float *row = ring + cstage * STRIDE;
      if (++cstage == NS) cstage = 0;
      float tzw[PW][CV];
#pragma unroll
      for (int pw = 0; pw < PW; ++pw) {
        const float *q = row + soff[pw];
        // sm_100 packed fp32 (FFMA2 / FMUL2): both channels of the lane in one issue slot; each half is
        // rounded exactly like the scalar fmul / fma, so the pinned arithmetic is unchanged
        float2 z2;
#pragma unroll
        for (int j = 0; j < NXU; ++j) {
          const float2 t = *reinterpret_cast<const float2 *>(q + j * VOX);
          const float2 w2 = make_float2(tw[pw][j], tw[pw][j]);
          z2 = j == 0 ? __fmul2_rn(w2, t) : __ffma2_rn(w2, t, z2);
        }
        tzw[pw][0] = z2.x, tzw[pw][1] = z2.y;
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
            for (int c = 0; c < CV; ++c) tzw[pw][c] = fmaf(w, q[j * VOX + c], tzw[pw][c]);
          }
        }
      }
#pragma unroll
      for (int pw = 0; pw < PW; ++pw) {
        const float2 o = __ffma2_rn(make_float2(wz, wz), make_float2(tzw[pw][0], tzw[pw][1]),
                                    make_float2(t1[pw][0], t1[pw][1]));
        t1[pw][0] = o.x, t1[pw][1] = o.y;
      }
      __syncwarp();
      if (r + NS - 1 < nrows) issue();
      else cp_async_commit();
    }
    // y-stage, once per feature row index y
    const int yy = ylist[yi];
    float wy[ROWS];
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) wy[rr] = rr < rows ? ty.at(yy, rr) : 0.0f;
#pragma unroll
    for (int rr = 0; rr < ROWS; ++rr) {
      if (wy[rr] != 0.0f) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          const float2 o = __ffma2_rn(make_float2(wy[rr], wy[rr]), make_float2(t1[pw][0], t1[pw][1]),
                                      make_float2(acc[rr][pw][0], acc[rr][pw][1]));
          acc[rr][pw][0] = o.x, acc[rr][pw][1] = o.y;
        }
      }
    }
  }
  cp_async_wait<0>();
}

// Stage-in of a backward warp's grad_out tile, [c][bin][33] for its CV channel slots (lane = channel column, padded
// against bank conflicts): 4-byte cp.async copies that transpose on the fly (coalesced global reads), all in flight
// together and committed as one group.
template <int CV>
__device__ __forceinline__ void stage_in_grad(const RoiParams &p, const Item &it, int PW, float *stage, int lane) {
  const int C = p.C, NB = it.rows * PW;
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
    if (lim < (long long)(cols - 1) * col_stride + NB) total = 0;  // rare: zero the tile, copy nothing out of range
    if (total < 32 * NB) {
      for (int i = lane; i < NB * 33; i += 32) st[i] = 0.0f;
      __syncwarp();
    }
    const int ncol = total / NB;
    unsigned sp = (unsigned)__cvta_generic_to_shared(st + lane * 33);
    const float *gp = p.grad_out + g0 + lane;
    // one column (channel run of NB floats) at a time, lanes along the run (cf. copy_out_tile); four columns per
    // iteration through four address registers and immediate shared offsets: a copy still queued in the memory
    // pipeline does not hold up the address update of the next one
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
// Forward, channels-last, separable, rows staged through a per-warp cp.async ring (ring_rows).
//
// Same work split and arithmetic as roi_align3d_fwd_cl_kernel, but each voxel of a feature row is fetched once
// instead of once per tap, the loads of the next rows are in flight while the current row is reduced, and the
// register file no longer holds the taps, which raises occupancy.  Ring capacity per warp is RXR voxels per row;
// wider footprints take the literal path.
// ---------------------------------------------------------------------------------------------
template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB>
__global__ void __launch_bounds__(kWarps * 32, MINB) roi_align3d_fwd_ring_kernel(const RoiParams p) {
  using TB = Tables<PW>;
  constexpr int RING = NS * (RXR + 2) * 32 * CV;  // floats
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int LISTS = 384;                   // ylist[40] + zlist[32] bytes (pad to 80) + yoff[40] + zoff[32] ints
  constexpr int RING_OR_STAGE = RING > STAGE ? RING : STAGE;
  constexpr int WARP_FLOATS = (TB::FLOATS + LISTS / 4 + RING_OR_STAGE + 3) / 4 * 4;
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
  unsigned char *lists = reinterpret_cast<unsigned char *>(sm + ((TB::FLOATS + 3) / 4 * 4));
  float *ring = sm + ((TB::FLOATS + 3) / 4 * 4) + LISTS / 4;
  T.empty = true, T.fits = true;
  if (it.ok) build_tables<PW>(T, it, lane);
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);
  const int RX = T.xmax - T.xmin + 1;

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
    int soff[PW];
    float tw[PW][NXU];
    const bool long_bins = x_taps<PW, CV, NXU>(T.Dx, T.xlo, T.xhi, true, lane, soff, tw);
    int pstage = 0, cstage = 0;
    ring_rows<PW, ROWS, CV, NXU, NS, RXR>(acc, T, TabView{T.Dy, 8, 0}, ROWS, TabView{T.Dz, 1, 0}, soff, tw, long_bins,
                                          fb_roi, it.chunk, C, it.L.H, it.L.W, lists, ring, pstage, cstage, lane);
  }

  // ---- epilogue: divide by the sample count, transpose through smem, stream out ----
  const int NB = it.rows * PW;
  float *stage = ring;  // the ring is drained
  const long long out_base = (((long long)it.krow * C) * p.PD + it.pd) * p.PH * PW + (long long)it.ph0 * PW;
  const long long ch_stride = (long long)p.PD * p.PH * PW;
  copy_out_tile<ROWS, PW, CV>(acc, count, stage, lane, NB, it.chunk, C, p.out + out_base, ch_stride);
}

// Shared-memory layout of the ring2 kernel, shared by the kernel and its launcher.
template <int PW, int ROWS, int CV, int NS, int RXR>
struct Ring2Layout {
  static constexpr int RING = NS * (RXR + 2) * 32 * CV;
  static constexpr int STAGE = ROWS * PW * 33;
  // bytes: ylist[40] + zlist[40] bytes, yoff[40] + zoff[40] ints (0..400).  The 64 bytes at 416 are spare; the
  // size is kept so that the shared-memory footprint, and with it the occupancy, stay as measured.
  static constexpr int LISTS = 480;
  static constexpr int ALIGN = 4;  // floats
  static constexpr int RING_OR_STAGE = RING > STAGE ? RING : STAGE;
  static constexpr int WARP_FLOATS = (LISTS / 4 + RING_OR_STAGE + ALIGN - 1) / ALIGN * ALIGN;
  static constexpr size_t BYTES = ((size_t)CtaTables<PW, false>::FLOATS + (size_t)kWarps * WARP_FLOATS) * sizeof(float);
};

// ---------------------------------------------------------------------------------------------
// Forward ring kernel with CTA-shared per-RoI tables: the four warps of a CTA always work on the same
// RoI (grid = K x ceil(items per RoI / 4)), so the axis tables are built once per CTA by three warps in
// parallel (x, y and z bins) instead of once per warp, and sit once in shared memory.  Everything after
// the table build is the per-warp pipeline of roi_align3d_fwd_ring_kernel.
// ---------------------------------------------------------------------------------------------
template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB, bool MULTI>
__global__ void __launch_bounds__(kWarps * 32, MINB) roi_align3d_fwd_ring2_kernel(const RoiParams p) {
  using ST = CtaTables<PW, false>;
  using LY = Ring2Layout<PW, ROWS, CV, NS, RXR>;
  extern __shared__ __align__(128) float smem_r2[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  ST T;  // CTA-shared per-RoI tables (all warps of a CTA work on the same RoI)
  T.bind(smem_r2);
  float *sm = smem_r2 + ST::FLOATS + warp * LY::WARP_FLOATS;

  // CTA -> (RoI k, group of kWarps * p.items_per_warp consecutive sub-items); warp w takes sub-items
  // first + w, first + w + kWarps, ...  Sub-item order: channel chunk fastest, then pd, then ph-group, so with
  // nchunk == kWarps a warp keeps its channel chunk and walks the pd slices of one RoI.
  const int k = blockIdx.x / p.ctas_per_roi;
  const int items_per_warp = MULTI ? p.items_per_warp : 1;
  const int first = (blockIdx.x - k * p.ctas_per_roi) * kWarps * items_per_warp;
  Item it;
  it.krow = p.out_rows != nullptr ? __ldg(p.out_rows + k) : k;
  it.pd = 0, it.chunk = 0, it.ph0 = 0, it.rows = 0;
  roi_geometry(p, k, it);
  const int C = p.C;
  if (p.lvls_out != nullptr && blockIdx.x == k * p.ctas_per_roi && tid == 0) p.lvls_out[k] = it.lvl;

  build_cta_tables(T, it, p.PH, p.PD, warp, lane);
  // no block-level barriers below: warps run their sub-items independently

  unsigned char *lists = reinterpret_cast<unsigned char *>(sm);
  float *ring = sm + LY::LISTS / 4;
  const float count = (float)(it.axd.S * it.axh.S * it.axw.S);
  const int RX = T.xmax - T.xmin + 1;
  const bool use_ring = !T.empty && T.fits && RX <= RXR;

  // x-contraction constants are RoI-level: shared by all sub-items of the warp
  int soff[PW];
  float tw[PW][NXU];
  const bool long_bins = x_taps<PW, CV, NXU>(T.Dx, T.xlo, T.xhi, use_ring, lane, soff, tw);
  int pstage = 0, cstage = 0;  // ring cursors persist across sub-items (every issued row is consumed)

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

  if (!T.empty)
    ring_rows<PW, ROWS, CV, NXU, NS, RXR>(acc, T, TabView{T.Dy, PP2, it.ph0}, it.rows, TabView{T.Dz, PP2, it.pd}, soff,
                                          tw, long_bins, fb_roi, it.chunk, C, it.L.H, it.L.W, lists, ring, pstage,
                                          cstage, lane);

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
                                              bool active) {
  for (int r = 0; r < it.rows; ++r)
    for (int pw = 0; pw < PW; ++pw) {
      float top[CV];
#pragma unroll
      for (int c = 0; c < CV; ++c) top[c] = stage[(c * it.rows * PW + r * PW + pw) * 33 + lane];
      if (active) literal_bin_bwd<CV>(it, gb, C, it.pd, it.ph0 + r, pw, top);
    }
}

template <int PW, int ROWS, int CV, int RXR>
__global__ void __launch_bounds__(kWarps * 32) roi_align3d_bwd_cl_kernel(const RoiParams p) {
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

  const int NB = it.rows * PW;
  stage_in_grad<CV>(p, it, PW, stage, lane);
  build_tables<PW>(T, it, lane);  // overlaps the copies
  cp_async_wait<0>();
  __syncwarp();
  if (T.empty) return;
  const int RX = T.xmax - T.xmin + 1;
  if (!T.fits || RX > RXR) {
    literal_tile_bwd<CV>(it, gb, C, PW, stage, lane, active);
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

  // compact lists of the y rows / z slices that carry weight, the z slices in one ballot (RZ <= 32).  Kept here rather
  // than in weighted_rows: through the helper this kernel ran 6-8% slower (7-wide, B200 at 1000 W).
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
        for (int pw = 0; pw < PW; ++pw)
#pragma unroll
          for (int c = 0; c < CV; ++c) u[pw][c] = fmaf(wy[r], g[r][pw][c], u[pw][c]);
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
      for (int pw = 0; pw < PW; ++pw)
#pragma unroll
        for (int c = 0; c < CV; ++c) v[c] = fmaf(wx[pw], u[pw][c], v[c]);
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
#pragma unroll
          for (int c = 0; c < CV; ++c) v[c] = zw[zi] * uv[c];
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
template <int PW, int ROWS, int CV, int MINB>
__global__ void __launch_bounds__(kWarps * 32, MINB) roi_align3d_bwd2_kernel(const RoiParams p) {
  static_assert(CV == 2, "packed f32x2 arithmetic pairs the two channels of a lane");
  using ST = CtaTables<PW, true>;
  constexpr int PWP = ST::PWP;
  constexpr int STAGE = CV * ROWS * PW * 33;     // all CV slots of the grad tile at once
  constexpr int LISTS = 80;
  constexpr int WARP_FLOATS = (LISTS / 4 + STAGE + 3) / 4 * 4;
  extern __shared__ __align__(16) float smem_all[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  ST T;
  T.bind(smem_all);
  float *sm = smem_all + ST::FLOATS + warp * WARP_FLOATS;

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
    it.ph0 = (int)phg * ROWS;
    it.rows = min(ROWS, p.PH - it.ph0);
  }
  roi_geometry(p, k, it);
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

  // this warp's grad_out tile is in flight while the CTA builds the tables
  const int NB = it.rows * PW;
  if (valid) stage_in_grad<CV>(p, it, PW, stage, lane);
  build_cta_tables(T, it, p.PH, p.PD, warp, lane);
  if (!valid) return;  // padding warp of the last CTA of this RoI: no block-level barriers below
  cp_async_wait<0>();
  __syncwarp();
  if (T.empty) return;
  if (!T.fits) {
    literal_tile_bwd<CV>(it, gb, C, PW, stage, lane, active);
    return;
  }
  const int RX = T.xmax - T.xmin + 1;
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

  const TabView ty{T.Dy, PP2, it.ph0}, tz{T.Dz, PP2, it.pd};
  const int2 n = weighted_rows<ROWS>(ty, it.rows, T.ymax - T.ymin + 1, tz, T.zmax - T.zmin + 1, ylist, zlist, lane);
  const int ny = n.x, nz = n.y;

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
    zw[zi] = zi < nz ? tz.at(zrel, 0) : 0.0f;
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
      const float wy = r < it.rows ? ty.at(yy, r) : 0.0f;
      if (wy != 0.0f) {
#pragma unroll
        for (int pw = 0; pw < PW; ++pw) {
          const float2 o = __ffma2_rn(make_float2(wy, wy), make_float2(g[r][pw][0], g[r][pw][1]),
                                      make_float2(u[pw][0], u[pw][1]));
          u[pw][0] = o.x, u[pw][1] = o.y;
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
          const float4 t = *reinterpret_cast<const float4 *>(T.Dx + (xx + h) * PWP + t4 * 4);
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
          const float2 o = __ffma2_rn(make_float2(wx[h][pw], wx[h][pw]), make_float2(u[pw][0], u[pw][1]),
                                      make_float2(v[h][0], v[h][1]));
          v[h][0] = o.x, v[h][1] = o.y;
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
          const float2 t = __fmul2_rn(make_float2(zw[zi], zw[zi]), make_float2(v[h][0], v[h][1]));
          o[h][zi][0] = t.x, o[h][zi][1] = t.y;
        }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (xx + h >= RX || (has_gaps && !T.xany[xx + h])) continue;  // warp-uniform
#pragma unroll
        for (int zi = 0; zi < 4; ++zi)
          if (zi < nz) redv<CV>(ad[h][zi], o[h][zi]);
        for (int zi = 4; zi < nz; ++zi) {
          const int zrel = zlist[zi];
          const float wz = tz.at(zrel, 0);
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
extern int g_host_pipeline_kb;        // host_api.cu
extern int g_planar_smem_floats;      // roi_align3d_planar.cu
extern int g_topk_sieve;              // proposal.cu
extern thread_local cudaEvent_t g_timing_ev[2];  // roi_align3d_stream.cu
static int g_bwd_variant = 0;

using RoiKernel = void (*)(RoiParams);

// Per-warp grid: one warp per (RoI, chunk of 32*CV channels, pd, group of ROWS ph rows), kWarps warps per CTA.
static int launch_per_warp(RoiKernel kern, RoiParams &p, int CV, int ROWS, size_t smem, const char *what,
                           cudaStream_t st) {
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.total_items = (long long)p.K * p.nchunk * p.PD * p.nphg;
  ROI3D_CHECK_ARG(p.total_items < 2147483647LL, "%s: too many work items", what);
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)ceil_div_ll(p.total_items, kWarps), kWarps * 32, smem, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

// Per-RoI grid: the kWarps warps of a CTA work on one RoI, each on items_per_warp of its (chunk, pd, ph-group)
// sub-items; ctas_per_roi CTAs per RoI.
static int launch_per_roi(RoiKernel kern, RoiParams &p, int CV, int ROWS, int items_per_warp, size_t smem,
                          const char *what, cudaStream_t st) {
  p.nchunk = ceil_div(p.C, 32 * CV);
  p.nphg = ceil_div(p.PH, ROWS);
  p.items_per_roi = p.nchunk * p.PD * p.nphg;
  p.items_per_warp = items_per_warp;
  p.ctas_per_roi = ceil_div(p.items_per_roi, kWarps * items_per_warp);
  p.total_items = (long long)p.K * p.items_per_roi;
  const long long blocks = (long long)p.K * p.ctas_per_roi;
  ROI3D_CHECK_ARG(blocks < 2147483647LL, "%s: too many work items", what);
  ROI3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)blocks, kWarps * 32, smem, st>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

template <int PW, int ROWS, int CV, int NXU>
static int launch_fwd(RoiParams &p, cudaStream_t st) {
  using TB = Tables<PW>;
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int WARP_FLOATS = ((STAGE > TB::FLOATS ? STAGE : TB::FLOATS) + 3) / 4 * 4;  // 16-byte aligned per warp
  return launch_per_warp(roi_align3d_fwd_cl_kernel<PW, ROWS, CV, NXU>, p, CV, ROWS,
                         (size_t)kWarps * WARP_FLOATS * sizeof(float), "roi_align3d forward", st);
}

template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB = 0>
static int launch_fwd_ring(RoiParams &p, cudaStream_t st) {
  using TB = Tables<PW>;
  constexpr int RING = NS * (RXR + 2) * 32 * CV;
  constexpr int STAGE = ROWS * PW * 33;
  constexpr int RING_OR_STAGE = RING > STAGE ? RING : STAGE;
  constexpr int WARP_FLOATS = (TB::FLOATS + 384 / 4 + RING_OR_STAGE + 3) / 4 * 4;
  return launch_per_warp(roi_align3d_fwd_ring_kernel<PW, ROWS, CV, NXU, NS, RXR, MINB>, p, CV, ROWS,
                         (size_t)kWarps * WARP_FLOATS * sizeof(float), "roi_align3d forward", st);
}

template <int PW, int ROWS, int CV, int NXU, int NS, int RXR, int MINB = 0, bool MULTI = false, int ITEMS = 1>
static int launch_fwd_ring2(RoiParams &p, cudaStream_t st) {
  return launch_per_roi(roi_align3d_fwd_ring2_kernel<PW, ROWS, CV, NXU, NS, RXR, MINB, MULTI>, p, CV, ROWS,
                        MULTI ? ITEMS : 1, Ring2Layout<PW, ROWS, CV, NS, RXR>::BYTES, "roi_align3d forward", st);
}

template <int PW, int ROWS, int CV, int RXR>
static int launch_bwd(RoiParams &p, cudaStream_t st) {
  using TB = Tables<PW>;
  constexpr int STAGE = CV * ROWS * PW * 33;
  constexpr int UX = RXR * 32 * CV;
  constexpr int WARP_FLOATS = (TB::FLOATS + 80 / 4 + (STAGE > UX ? STAGE : UX) + 3) / 4 * 4;
  return launch_per_warp(roi_align3d_bwd_cl_kernel<PW, ROWS, CV, RXR>, p, CV, ROWS,
                         (size_t)kWarps * WARP_FLOATS * sizeof(float), "roi_align3d backward", st);
}

template <int PW, int ROWS, int CV, int MINB = 0>
static int launch_bwd2(RoiParams &p, cudaStream_t st) {
  ROI3D_CHECK_ARG(p.PH <= PP2 && p.PD <= PP2, "roi_align3d backward: table rows narrower than PH / PD");
  constexpr int WARP_FLOATS = (80 / 4 + CV * ROWS * PW * 33 + 3) / 4 * 4;
  return launch_per_roi(roi_align3d_bwd2_kernel<PW, ROWS, CV, MINB>, p, CV, ROWS, 1,
                        ((size_t)CtaTables<PW, true>::FLOATS + (size_t)kWarps * WARP_FLOATS) * sizeof(float),
                        "roi_align3d backward", st);
}

template <int CV>
static int launch_generic(RoiParams &p, bool fwd, cudaStream_t st) {
  return launch_per_warp(fwd ? roi_align3d_fwd_generic_kernel<CV> : roi_align3d_bwd_generic_kernel<CV>, p, CV, 1, 0,
                         "roi_align3d", st);
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

// Forward kernel selection.  g_fwd_variant (roi3d_set_tuning key 0): 0 = auto, 50 = the per-warp ring kernel even
// where the streamed kernel applies (A/B), 60 = the planar kernel on channels-last 7-wide outputs, 99 = literal.
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
    if (ring_ok && cvmax >= 2) {
      if (p.PH <= 16 && p.PD <= 16) return launch_fwd_ring2<7, 7, 2, 3, 5, 18, 2>(p, st);
      return launch_fwd_ring<7, 7, 2, 3, 4, 18, 2>(p, st);  // per-warp tables (PH or PD > 16)
    }
    if (cvmax == 1) return launch_fwd<7, 7, 1, 3>(p, st);
    return launch_fwd<7, 7, 2, 3>(p, st);
  }
  if (p.PW == 14) {
    if (ring_ok && cvmax >= 2) {
      if (p.PH <= 16 && p.PD <= 16) return launch_fwd_ring2<14, 4, 2, 3, 3, 18, 0, true, 7>(p, st);
      return launch_fwd_ring<14, 4, 2, 3, 3, 18>(p, st);  // per-warp tables (PH or PD > 16)
    }
    if (cvmax == 1) return launch_fwd<14, 7, 1, 3>(p, st);
    return launch_fwd<14, 4, 2, 3>(p, st);
  }
  if (cvmax >= 2) return launch_generic<2>(p, true, st);
  return launch_generic<1>(p, true, st);
}

// Backward kernel selection.  g_bwd_variant (key 1): 0 = auto, 50 = the CTA-shared-table kernel even where the
// streamed or planar kernel applies (A/B), 60 = the planar backward on 7-wide outputs.
static int dispatch_bwd(RoiParams &p, cudaStream_t st) {
  if (p.K == 0) return ROI3D_OK;
  const int cvmax = pick_cv(p, true);
  const int v = g_bwd_variant;
  if (p.PW == 7) {
    if (v == 60 && bwd_planar_ok(p)) return launch_bwd_planar(p, st);   // (A/B: the planar backward on 7-wide outputs)
    if (v == 0 && bwd_stream_ok(p)) return launch_bwd_stream(p, st);    // one red per voxel (roi_align3d_stream.cu)
    if (cvmax == 1) return launch_bwd<7, 7, 1, 40>(p, st);
    if ((v == 0 || v == 50) && p.PH <= 16 && p.PD <= 16) return launch_bwd2<7, 7, 2>(p, st);
    return launch_bwd<7, 7, 2, 26>(p, st);  // per-warp tables (PH / PD > 16, or v == 60 where the planar kernel does not apply)
  }
  if (p.PW == 14) {
    if ((v == 0 || v == 60) && bwd_planar_ok(p)) return launch_bwd_planar(p, st);   // transposed planar stages (roi_align3d_planar.cu)
    if (cvmax == 1) return launch_bwd<14, 7, 1, 40>(p, st);
    if ((v == 0 || v == 50) && p.PH <= 16 && p.PD <= 16) return launch_bwd2<14, 2, 2, 4>(p, st);  // 2 ph rows per warp
    return launch_bwd<14, 4, 2, 30>(p, st);  // per-warp tables (PH / PD > 16, or v == 60 where the planar kernel does not apply)
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
  const bool ok = key == 0    ? value == 0 || value == 50 || value == 60 || value == 99
                  : key == 1  ? value == 0 || value == 50 || value == 60
                  : key == 4  ? value >= -1
                  : key == 10 ? value >= 0
                  : key == 11 ? value == -1 || value == 0 || value == 2
                              : false;
  ROI3D_CHECK_ARG(ok, "roi3d_set_tuning: unsupported key %d / value %d", key, value);
  if (key == 0) g_fwd_variant = value;
  else if (key == 1) g_bwd_variant = value;
  else if (key == 4) g_host_pipeline_kb = value;
  else if (key == 10) g_planar_smem_floats = value;
  else g_topk_sieve = value;
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

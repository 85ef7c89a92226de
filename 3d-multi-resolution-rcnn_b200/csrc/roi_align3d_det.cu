// Deterministic RoIAlign3D / RoI-extractor backward for B200 (sm_100a): the gradient gathered by output tile.
//
// The atomic backward kernels (roi_align3d.cu, roi_align3d_stream.cu, roi_align3d_planar.cu) scatter every RoI's
// contribution into the gradient with float reds, so where two RoIs share a voxel the order of the additions -- and
// therefore the last bits of the gradient -- changes from run to run.  Here every gradient voxel has one owner:
//
//   - one CTA owns one tile of DT_Z x DT_Y x DT_X voxels x DT_CH channels of one level and one batch index, keeps
//     the tile's sums in registers and writes each voxel exactly once (no atomics on gradient memory; with
//     accumulate = 0 the store overwrites, so no zero-fill is needed);
//   - the CTA finds the RoIs whose footprint meets its tile with a ballot scan over per-RoI footprint boxes (one
//     small kernel computes them first), DT_SCAN RoIs per step, which yields them in ascending RoI index;
//   - it adds the RoIs in that order, and within one RoI in an order fixed by the tile geometry: the grad_out bins
//     whose weights reach the tile are walked pw-major, then pd, then ph; for every pw the z and y weights are
//     contracted first (V = sum_(pd,ph) Wz[pd][z] Wy[ph][y] g[pd][ph][pw]), then V / count is expanded along x.
//
// Nothing depends on the grid size, the SM count, other streams or timing, so the result is the same bits on every
// run.  Semantics are those of the atomic kernels: per-axis taps from axis_setup / axis_tap, out-of-range samples
// count in the divisor but contribute nothing, an adaptive-sampling RoI with S = 0 on some axis and a RoI whose
// batch index is out of range contribute nothing, levels are picked with roi_level.  Any PD / PH / PW and any C.
#include <limits.h>

#include "common.cuh"
#include "roi_align3d_shared.cuh"

namespace roi3d {

namespace {

constexpr int DT_Z = 4, DT_Y = 8, DT_X = 8;  // gradient tile in voxels (DT_Y == DT_X: one table row length)
constexpr int DT_CH = 64;                     // channels per CTA: lane l holds channels l and l + 32 of the chunk
constexpr int DT_WARPS = 8;                   // warp w owns tile z row w / 2 and y rows (w % 2) * 4 .. + 3
constexpr int DT_THREADS = DT_WARPS * 32;
constexpr int DT_GS = DT_CH + 1;              // padded row of the staged grad_out piece [bin][channel]
constexpr int DT_BCAP = 192;                  // grad_out bins staged at once (48.8 KB)
constexpr int DT_SCAN = DT_THREADS;           // RoIs tested per scan step, one per thread
static_assert(DT_Z * 2 == DT_WARPS && DT_Y == 8 && DT_X == 8, "warp -> (z row, four y rows) mapping");

struct DetArgs {
  RoiParams p;
  const int4 *boxes;                      // [K][2]: (level, batch, z0, z1), (y0, y1, x0, x1); level -1 = no contribution
  long long tile_end[ROI3D_MAX_LEVELS];   // CTAs of levels [0, l], cumulative
  int accumulate;
};

// Voxel span [lo, hi] of the valid taps of one RoI axis (hi < lo: none).
__device__ void axis_span(const Axis &a, int P, int size, int &lo, int &hi) {
  lo = INT_MAX, hi = -1;
  for (int p = 0; p < P; ++p)
    for (int i = 0; i < a.S; ++i) {
      const Tap t = axis_tap(axis_coord(a, p, i), size);
      if (t.valid) lo = min(lo, t.low), hi = max(hi, t.high);
    }
}

// Footprint box of every RoI on its level.  A RoI that contributes nothing (batch index out of range, S = 0 on an
// axis, no valid sample on an axis) gets level -1 and is never listed by a tile.
__global__ void roi_align3d_det_boxes_kernel(const __grid_constant__ RoiParams p, int4 *boxes) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= p.K) return;
  float r[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)k * 7 + i);
  const int lvl = p.num_levels > 1 ? roi_level(r, p.num_levels, p.inv_finest) : 0;
  const LevelDev &L = p.lv[lvl];
  const int b = (int)r[0];
  int4 h = make_int4(-1, 0, 0, -1), q = make_int4(0, -1, 0, -1);
  const Axis aw = axis_setup(r[1], r[3], L.scale, p.PW, p.sample_num);
  const Axis ah = axis_setup(r[2], r[4], L.scale, p.PH, p.sample_num);
  const Axis ad = axis_setup(r[5], r[6], L.scale_d, p.PD, p.sample_num);
  if (b >= 0 && b < p.B && aw.S > 0 && ah.S > 0 && ad.S > 0) {
    int z0, z1, y0, y1, x0, x1;
    axis_span(ad, p.PD, L.D, z0, z1);
    axis_span(ah, p.PH, L.H, y0, y1);
    axis_span(aw, p.PW, L.W, x0, x1);
    if (z1 >= z0 && y1 >= y0 && x1 >= x0) h = make_int4(lvl, b, z0, z1), q = make_int4(y0, y1, x0, x1);
  }
  boxes[2 * (long long)k] = h;
  boxes[2 * (long long)k + 1] = q;
}

__global__ void __launch_bounds__(DT_THREADS, 2) roi_align3d_bwd_det_kernel(const __grid_constant__ DetArgs a) {
  const RoiParams &p = a.p;
  extern __shared__ __align__(16) float smem_det[];
  float *G = smem_det;                                   // [DT_BCAP][DT_GS] staged grad_out piece
  float *Az = G + DT_BCAP * DT_GS;                       // [PD][DT_Z] tile-local weights (z, y, x tables contiguous)
  float *Ay = Az + p.PD * DT_Z;                          // [PH][DT_Y]
  float *Ax = Ay + p.PH * DT_Y;                          // [PW][DT_X]
  int *list = reinterpret_cast<int *>(Ax + p.PW * DT_X); // [DT_SCAN] RoIs of the scan step that meet the tile
  int *wcnt = list + DT_SCAN;                            // [DT_WARPS]
  int *rng = wcnt + DT_WARPS;                            // [3][2] first / last bin with a tap in the tile (z, y, x)

  // ---- this CTA's tile: level, then (batch, z, y, x tile, channel chunk), channel chunk fastest ----
  const long long cta = blockIdx.x;
  int lvl = 0;
  while (cta >= a.tile_end[lvl]) ++lvl;
  const LevelDev L = p.lv[lvl];
  long long t = cta - (lvl > 0 ? a.tile_end[lvl - 1] : 0);
  const int nchunk = (p.C + DT_CH - 1) / DT_CH;
  const int nx = (L.W + DT_X - 1) / DT_X, ny = (L.H + DT_Y - 1) / DT_Y, nz = (L.D + DT_Z - 1) / DT_Z;
  const int chunk = (int)(t % nchunk);
  t /= nchunk;
  const int tx0 = (int)(t % nx) * DT_X;
  t /= nx;
  const int ty0 = (int)(t % ny) * DT_Y;
  t /= ny;
  const int tz0 = (int)(t % nz) * DT_Z;
  const int b = (int)(t / nz);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wz = warp >> 1, wy0 = (warp & 1) * 4;
  const int C = p.C;
  const int c0 = chunk * DT_CH + lane;  // this lane's channels: c0, c0 + 32
  const long long pdhw = (long long)p.PD * p.PH * p.PW;
  const int ntab = p.PD * DT_Z + p.PH * DT_Y + p.PW * DT_X;
  const int nbins_axes = p.PD + p.PH + p.PW;

  float acc[4][DT_X][2];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int x = 0; x < DT_X; ++x) acc[r][x][0] = acc[r][x][1] = 0.0f;
  bool any = false;  // CTA-uniform: some RoI met the tile

  for (int base = 0; base < p.K; base += DT_SCAN) {
    // ---- ascending list of this step's RoIs whose footprint box meets the tile ----
    const int k = base + tid;
    bool hit = false;
    if (k < p.K) {
      const int4 h = __ldg(a.boxes + 2 * (long long)k);
      if (h.x == lvl && h.y == b && h.z <= tz0 + DT_Z - 1 && h.w >= tz0) {
        const int4 q = __ldg(a.boxes + 2 * (long long)k + 1);
        hit = q.x <= ty0 + DT_Y - 1 && q.y >= ty0 && q.z <= tx0 + DT_X - 1 && q.w >= tx0;
      }
    }
    const unsigned bal = __ballot_sync(FULL, hit);
    if (lane == 0) wcnt[warp] = __popc(bal);
    __syncthreads();
    int off = 0, n = 0;
#pragma unroll
    for (int w = 0; w < DT_WARPS; ++w) {
      const int c = wcnt[w];
      off += w < warp ? c : 0;
      n += c;
    }
    if (hit) list[off + __popc(bal & ((1u << lane) - 1u))] = k;
    __syncthreads();
    any |= n > 0;

    for (int li = 0; li < n; ++li) {
      const int kk = list[li];
      float r[7];
#pragma unroll
      for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)kk * 7 + i);
      const Axis aw = axis_setup(r[1], r[3], L.scale, p.PW, p.sample_num);
      const Axis ah = axis_setup(r[2], r[4], L.scale, p.PH, p.sample_num);
      const Axis ad = axis_setup(r[5], r[6], L.scale_d, p.PD, p.sample_num);
      const float inv = __frcp_rn((float)(ad.S * ah.S * aw.S));  // S > 0 on every axis of a listed RoI

      // ---- tile-local weight tables: one thread per bin adds its taps inside the tile in sample order ----
      for (int i = tid; i < ntab; i += DT_THREADS) Az[i] = 0.0f;
      if (tid < 6) rng[tid] = (tid & 1) ? -1 : INT_MAX;
      __syncthreads();
      for (int j = tid; j < nbins_axes; j += DT_THREADS) {
        const int axis = j < p.PD ? 0 : j < p.PD + p.PH ? 1 : 2;
        const int pb = axis == 0 ? j : axis == 1 ? j - p.PD : j - p.PD - p.PH;
        const Axis ax = axis == 0 ? ad : axis == 1 ? ah : aw;
        const int size = axis == 0 ? L.D : axis == 1 ? L.H : L.W;
        const int t0 = axis == 0 ? tz0 : axis == 1 ? ty0 : tx0;
        const int T = axis == 0 ? DT_Z : DT_Y;
        float *row = axis == 0 ? Az + pb * DT_Z : axis == 1 ? Ay + pb * DT_Y : Ax + pb * DT_X;
        bool touched = false;
        for (int i = 0; i < ax.S; ++i) {
          const Tap tp = axis_tap(axis_coord(ax, pb, i), size);
          if (!tp.valid) continue;  // counted in the divisor, contributes nothing
          const int lo = tp.low - t0, hi = tp.high - t0;
          if ((unsigned)lo < (unsigned)T) row[lo] += tp.h, touched = true;
          if ((unsigned)hi < (unsigned)T) row[hi] += tp.l, touched = true;
        }
        if (touched) {  // min / max: the same result in any order
          atomicMin(&rng[2 * axis], pb);
          atomicMax(&rng[2 * axis + 1], pb);
        }
      }
      __syncthreads();
      const int pd0 = rng[0], npd = rng[1] - rng[0] + 1;
      const int ph0 = rng[2], nph = rng[3] - rng[2] + 1;
      const int pw0 = rng[4], npw = rng[5] - rng[4] + 1;
      const int nb = (npd > 0 && nph > 0 && npw > 0) ? npw * npd * nph : 0;
      if (nb == 0) {
        __syncthreads();  // everyone has read rng before the next RoI resets it
        continue;
      }

      // ---- walk the bins pw-major, then pd, then ph, staged in pieces of DT_BCAP bins ----
      const float *gk = p.grad_out + (long long)kk * C * pdhw;
      float V[4][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}, {0.0f, 0.0f}, {0.0f, 0.0f}};
      int ipw = 0, ipd = 0, iph = 0;
      for (int s = 0; s < nb; s += DT_BCAP) {
        const int m = min(nb - s, DT_BCAP);
        // stage grad_out[kk][chunk channels][piece bins] transposed to [bin][channel] (bins fastest in the loads)
        for (int q = tid; q < m * DT_CH; q += DT_THREADS) {
          const int bl = q % m, ch = q / m;
          const int lb = s + bl;
          const int qh = lb % nph, q2 = lb / nph;
          const int qd = q2 % npd, qw = q2 / npd;
          const int c = chunk * DT_CH + ch;
          float v = 0.0f;
          if (c < C) v = __ldg(gk + (long long)c * pdhw + ((long long)(pd0 + qd) * p.PH + (ph0 + qh)) * p.PW + (pw0 + qw));
          G[bl * DT_GS + ch] = v;
        }
        __syncthreads();
        for (int bl = 0; bl < m; ++bl) {
          const float wzv = Az[(pd0 + ipd) * DT_Z + wz];
          if (wzv != 0.0f) {  // warp-uniform
            const float4 wy = *reinterpret_cast<const float4 *>(Ay + (ph0 + iph) * DT_Y + wy0);
            const float g0 = G[bl * DT_GS + lane], g1 = G[bl * DT_GS + lane + 32];
            const float w[4] = {wzv * wy.x, wzv * wy.y, wzv * wy.z, wzv * wy.w};
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
              V[rr][0] = fmaf(w[rr], g0, V[rr][0]);
              V[rr][1] = fmaf(w[rr], g1, V[rr][1]);
            }
          }
          if (++iph == nph) {
            iph = 0;
            if (++ipd == npd) {  // column pw0 + ipw finished: expand V / count along x
              ipd = 0;
              const float4 xa = *reinterpret_cast<const float4 *>(Ax + (pw0 + ipw) * DT_X);
              const float4 xb = *reinterpret_cast<const float4 *>(Ax + (pw0 + ipw) * DT_X + 4);
              const float wx[DT_X] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
              for (int rr = 0; rr < 4; ++rr)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  const float v = V[rr][j] * inv;
                  V[rr][j] = 0.0f;
#pragma unroll
                  for (int x = 0; x < DT_X; ++x) acc[rr][x][j] = fmaf(wx[x], v, acc[rr][x][j]);
                }
              ++ipw;
            }
          }
        }
        __syncthreads();  // G and the tables are free for the next piece / RoI
      }
    }
  }

  // ---- one store per voxel and channel: overwrite, or one fp32 add onto the old value ----
  if (a.accumulate && !any) return;  // nothing to add: the tile stays untouched
  const int z = tz0 + wz;
  if (z >= L.D) return;
  float *gb = L.grad + (long long)b * L.D * L.H * L.W * C;
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    const int y = ty0 + wy0 + rr;
    if (y >= L.H) break;
    const long long rowv = ((long long)z * L.H + y) * L.W;
#pragma unroll
    for (int x = 0; x < DT_X; ++x) {
      if (tx0 + x >= L.W) break;
      float *gp = gb + (rowv + tx0 + x) * C;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int c = c0 + 32 * j;
        if (c < C) gp[c] = a.accumulate ? __fadd_rn(gp[c], acc[rr][x][j]) : acc[rr][x][j];
      }
    }
  }
}

size_t det_smem_bytes(const RoiParams &p) {
  const size_t tab = (size_t)p.PD * DT_Z + (size_t)p.PH * DT_Y + (size_t)p.PW * DT_X;
  return ((size_t)DT_BCAP * DT_GS + tab + DT_SCAN + DT_WARPS + 8) * sizeof(float);
}

}  // namespace

int launch_bwd_det(RoiParams &p, int accumulate, cudaStream_t st) {
  DetArgs a;
  a.p = p;
  a.accumulate = accumulate ? 1 : 0;
  const long long nchunk = ceil_div(p.C, DT_CH);
  long long total = 0;
  for (int l = 0; l < ROI3D_MAX_LEVELS; ++l) {
    if (l < p.num_levels) {
      total += (long long)p.B * ceil_div(p.lv[l].D, DT_Z) * ceil_div(p.lv[l].H, DT_Y) * ceil_div(p.lv[l].W, DT_X) * nchunk;
      a.tile_end[l] = total;
    } else {
      a.tile_end[l] = LLONG_MAX;
    }
  }
  ROI3D_CHECK_ARG(total < 2147483647LL, "roi_align3d deterministic backward: too many gradient tiles");
  const size_t smem = det_smem_bytes(p);
  ROI3D_CHECK_ARG(smem <= 227 * 1024, "roi_align3d deterministic backward: output %dx%dx%d too large for the weight tables",
                  p.PD, p.PH, p.PW);
  int4 *boxes = nullptr;
  if (p.K > 0) {
    cudaMemPool_t pool;
    const int rc = stream_pool(&pool);
    if (rc) return rc;
    ROI3D_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void **>(&boxes), (size_t)p.K * 2 * sizeof(int4), pool, st));
    roi_align3d_det_boxes_kernel<<<ceil_div(p.K, 128), 128, 0, st>>>(p, boxes);
  }
  a.boxes = boxes;
  static PerDeviceSmemOptIn opt_in;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && opt_in.need(smem)) {
    e = cudaFuncSetAttribute(roi_align3d_bwd_det_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) opt_in.mark(smem);
  }
  if (e == cudaSuccess) {
    roi_align3d_bwd_det_kernel<<<(unsigned)total, DT_THREADS, smem, st>>>(a);
    e = cudaGetLastError();
  }
  if (boxes != nullptr) {
    const cudaError_t f = cudaFreeAsync(boxes, st);
    if (e == cudaSuccess) e = f;
  }
  if (e != cudaSuccess) {
    set_error("roi_align3d deterministic backward: %s", cudaGetErrorString(e));
    return ROI3D_ECUDA;
  }
  return ROI3D_OK;
}

}  // namespace roi3d

// RoIAlign3D forward, "streamed" kernel for B200 (sm_100a): persistent CTAs, TMA-fed, warp-specialised.
//
// Replaces (reference, /root/reference):
//   ROIAlignForward3D / bilinear_interpolate_3d   mmdet/ops/roi_align/src/roi_align_kernel.cu:214-291, :64-149
//   SingleRoIExtractor.forward / map_roi_levels    mmdet/models/roi_extractors/single_level.py:58-104
//
// Same separable formulation as roi_align3d.cu (per-axis tap tables built with the compiled reference's rounding
// sequence, common.cuh), different machine mapping:
//
//   * A small plan kernel reduces every RoI once to a 1.2 KB record (FPN level, footprint box, the <= 4 contiguous
//     taps of each x / y / z bin, TMA tiling) and ranks the RoIs by footprint (largest first) so that the dynamic
//     schedule of the main kernel ends on its cheapest items.
//   * The main kernel runs ONE persistent 16-warp CTA per SM.  A work item is (RoI, 64-channel chunk), items are taken
//     from an atomic counter, chunk-major so that the RoIs of one channel chunk (a quarter of the level: L2-sized) run
//     together.  Warp 14 is the producer: it streams the item's footprint -- (z, y) rows of RXB voxels x 64 channels
//     -- into a four-slot shared-memory ring with cp.async.bulk.tensor (TMA, 5-D maps over the channels-last level
//     [B][D][H][W][C], box = 64 channels x RXB voxels x {1,2,4,8} rows), one mbarrier per slot counting bytes; the
//     item's plan record rides on the first tile's barrier as a plain bulk copy.
//   * Warps 0..13 are bin owners: warp (pw, half) holds acc[pd][ph] for its output column pw and 4 (or 3) output rows
//     ph of all PD slices in registers, lanes = channel pairs (packed FFMA2 arithmetic).  For every feature row of a
//     tile inside the y support of its output rows it contracts the row along x ONCE for its pw bin (taps at a
//     warp-uniform offset: LDS.64 + FFMA2), folds the value into the slice partials of its output rows with the row's
//     dense y weights (one broadcast LDS.128), and at the end of a z slice folds the partials into the pd bins that
//     slice feeds.  (Owners used to be (ph, half of the pw bins): every row was then contracted by the ~2 output rows
//     whose support holds it -- 1.75x the shared-memory reads and x-stage arithmetic.)  Every row is read from HBM/L2
//     exactly once per item; owners never wait for each other.
//   * At the end of an item the owners scale by 1 / count and write their bins into a shared-memory image of the
//     item's [64 channels][PD*49] output block, which is contiguous in the [K, C, PD, PH, PW] output; warp 15 writes
//     it back with ONE bulk store (cp.async.bulk.global.shared::cta) while the owners already work on the next item.
//
// RoIs whose bins need more than four contiguous taps, or whose footprint is wider than the tiles, are flagged by the
// plan kernel and evaluated literally (reference sample loops, bit-exact) by the same owner warps.
//
// The file also holds the kernel's NCDHW twin (roi_align3d_fwd_stream_ncdhw_kernel: the reference's layout read in
// place, same plans / owners / storer, producers = warps issuing 16-byte cp.async; see the comment above it) and the
// streamed backward (roi_align3d_bwd_stream_kernel).
#include <cuda.h>

#include <mutex>
#include <vector>

#include "roi_align3d_shared.cuh"

namespace roi3d {

extern thread_local cudaEvent_t g_timing_ev[2];

namespace {

constexpr int ST_OWNERS = 14;          // 7 output rows x 2 halves of the 7 pw bins
constexpr int ST_WARPS = 16;           // owners + producer + storer
constexpr int ST_RMAX = 20;            // widest footprint box in x and y (voxels)
constexpr int ST_RZMAX = 24;           // deepest footprint box
constexpr int ST_CH = 64;              // channels per item
constexpr int ST_XCLS = 20;            // box widths 1, 2, ..., 20 voxels
constexpr int ST_YCLS = 4;             // box heights 1, 2, 4, 8 rows
constexpr int ST_MAX_LEVELS = 4;
constexpr int ST_SORT_MAX = 8192;      // RoIs ranked by footprint up to this K (identity order above)
constexpr int ST_MAX_TILE_ROWS = 32;   // one producer lane per tile row

// NCDHW twin (roi_align3d_fwd_stream_ncdhw_kernel): a ring slot is [64 channels][SN_S floats], SN_S = 4 x odd (16-byte
// aligned channel rows; lanes = channels then fall into 8 bank groups of 4 lanes, which read their four taps in rotated
// order: 32 different banks); the producers are SN_PROD warps issuing 16-byte cp.async (TMA delivers such 48..80-byte
// runs at ~10 B/clk/SM: tools/probe/tma_probe_ncdhw.cu; 4-byte cp.async retires about one lane per clock)
constexpr int SN_S = 164;                   // 4 x 41
constexpr int SN_SLOT = ST_CH * SN_S * 4;   // 41984 bytes = 328 x 128
constexpr int SN_PROD = 4;
constexpr int SN_WARPS = ST_OWNERS + SN_PROD + 1;
constexpr int SN_HALF = 32 * SN_S;          // lane l holds channels l and l + 32
constexpr int SN_EMAX = (SN_S / 4 + 31) / 32;   // 16-byte pieces per lane and tile

constexpr int PLAN_EMPTY = 1;          // output is 0 * (1 / count)
constexpr int PLAN_SLOW = 2;           // literal evaluation
constexpr int PLAN_X3 = 4;             // every x bin fits three taps

constexpr int TILE_FIRST = 1, TILE_LAST = 2, TILE_DONE = 4;

// One per RoI, written by roi_align3d_plan_kernel in schedule order (largest footprint first), copied to shared
// memory with the first tile of each item.  The first 16 words are the header the producer reads.
struct alignas(16) StreamPlan {
  int k, krow, lvl, b;
  int flags, x0, y0, z0;
  int RX, RY, RZ, RXB;
  int rows_per_tile, ntiles, nrows, xcls;
  float inv_count;
  int spt, tps, pad;       // spt = ceil(2^16 / RY): (row * spt) >> 16 == row / RY for the rows of a tile
  int xoff[8];             // first tap of bin pw, voxels from x0 (clamped so that all NT taps stay inside the box)
  float xw[8][4];
  int ylo[8];              // first row (from y0) with weight for bin ph, and how many
  int yn[8];
  float yw[8][4];
  float zwd[ST_RZMAX][8];  // dense: weight of slice z (from z0) in bin pd
  float ywd[ST_RMAX][8];   // dense: weight of row y (from y0) in bin ph
  float xwd[ST_RMAX][8];   // dense: weight of voxel x (from x0) in bin pw (the backward's x expansion)
};
static_assert(sizeof(StreamPlan) % 16 == 0, "bulk copies move multiples of 16 bytes");
constexpr int PLAN_BYTES = (int)sizeof(StreamPlan);

struct TileDesc {
  int plan, nrows, z, y;      // plan slot; rows in this tile; slice / row (from the box origin) of its first row
  int flags, rowfloats, chunk, pad;
};

struct StreamArgs {
  RoiParams p;
  const StreamPlan *plans;  // schedule order
  int *counter;
  const CUtensorMap *maps[ST_MAX_LEVELS];  // [xcls][ycls] per level, device memory
  int total_items;
  int pdhw;           // PD * 49
};

// shared-memory carve-up (bytes from the base) for a ring of NS slots of SLOT bytes
template <int NS, int SLOT>
struct Lay {
  static_assert(NS >= 2 && SLOT % 128 == 0, "ring geometry");
  static constexpr int RING = 0;
  static constexpr int STAGE = RING + NS * SLOT;
  static constexpr int STAGE_BYTES = ST_CH * 7 * 49 * 4;
  static constexpr int PLAN = STAGE + STAGE_BYTES;
  static constexpr int TDESC = PLAN + NS * PLAN_BYTES;
  static constexpr int SDESC = TDESC + NS * (int)sizeof(TileDesc);
  static constexpr int SCHED = SDESC + 2 * 16; // NCDHW twin: item index mailbox of the producer warps (two entries)
  static constexpr int BAR = SCHED + 16;       // full[NS], empty[NS], staging full, staging free
  static constexpr int TOTAL = BAR + (2 * NS + 2) * 8;
  static constexpr int LAUNCH = (TOTAL + 127) / 128 * 128;
  static_assert(STAGE % 128 == 0 && PLAN % 16 == 0 && BAR % 8 == 0, "alignment");
  static_assert(LAUNCH <= 232448, "shared memory budget of one CTA per SM");
};

// ---- PTX helpers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned s_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void st_mbar_init(unsigned mbar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void st_mbar_expect_tx(unsigned mbar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void st_mbar_arrive(unsigned mbar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(mbar) : "memory");
}
// Bounded: a protocol error traps (reported as a launch failure) instead of hanging the GPU.
__device__ __forceinline__ void st_mbar_wait(unsigned mbar, unsigned parity) {
  unsigned ok = 0;
#pragma unroll 1
  for (int spin = 0; spin < (1 << 22); ++spin) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok)
        : "r"(mbar), "r"(parity)
        : "memory");
    if (ok) return;
  }
  __trap();
}
__device__ __forceinline__ void st_bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(mbar)
               : "memory");
}
__device__ __forceinline__ void st_tma_5d(unsigned dst, const CUtensorMap *map, int c0, int c1, int c2, int c3, int c4,
                                          unsigned mbar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], "
      "[%7];\n" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(mbar)
      : "memory");
}
__device__ __forceinline__ void st_bulk_s2g(void *dst, unsigned src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}

__device__ __forceinline__ void add_tap(float (&w)[4], int i, float v) {
  if (i == 0) w[0] += v;
  else if (i == 1) w[1] += v;
  else if (i == 2) w[2] += v;
  else w[3] += v;
}

// ---------------------------------------------------------------------------------------------------------------
// Plan kernel: one warp per RoI.  Lanes 0..7 -> x bins, 8..15 -> y bins, 16..23 -> z bins.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) roi_align3d_plan_kernel(const RoiParams p, StreamPlan *plans, int *counter, int sort,
                                                               int slot_bytes, int counter_init, int ncdhw) {
  extern __shared__ float cost_s[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // programmatic dependent launch: the streamed kernel may be scheduled now; it waits (griddepcontrol.wait) for this
  // grid to finish before it touches the plans or the counter
  asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
  if (blockIdx.x == 0 && threadIdx.x == 0) *counter = counter_init;   // the first items of every CTA are static

  // ---- footprint cost of every RoI (each CTA computes all of them: K is small), then the rank of this CTA's RoIs
  if (sort) {
    for (int k = threadIdx.x; k < p.K; k += blockDim.x) {
      float r[7];
#pragma unroll
      for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)k * 7 + i);
      const int lvl = p.num_levels > 1 ? roi_level(r, p.num_levels, p.inv_finest) : 0;
      const float s = p.lv[lvl].scale, sd = p.lv[lvl].scale_d;
      const float wx = fminf(fmaxf((r[3] - r[1] + 1.0f) * s, 0.0f), 64.0f) + 2.0f;
      const float wy = fminf(fmaxf((r[4] - r[2] + 1.0f) * s, 0.0f), 64.0f) + 2.0f;
      const float wz = fminf(fmaxf((r[6] - r[5] + 1.0f) * sd, 0.0f), 64.0f) + 2.0f;
      if (sort == 2) {
        // spatial order: Morton code of the cell (16 x 16 x 8 voxels) that holds the RoI's centre, level-major --
        // RoIs that overlap run close together in time, so a line fetched for one is still in L2 for the next
        const int cx = min(31, max(0, (int)((r[1] + r[3]) * 0.5f * s) >> 4));
        const int cy = min(31, max(0, (int)((r[2] + r[4]) * 0.5f * s) >> 4));
        const int cz = min(31, max(0, (int)((r[5] + r[6]) * 0.5f * sd) >> 3));
        int code = 0;
#pragma unroll
        for (int bit = 0; bit < 5; ++bit)
          code |= (((cx >> bit) & 1) << (3 * bit)) | (((cy >> bit) & 1) << (3 * bit + 1)) | (((cz >> bit) & 1) << (3 * bit + 2));
        cost_s[k] = (float)((lvl << 15) | code);
      } else {
        cost_s[k] = -(wx * wy * wz);   // largest footprint first
      }
    }
    __syncthreads();
  }
  const int k = blockIdx.x * 8 + warp;
  if (k >= p.K) return;
  int rank = k;
  if (sort) {
    const float mine = cost_s[k];
    rank = 0;
    for (int j = lane; j < p.K; j += 32) {
      const float c = cost_s[j];
      rank += (c < mine) || (c == mine && j < k);
    }
    rank = __reduce_add_sync(FULL, rank);
  }

  // ---- the plan
  float r[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)k * 7 + i);
  const int lvl = p.num_levels > 1 ? roi_level(r, p.num_levels, p.inv_finest) : 0;
  const LevelDev L = p.lv[lvl];
  const int b = (int)r[0];
  const bool ok = b >= 0 && b < p.B;
  if (p.lvls_out != nullptr && lane == 0) p.lvls_out[k] = lvl;
  const Axis axw = axis_setup(r[1], r[3], L.scale, p.PW, p.sample_num);
  const Axis axh = axis_setup(r[2], r[4], L.scale, p.PH, p.sample_num);
  const Axis axd = axis_setup(r[5], r[6], L.scale_d, p.PD, p.sample_num);

  const int role = lane >> 3, bin = lane & 7;
  const int P = role == 0 ? p.PW : role == 1 ? p.PH : role == 2 ? p.PD : 0;
  const Axis ax = role == 1 ? axh : role == 2 ? axd : axw;
  const int asize = role == 1 ? L.H : role == 2 ? L.D : L.W;
  const bool active = bin < P;
  int lo = INT_MAX, hi = -1;
  if (active) {
    for (int i = 0; i < ax.S; ++i) {
      const Tap t = axis_tap(axis_coord(ax, bin, i), asize);
      if (t.valid) lo = min(lo, t.low), hi = max(hi, t.high);
    }
  }
  const int n = hi >= lo ? hi - lo + 1 : 0;
  bool slow = n > 4;
  float w[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  if (active && n > 0 && !slow) {
    for (int i = 0; i < ax.S; ++i) {
      const Tap t = axis_tap(axis_coord(ax, bin, i), asize);
      if (t.valid) {
        add_tap(w, t.low - lo, t.h);
        add_tap(w, t.high - lo, t.l);
      }
    }
  }
  const int x0 = __reduce_min_sync(FULL, role == 0 && n > 0 ? lo : INT_MAX);
  const int x1 = __reduce_max_sync(FULL, role == 0 && n > 0 ? hi : -1);
  const int y0 = __reduce_min_sync(FULL, role == 1 && n > 0 ? lo : INT_MAX);
  const int y1 = __reduce_max_sync(FULL, role == 1 && n > 0 ? hi : -1);
  const int z0 = __reduce_min_sync(FULL, role == 2 && n > 0 ? lo : INT_MAX);
  const int z1 = __reduce_max_sync(FULL, role == 2 && n > 0 ? hi : -1);
  const bool empty = !ok || x1 < x0 || y1 < y0 || z1 < z0;
  const int RX = empty ? 0 : x1 - x0 + 1, RY = empty ? 0 : y1 - y0 + 1, RZ = empty ? 0 : z1 - z0 + 1;
  slow = __any_sync(FULL, slow) || RX > ST_RMAX || RY > ST_RMAX || RZ > ST_RZMAX;
  if (empty) slow = false;
  const bool x3 = !ncdhw && !__any_sync(FULL, role == 0 && n > 3);
  const int NT = x3 ? 3 : 4;
  // box origin and width in x.  Channels-last: the footprint, at least the NT taps of one bin.  NCDHW: whole 16-byte
  // pieces of the level's rows (W % 4 == 0), so the origin moves left to a multiple of 4 and the width is rounded up.
  const int xa = (ncdhw && !empty) ? (x0 & ~3) : x0;
  const int RXB = ncdhw ? (empty ? 4 : ((x0 + RX - xa + 3) & ~3)) : max(4, RX);
  // Tiling: consecutive (z, y) rows of the footprint, as many as fit a ring slot (one producer lane per row).
  const int rows_per_tile = min(ST_MAX_TILE_ROWS, slot_bytes / (RXB * ST_CH * 4));
  const bool stream = !empty && !slow;
  const int nrows = stream ? RY * RZ : 0;
  const int ntiles = stream ? (nrows + rows_per_tile - 1) / rows_per_tile : 1;
  const int spt = stream ? (65536 + RY - 1) / RY : 0, tps = 0;  // spt: 2^16 / RY rounded up (row -> slice without a division)

  StreamPlan *pl = plans + rank;
  if (lane == 0) {
    pl->k = k;
    pl->krow = p.out_rows != nullptr ? __ldg(p.out_rows + k) : k;
    pl->lvl = lvl;
    pl->b = ok ? b : 0;
    pl->flags = (empty ? PLAN_EMPTY : 0) | (slow ? PLAN_SLOW : 0) | (x3 ? PLAN_X3 : 0);
    pl->x0 = empty ? 0 : xa, pl->y0 = empty ? 0 : y0, pl->z0 = empty ? 0 : z0;
    pl->RX = RX, pl->RY = RY, pl->RZ = RZ, pl->RXB = RXB;
    pl->rows_per_tile = rows_per_tile, pl->ntiles = ntiles, pl->nrows = nrows, pl->xcls = RXB - 1;
    // The reference divides by the sample count (roi_align_kernel.cu:288); 1/count is exact for the power-of-two
    // counts of fixed sample_num and within one ulp otherwise; count == 0 gives inf -> 0 * inf = NaN like its 0/0.
    pl->inv_count = __frcp_rn((float)(axd.S * axh.S * axw.S));
    pl->spt = spt, pl->tps = tps, pl->pad = 0;
  }
  // per-bin words; the x taps are shifted right so that tap NT-1 still lies inside the RXB-wide box (the shifted-in weights are 0)
  int off_d = 0;                                 // first voxel of this lane's bin in its dense table (x: after the shift)
  float wd[4] = {0.0f, 0.0f, 0.0f, 0.0f};        // and its weights
  const bool on = n > 0 && stream;
  if (role == 0) {
    int off = on ? lo - xa : 0;
    const int sh = max(0, off + NT - RXB);
    off -= sh;
    if (on) {
#pragma unroll
      for (int t = 0; t < 4; ++t)
        if (t + sh < 4) add_tap(wd, t + sh, w[t]);
    }
    off_d = off;
    pl->xoff[bin] = off;
    *reinterpret_cast<float4 *>(&pl->xw[bin][0]) = make_float4(wd[0], wd[1], wd[2], wd[3]);
  } else if (role == 1 || role == 2) {
    off_d = on ? lo - (role == 1 ? y0 : z0) : 0;
    if (on) wd[0] = w[0], wd[1] = w[1], wd[2] = w[2], wd[3] = w[3];
    if (role == 1) {
      pl->ylo[bin] = off_d;
      pl->yn[bin] = on ? n : 0;
      *reinterpret_cast<float4 *>(&pl->yw[bin][0]) = make_float4(wd[0], wd[1], wd[2], wd[3]);
    }
  }
  // dense [voxel][bin] tables (x, y, z), written by the whole warp: element e = voxel * 8 + bin takes its weight from the
  // lane that owns the bin (role * 8 + bin), consecutive lanes = consecutive floats
#pragma unroll 1
  for (int tb = 0; tb < 3; ++tb) {
    const int nvox = tb == 2 ? ST_RZMAX : ST_RMAX;
    float *base = tb == 0 ? &pl->xwd[0][0] : tb == 1 ? &pl->ywd[0][0] : &pl->zwd[0][0];
    for (int e0 = 0; e0 < nvox * 8; e0 += 32) {
      const int e = e0 + lane, src = tb * 8 + (e & 7);
      const int so = __shfl_sync(FULL, off_d, src);
      const float s0 = __shfl_sync(FULL, wd[0], src), s1 = __shfl_sync(FULL, wd[1], src);
      const float s2 = __shfl_sync(FULL, wd[2], src), s3 = __shfl_sync(FULL, wd[3], src);
      const int t = (e >> 3) - so;
      base[e] = t == 0 ? s0 : t == 1 ? s1 : t == 2 ? s2 : t == 3 ? s3 : 0.0f;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Owner: literal evaluation of this owner's bins of a RoI the tap tables cannot express (rare).
// ---------------------------------------------------------------------------------------------------------------
template <int NPH, bool NC>
__device__ __noinline__ void owner_literal(const RoiParams &p, int k, int lvl, int chunk, int ph0, int pw, int lane,
                                           float *staging, int pdhw) {
  Item it;
  it.k = k, it.krow = k, it.chunk = chunk, it.pd = 0, it.ph0 = ph0, it.rows = 1, it.lvl = lvl;
  float r[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) r[i] = __ldg(p.rois + (long long)k * 7 + i);
  it.L = p.lv[lvl];
  it.b = (int)r[0];
  it.ok = true;
  it.axw = axis_setup(r[1], r[3], it.L.scale, p.PW, p.sample_num);
  it.axh = axis_setup(r[2], r[4], it.L.scale, p.PH, p.sample_num);
  it.axd = axis_setup(r[5], r[6], it.L.scale_d, p.PD, p.sample_num);
  const long long vox = (long long)it.L.D * it.L.H * it.L.W;
  if constexpr (NC) {
    // NCDHW level: channels lane and lane + 32 of the chunk, one plane each
    const long long sy = it.L.W, sz = (long long)it.L.H * it.L.W;
    const float *f0 = it.L.feats + ((long long)it.b * p.C + chunk * ST_CH + lane) * vox;
    const float *f1 = f0 + 32 * vox;
    for (int pd = 0; pd < p.PD; ++pd)
      for (int j = 0; j < NPH; ++j) {
        const int idx = pd * 49 + (ph0 + j) * 7 + pw;
        staging[lane * pdhw + idx] = literal_bin_strided(it.axw, it.axh, it.axd, it.L.D, it.L.H, it.L.W, f0, sz, sy, 1, pd, ph0 + j, pw);
        staging[(lane + 32) * pdhw + idx] = literal_bin_strided(it.axw, it.axh, it.axd, it.L.D, it.L.H, it.L.W, f1, sz, sy, 1, pd, ph0 + j, pw);
      }
  } else {
    const float *fb = it.L.feats + (long long)it.b * vox * p.C + chunk * ST_CH + lane * 2;
    for (int pd = 0; pd < p.PD; ++pd)
      for (int j = 0; j < NPH; ++j) {
        float v[2];
        literal_bin_fwd<2>(it, fb, p.C, pd, ph0 + j, pw, v);
        const int idx = pd * 49 + (ph0 + j) * 7 + pw;
        staging[(2 * lane) * pdhw + idx] = v[0];
        staging[(2 * lane + 1) * pdhw + idx] = v[1];
      }
  }
}

// x-contraction of one feature row for this owner's pw bin, then the fold into the slice partials of its NPH output rows
// with the row's (dense) y weights: a row outside a bin's support has weight 0
template <int NT, int NPH, bool NC>
__device__ __forceinline__ void row_visit(const float *q, const float (&xw)[4], const float *ywrow, float2 (&t2)[NPH],
                                          const int3 rot) {
  // channels-last tile: taps ST_CH floats apart, the lane's two channels adjacent; NCDHW tile: taps adjacent, the lane's
  // two channels SN_HALF floats apart
  float2 v0, v1, v2;
  if constexpr (NC) {
    // q points at this lane's FIRST tap in its rotated order; steps 1..3 are at the lane's offsets (xw is rotated alike)
    v0 = make_float2(q[0], q[SN_HALF]);
    v1 = make_float2(q[rot.x], q[rot.x + SN_HALF]);
    v2 = make_float2(q[rot.y], q[rot.y + SN_HALF]);
  } else {
    v0 = *reinterpret_cast<const float2 *>(q);
    v1 = *reinterpret_cast<const float2 *>(q + ST_CH);
    v2 = *reinterpret_cast<const float2 *>(q + 2 * ST_CH);
  }
  const float4 wy = *reinterpret_cast<const float4 *>(ywrow);
  float2 x = __fmul2_rn(make_float2(xw[0], xw[0]), v0);
  x = __ffma2_rn(make_float2(xw[1], xw[1]), v1, x);
  x = __ffma2_rn(make_float2(xw[2], xw[2]), v2, x);
  if constexpr (NT == 4) {
    float2 v3;
    if constexpr (NC) v3 = make_float2(q[rot.z], q[rot.z + SN_HALF]);
    else v3 = *reinterpret_cast<const float2 *>(q + 3 * ST_CH);
    x = __ffma2_rn(make_float2(xw[3], xw[3]), v3, x);
  }
  t2[0] = __ffma2_rn(make_float2(wy.x, wy.x), x, t2[0]);
  t2[1] = __ffma2_rn(make_float2(wy.y, wy.y), x, t2[1]);
  t2[2] = __ffma2_rn(make_float2(wy.z, wy.z), x, t2[2]);
  if constexpr (NPH == 4) t2[3] = __ffma2_rn(make_float2(wy.w, wy.w), x, t2[3]);
}

// All rows of one tile that carry weight for this owner; z fold at the end of every slice the tile completes.
// The tile holds rows [y, y + nrows) of the footprint's (slice, row) sequence starting in slice z.
template <int NT, int NPH, bool NC>
__device__ __forceinline__ void owner_tile(int nrows, int z, int y, int rowfloats, const StreamPlan *P, const float *tile,
                                           int ph0, int RY, int ylo, int yhi1, const float (&xw)[4], float2 (&t2)[NPH],
                                           float2 (&acc)[7][NPH], const int3 rot) {
  int left = nrows;
  const float *rowp = tile;
  while (left > 0) {
    const int seg = min(left, RY - y);
    const int ya = max(y, ylo), yb = min(y + seg, yhi1);
    const float *q = rowp + (ya - y) * rowfloats;
    const float *yw = &P->ywd[ya][ph0];
#pragma unroll 2
    for (int yy = ya; yy < yb; ++yy) {
      row_visit<NT, NPH, NC>(q, xw, yw, t2, rot);
      q += rowfloats, yw += 8;
    }
    rowp += seg * rowfloats;
    y += seg, left -= seg;
    if (y == RY) {
      const float4 wa = *reinterpret_cast<const float4 *>(&P->zwd[z][0]);
      const float4 wb = *reinterpret_cast<const float4 *>(&P->zwd[z][4]);
      const float wz[7] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z};
#pragma unroll
      for (int pd = 0; pd < 7; ++pd) {
        if (wz[pd] != 0.0f) {
          const float2 w2 = make_float2(wz[pd], wz[pd]);
#pragma unroll
          for (int j = 0; j < NPH; ++j) acc[pd][j] = __ffma2_rn(w2, t2[j], acc[pd][j]);
        }
      }
#pragma unroll
      for (int j = 0; j < NPH; ++j) t2[j] = make_float2(0.0f, 0.0f);
      y = 0, ++z;
    }
  }
}

// Owner warp (pw, half of the output rows): ph0 = 0 with NPH = 4 rows, or ph0 = 4 with NPH = 3.  The first tile of an
// item carries the plan record (or the end-of-work mark); every tile has a descriptor (rows, first slice / row) written by
// the producer before it arms the slot's barrier.
// (Tried and dropped: letting an owner skip the wait for tiles that hold none of its rows -- slower, and a parity
// wait can alias once a warp is more than one use of a slot ahead.)
template <int NPH, int NS, int SLOT, bool NC = false>
__device__ __forceinline__ void owner_loop(const StreamArgs &a, unsigned char *smem, int ph0, int pw, int warp, int lane) {
  using L = Lay<NS, SLOT>;
  const unsigned bar0 = s_u32(smem + L::BAR);
  const unsigned sfull = bar0 + 2 * NS * 8, sfree = sfull + 8;
  float *staging = reinterpret_cast<float *>(smem + L::STAGE);
  const TileDesc *tdesc = reinterpret_cast<const TileDesc *>(smem + L::TDESC);
  const int pdhw = a.pdhw;
  unsigned tile_seq = 0, item_seq = 0;
  for (;;) {  // items
    unsigned slot = tile_seq % NS;
    st_mbar_wait(bar0 + slot * 8, (tile_seq / NS) & 1);
    const TileDesc d = tdesc[slot];
    if (d.flags & TILE_DONE) break;
    const StreamPlan *P = reinterpret_cast<const StreamPlan *>(smem + L::PLAN + d.plan * PLAN_BYTES);
    const int pflags = P->flags;
    int krow = 0;
    bool released = false;
    if (!(pflags & PLAN_SLOW)) {
      // ---- streamed item: acc lives in registers from the first tile to the epilogue
      float2 acc[7][NPH], t2[NPH];
      float xw[4];
#pragma unroll
      for (int pd = 0; pd < 7; ++pd)
#pragma unroll
        for (int j = 0; j < NPH; ++j) acc[pd][j] = make_float2(0.0f, 0.0f);
#pragma unroll
      for (int j = 0; j < NPH; ++j) t2[j] = make_float2(0.0f, 0.0f);
      const int xo = NC ? P->xoff[pw] : P->xoff[pw] * ST_CH;
      int3 rot = make_int3(0, 0, 0);
      int first = 0;
      {
        const float4 w4 = *reinterpret_cast<const float4 *>(&P->xw[pw][0]);
        xw[0] = w4.x, xw[1] = w4.y, xw[2] = w4.z, xw[3] = w4.w;
        if constexpr (NC) {
          // step i reads tap (i + lane / 8) % 4: offsets of steps 1..3 relative to step 0, weights in step order
          const int r0 = (lane >> 3) & 3;
          const float t0 = xw[0], t1 = xw[1], t2w = xw[2], t3 = xw[3];
          xw[0] = r0 == 0 ? t0 : r0 == 1 ? t1 : r0 == 2 ? t2w : t3;
          xw[1] = r0 == 0 ? t1 : r0 == 1 ? t2w : r0 == 2 ? t3 : t0;
          xw[2] = r0 == 0 ? t2w : r0 == 1 ? t3 : r0 == 2 ? t0 : t1;
          xw[3] = r0 == 0 ? t3 : r0 == 1 ? t0 : r0 == 2 ? t1 : t2w;
          first = r0;
          rot = make_int3(((r0 + 1) & 3) - r0, ((r0 + 2) & 3) - r0, ((r0 + 3) & 3) - r0);
        }
      }
      // rows with weight for any of this owner's output rows
      const int RY = P->RY;
      int ylo = RY, yhi1 = 0;
#pragma unroll
      for (int j = 0; j < NPH; ++j) {
        const int n = P->yn[ph0 + j], lo = P->ylo[ph0 + j];
        if (n > 0) ylo = min(ylo, lo), yhi1 = max(yhi1, lo + n);
      }
      TileDesc dt = d;
      for (;;) {  // tiles of the item
        if (dt.nrows > 0) {
          const float *tile = reinterpret_cast<const float *>(smem + L::RING + slot * SLOT) + (NC ? lane * SN_S + first : lane * 2) + xo;
          if (!NC && (pflags & PLAN_X3))
            owner_tile<3, NPH, NC>(dt.nrows, dt.z, dt.y, dt.rowfloats, P, tile, ph0, RY, ylo, yhi1, xw, t2, acc, rot);
          else
            owner_tile<4, NPH, NC>(dt.nrows, dt.z, dt.y, dt.rowfloats, P, tile, ph0, RY, ylo, yhi1, xw, t2, acc, rot);
        }
        ++tile_seq;
        if (dt.flags & TILE_LAST) break;
        __syncwarp();
        if (lane == 0) st_mbar_arrive(bar0 + (NS + slot) * 8);  // slot free
        slot = tile_seq % NS;
        st_mbar_wait(bar0 + slot * 8, (tile_seq / NS) & 1);     // the next tile's bytes have landed
        dt = tdesc[slot];
      }
      // the item's last slot and its plan record go back to the producer BEFORE the epilogue (what the epilogue needs
      // of the plan is in registers): the producer fills it while the owners wait for the staging image and write it
      const float inv = P->inv_count;
      krow = P->krow;
      released = true;
      __syncwarp();
      if (lane == 0) st_mbar_arrive(bar0 + (NS + slot) * 8);
      // the staging image is free once the storer has read out the previous item
      st_mbar_wait(sfree, (item_seq & 1) ^ 1);
      const float2 inv2 = make_float2(inv, inv);
      float *s0 = staging + (NC ? lane : 2 * lane) * pdhw + ph0 * 7 + pw;
      const int second = NC ? 32 * pdhw : pdhw;   // the lane's other channel
#pragma unroll
      for (int pd = 0; pd < 7; ++pd) {
        if (pd * 49 < pdhw) {
#pragma unroll
          for (int j = 0; j < NPH; ++j) {
            const float2 v = __fmul2_rn(acc[pd][j], inv2);
            s0[pd * 49 + j * 7] = v.x;
            s0[second + pd * 49 + j * 7] = v.y;
          }
        }
      }
    } else {
      // ---- literal item (one descriptor-only tile)
      ++tile_seq;
      st_mbar_wait(sfree, (item_seq & 1) ^ 1);
      owner_literal<NPH, NC>(a.p, P->k, P->lvl, d.chunk, ph0, pw, lane, staging, pdhw);
      krow = P->krow;
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");  // generic-proxy writes -> visible to the bulk store
    if (warp == 0 && lane == 0) {
      int *sd = reinterpret_cast<int *>(smem + L::SDESC + (item_seq & 1) * 16);
      sd[0] = krow, sd[1] = d.chunk, sd[2] = 0;
    }
    __syncwarp();
    if (lane == 0) {
      if (!released) st_mbar_arrive(bar0 + (NS + slot) * 8);  // (literal item) its slot and plan record are free
      st_mbar_arrive(sfull);
    }
    ++item_seq;
  }
  // no more items: tell the storer.  Like an item's arrivals these wait for the previous hand-back of the staging
  // image, otherwise an owner that runs ahead would arrive twice in the phase of the item the others still write.
  st_mbar_wait(sfree, (item_seq & 1) ^ 1);
  if (lane == 0) {
    if (warp == 0) reinterpret_cast<int *>(smem + L::SDESC + (item_seq & 1) * 16)[2] = 1;
    st_mbar_arrive(sfull);
  }
}

// Producer warp.  Lane l < 22 keeps word l of an item's header (the first 20 plan words, the chunk, the schedule slot)
// for the current item and the next one; the atomic ticket of item i+3 and the header load of item i+2 are in flight
// while the tiles of item i are issued.  A tile's rows are spread over the lanes: lane l looks at row l (slice and row
// from a multiply by the plan's 2^16 / RY instead of a division), the lanes that start a {8,4,2,1}-row box issue its
// TMA copy.
template <int NS, int SLOT>
__device__ __forceinline__ void producer_loop(const StreamArgs &a, unsigned char *smem, int lane) {
  using L = Lay<NS, SLOT>;
  const unsigned bar0 = s_u32(smem + L::BAR);
  TileDesc *tdesc = reinterpret_cast<TileDesc *>(smem + L::TDESC);
  const int K = a.p.K, total = a.total_items;
  auto ticket = [&]() -> int { return lane == 0 ? atomicAdd(a.counter, 1) : 0; };
  auto header = [&](int idx) -> int {
    if (idx >= total) return 0;
    const int chunk = idx / K, r = idx - chunk * K;
    if (lane < 20) return __ldg(reinterpret_cast<const int *>(a.plans + r) + lane);
    return lane == 20 ? chunk : r;
  };
  // the first three items of a CTA are static (blockIdx.x + {0, 1, 2} * grid; the counter starts behind them): no chain
  // of dependent atomic / header round trips before the first tile is requested
  int idx_cur = (int)blockIdx.x, idx_n1 = (int)(blockIdx.x + gridDim.x);
  int h_cur = header(idx_cur);
  int h_n1 = header(idx_n1);
  int t_n2 = (int)(blockIdx.x + 2 * gridDim.x);
  unsigned tile_seq = 0, item_seq = 0;
  while (idx_cur < total) {
    const int idx_n2 = __shfl_sync(FULL, t_n2, 0);
    t_n2 = ticket();                   // item i+3
    const int h_n2 = header(idx_n2);   // item i+2, consumed in the next trip
    const int lvl = __shfl_sync(FULL, h_cur, 2), b = __shfl_sync(FULL, h_cur, 3);
    const int x0 = __shfl_sync(FULL, h_cur, 5), y0 = __shfl_sync(FULL, h_cur, 6), z0 = __shfl_sync(FULL, h_cur, 7);
    const int RY = __shfl_sync(FULL, h_cur, 9), RZ = __shfl_sync(FULL, h_cur, 10), RXB = __shfl_sync(FULL, h_cur, 11);
    const int rpt = __shfl_sync(FULL, h_cur, 12), ntiles = __shfl_sync(FULL, h_cur, 13);
    const int xcls = __shfl_sync(FULL, h_cur, 15), spt = __shfl_sync(FULL, h_cur, 17), tps = __shfl_sync(FULL, h_cur, 18);
    const int chunk = __shfl_sync(FULL, h_cur, 20), r_sched = __shfl_sync(FULL, h_cur, 21);
    const int rowbytes = RXB * ST_CH * 4;
    const CUtensorMap *maps = a.maps[lvl] + xcls * ST_YCLS;
    const unsigned pslot = item_seq % NS;
    const int nrows = __shfl_sync(FULL, h_cur, 14), magic = spt;
    const int c0 = chunk * ST_CH;
    (void)tps, (void)RZ;
    int r = 0, ys = 0, zs = 0;  // first row of the next tile: index, and (row, slice) from the box origin
    for (int t = 0; t < ntiles; ++t) {
      const unsigned slot = tile_seq % NS;
      st_mbar_wait(bar0 + (NS + slot) * 8, ((tile_seq / NS) & 1) ^ 1);
      const unsigned full = bar0 + slot * 8;
      const int tr = min(rpt, nrows - r);
      if (lane == 0) {
        TileDesc d;
        d.plan = (int)pslot, d.nrows = tr, d.z = zs, d.y = ys;
        d.flags = (t == 0 ? TILE_FIRST : 0) | (t == ntiles - 1 ? TILE_LAST : 0);
        d.rowfloats = RXB * ST_CH, d.chunk = chunk, d.pad = 0;
        tdesc[slot] = d;
        st_mbar_expect_tx(full, (unsigned)(tr * rowbytes + (t == 0 ? PLAN_BYTES : 0)));
        if (t == 0) st_bulk_g2s(s_u32(smem + L::PLAN + pslot * PLAN_BYTES), a.plans + r_sched, PLAN_BYTES, full);
      }
      __syncwarp();
      // row `lane` of the tile: slice dz (from zs) and row y; the slice's run of rows inside this tile is [seg0, seg1);
      // the lanes at the start of a box of its {8,...,8,4,2,1}-row cover issue the copy
      const int pos = ys + lane;
      const int dz = (pos * magic) >> 16;
      const int y = pos - dz * RY;
      const int seg0 = dz == 0 ? ys : 0;
      const int seg1 = min(RY, ys + tr - dz * RY);
      const int n = seg1 - seg0, p = y - seg0;
      const int n8 = n & ~7, rem = n - n8;
      int yc = -1;
      if (p < n8) {
        if ((p & 7) == 0) yc = 3;
      } else {
        const int q = p - n8;
        if (q == 0 && (rem & 4)) yc = 2;
        else if (q == (rem & 4) && (rem & 2)) yc = 1;
        else if (q == (rem & 6) && (rem & 1)) yc = 0;
      }
      if (lane < tr && yc >= 0)
        st_tma_5d(s_u32(smem + L::RING + slot * SLOT) + lane * rowbytes, maps + yc, c0, x0, y0 + y, z0 + zs + dz, b, full);
      r += tr;
      {
        const int pe = ys + tr;
        const int de = (pe * magic) >> 16;
        zs += de, ys = pe - de * RY;
      }
      ++tile_seq;
    }
    ++item_seq;
    idx_cur = idx_n1, h_cur = h_n1;
    idx_n1 = idx_n2, h_n1 = h_n2;
  }
  // sentinel tile
  const unsigned slot = tile_seq % NS;
  st_mbar_wait(bar0 + (NS + slot) * 8, ((tile_seq / NS) & 1) ^ 1);
  if (lane == 0) {
    TileDesc d;
    d.plan = 0, d.nrows = 0, d.z = 0, d.y = 0, d.flags = TILE_DONE, d.rowfloats = 0, d.chunk = 0, d.pad = 0;
    tdesc[slot] = d;
    st_mbar_arrive(bar0 + slot * 8);
  }
}

// Storer warp: one bulk store per item, the staging image is handed back as soon as it has been read.
template <int NS, int SLOT>
__device__ __forceinline__ void storer_loop(const StreamArgs &a, unsigned char *smem, int lane) {
  using L = Lay<NS, SLOT>;
  if (lane != 0) return;
  const unsigned bar0 = s_u32(smem + L::BAR);
  const unsigned sfull = bar0 + 2 * NS * 8, sfree = sfull + 8;
  const unsigned stage_s = s_u32(smem + L::STAGE);
  const unsigned bytes = (unsigned)(ST_CH * a.pdhw * 4);
  for (unsigned n = 0;; ++n) {
    st_mbar_wait(sfull, n & 1);
    const int *sd = reinterpret_cast<const int *>(smem + L::SDESC + (n & 1) * 16);
    if (sd[2]) break;
    float *dst = a.p.out + ((long long)sd[0] * a.p.C + (long long)sd[1] * ST_CH) * a.pdhw;
    st_bulk_s2g(dst, stage_s, bytes);
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    st_mbar_arrive(sfree);
  }
  asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");
}

template <int NS, int SLOT>
__global__ void __launch_bounds__(ST_WARPS * 32, 1) roi_align3d_fwd_stream_kernel(const __grid_constant__ StreamArgs a) {
  using L = Lay<NS, SLOT>;
  extern __shared__ __align__(1024) unsigned char smem[];  // no static shared memory: the window starts at offset 0
  if ((s_u32(smem) & 127u) != 0) __trap();                  // TMA destinations need 128-byte alignment
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned bar0 = s_u32(smem + L::BAR);
  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      st_mbar_init(bar0 + s * 8, 1);                 // full: the producer's arrive + the tile's bytes
      st_mbar_init(bar0 + (NS + s) * 8, ST_OWNERS);   // empty: one arrive per owner warp
    }
    st_mbar_init(bar0 + 2 * NS * 8, ST_OWNERS);       // staging full
    st_mbar_init(bar0 + 2 * NS * 8 + 8, 1);           // staging free
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  // launched as a programmatic dependent of the plan kernel: everything above overlapped with it
  asm volatile("griddepcontrol.wait;\n" ::: "memory");

  if (warp < ST_OWNERS) {
    if (warp < 7) owner_loop<4, NS, SLOT>(a, smem, 0, warp, warp, lane);
    else owner_loop<3, NS, SLOT>(a, smem, 4, warp - 7, warp, lane);
    return;
  }
  if (warp == ST_OWNERS) {
    producer_loop<NS, SLOT>(a, smem, lane);
    return;
  }

  storer_loop<NS, SLOT>(a, smem, lane);
}

// ---------------------------------------------------------------------------------------------------------------
// NCDHW twin: the reference's layout (roi_align_cuda.cpp:35-39) read in place.
//
// Same plans, owners and storer; what changes is the supply.  In NCDHW the 64 channels of a voxel are D*H*W floats
// apart and only the x-run of a footprint row (RX ~ 11 floats) is contiguous.  TMA needs 16-byte aligned box origins
// and moves such 48..80-byte runs at ~10 B/clk/SM (tools/probe/tma_probe_ncdhw.cu); 4-byte cp.async retires about one
// lane per clock (measured: 540 us of supply on C2).  So the producers are SN_PROD warps that issue 16-byte cp.async
// (LDGSTS.128) over whole 16-byte pieces of the level's rows (W % 4 == 0; the plan widens the box to multiples of 4
// voxels): a tile is a run of consecutive (z, y) rows of the footprint, stored per channel as [row][RXB] in a slot of
// [64 channels][SN_S floats]; lane l of a producer warp owns pieces l and l + 32 of the tile (their offset inside a
// channel's volume is computed once per tile) and walks its 64 / SN_PROD channels.  Every producer lane arrives on the
// slot's barrier through cp.async.mbarrier.arrive.noinc (the arrival fires when the lane's copies have landed).
// SN_S = 4 x odd: the owners' lanes = channels fall into 8 groups of 4 lanes per 4-bank group; the four lanes of a
// group read the four taps of a row in rotated order (tap (i + lane / 8) % 4 in step i), so every LDS.32 touches 32
// different banks.
// Schedule order is spatial (Morton order of the RoI centres, level-major) instead of largest-first: DRAM reads on C2
// 1.17 GB -> 0.93 GB (a line fetched for one RoI is still in L2 for its neighbours), same time; items are tickets of an
// atomic counter.  What bounds it (measured on C2): the LSU retires about one cp.async lane per clock whatever its size
// (16 B/clk/SM at best; 778 MB of row pieces in 210 us with the owners idle), a two-slot ring is as fast as three, and the
// owners' LDS traffic shares that pipe (317 us with everything on; planar kernel on the same call: 392 us).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_cp_async16(unsigned dst, const float *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void st_cp_async_arrive(unsigned mbar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];\n" ::"r"(mbar) : "memory");
}

template <int NS>
__device__ __forceinline__ void producer_loop_ncdhw(const StreamArgs &a, unsigned char *smem, int pwarp, int lane) {
  using L = Lay<NS, SN_SLOT>;
  const unsigned bar0 = s_u32(smem + L::BAR);
  TileDesc *tdesc = reinterpret_cast<TileDesc *>(smem + L::TDESC);
  const int K = a.p.K, total = a.total_items, C = a.p.C;
  const bool leader = pwarp == 0 && lane == 0;
  constexpr int CPW = ST_CH / SN_PROD;   // channels per producer warp
  unsigned tile_seq = 0, item_seq = 0;
  // Items: the first two of a CTA are static (blockIdx.x, + grid), later ones are tickets of the atomic counter (it starts
  // at 2 * grid) drawn by the leader one item ahead; the producer warps agree on an item through a two-entry mailbox and
  // one named barrier per item.
  volatile int *sched = reinterpret_cast<volatile int *>(smem + L::SCHED);
  int idx_cur = (int)blockIdx.x, idx_n1 = (int)(blockIdx.x + gridDim.x);
  int t_n2 = leader ? atomicAdd(a.counter, 1) : 0;
  for (;; ++item_seq) {
    if (leader) sched[item_seq & 1] = idx_cur;
    asm volatile("bar.sync 1, %0;\n" ::"n"(SN_PROD * 32) : "memory");
    const int idx = sched[item_seq & 1];
    if (idx >= total) break;
    if (leader) {
      idx_cur = idx_n1, idx_n1 = t_n2;
      t_n2 = atomicAdd(a.counter, 1);
    }
    const int chunk = idx / K, r_sched = idx - chunk * K;
    const int h = lane < 20 ? __ldg(reinterpret_cast<const int *>(a.plans + r_sched) + lane) : 0;
    const int lvl = __shfl_sync(FULL, h, 2), b = __shfl_sync(FULL, h, 3);
    const int x0 = __shfl_sync(FULL, h, 5), y0 = __shfl_sync(FULL, h, 6), z0 = __shfl_sync(FULL, h, 7);
    const int RY = __shfl_sync(FULL, h, 9), RXB = __shfl_sync(FULL, h, 11);
    const int rpt = __shfl_sync(FULL, h, 12), ntiles = __shfl_sync(FULL, h, 13), nrows = __shfl_sync(FULL, h, 14);
    const int magic_y = __shfl_sync(FULL, h, 17);
    const int npr = RXB >> 2;                       // 16-byte pieces per row
    const int magic_x = (65536 + npr - 1) / npr;
    const LevelDev Lv = a.p.lv[lvl];
    const int Wd = Lv.W, HW = Lv.H * Lv.W;
    const long long vox = (long long)Lv.D * HW;
    const float *base = Lv.feats + ((long long)b * C + chunk * ST_CH + pwarp * CPW) * vox;
    const unsigned pslot = item_seq % NS;
    int r = 0, ys = 0, zs = 0;   // first row of the next tile: index, and (row, slice) from the box origin
    for (int t = 0; t < ntiles; ++t) {
      const unsigned slot = tile_seq % NS;
      const int tr = min(rpt, nrows - r);
      // this lane's 16-byte pieces of the tile (piece p = row * RXB / 4 + quarter lands at float 4 p of every channel
      // row): offset inside a channel's volume, -1 = none
      const int np = tr * npr;
      int off[SN_EMAX];
#pragma unroll
      for (int j = 0; j < SN_EMAX; ++j) {
        const int pc = lane + 32 * j;
        const int row = (pc * magic_x) >> 16, q = pc - row * npr;
        const int pos = ys + row;
        const int dz = (pos * magic_y) >> 16, y = pos - dz * RY;
        off[j] = pc < np ? (z0 + zs + dz) * HW + (y0 + y) * Wd + x0 + 4 * q : -1;
      }
      st_mbar_wait(bar0 + (NS + slot) * 8, ((tile_seq / NS) & 1) ^ 1);
      const unsigned full = bar0 + slot * 8;
      if (leader) {
        TileDesc d;
        d.plan = (int)pslot, d.nrows = tr, d.z = zs, d.y = ys;
        d.flags = (t == 0 ? TILE_FIRST : 0) | (t == ntiles - 1 ? TILE_LAST : 0);
        d.rowfloats = RXB, d.chunk = chunk, d.pad = 0;
        tdesc[slot] = d;
        st_mbar_expect_tx(full, t == 0 ? (unsigned)PLAN_BYTES : 0u);
        if (t == 0) st_bulk_g2s(s_u32(smem + L::PLAN + pslot * PLAN_BYTES), a.plans + r_sched, PLAN_BYTES, full);
      }
      const unsigned dst0 = s_u32(smem + L::RING + slot * SN_SLOT) + (unsigned)((pwarp * CPW * SN_S + lane * 4) * 4);
      const float *src = base;
#pragma unroll 4
      for (int c = 0; c < CPW; ++c) {
#pragma unroll
        for (int j = 0; j < SN_EMAX; ++j)
          if (off[j] >= 0) st_cp_async16(dst0 + (unsigned)((c * SN_S + 128 * j) * 4), src + off[j]);
        src += vox;
      }
      st_cp_async_arrive(full);
      r += tr;
      {
        const int pe = ys + tr;
        const int de = (pe * magic_y) >> 16;
        zs += de, ys = pe - de * RY;
      }
      ++tile_seq;
    }
  }
  // sentinel tile
  const unsigned slot = tile_seq % NS;
  st_mbar_wait(bar0 + (NS + slot) * 8, ((tile_seq / NS) & 1) ^ 1);
  if (leader) {
    TileDesc d;
    d.plan = 0, d.nrows = 0, d.z = 0, d.y = 0, d.flags = TILE_DONE, d.rowfloats = 0, d.chunk = 0, d.pad = 0;
    tdesc[slot] = d;
    st_mbar_arrive(bar0 + slot * 8);
  }
  st_cp_async_arrive(bar0 + slot * 8);
}

template <int NS>
__global__ void __launch_bounds__(SN_WARPS * 32, 1) roi_align3d_fwd_stream_ncdhw_kernel(const __grid_constant__ StreamArgs a) {
  using L = Lay<NS, SN_SLOT>;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned bar0 = s_u32(smem + L::BAR);
  if (threadIdx.x == 0) {
    for (int s = 0; s < NS; ++s) {
      st_mbar_init(bar0 + s * 8, SN_PROD * 32 + 1);   // full: every producer lane's copies + the leader's arrive (+ plan bytes)
      st_mbar_init(bar0 + (NS + s) * 8, ST_OWNERS);    // empty: one arrive per owner warp
    }
    st_mbar_init(bar0 + 2 * NS * 8, ST_OWNERS);        // staging full
    st_mbar_init(bar0 + 2 * NS * 8 + 8, 1);            // staging free
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  asm volatile("griddepcontrol.wait;\n" ::: "memory");

  if (warp < ST_OWNERS) {
    if (warp < 7) owner_loop<4, NS, SN_SLOT, true>(a, smem, 0, warp, warp, lane);
    else owner_loop<3, NS, SN_SLOT, true>(a, smem, 4, warp - 7, warp, lane);
    return;
  }
  if (warp < ST_OWNERS + SN_PROD) {
    producer_loop_ncdhw<NS>(a, smem, warp - ST_OWNERS, lane);
    return;
  }
  storer_loop<NS, SN_SLOT>(a, smem, lane);
}

// =================================================================================================================
// Backward of the streamed formulation (bbox branch: 7 x 7 x PD outputs, channels-last gradients, C % 64 == 0).
//
// Replaces (reference): ROIAlignBackward3D / bilinear_interpolate_gradient_3d, roi_align_kernel.cu:519-636, :383-442.
// Same plans and schedule as the forward (one persistent 16-warp CTA per SM, items = (RoI, 64-channel chunk), largest
// footprints first, round-robin over the CTAs).  The item's grad_out block [64 channels][PD * 49] is copied into shared
// memory TRANSPOSED ([element][channel], 4-byte cp.async, the next item's block in flight while this one is reduced),
// so that lanes = channel pairs read it with LDS.64.  The unit of work is then one (z, y) ROW of the footprint per
// warp: V[pw] = sum over the (ph, pd) bins that hold (y, z) of wy * wz * g[pd][ph][pw]  (a handful of warp-uniform
// non-zero weight pairs, 7 LDS.64 + FFMA2 each), then for every voxel x of the row sum_pw wx[x][pw] * V[pw] and ONE
// 8-byte vector red per lane: every voxel of the footprint receives exactly one red per RoI and channel -- the
// per-warp kernel (roi_align3d_bwd2_kernel) issues one per (voxel, pd bin whose support holds z), ~2.6x as many.
// =================================================================================================================
constexpr int SB_GSTRIDE = 66;                              // floats per element of the transposed image (2-way STS conflicts)
constexpr int SB_GBYTES = (343 * SB_GSTRIDE * 4 + 15) / 16 * 16;
constexpr int SB_PLAN = 2 * SB_GBYTES;
constexpr int SB_TOTAL = SB_PLAN + 2 * PLAN_BYTES;
static_assert(SB_TOTAL <= 232448, "shared memory budget of one CTA per SM");

__global__ void __launch_bounds__(ST_WARPS * 32, 1) roi_align3d_bwd_stream_kernel(const __grid_constant__ StreamArgs a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int K = a.p.K, total = a.total_items, pdhw = a.pdhw, C = a.p.C;
  asm volatile("griddepcontrol.wait;\n" ::: "memory");   // the plans come from the kernel launched just before

  auto issue_load = [&](int idx, int buf) {
    const int chunk = idx / K, r = idx - chunk * K;
    const StreamPlan *gp = a.plans + r;
    if (tid < PLAN_BYTES / 16) {
      const unsigned dst = s_u32(smem + SB_PLAN + buf * PLAN_BYTES) + tid * 16;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(reinterpret_cast<const char *>(gp) + tid * 16)
                   : "memory");
    }
    const int k = __ldcg(&gp->k);
    const float *src = a.p.grad_out + ((long long)k * C + (long long)chunk * ST_CH) * pdhw;
    const unsigned g0 = s_u32(smem + buf * SB_GBYTES);
    for (int ch = warp; ch < ST_CH; ch += ST_WARPS) {
      const float *sp = src + (long long)ch * pdhw;
      for (int e = lane; e < pdhw; e += 32) {
        const unsigned dst = g0 + (unsigned)(e * SB_GSTRIDE + ch) * 4u;
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(sp + e) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };

  int idx = (int)blockIdx.x;
  if (idx < total) issue_load(idx, 0);
  for (int it_n = 0; idx < total; ++it_n, idx += (int)gridDim.x) {
    const int buf = it_n & 1;
    const int nxt = idx + (int)gridDim.x;
    if (nxt < total) {
      issue_load(nxt, buf ^ 1);
      asm volatile("cp.async.wait_group 1;\n" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    }
    __syncthreads();
    const StreamPlan *P = reinterpret_cast<const StreamPlan *>(smem + SB_PLAN + buf * PLAN_BYTES);
    const float *G = reinterpret_cast<const float *>(smem + buf * SB_GBYTES) + lane * 2;
    const int chunk = idx / K;
    const int pflags = P->flags;
    if (!(pflags & (PLAN_EMPTY | PLAN_SLOW))) {
      const LevelDev L = a.p.lv[P->lvl];
      const int RY = P->RY, RX = P->RX, nrows = P->nrows, spt = P->spt;
      const float inv = P->inv_count;
      float *gbase = L.grad + ((((long long)P->b * L.D + P->z0) * L.H + P->y0) * L.W + P->x0) * C + chunk * ST_CH + lane * 2;
      for (int row = warp; row < nrows; row += ST_WARPS) {
        const int z = (row * spt) >> 16, y = row - z * RY;
        float wy[8], wz[8];
        {
          const float4 ya = *reinterpret_cast<const float4 *>(&P->ywd[y][0]), yb = *reinterpret_cast<const float4 *>(&P->ywd[y][4]);
          const float4 za = *reinterpret_cast<const float4 *>(&P->zwd[z][0]), zb = *reinterpret_cast<const float4 *>(&P->zwd[z][4]);
          wy[0] = ya.x, wy[1] = ya.y, wy[2] = ya.z, wy[3] = ya.w, wy[4] = yb.x, wy[5] = yb.y, wy[6] = yb.z, wy[7] = yb.w;
          wz[0] = za.x * inv, wz[1] = za.y * inv, wz[2] = za.z * inv, wz[3] = za.w * inv;
          wz[4] = zb.x * inv, wz[5] = zb.y * inv, wz[6] = zb.z * inv, wz[7] = zb.w * inv;
        }
        float2 V[7];
#pragma unroll
        for (int pw = 0; pw < 7; ++pw) V[pw] = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int ph = 0; ph < 7; ++ph) {
          if (wy[ph] != 0.0f) {   // warp-uniform
#pragma unroll
            for (int pd = 0; pd < 7; ++pd) {
              if (wz[pd] != 0.0f) {
                const float w = wy[ph] * wz[pd];
                const float2 w2 = make_float2(w, w);
                const float *gp = G + (pd * 49 + ph * 7) * SB_GSTRIDE;
#pragma unroll
                for (int pw = 0; pw < 7; ++pw)
                  V[pw] = __ffma2_rn(w2, *reinterpret_cast<const float2 *>(gp + pw * SB_GSTRIDE), V[pw]);
              }
            }
          }
        }
        float *dst = gbase + ((long long)z * L.H + y) * L.W * C;
        const float4 *xw4 = reinterpret_cast<const float4 *>(&P->xwd[0][0]);
#pragma unroll 2
        for (int x = 0; x < RX; ++x) {
          const float4 xa = xw4[0], xb = xw4[1];
          float2 acc = __fmul2_rn(make_float2(xa.x, xa.x), V[0]);
          acc = __ffma2_rn(make_float2(xa.y, xa.y), V[1], acc);
          acc = __ffma2_rn(make_float2(xa.z, xa.z), V[2], acc);
          acc = __ffma2_rn(make_float2(xa.w, xa.w), V[3], acc);
          acc = __ffma2_rn(make_float2(xb.x, xb.x), V[4], acc);
          acc = __ffma2_rn(make_float2(xb.y, xb.y), V[5], acc);
          acc = __ffma2_rn(make_float2(xb.z, xb.z), V[6], acc);
          atomicAdd(reinterpret_cast<float2 *>(dst), acc);
          dst += C, xw4 += 2;
        }
      }
    } else if (pflags & PLAN_SLOW) {
      // literal gradient of the bins of a RoI the tables cannot express (rare): one bin per warp and trip
      Item it;
      const int k = P->k;
      it.k = k, it.krow = k, it.chunk = chunk, it.pd = 0, it.ph0 = 0, it.rows = 1, it.lvl = P->lvl;
      float r[7];
#pragma unroll
      for (int i = 0; i < 7; ++i) r[i] = __ldg(a.p.rois + (long long)k * 7 + i);
      it.L = a.p.lv[it.lvl];
      it.b = (int)r[0];
      it.ok = true;
      it.axw = axis_setup(r[1], r[3], it.L.scale, a.p.PW, a.p.sample_num);
      it.axh = axis_setup(r[2], r[4], it.L.scale, a.p.PH, a.p.sample_num);
      it.axd = axis_setup(r[5], r[6], it.L.scale_d, a.p.PD, a.p.sample_num);
      const long long vox = (long long)it.L.D * it.L.H * it.L.W;
      float *gb = it.L.grad + (long long)it.b * vox * C + chunk * ST_CH + lane * 2;
      for (int e = warp; e < pdhw; e += ST_WARPS) {
        const int pd = e / 49, q = e - pd * 49, ph = q / 7, pw = q - ph * 7;
        const float2 t2 = *reinterpret_cast<const float2 *>(G + e * SB_GSTRIDE);
        const float top[2] = {t2.x, t2.y};
        literal_bin_bwd<2>(it, gb, C, pd, ph, pw, top);
      }
    }
    __syncthreads();   // everyone is done with this buffer before the next trip's loads overwrite it
  }
}

// ---- host: tensor maps -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(ptr);
  }();
  return fn;
}

// Device-resident map tables, one per (device, level pointer, shape): a detector hands the same FPN buffers to the
// extractor call after call, so the 40 descriptors of a level are encoded and uploaded once.  Entries are immutable;
// the oldest is dropped with cudaFree (which waits for the device) when the cache is full.
struct MapEntry {
  int dev;
  const void *ptr;
  int B, C, D, H, W;
  CUtensorMap *maps_dev;
};
std::mutex g_map_mutex;
std::vector<MapEntry> g_map_cache;
constexpr size_t MAP_CACHE_MAX = 64;

int level_maps(const LevelDev &L, int B, int C, const CUtensorMap **out) {
  int dev = 0;
  ROI3D_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_map_mutex);
  for (size_t i = 0; i < g_map_cache.size(); ++i) {
    const MapEntry &e = g_map_cache[i];
    if (e.dev == dev && e.ptr == L.feats && e.B == B && e.C == C && e.D == L.D && e.H == L.H && e.W == L.W) {
      *out = e.maps_dev;
      return ROI3D_OK;
    }
  }
  EncodeTiledFn enc = encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return ROI3D_ECUDA;
  }
  CUtensorMap host[ST_XCLS * ST_YCLS];
  const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)L.W, (cuuint64_t)L.H, (cuuint64_t)L.D, (cuuint64_t)B};
  const cuuint64_t strides[4] = {(cuuint64_t)C * 4, (cuuint64_t)L.W * C * 4, (cuuint64_t)L.H * L.W * C * 4,
                                 (cuuint64_t)L.D * L.H * L.W * C * 4};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  for (int xc = 0; xc < ST_XCLS; ++xc)
    for (int yc = 0; yc < ST_YCLS; ++yc) {
      const cuuint32_t box[5] = {(cuuint32_t)ST_CH, (cuuint32_t)(xc + 1), (cuuint32_t)(1 << yc), 1, 1};
      const CUresult r = enc(&host[xc * ST_YCLS + yc], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float *>(L.feats),
                             dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (CUresult %d) for a %dx%dx%dx%dx%d level", (int)r, B, C, L.D, L.H, L.W);
        return ROI3D_ECUDA;
      }
    }
  if (g_map_cache.size() >= MAP_CACHE_MAX) {
    cudaFree(g_map_cache.front().maps_dev);
    g_map_cache.erase(g_map_cache.begin());
  }
  MapEntry e;
  e.dev = dev, e.ptr = L.feats, e.B = B, e.C = C, e.D = L.D, e.H = L.H, e.W = L.W, e.maps_dev = nullptr;
  ROI3D_CUDA(cudaMalloc(&e.maps_dev, sizeof(host)));
  ROI3D_CUDA(cudaMemcpy(e.maps_dev, host, sizeof(host), cudaMemcpyHostToDevice));
  g_map_cache.push_back(e);
  *out = e.maps_dev;
  return ROI3D_OK;
}

}  // namespace

bool fwd_stream_ok(const RoiParams &p) {
  if (p.PW != 7 || p.PH != 7 || p.PD < 1 || p.PD > 7) return false;
  if (p.layout == ROI3D_NCDHW)   // 32-bit offsets inside one channel's volume
    for (int l = 0; l < p.num_levels; ++l)
      if ((long long)p.lv[l].D * p.lv[l].H * p.lv[l].W >= 2147483647LL || p.lv[l].W % 4 != 0) return false;   // 16-byte row pieces
  if (p.C % ST_CH != 0 || p.num_levels > ST_MAX_LEVELS) return false;
  if ((reinterpret_cast<uintptr_t>(p.out) & 15) != 0) return false;
  if ((long long)p.K * (p.C / ST_CH) >= 2147483647LL) return false;
  for (int l = 0; l < p.num_levels; ++l) {
    if ((reinterpret_cast<uintptr_t>(p.lv[l].feats) & 15) != 0) return false;
    if ((long long)p.lv[l].D * p.lv[l].H * p.lv[l].W * p.C * 4 >= (1LL << 40)) return false;  // TMA stride field
  }
  if (p.out_rows != nullptr) {
    // a row-mapped output may be mapped host memory (roi3d_roi_align3d_forward_host): bulk stores stay on device memory
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p.out) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
      cudaGetLastError();
      return false;
    }
  }
  return true;
}

// Plans and the work counter come from a private stream-ordered pool: no host sync, re-entrant across streams, and
// (release threshold = max) the pages stay with the pool between calls instead of going back to the driver at every
// synchronisation as the default pool would do.
int stream_pool(cudaMemPool_t *out) {
  static std::mutex mu;
  static cudaMemPool_t pools[64] = {};
  int dev = 0;
  ROI3D_CUDA(cudaGetDevice(&dev));
  ROI3D_CHECK_ARG(dev >= 0 && dev < 64, "device index %d out of range", dev);
  std::lock_guard<std::mutex> lock(mu);
  if (pools[dev] == nullptr) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool = nullptr;
    ROI3D_CUDA(cudaMemPoolCreate(&pool, &props));
    unsigned long long keep = ~0ULL;
    ROI3D_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    pools[dev] = pool;
  }
  *out = pools[dev];
  return ROI3D_OK;
}


namespace {

// Plan workspace of the streamed kernels: one grow-only buffer per (device, stream).  Calls on one stream are ordered, so
// the next call's plan kernel cannot overwrite plans the previous call's main kernel still reads; calls on different
// streams get different buffers (re-entrant across streams).  (A stream-ordered pool allocation per call costs ~3 us of
// stream work around each launch pair.)
struct PlanWs {
  int dev;
  cudaStream_t st;
  unsigned char *ptr;
  size_t bytes;
};
std::mutex g_planws_mutex;
std::vector<PlanWs> g_planws;

int plan_workspace(size_t bytes, cudaStream_t st, unsigned char **out) {
  int dev = 0;
  ROI3D_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_planws_mutex);
  for (PlanWs &e : g_planws) {
    if (e.dev == dev && e.st == st) {
      if (e.bytes < bytes) {
        // the old buffer may still be read by work enqueued on this stream: release it in stream order
        ROI3D_CUDA(cudaFreeAsync(e.ptr, st));
        e.ptr = nullptr, e.bytes = 0;
        ROI3D_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&e.ptr), bytes, st));
        e.bytes = bytes;
      }
      *out = e.ptr;
      return ROI3D_OK;
    }
  }
  PlanWs e;
  e.dev = dev, e.st = st, e.ptr = nullptr, e.bytes = bytes < (1u << 20) ? (1u << 20) : bytes;
  ROI3D_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&e.ptr), e.bytes, st));
  if (g_planws.size() >= 256) {   // streams come and go: forget the oldest entry (its buffer is released in ITS stream's order)
    cudaFreeAsync(g_planws.front().ptr, g_planws.front().st);
    g_planws.erase(g_planws.begin());
  }
  g_planws.push_back(e);
  *out = e.ptr;
  return ROI3D_OK;
}

// Under stream capture the workspace comes from the stream-ordered pool instead (alloc / free nodes inside the graph: a
// replayed graph owns its plans); *pooled tells the caller to free it after the launches.
int acquire_plan_ws(size_t bytes, cudaStream_t st, unsigned char **ws, bool *pooled) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  ROI3D_CUDA(cudaStreamIsCapturing(st, &cap));
  cudaMemPool_t pool;
  if (cap == cudaStreamCaptureStatusNone) {
    const int rc0 = stream_pool(&pool);   // created here, outside any capture (pool creation is not capturable)
    if (rc0) return rc0;
    *pooled = false;
    return plan_workspace(bytes, st, ws);
  }
  const int rc = stream_pool(&pool);
  if (rc) return rc;
  ROI3D_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void **>(ws), bytes, pool, st));
  *pooled = true;
  return ROI3D_OK;
}

template <int NS, int SLOT, bool NC = false>
int launch_cfg(const RoiParams &p, StreamArgs &a, cudaStream_t st, int sm_count) {
  using L = Lay<NS, SLOT>;
  auto kernel = [] {
    if constexpr (NC) return roi_align3d_fwd_stream_ncdhw_kernel<NS>;
    else return roi_align3d_fwd_stream_kernel<NS, SLOT>;
  }();
  const size_t plan_bytes = (size_t)p.K * sizeof(StreamPlan);
  unsigned char *ws = nullptr;
  bool pooled = false;
  int rc = acquire_plan_ws(plan_bytes + 16, st, &ws, &pooled);
  if (rc) return rc;
  StreamPlan *plans = reinterpret_cast<StreamPlan *>(ws);
  int *counter = reinterpret_cast<int *>(ws + plan_bytes);
  const int sort = p.K <= ST_SORT_MAX ? 1 : 0;
  const int grid = a.total_items < sm_count ? a.total_items : sm_count;
  roi_align3d_plan_kernel<<<ceil_div(p.K, 8), 256, sort ? p.K * sizeof(float) : 0, st>>>(p, plans, counter, NC && sort ? 2 : sort, SLOT, NC ? 2 * grid : 3 * grid, NC ? 1 : 0);
  ROI3D_LAUNCH_CHECK();
  a.plans = plans, a.counter = counter;
  static PerDeviceSmemOptIn opt_in;   // (one per instantiation = per kernel)
  if (opt_in.need(L::LAUNCH)) {
    ROI3D_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L::LAUNCH));
    opt_in.mark(L::LAUNCH);
  }
  if (g_timing_ev[0] != nullptr) ROI3D_CUDA(cudaEventRecord(g_timing_ev[0], st));   // (measurement hook, see roi3d_set_kernel_timing_events)
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid), cfg.blockDim = dim3((NC ? SN_WARPS : ST_WARPS) * 32), cfg.dynamicSmemBytes = L::LAUNCH, cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    ROI3D_CUDA(cudaLaunchKernelEx(&cfg, kernel, a));
  }
  ROI3D_LAUNCH_CHECK();
  if (g_timing_ev[1] != nullptr) ROI3D_CUDA(cudaEventRecord(g_timing_ev[1], st));
  if (pooled) ROI3D_CUDA(cudaFreeAsync(ws, st));
  return ROI3D_OK;
}

}  // namespace

// Measurement hook: when set, launch_fwd_stream records these events right before and right after the launch of the
// streamed forward kernel, so that a benchmark can time the dominant kernel by itself (without the plan kernel).
thread_local cudaEvent_t g_timing_ev[2] = {nullptr, nullptr};

int launch_fwd_stream(RoiParams &p, cudaStream_t st) {
  int sm_count = 0;
  {
    const int rc = current_sm_count(&sm_count);
    if (rc) return rc;
  }
  StreamArgs a;
  a.p = p;
  for (int l = 0; l < ST_MAX_LEVELS; ++l) a.maps[l] = nullptr;
  a.total_items = p.K * (p.C / ST_CH);
  a.pdhw = p.PD * 49;
  if (p.layout == ROI3D_NCDHW) {   // cp.async producers, no tensor maps
    return launch_cfg<3, SN_SLOT, true>(p, a, st, sm_count);
  }
  for (int l = 0; l < p.num_levels; ++l) {
    const int rc = level_maps(p.lv[l], p.B, p.C, &a.maps[l]);
    if (rc) return rc;
  }
  // ring geometry (measured on C2, whole call): 3 x 42 KB 154 us, 4 x 32 KB 156 us, 4 x 30 KB 160 us, 5 x 24 KB 166 us,
  // 4 x 20 KB 185 us, 8 x 15 KB 215 us -- per-tile hand-offs cost more than a shallower ring
  return launch_cfg<3, 43008>(p, a, st, sm_count);
}

bool bwd_stream_ok(const RoiParams &p) {
  if (p.PW != 7 || p.PH != 7 || p.PD < 1 || p.PD > 7) return false;
  if (p.C % ST_CH != 0 || p.num_levels > ST_MAX_LEVELS || p.bug_compat) return false;
  if ((long long)p.K * (p.C / ST_CH) >= 2147483647LL) return false;
  for (int l = 0; l < p.num_levels; ++l)
    if ((reinterpret_cast<uintptr_t>(p.lv[l].grad) & 7) != 0) return false;
  return (reinterpret_cast<uintptr_t>(p.grad_out) & 3) == 0;
}

int launch_bwd_stream(RoiParams &p, cudaStream_t st) {
  int sm_count = 0;
  {
    const int rc = current_sm_count(&sm_count);
    if (rc) return rc;
  }
  StreamArgs a;
  a.p = p;
  for (int l = 0; l < ST_MAX_LEVELS; ++l) a.maps[l] = nullptr;
  a.total_items = p.K * (p.C / ST_CH);
  a.pdhw = p.PD * 49;
  const size_t plan_bytes = (size_t)p.K * sizeof(StreamPlan);
  unsigned char *ws = nullptr;
  bool pooled = false;
  int rc = acquire_plan_ws(plan_bytes + 16, st, &ws, &pooled);
  if (rc) return rc;
  StreamPlan *plans = reinterpret_cast<StreamPlan *>(ws);
  int *counter = reinterpret_cast<int *>(ws + plan_bytes);
  const int sort = p.K <= ST_SORT_MAX ? 1 : 0;
  const int grid = a.total_items < sm_count ? a.total_items : sm_count;
  RoiParams pp = p;
  pp.lvls_out = nullptr;   // (the forward reports the levels)
  roi_align3d_plan_kernel<<<ceil_div(p.K, 8), 256, sort ? p.K * sizeof(float) : 0, st>>>(pp, plans, counter, sort, 43008, 0, 0);
  ROI3D_LAUNCH_CHECK();
  a.plans = plans, a.counter = counter;
  static PerDeviceSmemOptIn opt_in;
  if (opt_in.need(SB_TOTAL)) {
    ROI3D_CUDA(cudaFuncSetAttribute(roi_align3d_bwd_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SB_TOTAL));
    opt_in.mark(SB_TOTAL);
  }
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid), cfg.blockDim = dim3(ST_WARPS * 32), cfg.dynamicSmemBytes = SB_TOTAL, cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    ROI3D_CUDA(cudaLaunchKernelEx(&cfg, roi_align3d_bwd_stream_kernel, a));
  }
  ROI3D_LAUNCH_CHECK();
  if (pooled) ROI3D_CUDA(cudaFreeAsync(ws, st));
  return ROI3D_OK;
}

}  // namespace roi3d

// RPN proposal path pieces for B200 (sm_100a): segmented radix-select top-k and the fused
// anchor-generation + delta2bbox3D decode.
//
// Replaces (reference, /root/reference):
//   scores.topk(nms_pre) / scores.topk(max_num)      mmdet/models/anchor_heads/rpn_head_3d.py:108-112, :147
//   sigmoid over every anchor                         rpn_head_3d.py:87-90
//   AnchorGenerator3D.grid_anchors (numpy + H2D)      mmdet/core/anchor/anchor_generator_3d.py:56-71
//   delta2bbox3D (~25 elementwise launches)           mmdet/core/bbox/transforms.py:105-160
//
// Top-k.  Keys are 64-bit: (order-preserving score bits) << 32 | ~logical_index, so keys are unique and
// "descending key" is exactly "descending score, ties -> lower index" (the build's tie rule; torch's own
// tie order is unspecified).  The logical index of an RPN score is its position after
// permute(2,3,1,0).reshape(-1) of the [A,D,H,W] map -- the order the reference's anchors are generated
// in -- while memory is read in its native, coalesced order.  Six MSB-first histogram passes
// (11/11/10 bits over the score word, 11/11/10 over the index word) find the k-th largest key exactly;
// one collect pass appends the k keys >= it; a rank-by-counting pass sorts them.  Every (volume, level)
// segment shares each launch; nothing syncs the host.
#include <cooperative_groups.h>

#include "common.cuh"

namespace roi3d {
namespace cg = cooperative_groups;

constexpr int kMaxSeg = 64;
constexpr int kBins = 2048;
constexpr int kItemsPerThread = 16;
constexpr int kTopkThreads = 256;
constexpr int kItemsPerCta = kItemsPerThread * kTopkThreads;

struct SegDesc {
  long long off;
  unsigned len;
  int A, D, H, W;  // A == 0: logical index == memory index
  const unsigned char *mask;  // optional, indexed by LOGICAL index: 0 = the element does not take part (rpn_head_3d.py:97-106)
  long long koff;             // this segment's first entry in the key buffer (see topk_hist_kernel)
};

struct SegTable {
  SegDesc s[kMaxSeg];
  // flat grids of the full passes over long segments: segment i owns CTAs [cta0[i], cta0[i + 1]) of kFirstItemsPerCta
  // elements each (none for a segment that the tail kernel finishes alone)
  unsigned cta0[kMaxSeg + 1];
};

// CTA index of a flat grid -> its segment (binary search over the <= 64 prefix sums in the kernel parameters)
__device__ __forceinline__ int flat_segment(const SegTable &tab, unsigned cta) {
  int lo = 0, hi = kMaxSeg;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (tab.cta0[mid] <= cta) lo = mid; else hi = mid;
  }
  return lo;
}

struct SegState {           // device, per segment
  unsigned long long prefix;  // key bits decided so far (left-aligned value of the decided digits)
  int k_rem;                // how many keys still to take inside the current prefix
  int k_take;               // min(k, len)
  int cand_count;
  int bnd_count;            // keys inside the boundary bin after the second digit pass (topk_split_kernel); read as
                            // unsigned: a segment of more than 2^31 elements can put more than INT_MAX keys there
  unsigned eff_len;         // elements taking part: len, or the number of set mask bytes (known after digit pass 0)
  float sieve_t;            // sieve path: raw-score threshold picked from a sample of the segment (topk_sample_kernel)
  int sieve_count;          // sieve path: elements with a raw score >= sieve_t (may exceed the list's capacity; unsigned
                            // like bnd_count)
  int need_slow;            // 1: the digit passes run for this segment (sieve off, or its result could not be proven exact)
};

__device__ __forceinline__ unsigned okey(float s) {
  if (s != s) return 0xFFFFFFFFu;   // NaN of either sign ranks above everything, as torch.topk has it
  s = s + 0.0f;
  unsigned u = __float_as_uint(s);
  const unsigned k = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return k != 0u ? k : 1u;  // 0 is reserved for "masked out" in the key buffer (only -NaN with a full payload maps there)
}

__device__ __forceinline__ float okey_inv(unsigned k) {
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}

// torch's fp32 sigmoid: 1 / (1 + exp(-x))   (rpn_head_3d.py:90)
__device__ __forceinline__ float sigmoid_ref(float x) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))); }

__device__ __forceinline__ unsigned logical_index(const SegDesc &d, unsigned m) {
  if (d.A == 0) return m;
  // memory m = ((a*D + z)*H + y)*W + x  ->  logical ((y*W + x)*D + z)*A + a
  const unsigned x = m % d.W;
  unsigned t = m / d.W;
  const unsigned y = t % d.H;
  t /= d.H;
  const unsigned z = t % d.D;
  const unsigned a = t / d.D;
  return ((y * d.W + x) * d.D + z) * d.A + a;
}

// pass p: digit position and width.  Score word: bits 63..53, 52..42, 41..32; index word: 31..21, 20..10, 9..0
__device__ __forceinline__ void pass_geometry(int pass, int &shift, int &bits) {
  const int sh[6] = {53, 42, 32, 21, 10, 0};
  const int bw[6] = {11, 11, 10, 11, 11, 10};
  shift = sh[pass], bits = bw[pass];
}

// Bin of h[0, kBins) (shared memory) where the descending cumulative count reaches `need` (1 <= need <= total): returns
// the bin, leaves what is still needed inside it in `need`, and tells whether the bin holds exactly that many.  The
// whole CTA calls it; warp 0 works: lanes sum 64 bins each (rotated, so that the 32 lanes read 32 banks), a shuffle scan
// finds the lane that crosses, the same again over that lane's 64 bins.  Three barriers (before, after, and after the
// result is read).
__device__ __forceinline__ unsigned find_bin_desc(const unsigned *h, unsigned &need, bool &exact, int tid) {
  __shared__ unsigned s_fb[3];
  static_assert(kBins == 2048, "32 lanes x 64 bins");
  __syncthreads();
  if (tid < 32) {
    const int lane = tid;
    unsigned sum = 0;
#pragma unroll 16
    for (int j = 0; j < 64; ++j) sum += h[lane * 64 + ((j + lane) & 63)];
    unsigned incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_down_sync(0xffffffffu, incl, o);
      if (lane + o < 32) incl += v;
    }
    const unsigned above = incl - sum;
    const unsigned ball = __ballot_sync(0xffffffffu, above < need && above + sum >= need);
    const int L = ball ? __ffs(ball) - 1 : 0;
    const unsigned aboveL = __shfl_sync(0xffffffffu, above, L);
    const unsigned c0 = h[L * 64 + 2 * lane], c1 = h[L * 64 + 2 * lane + 1];
    const unsigned s2 = c0 + c1;
    unsigned incl2 = s2;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_down_sync(0xffffffffu, incl2, o);
      if (lane + o < 32) incl2 += v;
    }
    const unsigned above2 = aboveL + incl2 - s2;
    if (above2 < need && above2 + s2 >= need) {
      const bool hi = above2 + c1 >= need;
      const unsigned rem = hi ? need - above2 : need - above2 - c1;
      s_fb[0] = (unsigned)(L * 64 + 2 * lane + (hi ? 1 : 0)), s_fb[1] = rem, s_fb[2] = (hi ? c1 : c0) == rem;
    }
  }
  __syncthreads();
  const unsigned bin = s_fb[0];
  need = s_fb[1];
  exact = s_fb[2] != 0u;
  __syncthreads();   // nobody is still reading the result when a caller goes on to write shared memory
  return bin;
}

// Pick the digit where the descending cumulative count crosses k_rem (256 threads; run by the LAST CTA of a
// segment's histogram pass, see topk_hist_kernel).
__device__ __forceinline__ void scan_segment(unsigned *__restrict__ hist, SegState *__restrict__ state, int seg, int pass) {
  SegState st = state[seg];
  unsigned *g = hist + (long long)seg * kBins;
  __shared__ unsigned part[256];
  __shared__ int s_digit, s_krem;
  const bool act = threadIdx.x < 256;   // CTAs larger than 256 threads: the rest only keep the barriers company
  // thread t owns bins [8t, 8t+8) ; descending order means high bins first
  unsigned loc[8], sum = 0;
  if (act) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      loc[i] = __ldcg(g + threadIdx.x * 8 + i);  // written by other CTAs' atomics: read through L2
      sum += loc[i];
      g[threadIdx.x * 8 + i] = 0;  // leave the histogram clean for the next pass
    }
    part[threadIdx.x] = sum;
  }
  __syncthreads();
  // suffix sum over threads above me (256 entries; simple serial-in-smem log scan)
  for (int o = 1; o < 256; o <<= 1) {
    unsigned v = (act && threadIdx.x + o < 256) ? part[threadIdx.x + o] : 0u;
    __syncthreads();
    if (act) part[threadIdx.x] += v;
    __syncthreads();
  }
  const unsigned above = act ? part[threadIdx.x] - sum : 0u;  // keys in bins strictly above my 8 bins
  if (pass == 0) {
    // the first histogram counts every element that takes part: a masked segment learns its effective length here
    const unsigned total = part[0];
    st.eff_len = total;
    if (total < (unsigned)st.k_take) st.k_take = (int)total, st.k_rem = (int)total;
  }
  const unsigned k = (unsigned)st.k_rem;
  if (k == 0) {  // nothing to select (all masked out)
    __syncthreads();
    if (threadIdx.x == 0) state[seg] = st;
    return;
  }
  if (act && above < k && above + sum >= k) {
    unsigned cum = above;
    for (int i = 7; i >= 0; --i) {
      if (cum + loc[i] >= k) {
        s_digit = threadIdx.x * 8 + i;
        s_krem = (int)(k - cum);
        break;
      }
      cum += loc[i];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int shift, bits;
    pass_geometry(pass, shift, bits);
    st.prefix |= (unsigned long long)(unsigned)s_digit << shift;
    st.k_rem = s_krem;
    state[seg] = st;
  }
}

constexpr int kBndCap = 4096;  // boundary keys kept per segment after two digit passes; more (mass ties) -> full passes

// bnd != nullptr (passes 2..5): if the segment's boundary bin fitted kBndCap keys, the pass runs over those keys only
// instead of re-reading and re-scoring the whole segment.
// keys (optional u32 buffer, one entry per score): digit pass 0 stores every element's order-preserving key there (0 =
// the element does not take part: masked out), so that the sigmoid, the mask lookup and the HBM read happen ONCE; the
// later full passes (digit pass 1, the split, and the rare overflow passes) read the keys back from L2.
// Digit pass 0 of a full segment runs in topk_first_kernel (lane-private counters); this kernel takes the later passes.
template <bool SIGMOID>
__global__ void __launch_bounds__(kTopkThreads) topk_hist_kernel(const float *__restrict__ scores, const SegTable tab,
                                                                 const SegState *__restrict__ state, int pass,
                                                                 unsigned *__restrict__ hist /*[nseg][kBins]*/,
                                                                 const unsigned long long *__restrict__ bnd,
                                                                 int *__restrict__ tickets, unsigned *__restrict__ keys,
                                                                 unsigned small_max) {
  const int seg = blockIdx.y;
  const SegDesc d = tab.s[seg];
  if (d.len <= small_max) return;   // (0 when the tail kernel is not in use: k > kBitonicMax)
  const SegState st = state[seg];
  const bool use_b = bnd != nullptr && (unsigned)st.bnd_count <= (unsigned)kBndCap;
  const long long len = use_b ? (long long)st.bnd_count : (long long)d.len;
  if ((long long)blockIdx.x * kItemsPerCta >= len) return;
  if (st.k_take <= 0) return;
  __shared__ unsigned h[kBins];
  for (int i = threadIdx.x; i < kBins; i += kTopkThreads) h[i] = 0;
  __syncthreads();
  int shift, bits;
  pass_geometry(pass, shift, bits);
  const unsigned dmask = (1u << bits) - 1u;
  const bool low_word = pass >= 3;
  const unsigned pre_hi = (unsigned)(st.prefix >> 32);
  const float *src = scores + d.off;
  const unsigned long long *bsrc = bnd + (long long)seg * kBndCap;
  unsigned *kbuf = keys != nullptr ? keys + d.koff : nullptr;
  // grid-stride over the segment: the boundary passes are launched with a few CTAs per segment (the usual case
  // needs one); a segment that overflowed the boundary buffer is then walked by those few CTAs
  const bool from_keys = !use_b && kbuf != nullptr && pass > 0;
  for (long long base = (long long)blockIdx.x * kItemsPerCta; base < len; base += (long long)gridDim.x * kItemsPerCta) {
  unsigned kpre[kItemsPerThread];   // key-buffer passes: all of a thread's loads are issued before the first atomic
  if (from_keys) {
#pragma unroll
    for (int it = 0; it < kItemsPerThread; ++it) {
      const long long m = base + (long long)it * kTopkThreads + threadIdx.x;
      kpre[it] = m < len ? __ldg(kbuf + m) : 0u;
    }
  }
#pragma unroll
  for (int it = 0; it < kItemsPerThread; ++it) {
    const long long m = base + (long long)it * kTopkThreads + threadIdx.x;
    unsigned bin = 0xFFFFFFFFu;  // no contribution
    if (m < len) {
      unsigned kh, kl_b = 0;
      bool take = true;
      if (use_b) {
        const unsigned long long key = bsrc[m];
        kh = (unsigned)(key >> 32), kl_b = (unsigned)key;
      } else if (from_keys) {
        kh = kpre[it];
        take = kh != 0u;
      } else {
        take = d.mask == nullptr || __ldg(d.mask + logical_index(d, (unsigned)m)) != 0;
        float v = __ldg(src + m);
        if (SIGMOID) v = sigmoid_ref(v);
        kh = take ? okey(v) : 0u;
        if (kbuf != nullptr) kbuf[m] = kh;
      }
      if (take) {
        if (!low_word) {
          // participates iff the already-decided high digits match
          const int decided = 32 - (shift - 32) - bits;  // number of decided bits of the score word
          const bool match = decided == 0 || (kh >> (32 - decided)) == (pre_hi >> (32 - decided));
          if (match) bin = (kh >> (shift - 32)) & dmask;
        } else if (kh == pre_hi) {
          const unsigned kl = use_b ? kl_b : ~logical_index(d, (unsigned)m);
          const unsigned pre_lo = (unsigned)st.prefix;
          const int decided = 32 - shift - bits;
          const bool match = decided == 0 || (kl >> (32 - decided)) == (pre_lo >> (32 - decided));
          if (match) bin = (kl >> shift) & dmask;
        }
      }
    }
    if (bin != 0xFFFFFFFFu) atomicAdd(&h[bin], 1u);
  }
  }
  __syncthreads();
  unsigned *g = hist + (long long)seg * kBins;
  for (int i = threadIdx.x; i < kBins; i += kTopkThreads) {
    const unsigned c = h[i];
    if (c) atomicAdd(&g[i], c);
  }
  // the last CTA of this segment to get here scans the finished histogram (no separate scan launch)
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const long long want = (len + kItemsPerCta - 1) / kItemsPerCta;
    const int nct = (int)(want < (long long)gridDim.x ? want : (long long)gridDim.x);
    s_last = atomicAdd(&tickets[seg], 1) == nct - 1;
    if (s_last) tickets[seg] = 0;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    scan_segment(hist, const_cast<SegState *>(state), seg, pass);
  }
}

// Digit pass 0 over whole segments.  Sigmoid scores crowd into a handful of exponent bins (half of them share ONE
// 11-bit prefix), which serialises shared-memory atomics on a common histogram up to 32-fold.  Here every lane counts
// in its own 16-bit counter: table [bin][16 words], lanes 2j / 2j+1 share word j (low / high half), so an atomic
// instruction never meets more than a two-way conflict, whatever the distribution.  A (bin, lane) counter sees at
// most kFirstItemsPerThread * 16 warps = 1024 increments.  The pass also stores every element's order-preserving key
// (0 = masked out) when a key buffer is given, 16 bytes per thread and load.
constexpr int kFirstThreads = 1024;
constexpr int kFirstItemsPerThread = 32;
constexpr int kFirstItemsPerCta = kFirstThreads * kFirstItemsPerThread;
constexpr int kFirstSmemBytes = kBins * 16 * 4;

template <bool SIGMOID>
__device__ __forceinline__ unsigned first_key(const SegDesc &d, unsigned m, float v) {
  const bool take = d.mask == nullptr || __ldg(d.mask + logical_index(d, m)) != 0;
  if (SIGMOID) v = sigmoid_ref(v);
  return take ? okey(v) : 0u;
}

// last CTA of a segment's flat range runs the scan (no separate launch)
__device__ __forceinline__ void flat_finish(const SegTable &tab, int seg, unsigned *hist, SegState *state, int *tickets, int pass,
                                            int ctas_per_chunk = 1) {
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const int nct = (int)(tab.cta0[seg + 1] - tab.cta0[seg]) * ctas_per_chunk;
    s_last = atomicAdd(&tickets[seg], 1) == nct - 1;
    if (s_last) tickets[seg] = 0;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    scan_segment(hist, state, seg, pass);
  }
}

template <bool SIGMOID>
__global__ void __launch_bounds__(kFirstThreads, 1) topk_first_kernel(const float *__restrict__ scores, const SegTable tab,
                                                                      SegState *__restrict__ state, unsigned *__restrict__ hist,
                                                                      int *__restrict__ tickets, unsigned *__restrict__ keys) {
  extern __shared__ __align__(16) unsigned ftab[];   // [kBins][16]
  const int seg = flat_segment(tab, blockIdx.x);
  const SegDesc d = tab.s[seg];
  if (!state[seg].need_slow) return;   // the sieve path already finished this segment
  const unsigned len = d.len;
  const unsigned base = (blockIdx.x - tab.cta0[seg]) * (unsigned)kFirstItemsPerCta;
  for (int i = threadIdx.x; i < kBins * 4; i += kFirstThreads) reinterpret_cast<uint4 *>(ftab)[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  const float *src = scores + d.off;
  unsigned *kbuf = keys != nullptr ? keys + d.koff : nullptr;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned inc = (lane & 1u) ? 0x10000u : 1u;
  unsigned *col = ftab + (lane >> 1);
  const bool vec = (reinterpret_cast<uintptr_t>(src) & 15) == 0;   // (the key buffer's segments are 16-byte aligned)
  if (vec) {
    constexpr int NB = 4;   // 16-byte loads in flight per thread: issued together, then scored
#pragma unroll 1
    for (int it0 = 0; it0 < kFirstItemsPerThread / 4; it0 += NB) {
      float4 v[NB];
#pragma unroll
      for (int u = 0; u < NB; ++u) {
        const unsigned m = base + ((unsigned)(it0 + u) * kFirstThreads + threadIdx.x) * 4u;
        v[u] = m + 4u <= len ? __ldcs(reinterpret_cast<const float4 *>(src + m)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < NB; ++u) {
        const unsigned m = base + ((unsigned)(it0 + u) * kFirstThreads + threadIdx.x) * 4u;
        if (m + 4u <= len) {
          uint4 kk;
          kk.x = first_key<SIGMOID>(d, m, v[u].x), kk.y = first_key<SIGMOID>(d, m + 1, v[u].y);
          kk.z = first_key<SIGMOID>(d, m + 2, v[u].z), kk.w = first_key<SIGMOID>(d, m + 3, v[u].w);
          if (kbuf != nullptr) *reinterpret_cast<uint4 *>(kbuf + m) = kk;
          if (kk.x) atomicAdd(col + (kk.x >> 21) * 16, inc);
          if (kk.y) atomicAdd(col + (kk.y >> 21) * 16, inc);
          if (kk.z) atomicAdd(col + (kk.z >> 21) * 16, inc);
          if (kk.w) atomicAdd(col + (kk.w >> 21) * 16, inc);
        } else {
          for (unsigned mm = m; mm < len; ++mm) {
            const unsigned kh = first_key<SIGMOID>(d, mm, __ldg(src + mm));
            if (kbuf != nullptr) kbuf[mm] = kh;
            if (kh) atomicAdd(col + (kh >> 21) * 16, inc);
          }
        }
      }
    }
  } else {
#pragma unroll 4
    for (int it = 0; it < kFirstItemsPerThread; ++it) {
      const unsigned m = base + (unsigned)it * kFirstThreads + threadIdx.x;
      if (m < len) {
        const unsigned kh = first_key<SIGMOID>(d, m, __ldg(src + m));
        if (kbuf != nullptr) kbuf[m] = kh;
        if (kh) atomicAdd(col + (kh >> 21) * 16, inc);
      }
    }
  }
  __syncthreads();
  unsigned *g = hist + (long long)seg * kBins;
  for (int b = threadIdx.x; b < kBins; b += kFirstThreads) {
    const uint4 *row = reinterpret_cast<const uint4 *>(ftab + b * 16);
    unsigned c = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 w = row[q];
      c += (w.x & 0xFFFFu) + (w.x >> 16) + (w.y & 0xFFFFu) + (w.y >> 16) + (w.z & 0xFFFFu) + (w.z >> 16) + (w.w & 0xFFFFu) +
           (w.w >> 16);
    }
    if (c) atomicAdd(&g[b], c);
  }
  flat_finish(tab, seg, hist, state, tickets, 0);
}

// Digit pass 1 and the split pass in their key-buffer form: one u32 load per element, flat grid, every load of a batch
// issued before the first atomic.  (The generic kernels above remain for callers without a key buffer and k > kBitonicMax.)
constexpr int kKeyThreads = 256;
constexpr int kKeyBatch = 16;
constexpr int kKeySub = 4;   // CTAs per chunk of kFirstItemsPerCta keys: short CTAs, ten per SM, hide the load latency
constexpr int kKeyItemsPerCta = kFirstItemsPerCta / kKeySub;

// a thread's batch of kKeyBatch keys, kKeyThreads apart: whole batches are loaded from one pointer with immediate offsets
__device__ __forceinline__ void load_key_batch(const unsigned *__restrict__ p, unsigned m0, unsigned end, unsigned (&kk)[kKeyBatch]) {
  if (m0 + (kKeyBatch - 1) * kKeyThreads < end) {
#pragma unroll
    for (int u = 0; u < kKeyBatch; ++u) kk[u] = __ldg(p + u * kKeyThreads);
  } else {
#pragma unroll
    for (int u = 0; u < kKeyBatch; ++u) kk[u] = m0 + u * kKeyThreads < end ? __ldg(p + u * kKeyThreads) : 0u;
  }
}

__global__ void __launch_bounds__(kKeyThreads) topk_second_kernel(const SegTable tab, SegState *__restrict__ state,
                                                                  unsigned *__restrict__ hist, int *__restrict__ tickets,
                                                                  const unsigned *__restrict__ keys) {
  __shared__ unsigned h[kBins];
  const unsigned chunk = blockIdx.x / kKeySub, sub = blockIdx.x - chunk * kKeySub;
  const int seg = flat_segment(tab, chunk);
  const SegDesc d = tab.s[seg];
  if (!state[seg].need_slow) return;
  const unsigned top11 = (unsigned)(state[seg].prefix >> 53);
  const bool live = state[seg].k_take > 0;
  for (int i = threadIdx.x; i < kBins; i += kKeyThreads) h[i] = 0;
  __syncthreads();
  const unsigned *kb = keys + d.koff;
  const unsigned base = (chunk - tab.cta0[seg]) * (unsigned)kFirstItemsPerCta + sub * (unsigned)kKeyItemsPerCta;
  const unsigned end = min(d.len, base + (unsigned)kKeyItemsPerCta);
  if (live) {
    for (unsigned m0 = base + threadIdx.x; m0 < end; m0 += kKeyThreads * kKeyBatch) {
      unsigned kk[kKeyBatch];
      load_key_batch(kb + m0, m0, end, kk);
#pragma unroll
      for (int u = 0; u < kKeyBatch; ++u)
        if (kk[u] != 0u && (kk[u] >> 21) == top11) atomicAdd(&h[(kk[u] >> 10) & 0x7FFu], 1u);
    }
  }
  __syncthreads();
  unsigned *g = hist + (long long)seg * kBins;
  for (int i = threadIdx.x; i < kBins; i += kKeyThreads) {
    const unsigned c = h[i];
    if (c) atomicAdd(&g[i], c);
  }
  flat_finish(tab, seg, hist, state, tickets, 1, kKeySub);
}

constexpr int kSplitStage = 1024;   // selected keys a CTA stages before it reserves their slots with one atomic per list
__global__ void __launch_bounds__(kKeyThreads) topk_split_keys_kernel(const SegTable tab, SegState *__restrict__ state, int k,
                                                                      unsigned long long *__restrict__ cand,
                                                                      unsigned long long *__restrict__ bnd,
                                                                      const unsigned *__restrict__ keys) {
  __shared__ unsigned long long stage[2][kSplitStage];   // [0]: above the boundary bin, [1]: inside it
  __shared__ int s_n[2], s_base[2];
  const unsigned chunk = blockIdx.x / kKeySub, sub = blockIdx.x - chunk * kKeySub;
  const int seg = flat_segment(tab, chunk);
  const SegDesc d = tab.s[seg];
  if (state[seg].k_take <= 0 || !state[seg].need_slow) return;
  const unsigned p22 = (unsigned)(state[seg].prefix >> 42);  // the 22 decided bits
  const unsigned *kb = keys + d.koff;
  const unsigned base = (chunk - tab.cta0[seg]) * (unsigned)kFirstItemsPerCta + sub * (unsigned)kKeyItemsPerCta;
  const unsigned end = min(d.len, base + (unsigned)kKeyItemsPerCta);
  if (threadIdx.x < 2) s_n[threadIdx.x] = 0;
  __syncthreads();
  for (unsigned m0 = base + threadIdx.x; m0 < end; m0 += kKeyThreads * kKeyBatch) {
    unsigned kk[kKeyBatch];
    load_key_batch(kb + m0, m0, end, kk);
#pragma unroll
    for (int u = 0; u < kKeyBatch; ++u) {
      const unsigned h22 = kk[u] >> 10;
      if (kk[u] != 0u && h22 >= p22) {
        const unsigned li = logical_index(d, m0 + u * kKeyThreads);
        const unsigned long long key = ((unsigned long long)kk[u] << 32) | (unsigned)~li;
        const int which = h22 > p22 ? 0 : 1;
        const int pos = atomicAdd(&s_n[which], 1);
        if (pos < kSplitStage) {
          stage[which][pos] = key;
        } else if (which == 0) {   // staging full (a CTA rarely holds this many): straight to the lists
          const int gp = atomicAdd(&state[seg].cand_count, 1);
          if (gp < k) cand[(long long)seg * k + gp] = key;
        } else {
          const int gp = atomicAdd(&state[seg].bnd_count, 1);
          if ((unsigned)gp < (unsigned)kBndCap) bnd[(long long)seg * kBndCap + gp] = key;
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    const int n = min(s_n[threadIdx.x], kSplitStage);
    s_base[threadIdx.x] = n > 0 ? atomicAdd(threadIdx.x == 0 ? &state[seg].cand_count : &state[seg].bnd_count, n) : 0;
  }
  __syncthreads();
  for (int which = 0; which < 2; ++which) {
    const int n = min(s_n[which], kSplitStage), gb = s_base[which];
    const int cap = which == 0 ? k : kBndCap;
    unsigned long long *dst = which == 0 ? cand + (long long)seg * k : bnd + (long long)seg * kBndCap;
    for (int i = threadIdx.x; i < n; i += kKeyThreads) {
      const unsigned at = (unsigned)gb + (unsigned)i;
      if (at < (unsigned)cap) dst[at] = stage[which][i];
    }
  }
}

template <bool SIGMOID>
__global__ void __launch_bounds__(kTopkThreads) topk_collect_kernel(const float *__restrict__ scores,
                                                                    const SegTable tab, SegState *__restrict__ state,
                                                                    int k, unsigned long long *__restrict__ cand,
                                                                    const unsigned long long *__restrict__ bnd,
                                                                    const unsigned *__restrict__ keys) {
  const int seg = blockIdx.y;
  const SegDesc d = tab.s[seg];
  const long long base = (long long)blockIdx.x * kItemsPerCta;
  const SegState st = state[seg];
  const bool use_b = bnd != nullptr && (unsigned)st.bnd_count <= (unsigned)kBndCap;  // keys above the boundary bin are in cand already
  const long long len = use_b ? (long long)st.bnd_count : (long long)d.len;
  if (base >= len) return;
  if (st.k_take <= 0) return;
  const unsigned thr_hi = (unsigned)(st.prefix >> 32);
  const float *src = scores + d.off;
  const unsigned long long *bsrc = bnd + (long long)seg * kBndCap;
  for (long long base2 = base; base2 < len; base2 += (long long)gridDim.x * kItemsPerCta)
#pragma unroll 4
  for (int it = 0; it < kItemsPerThread; ++it) {
    const long long m = base2 + (long long)it * kTopkThreads + threadIdx.x;
    if (m < len) {
      unsigned long long key;
      if (use_b) {
        key = bsrc[m];
      } else if (keys != nullptr) {
        const unsigned kh = __ldg(keys + d.koff + m);   // 0 (masked out) is below every threshold that selects anything
        if (kh == 0u || kh < thr_hi) continue;
        key = ((unsigned long long)kh << 32) | (unsigned)~logical_index(d, (unsigned)m);
      } else {
        float v = __ldg(src + m);
        if (SIGMOID) v = sigmoid_ref(v);
        const unsigned kh = okey(v);
        if (kh < thr_hi) continue;
        const unsigned li = logical_index(d, (unsigned)m);
        if (d.mask != nullptr && !__ldg(d.mask + li)) continue;
        key = ((unsigned long long)kh << 32) | (unsigned)~li;
      }
      if (key >= st.prefix) {
        const int pos = atomicAdd(&state[seg].cand_count, 1);
        if (pos < k) cand[(long long)seg * k + pos] = key;
      }
    }
  }
}

// After the first two digit passes (22 bits of the score word decided): one pass over the whole segment that
// (a) appends every key ABOVE the boundary bin to the result candidates -- they are certainly selected -- and
// (b) copies the keys INSIDE the boundary bin to a small buffer, on which the remaining four digit passes and the
// final collect run.  Five of the seven full passes over the scores disappear.
template <bool SIGMOID>
__global__ void __launch_bounds__(kTopkThreads) topk_split_kernel(const float *__restrict__ scores, const SegTable tab,
                                                                  SegState *__restrict__ state, int k,
                                                                  unsigned long long *__restrict__ cand,
                                                                  unsigned long long *__restrict__ bnd,
                                                                  const unsigned *__restrict__ keys, unsigned small_max) {
  const int seg = blockIdx.y;
  const SegDesc d = tab.s[seg];
  const long long base = (long long)blockIdx.x * kItemsPerCta;
  if (base >= (long long)d.len || d.len <= small_max) return;
  const SegState st = state[seg];
  if (st.k_take <= 0) return;
  const unsigned p22 = (unsigned)(st.prefix >> 42);  // the 22 decided bits
  const float *src = scores + d.off;
  unsigned kpre[kItemsPerThread];   // key-buffer form: all loads first
  if (keys != nullptr) {
#pragma unroll
    for (int it = 0; it < kItemsPerThread; ++it) {
      const long long m = base + (long long)it * kTopkThreads + threadIdx.x;
      kpre[it] = m < (long long)d.len ? __ldg(keys + d.koff + m) : 0u;
    }
  }
#pragma unroll
  for (int it = 0; it < kItemsPerThread; ++it) {
    const long long m = base + (long long)it * kTopkThreads + threadIdx.x;
    if (m < (long long)d.len) {
      unsigned kh;
      if (keys != nullptr) {
        kh = kpre[it];
        if (kh == 0u) continue;
      } else {
        float v = __ldg(src + m);
        if (SIGMOID) v = sigmoid_ref(v);
        kh = okey(v);
      }
      const unsigned h22 = kh >> 10;
      if (h22 >= p22) {
        const unsigned li = logical_index(d, (unsigned)m);
        if (keys == nullptr && d.mask != nullptr && !__ldg(d.mask + li)) continue;
        const unsigned long long key = ((unsigned long long)kh << 32) | (unsigned)~li;
        if (h22 > p22) {
          const int pos = atomicAdd(&state[seg].cand_count, 1);
          if (pos < k) cand[(long long)seg * k + pos] = key;
        } else {
          const int pos = atomicAdd(&state[seg].bnd_count, 1);
          if ((unsigned)pos < (unsigned)kBndCap) bnd[(long long)seg * kBndCap + pos] = key;
        }
      }
    }
  }
}

// Boundary bin larger than the buffer (mass ties): forget the split, the full-data passes and collect take over.
__global__ void topk_after_split_kernel(SegState *state, int nseg) {
  const int s = threadIdx.x;
  if (s < nseg && (unsigned)state[s].bnd_count > (unsigned)kBndCap) state[s].cand_count = 0;
}

// rank-by-counting sort of the (unique) candidate keys, descending.  grid (ceil(k/256), nseg).
// by_index (a segment no longer than k, when the caller asks for it): the whole segment is selected and is returned
// in ascending logical index instead -- the reference only sorts a level that has more than nms_pre anchors
// (rpn_head_3d.py:96,108-112).  The low key word is ~index, so "descending low word" is ascending index.
__global__ void __launch_bounds__(256) topk_sort_kernel(const unsigned long long *__restrict__ cand,
                                                        const SegState *__restrict__ state, const SegTable tab,
                                                        int small_by_index, int k, int64_t *__restrict__ out_idx,
                                                        float *__restrict__ out_val) {
  const int seg = blockIdx.y;
  const int n = state[seg].k_take;
  const bool by_index = small_by_index && state[seg].eff_len <= (unsigned)k;
  if ((int)(blockIdx.x * 256) >= n) return;
  const unsigned long long *c = cand + (long long)seg * k;
  const int i = blockIdx.x * 256 + threadIdx.x;
  const unsigned long long ki = i < n ? c[i] : 0ULL;
  __shared__ unsigned long long keys[256];
  int rank = 0;
  for (int j0 = 0; j0 < n; j0 += 256) {
    __syncthreads();
    keys[threadIdx.x] = (j0 + threadIdx.x) < n ? c[j0 + threadIdx.x] : 0ULL;
    __syncthreads();
    const int lim = min(256, n - j0);
    if (i < n) {
#pragma unroll 8
      for (int t = 0; t < lim; ++t) rank += by_index ? ((unsigned)keys[t] > (unsigned)ki) : (keys[t] > ki);
    }
  }
  if (i < n) {
    out_idx[(long long)seg * k + rank] = (int64_t)(unsigned)~(unsigned)ki;
    out_val[(long long)seg * k + rank] = okey_inv((unsigned)(ki >> 32));
  }
}

// k up to kBitonicMax: the tail kernel (below) finishes every segment in one launch; above it the rank-by-counting sort.
// ------------------------------------------------------------------------------------------------
// Sieve path (k <= kBitonicMax, no masks): ONE pass over the scores at memory speed instead of three digit passes.
//   * topk_sample_kernel (one cluster of CTAs per long segment; also initialises the segment states) reads a jittered sample of at
//     most kSieveSample RAW scores and picks the threshold T whose rank in the sample predicts k + kBndCap / 2
//     elements >= T in the whole segment (capacity of the list: k + kBndCap, the slow path's two lists end to end);
//   * topk_sieve_kernel streams the segment once: `x < T` drops an element without scoring it (no expf, no division
//     for 99.7 % of the anchors); the others are scored exactly and appended as 64-bit keys;
//   * the tail kernel sorts the list and PROVES the result: the list must hold at least k keys without overflowing, and
//     the k-th score must exceed sigmoid(T) by more than the rounding slack of the fp32 sigmoid (every dropped element
//     has x < T, hence a score below that bound) -- for raw scores: the k-th key >= key(T).  A segment that fails the
//     proof (mass ties, saturated scores, an unlucky sample) goes through the digit passes, which are launched behind
//     the tail and return at once for every segment that passed.
// The result is the same bit for bit: same keys, same order.
// ------------------------------------------------------------------------------------------------
constexpr int kSieveSample = 32768;
constexpr int kSieveCluster = 8;      // CTAs per segment in the sampling kernel
constexpr int kSieveThreads = 512;    // 8 sample keys per thread, kept in registers

__device__ __forceinline__ unsigned sieve_hash(unsigned i) {
  i ^= i >> 16, i *= 0x7feb352du, i ^= i >> 15, i *= 0x846ca68bu, i ^= i >> 16;
  return i;
}

__global__ void __cluster_dims__(kSieveCluster, 1, 1) __launch_bounds__(kSieveThreads)
    topk_sample_kernel(const float *__restrict__ scores, const SegTable tab, SegState *__restrict__ state,
                       int *__restrict__ tickets, unsigned *__restrict__ hist, int k, unsigned small_max) {
  // One CLUSTER of kSieveCluster CTAs per segment: a single SM gathers scattered 32-byte sectors too slowly (a 32 K
  // sample is 1 MB of them).  Every CTA keeps its share of the sample keys in registers; per digit the CTAs count into
  // their own table, CTA r adds up bins [r * 256, r * 256 + 256) of all tables through distributed shared memory and
  // writes the totals into every CTA's copy, and every CTA scans its copy -- two cluster barriers per digit.
  __shared__ unsigned h[kBins], tot[kBins];
  cg::cluster_group cluster = cg::this_cluster();
  const int seg = blockIdx.x / kSieveCluster, rank = (int)cluster.block_rank(), tid = threadIdx.x;
  const SegDesc d = tab.s[seg];
  const unsigned len = d.len;
  if (tid == 0 && rank == 0) {
    tickets[seg] = 0;
    SegState st;
    st.prefix = 0ULL;
    st.k_take = (int)min((unsigned)k, len);
    st.k_rem = st.k_take;
    st.cand_count = 0, st.bnd_count = 0;
    st.eff_len = len;
    st.sieve_t = 0.0f, st.sieve_count = 0, st.need_slow = 1;
    state[seg] = st;
  }
  if (len <= small_max) return;   // the whole cluster
  // the digit passes' global histogram of this segment starts out clean (no memset node in front of the path)
  if (tid < kBins / kSieveCluster) hist[(long long)seg * kBins + rank * (kBins / kSieveCluster) + tid] = 0u;
  const float *src = scores + d.off;
  const unsigned S = min(len, (unsigned)kSieveSample), step = len / S;
  // rank of T in the sample: predicts k + kBndCap / 2 elements >= T in the segment; a segment that is sampled whole
  // needs no statistical slack, only room for the proof (the k-th score must clear sigmoid(T) by the rounding margin)
  unsigned need = S == len ? (unsigned)(k + kBndCap / 16)
                           : (unsigned)(((unsigned long long)(k + kBndCap / 2) * S + len - 1) / len);
  need = max(1u, min(need, S));
  constexpr int PER = kSieveSample / kSieveCluster / kSieveThreads;
  unsigned key[PER];
#pragma unroll
  for (int u = 0; u < PER; ++u) {
    const unsigned i = ((unsigned)u * kSieveCluster + rank) * kSieveThreads + tid;
    key[u] = 0u;
    if (i < S) key[u] = okey(__ldg(src + (size_t)i * step + (step > 1u ? sieve_hash(i) % step : 0u)));
  }
  // two 11-bit digits: T is the lower edge of the 22-bit bin that holds the sample's need-th largest key (the last ten
  // bits would move it by 2^-13 of its value -- any threshold is valid, the tail proves the result)
  unsigned prefix = 0u;
#pragma unroll
  for (int dg = 0; dg < 2; ++dg) {
    const int shift = dg == 0 ? 21 : 10;
    for (int b = tid; b < kBins; b += kSieveThreads) h[b] = 0u;
    __syncthreads();
#pragma unroll
    for (int u = 0; u < PER; ++u)
      if (key[u] && (dg == 0 || (key[u] >> 21) == prefix)) atomicAdd(&h[(key[u] >> shift) & 0x7FFu], 1u);
    cluster.sync();
    if (tid < kBins / kSieveCluster) {
      const int b = rank * (kBins / kSieveCluster) + tid;
      unsigned c = 0;
#pragma unroll
      for (int r = 0; r < kSieveCluster; ++r) c += *cluster.map_shared_rank(h + b, r);
#pragma unroll
      for (int r = 0; r < kSieveCluster; ++r) *cluster.map_shared_rank(tot + b, r) = c;
    }
    cluster.sync();
    bool exact;
    const unsigned dgt = find_bin_desc(tot, need, exact, tid);
    prefix = (prefix << 11) | dgt;
  }
  prefix <<= 10;
  if (tid == 0 && rank == 0) state[seg].sieve_t = okey_inv(prefix);
}

constexpr int kSieveStage = 2048;   // keys a CTA stages before it reserves their slots in the list with ONE global atomic
constexpr int kSieveBatch = kKeyItemsPerCta / kKeyThreads / 4;   // 16-byte loads per thread, all issued before the first compare
static_assert(kSieveBatch * 4 <= 32, "one bit per element in a thread's batch");

// ONE copy of the rare path in the kernel (inlined at each of the 32 compares the code outgrew the instruction cache:
// 'no instruction' was the top stall): a thread only notes WHICH of its elements passed and walks that bit mask
// afterwards, reading the score again (an L1 / L2 hit).
template <bool SIGMOID>
__global__ void __launch_bounds__(kKeyThreads) topk_sieve_kernel(const float *__restrict__ scores, const SegTable tab,
                                                                 SegState *__restrict__ state, int k,
                                                                 unsigned long long *__restrict__ lists) {
  __shared__ unsigned long long stage[kSieveStage];
  __shared__ int s_n, s_base;
  const unsigned chunk = blockIdx.x / kKeySub, sub = blockIdx.x - chunk * kKeySub;
  const int seg = flat_segment(tab, chunk);
  const SegDesc d = tab.s[seg];
  const int cap = k + kBndCap;
  SegState *st = state + seg;
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  const float T = st->sieve_t;
  unsigned long long *list = lists + (long long)seg * cap;
  const float *src = scores + d.off;
  const unsigned base = (chunk - tab.cta0[seg]) * (unsigned)kFirstItemsPerCta + sub * (unsigned)kKeyItemsPerCta;
  const unsigned end = min(d.len, base + (unsigned)kKeyItemsPerCta);
  const bool vec = (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  // element j of the thread's batch: vec -> base + ((j / 4) * kKeyThreads + tid) * 4 + j % 4, else base + j * kKeyThreads + tid
  unsigned mask = 0u;
  if (vec) {
    float4 v[kSieveBatch];
#pragma unroll
    for (int u = 0; u < kSieveBatch; ++u) {
      const unsigned m = base + ((unsigned)u * kKeyThreads + threadIdx.x) * 4u;
      v[u] = m + 4u <= end ? __ldcs(reinterpret_cast<const float4 *>(src + m)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < kSieveBatch; ++u) {
      const unsigned m = base + ((unsigned)u * kKeyThreads + threadIdx.x) * 4u;
      if (m + 4u <= end) {
        mask |= (v[u].x < T ? 0u : 1u) << (4 * u) | (v[u].y < T ? 0u : 2u) << (4 * u) | (v[u].z < T ? 0u : 4u) << (4 * u) |
                (v[u].w < T ? 0u : 8u) << (4 * u);
      } else if (m < end) {
        mask |= ((1u << (end - m)) - 1u) << (4 * u);   // the segment's last, partial vector: looked at one by one below
      }
    }
  } else {
#pragma unroll 4
    for (int j = 0; j < kSieveBatch * 4; ++j) {
      const unsigned m = base + (unsigned)j * kKeyThreads + threadIdx.x;
      if (m < end && !(__ldg(src + m) < T)) mask |= 1u << j;
    }
  }
  while (mask) {
    const int j = __ffs(mask) - 1;
    mask &= mask - 1u;
    const unsigned m = vec ? base + ((unsigned)(j >> 2) * kKeyThreads + threadIdx.x) * 4u + (unsigned)(j & 3)
                           : base + (unsigned)j * kKeyThreads + threadIdx.x;
    const float x = __ldg(src + m);
    if (x < T) continue;   // NaN stays in
    const unsigned kh = okey(SIGMOID ? sigmoid_ref(x) : x);
    const unsigned long long key = ((unsigned long long)kh << 32) | (unsigned)~logical_index(d, m);
    const int pos = atomicAdd(&s_n, 1);   // (same-address shared-memory atomics are cheap: aggregating them per warp was slower)
    if (pos < kSieveStage) {
      stage[pos] = key;
    } else {   // staging full (a segment of a few CTAs puts a large share of its elements on the list)
      const int gp = atomicAdd(&st->sieve_count, 1);
      if ((unsigned)gp < (unsigned)cap) list[gp] = key;
    }
  }
  __syncthreads();
  const int n = min(s_n, kSieveStage);
  if (n == 0) return;
  if (threadIdx.x == 0) s_base = atomicAdd(&st->sieve_count, n);
  __syncthreads();
  const int gb = s_base;
  for (int i = threadIdx.x; i < n; i += kKeyThreads) {
    const unsigned at = (unsigned)gb + (unsigned)i;
    if (at < (unsigned)cap) list[at] = stage[i];
  }
}

constexpr int kBitonicMax = 4096;

// ------------------------------------------------------------------------------------------------
// Tail of the selection, ONE launch, one CTA per segment (k <= kBitonicMax): what used to be four digit passes over
// the boundary buffer, the collect pass, the final sort and the report -- seven launches of ~10 us each, all of it
// latency (a few global round trips per launch), for a few dozen boundary keys.
//   * a segment of at most kSmallMax elements never enters the digit passes: the CTA scores it, sorts it in shared
//     memory and writes the result (the final `topk(max_num)` over 5 x 1000 rows per image is this case);
//   * otherwise the boundary keys the split pass put aside are sorted and the k_rem largest join the certain keys;
//   * a boundary bin that overflowed its buffer (mass ties) is resolved by this CTA alone with the remaining digit
//     passes over the whole segment -- slow, and only for degenerate inputs.
// Rows past a segment's count are filled with -1 / 0 here (no separate fills of the outputs).
// ------------------------------------------------------------------------------------------------
constexpr int kSmallMax = 8192;
constexpr int kTailThreads = 1024;
constexpr int kTailSmemBytes = kSmallMax * 8 + 4096 * 8 + kBins * 4;   // keys, selected keys (k <= kBitonicMax), histogram

template <bool SIGMOID>
__device__ __forceinline__ unsigned long long tail_key64(const SegDesc &d, const float *src, const unsigned *kbuf, unsigned m) {
  const unsigned li = logical_index(d, m);
  unsigned kh;
  if (kbuf != nullptr) {
    kh = __ldg(kbuf + m);
  } else {
    const bool take = d.mask == nullptr || __ldg(d.mask + li) != 0;
    float v = __ldg(src + m);
    if (SIGMOID) v = sigmoid_ref(v);
    kh = take ? okey(v) : 0u;
  }
  return kh != 0u ? (((unsigned long long)kh << 32) | (unsigned)~li) : 0ULL;
}

__device__ __forceinline__ int pow2_at_least(int n) {
  int p = 2;
  while (p < n) p <<= 1;
  return p;
}

// descending bitonic sort of sk[0, npow2) by the whole CTA; ends with a barrier.  A thread's PAIRS compare-exchanges of
// a stage are independent: all loads are issued before the first store (the stage is latency-bound)
template <int PAIRS>
__device__ __forceinline__ void tail_bitonic_p(unsigned long long *sk, int npow2, int tid) {
  const int half = npow2 >> 1;
  for (int size = 2; size <= npow2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      unsigned long long a[PAIRS], b[PAIRS];
      int lo[PAIRS];
#pragma unroll
      for (int u = 0; u < PAIRS; ++u) {
        const int t = tid + u * kTailThreads;
        lo[u] = 2 * t - (t & (stride - 1));
        if (PAIRS > 1 || t < half) a[u] = sk[lo[u]], b[u] = sk[lo[u] + stride];
      }
#pragma unroll
      for (int u = 0; u < PAIRS; ++u) {
        const int t = tid + u * kTailThreads;
        if (PAIRS > 1 || t < half) {
          const bool desc = (lo[u] & size) == 0;
          if (desc ? (a[u] < b[u]) : (a[u] > b[u])) sk[lo[u]] = b[u], sk[lo[u] + stride] = a[u];
        }
      }
      __syncthreads();
    }
  }
}
// npow2 <= 2 * kTailThreads: thread t keeps elements 2t and 2t + 1 in registers.  Stride 1 is a compare inside the
// thread, strides 2..32 are warp shuffles (partner lane = lane ^ stride / 2, both elements travel), only strides >= 64
// go through shared memory: 20 barriers for 2048 keys instead of 66.
__device__ __forceinline__ void tail_bitonic_regs(unsigned long long *sk, int npow2, int tid) {
  const int e0 = 2 * tid;
  const bool mine = e0 < npow2;
  unsigned long long x0 = mine ? sk[e0] : 0ULL, x1 = mine ? sk[e0 + 1] : 0ULL;
  for (int size = 2; size <= npow2; size <<= 1) {
    const bool desc = (e0 & size) == 0;
    int j = size >> 1;
    if (j >= 64) {
      if (mine) sk[e0] = x0, sk[e0 + 1] = x1;
      __syncthreads();
      for (; j >= 64; j >>= 1) {
        if (tid < (npow2 >> 1)) {
          const int lo = 2 * tid - (tid & (j - 1));
          const unsigned long long a = sk[lo], b = sk[lo + j];
          if (((lo & size) == 0) ? (a < b) : (a > b)) sk[lo] = b, sk[lo + j] = a;
        }
        __syncthreads();
      }
      if (mine) x0 = sk[e0], x1 = sk[e0 + 1];
    }
    for (; j >= 2; j >>= 1) {
      const unsigned long long y0 = __shfl_xor_sync(0xffffffffu, x0, j >> 1), y1 = __shfl_xor_sync(0xffffffffu, x1, j >> 1);
      const bool keep_max = ((tid & (j >> 1)) == 0) == desc;
      x0 = keep_max ? (x0 > y0 ? x0 : y0) : (x0 < y0 ? x0 : y0);
      x1 = keep_max ? (x1 > y1 ? x1 : y1) : (x1 < y1 ? x1 : y1);
    }
    if (desc ? (x0 < x1) : (x0 > x1)) {
      const unsigned long long t = x0;
      x0 = x1, x1 = t;
    }
  }
  if (mine) sk[e0] = x0, sk[e0 + 1] = x1;   // (reads of other threads' elements all lie behind a barrier already)
  __syncthreads();
}

// (not inlined: four call sites x three variants made the tail kernel 70 KB of mostly straight-line code)
__device__ __noinline__ void tail_bitonic(unsigned long long *sk, int npow2, int tid) {
  if (npow2 <= 2 * kTailThreads) tail_bitonic_regs(sk, npow2, tid);        // one pair per thread, in registers
  else if (npow2 == 4 * kTailThreads) tail_bitonic_p<2>(sk, npow2, tid);
  else tail_bitonic_p<4>(sk, npow2, tid);                                  // 8 * kTailThreads = kSmallMax
}

__device__ __forceinline__ unsigned long long swap_words(unsigned long long v) {
  return ((unsigned long long)(unsigned)v << 32) | (v >> 32);
}

// The need-th largest of the non-zero keys sk[0, n) (need <= their count): MSB-first 11/11/10-bit digits like the global
// passes, histogram and scan in shared memory.  Stops as soon as a digit's bin holds exactly what is still needed (the
// returned threshold then has its undecided bits clear): every key >= the result is selected, and there are `need` of them.
__device__ __noinline__ unsigned long long tail_select(const unsigned long long *sk, int n, int need, unsigned *h, int tid) {
  unsigned long long prefix = 0ULL;
  for (int pass = 0; pass < 6; ++pass) {
    int shift, bits;
    pass_geometry(pass, shift, bits);
    const int decided = 64 - shift - bits;
    for (int i = tid; i < kBins; i += kTailThreads) h[i] = 0u;
    __syncthreads();
    for (int i = tid; i < n; i += kTailThreads) {
      const unsigned long long key = sk[i];
      if (key != 0ULL && (decided == 0 || (key >> (64 - decided)) == (prefix >> (64 - decided))))
        atomicAdd(&h[(unsigned)(key >> shift) & ((1u << bits) - 1u)], 1u);
    }
    unsigned nd = (unsigned)need;
    bool done;
    const unsigned digit = find_bin_desc(h, nd, done, tid);   // (its first barrier closes the counting above)
    prefix |= (unsigned long long)digit << shift;
    need = (int)nd;
    if (done) break;
  }
  return prefix;
}

template <bool SIGMOID>
__global__ void __launch_bounds__(kTailThreads) topk_tail_kernel(const float *__restrict__ scores, const SegTable tab,
                                                                 SegState *__restrict__ state, unsigned *__restrict__ hist,
                                                                 int k, const unsigned long long *__restrict__ cand,
                                                                 const unsigned long long *__restrict__ bnd,
                                                                 const unsigned *__restrict__ keys, unsigned small_max,
                                                                 int small_by_index, int64_t *__restrict__ out_idx,
                                                                 float *__restrict__ out_val, int32_t *__restrict__ out_count,
                                                                 unsigned char *__restrict__ out_sorted, int phase) {
  // phase 0: every segment, long ones through the digit passes' lists; phase 1: sieve path -- short segments and the
  // sieve lists of the long ones (3: the same, but every long segment gives up -- tests); phase 2: behind the guarded
  // digit passes -- only the segments the sieve gave up on
  extern __shared__ __align__(16) unsigned long long sk[];   // kSmallMax keys | kBitonicMax selected keys | kBins counters
  __shared__ int s_cnt;
  const int seg = blockIdx.x, tid = threadIdx.x;
  const SegDesc d = tab.s[seg];
  if (phase == 2 && (d.len <= small_max || !state[seg].need_slow)) return;
  const float *src = scores + d.off;
  int n_out = 0;
  bool by_index = false;
  if (tid == 0) s_cnt = 0;
  __syncthreads();
  unsigned long long *res = sk;   // where the sorted result ends up
  if (d.len > small_max && (phase == 1 || phase == 3)) {
    // ---- sieve path: select the k largest of the list, sort, prove that nothing outside the list can belong (see above)
    const SegState st = state[seg];
    const int cap = k + kBndCap, nc = st.sieve_count;
    if ((unsigned)nc < (unsigned)k || (unsigned)nc > (unsigned)cap || phase == 3) return;   // need_slow stays 1
    for (int i = tid; i < nc; i += kTailThreads) sk[i] = cand[(long long)seg * cap + i];
    __syncthreads();
    unsigned long long *sk2 = sk + kSmallMax;
    unsigned *h = reinterpret_cast<unsigned *>(sk2 + kBitonicMax);
    const unsigned long long thr = nc > k ? tail_select(sk, nc, k, h, tid) : 0ULL;
    for (int i = tid; i < nc; i += kTailThreads) {
      const unsigned long long key = sk[i];
      if (key >= thr) {
        const int pos = atomicAdd(&s_cnt, 1);
        if (pos < kBitonicMax) sk2[pos] = key;
      }
    }
    res = sk2, n_out = k;
    const int np2 = pow2_at_least(k);
    __syncthreads();
    for (int i = k + tid; i < np2; i += kTailThreads) res[i] = 0ULL;
    __syncthreads();
    tail_bitonic(res, np2, tid);
    const unsigned kth = (unsigned)(res[k - 1] >> 32);
    bool proven;
    if (SIGMOID) {
      // fp32 sigmoid = true sigmoid within 1.5 * 2^-22 relative (expf 2 ulp, one add, one division) where the result is
      // normal: a dropped x < T scores at most sigmoid_ref(T) * (1 + 2^-20); twice that slack and an absolute term for
      // subnormal scores are asked for here
      const double bound = (double)sigmoid_ref(st.sieve_t) * (1.0 + 1.9073486328125e-6) + 1e-37;
      proven = (double)okey_inv(kth) > bound;   // false for NaN
    } else {
      proven = kth >= okey(st.sieve_t);
    }
    if (!proven) return;
    if (tid == 0) state[seg].need_slow = 0;
  } else if (d.len <= small_max) {
    // ---- small segment: score; select the k largest if there are more (radix select in shared memory); sort
    const int len = (int)d.len;
    int mine = 0;
    for (int i = tid; i < len; i += kTailThreads) {
      const unsigned long long key = tail_key64<SIGMOID>(d, src, nullptr, (unsigned)i);
      sk[i] = key;
      mine += key != 0ULL;
    }
    mine = __reduce_add_sync(0xffffffffu, mine);
    if ((tid & 31) == 0 && mine) atomicAdd(&s_cnt, mine);
    __syncthreads();
    const int eff = s_cnt;
    n_out = min(k, eff);
    by_index = small_by_index && eff <= k;
    int nsort = len;
    if (eff > k) {
      unsigned long long *sk2 = sk + kSmallMax;
      unsigned *h = reinterpret_cast<unsigned *>(sk2 + kBitonicMax);
      const unsigned long long thr = tail_select(sk, len, k, h, tid);
      if (tid == 0) s_cnt = 0;
      __syncthreads();
      for (int i = tid; i < len; i += kTailThreads) {
        const unsigned long long key = sk[i];
        if (key != 0ULL && key >= thr) {
          const int pos = atomicAdd(&s_cnt, 1);
          if (pos < kBitonicMax) sk2[pos] = key;
        }
      }
      res = sk2, nsort = n_out;
    }
    const int np2 = pow2_at_least(nsort);
    __syncthreads();
    for (int i = nsort + tid; i < np2; i += kTailThreads) res[i] = 0ULL;
    if (by_index)
      for (int i = tid; i < nsort; i += kTailThreads) res[i] = swap_words(res[i]);   // index word leads (0 stays 0)
    __syncthreads();
    tail_bitonic(res, np2, tid);
  } else {
    SegState st = state[seg];
    n_out = st.k_take;
    by_index = small_by_index && st.eff_len <= (unsigned)k;
    if (n_out > 0) {
      if ((unsigned)st.bnd_count <= (unsigned)kBndCap) {
        // ---- the k_rem largest keys of the boundary bin join the cand_count certain ones
        const int nb = st.bnd_count, need = st.k_rem, c = n_out - need;
        const int np2 = pow2_at_least(nb);
        for (int i = tid; i < np2; i += kTailThreads) sk[i] = i < nb ? bnd[(long long)seg * kBndCap + i] : 0ULL;
        __syncthreads();
        tail_bitonic(sk, np2, tid);
        unsigned long long pick[kBndCap / kTailThreads];
#pragma unroll
        for (int j = 0; j < kBndCap / kTailThreads; ++j) {
          const int i = tid + j * kTailThreads;
          pick[j] = i < need ? sk[i] : 0ULL;
        }
        __syncthreads();
        for (int i = tid; i < c; i += kTailThreads) sk[i] = cand[(long long)seg * k + i];
#pragma unroll
        for (int j = 0; j < kBndCap / kTailThreads; ++j) {
          const int i = tid + j * kTailThreads;
          if (i < need) sk[c + i] = pick[j];
        }
      } else {
        // ---- mass ties: the remaining digit passes over the whole segment, by this CTA alone
        const unsigned *kbuf = keys != nullptr ? keys + d.koff : nullptr;
        unsigned *g = hist + (long long)seg * kBins;   // all zero: every scan leaves it clean
        for (int pass = 2; pass < 6; ++pass) {
          int shift, bits;
          pass_geometry(pass, shift, bits);
          const int decided = 64 - shift - bits;
          for (unsigned m = tid; m < d.len; m += kTailThreads) {
            const unsigned long long key = tail_key64<SIGMOID>(d, src, kbuf, m);
            if (key != 0ULL && (key >> (64 - decided)) == (st.prefix >> (64 - decided)))
              atomicAdd(&g[(unsigned)(key >> shift) & ((1u << bits) - 1u)], 1u);
          }
          __threadfence();
          __syncthreads();
          scan_segment(hist, state, seg, pass);
          __threadfence();
          __syncthreads();
          st.prefix = __ldcg(&state[seg].prefix), st.k_rem = __ldcg(&state[seg].k_rem);
        }
        for (unsigned m = tid; m < d.len; m += kTailThreads) {
          const unsigned long long key = tail_key64<SIGMOID>(d, src, kbuf, m);
          if (key != 0ULL && key >= st.prefix) {
            const int pos = atomicAdd(&s_cnt, 1);
            if (pos < kSmallMax) sk[pos] = key;
          }
        }
      }
      __syncthreads();
      const int np2 = pow2_at_least(n_out);
      for (int i = n_out + tid; i < np2; i += kTailThreads) sk[i] = 0ULL;
      if (by_index)
        for (int i = tid; i < n_out; i += kTailThreads) sk[i] = swap_words(sk[i]);
      __syncthreads();
      tail_bitonic(sk, np2, tid);
    }
  }
  for (int i = tid; i < k; i += kTailThreads) {
    long long oi = -1;
    float ov = 0.0f;
    if (i < n_out) {
      unsigned long long v = res[i];
      if (by_index) v = swap_words(v);
      oi = (long long)(unsigned)~(unsigned)v;
      ov = okey_inv((unsigned)(v >> 32));
    }
    out_idx[(long long)seg * k + i] = oi;
    out_val[(long long)seg * k + i] = ov;
  }
  if (tid == 0) {
    if (out_count != nullptr) out_count[seg] = n_out;
    if (out_sorted != nullptr) out_sorted[seg] = !by_index;
  }
}

__global__ void topk_init_kernel(SegState *state, int *tickets, const SegTable tab, int nseg, int k) {
  const int s = threadIdx.x;
  if (s >= nseg) return;
  tickets[s] = 0;
  SegState st;
  st.prefix = 0ULL;
  st.k_take = (int)min((unsigned)k, tab.s[s].len);
  st.k_rem = st.k_take;
  st.cand_count = 0;
  st.bnd_count = 0;
  st.eff_len = tab.s[s].len;
  st.sieve_t = 0.0f, st.sieve_count = 0, st.need_slow = 1;
  state[s] = st;
}

// What the callers downstream need to know about each segment without a host read: how many rows came back and
// whether they are in score order (1) or, for a small segment returned whole, in ascending logical index (0).
__global__ void topk_report_kernel(const SegState *state, int nseg, int k, int small_by_index, int32_t *out_count,
                                   unsigned char *out_sorted) {
  const int s = threadIdx.x;
  if (s >= nseg) return;
  if (out_count != nullptr) out_count[s] = state[s].k_take;
  if (out_sorted != nullptr) out_sorted[s] = !(small_by_index && state[s].eff_len <= (unsigned)k);
}

// ------------------------------------------------------------------------------------------------
// Fused anchors + delta2bbox3D + score append for selected anchors of one level.
// ------------------------------------------------------------------------------------------------
struct DecodeParams {
  const float *bbox_pred;  // [6A, D, H, W]
  int A, D, H, W;
  float stride, dstride;
  float base[16][6];
  float means[6], stds[6];
  float img_h, img_w, img_d;
  float max_ratio;
  const int64_t *idx;
  const float *scores;
  int n;
  float *out;
};

__global__ void __launch_bounds__(256) decode_proposals_kernel(const DecodeParams p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n) return;
  float *o = p.out + (long long)i * 7;
  const long long li = p.idx[i];
  if (li < 0) {
#pragma unroll
    for (int j = 0; j < 7; ++j) o[j] = 0.0f;
    return;
  }
  // logical index ((y*W + x)*D + z)*A + a   (anchor_generator_3d.py:59-70, np.meshgrid 'xy' order)
  long long t = li;
  const int a = (int)(t % p.A);
  t /= p.A;
  const int z = (int)(t % p.D);
  t /= p.D;
  const int x = (int)(t % p.W);
  const int y = (int)(t / p.W);
  const float sx = (float)x * p.stride, sy = (float)y * p.stride, sz = (float)z * p.dstride;
  const float ax1 = __fadd_rn(p.base[a][0], sx), ay1 = __fadd_rn(p.base[a][1], sy);
  const float ax2 = __fadd_rn(p.base[a][2], sx), ay2 = __fadd_rn(p.base[a][3], sy);
  const float az1 = __fadd_rn(p.base[a][4], sz), az2 = __fadd_rn(p.base[a][5], sz);
  const long long plane = (long long)p.D * p.H * p.W;
  const long long sp = ((long long)z * p.H + y) * p.W + x;
  float d[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    const float raw = __ldg(p.bbox_pred + (long long)(a * 6 + j) * plane + sp);
    d[j] = __fadd_rn(__fmul_rn(raw, p.stds[j]), p.means[j]);  // deltas * stds + means (transforms.py:114)
  }
  const float mr = p.max_ratio;
  const float dx = d[0], dy = d[1];
  const float dw = fminf(fmaxf(d[2], -mr), mr), dh = fminf(fmaxf(d[3], -mr), mr);
  const float dz = fminf(fmaxf(d[4], -mr), mr), dd = fminf(fmaxf(d[5], -mr), mr);
  const float px = __fmul_rn(__fadd_rn(ax1, ax2), 0.5f), py = __fmul_rn(__fadd_rn(ay1, ay2), 0.5f);
  const float pz = __fmul_rn(__fadd_rn(az1, az2), 0.5f);
  const float pw = __fadd_rn(__fsub_rn(ax2, ax1), 1.0f), ph = __fadd_rn(__fsub_rn(ay2, ay1), 1.0f);
  const float pdz = __fadd_rn(__fsub_rn(az2, az1), 1.0f);
  const float gw = __fmul_rn(pw, expf(dw)), gh = __fmul_rn(ph, expf(dh)), gd = __fmul_rn(pdz, expf(dd));
  const float gx = __fadd_rn(px, __fmul_rn(pw, dx)), gy = __fadd_rn(py, __fmul_rn(ph, dy));
  const float gz = __fadd_rn(pz, __fmul_rn(pdz, dz));
  float x1 = __fadd_rn(__fsub_rn(gx, __fmul_rn(gw, 0.5f)), 0.5f), y1 = __fadd_rn(__fsub_rn(gy, __fmul_rn(gh, 0.5f)), 0.5f);
  float x2 = __fsub_rn(__fadd_rn(gx, __fmul_rn(gw, 0.5f)), 0.5f), y2 = __fsub_rn(__fadd_rn(gy, __fmul_rn(gh, 0.5f)), 0.5f);
  float z1 = __fadd_rn(__fsub_rn(gz, __fmul_rn(gd, 0.5f)), 0.5f), z2 = __fsub_rn(__fadd_rn(gz, __fmul_rn(gd, 0.5f)), 0.5f);
  if (p.img_w > 0.0f) {
    x1 = fminf(fmaxf(x1, 0.0f), p.img_w - 1.0f), x2 = fminf(fmaxf(x2, 0.0f), p.img_w - 1.0f);
    y1 = fminf(fmaxf(y1, 0.0f), p.img_h - 1.0f), y2 = fminf(fmaxf(y2, 0.0f), p.img_h - 1.0f);
    z1 = fminf(fmaxf(z1, 0.0f), p.img_d - 1.0f), z2 = fminf(fmaxf(z2, 0.0f), p.img_d - 1.0f);
  }
  o[0] = x1, o[1] = y1, o[2] = x2, o[3] = y2, o[4] = z1, o[5] = z2;
  o[6] = p.scores ? p.scores[i] : 0.0f;
}

// Batched form: one launch decodes the selected anchors of every (image, level) segment.
struct DecodeSeg {
  const float *bbox_pred;  // [6A, D, H, W] of this (image, level)
  int A, D, H, W;
  int level;               // index into DecodeBatch::base / stride tables
  float img_h, img_w, img_d;
};

struct DecodeBatch {
  DecodeSeg seg[kMaxSeg];
  float base[ROI3D_MAX_LEVELS][4][6];
  float stride[ROI3D_MAX_LEVELS], dstride[ROI3D_MAX_LEVELS];
  float means[6], stds[6];
  float max_ratio;
  const int64_t *idx;   // [nseg, k]
  const float *scores;  // [nseg, k]
  int k;
  float *out;           // [nseg, k, 7]
};

__global__ void __launch_bounds__(256) decode_proposals_batched_kernel(const DecodeBatch b) {
  const int s = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b.k) return;
  DecodeParams p;
  const DecodeSeg &sg = b.seg[s];
  p.bbox_pred = sg.bbox_pred, p.A = sg.A, p.D = sg.D, p.H = sg.H, p.W = sg.W;
  p.stride = b.stride[sg.level], p.dstride = b.dstride[sg.level];
  float *o = b.out + ((long long)s * b.k + i) * 7;
  const long long li = b.idx[(long long)s * b.k + i];
  if (li < 0) {
#pragma unroll
    for (int j = 0; j < 7; ++j) o[j] = 0.0f;
    return;
  }
  long long t = li;
  const int a = (int)(t % p.A);
  t /= p.A;
  const int z = (int)(t % p.D);
  t /= p.D;
  const int x = (int)(t % p.W);
  const int y = (int)(t / p.W);
  const float *bs = b.base[sg.level][a];
  const float sx = (float)x * p.stride, sy = (float)y * p.stride, sz = (float)z * p.dstride;
  const float ax1 = __fadd_rn(bs[0], sx), ay1 = __fadd_rn(bs[1], sy);
  const float ax2 = __fadd_rn(bs[2], sx), ay2 = __fadd_rn(bs[3], sy);
  const float az1 = __fadd_rn(bs[4], sz), az2 = __fadd_rn(bs[5], sz);
  const long long plane = (long long)p.D * p.H * p.W;
  const long long sp = ((long long)z * p.H + y) * p.W + x;
  float d[6];
#pragma unroll
  for (int j = 0; j < 6; ++j)
    d[j] = __fadd_rn(__fmul_rn(__ldg(p.bbox_pred + (long long)(a * 6 + j) * plane + sp), b.stds[j]), b.means[j]);
  const float mr = b.max_ratio;
  const float dw = fminf(fmaxf(d[2], -mr), mr), dh = fminf(fmaxf(d[3], -mr), mr);
  const float dz = fminf(fmaxf(d[4], -mr), mr), dd = fminf(fmaxf(d[5], -mr), mr);
  const float px = __fmul_rn(__fadd_rn(ax1, ax2), 0.5f), py = __fmul_rn(__fadd_rn(ay1, ay2), 0.5f);
  const float pz = __fmul_rn(__fadd_rn(az1, az2), 0.5f);
  const float pw = __fadd_rn(__fsub_rn(ax2, ax1), 1.0f), ph = __fadd_rn(__fsub_rn(ay2, ay1), 1.0f);
  const float pdz = __fadd_rn(__fsub_rn(az2, az1), 1.0f);
  const float gw = __fmul_rn(pw, expf(dw)), gh = __fmul_rn(ph, expf(dh)), gd = __fmul_rn(pdz, expf(dd));
  const float gx = __fadd_rn(px, __fmul_rn(pw, d[0])), gy = __fadd_rn(py, __fmul_rn(ph, d[1]));
  const float gz = __fadd_rn(pz, __fmul_rn(pdz, dz));
  float x1 = __fadd_rn(__fsub_rn(gx, __fmul_rn(gw, 0.5f)), 0.5f), y1 = __fadd_rn(__fsub_rn(gy, __fmul_rn(gh, 0.5f)), 0.5f);
  float x2 = __fsub_rn(__fadd_rn(gx, __fmul_rn(gw, 0.5f)), 0.5f), y2 = __fsub_rn(__fadd_rn(gy, __fmul_rn(gh, 0.5f)), 0.5f);
  float z1 = __fadd_rn(__fsub_rn(gz, __fmul_rn(gd, 0.5f)), 0.5f), z2 = __fsub_rn(__fadd_rn(gz, __fmul_rn(gd, 0.5f)), 0.5f);
  if (sg.img_w > 0.0f) {
    x1 = fminf(fmaxf(x1, 0.0f), sg.img_w - 1.0f), x2 = fminf(fmaxf(x2, 0.0f), sg.img_w - 1.0f);
    y1 = fminf(fmaxf(y1, 0.0f), sg.img_h - 1.0f), y2 = fminf(fmaxf(y2, 0.0f), sg.img_h - 1.0f);
    z1 = fminf(fmaxf(z1, 0.0f), sg.img_d - 1.0f), z2 = fminf(fmaxf(z2, 0.0f), sg.img_d - 1.0f);
  }
  o[0] = x1, o[1] = y1, o[2] = x2, o[3] = y2, o[4] = z1, o[5] = z2;
  o[6] = b.scores ? b.scores[(long long)s * b.k + i] : 0.0f;
}

// ------------------------------------------------------------------------------------------------
// Tail of RPNHead3D.get_bboxes_single for every (image, level) segment at once (rpn_head_3d.py:135-148):
// proposals[:nms_post] of each level in NMS return order, concatenated per image in level order; scores of the
// unused tail are -inf so that the following top-k(max_num) ignores them.
// grid (ceil(P/256), B*L).  keep_sel[s] picks, per segment, the score-ordered or the index-ordered keep list.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rpn_collect_kernel(const float *__restrict__ dets, int k,
                                                          const int64_t *__restrict__ keep_by_score,
                                                          const int64_t *__restrict__ keep_by_index,
                                                          const int32_t *__restrict__ num_keep,
                                                          const unsigned char *__restrict__ use_index_order, int L, int P,
                                                          float *__restrict__ cat_props, float *__restrict__ cat_scores,
                                                          int32_t *__restrict__ n_valid) {
  const int seg = blockIdx.y, b = seg / L, l = seg - b * L;
  const int i = blockIdx.x * 256 + threadIdx.x;
  int before = 0, total = 0, mine = 0;
  for (int q = 0; q < L; ++q) {
    const int c = min(max(num_keep[b * L + q], 0), P);
    if (q < l) before += c;
    if (q == l) mine = c;
    total += c;
  }
  if (l == 0 && i == 0) n_valid[b] = total;
  if (i >= P) return;
  const long long row0 = (long long)b * L * P;
  if (i < mine) {
    const int64_t *keep = (use_index_order != nullptr && use_index_order[seg]) ? keep_by_index : keep_by_score;
    long long r = keep[(long long)seg * k + i];
    r = r < 0 ? 0 : (r >= k ? k - 1 : r);
    const float *src = dets + ((long long)seg * k + r) * 7;
    float *dst = cat_props + (row0 + before + i) * 7;
#pragma unroll
    for (int q = 0; q < 7; ++q) dst[q] = src[q];
    cat_scores[row0 + before + i] = src[6];
  } else {
    // this segment's unused slots fill the image's tail: total + (slack of earlier levels) + own slack position
    const int slack_before = l * P - before;
    const long long pos = row0 + total + slack_before + (i - mine);
    cat_scores[pos] = -INFINITY;
  }
}

// out[b][j] = rows[b][idx[b][j]] (7 floats); idx < 0 -> zeros.  grid (ceil(n/256), B)
__global__ void __launch_bounds__(256) gather_rows7_kernel(const float *__restrict__ rows, int rows_per_seg,
                                                           const int64_t *__restrict__ idx, int n,
                                                           float *__restrict__ out) {
  const int b = blockIdx.y, j = blockIdx.x * 256 + threadIdx.x;
  if (j >= n) return;
  const long long r = idx[(long long)b * n + j];
  float *dst = out + ((long long)b * n + j) * 7;
  if (r < 0 || r >= rows_per_seg) {
#pragma unroll
    for (int q = 0; q < 7; ++q) dst[q] = 0.0f;
    return;
  }
  const float *src = rows + ((long long)b * rows_per_seg + r) * 7;
#pragma unroll
  for (int q = 0; q < 7; ++q) dst[q] = src[q];
}

// ------------------------------------------------------------------------------------------------
// `min_bbox_size` filter of get_bboxes_single (mmdet v0.6.0 RPNHead): keep a row iff (x2 - x1) + 1 >= m and
// (y2 - y1) + 1 >= m, each operation one fp32 rounding as torch evaluates it; NaN fails.  Depth is not compared.
// Stable in-place compaction of the first counts_in[s] rows of each segment, one CTA per segment: per chunk of
// kFilterThreads * kFilterRows rows every thread holds its rows in registers, warp ballots give each (row slot, warp)
// its count, warp 0 scans the counts, and the survivors are written at the running offset.  A write never reaches
// past the chunk being processed (the offset never exceeds the chunk start), and every read of the chunk happens
// before the first barrier, so rows are not overwritten before they are read.  Two barriers per chunk also order the
// shared counts and offsets across chunks: a chunk's counts are written after the previous chunk's second barrier,
// its offsets after its own first one.  The count lands in counts_out[s].
// ------------------------------------------------------------------------------------------------
constexpr int kFilterThreads = 512;
constexpr int kFilterRows = 4;                                   // rows per thread per chunk
constexpr int kFilterWarps = kFilterThreads / 32;
constexpr int kFilterSlots = kFilterRows * kFilterWarps;         // (row slot, warp) counts per chunk, scanned by warp 0
static_assert(kFilterSlots == 64, "warp 0 scans two slots per lane");

__global__ void __launch_bounds__(kFilterThreads) filter_min_size_rows7_kernel(float *__restrict__ dets, int k,
                                                                                const int32_t *counts_in, float m,
                                                                                int32_t *counts_out) {
  __shared__ int slot_cnt[kFilterSlots];
  __shared__ int slot_off[kFilterSlots + 1];
  const int s = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = min(max(counts_in[s], 0), k);
  float *d = dets + (long long)s * k * 7;
  int kept = 0;   // rows written so far (the same in every thread)
  for (int base = 0; base < n; base += kFilterThreads * kFilterRows) {
    float r[kFilterRows][7];
    bool pass[kFilterRows];
    unsigned ball[kFilterRows];
#pragma unroll
    for (int j = 0; j < kFilterRows; ++j) {
      const int i = base + j * kFilterThreads + threadIdx.x;
      pass[j] = false;
      if (i < n) {
#pragma unroll
        for (int q = 0; q < 7; ++q) r[j][q] = d[(long long)i * 7 + q];
        const float w = __fadd_rn(__fsub_rn(r[j][2], r[j][0]), 1.0f);
        const float h = __fadd_rn(__fsub_rn(r[j][3], r[j][1]), 1.0f);
        pass[j] = (w >= m) && (h >= m);
      }
      ball[j] = __ballot_sync(0xffffffffu, pass[j]);
      if (lane == 0) slot_cnt[j * kFilterWarps + warp] = __popc(ball[j]);
    }
    __syncthreads();
    if (warp == 0) {   // exclusive scan of the 64 slot counts in (row slot, warp) order = row order
      const int a = slot_cnt[2 * lane], b = slot_cnt[2 * lane + 1];
      int incl = a + b;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      slot_off[2 * lane] = incl - a - b;
      slot_off[2 * lane + 1] = incl - b;
      if (lane == 31) slot_off[kFilterSlots] = incl;
    }
    __syncthreads();
    const unsigned below = (1u << lane) - 1u;
#pragma unroll
    for (int j = 0; j < kFilterRows; ++j) {
      if (!pass[j]) continue;
      const int i = base + j * kFilterThreads + threadIdx.x;
      const int o = kept + slot_off[j * kFilterWarps + warp] + __popc(ball[j] & below);
      if (o != i) {
#pragma unroll
        for (int q = 0; q < 7; ++q) d[(long long)o * 7 + q] = r[j][q];
      }
    }
    kept += slot_off[kFilterSlots];
  }
  __syncthreads();   // counts_out may be counts_in: every thread has read its count
  if (threadIdx.x == 0) counts_out[s] = kept;
}

int g_topk_sieve = 0;   // roi3d_set_tuning key 11: 0 = sieve path where it applies, -1 = digit passes only, 2 = sieve gives up (tests)

}  // namespace roi3d

using namespace roi3d;

extern "C" {

// Longest segment: the kernels index a segment's elements with 32-bit unsigned integers and add up to one flat-grid
// chunk (kFirstItemsPerCta = 32768 elements) to an index before they compare it with the end, so the length keeps
// 64 K of margin below 2^32.
static const long long kMaxSegLen = 0xFFFF0000LL;
static const size_t kStateBytes = 4096;                                     // kMaxSeg * sizeof(SegState) + tickets, rounded up
static const size_t kHistBytes = (size_t)kMaxSeg * kBins * sizeof(unsigned);  // 512 KiB

size_t roi3d_topk_workspace_bytes(int nseg, int k) {
  if (nseg <= 0 || k <= 0) return 256;
  const size_t ns = (size_t)(nseg < kMaxSeg ? nseg : kMaxSeg);
  const size_t b = kStateBytes + kHistBytes + ns * (size_t)k * sizeof(unsigned long long) +
                   ns * (size_t)kBndCap * sizeof(unsigned long long);
  return (b + 255) / 256 * 256;
}

size_t roi3d_topk_workspace_bytes_keys(int nseg, int k, int64_t total_len) {
  const size_t base = roi3d_topk_workspace_bytes(nseg, k);
  if (nseg <= 0 || k <= 0 || total_len <= 0) return base;
  return base + (((size_t)total_len + 4 * (size_t)nseg) * sizeof(unsigned) + 255) / 256 * 256;
}

int roi3d_topk_segmented(const float *scores_dev, const int64_t *seg_off, const int64_t *seg_len,
                         const int32_t *seg_adhw, int nseg, int k, int apply_sigmoid, int64_t *out_idx_dev,
                         float *out_val_dev, void *workspace_dev, size_t workspace_bytes, void *stream) {
  return roi3d_topk_segmented_ex(scores_dev, seg_off, seg_len, seg_adhw, nseg, k, apply_sigmoid, 0, out_idx_dev,
                                 out_val_dev, workspace_dev, workspace_bytes, stream);
}

int roi3d_topk_segmented_ex(const float *scores_dev, const int64_t *seg_off, const int64_t *seg_len,
                            const int32_t *seg_adhw, int nseg, int k, int apply_sigmoid, int small_segments_in_index_order,
                            int64_t *out_idx_dev, float *out_val_dev, void *workspace_dev, size_t workspace_bytes,
                            void *stream) {
  return roi3d_topk_segmented_masked(scores_dev, seg_off, seg_len, seg_adhw, nullptr, nseg, k, apply_sigmoid,
                                     small_segments_in_index_order, out_idx_dev, out_val_dev, nullptr, nullptr,
                                     workspace_dev, workspace_bytes, stream);
}

int roi3d_topk_segmented_masked(const float *scores_dev, const int64_t *seg_off, const int64_t *seg_len,
                                const int32_t *seg_adhw, const uint8_t *const *seg_mask_dev_ptrs, int nseg, int k,
                                int apply_sigmoid, int small_segments_in_index_order, int64_t *out_idx_dev,
                                float *out_val_dev, int32_t *out_count_dev, uint8_t *out_sorted_dev, void *workspace_dev,
                                size_t workspace_bytes, void *stream) {
  ROI3D_CHECK_ARG(nseg >= 0 && k >= 0, "bad sizes");
  if (nseg == 0 || k == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(scores_dev && seg_off && seg_len && out_idx_dev && out_val_dev && workspace_dev, "NULL pointer");
  ROI3D_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace_dev) & 255) == 0, "workspace must be 256-byte aligned");
  if (workspace_bytes < roi3d_topk_workspace_bytes(nseg, k)) {
    set_error("topk workspace too small: %zu < %zu", workspace_bytes, roi3d_topk_workspace_bytes(nseg, k));
    return ROI3D_ENOMEM;
  }
  cudaStream_t st = (cudaStream_t)stream;
  // k <= kBitonicMax: the tail kernel finishes every segment in one launch (and fills the unused rows itself)
  const bool tail = k <= kBitonicMax;
  const unsigned small_max = tail ? (unsigned)kSmallMax : 0u;
  if (!tail) {
    ROI3D_CUDA(cudaMemsetAsync(out_idx_dev, 0xFF, sizeof(int64_t) * (size_t)nseg * k, st));
    ROI3D_CUDA(cudaMemsetAsync(out_val_dev, 0, sizeof(float) * (size_t)nseg * k, st));
  }
  // optional key buffer behind the base workspace (roi3d_topk_workspace_bytes_keys): one u32 per score of a batch of
  // kMaxSeg segments, written by the first digit pass and read back (from L2) by the later full passes
  long long total_len = 0;
  for (int s = 0; s < nseg; ++s) total_len += seg_len[s] > 0 ? seg_len[s] : 0;
  const size_t base_bytes = roi3d_topk_workspace_bytes(nseg, k);
  unsigned *keys = workspace_bytes >= roi3d_topk_workspace_bytes_keys(nseg, k, total_len) && total_len > 0
                       ? reinterpret_cast<unsigned *>(static_cast<char *>(workspace_dev) + base_bytes)
                       : nullptr;
  for (int s0 = 0; s0 < nseg; s0 += kMaxSeg) {
    const int ns = nseg - s0 < kMaxSeg ? nseg - s0 : kMaxSeg;
    SegTable tab;
    long long maxlen = 0, koff = 0;   // maxlen: over the segments that go through the digit passes
    for (int s = 0; s < ns; ++s) {
      ROI3D_CHECK_ARG(seg_len[s0 + s] >= 0 && seg_len[s0 + s] <= kMaxSegLen, "segment %d: length %lld outside [0, %lld]", s0 + s,
                      (long long)seg_len[s0 + s], kMaxSegLen);
      tab.s[s].off = seg_off[s0 + s];
      tab.s[s].len = (unsigned)seg_len[s0 + s];
      if (seg_adhw) {
        tab.s[s].A = seg_adhw[(s0 + s) * 4 + 0], tab.s[s].D = seg_adhw[(s0 + s) * 4 + 1];
        tab.s[s].H = seg_adhw[(s0 + s) * 4 + 2], tab.s[s].W = seg_adhw[(s0 + s) * 4 + 3];
        ROI3D_CHECK_ARG(tab.s[s].A == 0 || (long long)tab.s[s].A * tab.s[s].D * tab.s[s].H * tab.s[s].W == seg_len[s0 + s],
                        "segment %d: A*D*H*W != len", s0 + s);
      } else {
        tab.s[s].A = tab.s[s].D = tab.s[s].H = tab.s[s].W = 0;
      }
      tab.s[s].mask = seg_mask_dev_ptrs != nullptr ? seg_mask_dev_ptrs[s0 + s] : nullptr;
      tab.s[s].koff = koff;
      koff += (seg_len[s0 + s] + 3) / 4 * 4;   // every segment's keys start on a 16-byte boundary
      if (seg_len[s0 + s] > (long long)small_max && seg_len[s0 + s] > maxlen) maxlen = seg_len[s0 + s];
    }
    {
      unsigned c = 0;
      for (int s = 0; s <= kMaxSeg; ++s) {
        tab.cta0[s] = c;
        if (s < ns && seg_len[s0 + s] > (long long)small_max) c += (unsigned)ceil_div_ll(seg_len[s0 + s], kFirstItemsPerCta);
      }
    }
    const unsigned flat_ctas = tab.cta0[kMaxSeg];
    static_assert(sizeof(SegState) * kMaxSeg + sizeof(int) * kMaxSeg <= 4096, "state block");
    char *b = static_cast<char *>(workspace_dev);
    SegState *state = reinterpret_cast<SegState *>(b);
    unsigned *hist = reinterpret_cast<unsigned *>(b + kStateBytes);
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(b + kStateBytes + kHistBytes);
    unsigned long long *bnd = cand + (size_t)(nseg < kMaxSeg ? nseg : kMaxSeg) * k;
    int *tickets = reinterpret_cast<int *>(b + sizeof(SegState) * kMaxSeg);  // inside the 4 KB state block
    int32_t *cnt_out = out_count_dev ? out_count_dev + s0 : nullptr;
    uint8_t *srt_out = out_sorted_dev ? out_sorted_dev + s0 : nullptr;
    // sieve path (see topk_sample_kernel): one pass over the scores; needs the key buffer for its guarded fallback
    bool sieve = tail && keys != nullptr && maxlen > 0 && g_topk_sieve >= 0;
    for (int s = 0; s < ns && sieve; ++s) sieve = tab.s[s].mask == nullptr;
    if (sieve) {
      static PerDeviceSmemOptIn tail_opt_in;
      if (tail_opt_in.need(kTailSmemBytes)) {
        ROI3D_CUDA(cudaFuncSetAttribute(topk_tail_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmemBytes));
        ROI3D_CUDA(cudaFuncSetAttribute(topk_tail_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmemBytes));
        tail_opt_in.mark(kTailSmemBytes);
      }
      topk_sample_kernel<<<ns * kSieveCluster, kSieveThreads, 0, st>>>(scores_dev, tab, state, tickets, hist, k, small_max);
      ROI3D_LAUNCH_CHECK();
      const int phase = g_topk_sieve == 2 ? 3 : 1;
      if (apply_sigmoid) {
        topk_sieve_kernel<true><<<flat_ctas * kKeySub, kKeyThreads, 0, st>>>(scores_dev, tab, state, k, cand);
        ROI3D_LAUNCH_CHECK();
        topk_tail_kernel<true><<<ns, kTailThreads, kTailSmemBytes, st>>>(
            scores_dev, tab, state, hist, k, cand, bnd, keys, small_max, small_segments_in_index_order,
            out_idx_dev + (size_t)s0 * k, out_val_dev + (size_t)s0 * k, cnt_out, srt_out, phase);
      } else {
        topk_sieve_kernel<false><<<flat_ctas * kKeySub, kKeyThreads, 0, st>>>(scores_dev, tab, state, k, cand);
        ROI3D_LAUNCH_CHECK();
        topk_tail_kernel<false><<<ns, kTailThreads, kTailSmemBytes, st>>>(
            scores_dev, tab, state, hist, k, cand, bnd, keys, small_max, small_segments_in_index_order,
            out_idx_dev + (size_t)s0 * k, out_val_dev + (size_t)s0 * k, cnt_out, srt_out, phase);
      }
      ROI3D_LAUNCH_CHECK();
    } else if (maxlen > 0 || !tail) {
      topk_init_kernel<<<1, kMaxSeg, 0, st>>>(state, tickets, tab, ns, k);
      ROI3D_LAUNCH_CHECK();
    }
    if (maxlen > 0) {
      if (!sieve) ROI3D_CUDA(cudaMemsetAsync(hist, 0, (size_t)ns * kBins * sizeof(unsigned), st));
      const dim3 grid((unsigned)ceil_div_ll(maxlen, kItemsPerCta), ns);
      const dim3 grid2((unsigned)(grid.x < 8 ? grid.x : 8), ns);  // boundary passes: see topk_hist_kernel
      {
        static PerDeviceSmemOptIn opt_in;
        if (opt_in.need(kFirstSmemBytes)) {
          ROI3D_CUDA(cudaFuncSetAttribute(topk_first_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFirstSmemBytes));
          ROI3D_CUDA(cudaFuncSetAttribute(topk_first_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFirstSmemBytes));
          opt_in.mark(kFirstSmemBytes);
        }
        if (apply_sigmoid)
          topk_first_kernel<true><<<flat_ctas, kFirstThreads, kFirstSmemBytes, st>>>(scores_dev, tab, state, hist, tickets, keys);
        else
          topk_first_kernel<false><<<flat_ctas, kFirstThreads, kFirstSmemBytes, st>>>(scores_dev, tab, state, hist, tickets, keys);
        ROI3D_LAUNCH_CHECK();
      }
      if (keys != nullptr) {  // digit pass 1 and the split over the stored keys
        topk_second_kernel<<<flat_ctas * kKeySub, kKeyThreads, 0, st>>>(tab, state, hist, tickets, keys);
        ROI3D_LAUNCH_CHECK();
        topk_split_keys_kernel<<<flat_ctas * kKeySub, kKeyThreads, 0, st>>>(tab, state, k, cand, bnd, keys);
        ROI3D_LAUNCH_CHECK();
        if (!tail) {
          topk_after_split_kernel<<<1, kMaxSeg, 0, st>>>(state, ns);
          ROI3D_LAUNCH_CHECK();
        }
      }
      for (int pass = keys != nullptr ? 2 : 1; pass < (tail ? 2 : 6); ++pass) {
        const unsigned long long *b2 = pass >= 2 ? bnd : nullptr;
        const dim3 g = pass >= 2 ? grid2 : grid;
        if (apply_sigmoid)
          topk_hist_kernel<true><<<g, kTopkThreads, 0, st>>>(scores_dev, tab, state, pass, hist, b2, tickets, keys, small_max);
        else
          topk_hist_kernel<false><<<g, kTopkThreads, 0, st>>>(scores_dev, tab, state, pass, hist, b2, tickets, keys, small_max);
        ROI3D_LAUNCH_CHECK();
        if (pass == 1) {  // 22 bits decided: split off the certain keys and the boundary bin
          if (apply_sigmoid)
            topk_split_kernel<true><<<grid, kTopkThreads, 0, st>>>(scores_dev, tab, state, k, cand, bnd, keys, small_max);
          else
            topk_split_kernel<false><<<grid, kTopkThreads, 0, st>>>(scores_dev, tab, state, k, cand, bnd, keys, small_max);
          ROI3D_LAUNCH_CHECK();
          if (!tail) {
            topk_after_split_kernel<<<1, kMaxSeg, 0, st>>>(state, ns);
            ROI3D_LAUNCH_CHECK();
          }
        }
      }
      if (!tail) {
        if (apply_sigmoid)
          topk_collect_kernel<true><<<grid2, kTopkThreads, 0, st>>>(scores_dev, tab, state, k, cand, bnd, keys);
        else
          topk_collect_kernel<false><<<grid2, kTopkThreads, 0, st>>>(scores_dev, tab, state, k, cand, bnd, keys);
        ROI3D_LAUNCH_CHECK();
      }
    }
    if (tail) {
      static PerDeviceSmemOptIn tail_opt_in;
      if (tail_opt_in.need(kTailSmemBytes)) {
        ROI3D_CUDA(cudaFuncSetAttribute(topk_tail_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmemBytes));
        ROI3D_CUDA(cudaFuncSetAttribute(topk_tail_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTailSmemBytes));
        tail_opt_in.mark(kTailSmemBytes);
      }
      if (apply_sigmoid)
        topk_tail_kernel<true><<<ns, kTailThreads, kTailSmemBytes, st>>>(
            scores_dev, tab, state, hist, k, cand, bnd, keys, small_max, small_segments_in_index_order,
            out_idx_dev + (size_t)s0 * k, out_val_dev + (size_t)s0 * k, cnt_out, srt_out, sieve ? 2 : 0);
      else
        topk_tail_kernel<false><<<ns, kTailThreads, kTailSmemBytes, st>>>(
            scores_dev, tab, state, hist, k, cand, bnd, keys, small_max, small_segments_in_index_order,
            out_idx_dev + (size_t)s0 * k, out_val_dev + (size_t)s0 * k, cnt_out, srt_out, sieve ? 2 : 0);
      ROI3D_LAUNCH_CHECK();
      continue;
    }
    topk_sort_kernel<<<dim3(ceil_div(k, 256), ns), 256, 0, st>>>(cand, state, tab, small_segments_in_index_order, k,
                                                                out_idx_dev + (size_t)s0 * k, out_val_dev + (size_t)s0 * k);
    ROI3D_LAUNCH_CHECK();
    if (cnt_out != nullptr || srt_out != nullptr) {
      topk_report_kernel<<<1, kMaxSeg, 0, st>>>(state, ns, k, small_segments_in_index_order, cnt_out, srt_out);
      ROI3D_LAUNCH_CHECK();
    }
  }
  return ROI3D_OK;
}

int roi3d_decode_proposals(const float *bbox_pred_dev, int A, int D, int H, int W, float stride, float depth_stride,
                           const float *base_anchors_host, const int64_t *idx_dev, const float *scores_dev, int n,
                           const float *means6_host, const float *stds6_host, float img_h, float img_w, float img_d,
                           float *out_dev, void *stream) {
  ROI3D_CHECK_ARG(n >= 0, "bad n");
  if (n == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(bbox_pred_dev && base_anchors_host && idx_dev && out_dev, "NULL pointer");
  ROI3D_CHECK_ARG(A >= 1 && A <= 16, "A=%d out of [1,16]", A);
  ROI3D_CHECK_ARG(D > 0 && H > 0 && W > 0, "bad dims");
  DecodeParams p;
  p.bbox_pred = bbox_pred_dev, p.A = A, p.D = D, p.H = H, p.W = W, p.stride = stride, p.dstride = depth_stride;
  for (int a = 0; a < A; ++a)
    for (int j = 0; j < 6; ++j) p.base[a][j] = base_anchors_host[a * 6 + j];
  for (int j = 0; j < 6; ++j) {
    p.means[j] = means6_host ? means6_host[j] : 0.0f;
    p.stds[j] = stds6_host ? stds6_host[j] : 1.0f;
  }
  p.img_h = img_h, p.img_w = img_w, p.img_d = img_d;
  // max_ratio = np.abs(np.log(16/1000)) evaluated in float64 then used as a python float by clamp
  p.max_ratio = (float)4.135166556742356;
  p.idx = idx_dev, p.scores = scores_dev, p.n = n, p.out = out_dev;
  decode_proposals_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(p);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

int roi3d_decode_proposals_batched(const float *const *bbox_pred_dev_ptrs, const int32_t *seg_adhw,
                                   const int32_t *seg_level, const float *seg_img_hwd, int nseg, int num_levels,
                                   int A, const float *base_anchors_host, const float *strides_host,
                                   const float *depth_strides_host, const int64_t *idx_dev, const float *scores_dev,
                                   int k, const float *means6_host, const float *stds6_host, float *out_dev,
                                   void *stream) {
  ROI3D_CHECK_ARG(nseg >= 0 && k >= 0, "bad sizes");
  if (nseg == 0 || k == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(bbox_pred_dev_ptrs && seg_adhw && seg_level && base_anchors_host && strides_host &&
                      depth_strides_host && idx_dev && out_dev,
                  "NULL pointer");
  ROI3D_CHECK_ARG(A >= 1 && A <= 4, "batched decode supports 1..4 base anchors per level, got %d", A);
  ROI3D_CHECK_ARG(num_levels >= 1 && num_levels <= ROI3D_MAX_LEVELS, "num_levels out of range");
  cudaStream_t st = (cudaStream_t)stream;
  for (int s0 = 0; s0 < nseg; s0 += kMaxSeg) {
    const int ns = nseg - s0 < kMaxSeg ? nseg - s0 : kMaxSeg;
    DecodeBatch b;
    for (int s = 0; s < ns; ++s) {
      DecodeSeg &sg = b.seg[s];
      sg.bbox_pred = bbox_pred_dev_ptrs[s0 + s];
      sg.A = seg_adhw[(s0 + s) * 4 + 0], sg.D = seg_adhw[(s0 + s) * 4 + 1];
      sg.H = seg_adhw[(s0 + s) * 4 + 2], sg.W = seg_adhw[(s0 + s) * 4 + 3];
      sg.level = seg_level[s0 + s];
      ROI3D_CHECK_ARG(sg.A == A && sg.level >= 0 && sg.level < num_levels && sg.bbox_pred, "segment %d: bad descriptor", s0 + s);
      sg.img_h = seg_img_hwd ? seg_img_hwd[(s0 + s) * 3 + 0] : 0.0f;
      sg.img_w = seg_img_hwd ? seg_img_hwd[(s0 + s) * 3 + 1] : 0.0f;
      sg.img_d = seg_img_hwd ? seg_img_hwd[(s0 + s) * 3 + 2] : 0.0f;
    }
    for (int l = 0; l < num_levels; ++l) {
      for (int a = 0; a < A; ++a)
        for (int j = 0; j < 6; ++j) b.base[l][a][j] = base_anchors_host[(l * A + a) * 6 + j];
      b.stride[l] = strides_host[l], b.dstride[l] = depth_strides_host[l];
    }
    for (int j = 0; j < 6; ++j) {
      b.means[j] = means6_host ? means6_host[j] : 0.0f;
      b.stds[j] = stds6_host ? stds6_host[j] : 1.0f;
    }
    b.max_ratio = (float)4.135166556742356;
    b.idx = idx_dev + (size_t)s0 * k, b.scores = scores_dev ? scores_dev + (size_t)s0 * k : nullptr;
    b.k = k, b.out = out_dev + (size_t)s0 * k * 7;
    decode_proposals_batched_kernel<<<dim3(ceil_div(k, 256), ns), 256, 0, st>>>(b);
    ROI3D_LAUNCH_CHECK();
  }
  return ROI3D_OK;
}

int roi3d_rpn_collect(const float *dets_dev, int num_images, int num_levels, int k, const int64_t *keep_by_score_dev,
                      const int64_t *keep_by_index_dev, const int32_t *num_keep_dev,
                      const uint8_t *use_index_order_dev, int nms_post, float *cat_props_dev, float *cat_scores_dev,
                      int32_t *n_valid_dev, void *stream) {
  ROI3D_CHECK_ARG(num_images >= 0 && num_levels >= 1 && k >= 1 && nms_post >= 1, "bad sizes");
  if (num_images == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(dets_dev && keep_by_score_dev && num_keep_dev && cat_props_dev && cat_scores_dev && n_valid_dev,
                  "NULL pointer");
  ROI3D_CHECK_ARG(use_index_order_dev == nullptr || keep_by_index_dev != nullptr, "keep_by_index is NULL");
  ROI3D_CHECK_ARG((long long)num_images * num_levels <= 65535, "too many segments");
  const int P = nms_post < k ? nms_post : k;
  rpn_collect_kernel<<<dim3(ceil_div(P, 256), num_images * num_levels), 256, 0, (cudaStream_t)stream>>>(
      dets_dev, k, keep_by_score_dev, keep_by_index_dev, num_keep_dev, use_index_order_dev, num_levels, P, cat_props_dev,
      cat_scores_dev, n_valid_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

int roi3d_gather_rows7(const float *rows_dev, int nseg, int rows_per_seg, const int64_t *idx_dev, int n, float *out_dev,
                       void *stream) {
  ROI3D_CHECK_ARG(nseg >= 0 && rows_per_seg >= 0 && n >= 0 && nseg <= 65535, "bad sizes");
  if (nseg == 0 || n == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG(rows_dev && idx_dev && out_dev, "NULL pointer");
  gather_rows7_kernel<<<dim3(ceil_div(n, 256), nseg), 256, 0, (cudaStream_t)stream>>>(rows_dev, rows_per_seg, idx_dev, n,
                                                                                      out_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

int roi3d_filter_min_size_rows7(float *dets_dev, int nseg, int k, const int32_t *counts_in_dev, float min_size,
                                int32_t *counts_out_dev, void *stream) {
  ROI3D_CHECK_ARG(nseg >= 0 && k >= 0, "bad sizes: nseg=%d k=%d", nseg, k);
  ROI3D_CHECK_ARG(min_size == min_size, "min_size is NaN");
  if (nseg == 0) return ROI3D_OK;
  ROI3D_CHECK_ARG((dets_dev || k == 0) && counts_in_dev && counts_out_dev, "NULL pointer");
  filter_min_size_rows7_kernel<<<nseg, kFilterThreads, 0, (cudaStream_t)stream>>>(dets_dev, k, counts_in_dev, min_size,
                                                                                 counts_out_dev);
  ROI3D_LAUNCH_CHECK();
  return ROI3D_OK;
}

}  // extern "C"

"""Every path of the segmented top-k (csrc/proposal.cu), reached through the C ABI, checked against a plain reference --
and checked to be the path that actually ran.

`roi3d_topk_segmented_masked` chooses per call and per batch of 64 segments among: the tail kernel alone (every
segment at most 8192 long, k <= 4096), the sieve (no masks, a key buffer, k <= 4096) and its give-up, the digit passes
over the stored keys or over the raw scores (the workspace decides whether there is a key buffer), and for k > 4096
the non-tail passes (collect, rank sort, optional report).  Inside those, the boundary bin of the k-th key either fits
its 4096-key buffer or overflows into the full-data passes, and masks, index-order segments and empty segments take
their own branches.  COVERAGE names, for each row, the exact set of top-k kernel instantiations that must launch;
every GPU row asserts that set under torch.profiler and compares indices exactly, and values bit for bit, with a
reference computed in numpy from the same keys the kernels use.  Every row also checks, from its own input, the
branch-deciding facts it relies on (lengths against 8192, masked-in count against k, population of the k-th key's
22-bit bin against 4096), so that a row cannot drift onto another branch and keep its name.  The CPU tests at the
bottom list the top-k instantiations of the built library (a kernel without a row fails on any machine) and check
the argument errors that return before anything is launched.
"""
import ctypes
from collections import namedtuple

import numpy as np
import pytest

from kernel_inventory import built_kernels, launched_kernels, library_kernels

SMALL_MAX = 8192          # kSmallMax: longer segments go through the digit passes (or the sieve)
BITONIC_MAX = 4096        # kBitonicMax: larger k runs the non-tail passes
BND_CAP = 4096            # kBndCap: boundary-bin keys kept after two digit passes
MAX_SEG = 64              # kMaxSeg: segments per batch
MAX_SEG_LEN = 0xFFFF0000  # longest segment the C ABI accepts
EINVAL, ENOMEM = -1, -3
FLT_MAX = np.finfo(np.float32).max


# ------------------------------------------------------------------------------------------------ keys and reference
def okey(s):
    """The kernels' order-preserving key of fp32 scores: every NaN -> 0xFFFFFFFF, -0.0 -> the key of +0.0."""
    s = np.asarray(s, np.float32)
    with np.errstate(invalid="ignore"):
        u = (s + np.float32(0)).view(np.uint32)
    k = np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)
    k[np.isnan(s)] = 0xFFFFFFFF
    k[k == 0] = 1
    return k


def okey_inv(k):
    k = np.asarray(k, np.uint32)
    return np.where(k & np.uint32(0x80000000), k ^ np.uint32(0x80000000), ~k).astype(np.uint32)


def keys64(sc, li):
    """(okey(score) << 32) | ~logical_index: unique, and descending key = descending score, ties -> lower index."""
    return (okey(sc[li]).astype(np.uint64) << np.uint64(32)) | (~li.astype(np.uint32)).astype(np.uint64)


def seg_stats(sc, mask, k):
    """(masked-in count, population of the 22-bit bin that holds the min(k, count)-th largest key)."""
    li = np.arange(sc.size) if mask is None else np.flatnonzero(mask)
    eff = li.size
    n = min(k, eff)
    if n == 0:
        return eff, 0
    key = keys64(sc, li)
    kth = np.partition(key, eff - n)[eff - n]
    return eff, int(np.count_nonzero((okey(sc[li]) >> np.uint32(10)) == (kth >> np.uint64(42))))


def expect_segment(oracle, sc, mask, k, small_idx):
    """(indices, value bits, count, sorted flag) the kernels must return for one segment."""
    li = np.arange(sc.size) if mask is None else np.flatnonzero(mask)
    eff = li.size
    n = min(k, eff)
    want = li[np.argsort(keys64(sc, li))[::-1][:n]]
    s = sc[li]
    if oracle is not None and eff and not (np.isnan(s).any() or (np.signbit(s) & (s == 0)).any()):
        assert np.array_equal(li[oracle.topk(s, k)], want), "the oracle's top-k and the key order disagree"
    by_index = small_idx and eff <= k
    if by_index:
        want = li
    return want, okey_inv(okey(sc[want])), n, int(not by_index)


# ------------------------------------------------------------------------------------------------ inputs
Seg = namedtuple("Seg", "x adhw mask")   # x: memory order ([A, D, H, W] when adhw); mask: uint8 by LOGICAL index


def logical(sg):
    return sg.x.transpose(2, 3, 1, 0).reshape(-1) if sg.adhw else sg.x.reshape(-1)


def normal(g, n, scale=2.0):
    return (scale * g.standard_normal(n)).astype(np.float32)


def specials(g, n):
    """Negative bulk (<= -1) with planted NaNs of both signs and several payloads, +-inf, +-FLT_MAX, -0.0 next to
    +0.0 in both orders, and subnormals: everything but -inf / -FLT_MAX ranks above the bulk."""
    x = (-1.0 - np.abs(g.standard_normal(n))).astype(np.float32)
    bits = [0x7FC00000, 0xFFC00000, 0x7F800001, 0xFFFFFFFF, 0x7FFFFFFF, 0xFF800123,       # NaNs
            0x7F800000, 0xFF800000, 0x7F7FFFFF, 0xFF7FFFFF, 0x7F7FFFFF,                     # +inf -inf FLT_MAX -FLT_MAX
            0x80000000, 0x00000000, 0x00000000, 0x80000000,                                 # -0 +0, +0 -0
            0x00000001, 0x80000001, 0x007FFFFF, 0x807FFFFF, 0x00000002, 0x00000001]         # subnormals
    pos = np.sort(g.choice(n, len(bits), replace=False))
    x[pos] = np.array(bits, np.uint32).view(np.float32)
    return x


def const(n, v):
    return np.full(n, v, np.float32)


def three(g, n):
    return g.choice(np.array([0.25, 0.5, 0.75], np.float32), n)


def bins(g, n, above, inbin):
    """`above` scores above the 22-bit bin of 1.0, `inbin` scores inside it (1.0 + j ulp, j < 1024: many exact ties),
    the rest below it."""
    x = g.uniform(-5.0, 0.99, n).astype(np.float32)
    pos = g.permutation(n)[:above + inbin]
    x[pos[:above]] = 2.0 + 100.0 * g.random(above)
    x[pos[above:]] = (np.uint32(0x3F800000) + g.integers(0, 1024, inbin).astype(np.uint32)).view(np.float32)
    return x


def logits(g, shape, scale=2.0):
    return (scale * g.standard_normal(shape)).astype(np.float32)


def saturated(g, shape, n_one):
    """Logits whose sigmoid is exactly 1.0 (n_one of them), exactly 0.0, +-inf and NaN, over a normal bulk."""
    x = logits(g, shape).reshape(-1)
    pos = g.permutation(x.size)
    x[pos[:n_one]] = g.uniform(17.0, 60.0, n_one)
    nz = min(200, (x.size - n_one) // 4)
    x[pos[n_one:n_one + nz]] = g.uniform(-200.0, -104.0, nz)
    x[pos[n_one + nz:n_one + nz + 3]] = [np.inf, -np.inf, np.nan]
    x[pos[n_one + nz + 3:n_one + nz + 6]] = np.array([0xFFC00000, 0x7F800001, 0x7FC00000], np.uint32).view(np.float32)
    return x.reshape(shape)


def keep(g, n, cnt):
    m = np.zeros(n, np.uint8)
    m[g.choice(n, cnt, replace=False)] = 1
    return m


def flat(x, mask=None):
    return Seg(np.asarray(x, np.float32), False, mask)


def amap(x, mask=None):
    assert x.ndim == 4
    return Seg(np.asarray(x, np.float32), True, mask)


def edges(g, k, special=()):
    """Segments of length 0, 1, k, 8192, 8193, 32768 and 32769 (those listed in `special` get planted specials)."""
    return [flat(specials(g, n) if n in special else normal(g, n)) for n in (0, 1, k, 8192, 8193, 32768, 32769)]


def masked_set(g, k, idx_maps=False):
    """Long segments whose masked-in count is > k, == k, < k and 0, plus one unmasked small segment."""
    if idx_maps:
        shapes = [(3, 9, 33, 31), (1, 20, 40, 41), (3, 8, 32, 33), (1, 10, 30, 31)]
        maps = [logits(g, s) for s in shapes]
        cnts = [min(3 * k, maps[0].size - 1), k, k // 2, 0]
        return [amap(m, keep(g, m.size, c)) for m, c in zip(maps, cnts)] + [amap(logits(g, (1, 2, 5, 9)))]
    segs = [flat(normal(g, 8 * k), keep(g, 8 * k, 2 * k)), flat(normal(g, 5 * k), keep(g, 5 * k, k)),
            flat(specials(g, 6 * k), keep(g, 6 * k, k // 2)), flat(normal(g, 9000), keep(g, 9000, 0))]
    return segs + [flat(normal(g, 5000))]


MASK_CLAIMS = {0: ("long", "eff>k"), 1: ("long", "eff=k"), 2: ("long", "eff<k"), 3: ("long", "eff=0")}


def many(g, nseg, long_len, masks=False):
    """nseg mixed segments (empty, short, at 8192, long); every batch of 64 holds long ones; masks on some."""
    lens = [(0, 1, 300, 8192, long_len, 3000, long_len + 3001, 2000)[i % 8] for i in range(nseg)]
    lens[-1] = long_len + 7
    segs = []
    for i, n in enumerate(lens):
        m = keep(g, n, n // (2 + i % 3)) if masks and (i % 3 == 0 or i == nseg - 1) and n else None
        segs.append(flat(normal(g, n), m))
    return segs


# ------------------------------------------------------------------------------------------------ the map
def K(name, s=None):
    return "topk_%s_kernel" % name + ("" if s is None else "<%s>" % ("true" if s else "false"))


TAIL_FAMILIES = ("small", "sieve", "digit_keys", "digit_nokeys")


def family_kernels(family, s, report):
    ks = {
        "small": [K("tail", s)],
        "sieve": [K("sample"), K("sieve", s), K("first", s), K("second"), K("split_keys"), K("tail", s)],
        "digit_keys": [K("init"), K("first", s), K("second"), K("split_keys"), K("tail", s)],
        "digit_nokeys": [K("init"), K("first", s), K("hist", s), K("split", s), K("tail", s)],
        "nontail_keys": [K("init"), K("first", s), K("second"), K("split_keys"), K("after_split"), K("hist", s),
                         K("collect", s), K("sort")],
        "nontail_nokeys": [K("init"), K("first", s), K("hist", s), K("split", s), K("after_split"), K("collect", s),
                           K("sort")],
        "nontail_empty": [K("init"), K("sort")],
    }[family]
    if report and family not in TAIL_FAMILIES:
        ks.append(K("report"))
    return set(ks)


Row = namedtuple("Row", "tag family sigmoid k make ws tune small_idx report misalign claims")


def row(tag, family, sigmoid, k, make, ws="keys", tune=0, small_idx=False, report=False, misalign=False, claims=None):
    """family: the path (family_kernels); make(rng) -> [Seg]; ws: workspace size -- "keys" (roi3d_topk_workspace_
    bytes_keys: key buffer), "keys-1" (one byte less: none) or "base" (roi3d_topk_workspace_bytes: none); tune:
    roi3d_set_tuning key 11 (0 sieve where it applies, 2 the sieve gives up, -1 digit passes only); misalign: segment s
    starts 1 + s % 3 floats past a 16-byte boundary; claims: {segment: facts its input must satisfy}."""
    return Row(tag, family, sigmoid, k, make, ws, tune, small_idx, report, misalign, claims or {})


BND = {0: ("long", "pop=4096"), 1: ("long", "pop=4097"), 2: ("long", "pop>4096"), 3: ("long", "pop>4096")}


def bnd_set(g, k, above):
    return [flat(bins(g, 30000, above, 4096)), flat(bins(g, 30000, above, 4097)), flat(const(50000, -3.0)),
            flat(three(g, 60000))]


COVERAGE = [
    # ---- tail kernel alone: every segment <= 8192
    row("small-edges-specials", "small", False, 4096,
        lambda g: [flat(normal(g, 0)), flat(normal(g, 1)), flat(specials(g, 4096)), flat(specials(g, 8192)),
                   flat(normal(g, 300)), flat(const(5000, 0.5))], misalign=True, report=True),
    row("small-k1", "small", False, 1,
        lambda g: [flat(normal(g, 1)), flat(specials(g, 8192)), flat(normal(g, 5)), flat(normal(g, 0))]),
    row("small-sigmoid-A3-A1-index-order", "small", True, 200,
        lambda g: [amap(saturated(g, (3, 2, 5, 7), 40)), amap(logits(g, (1, 2, 5, 9))),
                   amap(saturated(g, (3, 3, 9, 11), 300))], small_idx=True, report=True),
    row("small-masked-index-order", "small", False, 300,
        lambda g: [flat(specials(g, 2000), keep(g, 2000, 500)), flat(normal(g, 1000), keep(g, 1000, 300)),
                   flat(normal(g, 8192), keep(g, 8192, 100)), flat(normal(g, 50), keep(g, 50, 0))],
        small_idx=True, report=True, claims={0: ("eff>k",), 1: ("eff=k",), 2: ("eff<k",), 3: ("eff=0",)}),
    row("small-masked-sigmoid", "small", True, 300,
        lambda g: [amap(saturated(g, (3, 4, 10, 9), 100), keep(g, 1080, 700)),
                   amap(logits(g, (1, 4, 10, 9)), keep(g, 360, 300))], report=True,
        claims={0: ("eff>k",), 1: ("eff=k",)}),
    # ---- sieve: long segments, no mask, key buffer
    row("sieve-raw", "sieve", False, 2000,
        lambda g: [flat(normal(g, n)) for n in (8193, 32768, 32769, 150001, 5000, 0)], misalign=True, report=True),
    row("sieve-raw-specials", "sieve", False, 4096,
        lambda g: [flat(specials(g, 40000)), flat(specials(g, 8193)), flat(normal(g, 100000))]),
    row("sieve-sigmoid-A3-A1", "sieve", True, 2000,
        lambda g: [amap(logits(g, (3, 9, 33, 31))), amap(logits(g, (1, 20, 40, 41))), amap(logits(g, (1, 2, 5, 9)))],
        misalign=True),
    row("sieve-sigmoid-saturated", "sieve", True, 2000,
        lambda g: [amap(saturated(g, (3, 10, 30, 31), 6000)), amap(logits(g, (1, 16, 32, 33)))],
        claims={0: ("long", "pop>4096")}),
    row("sieve-boundary-bin", "sieve", False, 3000, lambda g: bnd_set(g, 3000, 1000), claims=BND),
    # ---- the sieve gives up on every long segment (key 11 = 2): must equal the digit passes bit for bit
    row("sieve-gives-up-raw", "sieve", False, 2000,
        lambda g: [flat(normal(g, 32769)), flat(specials(g, 50000)), flat(normal(g, 8193)), flat(normal(g, 3000))],
        tune=2, misalign=True, report=True),
    row("sieve-gives-up-sigmoid", "sieve", True, 4096,
        lambda g: [amap(saturated(g, (3, 8, 32, 33), 3000)), amap(logits(g, (1, 20, 40, 41)))], tune=2),
    row("sieve-gives-up-boundary-k1", "sieve", False, 1,
        lambda g: [flat(const(20000, 0.25)), flat(bins(g, 20000, 0, 4097))], tune=2,
        claims={0: ("long", "pop>4096"), 1: ("long", "pop=4097")}),
    # ---- digit passes over the key buffer (key 11 = -1, or masks)
    row("digit-keys-edges", "digit_keys", False, 4096, lambda g: edges(g, 4096, special=(8193, 32769)), tune=-1,
        misalign=True, report=True),
    row("digit-keys-k1", "digit_keys", False, 1,
        lambda g: [flat(specials(g, 8193)), flat(normal(g, 32768)), flat(normal(g, 5))], tune=-1),
    row("digit-keys-sigmoid", "digit_keys", True, 2000,
        lambda g: [amap(logits(g, (3, 9, 33, 31))), amap(saturated(g, (1, 10, 40, 41), 5000))], tune=-1,
        claims={1: ("long", "pop>4096")}),
    row("digit-keys-boundary-bin", "digit_keys", False, 3000, lambda g: bnd_set(g, 3000, 1000), tune=-1, claims=BND),
    row("digit-keys-masked", "digit_keys", False, 2000, lambda g: masked_set(g, 2000), report=True,
        claims=MASK_CLAIMS),
    row("digit-keys-masked-index-order-sigmoid", "digit_keys", True, 2000, lambda g: masked_set(g, 2000, True),
        small_idx=True, report=True, claims=MASK_CLAIMS),
    # ---- digit passes over the raw scores (no key buffer)
    row("digit-nokeys-raw-base", "digit_nokeys", False, 2000,
        lambda g: [flat(normal(g, 8193)), flat(normal(g, 32768)), flat(specials(g, 70001)), flat(normal(g, 300))],
        ws="base", misalign=True, report=True),
    row("digit-nokeys-edges-keys-1", "digit_nokeys", False, 4096, lambda g: edges(g, 4096, special=(32768,)),
        ws="keys-1"),
    row("digit-nokeys-sigmoid-keys-1", "digit_nokeys", True, 2000,
        lambda g: [amap(logits(g, (3, 9, 33, 31))), amap(logits(g, (1, 20, 40, 41)))], ws="keys-1", misalign=True),
    row("digit-nokeys-boundary-bin", "digit_nokeys", False, 3000, lambda g: bnd_set(g, 3000, 1000), ws="base",
        claims=BND),
    row("digit-nokeys-saturated", "digit_nokeys", True, 2000, lambda g: [amap(saturated(g, (3, 10, 30, 31), 6000))],
        ws="base", claims={0: ("long", "pop>4096")}),
    row("digit-nokeys-masked-index-order", "digit_nokeys", False, 2000, lambda g: masked_set(g, 2000), ws="base",
        small_idx=True, report=True, claims=MASK_CLAIMS),
    row("digit-nokeys-k1", "digit_nokeys", False, 1, lambda g: [flat(specials(g, 20000)), flat(normal(g, 8193))],
        ws="base"),
    # ---- k > 4096 over the key buffer
    row("nontail-keys-edges", "nontail_keys", False, 4097, lambda g: edges(g, 4097, special=(8193, 32769)),
        misalign=True, report=True),
    row("nontail-keys-raw", "nontail_keys", False, 5000,
        lambda g: [flat(normal(g, 100000)), flat(specials(g, 50000))]),
    row("nontail-keys-sigmoid", "nontail_keys", True, 5000,
        lambda g: [amap(logits(g, (3, 12, 40, 41))), amap(saturated(g, (1, 20, 40, 41), 8000)),
                   amap(logits(g, (1, 2, 5, 9)))], report=True, claims={1: ("long", "pop>4096")}),
    row("nontail-keys-boundary-bin", "nontail_keys", False, 5000, lambda g: bnd_set(g, 5000, 3000), claims=BND),
    row("nontail-keys-masked", "nontail_keys", False, 5000, lambda g: masked_set(g, 5000), report=True,
        claims=MASK_CLAIMS),
    row("nontail-keys-masked-index-order-sigmoid", "nontail_keys", True, 4097, lambda g: masked_set(g, 4097, True),
        small_idx=True, report=True, claims=MASK_CLAIMS),
    # ---- k > 4096 over the raw scores
    row("nontail-nokeys-edges", "nontail_nokeys", False, 4097, lambda g: edges(g, 4097, special=(4097, 32768)),
        ws="base", misalign=True, report=True),
    row("nontail-nokeys-sigmoid-keys-1", "nontail_nokeys", True, 5000,
        lambda g: [amap(logits(g, (3, 12, 40, 41))), amap(saturated(g, (1, 20, 40, 41), 8000))], ws="keys-1",
        report=True, claims={1: ("long", "pop>4096")}),
    row("nontail-nokeys-boundary-bin", "nontail_nokeys", False, 5000, lambda g: bnd_set(g, 5000, 3000), ws="base",
        claims=BND),
    row("nontail-nokeys-masked-index-order", "nontail_nokeys", False, 5000, lambda g: masked_set(g, 5000),
        ws="base", small_idx=True, report=True, claims=MASK_CLAIMS),
    row("nontail-nokeys-specials", "nontail_nokeys", False, 4097, lambda g: [flat(specials(g, 20000))], ws="base"),
    row("nontail-all-empty", "nontail_empty", False, 5000, lambda g: [flat(normal(g, 0))] * 3, report=True),
    # ---- more than 64 segments: several batches, per-batch output offsets, key-buffer offsets restart
    row("65-segments-sieve", "sieve", False, 2000, lambda g: many(g, 65, 9000), misalign=True, report=True),
    row("130-segments-masked-index-order", "digit_keys", False, 2000, lambda g: many(g, 130, 9000, masks=True),
        small_idx=True, report=True),
    row("65-segments-nontail-nokeys", "nontail_nokeys", False, 4097, lambda g: many(g, 65, 9000), ws="base",
        misalign=True, report=True),
    row("130-segments-nontail-keys-sigmoid-masked", "nontail_keys", True, 4097,
        lambda g: many(g, 130, 9000, masks=True), small_idx=True, report=True),
]


# ------------------------------------------------------------------------------------------------ preconditions
def _holds(claim, n, eff, pop, k):
    return {"long": n > SMALL_MAX, "eff>k": eff > k, "eff=k": eff == k, "eff<k": 0 < eff < k, "eff=0": eff == 0,
            "pop>4096": pop > BND_CAP, "pop=4096": pop == BND_CAP, "pop=4097": pop == BND_CAP + 1}[claim]


def check_row_preconditions(r, segs, scores):
    """The row's input takes the branches its family and claims name (scores: logical, as ranked)."""
    lens = [sg.x.size for sg in segs]
    keys = r.ws == "keys" and sum(lens) > 0
    assert (r.k <= BITONIC_MAX) == (r.family in TAIL_FAMILIES)
    for b in range(0, len(segs), MAX_SEG):
        bl, bm = lens[b:b + MAX_SEG], [sg.mask is not None for sg in segs[b:b + MAX_SEG]]
        if r.family == "small":
            assert max(bl) <= SMALL_MAX
        elif r.family in TAIL_FAMILIES:
            assert max(bl) > SMALL_MAX, "batch %d has no long segment" % (b // MAX_SEG)
        elif r.family == "nontail_empty":
            assert max(bl) == 0
        else:
            assert max(bl) > 0
        if r.family == "sieve":
            assert keys and not any(bm) and r.tune in (0, 2)
        if r.family == "digit_keys":
            assert keys and (r.tune == -1 or any(bm)), "the sieve would take batch %d" % (b // MAX_SEG)
    if r.family in ("digit_nokeys", "nontail_nokeys"):
        assert not keys
    if r.family == "nontail_keys":
        assert keys
    if r.ws == "keys-1":
        assert sum(lens) > 0
    for s, claims in r.claims.items():
        eff, pop = seg_stats(scores[s], segs[s].mask, r.k)
        for c in claims:
            assert _holds(c, lens[s], eff, pop, r.k), (r.tag, s, c, lens[s], eff, pop)


def _seed(tag):
    return sum((i + 1) * ord(c) for i, c in enumerate(tag)) % 100003


def _np_sigmoid(x):
    with np.errstate(over="ignore", invalid="ignore"):
        return (1.0 / (1.0 + np.exp(-x.astype(np.float64)))).astype(np.float32)


# ------------------------------------------------------------------------------------------------ GPU runner
@pytest.fixture(scope="module")
def dev():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


Placed = namedtuple("Placed", "buf offs lens adhw masks")
WS_FILL = 0xAB
Result = namedtuple("Result", "idx val cnt srt")   # val: uint32 bit patterns


def place(dev, segs, misalign):
    """All segments in one device buffer; misalign: segment s starts 1 + s % 3 floats past a 16-byte boundary."""
    import torch
    offs, cur = [], 0
    for i, sg in enumerate(segs):
        cur = -(-cur // 4) * 4 + ((1 + i % 3) if misalign else 0)
        offs.append(cur)
        cur += sg.x.size
    host = np.zeros(cur + 4, np.float32)
    for o, sg in zip(offs, segs):
        host[o:o + sg.x.size] = sg.x.reshape(-1)
    buf = torch.from_numpy(host).to(dev)
    assert buf.data_ptr() % 16 == 0
    adhw = None
    if any(sg.adhw for sg in segs):
        adhw = np.array([list(sg.x.shape) if sg.adhw else [0, 0, 0, 0] for sg in segs], np.int32)
    masks = [None if sg.mask is None else torch.from_numpy(sg.mask).to(dev) for sg in segs]
    return Placed(buf, offs, [sg.x.size for sg in segs], adhw, masks)


def call_topk(dev, p, k, sigmoid, ws="keys", small_idx=False, report=False, tune=0, profile=True, ws_probe=None):
    """roi3d_topk_segmented_masked on placed segments with a workspace of the chosen size.  Returns (Result, names of
    the launched kernels or None).  ws_probe: called after the call with (the workspace as bytes, its base size); the
    workspace is filled with WS_FILL before the call."""
    import torch
    import roi3d_b200
    from roi3d_b200._util import stream_ptr
    lib = roi3d_b200._lib.lib
    nseg = len(p.lens)
    off_a, len_a = np.asarray(p.offs, np.int64), np.asarray(p.lens, np.int64)
    base = lib.roi3d_topk_workspace_bytes(nseg, k)
    full = lib.roi3d_topk_workspace_bytes_keys(nseg, k, int(len_a.sum()))
    nbytes = {"base": base, "keys-1": full - 1, "keys": full}[ws]
    assert nbytes >= base
    wbuf = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
    wptr = wbuf.data_ptr() + (-wbuf.data_ptr()) % 256
    if ws_probe is not None:
        wbuf.fill_(WS_FILL)
    idx = torch.full((nseg, k), -77, dtype=torch.int64, device=dev)
    val = torch.full((nseg, k), float("nan"), device=dev)
    cnt = torch.full((nseg,), -77, dtype=torch.int32, device=dev) if report else None
    srt = torch.full((nseg,), 77, dtype=torch.uint8, device=dev) if report else None
    mask_p = None
    if any(m is not None for m in p.masks or []):
        mask_p = (ctypes.c_void_p * nseg)(*[None if m is None else m.data_ptr() for m in p.masks])
    adhw_p = p.adhw.ctypes.data if p.adhw is not None else None

    def fn():
        roi3d_b200._lib.check(lib.roi3d_topk_segmented_masked(
            p.buf.data_ptr(), off_a.ctypes.data, len_a.ctypes.data, adhw_p, mask_p, nseg, k, int(sigmoid),
            int(small_idx), idx.data_ptr(), val.data_ptr(), None if cnt is None else cnt.data_ptr(),
            None if srt is None else srt.data_ptr(), wptr, nbytes, stream_ptr()))
    roi3d_b200._lib.set_tuning(11, tune)
    try:
        names = launched_kernels(fn) if profile else fn()
        torch.cuda.synchronize()
    finally:
        roi3d_b200._lib.set_tuning(11, 0)
    if ws_probe is not None:
        w0 = wptr - wbuf.data_ptr()
        ws_probe(wbuf[w0:w0 + nbytes], base)
    del wbuf
    return Result(idx.cpu().numpy(), val.cpu().numpy().view(np.uint32),
                  None if cnt is None else cnt.cpu().numpy(), None if srt is None else srt.cpu().numpy()), names


def call_topk_segmented(dev, p, segs, r):
    """The same segments through the Python wrapper (views of the same buffer, so the same alignment)."""
    import roi3d_b200
    from roi3d_b200.models.anchor_heads import topk_segmented
    views = [p.buf[o:o + n].view(sg.x.shape) for o, n, sg in zip(p.offs, p.lens, segs)]
    roi3d_b200._lib.set_tuning(11, r.tune)
    try:
        out = topk_segmented(views, r.k, apply_sigmoid=r.sigmoid, permute_adhw=segs[0].adhw,
                             small_in_index_order=r.small_idx, masks=p.masks, report=r.report)
    finally:
        roi3d_b200._lib.set_tuning(11, 0)
    idx, val = out[0].cpu().numpy(), out[1].cpu().numpy().view(np.uint32)
    return Result(idx, val, out[2].cpu().numpy() if r.report else None, out[3].cpu().numpy() if r.report else None)


def gpu_scores(dev, sg, sigmoid):
    """Logical scores as the kernels rank them; sigmoid rows use torch's CUDA sigmoid (device expf can differ from
    the host's in the last bit)."""
    import torch
    x = np.ascontiguousarray(logical(sg))
    return torch.from_numpy(x).to(dev).sigmoid().cpu().numpy() if sigmoid else x


def check_result(oracle, got, segs, scores, k, small_idx, report, what=""):
    for s, (sg, sc) in enumerate(zip(segs, scores)):
        want, bits, n, srt = expect_segment(oracle, sc, sg.mask, k, small_idx)
        m = len(want)
        assert np.array_equal(got.idx[s, :m], want), "%s segment %d: indices" % (what, s)
        assert np.array_equal(got.val[s, :m], bits), "%s segment %d: values" % (what, s)
        assert (got.idx[s, m:] == -1).all() and (got.val[s, m:] == 0).all(), "%s segment %d: padding" % (what, s)
        if report:
            assert got.cnt[s] == n and got.srt[s] == srt, "%s segment %d: report" % (what, s)


def _same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b) if x is not None)


@pytest.mark.gpu
@pytest.mark.parametrize("r", COVERAGE, ids=lambda r: r.tag)
def test_topk_path_row(oracle, dev, r):
    segs = r.make(np.random.default_rng(_seed(r.tag)))
    scores = [gpu_scores(dev, sg, r.sigmoid) for sg in segs]
    check_row_preconditions(r, segs, scores)
    p = place(dev, segs, r.misalign)
    got, names = call_topk(dev, p, r.k, r.sigmoid, r.ws, r.small_idx, r.report, r.tune)
    assert library_kernels(names) == family_kernels(r.family, r.sigmoid, r.report), sorted(library_kernels(names))
    check_result(oracle, got, segs, scores, r.k, r.small_idx, r.report)
    if r.tune == 2:   # the sieve's fallback returns what the digit passes alone return, bit for bit
        digits, _ = call_topk(dev, p, r.k, r.sigmoid, r.ws, r.small_idx, r.report, -1, profile=False)
        assert _same(got, digits)
    if r.ws == "keys" and len({sg.adhw for sg in segs}) == 1:   # what the production wrapper passes
        assert _same(got, call_topk_segmented(dev, p, segs, r))


@pytest.mark.gpu
def test_topk_k4096_and_k4097_agree(oracle, dev):
    """The same segments through the tail path (k = 4096) and the non-tail path (k = 4097) agree on their common
    rows."""
    g = np.random.default_rng(4097)
    segs = [flat(normal(g, 0)), flat(normal(g, 1)), flat(specials(g, 4096)), flat(normal(g, 4097)),
            flat(specials(g, 8192)), flat(normal(g, 8193)), flat(normal(g, 32768)), flat(specials(g, 32769))]
    scores = [logical(sg) for sg in segs]
    p = place(dev, segs, False)
    a, na = call_topk(dev, p, 4096, False)
    b, nb = call_topk(dev, p, 4097, False, report=True)
    assert library_kernels(na) == family_kernels("sieve", False, False)
    assert library_kernels(nb) == family_kernels("nontail_keys", False, True)
    check_result(oracle, a, segs, scores, 4096, False, False, "k=4096")
    check_result(oracle, b, segs, scores, 4097, False, True, "k=4097")
    assert np.array_equal(a.idx, b.idx[:, :4096]) and np.array_equal(a.val, b.val[:, :4096])


def sieve_sample_positions(n):
    """Positions topk_sample_kernel reads in a segment of n > 32768 scores: one per stride, jittered by its hash."""
    S = 32768
    step = n // S
    i = np.arange(S, dtype=np.uint64)
    h = i ^ (i >> np.uint64(16))
    h = (h * np.uint64(0x7feb352d)) & np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(15)
    h = (h * np.uint64(0x846ca68b)) & np.uint64(0xFFFFFFFF)
    h ^= h >> np.uint64(16)
    return i * np.uint64(step) + h % np.uint64(step)


@pytest.mark.gpu
@pytest.mark.parametrize("bulk", ["proven", "constant"])
def test_topk_segment_past_2_31(dev, bulk):
    """One segment of 2^31 + 4099 scores (8.6 GB, plus 8.6 GB of keys) with maxima planted on both sides of index
    2^31, ties included; the answer follows from the planted values alone.
    "proven": the bulk lies in [-1, 0) and k = the planted count.  The smallest planted value, 1.0, sits at one of the
    positions the sieve samples and is the sample's largest score, so the threshold is 1.0: exactly k scores pass it,
    the list proves itself, and the digit passes never write the key buffer.
    "constant": the bulk is -1.0, so more than 2^31 elements pass the sieve's threshold (the list overflows, the sieve
    gives up) and share the k-th key's bin (the boundary buffer overflows, the tail's full-data passes decide); the
    rest of k = 4096 are the bulk's lowest indices, and the digit passes write the key buffer."""
    import torch
    n = 2 ** 31 + 4099
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < 24 * 2 ** 30:
        pytest.skip("needs 24 GB of free device memory for 17.2 GB of scores and keys; %.1f GB free" % (free / 2 ** 30))
    planted = {2 ** 31 + 2: np.inf, 2 ** 31: 7.0, 2 ** 31 + 1: 7.0, 17: 5.0, n - 1: 5.0, 2 ** 31 - 1: 3.0,
               2 ** 31 + 5: 3.0, 3: 2.0, 2 ** 31 + 4000: 2.0, 2 ** 31 + 4001: 2.5}
    if bulk == "proven":
        sampled = sieve_sample_positions(n)
        p0 = int(sampled[100])
        planted[p0] = 1.0
        planted[2 ** 31 + 7] = 1.0                              # ties with p0, which comes first
        assert set(planted) & set(sampled.tolist()) == {p0}
    order = sorted(planted, key=lambda i: (-planted[i], i))
    if bulk == "proven":
        k = len(planted)
        want = order
    else:
        k = 4096
        rest = [i for i in range(k + len(planted)) if i not in planted]
        want = order + rest[:k - len(planted)]
    keybuf = []

    def probe(ws, base):
        """Whether the first and the last 16 MB of the key buffer were written."""
        kb = ws[base:base + 4 * n]
        keybuf.append([bool((part != WS_FILL).any()) for part in (kb[:1 << 24], kb[-(1 << 24):])])

    try:
        buf = torch.empty(n + 4, dtype=torch.float32, device=dev)
        if bulk == "proven":
            buf.uniform_(-1.0, 0.0)
            buf.clamp_(max=-1e-30)                              # strictly below the threshold
        else:
            buf.fill_(-1.0)
        pos = torch.tensor(list(planted), dtype=torch.int64, device=dev)
        buf[pos] = torch.tensor([planted[i] for i in planted], dtype=torch.float32, device=dev)
        got, names = call_topk(dev, Placed(buf, [0], [n], None, [None]), k, False, "keys", report=True,
                               ws_probe=probe)
        assert library_kernels(names) == family_kernels("sieve", False, False)
        assert np.array_equal(got.idx[0], np.array(want, np.int64))
        vals = buf[torch.tensor(want, dtype=torch.int64, device=dev)].cpu().numpy()
        assert np.array_equal(got.val[0], vals.view(np.uint32))
        assert got.cnt[0] == k and got.srt[0] == 1
        # the proven sieve leaves the key buffer alone; the digit passes write all of it
        assert keybuf == [[bulk == "constant"] * 2], keybuf
    finally:
        buf = None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ end to end
def _e2e(oracle, dev, dims, nms_pre, keep_frac, seed):
    import torch
    from roi3d_b200 import RPNProposal3D
    from test_gpu_parity import _rpn_inputs
    strides, dstrides = [4, 8], [2, 4]
    cls, reg = _rpn_inputs(1, dims, seed)
    img = (dims[0][1] * 4, dims[0][2] * 4, 3, dims[0][0] * 2)
    cfg = dict(nms_pre=nms_pre, nms_post=1000, max_num=1000, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=strides,
                         anchor_strides_depth=dstrides)
    kw = {}
    if keep_frac:
        rng = np.random.default_rng(seed + 1)
        masks = [(rng.random(int(np.prod(d))) < keep_frac).astype(np.uint8) for d in dims]
        head.pos_indices = [torch.from_numpy(m).to(dev) for m in masks]
        kw["pos_indices"] = masks
    cls_t = [torch.from_numpy(c).to(dev) for c in cls]
    res = []
    names = launched_kernels(lambda: res.append(head.get_proposals(cls_t, [torch.from_numpy(r).to(dev) for r in reg],
                                                                   [dict(img_shape=img, scale_factor=1.0)], cfg)))
    anchors = [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
               for d, s, ds in zip(dims, strides, dstrides)]
    scores = [c[0].permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy() for c in cls_t]
    want = oracle.get_bboxes_single([c[0] for c in cls], [r[0] for r in reg], anchors, img, nms_pre, 1000, 1000, 0.7,
                                    scores=scores, **kw)
    got = res[0][0].cpu().numpy()
    assert got.shape == want.shape and np.abs(got - want).max() <= 1e-3
    return library_kernels(names)


@pytest.mark.gpu
def test_rpn_nms_pre_0_runs_the_non_tail_top_k(oracle, dev):
    """nms_pre = 0: k = the largest level (4608 anchors > 4096), every level comes back whole in anchor order through
    the non-tail passes."""
    ks = _e2e(oracle, dev, [(8, 24, 24), (4, 12, 12)], 0, None, 61)
    assert {K("collect", True), K("sort")} <= ks, sorted(ks)


@pytest.mark.gpu
def test_rpn_masked_level_past_8192_anchors(oracle, dev):
    """nms_pre = 5000 with pos_indices on a 10240-anchor level (about 6100 masked in): the masked non-tail top-k with
    its device-side report; the 1280-anchor level stays unmasked and unsorted."""
    ks = _e2e(oracle, dev, [(8, 32, 40), (4, 16, 20)], 5000, 0.6, 62)
    assert {K("collect", True), K("sort"), K("report")} <= ks, sorted(ks)


# ------------------------------------------------------------------------------------------------ CPU checks
def test_every_topk_kernel_has_a_coverage_row():
    """The top-k instantiations in the built library are exactly the union of the COVERAGE rows' kernel sets: a
    kernel added without a row fails this test on any machine."""
    built = built_kernels("topk_")
    covered = set().union(*(family_kernels(r.family, r.sigmoid, r.report) for r in COVERAGE))
    assert built == covered, "built, no row: %s; row, not built: %s" % (sorted(built - covered), sorted(covered - built))
    assert len(built) == 19


def test_coverage_rows_are_well_formed():
    tags = [r.tag for r in COVERAGE]
    assert len(tags) == len(set(tags))
    for r in COVERAGE:
        assert r.ws in ("keys", "keys-1", "base") and r.tune in (-1, 0, 2)
        assert r.tune == 0 or r.family in TAIL_FAMILIES
        segs = r.make(np.random.default_rng(_seed(r.tag)))
        scores = [_np_sigmoid(logical(sg)) if r.sigmoid else logical(sg) for sg in segs]
        for sg in segs:
            assert sg.mask is None or sg.mask.shape == (sg.x.size,)
        check_row_preconditions(r, segs, scores)


def test_reference_keys_follow_the_value_rule():
    """The reference's keys: NaN of either sign above +inf, -0.0 equal to +0.0, values mapped back as documented."""
    x = np.array([0xFFC00000, 0x7F800000, 0x80000000, 0x00000000, 0x00000001, 0x7FC00001, 0xFF7FFFFF],
                 np.uint32).view(np.float32)
    k = okey(x)
    assert k[0] == k[5] == 0xFFFFFFFF and k[1] < k[0] and k[2] == k[3] and k[4] > k[3] and k[6] > 0
    assert list(okey_inv(k)) == [0x7FFFFFFF, 0x7F800000, 0, 0, 1, 0x7FFFFFFF, 0xFF7FFFFF]
    got, bits, n, srt = expect_segment(None, x, None, 7, False)
    assert list(got) == [0, 5, 1, 4, 2, 3, 6] and n == 7 and srt == 1


def _call_fake(lens, adhw=None, k=100, ws_off=0, ws_short=0):
    """roi3d_topk_segmented_masked with placeholder device pointers: only for calls rejected before any launch.  The
    callers add a segment with a bad A*D*H*W after the one under test, so that even a missing check returns before
    anything is launched."""
    import roi3d_b200
    lib = roi3d_b200._lib.lib
    fake = 1 << 20
    nseg = len(lens)
    ln, off = np.asarray(lens, np.int64), np.zeros(nseg, np.int64)
    ad = None if adhw is None else np.asarray(adhw, np.int32)
    nbytes = lib.roi3d_topk_workspace_bytes(nseg, k) - ws_short
    rc = lib.roi3d_topk_segmented_masked(fake, off.ctypes.data, ln.ctypes.data, None if ad is None else ad.ctypes.data,
                                         None, nseg, k, 0, 0, fake, fake, None, None, fake + ws_off, nbytes, None)
    msg = lib.roi3d_last_error()
    return rc, msg.decode() if msg else ""


BAD = [1, 1, 1, 4]   # 4 != len 5


def test_topk_rejects_segments_past_the_length_bound():
    assert MAX_SEG_LEN == 0xFFFF0000
    rc, msg = _call_fake([MAX_SEG_LEN, MAX_SEG_LEN + 1, 5], [[0, 0, 0, 0], [0, 0, 0, 0], BAD])
    assert rc == EINVAL and "segment 1" in msg and "length" in msg, msg      # segment 0, at the bound, passed
    rc, msg = _call_fake([2 ** 32 - 2, 5], [[0, 0, 0, 0], BAD])              # the longest the old check accepted
    assert rc == EINVAL and "segment 0" in msg and "length" in msg, msg
    rc, msg = _call_fake([-1, 5], [[0, 0, 0, 0], BAD])
    assert rc == EINVAL and "segment 0" in msg and "length" in msg, msg


def test_topk_rejects_bad_maps_and_workspaces():
    rc, msg = _call_fake([5], [BAD])
    assert rc == EINVAL and "A*D*H*W" in msg, msg
    rc, msg = _call_fake([5], [BAD], ws_off=16)
    assert rc == EINVAL and "aligned" in msg, msg
    rc, msg = _call_fake([5], [BAD], ws_short=1)
    assert rc == ENOMEM and "workspace" in msg, msg

"""`min_bbox_size > 0` in the RPN proposal path: per (image, level), after the decode with its clamp and before that
level's NMS, a proposal is kept iff (x2 - x1) + 1 >= m and (y2 - y1) + 1 >= m in fp32 (mmdetection v0.6.0
RPNHead.get_bboxes_single; depth is not compared).  On the device this is `filter_min_size_rows7_kernel`
(`roi3d_filter_min_size_rows7`), a stable in-place compaction of the decoded rows.

The reference is `min_bbox_size_oracle` (tests/): oracle.get_bboxes_single with the filter between decode and NMS.
CPU: a literal torch transcription of the v0.6 snippet equals its `filter_min_bbox_size` bit for bit, its
get_bboxes_single at min_bbox_size = 0 equals oracle.get_bboxes_single, the ABI rejects bad arguments, and the built
library holds exactly the kernel the GPU rows name.
GPU: `RPNProposal3D.get_proposals` against `min_bbox_size_oracle.get_bboxes_single(..., min_bbox_size=m)`, bit for
bit.  The size
deltas are drawn from values whose device `expf` equals the host libm's (the oracle's decode calls libm), so the
device decode and the oracle's agree bit for bit and the proposals can be compared exactly; every case first checks,
from its own decoded rows, the fraction of rows its `m` drops.
"""
import ctypes
import ctypes.util
import functools

import numpy as np
import pytest
import torch

import min_bbox_size_oracle as mbo
from kernel_inventory import built_kernels, launched_kernels, library_kernels

EINVAL = -1
FILTER = "filter_min_size_rows7_kernel"
C4_STRIDES, C4_DSTRIDES = [4, 8, 16, 32, 64], [2, 4, 8, 16, 32]
STRIDES, DSTRIDES = C4_STRIDES[:3], C4_DSTRIDES[:3]
DIMS = [(8, 24, 24), (4, 12, 12), (2, 6, 6)]        # 4608, 576 and 72 anchors (A = 1)
IMG = (96, 96, 3, 16)
CFG = dict(nms_pre=300, nms_post=100, max_num=150, nms_thr=0.7, nms_across_levels=False)
M_SOME = 11.3        # drops some rows of every level (checked per case); not exactly representable in fp32
M_ALL = 1.0e4        # wider than every image: drops every row
C4_M = 9.5           # the C4 case here and in tools/bench_rpn_min_bbox_size.py
F32 = np.float32


def _next(x, direction):
    return np.nextafter(F32(x), F32(direction), dtype=F32)


# ------------------------------------------------------------------------------------------------ CPU
def _v06_filter(proposals, scores, min_bbox_size):
    """mmdetection v0.6.0 RPNHead.get_bboxes_single, the `cfg.min_bbox_size > 0` branch, on torch CPU tensors."""
    w = proposals[:, 2] - proposals[:, 0] + 1
    h = proposals[:, 3] - proposals[:, 1] + 1
    valid_inds = torch.nonzero((w >= min_bbox_size) & (h >= min_bbox_size)).squeeze()
    proposals = proposals[valid_inds, :]
    scores = scores[valid_inds]
    return proposals, scores


def _v06_clamp(proposals, max_shape):
    """The clamp at the end of v0.6.0's delta2bbox, applied to 3-D rows (x to W - 1, y to H - 1, z to D - 1)."""
    p = proposals.clone()
    for cols, hi in (((0, 2), max_shape[1] - 1), ((1, 3), max_shape[0] - 1), ((4, 5), max_shape[3] - 1)):
        for c in cols:
            p[:, c] = p[:, c].clamp(min=0, max=hi)
    return p


def _torch_rows(proposals, scores, m):
    """The v0.6 filter with the one-survivor case kept two-dimensional (`.squeeze()` leaves a 0-d index there)."""
    p, s = _v06_filter(torch.from_numpy(proposals), torch.from_numpy(scores), m)
    if p.dim() == 1:
        p, s = p[None], s.reshape(1)
    return np.concatenate([p.numpy(), s.numpy()[:, None]], 1)


def _boundary_rows():
    """Rows whose width or height sits exactly at 8, one ulp either side, at other small values, or is NaN / inf."""
    ws = [F32(8), _next(8, 0), _next(8, 9), F32(7), F32(9), F32(0.5), F32(1), F32(12.3), F32(11.3), _next(11.3, 0),
          _next(11.3, 12), F32(np.float32(11.3) + F32(1e-6))]
    rows = []
    for w in ws:
        for h in (F32(8), _next(8, 0), _next(8, 9), F32(20)):
            x1 = F32(3.25)
            rows.append([x1, F32(5), x1 + w - F32(1), F32(5) + h - F32(1), F32(0), F32(3)])
    nan, inf = np.nan, np.inf
    rows += [[nan, 0, 10, 10, 0, 3], [0, nan, 10, 10, 0, 3], [0, 0, nan, 10, 0, 3], [0, 0, 10, nan, 0, 3],
             [0, 0, 10, 10, nan, nan], [-inf, 0, 10, 10, 0, 3], [0, 0, inf, 10, 0, 3], [0, 0, 10, inf, 0, 3],
             [inf, 0, inf, 10, 0, 3], [0, -inf, 10, -inf, 0, 3], [0, 0, -inf, 10, 0, 3], [3, 3, 3, 3, 0, 0],
             [10, 10, 2, 2, 0, 3], [0, 0, 9, 9, 5, 2]]
    return np.asarray(rows, F32)


M_VALUES = [8, 8.0, float(_next(8, 0)), float(_next(8, 9)), 8 + 1e-7, 8 - 1e-7, 11.3, 0.1, 1 / 3, 1, 1e-45, 1e30]


def test_torch_transcription_equals_the_oracle_filter(oracle):
    """The v0.6 snippet on torch CPU tensors and the oracle's filter keep the same rows, bit for bit, for boundary,
    one-ulp, NaN and infinite coordinates and for `m` values that fp32 cannot hold exactly."""
    rows = _boundary_rows()
    rng = np.random.default_rng(0)
    rnd = np.concatenate([rng.uniform(-5, 40, (400, 2)), rng.uniform(-5, 40, (400, 2)), rng.uniform(0, 9, (400, 2))],
                         1).astype(F32)
    rnd[:, 2:4] = rnd[:, 0:2] + rng.choice([F32(7), _next(7, 0), _next(7, 8), F32(6.5), F32(10)], (400, 2))
    for props in (rows, rnd, np.concatenate([rows, rnd])):
        scores = np.arange(props.shape[0], dtype=F32) / F32(props.shape[0])
        full = np.concatenate([props, scores[:, None]], 1)
        for m in M_VALUES:
            want = mbo.filter_min_bbox_size(full, m)
            got = _torch_rows(props, scores, m)
            assert got.shape == want.shape and got.tobytes() == want.tobytes(), m
    # the values are compared in fp32: 8 + 1e-7 is 8 there, so a row 8 wide stays
    exact8 = rows[:1]
    assert mbo.filter_min_bbox_size(np.concatenate([exact8, [[0.5]]], 1), 8 + 1e-7).shape == (1, 7)
    assert mbo.filter_min_bbox_size(np.concatenate([exact8, [[0.5]]], 1), float(_next(8, 9))).shape == (0, 7)
    # NaN widths are dropped whatever m is
    nan_rows = rows[np.isnan(rows[:, :4]).any(1)]
    assert mbo.filter_min_bbox_size(nan_rows, 1e-30).shape == (0, 6)


def test_clamp_then_filter_matches_the_oracle_decode(oracle):
    """v0.6 order: delta2bbox's clamp to img_shape, then the filter.  The torch side clamps the oracle's unclamped
    decode and filters it; the oracle decodes with the clamp and filters; the kept rows are equal bit for bit.  The
    clamp makes boxes that stick out of the image small, and infinite deltas give infinite coordinates before it."""
    rng = np.random.default_rng(1)
    anchors = oracle.grid_anchors(oracle.gen_base_anchors(4, [2], [2], [1.0], 2), (4, 12, 12), 4, 2)
    n = anchors.shape[0]
    deltas = np.concatenate([rng.normal(0, 0.8, (n, 2)), rng.uniform(-1.5, 1.5, (n, 2)), rng.normal(0, 0.5, (n, 1)),
                             rng.uniform(-1, 1, (n, 1))], 1).astype(F32)
    deltas[::3, 2:4] = 0            # widths of exactly 8 before the clamp, or a few ulps off through the centre's rounding
    deltas[5, 0], deltas[6, 1], deltas[7, 0] = np.inf, -np.inf, F32(3e38)
    img = (40, 44, 3, 8)
    raw = oracle.delta2bbox3d(anchors, deltas)
    clamped = oracle.delta2bbox3d(anchors, deltas, max_shape=img)
    t_clamped = _v06_clamp(torch.from_numpy(raw), img).numpy()
    assert t_clamped.tobytes() == clamped.tobytes()
    scores = rng.uniform(0, 1, n).astype(F32)
    full = np.concatenate([clamped, scores[:, None]], 1)
    w = (clamped[:, 2] - clamped[:, 0]) + F32(1)
    assert (w == 8).any() and ((w < 8) & (w > 7.999)).any() and ((w > 8) & (w < 8.001)).any() and (w < 4).any()
    for m in M_VALUES:
        want = mbo.filter_min_bbox_size(full, m)
        got = _torch_rows(t_clamped, scores, m)
        assert got.shape == want.shape and got.tobytes() == want.tobytes(), m


@pytest.mark.parametrize("kw", [dict(), dict(nms_pre=0, nms_post=60, max_num=90), dict(nms_across_levels=True),
                                dict(masked=True)])
def test_reference_at_zero_is_the_oracle(oracle, kw):
    """At min_bbox_size = 0 the test reference is oracle.get_bboxes_single, bit for bit: it restates that loop."""
    kw = dict(kw)
    masked = kw.pop("masked", False)
    cfg = dict(CFG, **kw)
    rng = np.random.default_rng(3)
    cls = [(2 * rng.standard_normal((1, 1) + d)).astype(F32) for d in DIMS]
    reg = [(0.6 * rng.standard_normal((1, 6) + d)).astype(F32) for d in DIMS]
    masks = [(rng.random(int(np.prod(d))) < 0.6).astype(np.uint8) for d in DIMS] if masked else None
    args = ([c[0] for c in cls], [r[0] for r in reg], _anchors(oracle, DIMS), IMG, cfg['nms_pre'], cfg['nms_post'],
            cfg['max_num'], cfg['nms_thr'])
    want = oracle.get_bboxes_single(*args, nms_across_levels=cfg['nms_across_levels'], pos_indices=masks)
    got = mbo.get_bboxes_single(*args, nms_across_levels=cfg['nms_across_levels'], pos_indices=masks, min_bbox_size=0)
    assert want.shape[0] > 0 and got.shape == want.shape and got.tobytes() == want.tobytes()


def test_filter_abi_rejects_bad_arguments():
    import roi3d_b200
    lib = roi3d_b200._lib.lib
    fake = 1 << 20

    def call(dets, nseg, k, cin, m, cout):
        rc = lib.roi3d_filter_min_size_rows7(dets, nseg, k, cin, m, cout, None)
        msg = lib.roi3d_last_error()
        return rc, msg.decode() if msg else ""

    for args, text in [((fake, -1, 4, fake, 8.0, fake), "sizes"), ((fake, 2, -1, fake, 8.0, fake), "sizes"),
                       ((None, 2, 4, fake, 8.0, fake), "NULL"), ((fake, 2, 4, None, 8.0, fake), "NULL"),
                       ((fake, 2, 4, fake, 8.0, None), "NULL"), ((fake, 2, 4, fake, float("nan"), fake), "NaN")]:
        rc, msg = call(*args)
        assert rc == EINVAL and text in msg, (args, msg)
    assert call(None, 0, 4, None, 8.0, None)[0] == 0       # no segment: nothing to do


def test_every_filter_instantiation_has_a_gpu_row():
    assert built_kernels("filter_min_size") == {FILTER}


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@functools.lru_cache(maxsize=None)
def _size_delta_pool():
    """fp32 values in [-1.2, 1.2] whose device expf (torch.exp on CUDA, the same libdevice expf the decode kernel
    calls) equals the host libm's expf (the oracle's decode)."""
    libm = ctypes.CDLL(ctypes.util.find_library("m"))
    libm.expf.argtypes, libm.expf.restype = [ctypes.c_float], ctypes.c_float
    cand = np.random.default_rng(123).uniform(-1.2, 1.2, 8192).astype(F32)
    cand = np.concatenate([cand, F32([0.0])])
    dev_exp = torch.exp(torch.from_numpy(cand).cuda()).cpu().numpy()
    host_exp = np.array([libm.expf(float(v)) for v in cand], F32)
    pool = cand[dev_exp.view(np.uint32) == host_exp.view(np.uint32)]
    assert pool.size >= 2048 and 0.0 in pool, pool.size
    return pool


def _inputs(seed, B, dims=DIMS, shift=0.6):
    """Logits ~ 2 N(0, 1); position deltas ~ shift N(0, 1), so that boxes leave the image and the clamp shrinks them;
    size deltas from the pool, so that widths span about 0.3x to 3.3x the anchor."""
    rng = np.random.default_rng(seed)
    pool = _size_delta_pool()
    cls = [(2 * rng.standard_normal((B, 1) + d)).astype(F32) for d in dims]
    reg = []
    for d in dims:
        r = (shift * rng.standard_normal((B, 6) + d)).astype(F32)
        r[:, [2, 3, 5]] = rng.choice(pool, (B, 3) + d)
        reg.append(r)
    return cls, reg


def _head(levels=3):
    from roi3d_b200 import RPNProposal3D
    return RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0],
                         anchor_strides=C4_STRIDES[:levels], anchor_strides_depth=C4_DSTRIDES[:levels])


def _anchors(oracle, dims):
    return [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
            for d, s, ds in zip(dims, C4_STRIDES, C4_DSTRIDES)]


def _scores(cls_t, b):
    # the device's sigmoid, which the top-k's fused sigmoid equals bit for bit (glibc's expf may differ in the last bit)
    return [c[b].permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy() for c in cls_t]


def _decoded(oracle, reg, b, scores, anchors, img, nms_pre, masks):
    """Per level, the rows the filter sees for image b: oracle.get_bboxes_single's steps up to the clamped decode."""
    out = []
    for lvl, (r, anc) in enumerate(zip(reg, anchors)):
        sc, d = scores[lvl], np.transpose(r[b], (2, 3, 1, 0)).reshape(-1, 6)
        if masks is not None and nms_pre > 0 and sc.shape[0] > nms_pre:
            sel = masks[lvl].astype(bool)
            sc, d, anc = sc[sel], d[sel], anc[sel]
        if nms_pre > 0 and sc.shape[0] > nms_pre:
            idx = oracle.topk(sc, nms_pre)
            d, anc = d[idx], anc[idx]
        out.append(oracle.delta2bbox3d(anc, d, max_shape=img))
    return out


def _dropped(oracle, rows, m):
    return 1.0 - mbo.filter_min_bbox_size(rows, m).shape[0] / rows.shape[0]


def _run(oracle, dev, head, cls, reg, imgs, cfg, m, masks=None, expect=None, tensors=None):
    """get_proposals at min_bbox_size = m against the oracle, bit for bit, per image.  expect names the fraction of
    decoded rows m drops on every level of every image ('none', 'some', 'all'), checked first.  tensors: the device
    copies of cls / reg to call with (a CUDA graph is keyed on their addresses)."""
    dims = [tuple(c.shape[2:]) for c in cls]
    cfg = dict(cfg, min_bbox_size=m)
    if tensors is None:
        tensors = ([torch.from_numpy(c).to(dev) for c in cls], [torch.from_numpy(r).to(dev) for r in reg])
    cls_t, reg_t = tensors
    anchors = _anchors(oracle, dims)
    metas = [dict(img_shape=img, scale_factor=1.0) for img in imgs]
    wants = []
    for b, img in enumerate(imgs):
        sc = _scores(cls_t, b)
        if expect is not None:
            fr = [_dropped(oracle, rows, m) for rows in _decoded(oracle, reg, b, sc, anchors, img, cfg['nms_pre'], masks)]
            ok = {"none": all(f == 0 for f in fr), "some": all(0 < f < 1 for f in fr), "all": all(f == 1 for f in fr)}
            assert ok[expect], (b, fr)
        wants.append(mbo.get_bboxes_single([c[b] for c in cls], [r[b] for r in reg], anchors, img, cfg['nms_pre'],
                                              cfg['nms_post'], cfg['max_num'], cfg['nms_thr'],
                                              nms_across_levels=cfg['nms_across_levels'], pos_indices=masks, scores=sc,
                                              min_bbox_size=m))
    got = head.get_proposals(cls_t, reg_t, metas, cfg)
    assert len(got) == len(imgs)
    for b, (g, want) in enumerate(zip(got, wants)):
        g = g.cpu().numpy()
        assert g.shape == want.shape and g.tobytes() == want.tobytes(), (b, g.shape, want.shape)
    return got, wants


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_size_delta_pool_decodes_bit_identically(oracle, dev):
    """The premise of the exact comparisons: on the pool's deltas the device decode equals the oracle's bit for bit."""
    from roi3d_b200 import AnchorGenerator3D
    from roi3d_b200.models.anchor_heads import decode_proposals
    cls, reg = _inputs(7, 1)
    for lvl, (d, s, ds) in enumerate(zip(DIMS, STRIDES, DSTRIDES)):
        gen = AnchorGenerator3D(s, [2], [2], [1.0], ds)
        n = int(np.prod(d))
        idx = np.arange(n, dtype=np.int64)
        got = decode_proposals(torch.from_numpy(reg[lvl][0]).to(dev), gen.base_anchors, s, ds,
                               torch.from_numpy(idx).to(dev), None, (0,) * 6, (1,) * 6, IMG).cpu().numpy()
        want = oracle.delta2bbox3d(_anchors(oracle, DIMS)[lvl], np.transpose(reg[lvl][0], (2, 3, 1, 0)).reshape(-1, 6),
                                   max_shape=IMG)
        assert got[:, :6].tobytes() == want.tobytes(), lvl


CASES = {
    # name: (images, cfg overrides, masked)
    "sorted": ([IMG], dict(nms_pre=100), False),                     # levels 0 and 1 score-sorted, level 2 in anchor order
    "index_order": ([IMG], dict(nms_pre=0, nms_post=60, max_num=90), False),
    "masked": ([IMG], dict(nms_pre=300), True),                      # pos_indices on the two levels above nms_pre
    "across": ([IMG, IMG], dict(nms_pre=200, nms_across_levels=True), False),
    "batch3": ([IMG, (60, 84, 3, 12), (56, 96, 3, 9)], dict(nms_pre=200), False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("expect,m", [("none", 0), ("some", M_SOME), ("all", M_ALL)])
@pytest.mark.parametrize("case", sorted(CASES))
def test_get_proposals_matches_oracle(oracle, dev, case, expect, m):
    imgs, over, masked = CASES[case]
    cls, reg = _inputs(11 + sorted(CASES).index(case), len(imgs))
    head = _head()
    masks = None
    if masked:
        rng = np.random.default_rng(5)
        masks = [(rng.random(int(np.prod(d))) < 0.6).astype(np.uint8) for d in DIMS]
        head.pos_indices = [torch.from_numpy(mk).to(dev) for mk in masks]
    got, _ = _run(oracle, dev, head, cls, reg, imgs, dict(CFG, **over), m, masks, expect)
    if expect == "all":
        assert all(tuple(g.shape) == (0, 7) for g in got)
    else:
        assert all(g.shape[0] > 0 for g in got)


@pytest.mark.gpu
@pytest.mark.parametrize("m", [8, 8 + 1e-7, float(_next(8, 0)), float(_next(8, 9))])
def test_boundary_rows_and_nan_deltas(oracle, dev, m):
    """Half of the level-0 anchors get zero size deltas: their widths and heights are 8 exactly or a few ulps off (the
    centre's rounding), so m = 8 and its fp32 neighbours split them by the last bits.  Some rows have NaN deltas."""
    cls, reg = _inputs(21, 1, shift=0.3)
    rng = np.random.default_rng(22)
    zero = rng.random(DIMS[0]) < 0.5
    for c in (2, 3):
        reg[0][0, c][zero] = 0.0
    for lvl in (0, 1):
        for c in (0, 1, 2, 3):
            reg[lvl][0, c][rng.random(DIMS[lvl]) < 0.02] = np.nan
        cls[lvl][0, 0][np.isnan(reg[lvl][0, 0])] = 6.0    # high scores: the NaN rows reach the filter
    cfg = dict(CFG, nms_pre=1000)
    cls_t = [torch.from_numpy(c).to(dev) for c in cls]
    lvl0 = _decoded(oracle, reg, 0, _scores(cls_t, 0), _anchors(oracle, DIMS), IMG, 1000, None)[0]
    w, h = (lvl0[:, 2] - lvl0[:, 0]) + F32(1), (lvl0[:, 3] - lvl0[:, 1]) + F32(1)
    for a in (w, h):
        assert (a == 8).any() and ((a < 8) & (a > 7.999)).any() and ((a > 8) & (a < 8.001)).any()
    assert ((w == 8) & (h == 8)).any() and (lvl0[:, 0] == lvl0[:, 2]).any()   # NaN x deltas clamp to a 1-wide box
    _run(oracle, dev, _head(), cls, reg, [IMG], cfg, m)


@pytest.mark.gpu
def test_one_row_segment_and_an_image_with_no_proposals(oracle, dev):
    """Image 0 keeps exactly one row on levels 1 and 2 and none on level 0; image 1 keeps none anywhere and returns a
    [0, 7] tensor, also through get_bboxes_single."""
    cls, reg = _inputs(31, 2)
    m = 4.0
    for lvl, d in enumerate(DIMS):
        reg[lvl][:, [2, 3]] = -3.0                              # boxes of 0.05x the anchor: below m everywhere
        if lvl > 0:
            z, y, x = d[0] // 2, d[1] // 2, d[2] // 2
            reg[lvl][0, :, z, y, x] = 0.0                      # one anchor-sized box in the middle of image 0
            cls[lvl][0, 0, z, y, x] = 9.0
    cls_t = [torch.from_numpy(c).to(dev) for c in cls]
    anchors = _anchors(oracle, DIMS)
    kept = [[mbo.filter_min_bbox_size(rows, m).shape[0] for rows in
             _decoded(oracle, reg, b, _scores(cls_t, b), anchors, IMG, CFG['nms_pre'], None)] for b in range(2)]
    assert kept == [[0, 1, 1], [0, 0, 0]], kept
    head = _head()
    got, wants = _run(oracle, dev, head, cls, reg, [IMG, IMG], CFG, m)
    assert got[0].shape == (2, 7) and tuple(got[1].shape) == (0, 7)
    for b in range(2):
        one = head.get_bboxes_single([c[b] for c in cls_t], [torch.from_numpy(r[b]).to(dev) for r in reg], IMG,
                                     dict(CFG, min_bbox_size=m))
        assert one.cpu().numpy().tobytes() == wants[b].tobytes() and one.shape == wants[b].shape


@pytest.mark.gpu
def test_cuda_graph_replays_each_min_size(oracle, dev):
    """cuda_graph = True: one graph per min_bbox_size; replays alternating between two values and 0 each give that
    value's oracle result."""
    cls, reg = _inputs(41, 2)
    imgs = [IMG, (72, 80, 3, 14)]
    tensors = ([torch.from_numpy(c).to(dev) for c in cls], [torch.from_numpy(r).to(dev) for r in reg])
    head = _head()
    head.cuda_graph = True
    for m in (M_SOME, 5.0, 0, M_SOME, 0, 5.0, M_SOME):
        _run(oracle, dev, head, cls, reg, imgs, CFG, m, tensors=tensors)
    assert len(head._graphs) == 3


@pytest.mark.gpu
def test_c4_full_size(oracle, dev):
    """C4 at full size: 8 volumes of 512x512x160, 5 levels (1 310 720 ... 320 anchors), nms_pre 2000, NMS 0.7,
    nms_post 1000, max_num 1000, at min_bbox_size = C4_M."""
    dims = [(80, 128, 128), (40, 64, 64), (20, 32, 32), (10, 16, 16), (5, 8, 8)]
    cls, reg = _inputs(61, 8, dims)
    cfg = dict(nms_pre=2000, nms_post=1000, max_num=1000, nms_thr=0.7, nms_across_levels=False)
    got, _ = _run(oracle, dev, _head(5), cls, reg, [(512, 512, 3, 160)] * 8, cfg, C4_M)
    assert all(g.shape[0] > 0 for g in got)


@pytest.mark.gpu
def test_filter_kernel_on_long_segments(oracle, dev):
    """The kernel alone on segments of a whole C4 level (1 310 720 rows, k unpadded): counts at k, below k, above k
    (clamped), 0 and negative; written to a separate count tensor and in place over the input counts."""
    import roi3d_b200
    lib = roi3d_b200._lib.lib
    k = 1310720 + 3
    counts = np.array([k, k - 1000, k + 7, 0, -5, 1], np.int32)
    nseg = counts.size
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)
    dets = torch.rand((nseg, k, 7), device=dev, generator=gen) * 30
    dets[..., 2:4] = dets[..., 0:2] + torch.rand((nseg, k, 2), device=dev, generator=gen) * 16 - 1
    dets[0, 5:9, 0] = float("nan")
    host = dets.cpu().numpy()
    m = 8.5
    for inplace in (False, True):
        d = dets.clone()
        cin = torch.from_numpy(counts).to(dev)
        cout = cin if inplace else torch.empty_like(cin)
        roi3d_b200._lib.check(lib.roi3d_filter_min_size_rows7(d.data_ptr(), nseg, k, cin.data_ptr(), m, cout.data_ptr(),
                                                              torch.cuda.current_stream().cuda_stream))
        got_n, got = cout.cpu().numpy(), d.cpu().numpy()
        if not inplace:
            assert np.array_equal(cin.cpu().numpy(), counts)
        for s in range(nseg):
            n = min(max(int(counts[s]), 0), k)
            want = mbo.filter_min_bbox_size(host[s, :n], m)
            assert got_n[s] == want.shape[0], (s, got_n[s], want.shape)
            assert got[s, :want.shape[0]].tobytes() == want.tobytes(), s
        assert 0 < got_n[0] < k


# The path's kernels at min_bbox_size = 0 for the two configurations below, in launch order, as the path ran them before
# the filter existed: the m = 0 path must stay exactly this.  TORCH stands for a kernel of torch's own (the masked path's
# `1 - presorted`).
TORCH = "(torch)"
_M0_COMMON = ["decode_proposals_batched_kernel", "nms3d_rank_kernel", "nms3d_mask_q_kernel<false>", "nms3d_sweep_kernel",
              "rpn_collect_kernel", "topk_tail_kernel<false>", "gather_rows7_kernel"]
M0_LAUNCHES = {
    "plain": ["topk_tail_kernel<true>"] + _M0_COMMON,
    "masked": ["topk_tail_kernel<true>", TORCH] + _M0_COMMON,
}


def _launch_list(dev, which, m):
    """Kernels of one eager get_proposals call in launch order: library kernels by key, torch's as TORCH."""
    cls, reg = _inputs(51, 2)
    head = _head()
    if which == "masked":
        rng = np.random.default_rng(52)
        head.pos_indices = [torch.from_numpy((rng.random(int(np.prod(d))) < 0.6).astype(np.uint8)).to(dev) for d in DIMS]
    cls_t = [torch.from_numpy(c).to(dev) for c in cls]
    reg_t = [torch.from_numpy(r).to(dev) for r in reg]
    metas = [dict(img_shape=IMG, scale_factor=1.0)] * 2
    head.get_proposals(cls_t, reg_t, metas, dict(CFG, min_bbox_size=m))    # first-call set-up out of the record
    names = launched_kernels(lambda: head.get_proposals(cls_t, reg_t, metas, dict(CFG, min_bbox_size=m)))
    return [next(iter(library_kernels([n])), TORCH) for n in names]


@pytest.mark.gpu
@pytest.mark.parametrize("which", sorted(M0_LAUNCHES))
def test_filter_launches_iff_min_size_is_positive(dev, which):
    """The filter kernel runs once, right after the decode, iff min_bbox_size > 0; at 0 the path launches exactly what
    it launched before the filter existed."""
    at0, at_m = _launch_list(dev, which, 0), _launch_list(dev, which, M_SOME)
    assert FILTER not in at0 and at_m.count(FILTER) == 1
    i = at_m.index(FILTER)
    assert at_m[i - 1] == "decode_proposals_batched_kernel" and at_m[:i] + at_m[i + 1:] == at0
    assert at0 == M0_LAUNCHES[which], at0

"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C ABI
(libroi3d_b200.so via the Python host mirror) and is compared with the CPU oracle on the same seeded inputs;
the reference's OWN kernels are represented by their outputs stored under tests/golden/ (tests/golden/make_golden.py).

Tolerances (BASELINE.json north_star): NMS keep lists bit-exact; RoIAlign forward 1e-5, backward 1e-4,
measured as max|a-b| / max(1, max|ref|)  (norm-relative: pure elementwise relative error is ill-conditioned on
zero-mean data, SURVEY section 7)."""
import os

import numpy as np
import pytest
import torch

import synth

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

FWD_TOL = 1e-5
BWD_TOL = 1e-4


def rel_err(a, ref):
    a, ref = np.asarray(a, np.float64), np.asarray(ref, np.float64)
    return float(np.abs(a - ref).max() / max(1.0, np.abs(ref).max())) if a.size else 0.0


def cl(x):
    return x.contiguous(memory_format=torch.channels_last_3d)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------ NMS
@pytest.mark.parametrize("n,thr", [(1, 0.5), (2, 0.5), (63, 0.7), (64, 0.7), (65, 0.3), (300, 0.5), (2000, 0.7),
                                   (2000, 0.1), (4097, 0.7)])
def test_nms_keep_bit_exact(oracle, dev, n, thr):
    from roi3d_b200.ops import nms
    dets = synth.c1_boxes(n, seed=n)
    want = oracle.nms3d(dets, thr)
    t = torch.from_numpy(dets).to(dev)
    kept, inds = nms(t, thr)
    assert inds.dtype == torch.int64 and inds.device == t.device
    assert np.array_equal(inds.cpu().numpy(), want)
    assert torch.equal(kept, t[inds])
    # numpy + device_id form (host-buffer C ABI entry)
    kept_np, inds_np = nms(dets, thr, device_id=0)
    assert isinstance(inds_np, np.ndarray) and np.array_equal(inds_np, want)
    assert np.array_equal(kept_np, dets[want])


def test_nms_ties_and_duplicates(oracle, dev):
    from roi3d_b200.ops import nms
    dets = synth.c1_boxes(500, seed=11)
    dets[:, 6] = np.round(dets[:, 6] * 8) / 8          # many equal scores
    dets[100:200, :6] = dets[0:100, :6]                # exact duplicate boxes
    want = oracle.nms3d(dets, 0.5)
    _, inds = nms(torch.from_numpy(dets).to(dev), 0.5)
    assert np.array_equal(inds.cpu().numpy(), want)


@pytest.mark.parametrize("thr", [0.5, 0.0, -0.25])
def test_nms_coarse_rejection_edge_cases(oracle, dev, thr):
    """The bit-matrix kernels skip a pair whose coarse cell masks miss each other (csrc/nms3d.cu).  The kept list must
    stay the oracle's where that shortcut could go wrong: boxes one voxel apart (the reference's +1 makes them touch),
    boxes stored inverted, huge and non-finite coordinates, sparse sets with far outliers, and a negative threshold
    (every pair with a finite iou suppresses, disjoint ones included)."""
    from roi3d_b200.ops import nms
    rng = np.random.default_rng(5)
    n = 700
    c = rng.uniform(0, 400, (n, 3)).astype(np.float32)
    h = rng.uniform(0.5, 6, (n, 3)).astype(np.float32)
    d = np.stack([c[:, 0] - h[:, 0], c[:, 1] - h[:, 1], c[:, 0] + h[:, 0], c[:, 1] + h[:, 1], c[:, 2] - h[:, 2],
                  c[:, 2] + h[:, 2], rng.uniform(0, 1, n).astype(np.float32)], 1).astype(np.float32)
    d[1, :6] = d[0, :6]
    d[1, [0, 2]] += (d[0, 2] - d[0, 0]) + 1.0            # abuts box 0 along x: extent + 1 - 1 > 0 in the reference
    d[2, :6] = d[0, :6]
    d[2, [0, 2]] += (d[0, 2] - d[0, 0]) + 2.0            # one voxel further: extent 0
    d[10, [0, 2]] = d[10, [2, 0]]                        # inverted box
    d[11, [0, 2]] = d[11, [2, 0]] + np.float32([3, -3])  # inverted by more than the margin
    d[20, :6] = [1e9, 1e9, 1e9 + 64, 1e9 + 64, 1e9, 1e9 + 64]    # far outlier stretches the CTA's grid
    d[21, :6] = [-3e38, -3e38, 3e38, 3e38, -3e38, 3e38]            # covers everything, sums overflow
    want = oracle.nms3d(d, thr)
    _, inds = nms(torch.from_numpy(d).to(dev), thr)
    assert np.array_equal(inds.cpu().numpy(), want)
    # a large sparse set: most 64 x 64 tiles see no overlap at all
    big = synth.c1_boxes(2000, seed=3)
    big[:, [0, 2]] *= 7
    big[:, [1, 3]] *= 5
    want = oracle.nms3d(big, thr)
    _, inds = nms(torch.from_numpy(big).to(dev), thr)
    assert np.array_equal(inds.cpu().numpy(), want)


def test_nms_batched_segments(oracle, dev):
    from roi3d_b200.ops import nms3d_batched
    sizes = [0, 1, 64, 130, 700, 2000]
    n_max = 2000
    dets = np.zeros((len(sizes), n_max, 7), np.float32)
    for s, n in enumerate(sizes):
        dets[s, :n] = synth.c1_boxes(n, seed=100 + s) if n else 0
    cnt = torch.tensor(sizes, dtype=torch.int32, device=dev)
    keep, keep_s, num = nms3d_batched(torch.from_numpy(dets).to(dev), cnt, 0.7)
    num = num.cpu().numpy()
    for s, n in enumerate(sizes):
        want, want_s = oracle.nms3d(dets[s, :n], 0.7, return_score_order=True)
        assert num[s] == len(want)
        assert np.array_equal(keep[s, :num[s]].cpu().numpy(), want)
        assert np.array_equal(keep_s[s, :num[s]].cpu().numpy(), want_s)


def _mirrored_copies(dets, keep, copies):
    """A stored NMS case copied into other octants (copy j negates x, y and / or z by the bits of j, which leaves every
    IoU inside the copy as it was; boxes of different copies can meet only on a mirror plane, and for the cases copied
    here no such contact reaches the threshold, which the oracle check confirms) with its scores scaled by 2^-j (exact:
    the order inside a copy stays, and no two scores are equal).  Greedy NMS then keeps in every copy what it kept in
    the original, so the reference's keep list of the whole set is the stored one repeated."""
    n, parts = dets.shape[0], []
    for j in range(copies):
        d = dets.copy()
        for bit, (lo, hi) in enumerate([(0, 2), (1, 3), (4, 5)]):
            if j >> bit & 1:
                d[:, [lo, hi]] = -dets[:, [hi, lo]]
        d[:, 6] = dets[:, 6] * np.float32(2.0 ** -j)
        parts.append(d)
    return np.concatenate(parts), np.concatenate([keep + j * n for j in range(copies)])


def test_nms_against_reference_kernel(oracle, dev):
    """The keep lists of the reference's own nms_cuda_3d, stored in tests/golden/nms3d_ref.npz (65 to 1000 boxes), and
    the three larger cases copied up to 2000-2100 boxes (the full 32-word mask panel) by _mirrored_copies."""
    from roi3d_b200.ops import nms
    z = np.load(os.path.join(GOLDEN, "nms3d_ref.npz"))
    for t, copies in [("a", 1), ("b", 1), ("c", 1), ("d", 1), ("a", 7), ("b", 7), ("d", 2)]:
        dets, ref = _mirrored_copies(z["%s_dets" % t], z["%s_keep" % t], copies)
        thr = float(z["%s_thr" % t])
        assert len(np.unique(dets[:, 6])) == len(dets)
        assert np.array_equal(ref, oracle.nms3d(dets, thr)), "oracle disagrees with the reference kernel"
        assert np.array_equal(nms(torch.from_numpy(dets).to(dev), thr)[1].cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------- RoIAlign
def _feats(shape, seed):
    return np.random.default_rng(seed).standard_normal(shape).astype(np.float32)


CASES = [
    # (B, C, D, H, W), out_size, out_size_depth, scale, scale_d, sample_num, n_rois
    ((1, 64, 10, 32, 32), 7, 7, 0.25, 0.5, 2, 24),
    ((2, 32, 9, 14, 15), 7, 3, 0.25, 0.5, 2, 16),       # real-config bbox shape 7x7x3
    ((1, 40, 12, 20, 20), 14, 14, 0.25, 0.5, 2, 12),    # C not a multiple of 32*CV
    ((2, 64, 8, 16, 16), 14, 10, 0.125, 0.25, 2, 10),   # real-config mask shape 14x14x10
    ((1, 6, 10, 16, 16), 7, 7, 0.25, 0.5, 0, 10),       # adaptive sampling, odd channel count
    ((1, 16, 6, 12, 12), 5, 4, 0.25, 0.5, 2, 8),        # generic output size
    ((1, 8, 20, 60, 60), 7, 7, 1.0, 1.0, 2, 6),         # footprint larger than the tables -> literal path
    ((1, 160, 8, 18, 18), 7, 7, 0.25, 0.5, 2, 14),      # three channel chunks (last one half full): warps of a CTA
    ((1, 160, 6, 12, 12), 14, 14, 0.25, 0.5, 2, 9),     # ... span RoI sub-items with different chunks and pd
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("layout", ["channels_last", "contiguous"])
def test_roi_align_forward(oracle, dev, case, layout):
    from roi3d_b200.ops import RoIAlign3D
    shape, ps, pdp, sc, scd, sn, k = case
    B, C, D, H, W = shape
    f = _feats(shape, 1)
    img = (int(W / sc), int(H / sc), int(D / scd))
    rois = np.concatenate([synth.c2_rois(k, seed=2, img=img, batch=B),
                           synth.adversarial_rois((D, H, W), sc, scd, batch=B)], 0)
    if sn == 0:  # adaptive sampling of a zero-size RoI is 0/0 in the reference; checked separately
        ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
        rois = rois[ok]
    want = oracle.roi_align3d_forward(f, rois, ps, pdp, sc, scd, sn)
    ft = torch.from_numpy(f).to(dev)
    if layout == "channels_last":
        ft = cl(ft)
    out = RoIAlign3D(ps, pdp, sc, scd, sn)(ft, torch.from_numpy(rois).to(dev))
    assert out.shape == want.shape and out.is_contiguous()
    assert rel_err(out.cpu().numpy(), want) <= FWD_TOL


def test_roi_align_forward_literal_path_is_bit_exact(oracle, dev):
    """Variant 99 evaluates the reference's sample loops literally: identical bits to oracle(contract=1)."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D
    f = _feats((1, 32, 10, 24, 24), 3)
    rois = synth.c2_rois(20, seed=4, img=(96, 96, 20))
    want = oracle.roi_align3d_forward(f, rois, 7, 7, 0.25, 0.5, 2)
    roi3d_b200._lib.set_tuning(0, 99)
    try:
        out = RoIAlign3D(7, 7, 0.25, 0.5, 2)(cl(torch.from_numpy(f).to(dev)), torch.from_numpy(rois).to(dev))
    finally:
        roi3d_b200._lib.set_tuning(0, 0)
    assert np.array_equal(out.cpu().numpy(), want)


def test_roi_align_adaptive_zero_size_is_nan_like_reference(oracle, dev):
    from roi3d_b200.ops import RoIAlign3D
    f = _feats((1, 32, 6, 8, 8), 5)
    rois = np.array([[0, 10, 10, 9, 9, 4, 3]], np.float32)
    want = oracle.roi_align3d_forward(f, rois, 7, 7, 0.25, 0.5, 0)
    out = RoIAlign3D(7, 7, 0.25, 0.5, 0)(cl(torch.from_numpy(f).to(dev)), torch.from_numpy(rois).to(dev))
    assert np.isnan(want).all() and torch.isnan(out).all()


def test_roi_align_empty_rois(dev):
    from roi3d_b200.ops import RoIAlign3D
    f = torch.zeros(1, 32, 4, 8, 8, device=dev)
    out = RoIAlign3D(7, 3, 0.25, 0.5, 2)(f, torch.zeros(0, 7, device=dev))
    assert out.shape == (0, 32, 3, 7, 7)


@pytest.mark.parametrize("case", CASES[:6] + CASES[7:])
@pytest.mark.parametrize("layout", ["channels_last", "contiguous"])
def test_roi_align_backward(oracle, dev, case, layout):
    from roi3d_b200.ops import RoIAlign3D
    shape, ps, pdp, sc, scd, sn, k = case
    B, C, D, H, W = shape
    img = (int(W / sc), int(H / sc), int(D / scd))
    rois = np.concatenate([synth.c2_rois(k, seed=2, img=img, batch=B),
                           synth.adversarial_rois((D, H, W), sc, scd, batch=B)], 0)
    ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
    rois = rois[ok] if sn == 0 else rois
    g = _feats((rois.shape[0], C, pdp, ps, ps), 6)
    want = oracle.roi_align3d_backward(g, rois, shape, sc, scd, sn)
    ft = torch.from_numpy(_feats(shape, 1)).to(dev)
    if layout == "channels_last":
        ft = cl(ft)
    ft.requires_grad_(True)
    out = RoIAlign3D(ps, pdp, sc, scd, sn)(ft, torch.from_numpy(rois).to(dev))
    out.backward(torch.from_numpy(g).to(dev))
    assert ft.grad.shape == tuple(shape)
    assert rel_err(ft.grad.cpu().numpy(), want) <= BWD_TOL


def test_roi_align_backward_bug_compat(oracle, dev):
    from roi3d_b200.ops import RoIAlign3D, set_bug_compat
    shape = (1, 32, 9, 15, 15)
    rois = synth.c2_rois(6, seed=5, img=(60, 60, 18))
    g = _feats((6, 32, 3, 7, 7), 7)
    want = oracle.roi_align3d_backward(g, rois, shape, 0.25, 0.5, 2, bug_compat=True)
    ft = cl(torch.zeros(shape, device=dev)).requires_grad_(True)
    set_bug_compat(True)
    try:
        RoIAlign3D(7, 3, 0.25, 0.5, 2)(ft, torch.from_numpy(rois).to(dev)).backward(torch.from_numpy(g).to(dev))
    finally:
        set_bug_compat(False)
    assert rel_err(ft.grad.cpu().numpy(), want) <= BWD_TOL


def test_roi_align_against_reference_kernels(dev):
    """The outputs of the reference's own forward3d / backward3d, stored in tests/golden/roi_align3d_ref.npz for 6
    channels, widened to 64 so that the product takes its streamed and planar kernels (they need C % 64 == 0 or
    C % 4 == 0).  The reference computes each channel from that channel alone and linearly, so a level whose channel c
    is s_c * feats[:, src_c] (s_c a power of two: exact) has the output s_c * out[:, src_c], and output gradients built
    the same way have the input gradient s_c * gin[:, src_c].  Non-cubic outputs: the reference's backward reads the
    wrong top_diff element, so only there does the product run with bug_compat.  Tuning variant 60 puts the cubic
    7-wide case on the planar forward and backward kernels as well."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D, set_bug_compat
    z = synth.load_roi_align_ref(os.path.join(GOLDEN, "roi_align3d_ref.npz"))
    rng = np.random.default_rng(64)
    src = rng.permutation(np.arange(64) % 6)
    s = rng.choice(np.float32([-2, -1, -0.5, 0.5, 1, 2]), 64)[None, :, None, None, None]

    def widen(a):
        return np.ascontiguousarray(a[:, src] * s)
    f, sc, scd = widen(z["feats"]), float(z["spatial_scale"]), float(z["spatial_scale_depth"])
    runs = [(t, layout, 0) for t in synth.ROI_ALIGN_REF_TAGS for layout in ("channels_last", "contiguous")]
    for tag, layout, variant in runs + [("c7", "channels_last", 60)]:
        ps, pdp, sn = (int(v) for v in z["%s_cfg" % tag])
        x = torch.from_numpy(f).to(dev)
        x = (cl(x) if layout == "channels_last" else x).requires_grad_(True)
        roi3d_b200._lib.set_tuning(0, variant)
        roi3d_b200._lib.set_tuning(1, variant)
        set_bug_compat(ps != pdp)
        try:
            out = RoIAlign3D(ps, pdp, sc, scd, sn)(x, torch.from_numpy(z["%s_rois" % tag]).to(dev))
            out.backward(torch.from_numpy(widen(z["%s_gout" % tag])).to(dev))
        finally:
            set_bug_compat(False)
            roi3d_b200._lib.set_tuning(0, 0)
            roi3d_b200._lib.set_tuning(1, 0)
        assert rel_err(out.detach().cpu().numpy(), widen(z["%s_out" % tag])) <= FWD_TOL, (tag, layout, variant)
        assert rel_err(x.grad.cpu().numpy(), widen(z["%s_gin" % tag])) <= BWD_TOL, (tag, layout, variant)


# ------------------------------------------------------------------------------- extractor / levels
def test_map_roi_levels_matches_oracle_and_torch(oracle, dev):
    from roi3d_b200 import SingleRoIExtractor
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=7, out_size_depth=7, sample_num=2), 32,
                            [4, 8, 16, 32], [2, 4, 8, 16])
    rois = synth.c3_rois(2000, vols=1, seed=4)
    # boundary sweep: volumes whose sqrt lands on / next to 56 * 2^k
    edge = []
    for k in range(0, 4):
        s = 56.0 * 2 ** k
        for dlt in (-2e-3, -1e-4, 0.0, 1e-4, 2e-3):
            w = np.float32(s * (1 + dlt))
            edge.append([0, 0, 0, w - 1, w - 1, 0, 0])
    rois = np.concatenate([rois, np.asarray(edge, np.float32)], 0)
    rt = torch.from_numpy(rois).to(dev)
    got = ex.map_roi_levels(rt, 4)
    assert got.dtype == torch.int64
    assert np.array_equal(got.cpu().numpy(), oracle.map_roi_levels(rois, 4))
    # the reference expression evaluated by torch's CUDA elementwise kernels (single_level.py:73-81)
    scale = torch.sqrt((rt[:, 3] - rt[:, 1] + 1) * (rt[:, 4] - rt[:, 2] + 1) * (rt[:, 6] - rt[:, 5] + 1))
    ref = torch.floor(torch.log2(scale / 56 + 1e-6)).clamp(min=0, max=3).long()
    assert torch.equal(got, ref)
    hist = np.bincount(got.cpu().numpy(), minlength=4)
    assert (hist > 0).all()


def _pyramid(B, C, seed, base=(10, 32, 32), levels=4):
    feats = []
    for l in range(levels):
        shape = (B, C) + tuple(max(1, s >> l) for s in base)
        feats.append(_feats(shape, seed + l))
    return feats


@pytest.mark.parametrize("ps,pdp", [(7, 7), (14, 10)])
def test_extractor_forward_backward_multilevel(oracle, dev, ps, pdp):
    from roi3d_b200 import SingleRoIExtractor
    B, C = 2, 64
    strides, dstrides = [4, 8, 16, 32], [2, 4, 8, 16]
    feats = _pyramid(B, C, 20)
    rois = synth.c3_rois(60, vols=B, seed=4, img=(128, 128, 20))
    lv = oracle.map_roi_levels(rois, 4)
    assert len(np.unique(lv)) >= 3
    want = np.zeros((rois.shape[0], C, pdp, ps, ps), np.float32)
    g = _feats(want.shape, 30)
    want_grads = []
    for l in range(4):
        sel = lv == l
        want[sel] = oracle.roi_align3d_forward(feats[l], rois[sel], ps, pdp, 1 / strides[l], 1 / dstrides[l], 2)
        want_grads.append(oracle.roi_align3d_backward(g[sel], rois[sel], feats[l].shape, 1 / strides[l],
                                                      1 / dstrides[l], 2))
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=ps, out_size_depth=pdp, sample_num=2), C, strides,
                            dstrides)
    ft = [cl(torch.from_numpy(f).to(dev)).requires_grad_(True) for f in feats]
    out = ex(ft, torch.from_numpy(rois).to(dev))
    assert rel_err(out.detach().cpu().numpy(), want) <= FWD_TOL
    out.backward(torch.from_numpy(g).to(dev))
    for l in range(4):
        assert rel_err(ft[l].grad.cpu().numpy(), want_grads[l]) <= BWD_TOL
    # NCDHW-contiguous inputs (the reference's layout) give the same values and contiguous grads
    ft2 = [torch.from_numpy(f).to(dev).requires_grad_(True) for f in feats]
    out2 = ex(ft2, torch.from_numpy(rois).to(dev))
    assert rel_err(out2.detach().cpu().numpy(), want) <= FWD_TOL   # NCDHW levels are read natively (planar kernel)
    out2.backward(torch.from_numpy(g).to(dev))
    for l in range(4):
        assert ft2[l].grad.is_contiguous()
        assert rel_err(ft2[l].grad.cpu().numpy(), want_grads[l]) <= BWD_TOL


# -------------------------------------------------------------------------------------- proposal path
def test_topk_segmented_exact(oracle, dev):
    from roi3d_b200.models.anchor_heads import topk_segmented
    rng = np.random.default_rng(40)
    segs = [rng.standard_normal(n).astype(np.float32) for n in (5, 300, 5000, 70000)]
    segs.append(np.round(rng.standard_normal(20000) * 4).astype(np.float32) / 4)    # heavy ties
    segs.append(np.full(3000, 0.25, np.float32))                                     # all equal
    k = 2000
    idx, val = topk_segmented([torch.from_numpy(s).to(dev) for s in segs], k)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    for s, seg in enumerate(segs):
        want = oracle.topk(seg, k)
        m = len(want)
        assert np.array_equal(idx[s, :m], want)
        assert np.array_equal(val[s, :m], seg[want])
        assert (idx[s, m:] == -1).all()


def test_topk_small_segments(oracle, dev):
    """Short segments only (the final topk(max_num) of the proposal path is such a call): ties, k > n, -inf padding
    and the 'small segments stay in index order' rule."""
    from roi3d_b200.models.anchor_heads import topk_segmented
    rng = np.random.default_rng(44)
    segs = [rng.standard_normal(n).astype(np.float32) for n in (1, 5, 300, 5000, 8192)]
    segs.append(np.round(rng.standard_normal(6000) * 4).astype(np.float32) / 4)     # heavy ties
    segs.append(np.full(3000, 0.25, np.float32))                                     # all equal
    segs.append(np.where(rng.random(4000) < 0.5, -np.inf, rng.standard_normal(4000)).astype(np.float32))  # -inf padding
    for k in (2000, 1, 8192):
        idx, val = topk_segmented([torch.from_numpy(s).to(dev) for s in segs], k)
        idx, val = idx.cpu().numpy(), val.cpu().numpy()
        for s, seg in enumerate(segs):
            want = oracle.topk(seg, k)
            m = len(want)
            assert np.array_equal(idx[s, :m], want)
            assert np.array_equal(val[s, :m], seg[want])
            assert (idx[s, m:] == -1).all() and (val[s, m:] == 0).all()
    k = 2000
    idx, val = topk_segmented([torch.from_numpy(s).to(dev) for s in segs], k, small_in_index_order=True)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    for s, seg in enumerate(segs):
        if len(seg) <= k:
            assert np.array_equal(idx[s, :len(seg)], np.arange(len(seg))) and np.array_equal(val[s, :len(seg)], seg)
        else:
            assert np.array_equal(idx[s], oracle.topk(seg, k))


def test_topk_mass_ties_overflow_the_boundary_buffer(oracle, dev):
    """More equal scores than the 4096-key boundary buffer holds: the full-data passes take over; order stays
    'descending score, ties to the lower index'."""
    from roi3d_b200.models.anchor_heads import topk_segmented
    rng = np.random.default_rng(45)
    segs = [np.full(100000, 0.5, np.float32),
            rng.choice(np.array([0.25, 0.5, 0.75], np.float32), 200000),
            rng.standard_normal(50000).astype(np.float32)]
    maps = [np.full((1, 10, 40, 50), 1.5, np.float32)]               # permuted + sigmoid, all equal
    for k in (2000, 7):
        idx, val = topk_segmented([torch.from_numpy(s).to(dev) for s in segs], k)
        for s, seg in enumerate(segs):
            want = oracle.topk(seg, k)
            assert np.array_equal(idx[s].cpu().numpy(), want) and np.array_equal(val[s].cpu().numpy(), seg[want])
        idx, val = topk_segmented([torch.from_numpy(m).to(dev) for m in maps], k, apply_sigmoid=True, permute_adhw=True)
        assert np.array_equal(idx[0].cpu().numpy(), np.arange(k))      # ties: lowest LOGICAL index first


def test_topk_permuted_sigmoid(oracle, dev):
    from roi3d_b200.models.anchor_heads import topk_segmented
    rng = np.random.default_rng(41)
    maps = [2 * rng.standard_normal(s).astype(np.float32)
            for s in ((1, 8, 16, 16), (3, 4, 6, 5), (1, 2, 3, 3), (2, 12, 24, 20))]
    maps[1] = np.round(maps[1])   # ties: the tie rule must use LOGICAL (permuted) indices
    k = 200
    idx, val = topk_segmented([torch.from_numpy(m).to(dev) for m in maps], k, apply_sigmoid=True,
                              permute_adhw=True)
    for s, m in enumerate(maps):
        t = torch.from_numpy(m).to(dev)
        flat = t.permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy()   # rpn_head_3d.py:87-90, on CUDA
        want = oracle.topk(flat, k)
        n = len(want)
        assert np.array_equal(idx[s, :n].cpu().numpy(), want)
        assert np.array_equal(val[s, :n].cpu().numpy(), flat[want])
    idx2, val2 = topk_segmented([torch.from_numpy(m).to(dev) for m in maps[:3]], k, apply_sigmoid=True,
                                permute_adhw=True)                           # same segments in a smaller batch
    assert torch.equal(idx2, idx[:3]) and torch.equal(val2, val[:3])


@pytest.mark.parametrize("mode", [0, 2, -1])
def test_topk_sieve_path_and_its_fallback(oracle, dev, mode):
    """The sieve path of the segmented top-k (sample -> threshold -> one pass -> proof, csrc/proposal.cu) returns the
    digit passes' result bit for bit: mode 0 = sieve where it applies, 2 = the sieve gives up on every long segment so
    that the guarded digit passes behind it run, -1 = digit passes only.  Inputs include the cases where the proof
    must fail on its own: saturated sigmoid scores (thousands of exact 1.0), constant segments, NaNs, a sorted ramp
    (the k largest in one corner), lengths around the sample size and a segment that starts off a 16-byte boundary."""
    import roi3d_b200
    from roi3d_b200.models.anchor_heads import topk_segmented
    rng = np.random.default_rng(77)
    raw = [rng.standard_normal(n).astype(np.float32) for n in (8193, 32768, 32769, 150001, 1310720)]
    raw.append(np.arange(200000, dtype=np.float32) / 7)                                   # ascending ramp
    raw.append(np.full(60000, -3.0, np.float32))                                          # constant
    raw.append(np.round(rng.standard_normal(90000) * 3).astype(np.float32))               # heavy ties
    withnan = rng.standard_normal(50000).astype(np.float32)
    withnan[::997] = np.nan
    raw.append(withnan)
    big = torch.from_numpy(np.concatenate([np.zeros(1, np.float32), raw[3]])).to(dev)
    roi3d_b200._lib.set_tuning(11, mode)
    try:
        for k in (2000, 100, 4096):
            segs = [torch.from_numpy(r).to(dev) for r in raw] + [big[1:]]                  # last: off a 16-byte boundary
            idx, val = topk_segmented(segs, k)
            for s, r in enumerate(raw + [raw[3]]):
                if np.isnan(r).any():
                    got = idx[s].cpu().numpy()
                    nn = int(np.isnan(r).sum())
                    assert np.isnan(r[got[:nn]]).all()                                     # NaNs lead, as in torch.topk
                    rest = np.where(np.isnan(r), -np.inf, r)
                    assert np.array_equal(got[nn:], oracle.topk(rest, k)[:k - nn])
                    continue
                want = oracle.topk(r, k)
                assert np.array_equal(idx[s].cpu().numpy(), want), (mode, k, s)
                assert np.array_equal(val[s].cpu().numpy(), r[want])
        # sigmoid scores in the reference's anchor order; x 12 saturates thousands of scores to exactly 1.0
        maps = [rng.standard_normal(sh).astype(np.float32) * sc
                for sh, sc in (((3, 20, 32, 32), 2.0), ((3, 20, 32, 32), 12.0), ((1, 80, 128, 128), 2.0), ((1, 40, 64, 64), 30.0))]
        idx, val = topk_segmented([torch.from_numpy(m).to(dev) for m in maps], 2000, apply_sigmoid=True, permute_adhw=True)
        for s, m in enumerate(maps):
            flat = torch.from_numpy(m).to(dev).permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy()
            want = oracle.topk(flat, 2000)
            assert np.array_equal(idx[s].cpu().numpy(), want), (mode, s)
            assert np.array_equal(val[s].cpu().numpy(), flat[want])
    finally:
        roi3d_b200._lib.set_tuning(11, 0)


def test_decode_matches_oracle(oracle, dev):
    from roi3d_b200 import AnchorGenerator3D
    from roi3d_b200.models.anchor_heads import decode_proposals
    rng = np.random.default_rng(42)
    A, D, H, W = 3, 5, 6, 7
    gen = AnchorGenerator3D(8, [2, 4, 8], [2, 3, 4], [1.0], 4)
    assert gen.num_base_anchors == 3
    reg = (0.5 * rng.standard_normal((6 * A, D, H, W))).astype(np.float32)
    reg[:, 0, 0, 0] = 50.0          # exercises the ratio clamp
    n_all = A * D * H * W
    idx = rng.permutation(n_all)[:150].astype(np.int64)
    idx[7] = -1
    sc = rng.uniform(0, 1, 150).astype(np.float32)
    img_shape = (48, 56, 3, 20)
    anchors = oracle.grid_anchors(oracle.gen_base_anchors(8, [2, 4, 8], [2, 3, 4], [1.0], 4), (D, H, W), 8, 4)
    assert np.array_equal(gen.grid_anchors((D, H, W), 8, 4, device=dev).cpu().numpy(), anchors)
    deltas = np.transpose(reg, (2, 3, 1, 0)).reshape(-1, 6)
    means, stds = (0.0, 0.1, 0, 0, 0, 0), (1.0, 0.5, 1, 1, 2, 1)
    sel = np.where(idx >= 0, idx, 0)
    want = oracle.delta2bbox3d(anchors[sel], deltas[sel], means, stds, img_shape)
    got = decode_proposals(torch.from_numpy(reg).to(dev), gen.base_anchors, 8, 4, torch.from_numpy(idx).to(dev),
                           torch.from_numpy(sc).to(dev), means, stds, img_shape).cpu().numpy()
    ok = idx >= 0
    assert np.abs(got[ok, :6] - want[ok]).max() <= 1e-3      # expf last-bit differences only (glibc vs CUDA)
    assert np.array_equal(got[ok, 6], sc[ok]) and np.all(got[~ok] == 0)
    # against today's torch CUDA ops evaluating the reference's expression (transforms.py:105-160) on the same device:
    # every step is an fp32 elementwise kernel there, and the fused kernels keep its operation order -> bit-exact
    tw = _torch_delta2bbox3d(torch.from_numpy(anchors[sel]).to(dev), torch.from_numpy(deltas[sel]).to(dev), means, stds,
                             img_shape).cpu().numpy()
    assert np.array_equal(got[ok, :6], tw[ok])
    # the bbox head's decode entry (class-wise deltas [n, 6k]) against the same expression
    from roi3d_b200 import delta2bbox3D
    rois_t = torch.from_numpy(anchors[sel]).to(dev)
    d3 = torch.from_numpy(np.concatenate([deltas[sel], 0.5 * deltas[sel][::-1], 3.0 * deltas[sel]], 1).astype(np.float32)).to(dev)
    for shape in (img_shape, None):
        mine = delta2bbox3D(rois_t, d3, means, stds, shape)
        ref = _torch_delta2bbox3d(rois_t, d3, means, stds, shape)
        assert mine.shape == d3.shape and torch.equal(mine, ref)
    assert delta2bbox3D(rois_t[:0], d3[:0], means, stds, img_shape).shape == (0, 18)


def _torch_delta2bbox3d(rois, deltas, means, stds, max_shape, wh_ratio_clip=16 / 1000):
    """The reference's delta2bbox3D expression (mmdet/core/bbox/transforms.py:105-160) with today's torch ops: the
    yardstick for the fused decode kernels (the reference ran it on torch 1.0.1 CUDA kernels, not available here)."""
    k = deltas.size(1) // 6
    d = deltas * deltas.new_tensor(stds).repeat(1, k) + deltas.new_tensor(means).repeat(1, k)
    mr = float(np.abs(np.log(wh_ratio_clip)))
    ctr, size = {}, {}
    for name, lo, hi in (("x", 0, 2), ("y", 1, 3), ("z", 4, 5)):
        p_c = ((rois[:, lo] + rois[:, hi]) * 0.5).unsqueeze(1)
        p_s = (rois[:, hi] - rois[:, lo] + 1.0).unsqueeze(1)
        size[name] = p_s * d[:, hi::6].clamp(-mr, mr).exp()
        ctr[name] = p_c + p_s * d[:, lo::6]
    lims = None if max_shape is None else {"x": max_shape[1] - 1, "y": max_shape[0] - 1, "z": max_shape[3] - 1}
    cols = {}
    for name in ("x", "y", "z"):
        v1 = ctr[name] - size[name] * 0.5 + 0.5
        v2 = ctr[name] + size[name] * 0.5 - 0.5
        if lims is not None:
            v1, v2 = v1.clamp(0, lims[name]), v2.clamp(0, lims[name])
        cols[name] = (v1, v2)
    return torch.stack([cols["x"][0], cols["y"][0], cols["x"][1], cols["y"][1], cols["z"][0], cols["z"][1]],
                       dim=-1).view_as(deltas)


def _rpn_inputs(B, dims, seed):
    rng = np.random.default_rng(seed)
    cls = [(2 * rng.standard_normal((B, 1) + d)).astype(np.float32) for d in dims]
    reg = [(0.1 * rng.standard_normal((B, 6) + d)).astype(np.float32) for d in dims]
    return cls, reg


def test_rpn_get_bboxes_matches_oracle(oracle, dev):
    from roi3d_b200 import RPNProposal3D
    B = 2
    dims = [(8, 16, 16), (4, 8, 8), (2, 4, 4)]
    strides, dstrides = [4, 8, 16], [2, 4, 8]
    cls, reg = _rpn_inputs(B, dims, 50)
    cfg = dict(nms_pre=300, nms_post=100, max_num=150, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=strides,
                         anchor_strides_depth=dstrides)
    metas = [dict(img_shape=(64, 64, 3, 16), scale_factor=1.0)] * B
    got, anchors_list = head.get_bboxes([torch.from_numpy(c).to(dev) for c in cls],
                                        [torch.from_numpy(r).to(dev) for r in reg], metas, cfg)
    assert len(got) == B and len(anchors_list) == B   # the reference's (result_list, anchors_list) pair
    for b in range(B):
        anchors = [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
                   for d, s, ds in zip(dims, strides, dstrides)]
        want = oracle.get_bboxes_single([c[b] for c in cls], [r[b] for r in reg], anchors, (64, 64, 3, 16),
                                        300, 100, 150, 0.7)
        g = got[b].cpu().numpy()
        assert g.shape == want.shape
        assert np.abs(g - want).max() <= 1e-3


@pytest.mark.parametrize("which", ["pos_indices", "pos_indices_test", "shape_mismatch", "few_left"])
def test_rpn_get_bboxes_pos_indices_filter(oracle, dev, which):
    """The head's cached inside-flag masks (anchor_head_3d.py:212,239-243) as rpn_head_3d.py:97-106 applies them: only
    on levels with more than nms_pre anchors, only when the mask has the scores' shape; a level left with no more than
    nms_pre anchors after masking is not sorted."""
    from roi3d_b200 import RPNProposal3D
    dims = [(8, 16, 16), (4, 8, 8), (2, 4, 4)]
    strides, dstrides = [4, 8, 16], [2, 4, 8]
    cls, reg = _rpn_inputs(1, dims, 51)
    nms_pre = 300
    cfg = dict(nms_pre=nms_pre, nms_post=100, max_num=150, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=strides,
                         anchor_strides_depth=dstrides)
    rng = np.random.default_rng(52)
    keep_frac = 0.1 if which == "few_left" else 0.6     # few_left: level 0 keeps ~200 < nms_pre of its 2048 anchors
    masks = [(rng.random(int(np.prod(d))) < keep_frac).astype(np.uint8) for d in dims]
    if which == "shape_mismatch":
        masks = [m[None].repeat(2, 0) for m in masks]    # [imgs, n] as images_to_levels leaves it for 2 images: ignored
    kw = {"pos_indices_test" if which == "pos_indices_test" else "pos_indices": masks}
    setattr(head, "pos_indices_test" if which == "pos_indices_test" else "pos_indices",
            [torch.from_numpy(m).to(dev) for m in masks])
    metas = [dict(img_shape=(64, 64, 3, 16), scale_factor=1.0)]
    got, _ = head.get_bboxes([torch.from_numpy(c).to(dev) for c in cls], [torch.from_numpy(r).to(dev) for r in reg],
                             metas, cfg)
    anchors = [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
               for d, s, ds in zip(dims, strides, dstrides)]
    want = oracle.get_bboxes_single([c[0] for c in cls], [r[0] for r in reg], anchors, (64, 64, 3, 16),
                                    nms_pre, 100, 150, 0.7, **kw)
    plain = oracle.get_bboxes_single([c[0] for c in cls], [r[0] for r in reg], anchors, (64, 64, 3, 16),
                                     nms_pre, 100, 150, 0.7)
    g = got[0].cpu().numpy()
    assert g.shape == want.shape and np.abs(g - want).max() <= 1e-3
    if which == "shape_mismatch":
        assert np.array_equal(want, plain)
    else:
        assert want.shape != plain.shape or not np.array_equal(want, plain)   # the mask really changed the proposals


@pytest.mark.parametrize("cfg_kw", [dict(nms_across_levels=True), dict(nms_pre=0, nms_post=60, max_num=90)])
def test_rpn_get_bboxes_across_levels_and_unsorted(oracle, dev, cfg_kw):
    """nms_across_levels=True (rpn_head_3d.py:140-142) and nms_pre <= 0 (no level is sorted: NMS sees anchor order and
    `proposals[:nms_post]` cuts in that order)."""
    from roi3d_b200 import RPNProposal3D
    B = 2
    dims = [(6, 12, 12), (3, 6, 6)]
    strides, dstrides = [4, 8], [2, 4]
    cls, reg = _rpn_inputs(B, dims, 53)
    cfg = dict(nms_pre=200, nms_post=100, max_num=120, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    cfg.update(cfg_kw)
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=strides,
                         anchor_strides_depth=dstrides)
    metas = [dict(img_shape=(48, 48, 3, 12), scale_factor=1.0)] * B
    got = head.get_proposals([torch.from_numpy(c).to(dev) for c in cls], [torch.from_numpy(r).to(dev) for r in reg],
                             metas, cfg)
    for b in range(B):
        anchors = [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
                   for d, s, ds in zip(dims, strides, dstrides)]
        want = oracle.get_bboxes_single([c[b] for c in cls], [r[b] for r in reg], anchors, (48, 48, 3, 12),
                                        cfg['nms_pre'], cfg['nms_post'], cfg['max_num'], 0.7,
                                        nms_across_levels=cfg['nms_across_levels'])
        g = got[b].cpu().numpy()
        assert g.shape == want.shape
        assert np.abs(g - want).max() <= 1e-3


def test_layout_conversion_reuse_is_scoped_and_sees_rewrites(oracle, dev):
    """NCDHW inputs are converted on every call unless the caller opens a reuse scope; a buffer rewritten through its
    address (what a CUDA-graph replay does: `_version` does not change) is therefore never served stale."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 2)
    # W = 18 is not a multiple of 4, so this NCDHW input cannot be read natively and is converted to channels-last
    f = torch.from_numpy(_feats((1, 64, 8, 16, 18), 60)).to(dev)
    rois = torch.from_numpy(synth.c2_rois(12, seed=61, img=(72, 64, 16))).to(dev)
    a = layer(f, rois)
    v0 = f._version
    raw = torch.from_numpy(_feats((1, 64, 8, 16, 18), 62)).to(dev)
    # rewrite the same storage without touching the version counter (a kernel writing through data_ptr)
    torch.cuda.current_stream().synchronize()
    f.data.copy_(raw)
    assert f._version == v0
    b = layer(f, rois)
    assert rel_err(b.cpu().numpy(), oracle.roi_align3d_forward(raw.cpu().numpy(), rois.cpu().numpy(), 7, 7, 0.25, 0.5, 2)) <= FWD_TOL
    assert not torch.equal(a, b)
    with roi3d_b200.reuse_layout_conversions():
        c1 = layer(f, rois)
        c2 = layer(f, rois)          # second call reuses the converted copy
        assert torch.equal(c1, c2) and torch.equal(c1, b)
        assert len(roi3d_b200._util._scopes[-1]) == 1
    assert not roi3d_b200._util._scopes


def test_multiclass_nms_matches_oracle(oracle, dev):
    from roi3d_b200 import multiclass_nms_3d
    rng = np.random.default_rng(60)
    n = 400
    d = synth.c1_boxes(n, seed=61)
    s1 = d[:, 6]
    s2 = rng.permutation(s1)
    scores = np.stack([1 - s1, s1, s2], 1).astype(np.float32)
    boxes = np.concatenate([d[:, :6] * 0, d[:, :6], d[:, :6] + 1.5], 1).astype(np.float32)
    for max_num in (2000, 37):
        want_b, want_l = oracle.multiclass_nms_3d(boxes, scores, 0.2, 0.5, max_num)
        got_b, got_l = multiclass_nms_3d(torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev), 0.2,
                                         dict(type='nms', iou_thr=0.5), max_num)
        assert np.array_equal(got_b.cpu().numpy(), want_b)
        assert np.array_equal(got_l.cpu().numpy(), want_l)
    got_b, got_l = multiclass_nms_3d(torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev), 5.0,
                                     dict(type='nms', iou_thr=0.5), 10)
    assert got_b.shape == (0, 7) and got_l.shape == (0,)


def test_roi_align_forward_wide_rois(oracle, dev):
    """RoIs wider than the 18-voxel row ring / the 40-voxel tables take the literal path: same tolerance."""
    from roi3d_b200.ops import RoIAlign3D
    shape = (1, 64, 8, 40, 72)
    f = _feats(shape, 12)
    rois = np.array([[0, 2, 3, 250, 120, 1, 12],       # 62 voxels wide: tables too small -> literal path
                     [0, 10, 8, 140, 150, 2, 14],      # 33 x 36 voxels
                     [0, 100.5, 20.25, 200, 60, 0, 9],  # 25 voxels wide
                     [0, 30, 30, 60, 60, 3, 8]], np.float32)
    for ps, pdp in [(7, 7), (14, 14)]:
        want = oracle.roi_align3d_forward(f, rois, ps, pdp, 0.25, 0.5, 2)
        out = RoIAlign3D(ps, pdp, 0.25, 0.5, 2)(cl(torch.from_numpy(f).to(dev)), torch.from_numpy(rois).to(dev))
        assert rel_err(out.cpu().numpy(), want) <= FWD_TOL


def test_reference_config_roi_stage(oracle, dev):
    """C5 harness at a small volume: the reference's config dicts build the drop-in modules unchanged and the whole
    RoI stage runs; the hot-path pieces inside it are re-checked against the oracle."""
    import roi3d_b200
    import roi_stage
    stage = roi_stage.RoIStage(max_masks=20).to(dev)
    assert stage.bbox_ex.roi_layers[0].out_size == 7 and stage.bbox_ex.roi_layers[0].out_size_depth == 3
    assert stage.mask_ex.roi_layers[3].spatial_scale == 1 / 32
    feats, cls, reg, metas = roi_stage.synthetic_inputs(1, vol_dhw=(32, 128, 128), device=dev)
    out = stage(feats, cls, reg, metas)
    det, lab, masks = out[0]
    assert det.shape[1] == 7 and lab.dtype == torch.int64 and det.shape[0] == lab.shape[0]
    assert det.shape[0] > 0, "random heads should leave some detections above score_thr=0.2"
    assert masks.shape[1:] == (2, 20, 28, 28)          # deconv doubles 10x14x14 (mask_size 28 / depth 20, config :121-122)
    # the extractor inside the stage vs the oracle, on the stage's own proposals
    props = stage.rpn.get_proposals(cls, reg, metas, roi_stage.TEST_CFG_RPN)
    rois = roi3d_b200.bbox2roi3D(props)[:64].contiguous()
    got = stage.bbox_ex(feats[:4], rois).cpu().numpy()
    rn = rois.cpu().numpy()
    lv = oracle.map_roi_levels(rn, 4)
    want = np.zeros_like(got)
    for l, (s, ds) in enumerate(zip([4, 8, 16, 32], [2, 4, 8, 16])):
        sel = lv == l
        if sel.any():
            want[sel] = oracle.roi_align3d_forward(feats[l].cpu().numpy(), rn[sel], 7, 3, 1 / s, 1 / ds, 2)
    assert rel_err(got, want) <= FWD_TOL


# --------------------------------------------------------------- full BASELINE sizes, size-independent properties
def test_c2_full_size_properties(oracle, dev):
    """BASELINE C2 at full size (256ch x 40x128x128, 512 RoIs): partition of unity, linearity, forward/backward
    adjointness, and a sampled check against the oracle on a channel subset."""
    from roi3d_b200.ops import RoIAlign3D
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    shape = (1, 256, 40, 128, 128)
    x = cl(torch.randn(shape, device=dev, generator=g))
    y = cl(torch.randn(shape, device=dev, generator=g))
    rois_np = synth.c2_rois(512, seed=2)
    rois = torch.from_numpy(rois_np).to(dev)
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 2)
    fx, fy = layer(x, rois), layer(y, rois)
    # every C2 RoI lies inside the map, so all 8 samples of every bin are valid: weights sum to one
    ones = layer(cl(torch.full(shape, 3.25, device=dev)), rois)
    assert float((ones - 3.25).abs().max()) <= 1e-5
    lin = layer(cl(2.0 * x - 0.5 * y), rois)
    assert float((lin - (2.0 * fx - 0.5 * fy)).abs().max()) <= 2e-5
    # sampled oracle check: 3 channels, all RoIs
    ch = [0, 101, 255]
    want = oracle.roi_align3d_forward(x[:, ch].cpu().numpy(), rois_np, 7, 7, 0.25, 0.5, 2)
    assert rel_err(fx[:, ch].cpu().numpy(), want) <= FWD_TOL
    # the same call on the reference's NCDHW tensor (read in place by the streamed kernel's NCDHW twin)
    xn = x.contiguous()
    assert xn.is_contiguous() and not xn.is_contiguous(memory_format=torch.channels_last_3d)
    fn = layer(xn, rois)
    assert float((fn - fx).abs().max()) <= 1e-5
    assert rel_err(fn[:, ch].cpu().numpy(), want) <= FWD_TOL
    del xn, fn
    # adjointness <f(x), g> == <x, f^T(g)> in float64
    xg = x.clone().requires_grad_(True)
    out = layer(xg, rois)
    gout = torch.randn(out.shape, device=dev, generator=g)
    out.backward(gout)
    lhs = float((out.detach().double() * gout.double()).sum())
    rhs = float((x.double() * xg.grad.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))


def test_c3_full_size_parity(oracle, dev):
    """BASELINE C3 at full size: mask branch 14x14x14 over 4 FPN levels (2 x 256 ch x {40x128x128 ... 5x16x16}), level
    mapping, 2 x 512 RoIs, forward AND backward.  The whole 2.9 GB output is produced on the device; the oracle checks
    three channels of every RoI (forward) and the three matching channel planes of every level's gradient (backward,
    with the other channels' grad_out zeroed), plus the level indices and a partition-of-unity pass."""
    from roi3d_b200 import SingleRoIExtractor
    B, C = 2, 256
    dims = [(40, 128, 128), (20, 64, 64), (10, 32, 32), (5, 16, 16)]
    strides, dstrides = [4, 8, 16, 32], [2, 4, 8, 16]
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)
    pyr = [cl(torch.randn((B, C) + d, device=dev, generator=gen)).requires_grad_(True) for d in dims]
    rois_np = synth.c3_rois(512, vols=B, seed=4)
    rois = torch.from_numpy(rois_np).to(dev)
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=14, out_size_depth=14, sample_num=2), C, strides, dstrides)
    lv = oracle.map_roi_levels(rois_np, 4)
    assert np.array_equal(ex.map_roi_levels(rois, 4).cpu().numpy(), lv)
    assert all((lv == l).sum() > 30 for l in range(4)), np.bincount(lv, minlength=4)   # all four levels populated
    out = ex(pyr, rois)
    assert out.shape == (1024, C, 14, 14, 14)
    ch = [0, 131, 255]
    got = out[:, ch].detach().cpu().numpy()
    want = np.zeros_like(got)
    for l in range(4):
        sel = lv == l
        f3 = pyr[l].detach()[:, ch].contiguous().cpu().numpy()
        want[sel] = oracle.roi_align3d_forward(f3, rois_np[sel], 14, 14, 1 / strides[l], 1 / dstrides[l], 2)
    assert rel_err(got, want) <= FWD_TOL
    # backward: gradient only through the three checked channels
    g3 = torch.randn((1024, 3, 14, 14, 14), device=dev, generator=gen)
    gout = torch.zeros_like(out)
    gout[:, ch] = g3
    out.backward(gout)
    del out, gout
    g3n = g3.cpu().numpy()
    for l in range(4):
        sel = lv == l
        wg = oracle.roi_align3d_backward(g3n[sel], rois_np[sel], (B, 3) + dims[l], 1 / strides[l], 1 / dstrides[l], 2)
        gl = pyr[l].grad
        assert rel_err(gl[:, ch].cpu().numpy(), wg) <= BWD_TOL
        others = [c for c in (1, 100, 254)]
        assert float(gl[:, others].abs().max()) == 0.0    # channels without grad_out receive nothing
    # weights of every bin sum to one wherever all samples fall inside the map
    ones = [cl(torch.full((B, 64) + d, 2.5, device=dev)) for d in dims]
    ex64 = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=14, out_size_depth=14, sample_num=2), 64, strides, dstrides)
    assert float((ex64(ones, rois) - 2.5).abs().max()) <= 1e-5


def test_c4_full_size_parity(oracle, dev):
    """BASELINE C4 at full size: 8 volumes of 512x512x160, 5 levels (1 310 720 ... 320 anchors, A = 1), nms_pre 2000,
    NMS 0.7, nms_post 1000, max_num 1000.  Per level the selected index sets and their order are exact against the
    oracle's stable top-k of torch-formula sigmoid scores; the final proposals match oracle.get_bboxes_single."""
    from roi3d_b200 import RPNProposal3D
    from roi3d_b200.models.anchor_heads import topk_segmented
    Bv = 8
    dims = [(80, 128, 128), (40, 64, 64), (20, 32, 32), (10, 16, 16), (5, 8, 8)]
    strides, dstrides = [4, 8, 16, 32, 64], [2, 4, 8, 16, 32]
    gen = torch.Generator(device=dev)
    gen.manual_seed(6)
    cls = [2 * torch.randn((Bv, 1) + d, device=dev, generator=gen) for d in dims]
    reg = [0.1 * torch.randn((Bv, 6) + d, device=dev, generator=gen) for d in dims]
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=strides,
                         anchor_strides_depth=dstrides)
    cfg = dict(nms_pre=2000, nms_post=1000, max_num=1000, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    metas = [dict(img_shape=(512, 512, 3, 160), scale_factor=1.0)] * Bv
    props = head.get_proposals(cls, reg, metas, cfg)
    # (1) per-level top-k: index sets and order, all 8 volumes of the three levels that are top-k'd
    segs = [cls[l][b] for b in range(Bv) for l in range(3)]
    idx, val = topk_segmented(segs, 2000, apply_sigmoid=True, permute_adhw=True, small_in_index_order=True)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    j = 0
    for b in range(Bv):
        for l in range(3):
            sc = cls[l][b].permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy()   # rpn_head_3d.py:87-90, on CUDA
            want = oracle.topk(sc, 2000)
            assert np.array_equal(idx[j], want), (b, l)
            assert np.array_equal(val[j], sc[want])
            j += 1
    # (2) final proposals of every volume
    anchors = [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
               for d, s, ds in zip(dims, strides, dstrides)]
    for b in range(Bv):
        # scores from the reference's own expression on CUDA (rpn_head_3d.py:87-90): glibc's expf can differ from the
        # device's in the last bit, which would reorder near-ties of the final top-k
        sc = [c[b].permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy() for c in cls]
        want = oracle.get_bboxes_single([c[b].cpu().numpy() for c in cls], [r[b].cpu().numpy() for r in reg], anchors,
                                        (512, 512, 3, 160), 2000, 1000, 1000, 0.7, scores=sc)
        g = props[b].cpu().numpy()
        assert g.shape == want.shape, (b, g.shape, want.shape)
        assert np.array_equal(g[:, 6], want[:, 6])     # scores exact: the same selection in the same order
        assert np.abs(g[:, :6] - want[:, :6]).max() <= 1e-3


def test_c1_full_size_properties(oracle, dev):
    """BASELINE C1 (2000 clustered boxes, thr 0.7): bit-exact keep, ascending order, idempotence, and no kept pair
    overlaps above the threshold."""
    from roi3d_b200.ops import nms
    dets = synth.c1_boxes(2000, seed=0)
    t = torch.from_numpy(dets).to(dev)
    kept, inds = nms(t, 0.7)
    assert np.array_equal(inds.cpu().numpy(), oracle.nms3d(dets, 0.7))
    assert bool((inds[1:] > inds[:-1]).all())
    kept2, inds2 = nms(kept, 0.7)
    assert inds2.numel() == kept.shape[0] and torch.equal(kept2, kept)
    k = kept.cpu().numpy()
    order = np.argsort(-k[:, 6], kind="stable")
    k = k[order]
    for i in range(0, len(k), 97):
        for j in range(i + 1, min(i + 40, len(k))):
            assert not oracle.iou3d(k[i, :6], k[j, :6]) > 0.7


def test_topk_full_p2_level_and_large_segment(oracle, dev):
    """Top-k over a full P2 level (1.31 M scores) and a 4.4 M-score segment (1.5x scale): same values as
    torch.topk, indices exact against the oracle's tie rule."""
    from roi3d_b200.models.anchor_heads import topk_segmented
    g = torch.Generator(device=dev)
    g.manual_seed(6)
    for n, k in [(80 * 128 * 128, 2000), (4423680, 2000)]:
        s = 2 * torch.randn(n, device=dev, generator=g)
        idx, val = topk_segmented([s], k)
        tv, ti = torch.topk(s, k)
        assert torch.equal(val[0], tv)
        assert torch.equal(s[idx[0]], tv)
        want = oracle.topk(s.cpu().numpy(), k)
        assert np.array_equal(idx[0].cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["NCDHW", "NDHWC"])
@pytest.mark.parametrize("pipeline_kb", [-1, 1])
def test_roi_align_host_entry(oracle, dev, layout, pipeline_kb):
    """roi3d_roi_align3d_forward_host (numpy in / out): the plain path and the z-slab pipelined path (forced on a
    small volume through tuning key 4) give the device path's bits and the oracle's values; RoIs that are empty,
    out of the volume or NaN still land in their own output rows."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D, roi_align_3d_host
    shape = (1, 64, 24, 20, 28)
    f = _feats(shape, 21)
    rois = np.concatenate([synth.c2_rois(96, seed=5, img=(112, 80, 48)),
                           synth.adversarial_rois(shape[2:], 0.25, 0.5)], 0)
    rois = rois[np.random.RandomState(0).permutation(len(rois))]
    want = oracle.roi_align3d_forward(f, rois, 7, 7, 0.25, 0.5, 2)
    dev_out = RoIAlign3D(7, 7, 0.25, 0.5, 2)(cl(torch.from_numpy(f).to(dev)), torch.from_numpy(rois).to(dev))
    src = f if layout == "NCDHW" else np.ascontiguousarray(f.transpose(0, 2, 3, 4, 1))
    pinned = torch.empty(dev_out.shape, dtype=torch.float32).pin_memory()  # mapped: the kernels store into it directly
    roi3d_b200._lib.set_tuning(4, pipeline_kb)
    try:
        got = roi_align_3d_host(src, rois, 7, 7, 0.25, 0.5, 2, layout=layout)
        again = roi_align_3d_host(src, rois, 7, 7, 0.25, 0.5, 2, layout=layout, out=pinned.numpy())
    finally:
        roi3d_b200._lib.set_tuning(4, 0)
    assert np.array_equal(got, dev_out.cpu().numpy(), equal_nan=True)
    assert np.array_equal(got, again, equal_nan=True)
    assert rel_err(got, want) <= FWD_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("out_size", [7, 14, 5])
def test_roi_align_forward_row_map(dev, out_size):
    """roi3d_roi_align3d_forward_rows: RoI k lands in output row out_rows[k], bit-identical to the plain call
    (ring kernels for 7 / 14 wide outputs, literal kernels for other widths, wide RoIs included)."""
    import roi3d_b200
    from roi3d_b200 import _lib
    from roi3d_b200.ops import RoIAlign3D
    from roi3d_b200._util import stream_ptr
    shape = (1, 64, 12, 40, 72)
    f = cl(torch.from_numpy(_feats(shape, 31)).to(dev))
    rois_np = np.concatenate([synth.c2_rois(40, seed=9, img=(288, 160, 24)),
                              np.array([[0, 2, 3, 250, 120, 1, 12]], np.float32)], 0)
    rois = torch.from_numpy(rois_np).to(dev)
    K = rois.shape[0]
    plain = RoIAlign3D(out_size, out_size, 0.25, 0.5, 2)(f, rois)
    perm = torch.randperm(K, generator=torch.Generator().manual_seed(1)).to(torch.int32).to(dev)
    out = torch.full_like(plain, float("nan"))
    fcl = f.permute(0, 2, 3, 4, 1)
    assert fcl.is_contiguous()
    _lib.check(_lib.lib.roi3d_roi_align3d_forward_rows(
        fcl.data_ptr(), _lib.NDHWC, 1, 64, 12, 40, 72, rois.data_ptr(), K, out_size, out_size, out_size, 0.25, 0.5, 2,
        out.data_ptr(), perm.data_ptr(), stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(out[perm.long()], plain)
    if out_size in (7, 14):
        # the same row map over the reference's NCDHW tensor (streamed kernel's NCDHW twin / planar kernel)
        fn = f.contiguous()
        plain_n = RoIAlign3D(out_size, out_size, 0.25, 0.5, 2)(fn, rois)
        out_n = torch.full_like(plain, float("nan"))
        _lib.check(_lib.lib.roi3d_roi_align3d_forward_rows(
            fn.data_ptr(), _lib.NCDHW, 1, 64, 12, 40, 72, rois.data_ptr(), K, out_size, out_size, out_size, 0.25, 0.5, 2,
            out_n.data_ptr(), perm.data_ptr(), stream_ptr()))
        torch.cuda.synchronize()
        assert torch.equal(out_n[perm.long()], plain_n)
        assert float((plain_n - plain).abs().max()) <= 1e-5


# ---------------------------------------------------------------------------------------------------------------
# SURVEY 8f N1: evaluation-time NMS (coco_utils.py:245-332) on the device, float64 IoU in numpy's operation order
# ---------------------------------------------------------------------------------------------------------------
def _eval_volumes(nvol, seed):
    rng = np.random.RandomState(seed)
    vols = []
    for v in range(nvol):
        n = int(rng.randint(0, 400)) if v else 300
        b = synth.c1_boxes(max(n, 1), seed=seed + v)[:n]
        if n:
            b[:, 6] = rng.permutation(np.linspace(0.05, 0.99, n)).astype(np.float32)
        vols.append(b)
    return vols


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.1, 0.3, 0.0])
def test_eval_nms_matches_numpy_reference(oracle, dev, thr):
    from roi3d_b200.core.evaluation import nms_3d_eval_batched
    vols = _eval_volumes(9, 40)
    # boxes whose IoU sits exactly on / next to the threshold in float64: identical boxes shifted by whole voxels
    edge = np.array([[0, 0, 9, 9, 0, 9, 0.9], [0, 0, 9, 9, 0, 9, 0.8], [9, 0, 18, 9, 0, 9, 0.7],
                     [0, 0, 9, 9, 8, 17, 0.6], [100, 100, 100, 100, 50, 50, 0.5], [100, 100, 100, 100, 50, 50, 0.5]],
                    np.float32)
    vols.append(edge)
    got = nms_3d_eval_batched(vols, thr, device=dev)
    assert len(got) == len(vols)
    for b, g in zip(vols, got):
        want = oracle.nms_3d_python(b.astype(np.float64), thr)
        assert np.array_equal(g, want)


@pytest.mark.gpu
def test_eval_nms_nan_box_is_dropped_like_numpy(oracle, dev):
    from roi3d_b200.core.evaluation import nms_3d_eval_batched
    b = synth.c1_boxes(64, seed=3)
    b[:, 6] = np.linspace(0.99, 0.1, 64, dtype=np.float32)
    b[10, 2] = np.nan
    with np.errstate(invalid="ignore"):
        want = oracle.nms_3d_python(b.astype(np.float64), 0.1)
    got = nms_3d_eval_batched([b], 0.1, device=dev)[0]
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_apply_nms_matches_reference_restatement(oracle, dev):
    """apply_nms over json-style results of several volumes (interleaved, one volume without detections)."""
    from roi3d_b200.core.evaluation import apply_nms, nms_3d_python
    vols = _eval_volumes(5, 60)
    name_to_id = {"vol%d.npy" % v: 100 + v for v in range(len(vols) + 1)}  # one extra volume with no results
    results = []
    for v, b in enumerate(vols):
        for i, row in enumerate(b):
            results.append(dict(image_id=100 + v, original_bbox=[float(x) for x in row], score=float(row[6]),
                                category_id=1, tag=(v, i)))
    rng = np.random.RandomState(1)
    results = [results[i] for i in rng.permutation(len(results))]
    want = oracle.apply_nms(name_to_id, results, 0.1, 0.3)
    with torch.cuda.device(dev):
        got = apply_nms(name_to_id, results, 0.1, 0.3)
        one = nms_3d_python(results[:50], [r['original_bbox'] for r in results[:50]], 0.1)
    assert [r['tag'] for r in got] == [r['tag'] for r in want] and len(got) > 0
    keep = oracle.nms_3d_python(np.array([r['original_bbox'] for r in results[:50]]), 0.1)
    assert [r['tag'] for r in one] == [results[i]['tag'] for i in keep]


# ---------------------------------------------------------------------------------------------------------------
# SURVEY 8f N2: dense 3D IoU, MaxIoU assigner, bbox2delta3d
# ---------------------------------------------------------------------------------------------------------------
def _assign_case(n, k, seed, dup=True):
    rng = np.random.default_rng(seed)
    gt = synth.c1_boxes(max(k, 8), seed=seed)[:k, :6].copy()
    boxes = synth.c1_boxes(n, seed=seed + 1)[:, :7].copy()
    # make a good share of the boxes overlap some gt, some of them exactly
    take = rng.integers(0, k, n // 3)
    boxes[: n // 3, :6] = gt[take] + rng.integers(-4, 5, (n // 3, 6)).astype(np.float32)
    if dup:
        boxes[5, :6] = gt[0]
        boxes[6, :6] = gt[0]          # two boxes tie for gt 0's maximum
        if k > 2:
            gt[2] = gt[1]             # two gts tie for the same boxes' argmax
    return boxes, gt


@pytest.mark.gpu
def test_bbox_overlaps3d_matches_oracle_and_torch(oracle, dev):
    from roi3d_b200.core.bbox import bbox_overlaps
    boxes, gt = _assign_case(1500, 37, 3)
    want = oracle.bbox_overlaps3d(gt, boxes[:, :6])
    g, b = torch.from_numpy(gt).to(dev), torch.from_numpy(boxes).to(dev)
    got = bbox_overlaps(g, b)          # boxes carry a 7th (score) column: stride 7
    assert got.shape == (37, 1500)
    assert np.array_equal(got.cpu().numpy(), want)
    # the reference's expression evaluated by today's torch CUDA elementwise kernels
    b1, b2 = g, b[:, :6]
    xa, ya = torch.max(b1[:, None, 0], b2[:, 0]), torch.max(b1[:, None, 1], b2[:, 1])
    xb, yb = torch.min(b1[:, None, 2], b2[:, 2]), torch.min(b1[:, None, 3], b2[:, 3])
    za, zb = torch.max(b1[:, None, 4], b2[:, 4]), torch.min(b1[:, None, 5], b2[:, 5])
    inter = (xb - xa + 1).clamp(min=0) * (yb - ya + 1).clamp(min=0) * (zb - za + 1).clamp(min=0)
    a1 = (b1[:, 2] - b1[:, 0] + 1) * (b1[:, 3] - b1[:, 1] + 1) * (b1[:, 5] - b1[:, 4] + 1)
    a2 = (b2[:, 2] - b2[:, 0] + 1) * (b2[:, 3] - b2[:, 1] + 1) * (b2[:, 5] - b2[:, 4] + 1)
    assert torch.equal(got, inter / (a1[:, None] + a2 - inter))
    assert bbox_overlaps(g[:0], b).shape == (0, 1500)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [
    dict(pos_iou_thr=0.7, neg_iou_thr=0.3, min_pos_iou=0.3, gt_max_assign_all=True),     # rpn assigner of the config
    dict(pos_iou_thr=0.5, neg_iou_thr=0.5, min_pos_iou=0.5, gt_max_assign_all=True),     # rcnn assigner
    dict(pos_iou_thr=0.6, neg_iou_thr=(0.1, 0.4), min_pos_iou=0.2, gt_max_assign_all=False),
])
@pytest.mark.parametrize("shape", [(3000, 12), (257, 1), (70000, 700)])
def test_max_iou_assigner_matches_oracle(oracle, dev, cfg, shape):
    from roi3d_b200.core.bbox import MaxIoUAssigner
    n, k = shape
    boxes, gt = _assign_case(n, k, 11 + k)
    labels = (np.arange(k) % 3 + 1).astype(np.int64)
    want_a, want_mo, want_l = oracle.assign_max_iou(boxes, gt, labels, **cfg)
    res = MaxIoUAssigner(**cfg).assign(torch.from_numpy(boxes).to(dev), torch.from_numpy(gt).to(dev),
                                       gt_labels=torch.from_numpy(labels).to(dev))
    assert res.num_gts == k and res.gt_inds.dtype == torch.int64 and res.labels.dtype == torch.int64
    assert np.array_equal(res.max_overlaps.cpu().numpy(), want_mo)
    assert np.array_equal(res.gt_inds.cpu().numpy(), want_a)
    assert np.array_equal(res.labels.cpu().numpy(), want_l)
    assert (want_a > 0).sum() > 0 and (want_a == 0).sum() > 0
    res2 = MaxIoUAssigner(**cfg).assign(torch.from_numpy(boxes).to(dev), [torch.from_numpy(gt).to(dev)])
    assert res2.labels is None and torch.equal(res2.gt_inds, res.gt_inds)


@pytest.mark.gpu
@pytest.mark.parametrize("wrt_candidates", [True, False])
@pytest.mark.parametrize("assign_all", [True, False])
def test_max_iou_assigner_ignore_regions(oracle, dev, wrt_candidates, assign_all):
    """The ignore-region branch (max_iou_assigner.py:101-111): boxes whose overlap with an ignore box exceeds
    ignore_iof_thr read -1 against every gt and stay "don't care" -- also when they would have been a gt's best box."""
    from roi3d_b200.core.bbox import MaxIoUAssigner
    n, k = 5000, 9
    boxes, gt = _assign_case(n, k, 31)
    labels = (np.arange(k) % 3 + 1).astype(np.int64)
    rng = np.random.default_rng(5)
    # ignore regions: two copies of gt boxes (so that some would-be positives are ignored) and two random boxes
    extra = boxes[rng.choice(n, 2, replace=False), :6] + np.float32(1.0)
    ign = np.concatenate([gt[[1, 4], :6], extra], 0).astype(np.float32)
    cfg = dict(pos_iou_thr=0.5, neg_iou_thr=0.3, min_pos_iou=0.2, gt_max_assign_all=assign_all, ignore_iof_thr=0.4,
               ignore_wrt_candidates=wrt_candidates)
    want_a, want_mo, want_l = oracle.assign_max_iou(boxes, gt, labels, gt_bboxes_ignore=ign, **cfg)
    plain_a, _, _ = oracle.assign_max_iou(boxes, gt, labels, **{**cfg, 'ignore_iof_thr': -1})
    assert (want_a != plain_a).sum() > 0 and (want_mo == -1).sum() > 0   # the branch changes something here
    res = MaxIoUAssigner(**cfg).assign(torch.from_numpy(boxes).to(dev), torch.from_numpy(gt).to(dev),
                                       gt_bboxes_ignore=torch.from_numpy(ign).to(dev), gt_labels=torch.from_numpy(labels).to(dev))
    assert np.array_equal(res.max_overlaps.cpu().numpy(), want_mo)
    assert np.array_equal(res.gt_inds.cpu().numpy(), want_a)
    assert np.array_equal(res.labels.cpu().numpy(), want_l)
    # an empty ignore list, or ignore_iof_thr <= 0, is the plain assigner
    res0 = MaxIoUAssigner(**cfg).assign(torch.from_numpy(boxes).to(dev), torch.from_numpy(gt).to(dev),
                                        gt_bboxes_ignore=torch.zeros(0, 6, device=dev))
    assert np.array_equal(res0.gt_inds.cpu().numpy(), plain_a)


@pytest.mark.gpu
def test_max_iou_assigner_errors_like_reference(dev):
    from roi3d_b200.core.bbox import MaxIoUAssigner
    a = MaxIoUAssigner(0.5, 0.5)
    with pytest.raises(ValueError):
        a.assign(torch.zeros(0, 6, device=dev), torch.zeros(2, 6, device=dev))
    with pytest.raises(ValueError):
        a.assign(torch.zeros(4, 6, device=dev), torch.zeros(0, 6, device=dev))
    with pytest.raises(NotImplementedError):
        a.assign(torch.zeros(4, 6), torch.zeros(1, 6))


@pytest.mark.gpu
def test_bbox2delta3d_matches_oracle(oracle, dev):
    from roi3d_b200.core.bbox import bbox2delta3d, delta2bbox3D
    rng = np.random.default_rng(0)
    lo, sz = rng.uniform(0, 400, (4000, 3)).astype(np.float32), rng.uniform(4, 60, (4000, 3)).astype(np.float32)
    p = np.stack([lo[:, 0], lo[:, 1], lo[:, 0] + sz[:, 0], lo[:, 1] + sz[:, 1], lo[:, 2], lo[:, 2] + sz[:, 2]], 1)
    g = p + rng.uniform(-1.5, 1.5, p.shape).astype(np.float32)
    means, stds = (0.0, 0.0, 0.0, 0.0, 0.0, 0.0), (0.1, 0.1, 0.2, 0.2, 0.1, 0.2)
    want = oracle.bbox2delta3d(p, g, means, stds)
    got = bbox2delta3d(torch.from_numpy(p).to(dev), torch.from_numpy(g).to(dev), means, stds)
    gn = got.cpu().numpy()
    # dx, dy, dz are pure IEEE arithmetic: exact; dw, dh, dd go through logf (device libm vs numpy's)
    assert np.array_equal(gn[:, [0, 1, 4]], want[:, [0, 1, 4]])
    assert np.isfinite(want).all()
    assert np.allclose(gn[:, [2, 3, 5]], want[:, [2, 3, 5]], rtol=1e-5, atol=1e-6)  # tolerance: 1e-5 relative
    back = delta2bbox3D(torch.from_numpy(p).to(dev), got, means, stds)
    assert (back - torch.from_numpy(g).to(dev)).abs().max() < 1e-2


# ---------------------------------------------------------------------------------------------------------------
# SURVEY 8f N3: anchors in closed form + valid / inside flags on the device
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", [
    # (featmap D,H,W), stride, depth stride, scales, depth scales, ratios, valid (d,h,w), img_shape (H,W,3,D), border
    ((5, 8, 6), 8, 4, [2], [2], [1.0], (5, 7, 6), (56, 48, 3, 20), 0),
    ((7, 9, 11), 4, 2, [2, 4], [2, 3], [0.5, 1.0, 2.0], (6, 9, 10), (36, 42, 3, 13), 3),
    ((3, 4, 5), 16, 8, [8], [2], [1.0], (3, 4, 5), (64, 80, 3, 24), -1),
])
def test_grid_anchors_and_inside_flags_match_oracle(oracle, dev, case):
    from roi3d_b200 import AnchorGenerator3D
    from roi3d_b200.core.anchor import anchor_inside_flags
    fm, st, sd, scales, dscales, ratios, valid, img_shape, border = case
    gen = AnchorGenerator3D(st, scales, dscales, ratios, sd)
    base = oracle.gen_base_anchors(st, scales, dscales, ratios, sd)
    assert np.array_equal(gen.base_anchors.numpy(), base)
    want_a = oracle.grid_anchors(base, fm, st, sd)
    want_v = oracle.valid_flags(fm, valid, base.shape[0])
    want_f = oracle.anchor_inside_flags(want_a, want_v, img_shape, border)
    got_a = gen.grid_anchors(fm, st, sd, device=dev)
    assert np.array_equal(got_a.cpu().numpy(), want_a)
    got_v = gen.valid_flags(fm, valid, device=dev)
    assert got_v.dtype == torch.uint8 and np.array_equal(got_v.cpu().numpy(), want_v)
    a2, f2 = gen.grid_anchors_and_inside_flags(fm, st, sd, valid, img_shape, border, device=dev)
    assert torch.equal(a2, got_a) and np.array_equal(f2.cpu().numpy(), want_f)
    assert torch.equal(anchor_inside_flags(got_a, got_v, img_shape, border), f2)
    if border >= 0:
        assert 0 < int(f2.sum()) < f2.numel()


STREAM_CASES = [
    # (B, C, D, H, W), out_size_depth, scale, scale_d, sample_num, n_rois, roi image size (W, H, D)
    ((2, 128, 10, 24, 40), 7, 0.25, 0.5, 2, 120, (160, 96, 20)),    # two chunks, more items than SMs
    ((1, 64, 12, 40, 40), 3, 0.25, 0.5, 2, 60, (160, 160, 24)),     # real-config bbox shape 7x7x3
    ((1, 64, 24, 96, 96), 7, 0.25, 0.5, 2, 40, (384, 384, 48)),     # c2-sized RoIs: multi-tile items, x boxes up to 20
    ((1, 64, 10, 20, 20), 7, 0.25, 0.5, 0, 30, (80, 80, 20)),       # adaptive sampling (S = ceil(bin))
    ((2, 64, 6, 12, 12), 7, 0.125, 0.25, 3, 30, (96, 96, 24)),      # three samples per bin, coarse level
    ((1, 192, 9, 14, 15), 1, 0.25, 0.5, 1, 20, (60, 56, 18)),       # one output slice, one sample per bin
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", STREAM_CASES)
def test_roi_align_forward_streamed_kernel(oracle, dev, case):
    """The persistent TMA-fed kernel (7x7xPD outputs, C % 64 == 0, channels-last): oracle tolerance, and the per-warp
    ring kernel (tuning variant 50) on the same inputs beside it."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D
    shape, pdp, sc, scd, sn, k, img = case
    B, C, D, H, W = shape
    f = _feats(shape, 33)
    rois = np.concatenate([synth.c2_rois(k, seed=6, img=img, batch=B),
                           synth.adversarial_rois(shape[2:], sc, scd, batch=B),
                           np.array([[B - 1, 2, 3, img[0] - 4, img[1] - 6, 1, img[2] - 3]], np.float32)], 0)
    if sn == 0:
        ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
        rois = rois[ok]
    ft = cl(torch.from_numpy(f).to(dev))
    rt = torch.from_numpy(rois).to(dev)
    want = oracle.roi_align3d_forward(f, rois, 7, pdp, sc, scd, sn)
    layer = RoIAlign3D(7, pdp, sc, scd, sn)
    out = layer(ft, rt)
    assert rel_err(out.cpu().numpy(), want) <= FWD_TOL
    roi3d_b200._lib.set_tuning(0, 50)
    try:
        ring = layer(ft, rt)
    finally:
        roi3d_b200._lib.set_tuning(0, 0)
    assert rel_err(out.cpu().numpy(), ring.cpu().numpy()) <= FWD_TOL
    # a second call on the same buffers (cached tensor maps, recycled workspace) gives the same bits
    assert torch.equal(layer(ft, rt), out)
    # the NCDHW twin (cp.async producers, the reference's layout read in place; W % 4 == 0, otherwise the planar kernel
    # or the conversion path take the call): same owners with the x taps summed in a lane-rotated order
    fn = torch.from_numpy(f).to(dev)
    assert fn.is_contiguous()
    nat = layer(fn, rt)
    assert rel_err(nat.cpu().numpy(), want) <= FWD_TOL
    assert rel_err(nat.cpu().numpy(), out.cpu().numpy()) <= FWD_TOL
    assert torch.equal(layer(fn, rt), nat)


@pytest.mark.gpu
def test_roi_align_streamed_kernel_two_streams(oracle, dev):
    """Two streams run the streamed kernel concurrently on different inputs: per-call workspaces, no shared scratch."""
    from roi3d_b200.ops import RoIAlign3D
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 2)
    fs = [_feats((1, 64, 10, 32, 32), 40 + i) for i in range(2)]
    rs = [synth.c2_rois(150, seed=50 + i, img=(128, 128, 20)) for i in range(2)]
    want = [oracle.roi_align3d_forward(f, r, 7, 7, 0.25, 0.5, 2) for f, r in zip(fs, rs)]
    fts = [cl(torch.from_numpy(f).to(dev)) for f in fs]
    rts = [torch.from_numpy(r).to(dev) for r in rs]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
    outs = [None, None]
    for _ in range(3):
        for i, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs[i] = layer(fts[i], rts[i])
    torch.cuda.synchronize()
    for i in range(2):
        assert rel_err(outs[i].cpu().numpy(), want[i]) <= FWD_TOL


# ---------------------------------------------------------------------------------------------------------------
# SURVEY 8f N4: mask paste (sigmoid -> skimage-style resize to the box -> threshold) on the device
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mask_paste_matches_resize_restatement(oracle, dev):
    from roi3d_b200.models.mask_heads import get_seg_masks, paste_masks_compact
    rng = np.random.default_rng(70)
    n, ncls = 24, 3
    logits = (3 * rng.standard_normal((n, ncls, 10, 14, 14))).astype(np.float32)
    # smooth blobs make realistic masks; raw noise keeps many values near the threshold (harder test)
    lo = np.stack([rng.uniform(0, 200, n), rng.uniform(0, 200, n), rng.uniform(0, 60, n)], 1)
    sz = np.stack([rng.choice([1, 2, 3, 7, 14, 15, 33, 80], n), rng.choice([1, 3, 9, 14, 27, 50], n),
                   rng.choice([1, 2, 5, 10, 11, 24], n)], 1)
    det = np.stack([lo[:, 0], lo[:, 1], lo[:, 0] + sz[:, 0] - 0.3, lo[:, 1] + sz[:, 1] - 0.6, lo[:, 2],
                    lo[:, 2] + sz[:, 2] - 0.5, rng.random(n)], 1).astype(np.float32)
    labels = rng.integers(0, ncls - 1, n)
    want_b, want_m, want_l = oracle.get_seg_masks_compact(logits, det, labels, 0.5)
    got_b, got_m, got_l = paste_masks_compact(torch.from_numpy(logits).to(dev), torch.from_numpy(det).to(dev),
                                              torch.from_numpy(labels).to(dev), 0.5)
    assert np.array_equal(got_b, want_b) and np.array_equal(got_l, want_l)
    total = diff = 0
    for g, w in zip(got_m, want_m):
        assert g.shape == w.shape and g.dtype == np.uint8
        total += g.size
        diff += int((g != w).sum())
    # float64 arithmetic in scipy's order; a voxel can only differ when its value is within an ulp of the threshold
    assert diff <= max(1, total // 100000), "%d of %d mask voxels differ" % (diff, total)
    segs = get_seg_masks(torch.from_numpy(logits).to(dev), torch.from_numpy(det).to(dev),
                         torch.from_numpy(labels).to(dev), dict(mask_thr_binary=0.5), (320, 320, 120), 1.0, True, ncls)
    assert len(segs) == ncls - 1 and sum(len(s) for s in segs) == n
    i0 = int(np.nonzero(labels == 0)[0][0])
    vol = segs[0][0]
    b = want_b[i0]
    assert vol.shape == (120, 320, 320) and vol.sum() == got_m[i0].sum()
    assert np.array_equal(vol[b[4]:b[4] + got_m[i0].shape[0], b[1]:b[1] + got_m[i0].shape[1],
                              b[0]:b[0] + got_m[i0].shape[2]], got_m[i0])


@pytest.mark.gpu
def test_rpn_get_bboxes_cuda_graph_replay(dev):
    """cuda_graph=True: the captured path returns the eager path's proposals, also after the input buffers have been
    refilled in place (same addresses, new values) and for a second set of buffers."""
    from roi3d_b200 import RPNProposal3D
    dims = [(8, 16, 16), (4, 8, 8), (2, 4, 4)]
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=[4, 8, 16],
                         anchor_strides_depth=[2, 4, 8])
    cfg = dict(nms_pre=300, nms_post=100, max_num=150, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    metas = [dict(img_shape=(64, 64, 3, 16), scale_factor=1.0)] * 2
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    cls = [2 * torch.randn((2, 1) + d, device=dev, generator=g) for d in dims]
    reg = [0.1 * torch.randn((2, 6) + d, device=dev, generator=g) for d in dims]
    for rnd in range(3):
        head.cuda_graph = False
        want = head.get_proposals(cls, reg, metas, cfg)
        head.cuda_graph = True
        got = head.get_proposals(cls, reg, metas, cfg)
        assert len(got) == len(want) == 2
        for a, b in zip(got, want):
            assert torch.equal(a, b) and a.shape[0] > 0
        for t in cls + reg:   # new values at the same addresses: the replay must see them
            t.copy_(torch.randn(t.shape, device=dev, generator=g) * (2 if t.shape[1] == 1 else 0.1))
    assert len(head._graphs) == 1


@pytest.mark.gpu
def test_nms_presorted_segments_skip_the_ranking(oracle, dev):
    """Segments flagged presorted (rows already in descending-score order, ties by row) give the same keep lists as the
    ranked path; unflagged segments in the same call are still ranked."""
    from roi3d_b200.ops import nms3d_batched
    a = synth.c1_boxes(1500, seed=3)
    a = a[np.argsort(-a[:, 6], kind="stable")]
    a[100:140, 6] = a[100, 6]                       # a run of equal scores: order by row
    b = synth.c1_boxes(1500, seed=4)                # not sorted
    dets = torch.from_numpy(np.stack([a, b])).to(dev)
    flags = torch.tensor([1, 0], dtype=torch.uint8, device=dev)
    k0, s0, n0 = nms3d_batched(dets, None, 0.5)
    k1, s1, n1 = nms3d_batched(dets, None, 0.5, presorted=flags)
    assert torch.equal(n0, n1)
    for seg in range(2):
        m = int(n0[seg])
        assert torch.equal(k0[seg, :m], k1[seg, :m]) and torch.equal(s0[seg, :m], s1[seg, :m])
    assert np.array_equal(k1[0, :int(n1[0])].cpu().numpy(), oracle.nms3d(a, 0.5))


@pytest.mark.parametrize("max_keep", [1, 64, 100, 1000, 5000])
def test_nms_limited_sweep_returns_a_prefix(oracle, dev, max_keep):
    """roi3d_nms3d_batched_limited: a presorted segment's sweep stops with the 64-box tile in which the kept count
    reaches max_keep -- the lists are a prefix of the full result (what `proposals[:nms_post]` reads), unflagged
    segments and segments that never reach the limit are swept in full."""
    from roi3d_b200.ops import nms3d_batched
    segs = []
    for seed, n in ((3, 2000), (4, 2000), (5, 700), (6, 2000)):
        a = synth.c1_boxes(n, seed=seed)
        a = a[np.argsort(-a[:, 6], kind="stable")]
        segs.append(np.concatenate([a, np.zeros((2000 - n, 7), np.float32)]))
    segs[3] = synth.c1_boxes(2000, seed=6)              # unsorted, unflagged
    dets = torch.from_numpy(np.stack(segs)).to(dev)
    cnt = torch.tensor([2000, 2000, 700, 2000], dtype=torch.int32, device=dev)
    flags = torch.tensor([1, 1, 1, 0], dtype=torch.uint8, device=dev)
    k0, s0, n0 = nms3d_batched(dets, cnt, 0.5, presorted=flags)
    k1, s1, n1 = nms3d_batched(dets, cnt, 0.5, presorted=flags, max_keep=max_keep)
    for seg in range(4):
        full, got = int(n0[seg]), int(n1[seg])
        if seg == 3 or full <= max_keep:
            assert got == full and torch.equal(k0[seg, :full], k1[seg, :full]) and torch.equal(s0[seg, :full], s1[seg, :full])
            continue
        assert max_keep <= got <= min(full, max_keep + 63)
        assert torch.equal(s1[seg, :got], s0[seg, :got])                              # a prefix in score order
        assert torch.equal(k1[seg, :got], torch.sort(s0[seg, :got]).values)           # the same boxes by index


# ---------------------------------------------------------------------------------------------------------------
# SURVEY 8f N2 / N4 (training halves): RandomSampler and mask targets
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [dict(num=512, pos_fraction=0.25, neg_pos_ub=-1, add_gt_as_proposals=True),
                                 dict(num=64, pos_fraction=0.5, neg_pos_ub=3, add_gt_as_proposals=False)])
def test_random_sampler_matches_reference_restatement(oracle, dev, cfg):
    """Same seed -> the same boxes as base_sampler.py:31-103 / random_sampler.py:19-58 restated in numpy."""
    from roi3d_b200.core.bbox import MaxIoUAssigner, RandomSampler
    props, gts = _assign_case(3000, 9, 77)
    labels = np.arange(1, 10, dtype=np.int64)
    pt, gt_t, lt = torch.from_numpy(props).to(dev), torch.from_numpy(gts).to(dev), torch.from_numpy(labels).to(dev)
    res = MaxIoUAssigner(0.5, 0.5, 0.5, True).assign(pt, gt_t, None, lt)
    gi = res.gt_inds.cpu().numpy()
    if cfg["add_gt_as_proposals"]:
        gi = np.concatenate([np.arange(1, 10), gi])
    np.random.seed(123)
    want_pos, want_neg = oracle.random_sample(gi, cfg["num"], cfg["pos_fraction"], cfg["neg_pos_ub"])
    np.random.seed(123)
    sr = RandomSampler(**cfg).sample(res, pt, gt_t, lt)
    assert np.array_equal(sr.pos_inds.cpu().numpy(), want_pos) and np.array_equal(sr.neg_inds.cpu().numpy(), want_neg)
    allb = np.concatenate([gts, props[:, :6]]) if cfg["add_gt_as_proposals"] else props[:, :6]
    assert np.array_equal(sr.pos_bboxes.cpu().numpy(), allb[want_pos])
    assert np.array_equal(sr.bboxes.cpu().numpy(), np.concatenate([allb[want_pos], allb[want_neg]]))
    assert np.array_equal(sr.pos_assigned_gt_inds.cpu().numpy(), gi[want_pos] - 1)
    assert np.array_equal(sr.pos_gt_bboxes.cpu().numpy(), gts[gi[want_pos] - 1])
    if cfg["add_gt_as_proposals"]:
        assert sr.pos_is_gt[:9].cpu().numpy().sum() >= 1 and sr.num_gts == 9


@pytest.mark.gpu
@pytest.mark.parametrize("values", ["0/255", "0/1"])
def test_mask_target_matches_resize_restatement(oracle, dev, values):
    """mask_target_single on the device vs the restated host algorithm (uint8 crop -> img_as_float -> float64 resize
    -> *255 -> uint8 -> nonzero): crops that are enlarged, shrunk (anti-aliasing), clipped by the volume border and a
    one-voxel box.  Parity unpinned by the reference (skimage is not installed; same restatement over scipy)."""
    from roi3d_b200.core.mask import mask_target, mask_target_single
    rng = np.random.default_rng(5)
    G, D, H, W = 3, 40, 96, 96
    gt = np.zeros((G, D, H, W), np.uint8)
    zz, yy, xx = np.mgrid[:D, :H, :W]
    for g in range(G):   # blobs
        c = rng.uniform([8, 20, 20], [32, 76, 76])
        r = rng.uniform([4, 8, 8], [12, 30, 30])
        gt[g] = (((zz - c[0]) / r[0]) ** 2 + ((yy - c[1]) / r[1]) ** 2 + ((xx - c[2]) / r[2]) ** 2 <= 1)
    if values == "0/255":
        gt *= 255
    n = 24
    lo = np.stack([rng.uniform(0, 80, n), rng.uniform(0, 80, n), rng.uniform(0, 30, n)], 1)
    sz = np.stack([rng.uniform(1, 70, n), rng.uniform(1, 70, n), rng.uniform(1, 30, n)], 1)
    props = np.stack([lo[:, 0], lo[:, 1], lo[:, 0] + sz[:, 0], lo[:, 1] + sz[:, 1], lo[:, 2], lo[:, 2] + sz[:, 2]], 1)
    props[0] = [10, 12, 10, 12, 5, 5]                 # one voxel
    props[1] = [60, 60, 140, 150, 30, 60]             # clipped by the volume
    props = props.astype(np.float32)
    inds = rng.integers(0, G, n)
    cfg = dict(mask_size=28, mask_size_depth=20)
    got = mask_target_single(torch.from_numpy(props).to(dev), torch.from_numpy(inds).to(dev), torch.from_numpy(gt), cfg)
    want, scaled = oracle.mask_target_single(props, inds, gt, 28, 20, return_scaled=True)
    assert got.shape == (n, 20, 28, 28) and got.dtype == torch.float32
    differ = got.cpu().numpy() != want
    if values == "0/255":
        assert int(differ.sum()) == 0, "%d of %d target voxels differ" % (int(differ.sum()), want.size)
    else:
        # {0,1} masks: the reference computes 255 * (sum_i w_i * (1/255)) and truncates to uint8, so a voxel inside the
        # mask is 1 or 0 depending on the LAST BIT of that sum (numpy's exp and pairwise sums vs the device's).  The
        # two restatements may only disagree exactly on that knife edge.
        assert float(differ.mean()) < 5e-3
        assert np.all(np.abs(scaled[differ] - 1.0) < 1e-9)
    assert 0 < want.mean() < 1
    both = mask_target([torch.from_numpy(props[:5]).to(dev), torch.from_numpy(props[5:9]).to(dev)],
                       [torch.from_numpy(inds[:5]).to(dev), torch.from_numpy(inds[5:9]).to(dev)],
                       [torch.from_numpy(gt).to(dev), torch.from_numpy(gt).to(dev)], cfg)
    assert torch.equal(both, got[:9])
    assert mask_target_single(torch.zeros((0, 6), device=dev), torch.zeros(0, dtype=torch.long, device=dev), gt, cfg).shape == (0, 28, 28)


PLANAR_CASES_FOR_BWD = [
    # PLANAR_CASES rows with 14-wide outputs (+ plane storage in floats, 0 = default)
    ((2, 20, 10, 32, 32), 14, 14, 0.125, 0.25, 2, 50, (256, 256, 40), 0),
    ((1, 12, 8, 16, 16), 14, 10, 0.25, 0.5, 2, 30, (64, 64, 16), 0),
    ((1, 8, 6, 12, 12), 14, 14, 0.25, 0.5, 3, 20, (48, 48, 12), 0),
    ((2, 20, 10, 32, 32), 14, 14, 0.125, 0.25, 2, 50, (256, 256, 40), 5000),
    ((1, 40, 12, 20, 20), 14, 14, 0.25, 0.5, 0, 12, (80, 80, 24), 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", STREAM_CASES)
def test_roi_align_backward_streamed_kernel(oracle, dev, case):
    """The streamed backward (7x7xPD outputs, C % 64 == 0, channels-last gradients; one vector red per voxel, RoI and
    channel): oracle tolerance, with the per-warp kernel (tuning variant 50) on the same inputs beside it.  The RoI set
    holds empty, inverted and whole-map RoIs (literal path inside the same launch)."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D
    shape, pdp, sc, scd, sn, k, img = case
    B, C, D, H, W = shape
    rois = np.concatenate([synth.c2_rois(k, seed=6, img=img, batch=B),
                           synth.adversarial_rois(shape[2:], sc, scd, batch=B),
                           np.array([[B - 1, 2, 3, img[0] - 4, img[1] - 6, 1, img[2] - 3]], np.float32)], 0)
    ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
    rois = rois[ok] if sn == 0 else rois
    g = _feats((rois.shape[0], C, pdp, 7, 7), 8)
    want = oracle.roi_align3d_backward(g, rois, shape, sc, scd, sn)
    grads = {}
    for variant in (0, 50):
        ft = cl(torch.zeros(shape, device=dev)).requires_grad_(True)
        roi3d_b200._lib.set_tuning(1, variant)
        try:
            RoIAlign3D(7, pdp, sc, scd, sn)(ft, torch.from_numpy(rois).to(dev)).backward(torch.from_numpy(g).to(dev))
        finally:
            roi3d_b200._lib.set_tuning(1, 0)
        grads[variant] = ft.grad.cpu().numpy()
        assert rel_err(grads[variant], want) <= BWD_TOL
    assert rel_err(grads[0], grads[50]) <= BWD_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in PLANAR_CASES_FOR_BWD])
def test_roi_align_backward_planar_kernel(oracle, dev, case):
    """The planar backward (14-wide outputs, channels-last gradients): oracle tolerance, per-warp kernel (variant 50)
    beside it; smem_floats = 5000 forces four channels per pass and sends the largest footprints down the literal path."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D
    shape, ps, pdp, sc, scd, sn, k, img, smem_floats = case
    B, C, D, H, W = shape
    rois = np.concatenate([synth.c2_rois(k, seed=72, img=img, batch=B),
                           synth.adversarial_rois(shape[2:], sc, scd, batch=B),
                           np.array([[B - 1, 2, 3, img[0] - 4, img[1] - 6, 1, img[2] - 3]], np.float32)], 0)
    ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
    rois = rois[ok] if sn == 0 else rois
    g = _feats((rois.shape[0], C, pdp, ps, ps), 9)
    want = oracle.roi_align3d_backward(g, rois, shape, sc, scd, sn)
    grads = {}
    for variant in (0, 50):
        ft = cl(torch.zeros(shape, device=dev)).requires_grad_(True)
        roi3d_b200._lib.set_tuning(1, variant)
        roi3d_b200._lib.set_tuning(10, smem_floats)
        try:
            RoIAlign3D(ps, pdp, sc, scd, sn)(ft, torch.from_numpy(rois).to(dev)).backward(torch.from_numpy(g).to(dev))
        finally:
            roi3d_b200._lib.set_tuning(1, 0)
            roi3d_b200._lib.set_tuning(10, 0)
        grads[variant] = ft.grad.cpu().numpy()
        assert rel_err(grads[variant], want) <= BWD_TOL
    assert rel_err(grads[0], grads[50]) <= BWD_TOL


PLANAR_CASES = [
    # (B, C, D, H, W), out_size, out_size_depth, scale, scale_d, sample_num, n_rois, roi image (W, H, D)
    ((2, 24, 10, 24, 40), 7, 7, 0.25, 0.5, 2, 60, (160, 96, 20)),
    ((1, 37, 12, 40, 40), 7, 3, 0.25, 0.5, 2, 40, (160, 160, 24)),     # odd channel count, 7x7x3
    ((1, 16, 24, 96, 96), 7, 7, 0.25, 0.5, 2, 40, (384, 384, 48)),     # c2-sized RoIs: big footprints, several passes
    ((2, 20, 10, 32, 32), 14, 14, 0.125, 0.25, 2, 50, (256, 256, 40)),  # mask shape on a coarse level
    ((1, 12, 8, 16, 16), 14, 10, 0.25, 0.5, 2, 30, (64, 64, 16)),      # real-config mask shape 14x14x10
    ((1, 8, 10, 20, 20), 7, 7, 0.25, 0.5, 0, 30, (80, 80, 20)),        # adaptive sampling
    ((1, 8, 6, 12, 12), 14, 14, 0.25, 0.5, 3, 20, (48, 48, 12)),       # three samples per bin
]


# Channels-last levels reach the planar kernel only with C % 4 == 0 (16-byte copies of four channels of a voxel); the
# odd-channel case runs channels-last in test_roi_align_kernel_coverage.py under the kernel that takes it.
PLANAR_RUNS = [pytest.param(case, layout, smem_floats, id="%d-%s-case%d" % (smem_floats, layout, i))
               for smem_floats in (0, 5000) for layout in ("NCDHW", "NDHWC") for i, case in enumerate(PLANAR_CASES)
               if layout == "NCDHW" or case[0][1] % 4 == 0]


@pytest.mark.gpu
@pytest.mark.parametrize("case,layout,smem_floats", PLANAR_RUNS)
def test_roi_align_forward_planar_kernel(oracle, dev, case, layout, smem_floats):
    """The planar kernel: the reference's NCDHW layout read natively (no conversion), and channels-last through the
    same kernel (tuning variant 60); 7- and 14-wide outputs, ragged channel groups, adversarial and over-wide RoIs.
    smem_floats = 5000 shrinks the plane storage (tuning key 10) so that footprints are walked in several z chunks with
    four channels per pass, and the largest ones fall back to the literal path."""
    import roi3d_b200
    from roi3d_b200.ops import RoIAlign3D
    shape, ps, pdp, sc, scd, sn, k, img = case
    B, C, D, H, W = shape
    f = _feats(shape, 71)
    rois = np.concatenate([synth.c2_rois(k, seed=72, img=img, batch=B),
                           synth.adversarial_rois(shape[2:], sc, scd, batch=B),
                           np.array([[B - 1, 2, 3, img[0] - 4, img[1] - 6, 1, img[2] - 3],       # whole map: literal path
                                     [0, img[0] - 30, 4, img[0] - 2, 40, 2, 9]], np.float32)], 0)  # touches the right border
    if sn == 0:
        ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
        rois = rois[ok]
    want = oracle.roi_align3d_forward(f, rois, ps, pdp, sc, scd, sn)
    ft = torch.from_numpy(f).to(dev)
    if layout == "NDHWC":
        ft = cl(ft)
    roi3d_b200._lib.set_tuning(0, 60)
    roi3d_b200._lib.set_tuning(10, smem_floats)
    try:
        out = RoIAlign3D(ps, pdp, sc, scd, sn)(ft, torch.from_numpy(rois).to(dev))
    finally:
        roi3d_b200._lib.set_tuning(0, 0)
        roi3d_b200._lib.set_tuning(10, 0)
    assert out.is_contiguous() and rel_err(out.cpu().numpy(), want) <= FWD_TOL


@pytest.mark.gpu
def test_second_device_in_one_process(oracle):
    """A process that drives two GPUs: the opt-in to large dynamic shared memory is a per-device kernel attribute, so
    every large-shared-memory kernel (streamed forward / backward, NCDHW twin, planar, NMS sweep, top-k) has to be set
    up on each device it runs on.  Skipped on a single-GPU box."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from roi3d_b200.ops import RoIAlign3D, nms
    f = _feats((1, 64, 10, 32, 32), 5)
    rois = synth.c2_rois(60, seed=6, img=(128, 128, 20))
    want = oracle.roi_align3d_forward(f, rois, 7, 7, 0.25, 0.5, 2)
    want14 = oracle.roi_align3d_forward(f, rois, 14, 14, 0.25, 0.5, 2)
    dets = synth.c1_boxes(700, seed=3)
    keep_want = oracle.nms3d(dets, 0.5)
    for d in (0, 1):
        dv = torch.device("cuda:%d" % d)
        rt = torch.from_numpy(rois).to(dv)
        x = cl(torch.from_numpy(f).to(dv)).requires_grad_(True)
        out = RoIAlign3D(7, 7, 0.25, 0.5, 2)(x, rt)
        assert rel_err(out.detach().cpu().numpy(), want) <= FWD_TOL
        out.backward(torch.ones_like(out))
        assert torch.isfinite(x.grad).all()
        assert rel_err(RoIAlign3D(7, 7, 0.25, 0.5, 2)(torch.from_numpy(f).to(dv), rt).cpu().numpy(), want) <= FWD_TOL
        assert rel_err(RoIAlign3D(14, 14, 0.25, 0.5, 2)(cl(torch.from_numpy(f).to(dv)), rt).cpu().numpy(), want14) <= FWD_TOL
        _, inds = nms(torch.from_numpy(dets).to(dv), 0.5)
        assert np.array_equal(inds.cpu().numpy(), keep_want)

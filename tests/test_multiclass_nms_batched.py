"""Batched multiclass 3D NMS (`multiclass_nms_3d_batched`, `roi3d_multiclass_nms3d_batched`), the per-image
`multiclass_nms_3d` built on it, and the fixed-shape helpers around them (`RPNProposal3D.get_proposals_padded`,
`bbox2roi3D_padded`).

The reference is the CPU oracle: `oracle.multiclass_nms_3d` for hard NMS and `soft_nms_oracle.multiclass_nms_3d` for
soft-NMS, both the reference's per-class loop.  For every image b the first det_counts[b] rows and labels of the batched
call equal the oracle on `bboxes[b, :counts[b]], scores[b, :counts[b]]` bit for bit, and the rest are zero rows with
label -1; `multiclass_nms_3d` on the same rows returns the oracle's result too.  The last test captures the whole
fixed-shape test-time RoI stage, proposals to mask head, in one CUDA graph.
"""
import numpy as np
import pytest
import torch

import soft_nms_oracle as soft_oracle
import synth
from kernel_inventory import built_kernels, launched_kernels, library_kernels

EINVAL = -1
MC_KERNELS = {"multiclass_select_kernel", "multiclass_collect_kernel", "multiclass_gather_kernel"}
NMS_CFGS = {
    "nms": dict(type='nms', iou_thr=0.5),
    "soft_linear": dict(type='soft_nms', iou_thr=0.5, min_score=0.05),
    "soft_gaussian": dict(type='soft_nms', iou_thr=0.3, method='gaussian', sigma=0.3, min_score=0.25),
}
TIES = np.array([0.3, 0.6, 0.9], np.float32)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def make_batch(B, n, C, shared_boxes, seed, counts=None):
    """[B, n, 6 or 6C] boxes, [B, n, C] scores and int32 [B] counts.  Boxes are clustered (C1), shifted per class;
    class scores are distinct on odd images and drawn from three values (ties within and across classes) on even ones.
    Rows past counts[b] hold NaN / inf boxes and scores of 1.0, which must never be read."""
    rng = np.random.default_rng(seed)
    boxes = np.empty((B, n, 6 if shared_boxes else 6 * C), np.float32)
    scores = np.empty((B, n, C), np.float32)
    for b in range(B):
        d = synth.c1_boxes(n, seed=seed + 17 * b)
        if shared_boxes:
            boxes[b] = d[:, :6]
        else:
            boxes[b] = np.concatenate([d[:, :6] + np.float32(1.5 * c) for c in range(C)], 1)
        for c in range(1, C):
            scores[b, :, c] = rng.choice(TIES, n) if b % 2 == 0 else rng.permutation(d[:, 6])
        scores[b, :, 0] = 1 - scores[b, :, 1]
    if counts is None:
        counts = rng.integers(0, n + 1, B)
        counts[0] = n
        if B > 2:
            counts[1] = 0
    counts = np.asarray(counts, np.int32)
    for b in range(B):
        pad = boxes[b, counts[b]:]
        pad[:] = np.float32(np.nan)
        pad[::3] = np.float32(np.inf)
        pad[1::3] = np.float32(-np.inf)
        scores[b, counts[b]:] = np.float32(1.0)
    return boxes, scores, counts


def run_batched(dev, boxes, scores, counts, score_thr, cfg, max_num):
    from roi3d_b200 import multiclass_nms_3d_batched
    det, lab, cnt = multiclass_nms_3d_batched(torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev),
                                              torch.from_numpy(counts).to(dev), score_thr, cfg, max_num)
    return det.cpu().numpy(), lab.cpu().numpy(), cnt.cpu().numpy()


def oracle_multiclass_nms(oracle, boxes, scores, score_thr, cfg, max_num):
    """The CPU oracle of multiclass_nms_3d for nms_cfg `cfg` on one image's [n, 6C or 6] boxes and [n, C] scores."""
    if cfg['type'] == 'nms':
        return oracle.multiclass_nms_3d(boxes, scores, score_thr, cfg['iou_thr'], max_num)
    kw = {key: v for key, v in cfg.items() if key not in ('type', 'iou_thr')}
    return soft_oracle.multiclass_nms_3d(boxes, scores, score_thr, cfg['iou_thr'], max_num, **kw)


def check_against_oracle(oracle, dev, boxes, scores, counts, score_thr, cfg, max_num):
    """The batched call, and multiclass_nms_3d on each image, equal the oracle per image; returns the oracle's results."""
    from roi3d_b200 import multiclass_nms_3d
    B, n, C = scores.shape
    det, lab, cnt = run_batched(dev, boxes, scores, counts, score_thr, cfg, max_num)
    M = max_num if max_num > 0 else (C - 1) * n
    assert det.shape == (B, M, 7) and lab.shape == (B, M) and cnt.shape == (B,)
    assert det.dtype == np.float32 and lab.dtype == np.int64 and cnt.dtype == np.int32
    wants = []
    for b in range(B):
        k = int(counts[b])
        wb, wl = oracle_multiclass_nms(oracle, boxes[b, :k], scores[b, :k], score_thr, cfg, max_num)
        m = int(cnt[b])
        assert m == wb.shape[0], (b, m, wb.shape[0])
        assert same_bits(det[b, :m], wb), b
        assert np.array_equal(lab[b, :m], wl), b
        assert same_bits(det[b, m:], np.zeros((M - m, 7), np.float32)) and (lab[b, m:] == -1).all(), b
        gb, gl = multiclass_nms_3d(torch.from_numpy(boxes[b, :k]).to(dev), torch.from_numpy(scores[b, :k]).to(dev),
                                   score_thr, cfg, max_num)
        assert gb.device == dev and gl.device == dev, b
        assert same_bits(gb.cpu().numpy(), wb) and same_bits(gl.cpu().numpy(), wl), b
        wants.append((wb, wl))
    return wants


# ------------------------------------------------------------------------------------------------ CPU
def test_built_kernels_are_the_three_new_ones():
    assert built_kernels("multiclass_") == MC_KERNELS


def test_abi_argument_errors_return_before_any_launch():
    """Every check runs before the first CUDA call, so fake device addresses are enough here."""
    from roi3d_b200 import _lib
    lib = _lib.lib
    A = 1 << 20

    def call(box_cols=18, B=2, n=100, C=3, nms_type=0, soft_method=1, bboxes=A, det_counts=A, ws=A):
        # a 256-byte workspace is too small for every valid call here: nothing can reach a launch
        return lib.roi3d_multiclass_nms3d_batched(bboxes, box_cols, A, A, B, n, C, 0.2, nms_type, 0.5, soft_method, 0.5,
                                                  0.001, 37, A, A, det_counts, ws, 256, None)

    cases = [
        (dict(nms_type=1, n=4097), b"n=4097"),
        (dict(nms_type=1, soft_method=0), b"soft_method=0"),
        (dict(nms_type=1, soft_method=3), b"soft_method=3"),
        (dict(nms_type=2), b"nms_type=2"),
        (dict(nms_type=-1), b"nms_type=-1"),
        (dict(box_cols=12), b"box_cols=12"),
        (dict(box_cols=7), b"box_cols=7"),
        (dict(C=1, box_cols=6), b"num_classes=1"),
        (dict(B=-1), b"bad sizes"),
        (dict(n=32769), b"n=32769"),
        (dict(bboxes=None), b"NULL input"),
        (dict(det_counts=None), b"NULL output"),
        (dict(ws=None), b"NULL workspace"),
        (dict(ws=A + 16), b"256-byte aligned"),
    ]
    for kw, msg in cases:
        assert call(**kw) == EINVAL, kw
        assert msg in lib.roi3d_last_error(), (kw, lib.roi3d_last_error())
    # a soft-NMS call at the 4096-row limit passes the argument checks (it then fails on the too-small workspace)
    assert call(nms_type=1, n=4096, ws=A) == -3 and b"workspace too small" in lib.roi3d_last_error()
    assert lib.roi3d_multiclass_nms3d_batched(None, 6, None, None, 0, 10, 2, 0.2, 0, 0.5, 1, 0.5, 0.001, -1, None, None,
                                              None, None, 0, None) == 0   # B == 0: nothing to do


def test_workspace_size_is_a_host_query():
    from roi3d_b200 import _lib
    lib = _lib.lib
    hard = lib.roi3d_multiclass_nms3d_workspace_bytes(8, 1000, 2, 2000, 0)
    soft = lib.roi3d_multiclass_nms3d_workspace_bytes(8, 1000, 2, 2000, 1)
    assert hard >= lib.roi3d_nms3d_workspace_bytes(8, 1000) + lib.roi3d_topk_workspace_bytes(8, 2000)
    assert soft >= 8 * 1000 * 7 * 4 * 2 + lib.roi3d_topk_workspace_bytes(8, 2000)
    assert hard % 256 == 0 and soft % 256 == 0
    assert lib.roi3d_multiclass_nms3d_workspace_bytes(8, 1000, 1, 2000, 0) == 256


def test_python_errors_without_gpu():
    from roi3d_b200 import multiclass_nms_3d_batched
    b, s, c = torch.zeros(2, 5, 12), torch.zeros(2, 5, 2), torch.zeros(2, dtype=torch.int32)
    with pytest.raises(NotImplementedError, match="CUDA"):
        multiclass_nms_3d_batched(b, s, c, 0.2, dict(type='nms', iou_thr=0.5))
    with pytest.raises(NotImplementedError, match="CUDA"):
        multiclass_nms_3d_batched(b, s, c, 0.2, dict(type='soft_nms', iou_thr=0.5))
    with pytest.raises(NotImplementedError, match="nms type"):
        multiclass_nms_3d_batched(b, s, c, 0.2, dict(type='nms_2d', iou_thr=0.5))
    with pytest.raises(ValueError, match="Invalid method"):
        multiclass_nms_3d_batched(b, s, c, 0.2, dict(type='soft_nms', iou_thr=0.5, method='cubic'))
    with pytest.raises(KeyError):
        multiclass_nms_3d_batched(b, s, c, 0.2, dict(type='nms'))


def test_bbox2roi3D_padded_rows():
    from roi3d_b200 import bbox2roi3D_padded
    rng = np.random.default_rng(3)
    boxes = rng.uniform(0, 100, (3, 5, 7)).astype(np.float32)
    boxes[0, 2:] = np.nan
    boxes[1, :] = np.inf
    boxes[2, 4, :3] = -np.inf
    counts = np.array([2, 0, 5], np.int32)
    rois = bbox2roi3D_padded(torch.from_numpy(boxes), torch.from_numpy(counts)).numpy()
    assert rois.shape == (15, 7) and rois.dtype == np.float32
    pad = np.array([-1, 0, 0, 0, 0, 0, 0], np.float32)
    for b in range(3):
        for r in range(5):
            row = rois[b * 5 + r]
            want = np.concatenate([[np.float32(b)], boxes[b, r, :6]]).astype(np.float32) if r < counts[b] else pad
            assert same_bits(row, want), (b, r, row)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name", sorted(NMS_CFGS))
@pytest.mark.parametrize("shared_boxes", [False, True], ids=["class_boxes", "shared_boxes"])
@pytest.mark.parametrize("C", [2, 3])
@pytest.mark.parametrize("B", [1, 3, 8])
def test_matches_per_image_multiclass_nms(oracle, dev, B, C, shared_boxes, cfg_name):
    n = 300
    counts = {1: [n], 3: [n, 0, 137]}.get(B)
    boxes, scores, counts = make_batch(B, n, C, shared_boxes, seed=100 * B + 10 * C + shared_boxes, counts=counts)
    cfg = NMS_CFGS[cfg_name]
    for max_num in (-1, 37, 2000):
        wants = check_against_oracle(oracle, dev, boxes, scores, counts, 0.2, cfg, max_num)
        if max_num == 37:   # the cut is reached on every full image
            assert all(wb.shape[0] == 37 for (wb, _), k in zip(wants, counts) if k == n)
    # a score threshold nothing passes
    det, lab, cnt = run_batched(dev, boxes, scores, counts, 5.0, cfg, 37)
    assert (cnt == 0).all() and (det == 0).all() and (lab == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name", sorted(NMS_CFGS))
def test_matches_oracles(oracle, dev, cfg_name):
    boxes, scores, counts = make_batch(3, 400, 3, False, seed=61, counts=[400, 250, 0])
    cfg = NMS_CFGS[cfg_name]
    det, lab, cnt = run_batched(dev, boxes, scores, counts, 0.2, cfg, 37)
    for b in range(3):
        k = int(counts[b])
        wb, wl = oracle_multiclass_nms(oracle, boxes[b, :k], scores[b, :k], 0.2, cfg, 37)
        assert int(cnt[b]) == wb.shape[0] and same_bits(det[b, :cnt[b]], wb) and np.array_equal(lab[b, :cnt[b]], wl)
    assert cnt[0] == 37 and cnt[2] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("cfg_name", sorted(NMS_CFGS))
def test_padding_rows_are_inert(dev, cfg_name):
    boxes, scores, counts = make_batch(4, 200, 3, False, seed=9, counts=[200, 50, 0, 120])
    clean_b, clean_s = boxes.copy(), scores.copy()
    for b in range(4):
        clean_b[b, counts[b]:] = 0
        clean_s[b, counts[b]:] = 0
    for max_num in (-1, 37):
        got = run_batched(dev, boxes, scores, counts, 0.2, NMS_CFGS[cfg_name], max_num)
        want = run_batched(dev, clean_b, clean_s, counts, 0.2, NMS_CFGS[cfg_name], max_num)
        assert all(same_bits(g, w) for g, w in zip(got, want))
        assert got[2][1] > 0


@pytest.mark.gpu
def test_errors_on_the_device_path(dev):
    from roi3d_b200 import _lib, multiclass_nms_3d_batched
    boxes, scores, counts = (torch.from_numpy(x).to(dev) for x in make_batch(2, 4097, 2, True, seed=1, counts=[5, 5]))
    with pytest.raises(_lib.Roi3dError, match="n=4097"):
        multiclass_nms_3d_batched(boxes, scores, counts, 0.2, dict(type='soft_nms', iou_thr=0.5))
    ok = multiclass_nms_3d_batched(boxes, scores, counts, 0.2, dict(type='nms', iou_thr=0.5), 10)
    assert ok[2].shape == (2,)
    with pytest.raises(ValueError, match="multi_bboxes"):
        multiclass_nms_3d_batched(boxes[:, :, :5].contiguous(), scores, counts, 0.2, dict(type='nms', iou_thr=0.5))
    with pytest.raises(ValueError, match="background"):
        multiclass_nms_3d_batched(boxes, scores[:, :, :1].contiguous(), counts, 0.2, dict(type='nms', iou_thr=0.5))
    with pytest.raises(ValueError, match="counts"):
        multiclass_nms_3d_batched(boxes, scores, counts.long(), 0.2, dict(type='nms', iou_thr=0.5))
    with pytest.raises(NotImplementedError, match="counts"):
        multiclass_nms_3d_batched(boxes, scores, counts.cpu(), 0.2, dict(type='nms', iou_thr=0.5))


@pytest.mark.gpu
def test_hard_nms_launches_exactly_its_kernels(dev):
    from roi3d_b200 import multiclass_nms_3d, multiclass_nms_3d_batched
    boxes, scores, counts = (torch.from_numpy(x).to(dev) for x in make_batch(2, 300, 3, False, seed=5))
    res = {}

    def run():
        res["r"] = multiclass_nms_3d_batched(boxes, scores, counts, 0.2, dict(type='nms', iou_thr=0.5), 37)
    want = MC_KERNELS | {"nms3d_rank_kernel", "nms3d_mask_q_kernel<false>", "nms3d_sweep_kernel", "topk_tail_kernel<false>"}
    assert library_kernels(launched_kernels(run)) == want
    # the per-image function runs the same kernels (image 0 uses all its rows)
    names = launched_kernels(lambda: multiclass_nms_3d(boxes[0], scores[0], 0.2, dict(type='nms', iou_thr=0.5), 37))
    assert library_kernels(names) == want
    names = launched_kernels(lambda: multiclass_nms_3d_batched(boxes, scores, counts, 0.2,
                                                              dict(type='soft_nms', iou_thr=0.5), 37))
    assert library_kernels(names) == MC_KERNELS | {"soft_nms3d_kernel<1>", "topk_tail_kernel<false>"}


def _rpn_inputs(dev, B, seed):
    dims = [(8, 24, 24), (4, 12, 12), (2, 6, 6)]
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    cls = [2 * torch.randn((B, 1) + d, device=dev, generator=g) for d in dims]
    reg = [0.3 * torch.randn((B, 6) + d, device=dev, generator=g) for d in dims]
    metas = [dict(img_shape=(96, 96, 3, 16), scale_factor=1.0)] * B
    return cls, reg, metas


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(nms_across_levels=True), dict(min_bbox_size=11.3),
                                dict(nms_pre=0, nms_post=60, max_num=90)], ids=["plain", "across", "min_size", "no_pre"])
def test_get_proposals_padded_equals_get_proposals(dev, kw):
    from roi3d_b200 import RPNProposal3D
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=[4, 8, 16],
                         anchor_strides_depth=[2, 4, 8])
    cfg = dict(dict(nms_pre=300, nms_post=100, max_num=150, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False), **kw)
    cls, reg, metas = _rpn_inputs(dev, 3, seed=11)
    want = head.get_proposals(cls, reg, metas, cfg)
    final, counts = head.get_proposals_padded(cls, reg, metas, cfg)
    assert counts.dtype == torch.int32 and counts.is_cuda and tuple(counts.shape) == (3,)
    counts = counts.cpu().numpy()
    assert (counts <= final.shape[1]).all() and (counts > 0).all()
    for b in range(3):
        assert same_bits(final[b, :counts[b]].cpu().numpy(), want[b].cpu().numpy()), b


@pytest.mark.gpu
def test_padded_rois_give_zero_extractor_rows(dev):
    import roi_stage
    from roi3d_b200 import bbox2roi3D_padded
    stage = roi_stage.RoIStage(max_masks=20).to(dev)
    feats, _cls, _reg, _metas = roi_stage.synthetic_inputs(2, vol_dhw=(32, 128, 128), device=dev)
    boxes = torch.from_numpy(synth.c1_boxes(40, seed=3, vol=(128, 128, 32))).to(dev).view(2, 20, 7).clone()
    boxes[0, 5:] = float('nan')
    counts = torch.tensor([5, 20], dtype=torch.int32, device=dev)
    rois = bbox2roi3D_padded(boxes, counts)
    out = stage.mask_ex(feats[:4], rois)
    assert torch.count_nonzero(out[5:20]) == 0
    assert torch.isfinite(out).all() and torch.count_nonzero(out[:5]) > 0 and torch.count_nonzero(out[20:]) > 0


def fixed_shape_stage(stage, feats, cls, reg, metas):
    """The test-time RoI stage of roi_stage.RoIStage with fixed shapes and no host read: padded proposals -> bbox
    extractor -> FC heads -> softmax -> delta2bbox3D -> batched multiclass NMS -> padded mask RoIs -> mask extractor ->
    mask head.  Returns every intermediate the checks read."""
    import roi_stage
    import roi3d_b200
    rcnn = roi_stage.TEST_CFG_RCNN
    final, pcounts = stage.rpn.get_proposals_padded(cls, reg, metas, roi_stage.TEST_CFG_RPN)
    B, kk = final.shape[:2]
    rois = roi3d_b200.bbox2roi3D_padded(final, pcounts)
    h = stage.fc(stage.bbox_ex(feats[:4], rois).flatten(1))
    scores = stage.fc_cls(h).softmax(dim=1)
    boxes = roi3d_b200.delta2bbox3D(rois[:, 1:], stage.fc_reg(h), [0.0] * 6, roi_stage.BBOX_TARGET_STDS,
                                    metas[0]['img_shape'])
    det, labels, dcounts = roi3d_b200.multiclass_nms_3d_batched(boxes.view(B, kk, -1), scores.view(B, kk, -1), pcounts,
                                                                rcnn['score_thr'], rcnn['nms'], rcnn['max_per_img'])
    m = stage.max_masks
    mrois = roi3d_b200.bbox2roi3D_padded(det[:, :m], dcounts.clamp(max=m))
    mfeats = stage.mask_ex(feats[:4], mrois)
    return dict(pcounts=pcounts, boxes=boxes.view(B, kk, -1), scores=scores.view(B, kk, -1), det=det, labels=labels,
                dcounts=dcounts, mrois=mrois, mfeats=mfeats, masks=stage.mask_head(mfeats))


@pytest.mark.gpu
def test_whole_roi_stage_as_one_cuda_graph(oracle, dev):
    import roi_stage
    stage = roi_stage.RoIStage(max_masks=20).to(dev).eval()
    feats, cls, reg, metas = roi_stage.synthetic_inputs(2, vol_dhw=(32, 128, 128), device=dev, seed=7)
    graph = torch.cuda.CUDAGraph()
    try:
        with torch.no_grad():
            _check_stage_graph(oracle, dev, stage, graph, feats, cls, reg, metas)
    finally:
        # the graph and its private memory pool go with this test: nothing captured outlives it
        del graph
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _check_stage_graph(oracle, dev, stage, graph, feats, cls, reg, metas):
    """Warm up, capture, replay on new inputs, and check the replay's detections against the oracle on the replay's own
    boxes and scores, and its mask RoIs and features against the extractor on the oracle's rows."""
    import roi_stage
    rcnn = roi_stage.TEST_CFG_RCNN
    B, m = feats[0].shape[0], stage.max_masks
    fixed_shape_stage(stage, feats, cls, reg, metas)     # warm-up: descriptor uploads, attributes, algorithms
    torch.cuda.synchronize()
    with torch.cuda.graph(graph):
        out = fixed_shape_stage(stage, feats, cls, reg, metas)
    new_feats, new_cls, new_reg, _ = roi_stage.synthetic_inputs(B, vol_dhw=(32, 128, 128), device=dev, seed=8)
    for dst, src in zip(feats + cls + reg, new_feats + new_cls + new_reg):
        dst.copy_(src)
    graph.replay()
    torch.cuda.synchronize()

    pcounts = out['pcounts'].cpu().numpy()
    dcounts = out['dcounts'].cpu().numpy()
    det, labels = out['det'].cpu().numpy(), out['labels'].cpu().numpy()
    mfeats = out['mfeats']
    assert (pcounts > 0).all() and (dcounts > 0).all()
    want_rois = torch.zeros((B * m, 7), device=dev)
    want_rois[:, 0] = -1
    for b in range(B):
        k = int(pcounts[b])
        wb, wl = oracle_multiclass_nms(oracle, out['boxes'][b, :k].cpu().numpy(), out['scores'][b, :k].cpu().numpy(),
                                       rcnn['score_thr'], rcnn['nms'], rcnn['max_per_img'])
        c = int(dcounts[b])
        assert c == wb.shape[0]
        assert same_bits(det[b, :c], wb) and np.array_equal(labels[b, :c], wl)
        assert (det[b, c:] == 0).all() and (labels[b, c:] == -1).all()
        cm = min(c, m)
        want_rois[b * m:b * m + cm, 0] = b
        want_rois[b * m:b * m + cm, 1:] = torch.from_numpy(wb[:cm, :6]).to(dev)
    assert torch.equal(out['mrois'], want_rois)
    want_feats = stage.mask_ex(feats[:4], want_rois)
    for b in range(B):
        cm = min(int(dcounts[b]), m)
        assert torch.equal(mfeats[b * m:b * m + cm], want_feats[b * m:b * m + cm])
        assert torch.count_nonzero(mfeats[b * m + cm:(b + 1) * m]) == 0
    assert out['masks'].shape[0] == B * m

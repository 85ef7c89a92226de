"""Pins the CPU oracle against fixtures produced by the REFERENCE's own CUDA kernels on a B200
(tests/golden/make_golden.py runs oracle/_ref there; the .npz files are committed).  No GPU, no /root/reference."""
import os

import numpy as np
import pytest

import synth

HERE = os.path.dirname(os.path.abspath(__file__))


def _load(name):
    path = os.path.join(HERE, "golden", name)
    if not os.path.exists(path):
        pytest.skip("%s not generated yet" % name)
    return synth.load_roi_align_ref(path) if name == "roi_align3d_ref.npz" else np.load(path)


@pytest.mark.parametrize("tag", ["c7", "m14x10", "b7x3", "a5"])
def test_roi_align_forward_is_bit_identical_to_reference_kernel(oracle, tag):
    z = _load("roi_align3d_ref.npz")
    ps, pdp, sn = (int(v) for v in z["%s_cfg" % tag])
    got = oracle.roi_align3d_forward(z["feats"], z["%s_rois" % tag], ps, pdp, float(z["spatial_scale"]),
                                     float(z["spatial_scale_depth"]), sn, contract=True)
    assert np.array_equal(got, z["%s_out" % tag])
    # the source-literal arithmetic (no FMA contraction) is close but NOT what the compiled kernel computes
    lit = oracle.roi_align3d_forward(z["feats"], z["%s_rois" % tag], ps, pdp, float(z["spatial_scale"]),
                                     float(z["spatial_scale_depth"]), sn, contract=False)
    assert np.abs(lit - z["%s_out" % tag]).max() < 1e-4


@pytest.mark.parametrize("tag", ["c7", "m14x10", "b7x3", "a5"])
def test_roi_align_backward_matches_reference_kernel(oracle, tag):
    """The reference accumulates with fp32 atomics in arbitrary order; the oracle sums in float64.
    Non-cubic outputs: the reference's own top_diff index (bug_compat) is what its kernel executed."""
    z = _load("roi_align3d_ref.npz")
    ps, pdp, sn = (int(v) for v in z["%s_cfg" % tag])
    want = z["%s_gin" % tag]
    got = oracle.roi_align3d_backward(z["%s_gout" % tag], z["%s_rois" % tag], z["feats"].shape,
                                      float(z["spatial_scale"]), float(z["spatial_scale_depth"]), sn,
                                      bug_compat=True, contract=True)
    assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max())
    if ps != pdp:
        fixed = oracle.roi_align3d_backward(z["%s_gout" % tag], z["%s_rois" % tag], z["feats"].shape,
                                            float(z["spatial_scale"]), float(z["spatial_scale_depth"]), sn,
                                            bug_compat=False, contract=True)
        assert np.abs(fixed - want).max() > 1e-3   # SURVEY F2: the reference's gradient is wrong here


@pytest.mark.parametrize("tag", ["a", "b", "c", "d"])
def test_nms_keep_list_equals_reference_kernel(oracle, tag):
    z = _load("nms3d_ref.npz")
    got = oracle.nms3d(z["%s_dets" % tag], float(z["%s_thr" % tag]), contract=True)
    assert np.array_equal(got, z["%s_keep" % tag])


def _assigner_cases():
    path = os.path.join(HERE, "golden", "assigner_ref.npz")
    return range(int(np.load(path)["num_cases"])) if os.path.exists(path) else []


@pytest.mark.parametrize("i", list(_assigner_cases()))
def test_assigner_equals_the_reference_assigner(oracle, i):
    """tests/golden/assigner_ref.npz holds the outputs of the REFERENCE's MaxIoUAssigner (its own Python, CPU tensors;
    tests/golden/make_assigner_golden.py), with and without ignore regions: the oracle restatement gives the same
    gt_inds, max_overlaps and labels, bit for bit."""
    z = _load("assigner_ref.npz")
    pos, neg, mpi, assign_all, ign_thr, wrt = (float(v) for v in z["cfg_%d" % i])
    a, mo, lab = oracle.assign_max_iou(z["boxes_%d" % i], z["gt_%d" % i], z["labels_%d" % i], pos_iou_thr=pos,
                                       neg_iou_thr=neg, min_pos_iou=mpi, gt_max_assign_all=bool(assign_all),
                                       ignore_iof_thr=ign_thr, ignore_wrt_candidates=bool(wrt),
                                       gt_bboxes_ignore=z["ign_%d" % i])
    assert np.array_equal(a, z["gt_inds_%d" % i])
    assert np.array_equal(mo, z["max_overlaps_%d" % i])
    assert np.array_equal(lab, z["assigned_labels_%d" % i])


@pytest.mark.gpu
@pytest.mark.parametrize("i", list(_assigner_cases()))
def test_device_assigner_equals_the_reference_assigner(i):
    """The same fixture against the product (roi3d_assign_max_iou_ignore through the MaxIoUAssigner mirror)."""
    import torch
    from roi3d_b200.core.bbox import MaxIoUAssigner
    z = _load("assigner_ref.npz")
    pos, neg, mpi, assign_all, ign_thr, wrt = (float(v) for v in z["cfg_%d" % i])
    dev = torch.device("cuda:0")
    res = MaxIoUAssigner(pos, neg, mpi, bool(assign_all), ign_thr, bool(wrt)).assign(
        torch.from_numpy(z["boxes_%d" % i]).to(dev), torch.from_numpy(z["gt_%d" % i]).to(dev),
        gt_bboxes_ignore=torch.from_numpy(z["ign_%d" % i]).to(dev), gt_labels=torch.from_numpy(z["labels_%d" % i]).to(dev))
    assert np.array_equal(res.gt_inds.cpu().numpy(), z["gt_inds_%d" % i])
    assert np.array_equal(res.max_overlaps.cpu().numpy(), z["max_overlaps_%d" % i])
    assert np.array_equal(res.labels.cpu().numpy(), z["assigned_labels_%d" % i])


# ---------------------------------------------------------------------------------------------------------------
# tests/golden/python_ref.npz: outputs of the reference's own pure-Python pieces (imported from /root/reference by
# tests/golden/make_python_ref_golden.py and run on CPU tensors) -- pins the oracle restatements of the rows next to
# the hot path (SURVEY 8f) to the reference itself.
# ---------------------------------------------------------------------------------------------------------------
ANCHOR_CASES = [
    ((5, 8, 6), 8, 4, [2], [2], [1.0], (5, 7, 6), (56, 48, 3, 20), 0),
    ((7, 9, 11), 4, 2, [2, 4], [2, 3], [0.5, 1.0, 2.0], (6, 9, 10), (36, 42, 3, 13), 3),
    ((3, 4, 5), 16, 8, [8], [2], [1.0], (3, 4, 5), (64, 80, 3, 24), -1),
]


@pytest.mark.parametrize("i", [0, 1, 2])
def test_anchor_generator_equals_the_reference_class(oracle, i):
    z = _load("python_ref.npz")
    fm, st, sd, scales, dscales, ratios, valid, img_shape, border = ANCHOR_CASES[i]
    base = oracle.gen_base_anchors(st, scales, dscales, ratios, sd)
    assert np.array_equal(base, z["anchor_base_%d" % i])
    grid = oracle.grid_anchors(base, fm, st, sd)
    assert np.array_equal(grid, z["anchor_grid_%d" % i])
    v = oracle.valid_flags(fm, valid, base.shape[0])
    assert np.array_equal(v, z["anchor_valid_%d" % i])
    assert np.array_equal(oracle.anchor_inside_flags(grid, v, img_shape, border), z["anchor_inside_%d" % i])


def test_bbox_transforms_equal_the_reference_functions(oracle):
    z = _load("python_ref.npz")
    means, stds = (0.0,) * 6, tuple(float(v) for v in z["t_stds"])
    d = oracle.bbox2delta3d(z["t_props"], z["t_gt"], means, stds)
    want = z["t_deltas"]
    # dx, dy, dz: IEEE add / mul / div only -> exact; dw, dh, dd go through log (numpy's vs torch's CPU libm)
    assert np.array_equal(d[:, [0, 1, 4]], want[:, [0, 1, 4]])
    assert np.allclose(d[:, [2, 3, 5]], want[:, [2, 3, 5]], rtol=1e-6, atol=1e-6)   # tolerance: 1e-6
    ms = tuple(int(v) for v in z["t_max_shape"])
    back = oracle.delta2bbox3d(z["t_props"], z["t_rand_deltas"], means, stds, max_shape=ms)
    assert np.abs(back - z["t_decoded"]).max() <= 1e-3                               # tolerance: 1e-3 px (exp)


@pytest.mark.parametrize("i", [0, 1])
def test_eval_nms_equals_the_reference_function(oracle, i):
    z = _load("python_ref.npz")
    assert np.array_equal(oracle.nms_3d_python(z["e_dets_%d" % i], 0.1), z["e_keep_%d" % i])


@pytest.mark.parametrize("i", [0, 1])
def test_random_sampler_equals_the_reference_class(oracle, i):
    """Same numpy seed -> the same sampled indices as the reference's RandomSampler.sample (gt boxes prepended when
    add_gt_as_proposals)."""
    z = _load("python_ref.npz")
    num, frac, ub, add_gt = z["s_cfg_%d" % i]
    gi = z["s_gt_inds_%d" % i]
    k = z["s_gt_%d" % i].shape[0]
    if add_gt:
        gi = np.concatenate([np.arange(1, k + 1), gi])
    np.random.seed(int(z["s_seed_%d" % i]))
    pos, neg = oracle.random_sample(gi, int(num), float(frac), float(ub))
    assert np.array_equal(pos, z["s_pos_inds_%d" % i]) and np.array_equal(neg, z["s_neg_inds_%d" % i])
    allb = np.concatenate([z["s_gt_%d" % i], z["s_boxes_%d" % i]]) if add_gt else z["s_boxes_%d" % i]
    assert np.array_equal(allb[pos], z["s_pos_bboxes_%d" % i])
    assert np.array_equal(gi[pos] - 1, z["s_pos_assigned_%d" % i])


def test_map_roi_levels_equals_the_reference_method(oracle):
    z = _load("python_ref.npz")
    assert np.array_equal(oracle.map_roi_levels(z["m_rois"], 4), z["m_levels"])


# ---- the same fixture against the product (device kernels through the Python mirror) ---------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("i", [0, 1, 2])
def test_device_anchor_generator_equals_the_reference_class(i):
    import torch
    from roi3d_b200 import AnchorGenerator3D
    z = _load("python_ref.npz")
    fm, st, sd, scales, dscales, ratios, valid, img_shape, border = ANCHOR_CASES[i]
    dev = torch.device("cuda:0")
    gen = AnchorGenerator3D(st, scales, dscales, ratios, sd)
    assert np.array_equal(gen.base_anchors.numpy(), z["anchor_base_%d" % i])
    a, f = gen.grid_anchors_and_inside_flags(fm, st, sd, valid, img_shape, border, device=dev)
    assert np.array_equal(a.cpu().numpy(), z["anchor_grid_%d" % i])
    assert np.array_equal(f.cpu().numpy(), z["anchor_inside_%d" % i])
    assert np.array_equal(gen.valid_flags(fm, valid, device=dev).cpu().numpy(), z["anchor_valid_%d" % i])


@pytest.mark.gpu
def test_device_eval_nms_map_levels_and_deltas_equal_the_reference():
    import torch
    import roi3d_b200
    from roi3d_b200.core.bbox import bbox2delta3d
    from roi3d_b200.core.evaluation import nms_3d_python
    z = _load("python_ref.npz")
    dev = torch.device("cuda:0")
    for i in (0, 1):
        dets = z["e_dets_%d" % i]
        kept = nms_3d_python(np.arange(len(dets)), dets, 0.1)
        assert np.array_equal(np.asarray(kept, dtype=np.int64), z["e_keep_%d" % i])
    ex = roi3d_b200.SingleRoIExtractor(dict(type='RoIAlign3D', out_size=7, out_size_depth=7, sample_num=2), 64,
                                       [4, 8, 16, 32], [2, 4, 8, 16])
    lv = ex.map_roi_levels(torch.from_numpy(z["m_rois"]).to(dev), 4)
    assert np.array_equal(lv.cpu().numpy(), z["m_levels"])
    d = bbox2delta3d(torch.from_numpy(z["t_props"]).to(dev), torch.from_numpy(z["t_gt"]).to(dev), (0.0,) * 6,
                     tuple(float(v) for v in z["t_stds"])).cpu().numpy()
    assert np.array_equal(d[:, [0, 1, 4]], z["t_deltas"][:, [0, 1, 4]])
    assert np.allclose(d[:, [2, 3, 5]], z["t_deltas"][:, [2, 3, 5]], rtol=1e-5, atol=1e-6)   # tolerance: 1e-5 (logf)


@pytest.mark.gpu
@pytest.mark.parametrize("i", [0, 1])
def test_device_random_sampler_equals_the_reference_class(i):
    import torch
    from roi3d_b200.core.bbox import AssignResult, RandomSampler
    z = _load("python_ref.npz")
    dev = torch.device("cuda:0")
    num, frac, ub, add_gt = z["s_cfg_%d" % i]
    gi, labels = z["s_gt_inds_%d" % i], z["s_labels_%d" % i]
    k = z["s_gt_%d" % i].shape[0]
    lab = labels[np.maximum(gi, 1) - 1] * (gi > 0)
    ar = AssignResult(k, torch.from_numpy(gi.copy()).to(dev), torch.zeros(len(gi), device=dev), labels=torch.from_numpy(lab).to(dev))
    np.random.seed(int(z["s_seed_%d" % i]))
    res = RandomSampler(int(num), float(frac), float(ub), bool(add_gt)).sample(
        ar, torch.from_numpy(z["s_boxes_%d" % i].copy()).to(dev), torch.from_numpy(z["s_gt_%d" % i]).to(dev),
        torch.from_numpy(labels).to(dev))
    assert np.array_equal(res.pos_inds.cpu().numpy(), z["s_pos_inds_%d" % i])
    assert np.array_equal(res.neg_inds.cpu().numpy(), z["s_neg_inds_%d" % i])
    assert np.array_equal(res.pos_bboxes.cpu().numpy(), z["s_pos_bboxes_%d" % i])
    assert np.array_equal(res.pos_assigned_gt_inds.cpu().numpy(), z["s_pos_assigned_%d" % i])

"""CPU oracle for the 3D RoI hot path -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this package, and only as the checker or the CPU baseline.  The product package
(``3d-multi-resolution-rcnn_b200/roi3d_b200``) never imports it.

The arithmetic lives in ``roi3d_oracle.c`` (each function cites the reference file:line it restates);
this module is the numpy/ctypes face of it plus the pure-numpy restatements of the reference's Python
glue (anchors, ``get_bboxes_single``, ``multiclass_nms_3d``, the numpy eval NMS).

Pinning status (see oracle/README.md):
  * 3D IoU: pinned by the reference's four known answers (mmdet/core/bbox/geometry.py:81-102).
  * RoIAlign3D fwd/bwd, 3D NMS: pinned against the reference's OWN kernels (oracle/_ref, built by
    oracle/build_ref.sh from /root/reference) run on the B200 box; outputs committed as fixtures under
    tests/golden/ (generator: tests/golden/make_golden.py).
  * level mapping, top-k tie order, delta2bbox3D last-bit behaviour: depend on torch==1.0.1 CUDA
    elementwise kernels that are not under /root/reference -> "parity unpinned" by the reference; the GPU
    tests compare against today's torch CUDA ops evaluating the same expressions.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liboracle.so")
_lib = None

_f32p = ctypes.POINTER(ctypes.c_float)
_i64p = ctypes.POINTER(ctypes.c_int64)
_u64p = ctypes.POINTER(ctypes.c_uint64)
_u8p = ctypes.POINTER(ctypes.c_ubyte)


def build(force=False):
    """Compile roi3d_oracle.c with gcc (about a second)."""
    src = os.path.join(_HERE, "roi3d_oracle.c")
    if (not force and os.path.exists(_LIB_PATH)
            and (not os.path.exists(src) or os.path.getmtime(_LIB_PATH) >= os.path.getmtime(src))):
        return _LIB_PATH
    subprocess.run(["make", "-s", "-C", _HERE, "_build/liboracle.so"], check=True)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.oracle_iou3d.restype = ctypes.c_float
        _lib.oracle_iou3d.argtypes = [_f32p, _f32p, ctypes.c_int]
        _lib.oracle_nms3d.restype = ctypes.c_int64
        _lib.oracle_nms3d.argtypes = [_f32p, ctypes.c_int64, ctypes.c_float, _i64p, _i64p, ctypes.c_int]
        _lib.oracle_nms3d_mask.restype = None
        _lib.oracle_nms3d_mask.argtypes = [_f32p, ctypes.c_int64, ctypes.c_float, _u64p, ctypes.c_int]
        _lib.oracle_argsort_desc_stable.restype = None
        _lib.oracle_argsort_desc_stable.argtypes = [_f32p, ctypes.c_int64, ctypes.c_int64, _i64p]
        _lib.oracle_roi_align3d_forward.restype = None
        _lib.oracle_roi_align3d_forward.argtypes = (
            [_f32p] + [ctypes.c_int] * 5 + [_f32p] + [ctypes.c_int] * 4 + [ctypes.c_float] * 2 +
            [ctypes.c_int, _f32p, ctypes.c_int])
        _lib.oracle_roi_align3d_backward.restype = None
        _lib.oracle_roi_align3d_backward.argtypes = (
            [_f32p, _f32p] + [ctypes.c_int] * 4 + [ctypes.c_float] * 2 + [ctypes.c_int, _f32p] +
            [ctypes.c_int] * 7)
        _lib.oracle_roi_align3d_unique_voxels.restype = ctypes.c_int64
        _lib.oracle_roi_align3d_unique_voxels.argtypes = (
            [_f32p] + [ctypes.c_int] * 8 + [ctypes.c_float] * 2 + [ctypes.c_int, _u8p])
        _lib.oracle_map_roi_levels.restype = None
        _lib.oracle_map_roi_levels.argtypes = [_f32p, ctypes.c_int64, ctypes.c_int, ctypes.c_float,
                                               ctypes.c_int, _i64p]
        _lib.oracle_delta2bbox3d.restype = None
        _lib.oracle_delta2bbox3d.argtypes = [_f32p, _f32p, ctypes.c_int64, _f32p, _f32p, ctypes.c_int,
                                             ctypes.c_float, ctypes.c_float, ctypes.c_float, _f32p]
        _lib.oracle_topk_desc_stable.restype = None
        _lib.oracle_topk_desc_stable.argtypes = [_f32p, ctypes.c_int64, ctypes.c_int64, _i64p]
        _lib.oracle_sigmoid.restype = None
        _lib.oracle_sigmoid.argtypes = [_f32p, ctypes.c_int64, _f32p]
        _lib.oracle_num_threads.restype = ctypes.c_int
        _lib.oracle_set_num_threads.argtypes = [ctypes.c_int]
    return _lib


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a, t=_f32p):
    return a.ctypes.data_as(t)


def num_threads():
    return int(lib().oracle_num_threads())


def set_num_threads(n):
    lib().oracle_set_num_threads(int(n))


# ----------------------------------------------------------------------------------------------
# C-backed restatements
# ----------------------------------------------------------------------------------------------
def iou3d(a, b, contract=True):
    """devIoU3d (mmdet/ops/nms/src/nms_kernel.cu:23-33); a, b = (x1,y1,x2,y2,z1,z2)."""
    a, b = _f32(a), _f32(b)
    return float(lib().oracle_iou3d(_p(a), _p(b), int(contract)))


def nms3d(dets, iou_thr, contract=True, return_score_order=False):
    """nms_cuda_3d (nms_kernel.cu:196-257): kept ORIGINAL indices, ascending (int64)."""
    dets = _f32(dets).reshape(-1, 7)
    n = dets.shape[0]
    keep = np.empty(max(n, 1), dtype=np.int64)
    so = np.empty(max(n, 1), dtype=np.int64)
    m = lib().oracle_nms3d(_p(dets), n, float(iou_thr), _p(keep, _i64p), _p(so, _i64p), int(contract))
    if return_score_order:
        return keep[:m].copy(), so[:m].copy()
    return keep[:m].copy()


def nms3d_mask(sorted_boxes, iou_thr, contract=True):
    """The suppression bit matrix nms_kernel_3d writes (nms_kernel.cu:81-129), [n, ceil(n/64)] uint64."""
    b = _f32(sorted_boxes).reshape(-1, 7)
    n = b.shape[0]
    cb = (n + 63) // 64
    mask = np.zeros((n, cb), dtype=np.uint64)
    lib().oracle_nms3d_mask(_p(b), n, float(iou_thr), _p(mask, _u64p), int(contract))
    return mask


def argsort_desc_stable(scores):
    s = _f32(scores).reshape(-1)
    order = np.empty(s.shape[0], dtype=np.int64)
    lib().oracle_argsort_desc_stable(_p(s), s.shape[0], 1, _p(order, _i64p))
    return order


def roi_align3d_forward(feats, rois, out_size, out_size_depth, spatial_scale, spatial_scale_depth,
                        sample_num=0, contract=True):
    """ROIAlignForward3D (roi_align_kernel.cu:214-291).  feats [B,C,D,H,W] (NCDHW), rois [K,7]; out_size is an int
    (square bins) or a (PH, PW) pair."""
    feats, rois = _f32(feats), _f32(rois).reshape(-1, 7)
    B, C, D, H, W = feats.shape
    K = rois.shape[0]
    PH, PW = (out_size, out_size) if np.ndim(out_size) == 0 else out_size
    PD, PH, PW = int(out_size_depth), int(PH), int(PW)
    out = np.empty((K, C, PD, PH, PW), dtype=np.float32)
    if K:
        lib().oracle_roi_align3d_forward(_p(feats), B, C, D, H, W, _p(rois), K, PD, PH, PW,
                                         float(spatial_scale), float(spatial_scale_depth), int(sample_num),
                                         _p(out), int(contract))
    return out


def roi_align3d_backward(grad_out, rois, feat_shape, spatial_scale, spatial_scale_depth, sample_num=0,
                         bug_compat=False, contract=True):
    """ROIAlignBackward3D (roi_align_kernel.cu:519-636); float64 accumulation of the fp32 terms."""
    grad_out, rois = _f32(grad_out), _f32(rois).reshape(-1, 7)
    K, C, PD, PH, PW = grad_out.shape
    B, C2, D, H, W = feat_shape
    assert C == C2
    gin = np.zeros((B, C, D, H, W), dtype=np.float32)
    lib().oracle_roi_align3d_backward(_p(grad_out), _p(rois), K, PD, PH, PW, float(spatial_scale),
                                      float(spatial_scale_depth), int(sample_num), _p(gin), B, C, D, H, W,
                                      int(bug_compat), int(contract))
    return gin


def roi_align3d_unique_voxels(rois, feat_shape, out_size, out_size_depth, spatial_scale,
                              spatial_scale_depth, sample_num=0):
    """U of SURVEY 8(d): distinct (b,z,y,x) voxels the RoI set reads."""
    rois = _f32(rois).reshape(-1, 7)
    B, _, D, H, W = feat_shape
    return int(lib().oracle_roi_align3d_unique_voxels(
        _p(rois), rois.shape[0], B, D, H, W, int(out_size_depth), int(out_size), int(out_size),
        float(spatial_scale), float(spatial_scale_depth), int(sample_num), None))


def map_roi_levels(rois, num_levels, finest_scale=56, recip_div=True):
    """SingleRoIExtractor.map_roi_levels (roi_extractors/single_level.py:58-82)."""
    rois = _f32(rois).reshape(-1, 7)
    out = np.empty(rois.shape[0], dtype=np.int64)
    lib().oracle_map_roi_levels(_p(rois), rois.shape[0], int(num_levels), float(finest_scale),
                                int(recip_div), _p(out, _i64p))
    return out


def delta2bbox3d(anchors, deltas, means=(0, 0, 0, 0, 0, 0), stds=(1, 1, 1, 1, 1, 1), max_shape=None):
    """delta2bbox3D (mmdet/core/bbox/transforms.py:105-160); max_shape = img_shape (H, W, 3, D)."""
    anchors, deltas = _f32(anchors).reshape(-1, 6), _f32(deltas).reshape(-1, 6)
    n = anchors.shape[0]
    out = np.empty((n, 6), dtype=np.float32)
    m, s = _f32(means), _f32(stds)
    if max_shape is None:
        has, mh, mw, md = 0, 0.0, 0.0, 0.0
    else:
        has, mh, mw, md = 1, float(max_shape[0]), float(max_shape[1]), float(max_shape[3])
    lib().oracle_delta2bbox3d(_p(anchors), _p(deltas), n, _p(m), _p(s), has, mh, mw, md, _p(out))
    return out


def topk(scores, k):
    """torch.topk restated with the build's tie rule (descending, ties -> lower index)."""
    s = _f32(scores).reshape(-1)
    k = int(min(k, s.shape[0]))
    idx = np.empty(max(k, 1), dtype=np.int64)
    lib().oracle_topk_desc_stable(_p(s), s.shape[0], k, _p(idx, _i64p))
    return idx[:k].copy()


def sigmoid(x):
    x = _f32(x)
    y = np.empty_like(x)
    lib().oracle_sigmoid(_p(x.reshape(-1)), x.size, _p(y.reshape(-1)))
    return y


# ----------------------------------------------------------------------------------------------
# numpy restatements of the reference's Python glue
# ----------------------------------------------------------------------------------------------
def nms_wrapper_3d(dets, iou_thr, contract=True):
    """mmdet.ops.nms for a CUDA [N,7] input (nms_wrapper.py:8-52): (dets[inds], inds)."""
    dets = _f32(dets).reshape(-1, 7)
    inds = nms3d(dets, iou_thr, contract) if dets.shape[0] else np.zeros(0, dtype=np.int64)
    return dets[inds, :], inds


def gen_base_anchors(base_size, scales, depth_scales, ratios, anchor_depth_base):
    """AnchorGenerator3D.gen_base_anchors (mmdet/core/anchor/anchor_generator_3d.py:22-53),
    scale_major=True, ctr=None."""
    w = h = np.float32(base_size)
    z = np.float32(anchor_depth_base)
    x_ctr, y_ctr, z_ctr = 0.5 * (w - 1), 0.5 * (h - 1), 0.5 * (z - 1)
    scales = np.asarray(scales, dtype=np.float32)
    dscales = np.asarray(depth_scales, dtype=np.float32)
    ratios = np.asarray(ratios, dtype=np.float32)
    h_ratios = np.sqrt(ratios)
    w_ratios = 1 / h_ratios
    ws = (w * w_ratios[:, None] * scales[None, :]).reshape(-1)
    hs = (h * h_ratios[:, None] * scales[None, :]).reshape(-1)
    zs = (z * h_ratios[:, None] * dscales[None, :]).reshape(-1)
    base = np.stack([x_ctr - 0.5 * (ws - 1), y_ctr - 0.5 * (hs - 1), x_ctr + 0.5 * (ws - 1),
                     y_ctr + 0.5 * (hs - 1), z_ctr - 0.5 * (zs - 1), z_ctr + 0.5 * (zs - 1)], axis=-1)
    return np.round(base.astype(np.float32)).astype(np.float32)  # torch.round: half to even, as np.round


def grid_anchors(base_anchors, featmap_size, stride, depth_stride):
    """AnchorGenerator3D.grid_anchors (anchor_generator_3d.py:56-71).  featmap_size = (D, H, W).
    np.meshgrid(x, y, z) with default 'xy' indexing flattens in (H, W, D) order, D fastest."""
    feat_z, feat_h, feat_w = featmap_size
    sx = np.arange(0, feat_w) * stride
    sy = np.arange(0, feat_h) * stride
    sz = np.arange(0, feat_z) * depth_stride
    xx, yy, zz = np.meshgrid(sx, sy, sz)
    xx, yy, zz = xx.flatten(), yy.flatten(), zz.flatten()
    shifts = np.column_stack((xx, yy, xx, yy, zz, zz)).astype(np.float32)
    allx = base_anchors[None, :, :] + shifts[:, None, :]
    return allx.reshape(-1, 6).astype(np.float32)


def get_bboxes_single(cls_scores, bbox_preds, mlvl_anchors, img_shape, nms_pre, nms_post, max_num, nms_thr,
                      target_means=(0, 0, 0, 0, 0, 0), target_stds=(1, 1, 1, 1, 1, 1),
                      nms_across_levels=False, contract=True, pos_indices=None, pos_indices_test=None, scores=None):
    """RPNHead3D.get_bboxes_single (mmdet/models/anchor_heads/rpn_head_3d.py:72-149), sigmoid scores,
    min_bbox_size == 0.  cls_scores[l]: [A, D, H, W]; bbox_preds[l]: [6A, D, H, W].  pos_indices / pos_indices_test:
    the head's cached per-level inside-flag masks (anchor_head_3d.py:212,239-243); a mask is applied only to a level
    with more than nms_pre anchors and only when its shape equals the scores' shape (:97-106).
    scores: optional per-level flat sigmoid scores to use instead of the host's 1/(1+expf(-x)) -- e.g. torch's CUDA
    sigmoid of the same logits, whose last bit can differ from glibc's expf and would otherwise reorder near-ties."""
    mlvl = []
    for lvl, (cls, reg, anchors) in enumerate(zip(cls_scores, bbox_preds, mlvl_anchors)):
        cls, reg = _f32(cls), _f32(reg)
        if scores is None:
            sc = sigmoid(np.transpose(cls, (2, 3, 1, 0)).reshape(-1))
        else:
            sc = _f32(scores[lvl]).reshape(-1)
        reg = np.transpose(reg, (2, 3, 1, 0)).reshape(-1, 6)
        anchors = _f32(anchors)
        if nms_pre > 0 and sc.shape[0] > nms_pre:
            sel = None
            if pos_indices is not None and np.asarray(pos_indices[lvl]).shape == sc.shape:
                sel = np.asarray(pos_indices[lvl]).astype(bool)
            elif pos_indices_test is not None and np.asarray(pos_indices_test[lvl]).shape == sc.shape:
                sel = np.asarray(pos_indices_test[lvl]).astype(bool)
            if sel is not None:
                sc, reg, anchors = sc[sel], reg[sel], anchors[sel]
        if nms_pre > 0 and sc.shape[0] > nms_pre:
            idx = topk(sc, nms_pre)
            reg, anchors, sc = reg[idx], anchors[idx], sc[idx]
        props = delta2bbox3d(anchors, reg, target_means, target_stds, img_shape)
        props = np.concatenate([props, sc[:, None]], axis=1)
        props, _ = nms_wrapper_3d(props, nms_thr, contract)
        mlvl.append(props[:nms_post])
    props = np.concatenate(mlvl, axis=0) if mlvl else np.zeros((0, 7), np.float32)
    if nms_across_levels:
        props, _ = nms_wrapper_3d(props, nms_thr, contract)
        props = props[:max_num]
    else:
        num = min(max_num, props.shape[0])
        props = props[topk(props[:, 6], num)]
    return props


def multiclass_nms_3d(multi_bboxes, multi_scores, score_thr, iou_thr, max_num=-1, contract=True):
    """multiclass_nms_3d (mmdet/core/post_processing/bbox_nms.py:57-106) with nms_cfg type 'nms'."""
    multi_bboxes, multi_scores = _f32(multi_bboxes), _f32(multi_scores)
    num_classes = multi_scores.shape[1]
    bboxes, labels = [], []
    for i in range(1, num_classes):
        sel = multi_scores[:, i] > np.float32(score_thr)
        if not sel.any():
            continue
        bb = multi_bboxes[sel, :] if multi_bboxes.shape[1] == 6 else multi_bboxes[sel, i * 6:(i + 1) * 6]
        dets = np.concatenate([bb, multi_scores[sel, i][:, None]], axis=1)
        dets, _ = nms_wrapper_3d(dets, iou_thr, contract)
        bboxes.append(dets)
        labels.append(np.full((dets.shape[0],), i - 1, dtype=np.int64))
    if bboxes:
        bboxes, labels = np.concatenate(bboxes), np.concatenate(labels)
        if bboxes.shape[0] > max_num:
            inds = argsort_desc_stable(bboxes[:, -1])[:max_num]
            bboxes, labels = bboxes[inds], labels[inds]
    else:
        bboxes, labels = np.zeros((0, 7), np.float32), np.zeros((0,), np.int64)
    return bboxes, labels


def nms_3d_python(boxes, iou_thr):
    """The reference's only CPU 3D-IoU NMS: nms_3d_python in mmdet/core/evaluation/coco_utils.py:245-282
    (numpy, keeps iou <= thr).  Returns kept indices in score order.  Dtype follows the input like numpy."""
    boxes = np.asarray(boxes)
    if len(boxes) == 0:
        return np.zeros(0, dtype=np.int64)
    x1, y1, x2, y2, z1, z2, s = (boxes[:, i] for i in range(7))
    vol = (x2 - x1 + 1) * (y2 - y1 + 1) * (z2 - z1 + 1)
    idxs = np.argsort(-s, kind="stable")
    keep = []
    while idxs.shape[0] > 0:
        i = idxs[0]
        keep.append(i)
        r = idxs[1:]
        xx1, yy1, zz1 = np.maximum(x1[r], x1[i]), np.maximum(y1[r], y1[i]), np.maximum(z1[r], z1[i])
        xx2, yy2, zz2 = np.minimum(x2[r], x2[i]), np.minimum(y2[r], y2[i]), np.minimum(z2[r], z2[i])
        inter = np.maximum(0, xx2 - xx1 + 1) * np.maximum(0, yy2 - yy1 + 1) * np.maximum(0, zz2 - zz1 + 1)
        iou = inter / (vol[i] + vol[r] - inter)
        nxt = np.nonzero(iou <= iou_thr)[0]
        if nxt.shape[0] == 0:
            break
        idxs = idxs[nxt + 1]
    return np.asarray(keep, dtype=np.int64)


def apply_nms(full_filename_to_id, json_results, nms_thresh=0.1, score_thresh=0):
    """apply_nms, mmdet/core/evaluation/coco_utils.py:306-332 (without the precomputed-proposal filter): per volume,
    scan all json results for the volume's image id, nms_3d_python on their 'original_bbox' rows (float64), keep the
    survivors in score order, drop those below score_thresh."""
    out = []
    for _filename, img_id in full_filename_to_id.items():
        cur = [r for r in json_results if r['image_id'] == img_id]
        if not cur:
            continue
        boxes = np.array([r['original_bbox'] for r in cur])
        for i in nms_3d_python(boxes, nms_thresh):
            if cur[i]['score'] < score_thresh:
                continue
            out.append(cur[i])
    return out


def bbox_overlaps3d(b1, b2):
    """bbox_overlaps, 6-column non-aligned branch (mmdet/core/bbox/geometry.py:49-60): fp32, one rounding per
    elementwise op like torch's separate kernels.  b1 [m,>=6], b2 [n,>=6] -> [m,n]."""
    b1, b2 = _f32(b1), _f32(b2)
    one = np.float32(1)
    xa = np.maximum(b1[:, None, 0], b2[None, :, 0])
    ya = np.maximum(b1[:, None, 1], b2[None, :, 1])
    xb = np.minimum(b1[:, None, 2], b2[None, :, 2])
    yb = np.minimum(b1[:, None, 3], b2[None, :, 3])
    za = np.maximum(b1[:, None, 4], b2[None, :, 4])
    zb = np.minimum(b1[:, None, 5], b2[None, :, 5])
    zero = np.float32(0)
    inter = np.maximum(xb - xa + one, zero) * np.maximum(yb - ya + one, zero) * np.maximum(zb - za + one, zero)
    a1 = (b1[:, 2] - b1[:, 0] + one) * (b1[:, 3] - b1[:, 1] + one) * (b1[:, 5] - b1[:, 4] + one)
    a2 = (b2[:, 2] - b2[:, 0] + one) * (b2[:, 3] - b2[:, 1] + one) * (b2[:, 5] - b2[:, 4] + one)
    with np.errstate(invalid="ignore", divide="ignore"):
        return (inter / (a1[:, None] + a2[None, :] - inter)).astype(np.float32)


def assign_max_iou(bboxes, gt_bboxes, gt_labels=None, pos_iou_thr=0.5, neg_iou_thr=0.5, min_pos_iou=0.0,
                   gt_max_assign_all=True, ignore_iof_thr=-1, ignore_wrt_candidates=True, gt_bboxes_ignore=None):
    """MaxIoUAssigner.assign + assign_wrt_overlaps (mmdet/core/bbox/assigners/max_iou_assigner.py:100-171), the
    ignore branch (:101-111) included: for 6-column boxes the reference's bbox_overlaps(..., mode='iof') is the IoU
    (geometry.py:49-60 never reads `mode`).  Ties of max(dim) go to the lowest index.  Pinned: tests/golden/
    assigner_ref.npz holds the outputs of the reference's own class on twelve seeded cases (test_golden.py).  Returns (assigned_gt_inds int64 [n], max_overlaps fp32 [n], labels int64 [n] or None)."""
    ov = bbox_overlaps3d(_f32(gt_bboxes)[:, :6], _f32(bboxes)[:, :6])  # [k, n]
    if ignore_iof_thr > 0 and gt_bboxes_ignore is not None and np.asarray(gt_bboxes_ignore).size > 0:
        gi = _f32(gt_bboxes_ignore)[:, :6]
        if ignore_wrt_candidates:
            ign_max = bbox_overlaps3d(_f32(bboxes)[:, :6], gi).max(axis=1)
        else:
            ign_max = bbox_overlaps3d(gi, _f32(bboxes)[:, :6]).max(axis=0)
        ov[:, ign_max > ignore_iof_thr] = -1
    k, n = ov.shape
    assigned = np.full(n, -1, dtype=np.int64)
    max_ov, argmax_ov = ov.max(axis=0), ov.argmax(axis=0)
    gt_max, gt_argmax = ov.max(axis=1), ov.argmax(axis=1)
    if isinstance(neg_iou_thr, float):
        assigned[(max_ov >= 0) & (max_ov < np.float32(neg_iou_thr))] = 0
    elif isinstance(neg_iou_thr, tuple):
        assigned[(max_ov >= np.float32(neg_iou_thr[0])) & (max_ov < np.float32(neg_iou_thr[1]))] = 0
    pos = max_ov >= np.float32(pos_iou_thr)
    assigned[pos] = argmax_ov[pos] + 1
    for i in range(k):
        if gt_max[i] >= np.float32(min_pos_iou):
            if gt_max_assign_all:
                assigned[ov[i, :] == gt_max[i]] = i + 1
            else:
                assigned[gt_argmax[i]] = i + 1
    labels = None
    if gt_labels is not None:
        gl = np.asarray(gt_labels, dtype=np.int64)
        labels = np.zeros(n, dtype=np.int64)
        p = assigned > 0
        labels[p] = gl[assigned[p] - 1]
    return assigned, max_ov.astype(np.float32), labels


def bbox2delta3d(proposals, gt, means=(0, 0, 0, 0, 0, 0), stds=(1, 1, 1, 1, 1, 1)):
    """bbox2delta3d (mmdet/core/bbox/transforms.py:33-63), fp32 numpy: (dx, dy, dw, dh, dz, dd)."""
    p, g = _f32(proposals), _f32(gt)
    half, one = np.float32(0.5), np.float32(1)
    cols = []
    enc = {}
    for name, lo, hi in (("x", 0, 2), ("y", 1, 3), ("z", 4, 5)):
        pc, ps = (p[:, lo] + p[:, hi]) * half, p[:, hi] - p[:, lo] + one
        gc, gs = (g[:, lo] + g[:, hi]) * half, g[:, hi] - g[:, lo] + one
        with np.errstate(invalid="ignore", divide="ignore"):
            enc[name] = ((gc - pc) / ps, np.log(gs / ps))
    cols = [enc["x"][0], enc["y"][0], enc["x"][1], enc["y"][1], enc["z"][0], enc["z"][1]]
    d = np.stack(cols, axis=-1).astype(np.float32)
    return ((d - _f32(np.asarray(means))[None]) / _f32(np.asarray(stds))[None]).astype(np.float32)


def valid_flags(featmap_size, valid_size, num_base_anchors):
    """AnchorGenerator3D.valid_flags (mmdet/core/anchor/anchor_generator_3d.py:73-92): np.meshgrid(x, y, z) order."""
    fz, fh, fw = featmap_size
    vd, vh, vw = valid_size
    vx, vy, vz = np.zeros(fw, np.uint8), np.zeros(fh, np.uint8), np.zeros(fz, np.uint8)
    vx[:vw], vy[:vh], vz[:vd] = 1, 1, 1
    xx, yy, zz = np.meshgrid(vx, vy, vz)
    v = xx.flatten() & yy.flatten() & zz.flatten()
    return np.repeat(v, num_base_anchors)


def anchor_inside_flags(flat_anchors, valid, img_shape, allowed_border=0):
    """anchor_inside_flags, 6-column branch (mmdet/core/anchor/anchor_target.py:203-217); img_shape = (H, W, 3, D)."""
    a = _f32(flat_anchors)
    if allowed_border < 0:
        return valid
    h, w, d = img_shape[0], img_shape[1], img_shape[3]
    ins = (a[:, 0] >= -allowed_border) & (a[:, 1] >= -allowed_border) & (a[:, 4] >= -allowed_border) & \
        (a[:, 2] < w + allowed_border) & (a[:, 3] < h + allowed_border) & (a[:, 5] < d + allowed_border)
    return valid & ins.astype(valid.dtype)


def resize_nd(image, output_shape):
    """skimage.transform.resize(image, output_shape) for a float n-D image with the defaults the reference uses
    (mmdet/models/mask_heads/fcn_mask_head_3d.py:181): scikit-image==0.18.0 (requirements.txt:24), n-dimensional
    branch of skimage/transform/_warps.py -- anti_aliasing on, sigma = max(0, (factors - 1) / 2), gaussian_filter
    and order-1 map_coordinates with ndimage mode 'mirror' (skimage mode 'reflect'), clip to the input range.
    The two primitives are scipy.ndimage's (scipy==1.5.4 pinned by the reference, requirements.txt:25; this image
    has a newer scipy whose order-1 / mirror behaviour is the same).  skimage itself is not installed: parity
    unpinned by the reference."""
    import scipy.ndimage as ndi
    image = np.asarray(image, dtype=np.float32)
    factors = np.divide(np.asarray(image.shape, dtype=np.float64), np.asarray(output_shape, dtype=np.float64))
    sigma = np.maximum(0, (factors - 1) / 2)
    img = ndi.gaussian_filter(image, sigma, cval=0, mode='mirror')
    coords = [factors[i] * (np.arange(d) + 0.5) - 0.5 for i, d in enumerate(output_shape)]
    cmap = np.array(np.meshgrid(*coords, sparse=False, indexing='ij'))
    out = ndi.map_coordinates(img, cmap, order=1, mode='mirror', cval=0)
    return np.clip(out, img.min(), img.max())


def get_seg_masks_compact(mask_logits, det_bboxes, det_labels, mask_thr_binary, scale_factor=1.0, class_agnostic=False):
    """The per-detection part of FCNMaskHead3D.get_seg_masks (fcn_mask_head_3d.py:144-185): returns (int boxes,
    list of uint8 (d, h, w) masks, 1-based labels).  mask_logits [n, classes, Dm, Hm, Wm]; sigmoid = oracle.sigmoid."""
    probs = sigmoid(np.asarray(mask_logits, dtype=np.float32))
    bboxes = np.asarray(det_bboxes, dtype=np.float32)[:, :6]
    labels = np.asarray(det_labels) + 1
    boxes, masks = [], []
    for i in range(bboxes.shape[0]):
        bbox = (bboxes[i, :] / scale_factor).astype(np.int32)
        w = max(bbox[2] - bbox[0] + 1, 1)
        h = max(bbox[3] - bbox[1] + 1, 1)
        d = max(bbox[5] - bbox[4] + 1, 1)
        m = probs[i, 0 if class_agnostic else labels[i]]
        masks.append((resize_nd(m, (d, h, w)) > mask_thr_binary).astype(np.uint8))
        boxes.append(bbox)
    return np.asarray(boxes, dtype=np.int32).reshape(-1, 6), masks, labels


def resize_nd_f64(image, output_shape):
    """skimage.transform.resize on a uint8 image as mask_target_single uses it (mmdet/core/mask/mask_target.py:42):
    img_as_float maps uint8 v to float64 v * (1 / 255); the rest is resize_nd in float64."""
    import scipy.ndimage as ndi
    image = np.multiply(np.asarray(image, dtype=np.uint8), 1.0 / 255, dtype=np.float64)
    factors = np.divide(np.asarray(image.shape, dtype=np.float64), np.asarray(output_shape, dtype=np.float64))
    sigma = np.maximum(0, (factors - 1) / 2)
    img = ndi.gaussian_filter(image, sigma, cval=0, mode='mirror')
    coords = [factors[i] * (np.arange(d) + 0.5) - 0.5 for i, d in enumerate(output_shape)]
    cmap = np.array(np.meshgrid(*coords, sparse=False, indexing='ij'))
    out = ndi.map_coordinates(img, cmap, order=1, mode='mirror', cval=0)
    return np.clip(out, img.min(), img.max())


def mask_target_single(pos_proposals, pos_assigned_gt_inds, gt_masks, mask_size, mask_size_depth, return_scaled=False):
    """mask_target_single (mmdet/core/mask/mask_target.py:17-50), 3D branch; gt_masks uint8 [G, D, H, W].
    return_scaled: also return the float64 `255 * resize(...)` values before the uint8 truncation."""
    props = np.asarray(pos_proposals, dtype=np.float32)
    out, scaled = [], []
    for i in range(props.shape[0]):
        x1, y1, x2, y2, z1, z2 = props[i].astype(np.int32)
        w, h, d = max(x2 - x1 + 1, 1), max(y2 - y1 + 1, 1), max(z2 - z1 + 1, 1)
        crop = np.asarray(gt_masks[int(pos_assigned_gt_inds[i])])[z1:z1 + d, y1:y1 + h, x1:x1 + w]
        t = 255 * resize_nd_f64(crop, (mask_size_depth, mask_size, mask_size))
        scaled.append(t)
        t = t.astype(np.uint8)
        t[t > 0] = 1
        out.append(t)
    if not out:
        return np.zeros((0, mask_size, mask_size), np.float32)
    if return_scaled:
        return np.stack(out).astype(np.float32), np.stack(scaled)
    return np.stack(out).astype(np.float32)


def random_sample(gt_inds, num, pos_fraction, neg_pos_ub=-1):
    """RandomSampler.sample's index selection (mmdet/core/bbox/samplers/base_sampler.py:73-101 with
    random_sampler.py:19-58) on a numpy gt_inds vector (after add_gt_); consumes np.random like the reference."""
    gt_inds = np.asarray(gt_inds)

    def pick(cands, n):
        if len(cands) <= n:
            return cands
        return cands[np.random.randint(low=0, high=len(cands), size=n)]
    pos = np.unique(pick(np.nonzero(gt_inds > 0)[0], int(num * pos_fraction)))
    n_neg = num - len(pos)
    if neg_pos_ub >= 0:
        n_neg = min(n_neg, int(neg_pos_ub * max(1, len(pos))))
    neg = np.unique(pick(np.nonzero(gt_inds == 0)[0], n_neg))
    return pos, neg


def nms_cpu_2d(dets, thr):
    """nms_cpu_kernel (mmdet/ops/nms/src/nms_cpu.cpp:5-59): 2-D NMS over columns 0-3 ranked by column 4,
    suppressing ovr >= thr -- what the reference's CPU wrapper runs even on 7-column input (SURVEY F3)."""
    dets = _f32(dets)
    n = dets.shape[0]
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    x1, y1, x2, y2, sc = dets[:, 0], dets[:, 1], dets[:, 2], dets[:, 3], dets[:, 4]
    areas = (x2 - x1 + 1) * (y2 - y1 + 1)
    order = argsort_desc_stable(sc)
    sup = np.zeros(n, dtype=bool)
    for _i in range(n):
        i = order[_i]
        if sup[i]:
            continue
        r = order[_i + 1:]
        r = r[~sup[r]]
        w = np.maximum(np.float32(0), np.minimum(x2[i], x2[r]) - np.maximum(x1[i], x1[r]) + 1)
        h = np.maximum(np.float32(0), np.minimum(y2[i], y2[r]) - np.maximum(y1[i], y1[r]) + 1)
        inter = w * h
        ovr = inter / (areas[i] + areas[r] - inter)
        sup[r[ovr >= np.float32(thr)]] = True
    return np.nonzero(~sup)[0].astype(np.int64)

"""CPU oracle of the RPN proposal path with `min_bbox_size > 0` -- TEST INFRASTRUCTURE ONLY (tests/ and
tools/bench_rpn_min_bbox_size.py).

`filter_min_bbox_size` is the filter of mmdetection v0.6.0's RPNHead.get_bboxes_single; `get_bboxes_single` is
oracle.get_bboxes_single (RPNHead3D.get_bboxes_single, mmdet/models/anchor_heads/rpn_head_3d.py:72-149) with that
filter between each level's decode and its NMS, built from the same oracle pieces.  At min_bbox_size <= 0 it is
oracle.get_bboxes_single step for step (a CPU test checks that they agree bit for bit)."""
import numpy as np

import oracle


def filter_min_bbox_size(props, min_bbox_size):
    """The `min_bbox_size` filter on decoded [n, >=4] rows: keep a row iff (x2 - x1) + 1 >= m and (y2 - y1) + 1 >= m in
    fp32, m = min_bbox_size rounded to fp32 (NaN fails); depth is not compared.  The kept rows, in order (one survivor
    stays a one-row array)."""
    props = np.ascontiguousarray(props, dtype=np.float32)
    m = np.float32(min_bbox_size)
    with np.errstate(invalid="ignore", over="ignore"):
        w = (props[:, 2] - props[:, 0]) + np.float32(1)
        h = (props[:, 3] - props[:, 1]) + np.float32(1)
        keep = (w >= m) & (h >= m)
    return props[keep]


def get_bboxes_single(cls_scores, bbox_preds, mlvl_anchors, img_shape, nms_pre, nms_post, max_num, nms_thr,
                      target_means=(0, 0, 0, 0, 0, 0), target_stds=(1, 1, 1, 1, 1, 1), nms_across_levels=False,
                      contract=True, pos_indices=None, pos_indices_test=None, scores=None, min_bbox_size=0):
    """oracle.get_bboxes_single's arguments, plus min_bbox_size (> 0: filter_min_bbox_size after each level's decode)."""
    mlvl = []
    for lvl, (cls, reg, anchors) in enumerate(zip(cls_scores, bbox_preds, mlvl_anchors)):
        cls, reg = np.asarray(cls, np.float32), np.asarray(reg, np.float32)
        if scores is None:
            sc = oracle.sigmoid(np.transpose(cls, (2, 3, 1, 0)).reshape(-1))
        else:
            sc = np.asarray(scores[lvl], np.float32).reshape(-1)
        reg = np.transpose(reg, (2, 3, 1, 0)).reshape(-1, 6)
        anchors = np.asarray(anchors, np.float32)
        if nms_pre > 0 and sc.shape[0] > nms_pre:
            sel = None
            if pos_indices is not None and np.asarray(pos_indices[lvl]).shape == sc.shape:
                sel = np.asarray(pos_indices[lvl]).astype(bool)
            elif pos_indices_test is not None and np.asarray(pos_indices_test[lvl]).shape == sc.shape:
                sel = np.asarray(pos_indices_test[lvl]).astype(bool)
            if sel is not None:
                sc, reg, anchors = sc[sel], reg[sel], anchors[sel]
        if nms_pre > 0 and sc.shape[0] > nms_pre:
            idx = oracle.topk(sc, nms_pre)
            reg, anchors, sc = reg[idx], anchors[idx], sc[idx]
        props = oracle.delta2bbox3d(anchors, reg, target_means, target_stds, img_shape)
        props = np.concatenate([props, sc[:, None]], axis=1)
        if min_bbox_size > 0:
            props = filter_min_bbox_size(props, min_bbox_size)
        props, _ = oracle.nms_wrapper_3d(props, nms_thr, contract)
        mlvl.append(props[:nms_post])
    props = np.concatenate(mlvl, axis=0) if mlvl else np.zeros((0, 7), np.float32)
    if nms_across_levels:
        props, _ = oracle.nms_wrapper_3d(props, nms_thr, contract)
        props = props[:max_num]
    else:
        num = min(max_num, props.shape[0])
        props = props[oracle.topk(props[:, 6], num)]
    return props

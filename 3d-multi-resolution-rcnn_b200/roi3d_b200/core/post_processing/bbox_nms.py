"""multiclass_nms_3d on the B200 NMS (reference: mmdet/core/post_processing/bbox_nms.py:57-106).

Same arguments and return value.  The reference loops over classes with a `.any()` host sync, a boolean-mask
gather and a host-synchronising NMS per class; here every class is one segment of a single batched NMS launch
and the only host read is the final per-class kept count (the result length is data dependent).
nms_cfg type 'nms' runs the hard 3D NMS; type 'soft_nms' runs the 3D soft-NMS with the remaining keys (iou_thr,
method, sigma, min_score) and keeps each class's rows in selection order with their decayed scores.
"""
import torch

from ...ops.nms import nms_wrapper


def multiclass_nms_3d(multi_bboxes, multi_scores, score_thr, nms_cfg, max_num=-1):
    """multi_bboxes [n, #class*6] or [n, 6]; multi_scores [n, #class] (class 0 = background).
    Returns (bboxes [k,7], labels [k] int64, 0-based)."""
    num_classes = multi_scores.shape[1]
    nms_cfg_ = dict(nms_cfg)
    nms_type = nms_cfg_.pop('type', 'nms')
    if nms_type not in ('nms', 'soft_nms'):
        raise NotImplementedError("nms type %r is not part of the 3D RoI hot path" % (nms_type,))
    iou_thr = float(nms_cfg_.pop('iou_thr'))
    n = multi_bboxes.shape[0]
    dev = multi_bboxes.device
    ncls = num_classes - 1
    if n == 0 or ncls <= 0:
        return multi_bboxes.new_zeros((0, 7)), multi_bboxes.new_zeros((0,), dtype=torch.long)
    scores = multi_scores[:, 1:].t().contiguous()                      # [ncls, n]
    if multi_bboxes.shape[1] == 6:
        boxes = multi_bboxes[None].expand(ncls, -1, -1)
    else:
        boxes = multi_bboxes.view(n, num_classes, 6)[:, 1:].permute(1, 0, 2)
    sel = scores > score_thr                                           # (:79)
    counts = sel.sum(dim=1).to(torch.int32)
    # stable compaction of the selected rows to the front of each class segment (original order kept)
    order = torch.sort((~sel).to(torch.uint8), dim=1, stable=True)[1]
    dets = torch.cat([torch.gather(boxes, 1, order[:, :, None].expand(-1, -1, 6)),
                      torch.gather(scores, 1, order)[:, :, None]], dim=2).contiguous()   # [ncls, n, 7]
    if nms_type == 'soft_nms':
        out, _, num = nms_wrapper.soft_nms3d_batched(dets, counts, iou_thr, **nms_cfg_)
    else:
        keep, _, num = nms_wrapper.nms3d_batched(dets, counts, iou_thr, want_score_order=False)
    num_h = num.tolist()                                               # the one host read
    bboxes, labels = [], []
    for c in range(ncls):
        if num_h[c] == 0:
            continue
        bboxes.append(out[c, :num_h[c]] if nms_type == 'soft_nms' else dets[c, keep[c, :num_h[c]]])
        labels.append(multi_bboxes.new_full((num_h[c],), c, dtype=torch.long))
    if not bboxes:
        return multi_bboxes.new_zeros((0, 7)), multi_bboxes.new_zeros((0,), dtype=torch.long)
    bboxes, labels = torch.cat(bboxes), torch.cat(labels)
    if bboxes.shape[0] > max_num:
        inds = torch.sort(bboxes[:, -1], descending=True, stable=True)[1][:max_num]
        bboxes, labels = bboxes[inds], labels[inds]
    return bboxes, labels

"""multiclass_nms_3d on the B200 NMS (reference: mmdet/core/post_processing/bbox_nms.py:57-106), and its batched,
fixed-shape form multiclass_nms_3d_batched.

Same arguments and return value.  The reference loops over classes with a `.any()` host sync, a boolean-mask
gather and a host-synchronising NMS per class; here every class is one segment of a single batched NMS launch
and the only host read is the final per-class kept count (the result length is data dependent).
nms_cfg type 'nms' runs the hard 3D NMS; type 'soft_nms' runs the 3D soft-NMS with the remaining keys (iou_thr,
method, sigma, min_score) and keeps each class's rows in selection order with their decayed scores.
"""
import torch

from ... import _lib
from ..._util import check_cuda_f32, device_guard, nvtx_range, stream_ptr, workspace
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


def multiclass_nms_3d_batched(multi_bboxes, multi_scores, counts, score_thr, nms_cfg, max_num=-1):
    """multiclass_nms_3d for B images in one call (roi3d_multiclass_nms3d_batched), with nothing read back to the host.

    multi_bboxes [B, n, #class*6] or [B, n, 6] and multi_scores [B, n, #class] fp32 CUDA (class 0 = background);
    counts int32 [B] CUDA: image b uses its first counts[b] rows (the rows past it are never read).  nms_cfg and max_num
    as in multiclass_nms_3d.  Returns device tensors (det [B, M, 7], labels [B, M] int64 0-based, det_counts [B] int32)
    with M = max_num if max_num > 0 else (#class - 1) * n: the first det_counts[b] rows of image b are
    multiclass_nms_3d(multi_bboxes[b, :counts[b]], multi_scores[b, :counts[b]], ...), the rows after them are zeros with
    label -1.  The shapes depend on the arguments only, so the call can be captured in a CUDA graph."""
    nms_cfg_ = dict(nms_cfg)
    nms_type = nms_cfg_.pop('type', 'nms')
    if nms_type not in ('nms', 'soft_nms'):
        raise NotImplementedError("nms type %r is not part of the 3D RoI hot path" % (nms_type,))
    iou_thr = float(nms_cfg_.pop('iou_thr'))
    method, sigma, min_score = 1, 0.5, 1e-3
    if nms_type == 'soft_nms':
        method_name = nms_cfg_.pop('method', 'linear')
        if method_name not in nms_wrapper.SOFT_NMS_METHODS:
            raise ValueError('Invalid method for SoftNMS: {}'.format(method_name))
        method = nms_wrapper.SOFT_NMS_METHODS[method_name]
        sigma = float(nms_cfg_.pop('sigma', sigma))
        min_score = float(nms_cfg_.pop('min_score', min_score))
        if nms_cfg_:
            raise TypeError("soft_nms: unexpected nms_cfg keys %s" % sorted(nms_cfg_))
    check_cuda_f32(multi_bboxes, "multi_bboxes", ndim=3)
    check_cuda_f32(multi_scores, "multi_scores", ndim=3)
    if not isinstance(counts, torch.Tensor) or not counts.is_cuda:
        raise NotImplementedError("counts must be an int32 CUDA tensor: the B200 path has no CPU implementation")
    B, n, num_classes = multi_scores.shape
    if num_classes < 2:
        raise ValueError("multi_scores [B, n, #class] needs #class >= 2 (class 0 is the background), got shape %s"
                         % (tuple(multi_scores.shape),))
    box_cols = multi_bboxes.shape[2]
    if tuple(multi_bboxes.shape[:2]) != (B, n) or box_cols not in (6, 6 * num_classes):
        raise ValueError("multi_bboxes must be [B, n, 6] or [B, n, %d] for multi_scores %s, got %s"
                         % (6 * num_classes, tuple(multi_scores.shape), tuple(multi_bboxes.shape)))
    if counts.dtype != torch.int32 or tuple(counts.shape) != (B,):
        raise ValueError("counts must be int32 [%d], got %s %s" % (B, counts.dtype, tuple(counts.shape)))
    max_num = int(max_num)
    soft = int(nms_type == 'soft_nms')
    M = max_num if max_num > 0 else (num_classes - 1) * n
    dev = multi_scores.device
    bboxes, scores, counts = multi_bboxes.contiguous(), multi_scores.contiguous(), counts.contiguous()
    det = torch.empty((B, M, 7), dtype=torch.float32, device=dev)
    labels = torch.empty((B, M), dtype=torch.int64, device=dev)
    det_counts = torch.empty((B,), dtype=torch.int32, device=dev)
    nbytes = _lib.lib.roi3d_multiclass_nms3d_workspace_bytes(B, n, num_classes, max_num, soft)
    _buf, ws = workspace(dev, nbytes)
    with device_guard(dev), nvtx_range("roi3d.multiclass_nms3d_batched"):
        _lib.check(_lib.lib.roi3d_multiclass_nms3d_batched(
            bboxes.data_ptr(), box_cols, scores.data_ptr(), counts.data_ptr(), B, n, num_classes, float(score_thr),
            soft, iou_thr, method, sigma, min_score, max_num, det.data_ptr(), labels.data_ptr(), det_counts.data_ptr(),
            ws, nbytes, stream_ptr()))
    return det, labels, det_counts

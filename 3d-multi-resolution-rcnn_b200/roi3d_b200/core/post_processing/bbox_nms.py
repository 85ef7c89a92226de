"""multiclass_nms_3d on the B200 (reference: mmdet/core/post_processing/bbox_nms.py:57-106), and its batched,
fixed-shape form multiclass_nms_3d_batched.

multiclass_nms_3d_batched is the implementation: one call of roi3d_multiclass_nms3d_batched runs the reference's
policy for B images on the device (score_thr select, stable per-class compaction, NMS or soft-NMS per class, class-major
concatenation, the `[:max_num]` cut) and reads nothing back to the host.  The reference instead loops over classes with
a `.any()` host sync, a boolean-mask gather and a host-synchronising NMS per class.  multiclass_nms_3d has the
reference's arguments and return value: it is the batched call at B = 1 plus one host read, the kept count, because
the length of its result depends on the data.
nms_cfg type 'nms' runs the hard 3D NMS; type 'soft_nms' runs the 3D soft-NMS with the remaining keys (iou_thr,
method, sigma, min_score) and keeps each class's rows in selection order with their decayed scores.
"""
import torch

from ... import _lib
from ..._util import check_cuda_f32, device_guard, nvtx_range, stream_ptr, workspace
from ...ops.nms import nms_wrapper


def _parse_nms_cfg(nms_cfg):
    """nms_cfg -> (soft, iou_thr, method, sigma, min_score) as roi3d_multiclass_nms3d_batched takes them."""
    cfg = dict(nms_cfg)
    nms_type = cfg.pop('type', 'nms')
    if nms_type not in ('nms', 'soft_nms'):
        raise NotImplementedError("nms type %r is not part of the 3D RoI hot path" % (nms_type,))
    iou_thr = float(cfg.pop('iou_thr'))
    method, sigma, min_score = 1, 0.5, 1e-3
    if nms_type == 'nms':
        return 0, iou_thr, method, sigma, min_score
    method_name = cfg.pop('method', 'linear')
    if method_name not in nms_wrapper.SOFT_NMS_METHODS:
        raise ValueError('Invalid method for SoftNMS: {}'.format(method_name))
    method = nms_wrapper.SOFT_NMS_METHODS[method_name]
    sigma = float(cfg.pop('sigma', sigma))
    min_score = float(cfg.pop('min_score', min_score))
    if cfg:
        raise TypeError("soft_nms: unexpected nms_cfg keys %s" % sorted(cfg))
    return 1, iou_thr, method, sigma, min_score


def multiclass_nms_3d(multi_bboxes, multi_scores, score_thr, nms_cfg, max_num=-1):
    """multi_bboxes [n, #class*6] or [n, 6]; multi_scores [n, #class] (class 0 = background).
    Returns (bboxes [k,7], labels [k] int64, 0-based).

    multiclass_nms_3d_batched on this one image, then one host read of its kept count."""
    num_classes = multi_scores.shape[1]
    n = multi_bboxes.shape[0]
    if n == 0 or num_classes < 2:
        _parse_nms_cfg(nms_cfg)   # an invalid nms_cfg raises here as it does on a non-empty input
        return multi_bboxes.new_zeros((0, 7)), multi_bboxes.new_zeros((0,), dtype=torch.long)
    counts = torch.full((1,), n, dtype=torch.int32, device=multi_bboxes.device)
    # no image keeps more than (#class - 1) * n rows: a larger max_num cuts nothing and would only size the outputs
    max_num = min(int(max_num), (num_classes - 1) * n)
    det, labels, det_counts = multiclass_nms_3d_batched(multi_bboxes[None], multi_scores[None], counts, score_thr,
                                                        nms_cfg, max_num)
    m = int(det_counts[0])   # the one host read: the result length is data dependent
    return det[0, :m], labels[0, :m]


def multiclass_nms_3d_batched(multi_bboxes, multi_scores, counts, score_thr, nms_cfg, max_num=-1):
    """multiclass_nms_3d for B images in one call (roi3d_multiclass_nms3d_batched), with nothing read back to the host.

    multi_bboxes [B, n, #class*6] or [B, n, 6] and multi_scores [B, n, #class] fp32 CUDA (class 0 = background);
    counts int32 [B] CUDA: image b uses its first counts[b] rows (the rows past it are never read).  score_thr, nms_cfg
    and max_num as in the reference's multiclass_nms_3d, including its `[:max_num]` slice rule: max_num = 0 keeps
    nothing, max_num < 0 keeps all but the last -max_num rows in descending score order.  Returns device tensors (det
    [B, M, 7], labels [B, M] int64 0-based, det_counts [B] int32) with M = max_num if max_num > 0 else (#class - 1) * n:
    the first det_counts[b] rows of image b are the reference's result on multi_bboxes[b, :counts[b]] and
    multi_scores[b, :counts[b]], the rows after them are zeros with label -1.  The shapes depend on the arguments only,
    so the call can be captured in a CUDA graph."""
    soft, iou_thr, method, sigma, min_score = _parse_nms_cfg(nms_cfg)
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

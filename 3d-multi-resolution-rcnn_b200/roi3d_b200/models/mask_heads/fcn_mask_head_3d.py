"""Mask paste of the 3D mask head on the device (SURVEY section 8f, N4).

Reference: FCNMaskHead3D.get_seg_masks, mmdet/models/mask_heads/fcn_mask_head_3d.py:124-187 -- for every detection,
on the host: sigmoid -> numpy, `skimage.transform.resize` to the box size, threshold, paste into a full-volume uint8
array.  Here every detection's resize + threshold runs in one launch of `roi3d_mask_paste_select`
(csrc/mask_paste.cu), which reads each detection's class channel of the head's output [n, classes, 20, 28, 28] in
place.  `paste_masks_device` keeps the box-sized binary masks on the device (what a B200 pipeline and
`parallel.gather_detections` use), `paste_masks_compact` reads them back, `get_seg_masks` returns the reference's
structure (a full-volume array per detection, grouped by class).
"""
import numpy as np
import torch

from ... import _lib
from ..._util import check_cuda_f32, device_guard, stream_ptr


def paste_masks_device(mask_pred, det_bboxes, det_labels, mask_thr_binary, scale_factor=1.0, class_agnostic=False):
    """mask_pred [n, num_classes, Dm, Hm, Wm] CUDA fp32 LOGITS (the head's output before sigmoid, as get_seg_masks
    receives it); det_bboxes [n, >=6]; det_labels [n] (0-based foreground labels).
    Returns device tensors (boxes int32 [n, 6], offsets int64 [n + 1], masks uint8 flat, labels int64 1-based):
    detection i's mask is masks[offsets[i]:offsets[i + 1]], shape (z2-z1+1, y2-y1+1, x2-x1+1) of its box (each at
    least 1).  One host read (the total mask size, to allocate the output)."""
    check_cuda_f32(mask_pred, "mask_pred", ndim=5)
    mask_pred = mask_pred.detach().contiguous()
    n, num_channels, Dm, Hm, Wm = mask_pred.shape
    dev = mask_pred.device
    b = det_bboxes.detach()[:, :6].to(dev, torch.float32)
    # the reference's integer box: (bboxes[i, :] / scale_factor).astype(np.int32)   (fcn_mask_head_3d.py:163); a
    # tensor divisor keeps torch from multiplying by the reciprocal, so the float32 quotient is numpy's
    boxes = (b / torch.full_like(b, float(scale_factor))).to(torch.int32).reshape(-1, 6).contiguous()
    labels = det_labels.detach().to(dev, torch.int64).reshape(-1) + 1
    size = (boxes[:, 2] - boxes[:, 0] + 1).clamp_min(1).long() * (boxes[:, 3] - boxes[:, 1] + 1).clamp_min(1).long() \
        * (boxes[:, 5] - boxes[:, 4] + 1).clamp_min(1).long()
    offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    torch.cumsum(size, 0, out=offsets[1:])
    out = torch.empty(int(offsets[-1]), dtype=torch.uint8, device=dev)
    if n:
        channel = None if class_agnostic else labels
        with device_guard(dev):
            _lib.check(_lib.lib.roi3d_mask_paste_select(
                mask_pred.data_ptr(), n, num_channels, Dm, Hm, Wm, None if channel is None else channel.data_ptr(),
                boxes.data_ptr(), offsets.data_ptr(), float(mask_thr_binary), out.data_ptr(), stream_ptr()))
    return boxes, offsets, out, labels


def paste_masks_compact(mask_pred, det_bboxes, det_labels, mask_thr_binary, scale_factor=1.0, class_agnostic=False):
    """Arguments as paste_masks_device.  Returns (boxes int32 [n, 6] numpy, masks: list of uint8 numpy arrays of shape
    (d, h, w), labels numpy 1-based)."""
    boxes_d, offsets_d, out_d, labels_d = paste_masks_device(mask_pred, det_bboxes, det_labels, mask_thr_binary,
                                                             scale_factor, class_agnostic)
    boxes, offsets, flat, labels = (t.cpu().numpy() for t in (boxes_d, offsets_d, out_d, labels_d))
    w = np.maximum(boxes[:, 2] - boxes[:, 0] + 1, 1)
    h = np.maximum(boxes[:, 3] - boxes[:, 1] + 1, 1)
    d = np.maximum(boxes[:, 5] - boxes[:, 4] + 1, 1)
    masks = [flat[offsets[i]:offsets[i + 1]].reshape(d[i], h[i], w[i]) for i in range(boxes.shape[0])]
    return boxes, masks, labels


def get_seg_masks(mask_pred, det_bboxes, det_labels, rcnn_test_cfg, ori_shape, scale_factor, rescale, num_classes,
                  class_agnostic=False):
    """Drop-in for FCNMaskHead3D.get_seg_masks (same arguments plus the head's num_classes / class_agnostic):
    returns cls_segms, a list per foreground class of full-volume uint8 masks (img_d, img_h, img_w)."""
    if not rescale:
        raise NotImplementedError("rescale=False stops in a debugger in the reference (fcn_mask_head_3d.py:153-157)")
    thr = rcnn_test_cfg['mask_thr_binary'] if isinstance(rcnn_test_cfg, dict) else rcnn_test_cfg.mask_thr_binary
    img_h, img_w, img_d = ori_shape[:3]
    boxes, masks, labels = paste_masks_compact(mask_pred, det_bboxes, det_labels, thr, scale_factor, class_agnostic)
    cls_segms = [[] for _ in range(num_classes - 1)]
    for i, m in enumerate(masks):
        b = boxes[i]
        dd, hh, ww = m.shape
        im_mask = np.zeros((img_d, img_h, img_w), dtype=np.uint8)
        im_mask[b[4]:b[4] + dd, b[1]:b[1] + hh, b[0]:b[0] + ww] = m
        cls_segms[labels[i] - 1].append(im_mask)
    return cls_segms

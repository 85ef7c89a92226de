"""`nms(dets, iou_thr, device_id=None)` and `soft_nms(dets, iou_thr, method, sigma, min_score)`: the reference's
dispatch wrappers (mmdet/ops/nms/nms_wrapper.py:8-52, :55-81) over the B200 3D NMS and 3D soft-NMS.

Same surface: Tensor or ndarray in, `(dets[inds, :], inds)` out in the input's type; N == 0 returns an empty
long index; `inds` are ORIGINAL row indices in ascending order (nms_kernel.cu:253-256).
Differences, all deliberate:
  * only the 3D form ([N,7] = x1,y1,x2,y2,z1,z2,score) exists here; 5-column (2-D) input raises
    (the reference's 3D config never produces it; on CUDA the reference leaves `inds` unbound for any other
    width, nms_wrapper.py:42-46);
  * there is no CPU path: a CPU tensor, or an ndarray without device_id, raises NotImplementedError instead of
    silently running the reference's 2-D `nms_cpu` on columns 0-4 (nms_wrapper.py:47-48, SURVEY F3);
  * the sweep runs on the device: one 4-byte D2H read (the kept count) instead of the reference's blocking
    copy of the whole bit matrix plus a host loop (nms_kernel.cu:225-249).

soft_nms is the reference's soft_nms_cpu loop (mmdet v0.6.0, soft_nms_cpu.pyx) in 3-D on [N,7] rows, run on the
device by roi3d_soft_nms3d_batched and equal to that loop bit for bit (include/roi3d_b200.h states the limits):
rows come back in selection order with the score each had when it was selected, `inds` are original row indices.
The reference's own soft_nms is 2-D, runs on the CPU and stops in a debugger on entry (nms_wrapper.py:56).  As for
nms, a CPU tensor and input other than [N,7] raise NotImplementedError; an ndarray runs on the current CUDA device.
"""
import ctypes

import numpy as np
import torch

from ... import _lib
from ..._util import check_cuda_f32, device_guard, nvtx_range, stream_ptr, workspace


_WS_BYTES = {}   # (nseg, n_max) -> workspace size (a ctypes round trip per call otherwise)


def nms3d_batched(dets, seg_counts, iou_thr, want_score_order=True, presorted=None, max_keep=0):
    """Batched device NMS.  dets [nseg, n_max, 7] fp32 CUDA; seg_counts int32 [nseg] CUDA or None.

    presorted: optional uint8 [nseg] CUDA tensor, 1 where the segment's rows already are in descending-score order
    (ties by ascending row), e.g. rows straight out of the segmented top-k: the ranking pass is skipped for them.
    max_keep > 0 (with presorted): the sweep of a presorted segment stops with the 64-box tile in which the kept count
    reaches max_keep -- the proposal path only reads `proposals[:nms_post]` (rpn_head_3d.py:135); the lists then hold
    that prefix of the full result (num_keep in [max_keep, max_keep + 63]).
    Returns (keep [nseg, n_max] int64, keep_by_score or None, num_keep [nseg] int32); nothing syncs.
    """
    check_cuda_f32(dets, "dets", ndim=3, last=7)
    dets = dets.contiguous()
    nseg, n_max, _ = dets.shape
    dev = dets.device
    keep = torch.empty((nseg, n_max), dtype=torch.int64, device=dev)
    keep_s = torch.empty((nseg, n_max), dtype=torch.int64, device=dev) if want_score_order else None
    if nseg == 0 or n_max == 0:
        return keep, keep_s, torch.zeros((nseg,), dtype=torch.int32, device=dev)
    num = torch.empty((nseg,), dtype=torch.int32, device=dev)  # written for every segment by the sweep kernel
    if seg_counts is not None:
        assert seg_counts.dtype == torch.int32 and seg_counts.is_cuda and seg_counts.numel() == nseg
        seg_counts = seg_counts.contiguous()
    nbytes = _WS_BYTES.get((nseg, n_max))
    if nbytes is None:
        if len(_WS_BYTES) > 256:
            _WS_BYTES.clear()
        nbytes = _WS_BYTES[(nseg, n_max)] = _lib.lib.roi3d_nms3d_workspace_bytes(nseg, n_max)
    _buf, ws = workspace(dev, nbytes)
    with device_guard(dev), nvtx_range("roi3d.nms3d_batched"):
        _lib.check(_lib.lib.roi3d_nms3d_batched_limited(
            dets.data_ptr(), None if seg_counts is None else seg_counts.data_ptr(),
            None if presorted is None else presorted.data_ptr(), nseg, n_max, float(iou_thr), int(max_keep),
            keep.data_ptr(), None if keep_s is None else keep_s.data_ptr(), num.data_ptr(), ws, nbytes,
            stream_ptr()))
    return keep, keep_s, num


def nms(dets, iou_thr, device_id=None):
    """Dispatch wrapper with the reference's signature (nms_wrapper.py:8)."""
    if isinstance(dets, torch.Tensor):
        is_numpy = False
        dets_th = dets
    elif isinstance(dets, np.ndarray):
        is_numpy = True
        if device_id is None:
            raise NotImplementedError(
                "nms: ndarray input without device_id would select the reference's CPU path, which is 2-D NMS "
                "on columns 0-4 (nms_cpu.cpp:12-16); the B200 path has no CPU implementation. Pass device_id.")
        dets_th = None
    else:
        raise TypeError('dets must be either a Tensor or numpy array, but got {}'.format(type(dets)))

    if is_numpy:
        if dets.ndim != 2 or dets.shape[1] != 7:
            raise NotImplementedError("nms: only [N,7] 3D boxes are supported, got shape %s" % (dets.shape,))
        n = dets.shape[0]
        if n == 0:
            inds = np.zeros(0, dtype=np.int64)
            return dets[inds, :], inds
        d32 = np.ascontiguousarray(dets, dtype=np.float32)
        keep = np.empty(n, dtype=np.int64)
        cnt = ctypes.c_int32(0)
        with torch.cuda.device(int(device_id)):
            _lib.check(_lib.lib.roi3d_nms3d_host(d32.ctypes.data, n, float(iou_thr), keep.ctypes.data,
                                                 ctypes.addressof(cnt)))
        inds = keep[:cnt.value].copy()
        return dets[inds, :], inds

    if dets_th.shape[0] == 0:
        inds = dets_th.new_zeros(0, dtype=torch.long)
        return dets[inds, :], inds
    if not dets_th.is_cuda:
        raise NotImplementedError(
            "nms: CPU tensors are not supported by the B200 path (the reference would run 2-D nms_cpu here, "
            "nms_wrapper.py:47-48); move dets to the GPU.")
    if dets_th.dim() != 2 or dets_th.shape[1] != 7:
        raise NotImplementedError("nms: only [N,7] 3D boxes are supported, got shape %s" % (tuple(dets_th.shape),))
    keep, _, num = nms3d_batched(dets_th.detach().unsqueeze(0), None, iou_thr, want_score_order=False)
    m = int(num.item())  # the one host read: the result length is data dependent
    inds = keep[0, :m]
    return dets[inds, :], inds


SOFT_NMS_METHODS = {'linear': 1, 'gaussian': 2}
SOFT_NMS_MAX_ROWS = 4096   # rows per segment the kernel takes (one CTA holds a segment's boxes in shared memory)


def soft_nms3d_batched(dets, seg_counts, iou_thr, method='linear', sigma=0.5, min_score=1e-3):
    """Batched device soft-NMS.  dets [nseg, n_max, 7] fp32 CUDA, n_max <= 4096; seg_counts int32 [nseg] CUDA or None.
    Returns (out_dets [nseg, n_max, 7] fp32, inds [nseg, n_max] int64, num_keep [nseg] int32): per segment the first
    num_keep rows in selection order, with the scores they had when selected, and their row indices; nothing syncs."""
    if method not in SOFT_NMS_METHODS:
        raise ValueError('Invalid method for SoftNMS: {}'.format(method))
    check_cuda_f32(dets, "dets", ndim=3, last=7)
    dets = dets.contiguous()
    nseg, n_max, _ = dets.shape
    dev = dets.device
    out = torch.empty((nseg, n_max, 7), dtype=torch.float32, device=dev)
    inds = torch.empty((nseg, n_max), dtype=torch.int64, device=dev)
    num = torch.empty((nseg,), dtype=torch.int32, device=dev)
    if seg_counts is not None:
        assert seg_counts.dtype == torch.int32 and seg_counts.is_cuda and seg_counts.numel() == nseg
        seg_counts = seg_counts.contiguous()
    with device_guard(dev), nvtx_range("roi3d.soft_nms3d_batched"):
        _lib.check(_lib.lib.roi3d_soft_nms3d_batched(
            dets.data_ptr(), None if seg_counts is None else seg_counts.data_ptr(), nseg, n_max,
            SOFT_NMS_METHODS[method], float(iou_thr), float(sigma), float(min_score), out.data_ptr(), inds.data_ptr(),
            num.data_ptr(), stream_ptr()))
    return out, inds, num


def soft_nms(dets, iou_thr, method='linear', sigma=0.5, min_score=1e-3):
    """Dispatch wrapper with the reference's signature (nms_wrapper.py:55): (new_dets, inds), a new tensor and int64
    indices on the input's device for a CUDA tensor (one host read: the count), float32 / int64 ndarrays for an
    ndarray (run on the current CUDA device)."""
    if isinstance(dets, torch.Tensor):
        is_numpy = False
    elif isinstance(dets, np.ndarray):
        is_numpy = True
    else:
        raise TypeError('dets must be either a Tensor or numpy array, but got {}'.format(type(dets)))
    if method not in SOFT_NMS_METHODS:
        raise ValueError('Invalid method for SoftNMS: {}'.format(method))

    if is_numpy:
        if dets.ndim != 2 or dets.shape[1] != 7:
            raise NotImplementedError("soft_nms: only [N,7] 3D boxes are supported, got shape %s" % (dets.shape,))
        if dets.shape[0] == 0:
            return np.zeros((0, 7), dtype=np.float32), np.zeros(0, dtype=np.int64)
        d = torch.from_numpy(np.ascontiguousarray(dets, dtype=np.float32)).to(torch.cuda.current_device())
        out, inds, num = soft_nms3d_batched(d[None], None, iou_thr, method, sigma, min_score)
        m = int(num.item())
        return out[0, :m].cpu().numpy(), inds[0, :m].cpu().numpy()

    if dets.shape[0] == 0:
        return dets.new_zeros((0,) + tuple(dets.shape[1:])), dets.new_zeros(0, dtype=torch.long)
    if not dets.is_cuda:
        raise NotImplementedError(
            "soft_nms: CPU tensors are not supported by the B200 path (the reference runs 2-D soft_nms_cpu on "
            "columns 0-4); move dets to the GPU.")
    if dets.dim() != 2 or dets.shape[1] != 7:
        raise NotImplementedError("soft_nms: only [N,7] 3D boxes are supported, got shape %s" % (tuple(dets.shape),))
    out, inds, num = soft_nms3d_batched(dets.detach().unsqueeze(0), None, iou_thr, method, sigma, min_score)
    m = int(num.item())  # the one host read: the result length is data dependent
    return out[0, :m], inds[0, :m]

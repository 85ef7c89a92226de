"""CPU oracle of the 3D soft-NMS -- TEST INFRASTRUCTURE ONLY (tests/ and tools/bench_soft_nms.py).

`soft_nms3d` is soft_nms_cpu (mmdet/ops/nms/src/soft_nms_cpu.pyx, mmdet v0.6.0) with a depth axis, written in the
reference's sequential form in soft_nms_oracle.c; `multiclass_nms_3d` is the reference's multiclass_nms_3d
(mmdet/core/post_processing/bbox_nms.py:57-106) with nms_cfg type 'soft_nms', the same per-class loop as
oracle.multiclass_nms_3d.  The C file is compiled with gcc on first use into a temporary directory, so the tree is
never written to."""
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

_f32p = ctypes.POINTER(ctypes.c_float)
_i64p = ctypes.POINTER(ctypes.c_int64)

METHODS = {'linear': 1, 'gaussian': 2}


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="soft_nms_oracle_")
        try:
            so = os.path.join(tmp, "libsoft_nms_oracle.so")
            cc = os.environ.get("CC", "gcc")
            subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden",
                            "-Wall", "-Wextra", os.path.join(_HERE, "soft_nms_oracle.c"), "-o", so, "-lm"], check=True)
            lb = ctypes.CDLL(so)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)   # the loaded library stays mapped
        lb.oracle_soft_nms3d.restype = ctypes.c_int64
        lb.oracle_soft_nms3d.argtypes = [_f32p, ctypes.c_int64, ctypes.c_float, ctypes.c_int, ctypes.c_float,
                                         ctypes.c_float, _f32p, _i64p]
        _lib = lb
    return _lib


def soft_nms3d(dets, iou_thr, method='linear', sigma=0.5, min_score=1e-3):
    """Through the wrapper's method names (nms_wrapper.py:55-81): (new_dets float32 [m,7] in selection order with the
    scores they had when selected, inds int64 [m] original row indices)."""
    if method not in METHODS:
        raise ValueError('Invalid method for SoftNMS: {}'.format(method))
    dets = np.ascontiguousarray(dets, dtype=np.float32).reshape(-1, 7)
    n = dets.shape[0]
    out = np.empty((max(n, 1), 7), dtype=np.float32)
    inds = np.empty(max(n, 1), dtype=np.int64)
    m = lib().oracle_soft_nms3d(dets.ctypes.data_as(_f32p), n, float(iou_thr), METHODS[method], float(sigma),
                                float(min_score), out.ctypes.data_as(_f32p), inds.ctypes.data_as(_i64p))
    return out[:m].copy(), inds[:m].copy()


def multiclass_nms_3d(multi_bboxes, multi_scores, score_thr, iou_thr, max_num=-1, **soft_nms_cfg):
    """multiclass_nms_3d with nms_cfg = dict(type='soft_nms', iou_thr=iou_thr, **soft_nms_cfg): each class's rows come
    out of soft_nms3d in selection order with their decayed scores; the max_num cut is the stable descending sort."""
    multi_bboxes = np.ascontiguousarray(multi_bboxes, dtype=np.float32)
    multi_scores = np.ascontiguousarray(multi_scores, dtype=np.float32)
    num_classes = multi_scores.shape[1]
    bboxes, labels = [], []
    for i in range(1, num_classes):
        sel = multi_scores[:, i] > np.float32(score_thr)
        if not sel.any():
            continue
        bb = multi_bboxes[sel, :] if multi_bboxes.shape[1] == 6 else multi_bboxes[sel, i * 6:(i + 1) * 6]
        dets = np.concatenate([bb, multi_scores[sel, i][:, None]], axis=1)
        dets, _ = soft_nms3d(dets, iou_thr, **soft_nms_cfg)
        bboxes.append(dets)
        labels.append(np.full((dets.shape[0],), i - 1, dtype=np.int64))
    if not bboxes:
        return np.zeros((0, 7), np.float32), np.zeros((0,), np.int64)
    bboxes, labels = np.concatenate(bboxes), np.concatenate(labels)
    if bboxes.shape[0] > max_num:
        inds = oracle.argsort_desc_stable(bboxes[:, -1])[:max_num]
        bboxes, labels = bboxes[inds], labels[inds]
    return bboxes, labels

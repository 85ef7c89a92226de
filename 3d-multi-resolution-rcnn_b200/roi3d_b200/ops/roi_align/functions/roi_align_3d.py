"""RoIAlignFunction3D: autograd face of the B200 RoIAlign3D kernels.

Mirrors mmdet/ops/roi_align/functions/roi_align_3d.py:9-38,69-89 of the reference (same positional
arguments, same saved state, same gradient arity), minus its breakpoint() on tuple out_size (:15) and the
redundant zero-fill of the output (:32).  CPU input raises NotImplementedError exactly as :36-37 does.
"""
import warnings

import torch
from torch.autograd import Function

from .... import _lib
from ...._util import (channels_last_to_contiguous, check_cuda_f32, forward_inputs, is_channels_last_3d, nvtx_range,
                      stream_ptr)


def _out_dims(out_size, out_size_depth):
    if isinstance(out_size, int):
        return int(out_size_depth), out_size, out_size
    if isinstance(out_size, tuple):
        if len(out_size) != 2 or not all(isinstance(v, int) for v in out_size):
            raise TypeError('"out_size" must be an integer or a tuple of two integers')
        return int(out_size_depth), out_size[0], out_size[1]
    raise TypeError('"out_size" must be an integer or tuple of integers')


class RoIAlignFunction3D(Function):

    @staticmethod
    def forward(ctx, features, rois, out_size, out_size_depth, spatial_scale, spatial_scale_depth, sample_num=0):
        out_d, out_h, out_w = _out_dims(out_size, out_size_depth)
        if isinstance(features, torch.Tensor) and not features.is_cuda:
            raise NotImplementedError  # reference: roi_align_3d.py:36-37
        check_cuda_f32(features, "features", ndim=5)
        check_cuda_f32(rois, "rois", ndim=2, last=7)
        ctx.spatial_scale = float(spatial_scale)
        ctx.spatial_scale_depth = float(spatial_scale_depth)
        ctx.sample_num = int(sample_num)
        ctx.feature_size = features.size()
        ctx.input_channels_last = is_channels_last_3d(features)
        rois = rois.contiguous()
        ctx.save_for_backward(rois)

        (feats_in,), layout = forward_inputs([features], out_h, out_w)
        B, C, D, H, W = features.shape
        K = rois.size(0)
        output = features.new_empty((K, C, out_d, out_h, out_w))
        if K > 0:
            with torch.cuda.device(features.device), nvtx_range("roi3d.roi_align3d.forward"):
                _lib.check(_lib.lib.roi3d_roi_align3d_forward(
                    feats_in.data_ptr(), layout, B, C, D, H, W, rois.data_ptr(), K, out_d, out_h, out_w,
                    ctx.spatial_scale, ctx.spatial_scale_depth, ctx.sample_num, output.data_ptr(), stream_ptr()))
        return output

    @staticmethod
    def backward(ctx, grad_output):
        rois = ctx.saved_tensors[0]
        assert ctx.feature_size is not None and grad_output.is_cuda
        B, C, D, H, W = ctx.feature_size
        grad_input = None
        if ctx.needs_input_grad[0]:
            grad_output = grad_output.contiguous()
            K, _, out_d, out_h, out_w = grad_output.shape
            grad_cl = torch.empty((B, C, D, H, W), dtype=grad_output.dtype, device=grad_output.device,
                                  memory_format=torch.channels_last_3d)
            with torch.cuda.device(grad_output.device), nvtx_range("roi3d.roi_align3d.backward"):
                if deterministic_backward("RoIAlignFunction3D.backward"):
                    # every voxel is written once (no zero-fill, no atomics): the same bits on every run
                    lv = _lib.level_array([grad_cl], [ctx.spatial_scale], [ctx.spatial_scale_depth], grads=[grad_cl])
                    _lib.check(_lib.lib.roi3d_extract_backward_deterministic(
                        lv, 1, B, C, rois.data_ptr(), K, out_d, out_h, out_w, ctx.sample_num, 56.0,
                        grad_output.data_ptr(), 0, stream_ptr()))
                else:
                    _lib.check(_lib.lib.roi3d_roi_align3d_backward(
                        grad_output.data_ptr(), rois.data_ptr(), K, out_d, out_h, out_w, ctx.spatial_scale,
                        ctx.spatial_scale_depth, ctx.sample_num, grad_cl.data_ptr(), _lib.NDHWC, B, C, D, H, W,
                        1, int(_BUG_COMPAT[0]), stream_ptr()))
            grad_input = grad_cl if ctx.input_channels_last else channels_last_to_contiguous(grad_cl)
        return grad_input, None, None, None, None, None, None


# The reference's backward reads the wrong top_diff element for non-cubic outputs
# (roi_align_kernel.cu:554-555, SURVEY F2).  Default: the correct gradient.  set_bug_compat(True) switches
# to the reference's indexing for A/B comparisons only.
_BUG_COMPAT = [False]


def set_bug_compat(flag):
    _BUG_COMPAT[0] = bool(flag)


def deterministic_backward(op):
    """True when the backward of `op` has to take the deterministic kernel: torch.use_deterministic_algorithms(True)
    is in force.  The default backward adds into the gradient with float atomics, so its last bits change from run to
    run wherever RoIs overlap.  bug_compat exists only in the atomic kernel: with the flag on it raises, as torch does
    for an op without a deterministic implementation, or under warn_only=True warns and keeps the atomic path."""
    if not torch.are_deterministic_algorithms_enabled():
        return False
    if _BUG_COMPAT[0]:
        msg = ("%s with set_bug_compat(True) does not have a deterministic implementation, but you set "
               "'torch.use_deterministic_algorithms(True)'. Call set_bug_compat(False), or use the 'warn_only=True' "
               "option to run the atomic backward with a warning." % op)
        if torch.is_deterministic_algorithms_warn_only_enabled():
            warnings.warn(msg, UserWarning)
            return False
        raise RuntimeError(msg)
    return True


roi_align_3d = RoIAlignFunction3D.apply
roi_align = roi_align_3d  # the reference's functions/roi_align_3d.py exports the 3D op under this name (:92)

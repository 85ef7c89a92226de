"""SingleRoIExtractor for 3D RoIs on the B200 kernels.

Same constructor keys, attributes and call signature as the reference's
mmdet/models/roi_extractors/single_level.py:24-104, so `bbox_roi_extractor=dict(type='SingleRoIExtractor',
roi_layer=dict(type='RoIAlign3D', out_size=7, out_size_depth=3, sample_num=2), out_channels=64,
featmap_strides=[4, 8, 16, 32], featmap_strides_depth=[2, 4, 8, 16])` from
configs/3d-multi-resolution-rcnn.py:40-45 builds it unchanged.

What is different underneath: the reference loops over levels in Python with two host syncs per level
(`inds.any()`, boolean-mask indexing), launches one RoIAlign per level into a temporary and index-adds it into
a zero-filled output (single_level.py:93-103).  Here level mapping, the per-level RoIAlign3D and the scatter
are ONE kernel launch that writes each RoI's block of the output exactly once, with no host sync; the backward
is one launch as well.
"""
import torch
import torch.nn as nn
from torch.autograd import Function

from ... import _lib, ops
from ..._util import (channels_last_to_contiguous, check_cuda_f32, forward_inputs, is_channels_last_3d, nvtx_range,
                      stream_ptr)
from ...ops.roi_align.functions.roi_align_3d import _BUG_COMPAT, _out_dims, deterministic_backward


class _MultiLevelRoIAlign3D(Function):
    """Fused map_roi_levels + per-level RoIAlign3D + scatter (single_level.py:84-104) and its gradient."""

    @staticmethod
    def forward(ctx, rois, out_dims, scales, scales_d, sample_num, finest_scale, *feats):
        check_cuda_f32(rois, "rois", ndim=2, last=7)
        for f in feats:
            check_cuda_f32(f, "feats", ndim=5)
        rois = rois.contiguous()
        out_d, out_h, out_w = out_dims
        B, C = feats[0].shape[:2]
        feats_in, layout = forward_inputs(feats, out_h, out_w)
        K = rois.size(0)
        out = feats[0].new_empty((K, C, out_d, out_h, out_w))
        ctx.cfg = (out_dims, tuple(scales), tuple(scales_d), int(sample_num), float(finest_scale))
        ctx.shapes = [tuple(f.shape) for f in feats]
        ctx.input_channels_last = [is_channels_last_3d(f) for f in feats]
        ctx.save_for_backward(rois)
        if K > 0:
            arr = _lib.level_array(feats_in, scales, scales_d, layout=layout)
            with torch.cuda.device(rois.device), nvtx_range("roi3d.extract.forward"):
                _lib.check(_lib.lib.roi3d_extract_forward(arr, len(feats), B, C, rois.data_ptr(), K, out_d, out_h,
                                                          out_w, int(sample_num), float(finest_scale),
                                                          out.data_ptr(), None, stream_ptr()))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        rois = ctx.saved_tensors[0]
        (out_d, out_h, out_w), scales, scales_d, sample_num, finest_scale = ctx.cfg
        nlev = len(ctx.shapes)
        need = ctx.needs_input_grad[6:]
        if not any(need):
            return (None,) * (6 + nlev)
        grad_out = grad_out.contiguous()
        K = rois.size(0)
        B, C = ctx.shapes[0][:2]
        grads = [torch.empty(s, dtype=grad_out.dtype, device=grad_out.device, memory_format=torch.channels_last_3d)
                 for s in ctx.shapes]
        arr = _lib.level_array(grads, scales, scales_d, grads=grads)
        with torch.cuda.device(grad_out.device):
            if deterministic_backward("SingleRoIExtractor backward"):
                # every voxel of every level is written once (no zero-fill, no atomics): the same bits on every run
                _lib.check(_lib.lib.roi3d_extract_backward_deterministic(
                    arr, nlev, B, C, rois.data_ptr(), K, out_d, out_h, out_w, sample_num, finest_scale,
                    grad_out.data_ptr(), 0, stream_ptr()))
            else:
                _lib.check(_lib.lib.roi3d_extract_backward(arr, nlev, B, C, rois.data_ptr(), K, out_d, out_h, out_w,
                                                           sample_num, finest_scale, grad_out.data_ptr(), 1,
                                                           int(_BUG_COMPAT[0]), stream_ptr()))
        outs = []
        for g, cl, nd in zip(grads, ctx.input_channels_last, need):
            outs.append(None if not nd else (g if cl else channels_last_to_contiguous(g)))
        return (None,) * 6 + tuple(outs)


class SingleRoIExtractor(nn.Module):
    """Extract RoI features from a single level feature map (3D RoIs).

    Args (reference single_level.py:24-35): roi_layer (dict), out_channels (int), featmap_strides (list),
    featmap_strides_depth (list or None), finest_scale (int).
    """

    def __init__(self, roi_layer, out_channels, featmap_strides, featmap_strides_depth=None, finest_scale=56):
        super(SingleRoIExtractor, self).__init__()
        self.roi_layers = self.build_roi_layers(roi_layer, featmap_strides, featmap_strides_depth)
        self.out_channels = out_channels
        self.featmap_strides = featmap_strides
        self.featmap_strides_depth = featmap_strides_depth
        self.finest_scale = finest_scale

    @property
    def num_inputs(self):
        """int: Input feature map levels."""
        return len(self.featmap_strides)

    def init_weights(self):
        pass

    def build_roi_layers(self, layer_cfg, featmap_strides, featmap_strides_depth=None):
        cfg = dict(layer_cfg)
        layer_type = cfg.pop('type')
        if not hasattr(ops, layer_type):  # the plugin seam: getattr(mmdet.ops, type) (single_level.py:48-49)
            raise KeyError("roi_layer type %r is not provided by roi3d_b200.ops" % (layer_type,))
        layer_cls = getattr(ops, layer_type)
        if featmap_strides_depth is None:
            raise NotImplementedError("2-D RoI layers (no featmap_strides_depth) are outside the 3D RoI hot path")
        return nn.ModuleList([
            layer_cls(spatial_scale=1 / s, spatial_scale_depth=1 / d, **cfg)
            for s, d in zip(featmap_strides, featmap_strides_depth)
        ])

    def map_roi_levels(self, rois, num_levels):
        """Level index (0-based, int64) of each RoI: floor(log2(sqrt(w*h*d)/finest_scale + 1e-6)) clamped to
        [0, num_levels-1] (single_level.py:58-82), one kernel instead of ~8 elementwise launches."""
        check_cuda_f32(rois, "rois", ndim=2, last=7)
        rois = rois.contiguous()
        lvls = torch.empty((rois.size(0),), dtype=torch.int64, device=rois.device)
        if rois.size(0):
            with torch.cuda.device(rois.device):
                _lib.check(_lib.lib.roi3d_map_roi_levels(rois.data_ptr(), rois.size(0), int(num_levels),
                                                         float(self.finest_scale), lvls.data_ptr(), stream_ptr()))
        return lvls

    def forward(self, feats, rois):
        if len(feats) == 1:
            return self.roi_layers[0](feats[0], rois)
        layer0 = self.roi_layers[0]
        out_dims = _out_dims(layer0.out_size, layer0.out_size_depth)
        num_levels = len(feats)
        scales = [self.roi_layers[i].spatial_scale for i in range(num_levels)]
        scales_d = [self.roi_layers[i].spatial_scale_depth for i in range(num_levels)]
        return _MultiLevelRoIAlign3D.apply(rois, out_dims, scales, scales_d, layer0.sample_num,
                                           float(self.finest_scale), *feats[:num_levels])

"""roi3d_b200: B200-native (sm_100a) 3D R-CNN RoI hot path -- RoIAlign3D fwd/bwd, 3D NMS, FPN level mapping and
the RPN proposal path -- behind the operator surface of arthur801031/3d-multi-resolution-rcnn's mmdet fork.

Module paths mirror the reference's (`mmdet.X` -> `roi3d_b200.X`):
    roi3d_b200.ops                       nms, soft_nms, RoIAlign3D, roi_align_3d        (mmdet/ops/__init__.py)
    roi3d_b200.ops.nms.nms_wrapper       nms(dets, iou_thr, device_id=None)             (mmdet/ops/nms/nms_wrapper.py)
    roi3d_b200.models.roi_extractors     SingleRoIExtractor                             (roi_extractors/single_level.py)
    roi3d_b200.models.anchor_heads       RPNProposal3D.get_bboxes[_single]              (anchor_heads/rpn_head_3d.py)
    roi3d_b200.core.anchor               AnchorGenerator3D                              (core/anchor/anchor_generator_3d.py)
    roi3d_b200.core.bbox                 delta2bbox3D, bbox2roi3D[_padded]              (core/bbox/transforms.py)
    roi3d_b200.core.post_processing      multiclass_nms_3d[_batched]                    (core/post_processing/bbox_nms.py)
    roi3d_b200.core.evaluation           apply_nms, nms_3d_python                       (core/evaluation/coco_utils.py)
    roi3d_b200.models.mask_heads         get_seg_masks (mask paste)                     (models/mask_heads/fcn_mask_head_3d.py)
    roi3d_b200.parallel                  shard_indices, gather_detections               (replaces eval_hooks.py:134-149)

Everything computes in hand-written CUDA (libroi3d_b200.so, C ABI in include/roi3d_b200.h).  Importing this
package fails if that library is missing: there is no CPU or PyTorch fallback.
"""
from . import _lib  # noqa: F401  (raises ImportError when libroi3d_b200.so is absent)
from . import ops
from ._util import reuse_layout_conversions
from .core.anchor import AnchorGenerator3D
from .core.bbox import bbox2roi3D, bbox2roi3D_padded, delta2bbox3D
from .core.post_processing import multiclass_nms_3d, multiclass_nms_3d_batched
from .core.evaluation import apply_nms, nms_3d_eval_batched
from .models.anchor_heads import RPNProposal3D
from .models.builder import build_roi_extractor, build_rpn_proposal
from .models.config import build_from_config, load_config
from .models.roi_extractors import SingleRoIExtractor
from .ops import RoIAlign3D, nms, roi_align_3d, soft_nms

__all__ = ['ops', 'nms', 'soft_nms', 'RoIAlign3D', 'roi_align_3d', 'SingleRoIExtractor', 'RPNProposal3D',
           'AnchorGenerator3D', 'delta2bbox3D', 'bbox2roi3D', 'bbox2roi3D_padded', 'multiclass_nms_3d',
           'multiclass_nms_3d_batched', 'build_roi_extractor',
           'build_rpn_proposal', 'build_from_config', 'load_config', 'reuse_layout_conversions', 'apply_nms', 'nms_3d_eval_batched']

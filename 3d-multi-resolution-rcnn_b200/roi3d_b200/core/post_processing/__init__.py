from .bbox_nms import multiclass_nms_3d, multiclass_nms_3d_batched

__all__ = ['multiclass_nms_3d', 'multiclass_nms_3d_batched']

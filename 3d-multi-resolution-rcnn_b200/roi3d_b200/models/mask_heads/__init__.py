from .fcn_mask_head_3d import get_seg_masks, paste_masks_compact, paste_masks_device

__all__ = ['get_seg_masks', 'paste_masks_compact', 'paste_masks_device']

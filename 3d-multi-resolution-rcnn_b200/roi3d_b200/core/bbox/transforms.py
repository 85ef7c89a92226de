"""3D box helpers of the proposal path (reference: mmdet/core/bbox/transforms.py)."""
import ctypes

import torch

from ... import _lib
from ..._util import check_cuda_f32, stream_ptr


def bbox2roi3D(bbox_list):
    """[n_i, >=6] boxes per image -> [K,7] rois (batch_ind, x1, y1, x2, y2, z1, z2), images in list order.
    Reference: bbox2roi3D, transforms.py:220-239.  Two concatenations for the whole batch instead of two per image."""
    ref = bbox_list[0]
    coords = torch.cat([b[:, :6] for b in bbox_list], dim=0) if len(bbox_list) > 1 else ref[:, :6]
    batch = torch.cat([ref.new_full((b.size(0), 1), i) for i, b in enumerate(bbox_list)], dim=0)
    return torch.cat([batch, coords], dim=1)


def bbox2roi3D_padded(boxes, counts):
    """Fixed-shape bbox2roi3D: boxes [B, n, >=6] holding counts[b] valid rows per image (counts: [B] integers on the
    same device) -> rois [B*n, 7].  Row b*n + r is (b, x1, y1, x2, y2, z1, z2) when r < counts[b] and exactly (-1, 0, 0, 0, 0, 0, 0)
    otherwise: the RoI extractors give a zero row for a batch index outside [0, B), and the coordinates are zeroed too,
    because padding rows may hold anything (NaN included) and would still reach the level map.  Reads nothing back to
    the host, so it can be captured in a CUDA graph with the rest of a fixed-shape stage."""
    B, n = boxes.shape[0], boxes.shape[1]
    valid = torch.arange(n, device=boxes.device)[None, :] < counts.reshape(B, 1)
    batch = torch.arange(B, device=boxes.device, dtype=boxes.dtype)[:, None].expand(B, n)
    batch = torch.where(valid, batch, -1.0)
    coords = torch.where(valid[:, :, None], boxes[:, :, :6], 0.0)
    return torch.cat([batch[:, :, None], coords], dim=2).reshape(B * n, 7)


def delta2bbox3D(rois, deltas, means=(0, 0, 0, 0, 0, 0), stds=(1, 1, 1, 1, 1, 1), max_shape=None,
                 wh_ratio_clip=16 / 1000, d_ratio_clip=64 / 1000):
    """Decode [n, 6k] class-wise deltas against [n, >=6] boxes, one kernel (roi3d_delta2bbox3d); the caller outside the
    fused proposal path is the bbox head.  Reference: delta2bbox3D, transforms.py:105-160 (about 60 elementwise
    launches); it clamps all of dw, dh, dz, dd with |log(wh_ratio_clip)| (:122-128) -- d_ratio_clip is accepted and
    unused, as there.  max_shape = img_shape (H, W, 3, D).  Returns a tensor shaped like `deltas`."""
    r, d = rois.float().contiguous(), deltas.float().contiguous()
    check_cuda_f32(r, "rois", ndim=2)
    check_cuda_f32(d, "deltas", ndim=2)
    if r.shape[1] < 6 or d.shape[1] % 6 != 0 or d.shape[0] != r.shape[0]:
        raise ValueError("delta2bbox3D: rois [n, >=6] and deltas [n, 6k] expected, got %s and %s"
                         % (tuple(r.shape), tuple(d.shape)))
    n, k = d.shape[0], d.shape[1] // 6
    out = torch.empty_like(d)
    m6 = (ctypes.c_float * 6)(*[float(x) for x in means])
    s6 = (ctypes.c_float * 6)(*[float(x) for x in stds])
    if max_shape is None:
        ih = iw = idp = 0.0
    else:
        ih, iw, idp = float(max_shape[0]), float(max_shape[1]), float(max_shape[3])
    if n:
        with torch.cuda.device(r.device):
            _lib.check(_lib.lib.roi3d_delta2bbox3d(r.data_ptr(), r.shape[1], d.data_ptr(), n, k, ctypes.addressof(m6),
                                                   ctypes.addressof(s6), float(wh_ratio_clip), ih, iw, idp,
                                                   out.data_ptr(), stream_ptr()))
    return out


def bbox2delta3d(proposals, gt, means=(0, 0, 0, 0, 0, 0), stds=(1, 1, 1, 1, 1, 1)):
    """Regression targets (dx, dy, dw, dh, dz, dd) of `gt` w.r.t. `proposals`, one kernel.
    Reference: bbox2delta3d, transforms.py:33-63 (about 30 elementwise launches)."""
    assert proposals.size() == gt.size()
    p, g = proposals.float().contiguous(), gt.float().contiguous()
    check_cuda_f32(p, "proposals", ndim=2)
    check_cuda_f32(g, "gt", ndim=2)
    if p.shape[1] < 6:
        raise NotImplementedError("bbox2delta3d: boxes need 6 columns")
    n = p.shape[0]
    out = p.new_empty((n, 6))
    m6 = (ctypes.c_float * 6)(*[float(x) for x in means])
    s6 = (ctypes.c_float * 6)(*[float(x) for x in stds])
    if n:
        with torch.cuda.device(p.device):
            _lib.check(_lib.lib.roi3d_bbox2delta3d(p.data_ptr(), p.shape[1], g.data_ptr(), g.shape[1], n,
                                                   ctypes.addressof(m6), ctypes.addressof(s6), out.data_ptr(),
                                                   stream_ptr()))
    return out

"""RPN proposal path on the B200 kernels: `get_bboxes` / `get_bboxes_single` of the reference's RPNHead3D
(mmdet/models/anchor_heads/rpn_head_3d.py:72-149, anchor_head_3d.py:232-268).

`RPNProposal3D` holds what the reference head holds for this path (anchor generators per level, strides, target
means/stds, use_sigmoid_cls) and exposes `get_bboxes(cls_scores, bbox_preds, img_metas, cfg)` with the same
arguments and the same return value: a list (one entry per image) of [<=max_num, 7] proposals
(x1,y1,x2,y2,z1,z2,score), and the list of anchors the reference also returns.

Per level the reference runs: permute + sigmoid over every anchor, topk(nms_pre), ~25 elementwise launches of
delta2bbox3D, cat, a host-synchronising NMS, slice; then cat + topk(max_num) (rpn_head_3d.py:82-148) -- for
every image separately, with anchors rebuilt in numpy and copied H2D on every call.  Here, for ALL images and
levels together: one segmented radix-select top-k (sigmoid fused, logical permuted indices), one fused
anchor+decode kernel per level, one batched NMS over every (image, level) segment, a handful of torch index ops,
one segmented top-k for the final cut, and a single host read of the result lengths at the end.

The head's cached inside-flag masks `pos_indices` / `pos_indices_test` (anchor_head_3d.py:212,239-243) are honoured
the way rpn_head_3d.py:97-106 applies them: on a level with more than nms_pre anchors, when the mask has the level's
shape, only the masked-in anchors take part in the top-k (the mask goes into the segmented top-k; nothing is
compacted).

`min_bbox_size > 0` drops, per (image, level), the decoded proposals whose width or height ((x2 - x1) + 1, (y2 - y1) + 1
in fp32) is below it, before that level's NMS, as mmdetection v0.6.0's RPNHead does; the fork's own branch stops in a
debugger (:125-132).  Depth is not compared: z is measured in slices, x and y in pixels, and one pixel threshold on the
depth would drop nearly every fine-level proposal (the level-0 anchors are 8 x 8 pixels by 4 slices).  The survivors
keep their order, so score-sorted levels stay sorted and index-order levels stay in anchor order.
"""
import ctypes

import numpy as np
import torch

from ... import _lib
from ..._util import check_cuda_f32, nvtx_range, stream_ptr, workspace
from ...core.anchor import AnchorGenerator3D
from ...ops.nms.nms_wrapper import nms3d_batched


def _cfg_get(cfg, key, default=None):
    if isinstance(cfg, dict):
        return cfg.get(key, default)
    return getattr(cfg, key, default)


def topk_segmented(scores_list, k, apply_sigmoid=False, permute_adhw=False, small_in_index_order=False, masks=None,
                   report=False):
    """Segmented top-k over a list of CUDA fp32 tensors (one segment each).

    permute_adhw=True: each tensor is an [A, D, H, W] score map and indices refer to
    permute(2,3,1,0).reshape(-1) positions (rpn_head_3d.py:87-89).  Returns (idx [nseg,k] int64, val [nseg,k]);
    rows past a segment's length hold -1 / 0.  Descending, ties -> lower index.  No host sync.
    small_in_index_order=True: a segment with no more than k elements comes back whole, in ascending index order
    (the reference does not sort a level that has at most nms_pre anchors, rpn_head_3d.py:96,108-112).
    masks: optional list (one entry per segment, None = no mask) of uint8 / bool CUDA tensors indexed like the returned
    indices; only elements whose mask byte is non-zero take part (`scores[pos_indices]`, rpn_head_3d.py:97-106), and
    "no more than k elements" then refers to the masked-in count.
    report=True additionally returns (count int32 [nseg], sorted uint8 [nseg]): rows returned per segment and whether
    they are in score order (1) or in ascending index order (0) -- device tensors, no host read.
    """
    segs = []
    for s in scores_list:
        check_cuda_f32(s, "scores")
        segs.append(s if s.is_contiguous() else s.contiguous())
    ptrs = [s.data_ptr() for s in segs]
    lens = [s.numel() for s in segs]
    adhw = [list(s.shape[-4:]) for s in segs] if permute_adhw else None
    mask_ptrs, keep = None, []
    if masks is not None and any(m is not None for m in masks):
        mask_ptrs = []
        for m, sc in zip(masks, segs):
            if m is None:
                mask_ptrs.append(None)
                continue
            m = _check_mask(m, sc.numel())
            keep.append(m)
            mask_ptrs.append(m.data_ptr())
    out = _topk_segmented_desc(segs[0].device, ptrs, lens, adhw, k, apply_sigmoid, small_in_index_order, mask_ptrs, report)
    del segs, keep
    return out


def _check_mask(m, numel):
    if m.dtype == torch.bool:
        m = m.view(torch.uint8)
    if m.dtype != torch.uint8 or not m.is_cuda or m.numel() != numel:
        raise ValueError("a top-k mask must be a uint8 / bool CUDA tensor with one entry per score")
    return m.contiguous()


_DESC_CACHE = {}


def _topk_segmented_desc(dev, ptrs, lens, adhw, k, apply_sigmoid, small_in_index_order, mask_ptrs, report):
    """topk_segmented on raw descriptors: device addresses, lengths and (optionally) [A, D, H, W] shapes of the segments.
    The caller keeps the tensors behind the addresses alive until the call is enqueued."""
    nseg = len(ptrs)
    # the host-side descriptor arrays only depend on the segments' relative addresses and shapes, which repeat from call
    # to call: built once per signature (three numpy constructions per call otherwise)
    # an empty segment reads nothing and its tensor's address may be 0: it takes offset 0 and plays no part in the base
    live = [q for q, n in zip(ptrs, lens) if n > 0]
    base = min(live) if live else None
    rel = [q - base if n > 0 else 0 for q, n in zip(ptrs, lens)]
    dkey = (tuple(rel), tuple(lens), None if adhw is None else tuple(map(tuple, adhw)))
    desc = _DESC_CACHE.get(dkey)
    if desc is None:
        off = np.array([r // 4 for r in rel], dtype=np.int64)
        ln = np.array(lens, dtype=np.int64)
        adhw_a = np.array(adhw, dtype=np.int32) if adhw is not None else None
        if len(_DESC_CACHE) > 64:
            _DESC_CACHE.clear()
        desc = _DESC_CACHE[dkey] = (off, ln, adhw_a, int(ln.sum()))
    off, ln, adhw_a, total_len = desc
    adhw_p = adhw_a.ctypes.data if adhw_a is not None else None
    idx = torch.empty((nseg, k), dtype=torch.int64, device=dev)
    val = torch.empty((nseg, k), dtype=torch.float32, device=dev)
    # base workspace + one u32 key per score (the first digit pass stores the keys, later passes re-read them from L2)
    nbytes = _lib.lib.roi3d_topk_workspace_bytes_keys(nseg, k, total_len)
    _buf, ws = workspace(dev, nbytes)
    if base is None:   # every segment empty: no score is read, but the entry wants a device address
        base = ws
    mask_p = (ctypes.c_void_p * nseg)(*mask_ptrs) if mask_ptrs is not None else None
    cnt = torch.empty((nseg,), dtype=torch.int32, device=dev) if report else None
    srt = torch.empty((nseg,), dtype=torch.uint8, device=dev) if report else None
    with torch.cuda.device(dev):
        _lib.check(_lib.lib.roi3d_topk_segmented_masked(
            base, off.ctypes.data, ln.ctypes.data, adhw_p, mask_p, nseg, int(k), int(bool(apply_sigmoid)),
            int(bool(small_in_index_order)), idx.data_ptr(), val.data_ptr(), None if cnt is None else cnt.data_ptr(),
            None if srt is None else srt.data_ptr(), ws, nbytes, stream_ptr()))
    del _buf
    if report:
        return idx, val, cnt, srt
    return idx, val


def decode_proposals(bbox_pred, base_anchors, stride, depth_stride, idx, scores, means, stds, img_shape):
    """Fused grid-anchor + delta2bbox3D + score append for the selected anchors of one level.
    bbox_pred [6A, D, H, W]; idx int64 [n] logical indices (-1 -> zero row); returns [n, 7]."""
    check_cuda_f32(bbox_pred, "bbox_pred", ndim=4)
    bbox_pred = bbox_pred.contiguous()
    A = base_anchors.shape[0]
    D, H, W = bbox_pred.shape[1:]
    n = idx.numel()
    out = torch.empty((n, 7), dtype=torch.float32, device=bbox_pred.device)
    base = np.ascontiguousarray(base_anchors.detach().cpu().numpy(), dtype=np.float32)
    m = np.asarray(means, dtype=np.float32)
    s = np.asarray(stds, dtype=np.float32)
    if img_shape is None:
        ih = iw = idp = 0.0
    else:
        ih, iw, idp = float(img_shape[0]), float(img_shape[1]), float(img_shape[3])  # (H, W, 3, D)
    with torch.cuda.device(bbox_pred.device):
        _lib.check(_lib.lib.roi3d_decode_proposals(bbox_pred.data_ptr(), A, D, H, W, float(stride),
                                                   float(depth_stride), base.ctypes.data, idx.data_ptr(),
                                                   None if scores is None else scores.data_ptr(), n,
                                                   m.ctypes.data, s.ctypes.data, ih, iw, idp, out.data_ptr(),
                                                   stream_ptr()))
    return out


class RPNProposal3D(object):
    """The proposal half of RPNHead3D/AnchorHead3D (anchor_head_3d.py:27-70 constructor keys)."""

    def __init__(self, anchor_scales=(8,), anchor_depth_scales=(2,), anchor_ratios=(1.0,),
                 anchor_strides=(4, 8, 16, 32, 64), anchor_strides_depth=(2, 4, 8, 16, 32),
                 anchor_base_sizes=None, anchor_base_depths=None, target_means=(.0, .0, .0, .0, .0, .0),
                 target_stds=(1.0, 1.0, 1.0, 1.0, 1.0, 1.0), use_sigmoid_cls=True):
        self.anchor_strides = list(anchor_strides)
        self.anchor_strides_depth = list(anchor_strides_depth)
        self.anchor_base_sizes = list(anchor_strides) if anchor_base_sizes is None else list(anchor_base_sizes)
        self.anchor_base_depths = (list(anchor_strides_depth) if anchor_base_depths is None
                                   else list(anchor_base_depths))
        self.target_means = tuple(target_means)
        self.target_stds = tuple(target_stds)
        self.use_sigmoid_cls = use_sigmoid_cls
        if not use_sigmoid_cls:
            raise NotImplementedError("softmax RPN scores are not used by configs/3d-multi-resolution-rcnn.py")
        self.anchor_generators = [
            AnchorGenerator3D(b, list(anchor_scales), list(anchor_depth_scales), list(anchor_ratios), d)
            for b, d in zip(self.anchor_base_sizes, self.anchor_base_depths)
        ]
        self.num_anchors = len(anchor_ratios) * len(anchor_scales)
        # the reference head's cached inside-flag masks (anchor_head_3d.py:67-68): per-level uint8 / bool CUDA tensors,
        # set by the training loss pass (:212) or by get_bboxes for different_img_size test configs (:239-243)
        self.pos_indices = None
        self.pos_indices_test = None
        self._desc_cache = {}  # (segment lengths, flags, device) -> device descriptor tensors of get_bboxes
        self.cuda_graph = False  # capture + replay the path per (input buffers, shapes, config); see get_bboxes
        self._graphs = {}

    def get_bboxes(self, cls_scores, bbox_preds, img_metas, cfg, rescale=False, img_meta_2=None, img_meta_3=None):
        """AnchorHead3D.get_bboxes (anchor_head_3d.py:232-268): same arguments, and the reference's return value
        `(result_list, anchors_list)` -- every 3D caller unpacks it (`proposal_list, _ = ...`).  anchors_list holds
        None per image: the reference only uses it for debug drawing (:270-547) and the anchors are never
        materialised here."""
        result = self.get_proposals(cls_scores, bbox_preds, img_metas, cfg, rescale, img_meta_2, img_meta_3)
        return result, [None] * len(result)

    def get_proposals(self, cls_scores, bbox_preds, img_metas, cfg, rescale=False, img_meta_2=None, img_meta_3=None):
        """The proposal list alone (first element of get_bboxes' return value).  With `self.cuda_graph = True`
        the ~45 launches of the path are captured once per (input buffers, shapes, config) into a CUDA graph and
        replayed: the path is launch-bound (0.6 ms of GPU time behind ~1 ms of host-side launching for 8 volumes),
        and inference loops hand the same activation buffers to every call."""
        if img_meta_2 is not None:
            img_metas = img_meta_2
        if img_meta_3 is not None:
            img_metas = img_meta_3
        if not self.cuda_graph:
            with nvtx_range("roi3d.rpn.get_bboxes"):
                final, n_valid, kk = self._enqueue(cls_scores, bbox_preds, img_metas, cfg)
        else:
            masks_now = [m for lst in (self.pos_indices, self.pos_indices_test) if lst is not None for m in lst]
            key = (tuple(t.data_ptr() for t in list(cls_scores) + list(bbox_preds) + masks_now),
                   tuple(tuple(t.shape) for t in list(cls_scores) + list(bbox_preds)),
                   tuple(tuple(m['img_shape']) for m in img_metas),
                   tuple(_cfg_get(cfg, n) for n in ('nms_pre', 'nms_post', 'max_num', 'nms_thr', 'min_bbox_size')))
            entry = self._graphs.get(key)
            if entry is None:
                self._enqueue(cls_scores, bbox_preds, img_metas, cfg)  # warm-up: scratch, descriptor cache, attributes
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    outs = self._enqueue(cls_scores, bbox_preds, img_metas, cfg)
                if len(self._graphs) >= 4:
                    self._graphs.clear()
                # the inputs are kept alive with the graph: their addresses are baked into it (the workspaces of the
                # captured calls are per-call torch allocations, so they live in the graph's own memory pool)
                entry = self._graphs[key] = (graph, outs, list(cls_scores) + list(bbox_preds))
            entry[0].replay()
            final, n_valid, kk = entry[1]
            # the graph's output buffer is overwritten by the next replay: ONE copy of the whole block, queued before
            # the host read below (a clone per image after it costs a launch + an idle gap each)
            final = final.clone()
        n_out = [min(int(v), kk) for v in n_valid.tolist()]  # the single host read of the whole path
        return [final[b, :n_out[b]] for b in range(len(n_out))]

    def get_proposals_padded(self, cls_scores, bbox_preds, img_metas, cfg):
        """get_proposals with fixed shapes and no host read: (final [B, kk, 7], counts int32 [B]) as device tensors, where
        final[b, :counts[b]] equals get_proposals(...)[b] and the rows past counts[b] are unspecified.  kk depends on
        the level shapes and the config only, so the call can be captured in a CUDA graph (as part of a larger stage);
        its first call per shape uploads small descriptor tensors from pageable memory, so run it once before a
        capture."""
        final, n_valid, kk = self._enqueue(cls_scores, bbox_preds, img_metas, cfg)
        return final, n_valid.clamp(max=kk)

    def _enqueue(self, cls_scores, bbox_preds, img_metas, cfg):
        """cls_scores[l]: [B, A, D, H, W]; bbox_preds[l]: [B, 6A, D, H, W]; img_metas[b]['img_shape'] = (H, W, 3, D).
        Same positional arguments as AnchorHead3D.get_bboxes (anchor_head_3d.py:232-233): `img_meta_2` / `img_meta_3`,
        when given, replace `img_metas` (the reference's swap for the 1.5x / third scale, :234-237).
        Returns the list of per-image proposals; with return_anchors=True the reference's 2-tuple
        (result_list, anchors_list) is returned, anchors_list holding None (the reference only uses it for debug
        drawing, anchor_head_3d.py:270-547).
        Queues every kernel of the path on the current stream and returns (final [B, kk, 7], n_valid int32 [B], kk)
        without touching the host."""
        assert len(cls_scores) == len(bbox_preds)
        nms_pre = int(_cfg_get(cfg, 'nms_pre'))
        nms_post = int(_cfg_get(cfg, 'nms_post'))
        max_num = int(_cfg_get(cfg, 'max_num'))
        nms_thr = float(_cfg_get(cfg, 'nms_thr'))
        min_size = float(_cfg_get(cfg, 'min_bbox_size', 0))
        across = bool(_cfg_get(cfg, 'nms_across_levels', False))
        L, B = len(cls_scores), len(img_metas)
        dev = cls_scores[0].device
        A = self.num_anchors

        # 1. top-k of sigmoid(score) per (image, level) segment, all in one pass set.  Segments are described by address:
        #    image b of level l starts b * A*D*H*W floats into the level's [B, A, D, H, W] tensor (no per-segment tensor
        #    views: 2 x B x L torch indexing calls cost more host time than the whole GPU path)
        cls_c, reg_c = [], []
        for l in range(L):
            c, r = cls_scores[l].detach(), bbox_preds[l].detach()
            check_cuda_f32(c, "cls_score", ndim=5)
            check_cuda_f32(r, "bbox_pred", ndim=5)
            assert c.shape[1] == A, "cls_score channels must equal num_anchors"
            assert c.shape[0] >= B and r.shape[0] >= B and tuple(r.shape[2:]) == tuple(c.shape[2:]) and r.shape[1] == 6 * A
            cls_c.append(c if c.is_contiguous() else c.contiguous())
            reg_c.append(r if r.is_contiguous() else r.contiguous())
        lvl_numel = [int(c.shape[1] * c.shape[2] * c.shape[3] * c.shape[4]) for c in cls_c]
        lvl_adhw = [[int(c.shape[1]), int(c.shape[2]), int(c.shape[3]), int(c.shape[4])] for c in cls_c]
        cls_ptr = [c.data_ptr() for c in cls_c]
        reg_ptr = [r.data_ptr() for r in reg_c]
        seg_meta = [(b, l) for b in range(B) for l in range(L)]
        seg_numel = [lvl_numel[l] for (_b, l) in seg_meta]
        seg_ptrs = [cls_ptr[l] + 4 * b * lvl_numel[l] for (b, l) in seg_meta]
        k = nms_pre if nms_pre > 0 else max(seg_numel)
        k = min(k, max(seg_numel))
        # Small descriptor tensors go up FIRST: a pageable host-to-device copy is stream-ordered and blocks the host,
        # so issued later it would wait for every kernel already queued and serialise the CPU with the GPU.
        counts = [min(k, n) for n in seg_numel]
        unsorted = [not (nms_pre > 0 and n > nms_pre) for n in seg_numel]
        # cached inside-flag masks: only on levels that are top-k'd, only when the shape matches (rpn_head_3d.py:96-106)
        masks = [None] * len(seg_meta)
        for j, (_b, l) in enumerate(seg_meta):
            if unsorted[j]:
                continue
            for lst in (self.pos_indices, self.pos_indices_test):
                if lst is not None and tuple(lst[l].shape) == (seg_numel[j],):
                    masks[j] = lst[l]
                    break
        masked = any(m is not None for m in masks)
        ckey = (tuple(counts), tuple(unsorted), dev)
        cached = self._desc_cache.get(ckey)
        if cached is None:  # they depend on the level shapes and the config only: uploaded once per shape signature
            cached = (torch.tensor(counts, dtype=torch.int32, device=dev),
                      torch.tensor(unsorted, dtype=torch.uint8, device=dev) if any(unsorted) else None,
                      torch.tensor([not u for u in unsorted], dtype=torch.uint8, device=dev))
            if len(self._desc_cache) > 16:
                self._desc_cache.clear()
            self._desc_cache[ckey] = cached
        seg_counts, use_idx, presorted = cached  # top-k'd levels reach the NMS already in score order
        # The reference only sorts a level when it has MORE than nms_pre anchors (rpn_head_3d.py:96,108-112);
        # a smaller level reaches NMS in anchor order, and `proposals[:nms_post]` then truncates in that order
        # (nms returns ascending input indices, nms_kernel.cu:253-256).  The top-k returns such segments whole in
        # ascending anchor order, and step 4 truncates them by original index instead of by score.
        # (nms_pre <= 0: no level is sorted, every level comes back whole in anchor order)
        seg_adhw = [lvl_adhw[l] for (_b, l) in seg_meta]
        if masked:  # the masked-in count decides, on the device, how many rows a level returns and whether it was sorted
            mask_keep = [None if m is None else _check_mask(m, seg_numel[j]) for j, m in enumerate(masks)]
            idx, val, seg_counts, presorted = _topk_segmented_desc(
                dev, seg_ptrs, seg_numel, seg_adhw, k, True, True, [None if m is None else m.data_ptr() for m in mask_keep], True)
            use_idx = 1 - presorted
            del mask_keep
        else:
            idx, val = _topk_segmented_desc(dev, seg_ptrs, seg_numel, seg_adhw, k, True, True, None, False)

        # 2. decode the selected anchors of every segment in ONE launch (anchors recomputed in closed form)
        dets = torch.empty((B * L, k, 7), dtype=torch.float32, device=dev)
        ptrs = (ctypes.c_void_p * len(seg_meta))(*[reg_ptr[l] + 4 * b * 6 * lvl_numel[l] for (b, l) in seg_meta])
        # host-side descriptors of the decode call depend on the level shapes, the image shapes and the head's constants only
        hkey = ("decode", B, tuple(tuple(a) for a in lvl_adhw), tuple(tuple(m['img_shape']) for m in img_metas[:B]))
        host = self._desc_cache.get(hkey)
        if host is None:
            host = (np.array(seg_adhw, dtype=np.int32),
                    np.array([l for (_b, l) in seg_meta], dtype=np.int32),
                    np.array([[img_metas[b]['img_shape'][0], img_metas[b]['img_shape'][1], img_metas[b]['img_shape'][3]]
                              for (b, _l) in seg_meta], dtype=np.float32),
                    np.ascontiguousarray(np.stack([g.base_anchors.numpy() for g in self.anchor_generators[:L]]),
                                         dtype=np.float32),
                    np.asarray(self.anchor_strides[:L], dtype=np.float32),
                    np.asarray(self.anchor_strides_depth[:L], dtype=np.float32),
                    np.asarray(self.target_means, dtype=np.float32),
                    np.asarray(self.target_stds, dtype=np.float32))
            if len(self._desc_cache) > 16:
                self._desc_cache.clear()
            self._desc_cache[hkey] = host
        adhw, lvl, img, base, strides, dstrides, means, stds = host
        with torch.cuda.device(dev):
            _lib.check(_lib.lib.roi3d_decode_proposals_batched(
                ptrs, adhw.ctypes.data, lvl.ctypes.data, img.ctypes.data, B * L, L, A, base.ctypes.data,
                strides.ctypes.data, dstrides.ctypes.data, idx.data_ptr(), val.data_ptr(), k, means.ctypes.data,
                stds.ctypes.data, dets.data_ptr(), stream_ptr()))
        if min_size > 0:
            # 2b. min_bbox_size: compact each segment's rows in place, in order, into a NEW count tensor (seg_counts may
            #     be the cached descriptor of this shape signature)
            kept = torch.empty_like(seg_counts)
            with torch.cuda.device(dev):
                _lib.check(_lib.lib.roi3d_filter_min_size_rows7(dets.data_ptr(), B * L, k, seg_counts.data_ptr(), min_size,
                                                                kept.data_ptr(), stream_ptr()))
            seg_counts = kept

        # 3. one batched NMS; kept rows in descending-score order
        #    (a score-sorted level only contributes proposals[:nms_post]: its sweep stops once that many are kept)
        keep_i, keep_s, num_keep = nms3d_batched(dets, seg_counts, nms_thr, want_score_order=True, presorted=presorted,
                                                 max_keep=nms_post)

        # 4. proposals[:nms_post] per segment (rpn_head_3d.py:135), per image cat in level order, topk(max_num)
        #    (:139-148): one collect kernel, one segmented top-k, one row gather
        P = min(nms_post, k)
        cat_props = torch.empty((B, L * P, 7), dtype=torch.float32, device=dev)
        cat_scores = torch.empty((B, L * P), dtype=torch.float32, device=dev)
        n_valid = torch.empty((B,), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib.roi3d_rpn_collect(
                dets.data_ptr(), B, L, k, keep_s.data_ptr(), keep_i.data_ptr(), num_keep.data_ptr(),
                None if use_idx is None else use_idx.data_ptr(), nms_post, cat_props.data_ptr(), cat_scores.data_ptr(),
                n_valid.data_ptr(), stream_ptr()))
        kk = min(max_num, L * P)
        if across:
            # rpn_head_3d.py:140-142: NMS over the concatenated levels, then the first max_num rows in the order nms
            # returns them (ascending position in the concatenation)
            fidx, _ks, nk = nms3d_batched(cat_props, n_valid, nms_thr)
            fidx = fidx[:, :kk].contiguous()
            n_valid = nk
        else:
            # (segments by address: B tensor views cost more host time than the launch)
            p0 = cat_scores.data_ptr()
            fidx, _ = _topk_segmented_desc(dev, [p0 + 4 * b * L * P for b in range(B)], [L * P] * B, None, kk, False, False,
                                           None, False)
        final = torch.empty((B, kk, 7), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib.roi3d_gather_rows7(cat_props.data_ptr(), B, L * P, fidx.data_ptr(), kk, final.data_ptr(),
                                                   stream_ptr()))
        return final, n_valid, kk

    def get_bboxes_single(self, cls_scores, bbox_preds, img_shape, cfg):
        """One image: cls_scores[l] [A, D, H, W], bbox_preds[l] [6A, D, H, W] (rpn_head_3d.py:72-79)."""
        out = self.get_proposals([c[None] for c in cls_scores], [r[None] for r in bbox_preds],
                                 [dict(img_shape=img_shape, scale_factor=1.0)], cfg)
        return out[0]

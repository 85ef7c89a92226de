"""ctypes binding of libroi3d_b200.so (the C ABI declared in include/roi3d_b200.h).

There is NO fallback: if the shared library is missing or fails to load, importing this module raises.
PyTorch is used above this layer only for device memory, streams and torch.distributed.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libroi3d_b200.so")

NCDHW = 0
NDHWC = 1
MAX_LEVELS = 8

c_void_p, c_int, c_float, c_size_t = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t


class Level(ctypes.Structure):
    """roi3d_level_t"""
    _fields_ = [("feats_dev", c_void_p), ("grad_dev", c_void_p), ("layout", ctypes.c_int32),
                ("D", ctypes.c_int32), ("H", ctypes.c_int32), ("W", ctypes.c_int32),
                ("spatial_scale", c_float), ("spatial_scale_depth", c_float)]


def level_array(tensors, scales, scales_d, grads=None, layout=NDHWC):
    """roi3d_level_t[] for the levels `tensors` ([B,C,D,H,W] each): feature pointers for a forward call, or with
    `grads` the gradient pointers of a backward call."""
    arr = (Level * len(tensors))()
    for i, t in enumerate(tensors):
        _, _, D, H, W = t.shape
        arr[i].feats_dev = t.data_ptr() if grads is None else None
        arr[i].grad_dev = None if grads is None else grads[i].data_ptr()
        arr[i].layout = layout
        arr[i].D, arr[i].H, arr[i].W = D, H, W
        arr[i].spatial_scale = scales[i]
        arr[i].spatial_scale_depth = scales_d[i]
    return arr


class Roi3dError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "roi3d_b200: %s not found. Build it with `bash 3d-multi-resolution-rcnn_b200/build.sh` "
            "(or __graft_entry__.build()). There is no CPU or PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    P = c_void_p
    sigs = {
        "roi3d_abi_version": (c_int, []),
        "roi3d_last_error": (ctypes.c_char_p, []),
        "roi3d_device_info": (c_int, [ctypes.POINTER(c_int)] * 3 + [ctypes.POINTER(c_size_t)]),
        "roi3d_set_tuning": (c_int, [c_int, c_int]),
        "roi3d_set_kernel_timing_events": (c_int, [P, P]),
        "roi3d_roi_align3d_forward": (c_int, [P, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int,
                                              c_int, c_float, c_float, c_int, P, P]),
        "roi3d_roi_align3d_forward_rows": (c_int, [P, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int,
                                                   c_int, c_int, c_float, c_float, c_int, P, P, P]),
        "roi3d_roi_align3d_backward": (c_int, [P, P, c_int, c_int, c_int, c_int, c_float, c_float, c_int, P, c_int,
                                               c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
        "roi3d_map_roi_levels": (c_int, [P, c_int, c_int, c_float, P, P]),
        "roi3d_extract_forward": (c_int, [ctypes.POINTER(Level), c_int, c_int, c_int, P, c_int, c_int, c_int, c_int,
                                          c_int, c_float, P, P, P]),
        "roi3d_extract_backward": (c_int, [ctypes.POINTER(Level), c_int, c_int, c_int, P, c_int, c_int, c_int, c_int,
                                           c_int, c_float, P, c_int, c_int, P]),
        "roi3d_extract_backward_deterministic": (c_int, [ctypes.POINTER(Level), c_int, c_int, c_int, P, c_int, c_int,
                                                         c_int, c_int, c_int, c_float, P, c_int, P]),
        "roi3d_ncdhw_to_ndhwc": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, P]),
        "roi3d_ndhwc_to_ncdhw": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, P]),
        "roi3d_nms3d_workspace_bytes": (c_size_t, [c_int, c_int]),
        "roi3d_nms3d_batched": (c_int, [P, P, c_int, c_int, c_float, P, P, P, P, c_size_t, P]),
        "roi3d_nms3d_batched_presorted": (c_int, [P, P, P, c_int, c_int, c_float, P, P, P, P, c_size_t, P]),
        "roi3d_nms3d_batched_limited": (c_int, [P, P, P, c_int, c_int, c_float, c_int, P, P, P, P, c_size_t, P]),
        "roi3d_nms3d_eval_batched": (c_int, [P, P, c_int, c_int, ctypes.c_double, P, P, P, P, c_size_t, P]),
        "roi3d_nms3d_host": (c_int, [P, c_int, c_float, P, P]),
        "roi3d_roi_align3d_forward_host": (c_int, [P, c_int, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int,
                                                   c_int, c_int, c_float, c_float, c_int, P]),
        "roi3d_mask_paste": (c_int, [P, c_int, c_int, c_int, c_int, P, P, c_float, P, P]),
        "roi3d_mask_target_workspace_bytes": (c_size_t, [P, c_int]),
        "roi3d_mask_target": (c_int, [P, c_int, c_int, c_int, c_int, P, P, c_int, c_int, c_int, c_int, P, P, c_size_t, P]),
        "roi3d_grid_anchors": (c_int, [c_int, c_int, c_int, c_int, c_float, c_float, P, c_int, c_int, c_int, c_float,
                                       c_float, c_float, c_int, P, P, P]),
        "roi3d_bbox_overlaps3d": (c_int, [P, c_int, c_int, P, c_int, c_int, P, P]),
        "roi3d_assign_workspace_bytes": (c_size_t, [c_int, c_int]),
        "roi3d_assign_max_iou": (c_int, [P, c_int, c_int, P, c_int, P, c_float, c_float, c_float, c_float, c_int, P, P, P,
                                         P, c_size_t, P]),
        "roi3d_assign_max_iou_ignore": (c_int, [P, c_int, c_int, P, c_int, P, P, c_float, c_float, c_float, c_float, c_int,
                                                P, P, P, P, c_size_t, P]),
        "roi3d_bbox2delta3d": (c_int, [P, c_int, P, c_int, c_int, P, P, P, P]),
        "roi3d_delta2bbox3d": (c_int, [P, c_int, P, c_int, c_int, P, P, c_float, c_float, c_float, c_float, P, P]),
        "roi3d_topk_workspace_bytes": (c_size_t, [c_int, c_int]),
        "roi3d_topk_workspace_bytes_keys": (c_size_t, [c_int, c_int, ctypes.c_int64]),
        "roi3d_topk_segmented": (c_int, [P, P, P, P, c_int, c_int, c_int, P, P, P, c_size_t, P]),
        "roi3d_topk_segmented_ex": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, P, P, P, c_size_t, P]),
        "roi3d_topk_segmented_masked": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, P, P, P, P, P, c_size_t, P]),
        "roi3d_rpn_collect": (c_int, [P, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P, P]),
        "roi3d_gather_rows7": (c_int, [P, c_int, c_int, P, c_int, P, P]),
        "roi3d_decode_proposals": (c_int, [P, c_int, c_int, c_int, c_int, c_float, c_float, P, P, P, c_int, P, P,
                                           c_float, c_float, c_float, P, P]),
        "roi3d_decode_proposals_batched": (c_int, [P, P, P, P, c_int, c_int, c_int, P, P, P, P, P, c_int, P, P, P, P]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.roi3d_abi_version() != 1:
        raise ImportError("roi3d_b200: ABI version mismatch (library %d, binding 1)" % lib.roi3d_abi_version())
    return lib, tuple(sigs)


lib, EXPORTS = _load()

# developer knob: pick a kernel variant for the whole process (see roi3d_set_tuning in the header)
for _key, _env in ((0, "ROI3D_FWD_VARIANT"), (1, "ROI3D_BWD_VARIANT"), (2, "ROI3D_FWD_ITEMS")):
    if os.environ.get(_env):
        lib.roi3d_set_tuning(_key, int(os.environ[_env]))


def check(rc):
    if rc != 0:
        msg = lib.roi3d_last_error()
        raise Roi3dError("libroi3d_b200: %s (code %d)" % (msg.decode() if msg else "error", rc))


def device_info():
    sm, mj, mn, l2 = c_int(), c_int(), c_int(), c_size_t()
    check(lib.roi3d_device_info(ctypes.byref(sm), ctypes.byref(mj), ctypes.byref(mn), ctypes.byref(l2)))
    return dict(sm_count=sm.value, cc=(mj.value, mn.value), l2_bytes=l2.value)


def set_tuning(key, value):
    check(lib.roi3d_set_tuning(int(key), int(value)))

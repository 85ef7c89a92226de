"""CPU checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every symbol that
include/roi3d_b200.h declares (no compute calls here)."""
import ctypes
import os
import re

from conftest import PKG, ROOT


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "roi3d_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(roi3d_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(os.path.join(PKG, "lib", "libroi3d_b200.so"))
    names = _declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "libroi3d_b200.so does not export %s" % n
    lib.roi3d_abi_version.restype = ctypes.c_int
    assert lib.roi3d_abi_version() == 1


def test_python_binding_covers_the_header():
    import roi3d_b200
    assert set(_declared_symbols()) == set(roi3d_b200._lib.EXPORTS)


def test_workspace_size_queries_are_host_only():
    import roi3d_b200
    lib = roi3d_b200._lib.lib
    n = 2000
    cb = (n + 63) // 64
    need = 32 * n + 4 * n + 8 * n * cb + n
    got = lib.roi3d_nms3d_workspace_bytes(1, n)
    assert need <= got <= need + 4 * 256
    assert lib.roi3d_topk_workspace_bytes(5, 2000) >= 5 * 2000 * 8


def test_surface_matches_reference_names():
    """Names a config / caller of the reference resolves (mmdet/ops/__init__.py:5-16, single_level.py:48-49,
    bbox_nms.py:75-77)."""
    import roi3d_b200
    from roi3d_b200 import ops
    from roi3d_b200.ops.nms import nms_wrapper
    for name in ("nms", "soft_nms", "RoIAlign3D"):
        assert hasattr(ops, name)
    assert callable(getattr(nms_wrapper, "nms"))
    ex = roi3d_b200.SingleRoIExtractor(dict(type='RoIAlign3D', out_size=7, out_size_depth=3, sample_num=2),
                                       out_channels=64, featmap_strides=[4, 8, 16, 32],
                                       featmap_strides_depth=[2, 4, 8, 16])
    assert ex.num_inputs == 4 and len(ex.roi_layers) == 4
    assert ex.roi_layers[1].spatial_scale == 1 / 8 and ex.roi_layers[1].spatial_scale_depth == 1 / 4
    assert ex.roi_layers[0].out_size == 7 and ex.roi_layers[0].out_size_depth == 3


def test_cpu_inputs_fail_loudly():
    import numpy as np
    import pytest
    import torch
    from roi3d_b200.ops import RoIAlign3D, nms
    with pytest.raises(NotImplementedError):
        RoIAlign3D(7, 7, 0.25, 0.5, 2)(torch.zeros(1, 4, 4, 4, 4), torch.zeros(1, 7))
    with pytest.raises(NotImplementedError):
        nms(torch.zeros(3, 7), 0.5)
    with pytest.raises(NotImplementedError):
        nms(np.zeros((3, 7), np.float32), 0.5)
    with pytest.raises(TypeError):
        nms([[0, 0, 1, 1, 0, 1, .5]], 0.5)
    d, i = nms(torch.zeros(0, 7), 0.5)
    assert d.shape == (0, 7) and i.dtype == torch.long and i.numel() == 0


def test_argument_errors_are_codes_with_messages_not_prints_or_exits():
    """Argument validation happens before any CUDA call, so it can be exercised without a GPU.  The reference prints
    and returns 0 (roi_align_cuda.cpp:80-83) or calls exit(-1) (roi_align_kernel.cu:679-682) on bad input."""
    import ctypes

    import roi3d_b200
    from roi3d_b200 import _lib
    lib = _lib.lib
    lv = (_lib.Level * 1)()
    lv[0].layout = 7                   # neither NCDHW nor NDHWC: must be refused, not mis-read
    lv[0].D, lv[0].H, lv[0].W = 4, 4, 4
    lv[0].feats_dev = 1 << 20
    rc = lib.roi3d_extract_forward(lv, 1, 1, 32, 1 << 20, 5, 7, 7, 7, 2, 56.0, 1 << 20, None, None)
    assert rc == -1 and b"layout" in lib.roi3d_last_error()
    rc = lib.roi3d_extract_forward(lv, 0, 1, 32, None, 0, 7, 7, 7, 2, 56.0, None, None, None)
    assert rc == -1 and b"num_levels" in lib.roi3d_last_error()
    rc = lib.roi3d_nms3d_batched(None, None, -1, 10, 0.5, None, None, None, None, 0, None)
    assert rc == -1
    rc = lib.roi3d_nms3d_batched(1 << 20, None, 1, 1 << 20, 0.5, 1 << 20, None, 1 << 20, 1 << 20, 1 << 30, None)
    assert rc == -1 and b"n_max" in lib.roi3d_last_error()
    with __import__("pytest").raises(_lib.Roi3dError):
        _lib.check(lib.roi3d_topk_segmented(None, None, None, None, 1, 5, 0, None, None, None, 0, None))
    assert lib.roi3d_set_tuning(77, 0) == -1
    # empty work is a no-op success, as in the reference wrapper (nms_wrapper.py:39-40)
    assert lib.roi3d_nms3d_batched(None, None, 0, 0, 0.5, None, None, None, None, 0, None) == 0
    n = ctypes.c_int32(7)
    assert lib.roi3d_nms3d_host(None, 0, 0.5, None, ctypes.addressof(n)) == 0 and n.value == 0


def test_set_tuning_accepts_exactly_the_documented_pairs():
    """roi3d_set_tuning takes the key / value pairs its header comment lists and refuses every other one with a message
    naming both, so that a call for a removed or misspelt variant cannot silently run the default kernels."""
    from roi3d_b200 import _lib
    lib = _lib.lib
    accepted = [(0, 0), (0, 50), (0, 60), (0, 99), (1, 0), (1, 50), (1, 60), (4, -1), (4, 0), (4, 1024),
                (10, 0), (10, 5000), (11, -1), (11, 0), (11, 2)]
    rejected = [(2, 0), (2, 7), (6, 0), (6, 1), (7, 0), (7, 1), (9, 0), (9, 2), (0, 1), (0, 40), (1, 1), (1, 3),
                (1, 99), (4, -2), (10, -1), (11, 1), (11, 5), (77, 0)]
    try:
        for key, value in accepted:
            assert lib.roi3d_set_tuning(key, value) == 0, (key, value)
        for key, value in rejected:
            assert lib.roi3d_set_tuning(key, value) == -1, (key, value)
            msg = lib.roi3d_last_error().decode()
            assert "key %d" % key in msg and "value %d" % value in msg, msg
    finally:
        for key in (0, 1, 4, 10, 11):
            assert lib.roi3d_set_tuning(key, 0) == 0

"""The deterministic RoIAlign3D / RoI-extractor backward (csrc/roi_align3d_det.cu, roi3d_extract_backward_deterministic)
that RoIAlign3D and SingleRoIExtractor take under torch.use_deterministic_algorithms(True): parity with the float64
oracle, the same bits on every run whatever else runs on the GPU, the accumulate / overwrite contract, CUDA-graph
capture, and the flag handling.  The module fixture turns torch's flag on for this file only and restores it."""
import contextlib
import ctypes

import numpy as np
import pytest
import torch

import synth
from test_gpu_parity import BWD_TOL, CASES, _feats, _pyramid, cl, rel_err


@pytest.fixture(scope="module", autouse=True)
def deterministic_flag():
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


@contextlib.contextmanager
def flag(on, warn_only=False):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _grad(layer, ft, rois, g):
    """d(layer(ft, rois)) / d ft for output gradient g, without touching ft.grad."""
    x = ft.detach().requires_grad_(True)
    out = layer(x, rois)
    (gx,) = torch.autograd.grad(out, x, g)
    return gx


def _det_entry(grads, scales, scales_d, rois, out_dims, sn, gout, accumulate, finest=56.0):
    from roi3d_b200 import _lib
    from roi3d_b200._util import stream_ptr
    B, C = grads[0].shape[:2]
    K = rois.size(0)
    arr = _lib.level_array(grads, scales, scales_d, grads=grads)
    _lib.check(_lib.lib.roi3d_extract_backward_deterministic(
        arr, len(grads), B, C, rois.data_ptr() if K else None, K, *out_dims, sn, finest,
        gout.data_ptr() if K else None, accumulate, stream_ptr()))


def _cl_empty(shape, dev, fill=None):
    t = torch.empty(shape, device=dev, memory_format=torch.channels_last_3d)
    if fill is not None:
        t.fill_(fill)
    return t


def _clustered_rois(k, seed, img, batch=1):
    """k RoIs whose centres lie within a few pixels of one spot: every voxel there is shared by hundreds of RoIs."""
    rng = np.random.default_rng(seed)
    W, H, D = img
    cx, cy, cz = W / 2 + rng.uniform(-4, 4, k), H / 2 + rng.uniform(-4, 4, k), D / 2 + rng.uniform(-2, 2, k)
    w, h, d = rng.uniform(12, 48, k), rng.uniform(12, 48, k), rng.uniform(4, 14, k)
    b = rng.integers(0, batch, k)
    return np.stack([b, cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2, cz - d / 2, cz + d / 2], 1).astype(np.float32)


# ------------------------------------------------------------------------------------------ 1. oracle parity
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("layout", ["channels_last", "contiguous"])
def test_det_backward_matches_oracle(oracle, dev, case, layout):
    """Every parity case, the wide-footprint one (CASES[6]) included, with the adversarial RoIs."""
    from roi3d_b200.ops import RoIAlign3D
    shape, ps, pdp, sc, scd, sn, k = case
    B, C, D, H, W = shape
    img = (int(W / sc), int(H / sc), int(D / scd))
    rois = np.concatenate([synth.c2_rois(k, seed=2, img=img, batch=B),
                           synth.adversarial_rois((D, H, W), sc, scd, batch=B)], 0)
    ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
    rois = rois[ok] if sn == 0 else rois          # (zero-size adaptive RoIs: test_det_skipped_rois_change_nothing)
    g = _feats((rois.shape[0], C, pdp, ps, ps), 6)
    want = oracle.roi_align3d_backward(g, rois, shape, sc, scd, sn)
    ft = torch.from_numpy(_feats(shape, 1)).to(dev)
    if layout == "channels_last":
        ft = cl(ft)
    ft.requires_grad_(True)
    out = RoIAlign3D(ps, pdp, sc, scd, sn)(ft, torch.from_numpy(rois).to(dev))
    out.backward(torch.from_numpy(g).to(dev))
    assert ft.grad.shape == tuple(shape)
    assert ft.grad.is_contiguous(memory_format=torch.channels_last_3d if layout == "channels_last"
                                 else torch.contiguous_format)
    assert rel_err(ft.grad.cpu().numpy(), want) <= BWD_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("ps,pdp", [(7, 7), (14, 10)])
def test_det_extractor_multilevel_matches_oracle(oracle, dev, ps, pdp):
    from roi3d_b200 import SingleRoIExtractor
    B, C = 2, 64
    strides, dstrides = [4, 8, 16, 32], [2, 4, 8, 16]
    feats = _pyramid(B, C, 20)
    rois = synth.c3_rois(60, vols=B, seed=4, img=(128, 128, 20))
    lv = oracle.map_roi_levels(rois, 4)
    assert len(np.unique(lv)) >= 3
    g = _feats((rois.shape[0], C, pdp, ps, ps), 30)
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=ps, out_size_depth=pdp, sample_num=2), C, strides,
                            dstrides)
    for layout in ("channels_last", "contiguous"):
        ft = [torch.from_numpy(f).to(dev) for f in feats]
        ft = [(cl(f) if layout == "channels_last" else f).requires_grad_(True) for f in ft]
        ex(ft, torch.from_numpy(rois).to(dev)).backward(torch.from_numpy(g).to(dev))
        for l in range(4):
            sel = lv == l
            want = oracle.roi_align3d_backward(g[sel], rois[sel], feats[l].shape, 1 / strides[l], 1 / dstrides[l], 2)
            assert rel_err(ft[l].grad.cpu().numpy(), want) <= BWD_TOL, (layout, l)


# ------------------------------------------------------------------------------------ 2. bit-for-bit repeatability
@pytest.mark.gpu
@pytest.mark.parametrize("ps,pdp,k", [(7, 3, 2000), (14, 10, 512)])
def test_det_backward_is_bitwise_repeatable_under_heavy_overlap(dev, ps, pdp, k):
    from roi3d_b200.models.roi_extractors.single_level import _MultiLevelRoIAlign3D
    from roi3d_b200.ops import RoIAlign3D
    shape = (1, 256, 16, 64, 64)
    sc, scd = 0.25, 0.5
    gen = torch.Generator(device=dev)
    gen.manual_seed(11)
    ft = cl(torch.randn(shape, device=dev, generator=gen))
    rois = torch.from_numpy(_clustered_rois(k, 12, (256, 256, 32))).to(dev)
    g = torch.randn((k, 256, pdp, ps, ps), device=dev, generator=gen)
    layer = RoIAlign3D(ps, pdp, sc, scd, 2)
    ref = _grad(layer, ft, rois, g)
    for _ in range(2):
        assert torch.equal(_grad(layer, ft, rois, g), ref)
    # once more while a large matmul occupies SMs from a second stream: a different CTA schedule
    side = torch.cuda.Stream()
    a = torch.randn((8192, 8192), device=dev, generator=gen)
    side.wait_stream(torch.cuda.current_stream())
    with flag(False), torch.cuda.stream(side):
        for _ in range(4):
            a = a @ a * (1.0 / 64)
    busy = _grad(layer, ft, rois, g)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    assert torch.equal(busy, ref)
    # the one-level extractor entry gives the same bits as RoIAlign3D
    x = ft.detach().requires_grad_(True)
    out = _MultiLevelRoIAlign3D.apply(rois, (pdp, ps, ps), [sc], [scd], 2, 56.0, x)
    (gx,) = torch.autograd.grad(out, x, g)
    assert torch.equal(gx, ref)
    # and the atomic path agrees within the backward tolerance
    with flag(False):
        atomic = _grad(layer, ft, rois, g)
    assert rel_err(ref.cpu().numpy(), atomic.cpu().numpy()) <= BWD_TOL


# ----------------------------------------------------------------------------------------- 3. long tile lists
@pytest.mark.gpu
def test_det_backward_long_tile_lists(oracle, dev):
    """20 000 RoIs on a 6 x 16 x 16 level: every tile's list spans many scan steps."""
    from roi3d_b200.ops import RoIAlign3D
    k = 20000
    rois_np = synth.c2_rois(k, seed=21, img=(64, 64, 12))
    rois = torch.from_numpy(rois_np).to(dev)
    layer = RoIAlign3D(7, 3, 0.25, 0.5, 2)
    for C in (64, 8):
        shape = (1, C, 6, 16, 16)
        ft = cl(torch.from_numpy(_feats(shape, 22)).to(dev))
        g_np = _feats((k, C, 3, 7, 7), 23)
        g = torch.from_numpy(g_np).to(dev)
        det = _grad(layer, ft, rois, g)
        with flag(False):
            atomic = _grad(layer, ft, rois, g)
        assert rel_err(det.cpu().numpy(), atomic.cpu().numpy()) <= BWD_TOL, C
        if C == 8:
            want = oracle.roi_align3d_backward(g_np, rois_np, shape, 0.25, 0.5, 2)
            assert rel_err(det.cpu().numpy(), want) <= BWD_TOL


# ---------------------------------------------------------------------------------------------- 4. skipped RoIs
@pytest.mark.gpu
def test_det_skipped_rois_change_nothing(dev):
    """A zero-size RoI under adaptive sampling (S = 0) and RoIs whose batch index is out of range add nothing: the
    gradient keeps its bits and holds no NaN."""
    from roi3d_b200.ops import RoIAlign3D
    shape = (1, 32, 6, 16, 16)
    ft = cl(torch.from_numpy(_feats(shape, 31)).to(dev))
    base = synth.c2_rois(30, seed=32, img=(64, 64, 12))
    extra = np.array([[0, 10, 10, 9, 9, 4, 3], [1, 8, 8, 30, 30, 2, 8], [-1, 8, 8, 30, 30, 2, 8]], np.float32)
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 0)
    g = torch.from_numpy(_feats((33, 32, 7, 7, 7), 33)).to(dev)
    ref = _grad(layer, ft, torch.from_numpy(base).to(dev), g[:30])
    got = _grad(layer, ft, torch.from_numpy(np.concatenate([base, extra])).to(dev), g)
    assert not torch.isnan(got).any()
    assert torch.equal(got, ref)


# ------------------------------------------------------------------------------------------------ 5. accumulate
@pytest.mark.gpu
def test_det_accumulate_and_overwrite(dev):
    B, C = 2, 48
    strides, dstrides = [4, 8], [2, 4]
    shapes = [(B, C, 10, 32, 32), (B, C, 5, 16, 16)]
    rois = torch.from_numpy(synth.c3_rois(40, vols=B, seed=41, img=(128, 128, 20))).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(42)
    gout = torch.randn((rois.size(0), C, 3, 7, 7), device=dev, generator=gen)
    args = ([1 / s for s in strides], [1 / d for d in dstrides], rois, (3, 7, 7), 2, gout)
    fresh = [_cl_empty(s, dev, float("nan")) for s in shapes]
    _det_entry(fresh, *args, accumulate=0)
    prefill = [cl(torch.randn(s, device=dev, generator=gen)) for s in shapes]
    acc = [p.clone(memory_format=torch.channels_last_3d) for p in prefill]
    _det_entry(acc, *args, accumulate=1)
    torch.cuda.synchronize()
    assert any(float(f.abs().max()) > 0 for f in fresh)
    for f, p, a in zip(fresh, prefill, acc):
        assert not torch.isnan(f).any()
        assert torch.equal(a, p + f)
    # K = 0: accumulate = 0 still overwrites every voxel of every level with zeros
    nan = [_cl_empty(s, dev, float("nan")) for s in shapes]
    _det_entry(nan, args[0], args[1], rois[:0], (3, 7, 7), 2, gout, accumulate=0)
    torch.cuda.synchronize()
    for t in nan:
        assert torch.equal(t, torch.zeros_like(t))


# ------------------------------------------------------------------------------------------------- 6. CUDA graph
@pytest.mark.gpu
def test_det_entry_in_a_cuda_graph(dev):
    shape = (1, 64, 10, 32, 32)
    rois = torch.from_numpy(_clustered_rois(300, 51, (128, 128, 20))).to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(52)
    gout = torch.randn((300, 64, 7, 7, 7), device=dev, generator=gen)
    eager = [_cl_empty(shape, dev)]
    _det_entry(eager, [0.25], [0.5], rois, (7, 7, 7), 2, gout, accumulate=0)
    torch.cuda.synchronize()
    out = [_cl_empty(shape, dev, float("nan"))]
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _det_entry(out, [0.25], [0.5], rois, (7, 7, 7), 2, gout, accumulate=0)
    for _ in range(2):
        out[0].fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out[0], eager[0])


# --------------------------------------------------------------------------------------- 7. full-size C2 and C3
@pytest.mark.gpu
def test_det_c2_full_size(dev):
    from roi3d_b200.ops import RoIAlign3D
    gen = torch.Generator(device=dev)
    gen.manual_seed(61)
    shape = (1, 256, 40, 128, 128)
    x = cl(torch.randn(shape, device=dev, generator=gen))
    rois = torch.from_numpy(synth.c2_rois(512, seed=2)).to(dev)
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 2)
    g = torch.randn((512, 256, 7, 7, 7), device=dev, generator=gen)
    det = _grad(layer, x, rois, g)
    assert torch.equal(_grad(layer, x, rois, g), det)
    with flag(False):
        atomic = _grad(layer, x, rois, g)
    assert rel_err(det.cpu().numpy(), atomic.cpu().numpy()) <= BWD_TOL


@pytest.mark.gpu
def test_det_c3_full_size(dev):
    from roi3d_b200 import SingleRoIExtractor
    B, C = 2, 256
    dims = [(40, 128, 128), (20, 64, 64), (10, 32, 32), (5, 16, 16)]
    gen = torch.Generator(device=dev)
    gen.manual_seed(62)
    pyr = [cl(torch.randn((B, C) + d, device=dev, generator=gen)).requires_grad_(True) for d in dims]
    rois = torch.from_numpy(synth.c3_rois(512, vols=B, seed=4)).to(dev)
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=14, out_size_depth=14, sample_num=2), C,
                            [4, 8, 16, 32], [2, 4, 8, 16])
    out = ex(pyr, rois)
    g = torch.randn(out.shape, device=dev, generator=gen)
    det = torch.autograd.grad(out, pyr, g, retain_graph=True)
    det2 = torch.autograd.grad(out, pyr, g, retain_graph=True)
    with flag(False):
        atomic = torch.autograd.grad(out, pyr, g)
    for l in range(4):
        assert torch.equal(det[l], det2[l]), l
        assert rel_err(det[l].cpu().numpy(), atomic[l].cpu().numpy()) <= BWD_TOL, l


# ---------------------------------------------------------------------------------------------- 8. flag handling
@pytest.mark.gpu
def test_flag_selects_the_kernel(dev, monkeypatch):
    """Flag on: the deterministic entry; flag off: the atomic entry, as before."""
    from roi3d_b200 import _lib
    from roi3d_b200.ops import RoIAlign3D
    calls = []
    real = _lib.lib.roi3d_extract_backward_deterministic

    def spy(*a):
        calls.append(1)
        return real(*a)
    monkeypatch.setattr(_lib.lib, "roi3d_extract_backward_deterministic", spy)
    ft = cl(torch.from_numpy(_feats((1, 32, 6, 16, 16), 71)).to(dev))
    rois = torch.from_numpy(synth.c2_rois(10, seed=72, img=(64, 64, 12))).to(dev)
    layer = RoIAlign3D(7, 3, 0.25, 0.5, 2)
    g = torch.ones((10, 32, 3, 7, 7), device=dev)
    with flag(False):
        off = _grad(layer, ft, rois, g)
    assert calls == []
    on = _grad(layer, ft, rois, g)
    assert calls == [1]
    assert rel_err(on.cpu().numpy(), off.cpu().numpy()) <= BWD_TOL


@pytest.mark.gpu
def test_bug_compat_raises_or_warns(oracle, dev):
    from roi3d_b200.ops import RoIAlign3D, set_bug_compat
    shape = (1, 32, 9, 15, 15)
    rois_np = synth.c2_rois(6, seed=5, img=(60, 60, 18))
    rois = torch.from_numpy(rois_np).to(dev)
    g = _feats((6, 32, 3, 7, 7), 7)
    layer = RoIAlign3D(7, 3, 0.25, 0.5, 2)
    ft = cl(torch.zeros(shape, device=dev))
    set_bug_compat(True)
    try:
        with pytest.raises(RuntimeError, match="RoIAlignFunction3D"):
            _grad(layer, ft, rois, torch.from_numpy(g).to(dev))
        with flag(True, warn_only=True), pytest.warns(UserWarning, match="deterministic"):
            got = _grad(layer, ft, rois, torch.from_numpy(g).to(dev))
    finally:
        set_bug_compat(False)
    want = oracle.roi_align3d_backward(g, rois_np, shape, 0.25, 0.5, 2, bug_compat=True)
    assert rel_err(got.cpu().numpy(), want) <= BWD_TOL


@pytest.mark.gpu
def test_forward_is_bitwise_repeatable_under_the_flag(dev):
    from roi3d_b200 import SingleRoIExtractor
    from roi3d_b200.ops import RoIAlign3D
    gen = torch.Generator(device=dev)
    gen.manual_seed(81)
    x = cl(torch.randn((1, 256, 40, 128, 128), device=dev, generator=gen))
    rois = torch.from_numpy(synth.c2_rois(512, seed=2)).to(dev)
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 2)
    assert torch.equal(layer(x, rois), layer(x, rois))
    del x
    feats = [cl(torch.from_numpy(f).to(dev)) for f in _pyramid(2, 64, 82)]
    rois = torch.from_numpy(synth.c3_rois(200, vols=2, seed=83, img=(128, 128, 20))).to(dev)
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=14, out_size_depth=10, sample_num=2), 64,
                            [4, 8, 16, 32], [2, 4, 8, 16])
    assert torch.equal(ex(feats, rois), ex(feats, rois))


# ------------------------------------------------------------------------------------------ 9. CPU, no GPU needed
def test_det_entry_argument_errors_before_any_cuda_call():
    from roi3d_b200 import _lib
    lib = _lib.lib
    fn = lib.roi3d_extract_backward_deterministic
    lv = (_lib.Level * 1)()
    lv[0].layout = _lib.NCDHW
    lv[0].D, lv[0].H, lv[0].W = 4, 4, 4
    lv[0].grad_dev = 1 << 20
    assert fn(lv, 1, 1, 32, 1 << 20, 5, 7, 7, 7, 2, 56.0, 1 << 20, 0, None) == -1
    assert b"layout" in lib.roi3d_last_error()
    lv[0].layout = _lib.NDHWC
    assert fn(lv, 0, 1, 32, 1 << 20, 5, 7, 7, 7, 2, 56.0, 1 << 20, 0, None) == -1
    assert b"num_levels" in lib.roi3d_last_error()
    assert fn(lv, 1, 1, 32, 1 << 20, 5, 7, 7, 7, 2, 56.0, None, 0, None) == -1
    assert b"grad_out" in lib.roi3d_last_error()
    assert ctypes.c_int(fn(lv, 1, 1, 32, 1 << 20, 5, 0, 7, 7, 2, 56.0, 1 << 20, 0, None)).value == -1

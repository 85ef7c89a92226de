"""3D soft-NMS: `ops.soft_nms`, `soft_nms3d_batched` and `multiclass_nms_3d(nms=dict(type='soft_nms'))`.

The chain of checks:
  * `ref_soft_nms_2d` below is a literal transcription of the reference loop (soft_nms_cpu, mmdet v0.6.0
    mmdet/ops/nms/src/soft_nms_cpu.pyx) with np.float32 scalars; `ref_soft_nms_3d` is the same loop with a depth axis.
    On the CPU they equal the C oracle (oracle_soft_nms3d in soft_nms_oracle.c) bit for bit: the 2-D loop on flat
    boxes (z1 = z2 = 0, where every depth factor is an exact 1), the 3-D loop on 3-D boxes;
  * on the GPU the kernel equals the C oracle bit for bit: rows, selection-time scores, indices and counts.
The oracle runs the loop in its sequential form (swaps and tail moves); the kernel renumbers the tail moves in closed
form, so the GPU rows with heavy drops check that form against the loop."""
import ctypes

import numpy as np
import pytest
import torch

import soft_nms_oracle as soft_oracle
import synth
from kernel_inventory import built_kernels, launched_kernels, library_kernels

METHOD = {'linear': 1, 'gaussian': 2}
F32 = np.float32


# --------------------------------------------------------------------------------- literal transcriptions (CPU)
def _max(a, b):
    return a if a >= b else b


def _min(a, b):
    return a if a <= b else b


def ref_soft_nms_2d(boxes_in, iou_thr, method=1, sigma=0.5, min_score=0.001):
    """soft_nms_cpu as written (2-D, [N,5] with the score in column 4); every scalar an np.float32."""
    boxes = np.array(boxes_in, dtype=np.float32, copy=True)
    N = boxes.shape[0]
    inds = np.arange(N)
    Nt, sigma, min_score = F32(iou_thr), F32(sigma), F32(min_score)
    for i in range(N):
        maxscore = boxes[i, 4]
        maxpos = i
        tx1, ty1, tx2, ty2, ts = boxes[i, 0], boxes[i, 1], boxes[i, 2], boxes[i, 3], boxes[i, 4]
        ti = inds[i]
        pos = i + 1
        while pos < N:
            if maxscore < boxes[pos, 4]:
                maxscore = boxes[pos, 4]
                maxpos = pos
            pos = pos + 1
        boxes[i, :] = boxes[maxpos, :]
        inds[i] = inds[maxpos]
        boxes[maxpos, 0], boxes[maxpos, 1], boxes[maxpos, 2], boxes[maxpos, 3], boxes[maxpos, 4] = tx1, ty1, tx2, ty2, ts
        inds[maxpos] = ti
        tx1, ty1, tx2, ty2, ts = boxes[i, 0], boxes[i, 1], boxes[i, 2], boxes[i, 3], boxes[i, 4]
        pos = i + 1
        while pos < N:
            x1, y1, x2, y2, s = boxes[pos, 0], boxes[pos, 1], boxes[pos, 2], boxes[pos, 3], boxes[pos, 4]
            area = (x2 - x1 + F32(1)) * (y2 - y1 + F32(1))
            iw = (_min(tx2, x2) - _max(tx1, x1) + F32(1))
            if iw > 0:
                ih = (_min(ty2, y2) - _max(ty1, y1) + F32(1))
                if ih > 0:
                    ua = F32((tx2 - tx1 + F32(1)) * (ty2 - ty1 + F32(1)) + area - iw * ih)
                    ov = iw * ih / ua
                    if method == 1:
                        weight = F32(1) - ov if ov > Nt else F32(1)
                    else:
                        weight = F32(np.exp(float(-(ov * ov) / sigma)))
                    boxes[pos, 4] = weight * boxes[pos, 4]
                    if boxes[pos, 4] < min_score:
                        boxes[pos, :] = boxes[N - 1, :]
                        inds[pos] = inds[N - 1]
                        N = N - 1
                        pos = pos - 1
            pos = pos + 1
    return boxes[:N], inds[:N]


def ref_soft_nms_3d(boxes_in, iou_thr, method=1, sigma=0.5, min_score=0.001):
    """The same loop on [N,7] = (x1,y1,x2,y2,z1,z2,score): a depth guard nested inside the others, volumes
    ((w*h)*d), inter = (iw*ih)*id, ua = (tarea + area) - inter."""
    boxes = np.array(boxes_in, dtype=np.float32, copy=True)
    N = boxes.shape[0]
    inds = np.arange(N)
    Nt, sigma, min_score = F32(iou_thr), F32(sigma), F32(min_score)
    one = F32(1)
    for i in range(N):
        maxscore = boxes[i, 6]
        maxpos = i
        t = boxes[i, :].copy()
        ti = inds[i]
        pos = i + 1
        while pos < N:
            if maxscore < boxes[pos, 6]:
                maxscore = boxes[pos, 6]
                maxpos = pos
            pos = pos + 1
        boxes[i, :] = boxes[maxpos, :]
        inds[i] = inds[maxpos]
        boxes[maxpos, :] = t
        inds[maxpos] = ti
        tx1, ty1, tx2, ty2, tz1, tz2 = (boxes[i, c] for c in range(6))
        pos = i + 1
        while pos < N:
            x1, y1, x2, y2, z1, z2 = (boxes[pos, c] for c in range(6))
            area = ((x2 - x1 + one) * (y2 - y1 + one)) * (z2 - z1 + one)
            iw = _min(tx2, x2) - _max(tx1, x1) + one
            if iw > 0:
                ih = _min(ty2, y2) - _max(ty1, y1) + one
                if ih > 0:
                    idp = _min(tz2, z2) - _max(tz1, z1) + one
                    if idp > 0:
                        tarea = ((tx2 - tx1 + one) * (ty2 - ty1 + one)) * (tz2 - tz1 + one)
                        inter = (iw * ih) * idp
                        ua = (tarea + area) - inter
                        ov = inter / ua
                        if method == 1:
                            weight = one - ov if ov > Nt else one
                        else:
                            weight = F32(np.exp(float(-(ov * ov) / sigma)))
                        boxes[pos, 6] = weight * boxes[pos, 6]
                        if boxes[pos, 6] < min_score:
                            boxes[pos, :] = boxes[N - 1, :]
                            inds[pos] = inds[N - 1]
                            N = N - 1
                            pos = pos - 1
            pos = pos + 1
    return boxes[:N], inds[:N]


# --------------------------------------------------------------------------------------------------- inputs
def dense_boxes(n, seed, levels=None, span=48.0):
    """Boxes packed into a small volume so most pairs overlap; scores from `levels` (tie-heavy) or distinct."""
    rng = np.random.default_rng(seed)
    lo = rng.uniform(0, span, (n, 3))
    size = rng.uniform(4, 20, (n, 3))
    hi = lo + size
    if levels is None:
        s = rng.permutation(np.linspace(0.05, 0.99, n)) if n else np.zeros(0)
    else:
        s = rng.choice(np.asarray(levels, np.float64), n)
    return np.stack([lo[:, 0], lo[:, 1], hi[:, 0], hi[:, 1], lo[:, 2], hi[:, 2], s], 1).astype(np.float32)


def tie_boxes(n, seed):
    """C1-style clustered boxes with scores drawn from five values."""
    d = synth.c1_boxes(max(n, 1), seed=seed)[:n]
    rng = np.random.default_rng(seed + 1)
    d[:, 6] = rng.choice(np.array([0.1, 0.25, 0.5, 0.75, 1.0], np.float32), n)
    return d


def edge_boxes(n, seed):
    """Dense boxes with tied scores, -0.0 next to +0.0, NaN scores, scores below min_score and a few disjoint rows."""
    d = dense_boxes(n, seed, levels=(0.02, 0.2, 0.5, 0.9))
    rng = np.random.default_rng(seed + 7)
    k = max(n // 16, 1)
    d[rng.choice(n, k), 6] = np.float32(np.nan)
    d[rng.choice(n, k), 6] = np.float32(-0.0)
    d[rng.choice(n, k), 6] = np.float32(0.0)
    d[rng.choice(n, k), 6] = np.float32(0.0004)                 # below every min_score used here
    far = rng.choice(n, k)
    d[far, :6] += np.float32(1000.0) + np.arange(k, dtype=np.float32)[:, None] * 100   # disjoint from everything
    return d


def flat(boxes5):
    """[N,5] 2-D rows -> [N,7] 3-D rows with z1 = z2 = 0."""
    b = np.asarray(boxes5, np.float32)
    z = np.zeros((b.shape[0], 1), np.float32)
    return np.concatenate([b[:, :4], z, z, b[:, 4:5]], 1)


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


CONFIGS = [('linear', 0.3, 0.5, 0.001), ('linear', 0.5, 0.5, 0.05), ('linear', 0.0, 0.5, 0.2),
           ('gaussian', 0.3, 0.5, 0.001), ('gaussian', 0.3, 0.2, 0.05), ('gaussian', 0.3, 1.5, 0.3)]


def _cpu_cases():
    yield "n0", dense_boxes(0, 1)
    yield "n1", dense_boxes(1, 2)
    yield "n2", dense_boxes(2, 3)
    yield "n2_same", np.repeat(dense_boxes(1, 4), 2, 0)
    yield "ties", dense_boxes(120, 5, levels=(0.2, 0.5, 0.9))
    yield "one_value", dense_boxes(60, 6, levels=(0.5,))
    yield "edge", edge_boxes(150, 8)
    yield "distinct", dense_boxes(150, 9)
    yield "c1_ties", tie_boxes(150, 10)


# -------------------------------------------------------------------------------------------------- CPU tests
@pytest.mark.parametrize("method,thr,sigma,min_score", CONFIGS)
def test_transcriptions_equal_oracle(method, thr, sigma, min_score):
    for name, d in _cpu_cases():
        want_d, want_i = soft_oracle.soft_nms3d(d, thr, method, sigma, min_score)
        got_d, got_i = ref_soft_nms_3d(d, thr, METHOD[method], sigma, min_score)
        assert same_bits(got_d, want_d) and np.array_equal(got_i, want_i), name
        # the 2-D reference loop on the same x / y rows equals the oracle on the flattened boxes
        d5 = d[:, [0, 1, 2, 3, 6]]
        ref_d, ref_i = ref_soft_nms_2d(d5, thr, METHOD[method], sigma, min_score)
        fl_d, fl_i = soft_oracle.soft_nms3d(flat(d5), thr, method, sigma, min_score)
        assert same_bits(flat(ref_d), fl_d) and np.array_equal(ref_i, fl_i), name


def test_oracle_properties():
    """Rules the kernel must reproduce, seen on the oracle: NaN selected only at position i and never dropped; a row
    below min_score survives until something overlaps it; selection-time scores; ±0 tie."""
    box = [0, 0, 9, 9, 0, 9]
    far = [100, 100, 109, 109, 100, 109]
    d = np.array([box + [np.nan], box + [0.9], far + [0.0001], box + [0.5]], np.float32)
    out, inds = soft_oracle.soft_nms3d(d, 0.3, 'linear', 0.5, 0.001)
    # position 0 holds the NaN: it is selected first; it never wins later and never drops
    assert inds[0] == 0 and np.isnan(out[0, 6])
    assert 2 in inds                                       # disjoint, below min_score, never tested: kept
    assert out[list(inds).index(2), 6] == np.float32(0.0001)
    z = np.array([box + [-0.0], far + [0.0]], np.float32)
    _, zi = soft_oracle.soft_nms3d(z, 0.3, 'linear', 0.5, -1.0)
    assert list(zi) == [0, 1]                              # -0.0 ties +0.0: the first position wins
    with pytest.raises(ValueError, match="Invalid method for SoftNMS"):
        soft_oracle.soft_nms3d(d, 0.3, 'hard')


def test_abi_argument_errors_return_before_any_launch():
    from roi3d_b200 import _lib
    lib = _lib.lib
    A = 1 << 20
    f = lib.roi3d_soft_nms3d_batched
    for method in (0, 3, -1):
        assert f(A, None, 1, 10, method, 0.3, 0.5, 1e-3, A, A, A, None) == -1
        assert b"method" in lib.roi3d_last_error()
    assert f(A, None, 1, 4097, 1, 0.3, 0.5, 1e-3, A, A, A, None) == -1
    assert b"n_max" in lib.roi3d_last_error() and b"4096" in lib.roi3d_last_error()
    assert f(A, None, -1, 10, 1, 0.3, 0.5, 1e-3, A, A, A, None) == -1
    assert f(A, None, 1, -5, 1, 0.3, 0.5, 1e-3, A, A, A, None) == -1
    assert f(A, None, 1, 10, 1, 0.3, 0.5, 1e-3, A, A, None, None) == -1          # num_keep NULL
    assert f(A, None, 1, 10, 1, 0.3, 0.5, 1e-3, None, A, A, None) == -1          # out_dets NULL
    assert f(A, None, 1, 10, 1, 0.3, 0.5, 1e-3, A, None, A, None) == -1          # inds NULL
    assert f(None, None, 1, 10, 1, 0.3, 0.5, 1e-3, A, A, A, None) == -1          # dets NULL
    assert f(None, None, 0, 10, 2, 0.3, 0.5, 1e-3, None, None, None, None) == 0  # no segments: nothing to do


def test_python_surface_errors_without_gpu():
    from roi3d_b200.core.post_processing.bbox_nms import multiclass_nms_3d
    from roi3d_b200.ops import soft_nms
    from roi3d_b200.ops.nms import nms_wrapper
    with pytest.raises(ValueError, match="Invalid method for SoftNMS"):
        soft_nms(np.zeros((3, 7), np.float32), 0.3, method='hard')
    with pytest.raises(NotImplementedError):
        soft_nms(torch.zeros(3, 7), 0.3)
    with pytest.raises(NotImplementedError):
        soft_nms(np.zeros((3, 5), np.float32), 0.3)
    with pytest.raises(TypeError):
        soft_nms([[0, 0, 1, 1, 0, 1, .5]], 0.3)
    d, i = soft_nms(np.zeros((0, 7), np.float32), 0.3)
    assert d.shape == (0, 7) and d.dtype == np.float32 and i.dtype == np.int64 and i.size == 0
    d, i = soft_nms(torch.zeros(0, 7), 0.3)
    assert d.shape == (0, 7) and i.dtype == torch.long and i.numel() == 0
    assert nms_wrapper.SOFT_NMS_MAX_ROWS == 4096
    with pytest.raises(NotImplementedError):
        multiclass_nms_3d(torch.zeros(3, 12), torch.zeros(3, 2), 0.2, dict(type='nms_match', iou_thr=0.5))
    # an empty input checks nms_cfg as a non-empty one does
    with pytest.raises(ValueError, match="Invalid method for SoftNMS"):
        multiclass_nms_3d(torch.zeros(0, 12), torch.zeros(0, 2), 0.2, dict(type='soft_nms', iou_thr=0.5, method='hard'))


# instantiation -> the GPU rows (n of test_soft_nms_matches_oracle) that launch it
COVERAGE = {"soft_nms3d_kernel<1>": (1, 63, 64, 65), "soft_nms3d_kernel<2>": (2000,), "soft_nms3d_kernel<4>": (4096,)}


def kernel_for(n_max):
    return "soft_nms3d_kernel<%d>" % (1 if n_max <= 1024 else 2 if n_max <= 2048 else 4)


def test_every_instantiation_has_a_gpu_row():
    assert built_kernels("soft_nms3d") == set(COVERAGE)
    for name, ns in COVERAGE.items():
        assert ns and all(kernel_for(n) == name for n in ns)
        assert all(n in GPU_NS for n in ns)


# -------------------------------------------------------------------------------------------------- GPU tests
GPU_NS = (1, 63, 64, 65, 2000, 4096)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _inputs(kind, n, seed):
    if kind == "c1":
        return synth.c1_boxes(n, seed=seed)
    if kind == "ties":
        return tie_boxes(n, seed)
    if kind == "dense_ties":
        return dense_boxes(n, seed, levels=(0.1, 0.3, 0.6, 0.9), span=8.0 * max(n, 8) ** (1 / 3))
    return edge_boxes(n, seed)


def _check_one(d, cfg, got_d, got_i, m):
    method, thr, sigma, min_score = cfg
    want_d, want_i = soft_oracle.soft_nms3d(d, thr, method, sigma, min_score)
    assert m == want_d.shape[0], (m, want_d.shape[0])
    assert np.array_equal(got_i[:m], want_i)
    assert same_bits(got_d[:m], want_d)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: "%s-%g-%g-%g" % c)
@pytest.mark.parametrize("kind", ["c1", "ties", "dense_ties", "edge"])
@pytest.mark.parametrize("n", GPU_NS)
def test_soft_nms_matches_oracle(dev, n, kind, cfg):
    from roi3d_b200.ops import soft_nms
    d = _inputs(kind, n, seed=n + 31)
    method, thr, sigma, min_score = cfg
    t = torch.from_numpy(d).to(dev)
    res = {}

    def run():
        res["d"], res["i"] = soft_nms(t, thr, method=method, sigma=sigma, min_score=min_score)
    names = launched_kernels(run)
    assert library_kernels(names) == {kernel_for(n)}
    got_d, got_i = res["d"], res["i"]
    assert got_d.device == t.device and got_d.dtype == torch.float32 and got_i.dtype == torch.int64
    _check_one(d, cfg, got_d.cpu().numpy(), got_i.cpu().numpy(), got_d.shape[0])


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [CONFIGS[1], CONFIGS[4]], ids=["linear", "gaussian"])
def test_many_segments_unequal_counts(dev, cfg):
    from roi3d_b200.ops.nms import nms_wrapper
    rng = np.random.default_rng(5)
    nseg, n_max = 70, 300
    counts = rng.integers(0, n_max + 1, nseg).astype(np.int32)
    counts[[0, 9, 33]] = 0
    counts[[1, 50]] = n_max
    counts[2] = 1
    segs = [(_inputs(("c1", "ties", "dense_ties", "edge")[s % 4], n_max, seed=100 + s)) for s in range(nseg)]
    dets = np.stack(segs)
    for s in range(nseg):
        dets[s, counts[s]:] = np.float32(1e9)     # rows past the count must be ignored
    res = {}

    def run():
        res["r"] = nms_wrapper.soft_nms3d_batched(torch.from_numpy(dets).to(dev), torch.from_numpy(counts).to(dev),
                                                  cfg[1], cfg[0], cfg[2], cfg[3])
    assert library_kernels(launched_kernels(run)) == {"soft_nms3d_kernel<1>"}
    out, inds, num = (x.cpu().numpy() for x in res["r"])
    for s in range(nseg):
        _check_one(dets[s, :counts[s]], cfg, out[s], inds[s], int(num[s]))
    # no counts: every segment has n_max rows
    out, inds, num = (x.cpu().numpy() for x in nms_wrapper.soft_nms3d_batched(
        torch.from_numpy(dets[:5]).to(dev), None, cfg[1], cfg[0], cfg[2], cfg[3]))
    for s in range(5):
        _check_one(dets[s], cfg, out[s], inds[s], int(num[s]))


@pytest.mark.gpu
def test_ndarray_input_and_limit(dev):
    from roi3d_b200 import _lib
    from roi3d_b200.ops import soft_nms
    d = edge_boxes(500, 77)
    got_d, got_i = soft_nms(d, 0.4, 'gaussian', 0.5, 0.01)
    assert isinstance(got_d, np.ndarray) and got_d.dtype == np.float32 and got_i.dtype == np.int64
    want_d, want_i = soft_oracle.soft_nms3d(d, 0.4, 'gaussian', 0.5, 0.01)
    assert same_bits(got_d, want_d) and np.array_equal(got_i, want_i)
    with pytest.raises(_lib.Roi3dError, match="n_max"):
        soft_nms(torch.from_numpy(synth.c1_boxes(4097, seed=3)).to(dev), 0.3)


@pytest.mark.gpu
def test_multiclass_soft_nms_runs_the_batched_kernels_and_matches_oracle(dev):
    from roi3d_b200 import multiclass_nms_3d
    rng = np.random.default_rng(60)
    n = 400
    d = synth.c1_boxes(n, seed=61)
    s1 = d[:, 6]
    s2 = rng.choice(np.array([0.3, 0.6, 0.9], np.float32), n)
    scores = np.stack([1 - s1, s1, s2], 1).astype(np.float32)
    boxes = np.concatenate([d[:, :6] * 0, d[:, :6], d[:, :6] + 1.5], 1).astype(np.float32)
    cfgs = [dict(iou_thr=0.5, min_score=0.05), dict(iou_thr=0.3, method='gaussian', sigma=0.3, min_score=0.25)]
    for cfg in cfgs:
        for max_num in (2000, 37):
            want_b, want_l = soft_oracle.multiclass_nms_3d(boxes, scores, 0.2, cfg['iou_thr'], max_num,
                                                           **{k: v for k, v in cfg.items() if k != 'iou_thr'})
            res = {}

            def run():
                res["r"] = multiclass_nms_3d(torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev), 0.2,
                                             dict(type='soft_nms', **cfg), max_num)
            assert library_kernels(launched_kernels(run)) == {"multiclass_select_kernel", "multiclass_collect_kernel",
                                                              "multiclass_gather_kernel", "soft_nms3d_kernel<1>",
                                                              "topk_tail_kernel<false>"}
            got_b, got_l = res["r"]
            assert same_bits(got_b.cpu().numpy(), want_b)
            assert np.array_equal(got_l.cpu().numpy(), want_l)
            assert max_num != 37 or got_b.shape[0] == 37


@pytest.mark.gpu
def test_reference_config_roi_stage_with_soft_nms(dev, monkeypatch):
    """The reference-config RoI stage with test_cfg.rcnn.nms switched to soft-NMS (the standard one-key mmdet switch);
    the stage's own boxes and scores are re-run through the oracle."""
    import roi3d_b200
    import roi_stage
    cfg = dict(roi_stage.TEST_CFG_RCNN, nms=dict(type='soft_nms', iou_thr=0.5, min_score=0.05))
    monkeypatch.setattr(roi_stage, "TEST_CFG_RCNN", cfg)
    calls = []
    real = roi3d_b200.multiclass_nms_3d

    def recording(boxes, scores, score_thr, nms_cfg, max_num=-1):
        out = real(boxes, scores, score_thr, nms_cfg, max_num)
        calls.append((boxes.cpu().numpy(), scores.cpu().numpy(), score_thr, dict(nms_cfg), max_num,
                      out[0].cpu().numpy(), out[1].cpu().numpy()))
        return out
    monkeypatch.setattr(roi3d_b200, "multiclass_nms_3d", recording)
    stage = roi_stage.RoIStage(max_masks=20).to(dev)
    feats, cls, reg, metas = roi_stage.synthetic_inputs(1, vol_dhw=(32, 128, 128), device=dev)
    det, lab, _ = stage(feats, cls, reg, metas)[0]
    assert len(calls) == 1 and det.shape[0] > 0
    boxes, scores, score_thr, nms_cfg, max_num, got_b, got_l = calls[0]
    assert nms_cfg == dict(type='soft_nms', iou_thr=0.5, min_score=0.05)
    want_b, want_l = soft_oracle.multiclass_nms_3d(boxes, scores, score_thr, 0.5, max_num, min_score=0.05)
    assert same_bits(got_b, want_b) and np.array_equal(got_l, want_l)
    assert same_bits(det.cpu().numpy(), want_b)

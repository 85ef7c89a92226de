"""Mask paste at the mask head's real output size (20 x 28 x 28 logits per class) and masks in the multi-GPU gather.

GPU: `paste_masks_compact` / `get_seg_masks` / `paste_masks_device` against the scipy restatement of
skimage.transform.resize (`oracle.get_seg_masks_compact`), the size bound of `roi3d_mask_paste_select`, the C5 RoI stage
end to end, and the fused class selection against a copy of the selected channel.
CPU: argument checks of the C entries (before any CUDA call) and `gather_detections(..., local_masks=...)` over gloo."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import PKG, ROOT

MAX_VOL = 52534                 # kPasteMaxVol in csrc/mask_paste.cu (documented in include/roi3d_b200.h)
LARGEST_SHAPE = (21, 41, 61)    # the largest volume <= MAX_VOL with every axis <= 64 (52,521 voxels)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _dets(rng, n, lo_max, sz_lo, sz_hi):
    lo = np.stack([rng.uniform(0, lo_max[0], n), rng.uniform(0, lo_max[1], n), rng.uniform(0, lo_max[2], n)], 1)
    sz = rng.integers(sz_lo, sz_hi + 1, (n, 3))
    return np.stack([lo[:, 0], lo[:, 1], lo[:, 0] + sz[:, 0] - 0.3, lo[:, 1] + sz[:, 1] - 0.6, lo[:, 2],
                     lo[:, 2] + sz[:, 2] - 0.5, rng.random(n)], 1).astype(np.float32)


def _count_diff(got_m, want_m):
    total = diff = 0
    for g, w in zip(got_m, want_m):
        assert g.shape == w.shape and g.dtype == np.uint8
        total += g.size
        diff += int((g != w).sum())
    return diff, total


def _check_against_oracle(oracle, dev, logits, det, labels, scale=1.0, agnostic=False):
    from roi3d_b200.models.mask_heads import paste_masks_compact
    want_b, want_m, want_l = oracle.get_seg_masks_compact(logits, det, labels, 0.5, scale, agnostic)
    got_b, got_m, got_l = paste_masks_compact(torch.from_numpy(logits).to(dev), torch.from_numpy(det).to(dev),
                                              torch.from_numpy(labels).to(dev), 0.5, scale, agnostic)
    assert np.array_equal(got_b, want_b) and np.array_equal(got_l, want_l)
    diff, total = _count_diff(got_m, want_m)
    # float64 arithmetic in scipy's order; a voxel can only differ when its value is within an ulp of the threshold
    assert diff <= max(1, total // 100000), "%d of %d mask voxels differ" % (diff, total)
    return got_m


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("agnostic", [False, True])
@pytest.mark.parametrize("scale", [1.0, 1.5])
def test_head_size_matches_resize_restatement(oracle, dev, agnostic, scale):
    """[n, 2, 20, 28, 28] logits, boxes of 1-90 voxels per axis: anti-aliasing up to sigma 13.5 and upsampling."""
    rng = np.random.default_rng(11 + int(agnostic) + int(10 * scale))
    n = 40
    logits = (3 * rng.standard_normal((n, 2, 20, 28, 28))).astype(np.float32)
    det = _dets(rng, n, (300, 300, 100), 1, 90)
    det[:8, 2:6:3] = det[:8, 0:5:4] + rng.integers(1, 4, (8, 2))       # a few very small boxes: the widest filters
    labels = rng.integers(0, 1, n) if not agnostic else rng.integers(0, 5, n)
    _check_against_oracle(oracle, dev, logits, det, labels, scale, agnostic)


@pytest.mark.gpu
def test_largest_mask_and_length_one_axis(oracle, dev):
    from roi3d_b200 import _lib
    rng = np.random.default_rng(5)
    for shape in (LARGEST_SHAPE, (1, 28, 28), (20, 1, 28)):
        n = 6
        logits = (3 * rng.standard_normal((n, 1) + shape)).astype(np.float32)
        det = _dets(rng, n, (100, 100, 40), 1, 70)
        _check_against_oracle(oracle, dev, logits, det, np.zeros(n, np.int64), agnostic=True)
    # one voxel past the bound: rejected before any launch
    lg = torch.zeros(16, device=dev)
    box = torch.zeros(6, dtype=torch.int32, device=dev)
    off = torch.zeros(2, dtype=torch.int64, device=dev)
    out = torch.zeros(1, dtype=torch.uint8, device=dev)
    rc = _lib.lib.roi3d_mask_paste_select(lg.data_ptr(), 1, 1, 1, 1, MAX_VOL + 1, None, box.data_ptr(), off.data_ptr(),
                                          0.5, out.data_ptr(), None)
    assert rc != 0 and b"exceeds 52534 voxels" in _lib.lib.roi3d_last_error()


@pytest.mark.gpu
def test_device_masks_and_fused_selection_bytes(dev):
    """paste_masks_device holds exactly paste_masks_compact's bytes; reading the class channel in place gives exactly
    the bytes of pasting a copy of the selected channels through roi3d_mask_paste."""
    from roi3d_b200 import _lib
    from roi3d_b200.models.mask_heads import paste_masks_compact, paste_masks_device
    rng = np.random.default_rng(3)
    n, ncls = 64, 4
    logits = torch.from_numpy((3 * rng.standard_normal((n, ncls, 20, 28, 28))).astype(np.float32)).to(dev)
    det = torch.from_numpy(_dets(rng, n, (400, 400, 120), 1, 60)).to(dev)
    labels = torch.from_numpy(rng.integers(0, ncls - 1, n)).to(dev)
    boxes, offsets, flat, lab = paste_masks_device(logits, det, labels, 0.5)
    cb, cm, cl = paste_masks_compact(logits, det, labels, 0.5)
    assert np.array_equal(boxes.cpu().numpy(), cb) and np.array_equal(lab.cpu().numpy(), cl)
    assert np.array_equal(flat.cpu().numpy(), np.concatenate([m.reshape(-1) for m in cm]))
    assert int(offsets[-1]) == flat.numel() and offsets.dtype == torch.int64
    sel = logits[torch.arange(n, device=dev), lab].contiguous()
    ref = torch.empty_like(flat)
    _lib.check(_lib.lib.roi3d_mask_paste(sel.data_ptr(), n, 20, 28, 28, boxes.data_ptr(), offsets.data_ptr(), 0.5,
                                         ref.data_ptr(), torch.cuda.current_stream().cuda_stream))
    assert torch.equal(ref, flat)
    # class-agnostic: channel 0 through a NULL channel pointer
    _, _, flat0, _ = paste_masks_device(logits, det, labels, 0.5, class_agnostic=True)
    sel0 = logits[:, 0].contiguous()
    _lib.check(_lib.lib.roi3d_mask_paste(sel0.data_ptr(), n, 20, 28, 28, boxes.data_ptr(), offsets.data_ptr(), 0.5,
                                         ref.data_ptr(), torch.cuda.current_stream().cuda_stream))
    assert torch.equal(ref, flat0)


@pytest.mark.gpu
def test_c5_roi_stage_masks_end_to_end(oracle, dev):
    """The C5 harness's own detections and [k, 2, 20, 28, 28] mask logits through get_seg_masks: every full-volume
    mask equals the oracle's box mask pasted into the same volume."""
    import roi_stage
    from roi3d_b200.models.mask_heads import get_seg_masks
    stage = roi_stage.RoIStage(max_masks=40).to(dev)
    D, H, W = 32, 128, 128
    feats, cls, reg, metas = roi_stage.synthetic_inputs(1, vol_dhw=(D, H, W), device=dev)
    det, lab, masks = stage(feats, cls, reg, metas)[0]
    k = masks.shape[0]
    assert k > 0 and masks.shape[1:] == (2, 20, 28, 28)
    det_m, lab_m = det[:k], lab[:k]
    segs = get_seg_masks(masks, det_m, lab_m, roi_stage.TEST_CFG_RCNN, (H, W, D), 1.0, True, 2)
    assert len(segs) == 1 and len(segs[0]) == k
    want_b, want_m, _ = oracle.get_seg_masks_compact(masks.cpu().numpy(), det_m.cpu().numpy(), lab_m.cpu().numpy(),
                                                     roi_stage.TEST_CFG_RCNN['mask_thr_binary'])
    total = diff = 0
    for got, b, m in zip(segs[0], want_b, want_m):
        want = np.zeros((D, H, W), np.uint8)
        want[b[4]:b[4] + m.shape[0], b[1]:b[1] + m.shape[1], b[0]:b[0] + m.shape[2]] = m
        assert got.shape == want.shape and got.dtype == np.uint8
        total += m.size
        diff += int((got != want).sum())
    assert diff <= max(1, total // 100000), "%d of %d mask voxels differ" % (diff, total)


# ------------------------------------------------------------------------------------------------------------- CPU
def _rc_msg(fn, *args):
    from roi3d_b200 import _lib
    rc = fn(*args)
    return rc, _lib.lib.roi3d_last_error().decode()


FAKE = 256   # a non-NULL address that is never dereferenced: every case below fails its checks before any CUDA call


@pytest.mark.parametrize("case, fragment", [
    (dict(n=-1), "n = -1"),
    (dict(C=0), "num_channels = 0"),
    (dict(C=-3), "num_channels = -3"),
    (dict(Dm=0), "Dm x Hm x Wm"),
    (dict(Wm=65, Dm=4), "longer than 64"),
    (dict(Dm=1, Hm=1, Wm=MAX_VOL + 1), "exceeds 52534 voxels"),
    (dict(Dm=64, Hm=64, Wm=64), "exceeds 52534 voxels"),
    (dict(logits=None), "logits pointer is NULL"),
    (dict(boxes=None), "boxes_dev is NULL"),
    (dict(offsets=None), "offsets_dev is NULL"),
    (dict(out=None), "out_dev is NULL"),
])
def test_paste_entries_reject_bad_arguments(case, fragment):
    from roi3d_b200 import _lib
    a = dict(logits=FAKE, n=3, C=2, Dm=20, Hm=28, Wm=28, boxes=FAKE, offsets=FAKE, out=FAKE)
    a.update(case)
    rc, msg = _rc_msg(_lib.lib.roi3d_mask_paste_select, a["logits"], a["n"], a["C"], a["Dm"], a["Hm"], a["Wm"], None,
                      a["boxes"], a["offsets"], 0.5, a["out"], None)
    assert rc != 0 and fragment in msg, msg
    if "C" not in case:
        rc, msg = _rc_msg(_lib.lib.roi3d_mask_paste, a["logits"], a["n"], a["Dm"], a["Hm"], a["Wm"], a["boxes"],
                          a["offsets"], 0.5, a["out"], None)
        assert rc != 0 and fragment in msg, msg


def test_head_size_is_within_the_bound():
    assert 20 * 28 * 28 <= MAX_VOL and np.prod(LARGEST_SHAPE) <= MAX_VOL


def _volume_masks(g, n):
    """Synthetic output of paste_masks_device for one volume of n detections."""
    lo = torch.randint(0, 50, (n, 3), generator=g)
    sz = torch.randint(1, 5, (n, 3), generator=g)
    boxes = torch.stack([lo[:, 0], lo[:, 1], lo[:, 0] + sz[:, 0] - 1, lo[:, 1] + sz[:, 1] - 1, lo[:, 2],
                         lo[:, 2] + sz[:, 2] - 1], 1).to(torch.int32)
    size = sz.prod(1)
    offsets = torch.zeros(n + 1, dtype=torch.int64)
    offsets[1:] = torch.cumsum(size, 0)
    flat = torch.randint(0, 2, (int(offsets[-1]),), generator=g).to(torch.uint8)
    return boxes, offsets, flat, torch.randint(1, 3, (n,), generator=g)


def _worker(rank, world, port, n_vol, q):
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from roi3d_b200.parallel import gather_detections, shard_indices
    mine = shard_indices(n_vol)
    g = torch.Generator().manual_seed(4321)
    counts = [int(torch.randint(0, 6, (1,), generator=g)) for _ in range(n_vol)]
    counts[0] = 0
    all_dets = [torch.rand((c, 7), generator=g) for c in counts]
    all_labels = [torch.randint(0, 3, (c,), generator=g) for c in counts]
    all_masks = [_volume_masks(g, c) for c in counts]
    out = gather_detections([all_dets[i] for i in mine], [all_labels[i] for i in mine], mine,
                            local_masks=[all_masks[i] for i in mine])
    ok = sorted(out.keys()) == list(range(n_vol))
    for i in range(n_vol):
        d, l, (b, o, f) = out[i]
        ok = ok and torch.equal(d, all_dets[i]) and torch.equal(l, all_labels[i])
        ok = ok and b.dtype == torch.int32 and o.dtype == torch.int64 and f.dtype == torch.uint8
        ok = ok and torch.equal(b, all_masks[i][0]) and torch.equal(o, all_masks[i][1]) and torch.equal(f, all_masks[i][2])
    plain = gather_detections([all_dets[i] for i in mine], [all_labels[i] for i in mine], mine)
    ok = ok and sorted(plain.keys()) == list(range(n_vol)) and all(len(v) == 2 for v in plain.values())
    ok = ok and all(torch.equal(plain[i][0], all_dets[i]) and torch.equal(plain[i][1], all_labels[i])
                    for i in range(n_vol))
    q.put((rank, bool(ok)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world, n_vol", [(2, 7), (3, 800), (2, 1)])
def test_gather_with_masks_gloo(world, n_vol):
    """Every rank receives every volume's boxes, labels and masks byte for byte: volumes without detections, ranks
    without volumes, and more than 256 volumes per rank (several rounds)."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29800 + (os.getpid() % 150) + world * 7 + n_vol % 5
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_vol, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(r for r, _ in res) == list(range(world))
    assert all(ok for _, ok in res)


def test_gather_with_masks_single_process():
    from roi3d_b200.parallel import gather_detections
    g = torch.Generator().manual_seed(1)
    m = _volume_masks(g, 3)
    out = gather_detections([torch.zeros(3, 7)], [torch.zeros(3, dtype=torch.int64)], [4], local_masks=[m])
    assert list(out.keys()) == [4] and len(out[4]) == 3 and all(a is b for a, b in zip(out[4][2], m[:3]))

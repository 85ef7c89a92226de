"""RPN proposal path (`RPNProposal3D.get_proposals`) at C4 with and without the `min_bbox_size` filter.

Workload: C4 as bench.py runs it -- 8 volumes of 512x512x160, 5 levels (1 310 720 ... 320 anchors, A = 1), logits
2 N(0, 1) and deltas 0.1 N(0, 1) from the same seed, nms_pre 2000, NMS 0.7, nms_post 1000, max_num 1000 -- at each
--min-sizes value (0 = no filter, the path bench.py times; 9.5 = the C4 test's value), eager and replayed as a CUDA
graph.  Time per call is the median of CUDA events around each of --iters calls after --warmup calls; a call ends with
its one host read, so the events span the launches and the gaps between them, as a caller sees it.  The top-k reads
the 48 MB of logits once per call; the decode gathers only the selected anchors' deltas.  Every value's proposals are
checked against tests/min_bbox_size_oracle.get_bboxes_single (shapes and scores exact, coordinates within 1e-3:
glibc's expf and CUDA's may differ in the last bit), and the graph's against the eager call's, bit for bit.  With a positive value the filter
kernel is also timed alone (CUDA events around its launch, rows restored outside the window) on 40 segments x 2000
rows (the C4 shape at nms_pre 2000) and on 8 whole level-0 segments of 1 310 720 rows (nms_pre <= 0), about half of
the rows kept.  Prints one JSON line with the device name and its power limit.

    python tools/bench_rpn_min_bbox_size.py [--iters 200] [--warmup 20] [--min-sizes 0,9.5] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "3d-multi-resolution-rcnn_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import min_bbox_size_oracle  # noqa: E402
import oracle  # noqa: E402
from roi3d_b200 import RPNProposal3D, _lib  # noqa: E402

DIMS = [(80, 128, 128), (40, 64, 64), (20, 32, 32), (10, 16, 16), (5, 8, 8)]
STRIDES, DSTRIDES = [4, 8, 16, 32, 64], [2, 4, 8, 16, 32]
IMG = (512, 512, 3, 160)
BV = 8


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def time_calls(call, iters, warmup):
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record()
        call()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) * 1e3 for a, b in ev]))


def check_oracle(props, cls, reg, cfg):
    anchors = [oracle.grid_anchors(oracle.gen_base_anchors(s, [2], [2], [1.0], ds), d, s, ds)
               for d, s, ds in zip(DIMS, STRIDES, DSTRIDES)]
    for b in range(BV):
        sc = [c[b].permute(2, 3, 1, 0).reshape(-1).sigmoid().cpu().numpy() for c in cls]
        want = min_bbox_size_oracle.get_bboxes_single(
            [c[b].cpu().numpy() for c in cls], [r[b].cpu().numpy() for r in reg], anchors, IMG, cfg['nms_pre'],
            cfg['nms_post'], cfg['max_num'], cfg['nms_thr'], scores=sc, min_bbox_size=cfg['min_bbox_size'])
        g = props[b].cpu().numpy()
        assert g.shape == want.shape, (b, g.shape, want.shape)
        assert np.array_equal(g[:, 6], want[:, 6]) and np.abs(g[:, :6] - want[:, :6]).max(initial=0) <= 1e-3, b


def filter_alone(m, nseg, k, iters, warmup, dev):
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    src = torch.rand((nseg, k, 7), device=dev, generator=gen) * 400
    src[..., 2:4] = src[..., 0:2] + torch.rand((nseg, k, 2), device=dev, generator=gen) * (2.8 * m) - 1
    dets = src.clone()
    cin = torch.full((nseg,), k, dtype=torch.int32, device=dev)
    cout = torch.empty_like(cin)
    stream = torch.cuda.current_stream().cuda_stream
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters + warmup)]
    for a, b in ev:
        dets.copy_(src)
        a.record()
        _lib.check(_lib.lib.roi3d_filter_min_size_rows7(dets.data_ptr(), nseg, k, cin.data_ptr(), m, cout.data_ptr(),
                                                        stream))
        b.record()
    torch.cuda.synchronize()
    us = float(np.median([a.elapsed_time(b) * 1e3 for a, b in ev[warmup:]]))
    return dict(nseg=nseg, rows=k, kept_fraction=round(float(cout.sum()) / (nseg * k), 3), kernel_us=round(us, 1))


def run(m, cls, reg, iters, warmup):
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0], anchor_strides=STRIDES,
                         anchor_strides_depth=DSTRIDES)
    cfg = dict(nms_pre=2000, nms_post=1000, max_num=1000, nms_thr=0.7, min_bbox_size=m, nms_across_levels=False)
    metas = [dict(img_shape=IMG, scale_factor=1.0)] * BV
    call = lambda: head.get_proposals(cls, reg, metas, cfg)  # noqa: E731
    props = call()
    check_oracle(props, cls, reg, cfg)
    eager_us = time_calls(call, iters, warmup)
    head.cuda_graph = True
    graph_us = time_calls(call, iters, warmup)
    props_g = call()
    assert all(torch.equal(a, b) for a, b in zip(props, props_g)), "graph replay differs from the eager call"
    out = dict(min_bbox_size=m, eager_us=round(eager_us, 1), cuda_graph_us=round(graph_us, 1),
               proposals_out=[int(p.shape[0]) for p in props], matches_oracle=True)
    if m > 0:
        out["filter_kernel_alone"] = [filter_alone(m, n, k, iters, warmup, cls[0].device)
                                      for n, k in ((40, 2000), (8, 1310720))]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--min-sizes", default="0,9.5")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_rpn_min_bbox_size.py needs a CUDA device"
    dev = torch.device("cuda:0")
    oracle.build()
    gen = torch.Generator(device=dev)
    gen.manual_seed(6)   # bench.py's C4 draw
    cls = [2 * torch.randn((BV, 1) + d, device=dev, generator=gen) for d in DIMS]
    reg = [0.1 * torch.randn((BV, 6) + d, device=dev, generator=gen) for d in DIMS]
    res = dict(device=torch.cuda.get_device_name(dev), power_limit=power_limit(), iters=a.iters, warmup=a.warmup,
               results=[run(float(m), cls, reg, a.iters, a.warmup) for m in a.min_sizes.split(",")])
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""3D soft-NMS (roi3d_soft_nms3d_batched) device time, with the single-threaded C oracle on the same inputs beside it.

Workloads:
  c1_2000_linear / c1_2000_gaussian  one segment of 2000 C1 boxes (synth.c1_boxes), iou_thr 0.3, min_score 1e-3
  stage_2x2000                       the RoI-stage shape: 2 classes x 2000 rows, linear, iou_thr 0.5, min_score 0.05
  seg64x300                          64 segments x 300 C1 rows, linear, iou_thr 0.3, min_score 1e-3
Soft-NMS is a chain of dependent selection steps, so its cost is latency per step; the inputs (at most 2 x 2000 rows)
sit in L2 after the first call, which is where a caller's freshly written detections are too.  Device time is the
median of CUDA events around each of --iters calls after --warmup calls; "us_per_step" divides it by the longest
segment's step count (its num_keep), the chain the launch waits for.  Every workload's output is checked against the
oracle bit for bit.  Prints one JSON line with the device name and its power limit.

    python tools/bench_soft_nms.py [--iters 200] [--warmup 20] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "3d-multi-resolution-rcnn_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import soft_nms_oracle  # noqa: E402
import synth  # noqa: E402
from roi3d_b200.ops.nms import nms_wrapper  # noqa: E402

WORKLOADS = {
    # name: (segments [nseg, n_max, 7], method, iou_thr, sigma, min_score)
    "c1_2000_linear": (lambda: synth.c1_boxes(2000, seed=0)[None], 'linear', 0.3, 0.5, 1e-3),
    "c1_2000_gaussian": (lambda: synth.c1_boxes(2000, seed=0)[None], 'gaussian', 0.3, 0.5, 1e-3),
    "stage_2x2000": (lambda: np.stack([synth.c1_boxes(2000, seed=1), synth.c1_boxes(2000, seed=2)]), 'linear', 0.5,
                     0.5, 0.05),
    "seg64x300": (lambda: np.stack([synth.c1_boxes(300, seed=10 + s) for s in range(64)]), 'linear', 0.3, 0.5, 1e-3),
}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run(name, iters, warmup, dev):
    make, method, thr, sigma, min_score = WORKLOADS[name]
    segs = make().astype(np.float32)
    d = torch.from_numpy(segs).to(dev)
    call = lambda: nms_wrapper.soft_nms3d_batched(d, None, thr, method, sigma, min_score)  # noqa: E731
    for _ in range(warmup):
        call()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record()
        call()
        b.record()
    torch.cuda.synchronize()
    dev_us = float(np.median([a.elapsed_time(b) * 1e3 for a, b in ev]))
    out, inds, num = (x.cpu().numpy() for x in call())
    t0 = time.perf_counter()
    want = [soft_nms_oracle.soft_nms3d(s, thr, method, sigma, min_score) for s in segs]
    oracle_us = (time.perf_counter() - t0) * 1e6
    for s, (wd, wi) in enumerate(want):
        m = int(num[s])
        assert m == wd.shape[0] and np.array_equal(inds[s, :m], wi) and out[s, :m].tobytes() == wd.tobytes(), \
            "%s: segment %d differs from the oracle" % (name, s)
    steps = int(num.max())
    return dict(workload=name, nseg=segs.shape[0], n_max=segs.shape[1], method=method, iou_thr=thr, sigma=sigma,
                min_score=min_score, kept=[int(x) for x in num[:4]], steps_longest=steps, device_us=round(dev_us, 1),
                us_per_step=round(dev_us / max(steps, 1), 4), oracle_cpu_us=round(oracle_us, 1), matches_oracle=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_soft_nms.py needs a CUDA device"
    dev = torch.device("cuda:0")
    soft_nms_oracle.lib()   # compiled before the timing starts; the loop itself is single-threaded C
    res = dict(device=torch.cuda.get_device_name(dev), power_limit=power_limit(), iters=a.iters, warmup=a.warmup,
               results=[run(w, a.iters, a.warmup, dev) for w in a.workloads.split(",")])
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

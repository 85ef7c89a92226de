"""Batched multiclass 3D NMS (roi3d_multiclass_nms3d_batched) and the per-image multiclass_nms_3d loop over the same
images, and the fixed-shape RoI stage captured as one CUDA graph against RoIStage.forward.

NMS workloads (score_thr 0.2, NMS iou_thr 0.5 as in the reference config's test_cfg.rcnn):
  b{B}_n1000_c2    B images of 1000 rows, 2 classes (background + 1), class-specific boxes, max_num 2000 (max_per_img)
  b8_n1000_c3_m37  8 images of 1000 rows, 3 classes, max_num 37 (the cut is reached)
  b1_n3000_c3_all  1 image of 3000 rows, 3 classes, max_num -1 (the reference's default): the cut sorts all
                   (C - 1) * n = 6000 rows, more than the 4096 the top-k's one-launch tail path takes
Boxes are C1 clusters (synth.c1_boxes), class scores uniform in [0, 1), so about 80 % of the rows pass the threshold.
Three ways per workload, each timed with a host clock around the call and a device synchronise, median over --iters
calls after --warmup:
  per_image_loop  multiclass_nms_3d on each image (one host read per image, as tests/roi_stage.py does)
  batched_eager   one multiclass_nms_3d_batched call
  batched_graph   the same call captured once in a CUDA graph and replayed
The per-image and the batched results are first checked bit for bit against the CPU oracle (oracle.multiclass_nms_3d).

Stage: 512 x 512 x 160 volume, B = 1, the reference config (tests/roi_stage.py): RoIStage.forward (eager, host reads)
and the fixed-shape stage of tests/test_multiclass_nms_batched.py (proposals to mask head) replayed as one CUDA graph.
Prints one JSON line with the device name and its power limit.

    python tools/bench_multiclass_nms_batched.py [--iters 200] [--warmup 20] [--out result.json]
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

import oracle  # noqa: E402
import roi_stage  # noqa: E402
import synth  # noqa: E402
from roi3d_b200 import multiclass_nms_3d, multiclass_nms_3d_batched  # noqa: E402
from test_multiclass_nms_batched import fixed_shape_stage  # noqa: E402

NMS = dict(type='nms', iou_thr=0.5)
SCORE_THR = 0.2
WORKLOADS = {
    # name: (B, n, C, max_num)
    "b1_n1000_c2": (1, 1000, 2, 2000),
    "b8_n1000_c2": (8, 1000, 2, 2000),
    "b8_n1000_c3_m37": (8, 1000, 3, 37),
    "b1_n3000_c3_all": (1, 3000, 3, -1),
}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def host_ms(fn, iters, warmup):
    """Median wall time of fn() followed by a device synchronise, in ms."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def graph_of(fn):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


def nms_inputs(B, n, C, dev, seed=0):
    rng = np.random.default_rng(seed)
    boxes = np.empty((B, n, 6 * C), np.float32)
    scores = np.empty((B, n, C), np.float32)
    for b in range(B):
        d = synth.c1_boxes(n, seed=seed + b)
        boxes[b] = np.concatenate([d[:, :6] + np.float32(c) for c in range(C)], 1)
        scores[b] = rng.uniform(0, 1, (n, C))
    counts = np.full(B, n, np.int32)
    return tuple(torch.from_numpy(x).to(dev) for x in (boxes, scores, counts))


def run_nms(name, iters, warmup, dev):
    B, n, C, max_num = WORKLOADS[name]
    boxes, scores, counts = nms_inputs(B, n, C, dev)
    per_image = lambda: [multiclass_nms_3d(boxes[b], scores[b], SCORE_THR, NMS, max_num) for b in range(B)]  # noqa: E731
    batched = lambda: multiclass_nms_3d_batched(boxes, scores, counts, SCORE_THR, NMS, max_num)  # noqa: E731
    got = per_image()
    det, lab, cnt = (x.cpu().numpy() for x in batched())
    for b in range(B):
        wb, wl = oracle.multiclass_nms_3d(boxes[b].cpu().numpy(), scores[b].cpu().numpy(), SCORE_THR, NMS['iou_thr'],
                                          max_num)
        m = int(cnt[b])
        assert m == wb.shape[0] and det[b, :m].tobytes() == wb.tobytes() and np.array_equal(lab[b, :m], wl), \
            "%s: image %d of the batched call differs from the oracle" % (name, b)
        gb, gl = (x.cpu().numpy() for x in got[b])
        assert gb.shape == wb.shape and gb.tobytes() == wb.tobytes() and np.array_equal(gl, wl), \
            "%s: image %d of multiclass_nms_3d differs from the oracle" % (name, b)
    g, _ = graph_of(batched)
    return dict(workload=name, B=B, n=n, num_classes=C, max_num=max_num, kept=[int(x) for x in cnt[:4]],
                per_image_loop_ms=round(host_ms(per_image, iters, warmup), 4),
                batched_eager_ms=round(host_ms(batched, iters, warmup), 4),
                batched_graph_ms=round(host_ms(g.replay, iters, warmup), 4), matches_oracle=True)


def run_stage(iters, warmup, dev):
    stage = roi_stage.RoIStage().to(dev)
    feats, cls, reg, metas = roi_stage.synthetic_inputs(1, device=dev)
    with torch.no_grad():
        eager_ms = host_ms(lambda: stage(feats, cls, reg, metas), iters, warmup)
        g, out = graph_of(lambda: fixed_shape_stage(stage, feats, cls, reg, metas))
        graph_ms = host_ms(g.replay, iters, warmup)
    return dict(workload="stage_512x512x160_b1", roi_stage_forward_eager_ms=round(eager_ms, 4),
                fixed_shape_stage_graph_ms=round(graph_ms, 4), proposals=int(out['pcounts'][0]),
                detections=int(out['dcounts'][0]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_multiclass_nms_batched.py needs a CUDA device"
    dev = torch.device("cuda:0")
    res = dict(device=torch.cuda.get_device_name(dev), power_limit=power_limit(), iters=a.iters, warmup=a.warmup,
               results=[run_nms(w, a.iters, a.warmup, dev) for w in WORKLOADS] + [run_stage(a.iters, a.warmup, dev)])
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""Deterministic vs atomic RoIAlign3D / extractor backward, timed in one process.

For each case both paths run on the same seeded inputs, alternating call by call:
  atomic        roi3d_extract_backward(zero_fill=1): the library's zero-fill of the gradients + the default kernel
  deterministic roi3d_extract_backward_deterministic(accumulate=0): overwrites every voxel, no fill
Times are CUDA-event medians over --iters calls after --warmup calls.  grad_out is rotated over enough copies that
every call reads more than the L2 holds.  The outputs of the two paths are compared (max |a - b| and the tests' norm-
relative error).  Prints one JSON line with the device name and its power limit.

    python tools/bench_det_bwd.py [--iters 100] [--warmup 10] [--cases c2,c3,cfg_bbox,cfg_mask]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "3d-multi-resolution-rcnn_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from roi3d_b200 import _lib  # noqa: E402
import synth  # noqa: E402

PYR = [(40, 128, 128), (20, 64, 64), (10, 32, 32), (5, 16, 16)]
STRIDES, DSTRIDES = [4, 8, 16, 32], [2, 4, 8, 16]
CASES = {
    # name: (B, C, level dims, out (PD, PH, PW), rois)
    "c2": (1, 256, PYR[:1], (7, 7, 7), lambda: synth.c2_rois(512, seed=2)),
    "c3": (2, 256, PYR, (14, 14, 14), lambda: synth.c3_rois(512, vols=2, seed=4)),
    "cfg_bbox": (2, 64, PYR, (3, 7, 7), lambda: synth.c3_rois(512, vols=2, seed=4)),
    "cfg_mask": (2, 64, PYR, (10, 14, 14), lambda: synth.c3_rois(512, vols=2, seed=4)),
}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run_case(name, iters, warmup, dev, l2_bytes):
    B, C, dims, (PD, PH, PW), make_rois = CASES[name]
    nlev = len(dims)
    rois = torch.from_numpy(make_rois()).to(dev)
    K = rois.size(0)
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    gout_bytes = K * C * PD * PH * PW * 4
    ncopy = max(1, min(8, -(-3 * l2_bytes // gout_bytes)))
    gouts = [torch.randn((K, C, PD, PH, PW), device=dev, generator=gen) for _ in range(ncopy)]
    shapes = [(B, C) + d for d in dims]
    grads = {p: [torch.empty(s, device=dev, memory_format=torch.channels_last_3d) for s in shapes]
             for p in ("atomic", "det")}
    scales, scales_d = [1 / s for s in STRIDES[:nlev]], [1 / d for d in DSTRIDES[:nlev]]
    arrs = {p: _lib.level_array(grads[p], scales, scales_d, grads=grads[p]) for p in grads}
    st = torch.cuda.current_stream().cuda_stream

    def call(path, i):
        g = gouts[i % ncopy].data_ptr()
        if path == "atomic":
            rc = _lib.lib.roi3d_extract_backward(arrs[path], nlev, B, C, rois.data_ptr(), K, PD, PH, PW, 2, 56.0, g, 1,
                                                 0, st)
        else:
            rc = _lib.lib.roi3d_extract_backward_deterministic(arrs[path], nlev, B, C, rois.data_ptr(), K, PD, PH, PW,
                                                               2, 56.0, g, 0, st)
        _lib.check(rc)

    ev = {p: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
          for p in grads}
    for i in range(warmup):
        call("atomic", i)
        call("det", i)
    torch.cuda.synchronize()
    for i in range(iters):
        for p in ("atomic", "det") if i % 2 == 0 else ("det", "atomic"):
            ev[p][i][0].record()
            call(p, i)
            ev[p][i][1].record()
    torch.cuda.synchronize()
    med = {}
    for p in grads:
        t = sorted(a.elapsed_time(b) * 1e3 for a, b in ev[p])
        med[p] = t[len(t) // 2]
    # same inputs: the last call of each path used the same grad_out copy (iters - 1)
    maxdiff, rel = 0.0, 0.0
    for a, d in zip(grads["atomic"], grads["det"]):
        diff = float((a.double() - d.double()).abs().max())
        maxdiff = max(maxdiff, diff)
        rel = max(rel, diff / max(1.0, float(a.double().abs().max())))
    det_again = [torch.empty_like(t) for t in grads["det"]]
    arr2 = _lib.level_array(det_again, scales, scales_d, grads=det_again)
    _lib.check(_lib.lib.roi3d_extract_backward_deterministic(arr2, nlev, B, C, rois.data_ptr(), K, PD, PH, PW, 2, 56.0,
                                                             gouts[(iters - 1) % ncopy].data_ptr(), 0, st))
    torch.cuda.synchronize()
    bitwise = all(torch.equal(a, b) for a, b in zip(det_again, grads["det"]))
    return dict(case=name, B=B, C=C, levels=nlev, out=[PD, PH, PW], K=K, grad_out_copies=ncopy,
                atomic_with_fill_us=round(med["atomic"], 1), deterministic_us=round(med["det"], 1),
                det_over_atomic=round(med["det"] / med["atomic"], 3), max_abs_diff=maxdiff, rel_err=rel,
                det_repeat_bitwise=bitwise)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--cases", default=",".join(CASES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_det_bwd.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    info = _lib.device_info()
    results = [run_case(c, args.iters, args.warmup, dev, info["l2_bytes"]) for c in args.cases.split(",")]
    print(json.dumps(dict(tool="bench_det_bwd", device=torch.cuda.get_device_name(dev), power_limit=power_limit(),
                          iters=args.iters, warmup=args.warmup, results=results)))


if __name__ == "__main__":
    main()

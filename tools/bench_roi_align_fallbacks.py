"""Times every RoIAlign3D instantiation of csrc/roi_align3d.cu: the kernels that take the inputs the streamed and
planar kernels reject.  bench.py reaches none of them.

Each case is a shape a user would run, changed in one respect so that the dispatcher sends it to the kernel it names:
  ring2 / bwd2   C2 (B=1, C=256, 40x128x128 level, K=512, 7x7x7) and C3's 14-wide extractor shape (B=2, C=256, four
                 levels, K=1024, 14x14x14), through tuning variant 50 (skip the streamed and planar kernels)
  ring / bwd_cl  the same level with PD = 17 (tables wider than the CTA-shared ones), channel counts C = 255
  fwd_cl         (one channel per lane) and C = 258 (two channels per lane, no 16-byte rows)
  generic        C2 with a 5x5x4 output
7-wide kernels use the C2 level, 14-wide ones the C3 pyramid.  Before timing, each case runs once under
torch.profiler and must launch the kernel it names.  Each timed call is one launch between two CUDA events.  Before
each one a 256 MB buffer is overwritten, so no call finds the previous call's features or gradients in the 126 MB L2.
Backward calls accumulate into the gradients (zero_fill = 0), so they time the kernel without the fill.  Prints one
JSON line with the device name and power limit and the median time of each case.

    python tools/bench_roi_align_fallbacks.py [--iters 20] [--warmup 3] [--cases name,name,...]
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
from kernel_inventory import kernel_key, launched_kernels, library_kernels  # noqa: E402
import synth  # noqa: E402

C2_LEVELS = [(40, 128, 128)]
C3_LEVELS = [(40, 128, 128), (20, 64, 64), (10, 32, 32), (5, 16, 16)]
STRIDES, DSTRIDES = [4, 8, 16, 32], [2, 4, 8, 16]


def c2(direction, kernel, C=256, out=(7, 7, 7), variant=0):
    return dict(direction=direction, kernel=kernel, B=1, C=C, levels=C2_LEVELS, out=out, variant=variant,
                rois=lambda: synth.c2_rois(512, seed=2))


def c3(direction, kernel, C=256, out=(14, 14, 14), variant=0):
    return dict(direction=direction, kernel=kernel, B=2, C=C, levels=C3_LEVELS, out=out, variant=variant,
                rois=lambda: synth.c3_rois(512, vols=2, seed=4))


CASES = {
    "fwd_ring2_7_c2": c2("fwd", "roi_align3d_fwd_ring2_kernel<7,7,2,3,5,18,2,false>", variant=50),
    "fwd_ring2_14_c3": c3("fwd", "roi_align3d_fwd_ring2_kernel<14,4,2,3,3,18,0,true>", variant=50),
    "bwd2_7_c2": c2("bwd", "roi_align3d_bwd2_kernel<7,7,2,0>", variant=50),
    "bwd2_14_c3": c3("bwd", "roi_align3d_bwd2_kernel<14,2,2,4>", variant=50),
    "fwd_ring_7_c2_pd17": c2("fwd", "roi_align3d_fwd_ring_kernel<7,7,2,3,4,18,2>", out=(17, 7, 7)),
    "fwd_ring_14_c3_pd17": c3("fwd", "roi_align3d_fwd_ring_kernel<14,4,2,3,3,18,0>", out=(17, 14, 14)),
    "fwd_cl_7_1_c2_c255": c2("fwd", "roi_align3d_fwd_cl_kernel<7,7,1,3>", C=255),
    "fwd_cl_7_2_c2_c258": c2("fwd", "roi_align3d_fwd_cl_kernel<7,7,2,3>", C=258),
    "fwd_cl_14_1_c3_c255": c3("fwd", "roi_align3d_fwd_cl_kernel<14,7,1,3>", C=255),
    "fwd_cl_14_2_c3_c258": c3("fwd", "roi_align3d_fwd_cl_kernel<14,4,2,3>", C=258),
    "bwd_cl_7_1_c2_c255": c2("bwd", "roi_align3d_bwd_cl_kernel<7,7,1,40>", C=255),
    "bwd_cl_7_2_c2_pd17": c2("bwd", "roi_align3d_bwd_cl_kernel<7,7,2,26>", out=(17, 7, 7)),
    "bwd_cl_14_1_c3_c255": c3("bwd", "roi_align3d_bwd_cl_kernel<14,7,1,40>", C=255),
    "bwd_cl_14_2_c3_pd17": c3("bwd", "roi_align3d_bwd_cl_kernel<14,4,2,30>", out=(17, 14, 14)),
    "fwd_generic_2_c2_5x5x4": c2("fwd", "roi_align3d_fwd_generic_kernel<2>", out=(4, 5, 5)),
    "fwd_generic_1_c2_c255_5x5x4": c2("fwd", "roi_align3d_fwd_generic_kernel<1>", C=255, out=(4, 5, 5)),
    "bwd_generic_2_c2_5x5x4": c2("bwd", "roi_align3d_bwd_generic_kernel<2>", out=(4, 5, 5)),
    "bwd_generic_1_c2_c255_5x5x4": c2("bwd", "roi_align3d_bwd_generic_kernel<1>", C=255, out=(4, 5, 5)),
}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run_case(name, iters, warmup, dev, flush):
    cs = CASES[name]
    B, C, (PD, PH, PW) = cs["B"], cs["C"], cs["out"]
    nlev = len(cs["levels"])
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    rois = torch.from_numpy(cs["rois"]()).to(dev)
    K = rois.size(0)
    levels = [torch.randn((B, C) + d, device=dev, generator=gen).contiguous(memory_format=torch.channels_last_3d)
              for d in cs["levels"]]
    scales, scales_d = [1 / s for s in STRIDES[:nlev]], [1 / d for d in DSTRIDES[:nlev]]
    st = torch.cuda.current_stream().cuda_stream
    key = 0 if cs["direction"] == "fwd" else 1
    if cs["direction"] == "fwd":
        out = torch.empty((K, C, PD, PH, PW), device=dev)
        arr = _lib.level_array(levels, scales, scales_d)

        def call():
            _lib.check(_lib.lib.roi3d_extract_forward(arr, nlev, B, C, rois.data_ptr(), K, PD, PH, PW, 2, 56.0,
                                                      out.data_ptr(), None, st))
    else:
        gout = torch.randn((K, C, PD, PH, PW), device=dev, generator=gen)
        arr = _lib.level_array(levels, scales, scales_d, grads=levels)

        def call():
            _lib.check(_lib.lib.roi3d_extract_backward(arr, nlev, B, C, rois.data_ptr(), K, PD, PH, PW, 2, 56.0,
                                                       gout.data_ptr(), 0, 0, st))
    _lib.set_tuning(key, cs["variant"])
    try:
        ran = library_kernels(launched_kernels(call))
        assert kernel_key(cs["kernel"]) in ran, "%s: expected %s, launched %s" % (name, cs["kernel"], sorted(ran))
        for _ in range(warmup):
            call()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in ev:
            flush.zero_()
            a.record()
            call()
            b.record()
        torch.cuda.synchronize()
    finally:
        _lib.set_tuning(key, 0)
    t = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    return dict(case=name, kernel=cs["kernel"], B=B, C=C, levels=nlev, out=[PD, PH, PW], K=K,
                median_us=round(t[len(t) // 2], 1), min_us=round(t[0], 1), max_us=round(t[-1], 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cases", default=",".join(CASES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_roi_align_fallbacks.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    flush = torch.empty(64 << 20, device=dev)  # 256 MB, twice the L2
    results = []
    for c in args.cases.split(","):
        results.append(run_case(c, args.iters, args.warmup, dev, flush))
        torch.cuda.empty_cache()
    print(json.dumps(dict(tool="bench_roi_align_fallbacks", device=torch.cuda.get_device_name(dev),
                          power_limit=power_limit(), iters=args.iters, warmup=args.warmup, l2_flush_mb=256,
                          results=results)))


if __name__ == "__main__":
    main()

"""Mask paste at the mask head's output size (20 x 28 x 28 logits, two classes) on the B200.

Reports the card and its power limit; the CUDA-event device time of one `roi3d_mask_paste_select` launch for
n = 100 and n = 2000 detections with boxes at microbleed scale (2-12 voxels in x and y, 1-6 slices), alone and with a
tail of large boxes (up to 120 x 120 x 40); the wall time of `paste_masks_compact` including the read-back; the scipy
restatement (`oracle.get_seg_masks_compact`) on the host for a sample, with the host's core count; and how many mask
voxels differ from it.  Prints one JSON object.

    python tools/bench_mask_paste.py [--iters 50] [--sample 100]
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
for p in (ROOT, os.path.join(ROOT, "3d-multi-resolution-rcnn_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def detections(rng, n, tail):
    """Microbleed-scale boxes; with `tail`, 5 % of them (at least one) are large boxes of 60-120 x 60-120 x 20-40."""
    sz = np.stack([rng.integers(2, 13, n), rng.integers(2, 13, n), rng.integers(1, 7, n)], 1)
    if tail:
        k = max(1, n // 20)
        idx = rng.choice(n, k, replace=False)
        sz[idx] = np.stack([rng.integers(60, 121, k), rng.integers(60, 121, k), rng.integers(20, 41, k)], 1)
        sz[idx[0]] = (120, 120, 40)
    lo = np.stack([rng.uniform(0, 380, n), rng.uniform(0, 380, n), rng.uniform(0, 110, n)], 1)
    return np.stack([lo[:, 0], lo[:, 1], lo[:, 0] + sz[:, 0] - 1, lo[:, 1] + sz[:, 1] - 1, lo[:, 2],
                     lo[:, 2] + sz[:, 2] - 1, rng.random(n)], 1).astype(np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--sample", type=int, default=100, help="detections the host restatement runs on")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_mask_paste.py measures on the GPU"
    import oracle
    from roi3d_b200 import _lib
    from roi3d_b200.models.mask_heads import paste_masks_compact, paste_masks_device
    dev = torch.device("cuda:0")
    name, power = card()
    res = dict(gpu=name, power_limit=power, host_cores=os.cpu_count(), mask_shape=[20, 28, 28], classes=2)
    rng = np.random.default_rng(2024)
    for n in (100, 2000):
        logits = torch.from_numpy((3 * rng.standard_normal((n, 2, 20, 28, 28))).astype(np.float32)).to(dev)
        labels = torch.zeros(n, dtype=torch.long, device=dev)
        for tail in (False, True):
            det_np = detections(rng, n, tail)
            det = torch.from_numpy(det_np).to(dev)
            boxes, offsets, out, lab = paste_masks_device(logits, det, labels, 0.5)
            stream = torch.cuda.current_stream().cuda_stream

            def launch():
                _lib.check(_lib.lib.roi3d_mask_paste_select(logits.data_ptr(), n, 2, 20, 28, 28, lab.data_ptr(),
                                                            boxes.data_ptr(), offsets.data_ptr(), 0.5, out.data_ptr(),
                                                            stream))
            for _ in range(5):
                launch()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            times = []
            for _ in range(args.iters):
                e0.record()
                launch()
                e1.record()
                e1.synchronize()
                times.append(e0.elapsed_time(e1) * 1e3)
            key = "n%d_%s" % (n, "tail" if tail else "microbleed")
            res[key + "_kernel_us_median"] = float(np.median(times))
            res[key + "_kernel_us_min"] = float(np.min(times))
            res[key + "_output_voxels"] = int(offsets[-1])
            res[key + "_largest_box_voxels"] = int((offsets[1:] - offsets[:-1]).max())
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            reps = 5
            for _ in range(reps):
                got_b, got_m, _ = paste_masks_compact(logits, det, labels, 0.5)
            res[key + "_paste_masks_compact_wall_us"] = (time.perf_counter() - t0) / reps * 1e6
            k = min(args.sample, n)
            lg = logits[:k].cpu().numpy()
            t0 = time.perf_counter()
            _, want_m, _ = oracle.get_seg_masks_compact(lg, det_np[:k], np.zeros(k, np.int64), 0.5)
            res[key + "_scipy_restatement_us_for_%d" % k] = (time.perf_counter() - t0) * 1e6
            res[key + "_voxels_differing_of_%d" % k] = int(sum(int((a != b).sum()) for a, b in zip(got_m[:k], want_m)))
            res[key + "_voxels_compared"] = int(sum(m.size for m in want_m))
    print(json.dumps(res))


if __name__ == "__main__":
    main()

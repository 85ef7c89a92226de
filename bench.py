#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native 3D RoI hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): RoIs/s of 3D RoIAlign forward on workload C2 = BASELINE.json configs[1]
("3D RoIAlign fwd on one synthetic FPN P2 level 256ch x 40x128x128, 512 RoIs, 7x7x7 out, sampling_ratio 2").
One "step" = one RoIAlign3D forward over one batch of 512 RoIs.  Every rank runs the same per-GPU workload on its own
volume (weak scaling, no data-path collective: volumes are independent, SURVEY 8e); `value` = N * 512 * K / max-over-ranks
device time.  One JSON line is printed by rank 0 with, besides the contract keys:
  roofline      dominant kernel (roi_align3d_fwd_stream_kernel; its 7 us plan kernel is inside the timed step too):
                algorithmic bytes / CUDA-event time vs MEASURED_PEAKS.json, for channels-last AND for NCDHW input
  cpu_baseline  the oracle (CPU restatement of the reference; the reference has no CPU RoIAlign) on a bounded sample
  e2e           the same metric through the C-ABI host-buffer entry (pinned host NCDHW features -> H2D -> layout
                conversion -> kernel -> D2H of the pooled features), i.e. what a caller holding host tensors pays
  extra         secondary rows: NCDHW-input path, RoIAlign backward, C3 (mask branch fwd+bwd, 4 levels), C1 3D NMS
  ranks         (N > 1) per-rank median step time: every rank runs the SAME RoIs and features (same seeds), so the
                spread is the machine's, not the draw's; after the timed region the ranks also run C4 -> C5 sharded one
                volume per rank and all-gather the detections over NCCL (the path's only collective)
`--impl reference` times the reference's own algorithm on the host cores (oracle port, all threads) on the same workload.
`--dump-outputs DIR` writes what the last timed step returned (a fixed sample of it, see dump_outputs) as .npy files, so
that two builds can be compared output for output: the inputs are seeded and the same from run to run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "3d-multi-resolution-rcnn_b200")
for _p in (ROOT, PKG, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "roialign3d_fwd_rois_per_sec"
UNIT = "RoIs/s"
C2 = dict(B=1, C=256, D=40, H=128, W=128, K=512, P=7, PD=7, scale=0.25, scale_d=0.5, sample_num=2)
WORKLOAD = ("C2: RoIAlign3D fwd, FPN P2 level 256ch x 40x128x128 fp32 (671 MB, > L2 so no flush needed), 512 RoIs, "
            "7x7x7 bins, sample_num 2; features resident in HBM in torch.channels_last_3d memory format")


CONFIG = {"workload": WORKLOAD, "l2": "inputs (671 MB features + 180 MB output) exceed the 126 MB L2",
          "per_gpu": "each rank runs C2 on its own copy of the same volume and RoIs; no collective on the data path",
          "e2e_layout": "host features NCDHW-contiguous (reference layout); conversion to channels-last "
                        "runs on the device inside the timed call"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary rows (C3, NMS, backward)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none to write")
    return args


# ---------------------------------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY 8d): output write + compulsory read of the U distinct voxels touched + rois
# ---------------------------------------------------------------------------------------------------------------
def unique_voxels(rois, D, H, W, P, PD, scale, scale_d, sample_num):
    """U = number of distinct (b,z,y,x) voxels the RoI set samples (host arithmetic in float32, same formulas as
    the kernel; used only to count bytes)."""
    f32 = np.float32
    touched = {}

    def axis(c1, c2, s, Pn, size):
        start = f32(c1) * f32(s)
        sz = max(f32(f32(c2) + f32(1)) * f32(s) - start, f32(0))
        b = f32(sz) / f32(Pn)
        S = sample_num if sample_num > 0 else int(np.ceil(b))
        m = np.zeros(size, bool)
        for p in range(Pn):
            for i in range(S):
                c = f32(start + f32(p) * b) + f32(f32(i + 0.5) * b) / f32(S)
                if c < -1.0 or c > size:
                    continue
                c = max(c, f32(0))
                lo = int(c)
                if lo >= size - 1:
                    lo = hi = size - 1
                else:
                    hi = lo + 1
                m[lo] = m[hi] = True
        return m

    for r in rois:
        b = int(r[0])
        vol = touched.setdefault(b, np.zeros((D, H, W), bool))
        mx, my, mz = axis(r[1], r[3], scale, P, W), axis(r[2], r[4], scale, P, H), axis(r[5], r[6], scale_d, PD, D)
        zs, ys, xs = np.nonzero(mz)[0], np.nonzero(my)[0], np.nonzero(mx)[0]
        if len(zs) and len(ys) and len(xs):
            vol[zs[0]:zs[-1] + 1, ys[0]:ys[-1] + 1, xs[0]:xs[-1] + 1] |= (mz[zs[0]:zs[-1] + 1, None, None] &
                                                                       my[None, ys[0]:ys[-1] + 1, None] &
                                                                       mx[None, None, xs[0]:xs[-1] + 1])
    return int(sum(int(v.sum()) for v in touched.values()))


# ---------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 8:
                self.rows.append((time.time(), parts))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [p for (t, p) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [p for (_t, p) in self.rows]
        if not rows:
            return None
        sm, mx, reasons = [], [], set()
        for p in rows:
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
def c2_inputs(torch, dev, rank):
    import synth
    g = torch.Generator(device=dev)
    g.manual_seed(1)   # the same volume and RoIs on every rank: the scaling curve measures the machine, not the draw
    feats = torch.randn((C2["B"], C2["C"], C2["D"], C2["H"], C2["W"]), device=dev, generator=g)
    feats_cl = feats.contiguous(memory_format=torch.channels_last_3d)
    rois_np = synth.c2_rois(C2["K"], seed=2)
    return feats, feats_cl, rois_np


DUMP_ROIS = 128   # of the 512 RoIs of a step: 128 x 256 x 7^3 fp32 = 45 MB


def dump_outputs(torch, out_dir, out):
    """The step returns the pooled features [512, 256, 7, 7, 7] fp32 (180 MB).  Writes those of a fixed, seeded
    sample of DUMP_ROIS RoIs, all channels, in ascending RoI order, as out_dir/roi_align3d_out.npy."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(out.shape[0], DUMP_ROIS, replace=False))
    sample = out.index_select(0, torch.from_numpy(idx).to(out.device))
    np.save(os.path.join(out_dir, "roi_align3d_out.npy"), sample.cpu().numpy())


def time_steps(torch, fn, steps, warmup, dist=None):
    """W warm-ups, then K steps bracketed by barrier + synchronize; device time by CUDA events on the launching
    stream; returns (total_ms max over ranks, per-step list of this rank)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for i in range(steps):
        fn()
        evs[i + 1].record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    total = evs[0].elapsed_time(evs[-1])
    per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
    if dist is not None:
        t = torch.tensor([total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    return total, per


def run_reference(args):
    """--impl reference: the reference's algorithm on the host cores.  The reference has no CPU RoIAlign
    (functions/roi_align_3d.py:36-37 raises NotImplementedError), so this is the oracle port (kind "port") with every
    host thread, on the same workload; each step is a bounded sample of the 512 RoIs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    import synth
    oracle.build()
    oracle.set_num_threads(os.cpu_count() or 1)  # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
    rng = np.random.default_rng(1)
    feats = rng.standard_normal((C2["B"], C2["C"], C2["D"], C2["H"], C2["W"]), dtype=np.float32)
    rois = synth.c2_rois(C2["K"], seed=2)
    cores = oracle.num_threads()
    # size the per-step sample so a step takes ~1 s
    t0 = time.perf_counter()
    oracle.roi_align3d_forward(feats, rois[:8], C2["P"], C2["PD"], C2["scale"], C2["scale_d"], C2["sample_num"])
    t8 = max(time.perf_counter() - t0, 1e-4)
    n = int(min(C2["K"], max(8, 8 * round(1.0 / t8))))
    # --steps / --warmup are honoured as given; the per-step sample (n RoIs, ~1 s of CPU work) keeps the run bounded
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    budget_steps = max(1, int(150.0 / max(t8 * n / 8.0, 1e-3)))   # never more than ~150 s of CPU work in total
    if steps + warmup > budget_steps:
        n = int(max(8, n * budget_steps // (steps + warmup)))
    for _ in range(warmup):
        oracle.roi_align3d_forward(feats, rois[:n], C2["P"], C2["PD"], C2["scale"], C2["scale_d"], C2["sample_num"])
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.roi_align3d_forward(feats, rois[:n], C2["P"], C2["PD"], C2["scale"], C2["scale_d"], C2["sample_num"])
    dt = time.perf_counter() - t0
    val = n * steps / dt
    sample = "%d of the 512 C2 RoIs per step, all 256 channels, oracle C port (gcc -O2 -fopenmp)" % n
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(CONFIG, note="CPU arm: host cores only, no GPU work; each step is a bounded sample of the workload"),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    import torch
    import roi3d_b200
    from roi3d_b200 import _lib
    from roi3d_b200.ops import RoIAlign3D, nms3d_batched

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    steps, warmup = max(1, args.steps), max(3, args.warmup)

    feats, feats_cl, rois_np = c2_inputs(torch, dev, rank)
    rois = torch.from_numpy(rois_np).to(dev)
    layer = RoIAlign3D(C2["P"], C2["PD"], C2["scale"], C2["scale_d"], C2["sample_num"])
    out = layer(feats_cl, rois)  # first call: context/library load outside any timed region
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    t_wall0 = time.time()

    # ---- headline: device-resident inputs ----------------------------------------------------------------
    launches = [0]
    last_out = [None]

    def step():
        out = layer(feats_cl, rois)
        launches[0] += 1
        if launches[0] == warmup + steps:   # only the last timed step's output is kept: the others reuse one buffer
            last_out[0] = out

    total_ms, per = time_steps(torch, step, steps, warmup, dist)
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, args.dump_outputs, last_out[0])
    last_out[0] = None
    gpu_launches = 2 * steps  # per step: roi_align3d_plan_kernel (7 us) + roi_align3d_fwd_stream_kernel
    value = world * C2["K"] * steps / (total_ms * 1e-3)
    kernel_ms = float(np.median(per))  # per-step event time = plan kernel + streamed kernel (+ the launch gap)
    # ---- the dominant kernel by itself: a second region of the same K steps in which the library records a CUDA
    #      event right before and right after the launch of roi_align3d_fwd_stream_kernel (roi3d_set_kernel_timing_events;
    #      the plan kernel then no longer overlaps the main kernel's start, so these steps are not the headline's)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a_, b_ in evs:   # torch creates the cudaEvent_t at the first record
        a_.record()
        b_.record()
    torch.cuda.synchronize()
    for a_, b_ in evs:
        _lib.check(_lib.lib.roi3d_set_kernel_timing_events(a_.cuda_event, b_.cuda_event))
        layer(feats_cl, rois)
    _lib.check(_lib.lib.roi3d_set_kernel_timing_events(None, None))
    torch.cuda.synchronize()
    main_kernel_ms = float(np.median([a_.elapsed_time(b_) for a_, b_ in evs]))
    rank_us = None
    if dist is not None:  # per-rank medians: same inputs everywhere, so the spread is contention / clocks
        t = torch.tensor([kernel_ms * 1e3], device=dev, dtype=torch.float64)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        rank_us = [float(x.item()) for x in allt]

    # ---- e2e: host buffers through the C-ABI host entry ---------------------------------------------------
    e2e_steps = max(1, min(steps, 10))
    feats_h = torch.empty(feats.shape, dtype=torch.float32).pin_memory()
    feats_h.copy_(feats)  # NCDHW, the reference's layout
    rois_h = torch.from_numpy(rois_np).pin_memory()
    out_h = torch.empty(out.shape, dtype=torch.float32).pin_memory()

    def e2e_step():
        _lib.check(_lib.lib.roi3d_roi_align3d_forward_host(
            feats_h.data_ptr(), _lib.NCDHW, C2["B"], C2["C"], C2["D"], C2["H"], C2["W"], rois_h.data_ptr(), C2["K"],
            C2["PD"], C2["P"], C2["P"], C2["scale"], C2["scale_d"], C2["sample_num"], out_h.data_ptr()))

    for _ in range(2):
        e2e_step()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()  # synchronous: returns after the D2H copy completed
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_val = world * C2["K"] * e2e_steps / e2e_s
    h2d = feats_h.numel() * 4 + rois_h.numel() * 4
    d2h = out_h.numel() * 4
    # outside the timed region: the host-buffer call returns what the device-resident call computes (same kernels)
    e2e_same = bool(torch.equal(out_h, layer(feats_cl, rois).cpu()))
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None

    # ---- N > 1: BASELINE configs 4-5 sharded one volume per rank + the path's only collective --------------------
    multi = None
    if dist is not None:
        multi = sharded_stage_and_gather(torch, dist, dev, rank, world)

    # ---- secondary rows -------------------------------------------------------------------------------------
    extra = {}
    if not args.no_extra and rank == 0:
        try:
            extra = secondary_rows(torch, dev, feats, feats_cl, rois, layer, nms3d_batched, kernel_ms * 1e3)
        except Exception as e:  # secondary rows never take the headline down
            extra = {"error": repr(e)}

    if rank == 0:
        # ---- roofline of the dominant kernel -----------------------------------------------------------------
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        U = unique_voxels(rois_np, C2["D"], C2["H"], C2["W"], C2["P"], C2["PD"], C2["scale"], C2["scale_d"],
                          C2["sample_num"])
        out_bytes = C2["K"] * C2["C"] * C2["PD"] * C2["P"] * C2["P"] * 4
        alg_bytes = out_bytes + U * C2["C"] * 4 + C2["K"] * 28
        achieved = alg_bytes / (main_kernel_ms * 1e-3) / 1e9          # the dominant kernel's own launch duration
        achieved_step = alg_bytes / (kernel_ms * 1e-3) / 1e9            # the whole step (plan kernel + launch gap included)
        traffic = None
        prof = os.path.join(ROOT, "profiles", "r02_s4_c2_fwd_stream_ncu_summary.json")   # ncu --set full of this kernel
        if not os.path.exists(prof):
            prof = os.path.join(ROOT, "profiles", "r02_final_c2_fwd_stream_ncu_summary.json")
        if os.path.exists(prof):
            try:
                traffic = json.load(open(prof)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "kernel": "roi_align3d_fwd_stream_kernel<3,43008>",
                    "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes": alg_bytes, "unique_voxels": U, "kernel_us": main_kernel_ms * 1e3,
                    "kernel_timing": "CUDA events recorded by the library right before / after the kernel's launch, "
                                     "median over a second region of the same K steps",
                    "whole_step": {"step_us": kernel_ms * 1e3, "achieved": achieved_step, "frac": achieved_step / peak,
                                   "note": "one step = roi_align3d_plan_kernel + the streamed kernel (programmatic "
                                           "dependent launch) + the launch gap to the next step; this is what "
                                           "ms_per_step and value measure"},
                    "output_only_gbs": out_bytes / (main_kernel_ms * 1e-3) / 1e9,
                    "layout": "channels-last (NDHWC) features resident in HBM"}
        if extra.get("c2_fwd_ncdhw_input_us"):
            # the reference's own layout, read in place by the streamed kernel's NCDHW twin (rows of a RoI are 40-70 bytes
            # of a 512-byte feature row: DRAM moves about 1 GB for the same algorithmic bytes)
            us = extra["c2_fwd_ncdhw_input_us"]
            roofline["ncdhw_input"] = {"kernel": extra.get("c2_fwd_ncdhw_input_kernel"), "kernel_us": us,
                                       "achieved": alg_bytes / (us * 1e-6) / 1e9,
                                       "frac": alg_bytes / (us * 1e-6) / 1e9 / peak,
                                       "convert_plus_streamed_us": extra.get("c2_fwd_ncdhw_convert_plus_streamed_us"),
                                       "note": "same algorithmic bytes as the channels-last call"}
        if extra.get("c3_fwd_output_gbs"):
            # the mask branch (C3, 14^3 bins, four levels): the 2.88 GB output is 93 % of its traffic; output bytes only
            roofline["c3_mask_branch"] = {
                "kernel": "roi_align3d_fwd_planar_kernel<14,*,14>", "kernel_us": extra["c3_fwd_us"],
                "achieved_output_only": extra["c3_fwd_output_gbs"], "frac_output_only": extra["c3_fwd_output_gbs"] / peak,
                "ncdhw": {"kernel_us": extra.get("c3_fwd_ncdhw_us"),
                          "frac_output_only": (extra.get("c3_fwd_ncdhw_output_gbs") or 0.0) / peak}}
        cpu = cpu_baseline() if world == 1 else None  # reported on rank 0 at N=1 only
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": CONFIG,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": e2e_s / e2e_steps * 1e3,
                    "identical_to_device_resident_call": e2e_same},
            "gpu_launches": gpu_launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "extra": extra,
        }
        if rank_us is not None:
            line["ranks"] = {"step_us_per_rank": rank_us, "min": min(rank_us), "median": float(np.median(rank_us)),
                             "max": max(rank_us)}
        if multi is not None:
            line["multi_gpu"] = multi
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def sharded_stage_and_gather(torch, dist, dev, rank, world):
    """BASELINE configs[3] / [4] as they are stated ("8 volumes sharded over 8 B200"): every rank runs the RoI stage of
    configs/3d-multi-resolution-rcnn.py (proposal path C4 -> extractors -> heads -> multiclass NMS, C5 harness) on its
    OWN 512x512x160 volume, then the per-volume detections are all-gathered over NCCL (roi3d_b200.parallel.
    gather_detections, replacing eval_hooks.py:134-149).  Device-timed per rank, max over ranks reported; rank 0 checks
    that it received every volume and that its own volume came back bit-identical."""
    import roi_stage
    from roi3d_b200.parallel import gather_detections
    stage = roi_stage.RoIStage(max_masks=50).to(dev)
    feats5, cls5, reg5, metas5 = roi_stage.synthetic_inputs(1, device=dev, seed=7 + rank)
    out5 = stage(feats5, cls5, reg5, metas5)          # warm-up (allocations, tensor maps, cuDNN plans)
    gather_detections([out5[0][0]], [out5[0][1]], [rank])
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    out5 = stage(feats5, cls5, reg5, metas5)
    e1.record()
    allv = gather_detections([out5[0][0]], [out5[0][1]], [rank])
    e2.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) * 1e3, e1.elapsed_time(e2) * 1e3], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ok = sorted(allv.keys()) == list(range(world)) and torch.equal(allv[rank][0].to(dev), out5[0][0]) and \
        torch.equal(allv[rank][1].to(dev), out5[0][1])
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    res = {"workload": "C4 -> C5: RoI stage of the reference config, one 512x512x160 volume per rank, then the "
                       "detections all-gathered (NCCL)",
           "volumes": world, "roi_stage_us_max_over_ranks": float(t[0].item()),
           "gather_detections_us_max_over_ranks": float(t[1].item()),
           "volumes_per_sec": world / (float(t[0].item() + t[1].item()) * 1e-6),
           "detections_per_volume": [int(allv[v][0].shape[0]) for v in sorted(allv.keys())],
           "gather_reassembled_on_every_rank": bool(flag.item())}
    del stage, feats5, cls5, reg5, out5
    torch.cuda.empty_cache()
    return res


def cpu_baseline():
    """The oracle (CPU port of the reference kernel) on a bounded sample of C2, on this box's host cores."""
    import oracle
    import synth
    oracle.build()
    oracle.set_num_threads(os.cpu_count() or 1)
    rng = np.random.default_rng(1)
    feats = rng.standard_normal((C2["B"], C2["C"], C2["D"], C2["H"], C2["W"]), dtype=np.float32)
    rois = synth.c2_rois(C2["K"], seed=2)
    cores = oracle.num_threads()
    t0 = time.perf_counter()
    oracle.roi_align3d_forward(feats, rois[:8], C2["P"], C2["PD"], C2["scale"], C2["scale_d"], C2["sample_num"])
    t8 = max(time.perf_counter() - t0, 1e-4)
    n = int(min(C2["K"], max(8, 8 * round(10.0 / t8))))  # about 10 s of CPU work
    # repeat the sample until about 10 s of CPU work have been timed (a fast many-core host finishes the whole
    # workload in well under a second; one pass would be a noisy baseline)
    passes, dt = 0, 0.0
    while dt < 10.0 and passes < 64:
        t0 = time.perf_counter()
        oracle.roi_align3d_forward(feats, rois[:n], C2["P"], C2["PD"], C2["scale"], C2["scale_d"], C2["sample_num"])
        dt += time.perf_counter() - t0
        passes += 1
    return {"value": n * passes / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d of the 512 C2 RoIs (all 256 channels, full P2 level), %d passes, %.1f s" % (n, passes, dt)}


def secondary_rows(torch, dev, feats, feats_cl, rois, layer, nms3d_batched, fwd_us):
    """Other BASELINE.json configs, timed the same way (CUDA events, median of a few iterations)."""
    import roi3d_b200
    import synth
    from roi3d_b200 import SingleRoIExtractor
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def med_us(fn, iters=10, warm=2, do_flush=True):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(iters):
            if do_flush:
                flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts))

    ex = {}
    # the headline step (plan kernel + streamed kernel) captured once and replayed as a CUDA graph of 20 steps: what the
    # step costs the GPU without the host's launch gaps (the headline itself is timed through eager calls)
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                layer(feats_cl, rois)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                for _ in range(20):
                    gout = layer(feats_cl, rois)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            graph.replay()
        b.record()
        torch.cuda.synchronize()
        ex["c2_fwd_step_cuda_graph_us"] = a.elapsed_time(b) * 1e3 / 100
        ex["c2_fwd_step_cuda_graph_identical"] = bool(torch.equal(gout, layer(feats_cl, rois)))
        del graph, gout
    except Exception as e:  # measurement only: never fail the bench line over it
        ex["c2_fwd_step_cuda_graph_error"] = repr(e)
    # C2 with the reference's NCDHW-contiguous input, as a lone call: the NCDHW twin of the streamed kernel reads the tensor
    # in place (16-byte cp.async producers); the planar kernel on the same call is timed beside it (tuning variant 60)
    us = med_us(lambda: layer(feats, rois), iters=5)
    ex["c2_fwd_ncdhw_input_us"] = us
    ex["c2_fwd_ncdhw_input_rois_per_sec"] = C2["K"] / (us * 1e-6)
    ex["c2_fwd_ncdhw_input_kernel"] = "roi_align3d_fwd_stream_ncdhw_kernel<3> (native NCDHW, no conversion)"
    roi3d_b200._lib.set_tuning(0, 60)
    try:
        ex["c2_fwd_ncdhw_input_planar_kernel_us"] = med_us(lambda: layer(feats, rois), iters=5)
    finally:
        roi3d_b200._lib.set_tuning(0, 0)
    # the other route: convert to channels-last once (reusable by every extractor call of a pass, see
    # roi3d_b200.reuse_layout_conversions) + the streamed kernel; a fresh scope per call = conversion paid every time
    import roi3d_b200 as _r3

    def conv_then_stream():
        with _r3.reuse_layout_conversions():
            layer(feats, rois)
    ex["c2_fwd_ncdhw_convert_plus_streamed_us"] = med_us(conv_then_stream, iters=5)
    # C2 backward (grad of the pooled features w.r.t. the level), zero-fill of the 671 MB gradient included
    fcl = feats_cl.detach().requires_grad_(True)
    out = layer(fcl, rois)
    g = torch.randn_like(out)

    def bwd():
        fcl.grad = None
        out.backward(g, retain_graph=True)
    us = med_us(bwd, iters=5)
    ex["c2_bwd_us_incl_zero_fill"] = us
    ex["c2_fwd_us"] = fwd_us
    ex["c2_fwd_bwd_rois_per_sec"] = C2["K"] / ((us + fwd_us) * 1e-6)
    del out, g, fcl
    torch.cuda.empty_cache()
    # C1: 3D NMS, 2000 boxes, thr 0.7 (device resident, no host sync) and 40 segments batched
    dets = torch.from_numpy(synth.c1_boxes(2000, seed=0)).to(dev)
    d1 = dets[None].contiguous()
    us = med_us(lambda: nms3d_batched(d1, None, 0.7), iters=30, do_flush=False)
    ex["c1_nms2000_us"] = us
    ex["c1_nms2000_boxes_per_sec"] = 2000 / (us * 1e-6)
    ex["c1_nms2000_iou_pairs_per_sec"] = 1999000 / (us * 1e-6)
    # the same call 200 times back to back (the launch queue never runs dry: device time per NMS without the host's
    # per-call latency), and the host's own CPU time per call (python glue + ctypes + three launches)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    a.record()
    for _ in range(200):
        nms3d_batched(d1, None, 0.7)
    b.record()
    host_us = (time.perf_counter() - t0) / 200 * 1e6
    torch.cuda.synchronize()
    ex["c1_nms2000_back_to_back_us"] = a.elapsed_time(b) * 1e3 / 200
    ex["c1_nms2000_host_cpu_us_per_call"] = host_us
    d40 = dets[None].repeat(40, 1, 1).contiguous()
    us = med_us(lambda: nms3d_batched(d40, None, 0.7), iters=10, do_flush=False)
    ex["c1_nms2000_x40_batched_us"] = us
    ex["c1_nms2000_x40_boxes_per_sec"] = 40 * 2000 / (us * 1e-6)
    # C1 as BASELINE.json states it: numpy boxes through the nms wrapper (host buffers: upload, kernels, read-back),
    # beside the reference's CPU paths restated in the oracle: its only CPU 3D-IoU NMS (numpy nms_3d_python) and
    # what its wrapper really runs on CPU input, the 2-D nms_cpu on columns 0-4 (SURVEY F3)
    import oracle  # CPU baseline legs only
    from roi3d_b200.ops import nms as nms_wrapper
    dn = synth.c1_boxes(2000, seed=0)
    nms_wrapper(dn, 0.7, device_id=dev.index or 0)
    t0 = time.perf_counter()
    for _ in range(20):
        _, keep_h = nms_wrapper(dn, 0.7, device_id=dev.index or 0)
    ex["c1_nms2000_numpy_in_wrapper_us"] = (time.perf_counter() - t0) / 20 * 1e6
    t0 = time.perf_counter()
    keep_np = oracle.nms_3d_python(dn, 0.7)
    ex["c1_nms2000_cpu_numpy_3d_us"] = (time.perf_counter() - t0) * 1e6
    t0 = time.perf_counter()
    oracle.nms_cpu_2d(dn, 0.7)
    ex["c1_nms2000_cpu_reference_wrapper_2d_semantics_us"] = (time.perf_counter() - t0) * 1e6
    # the reference's own natives built by oracle/build_ref.sh (oracle/_ref), timed beside: nms_cpu.cpp (the CPU path its
    # wrapper takes for numpy input: 2-D NMS on columns 0-4, SURVEY F3) and the CUDA kernels it ships (BASELINE.md 3:
    # "the kernel to beat"; nms_3d includes its blocking D2H + host sweep)
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import ref_nms_cpu
        dt_ = torch.from_numpy(dn)
        ref_nms_cpu.nms(dt_, 0.7)
        t0 = time.perf_counter()
        for _ in range(20):
            ref_nms_cpu.nms(dt_, 0.7)
        ex["c1_nms2000_ref_nms_cpu_cpp_us"] = (time.perf_counter() - t0) / 20 * 1e6
    except Exception as e:
        ex["ref_nms_cpu_error"] = repr(e)
    try:
        import ref_nms_cuda
        import ref_roi_align_cuda
        ex["ref_gpu_nms2000_us"] = med_us(lambda: ref_nms_cuda.nms_3d(dets, 0.7), iters=20, do_flush=False)
        ref_out = torch.zeros((C2["K"], C2["C"], C2["PD"], C2["P"], C2["P"]), device=dev)
        ex["ref_gpu_c2_fwd_us"] = med_us(lambda: ref_roi_align_cuda.forward3d(
            feats, rois, C2["PD"], C2["P"], C2["P"], C2["scale"], C2["scale_d"], C2["sample_num"], ref_out), iters=5)
        ex["ref_gpu_c2_fwd_max_abs_diff_vs_ours"] = float((layer(feats_cl, rois) - ref_out).abs().max())
        gref = torch.randn_like(ref_out)
        ref_gin = torch.zeros_like(feats)
        ex["ref_gpu_c2_bwd_us_no_zero_fill"] = med_us(lambda: ref_roi_align_cuda.backward3d(
            gref, rois, C2["PD"], C2["P"], C2["P"], C2["scale"], C2["scale_d"], C2["sample_num"], ref_gin), iters=3, warm=1)
        del ref_out, gref, ref_gin
    except Exception as e:
        ex["ref_gpu_error"] = repr(e)
    ex["c1_kept"] = int(len(keep_h))
    ex["c1_kept_matches_cpu_3d_set"] = bool(np.array_equal(np.sort(keep_np), np.sort(np.asarray(keep_h))))
    del d40
    # C3: mask branch, 14^3, 4 levels with level mapping, 2 volumes x 512 RoIs, fwd + bwd
    dims = [(40, 128, 128), (20, 64, 64), (10, 32, 32), (5, 16, 16)]
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)
    pyr = [torch.randn((2, 256) + d, device=dev, generator=gen).contiguous(memory_format=torch.channels_last_3d)
           for d in dims]
    r3 = torch.from_numpy(synth.c3_rois(512, vols=2, seed=4)).to(dev)
    ext = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=14, out_size_depth=14, sample_num=2), 256,
                             [4, 8, 16, 32], [2, 4, 8, 16])
    ex["c3_level_hist"] = torch.bincount(ext.map_roi_levels(r3, 4), minlength=4).tolist()
    us_f = med_us(lambda: ext(pyr, r3), iters=5)
    ex["c3_fwd_us"] = us_f
    pyr_nc = [t.contiguous() for t in pyr]   # the reference's NCDHW layout, read natively
    us_nc = med_us(lambda: ext(pyr_nc, r3), iters=5)
    ex["c3_fwd_ncdhw_us"] = us_nc
    del pyr_nc
    for t in pyr:
        t.requires_grad_(True)
    o3 = ext(pyr, r3)
    g3 = torch.randn_like(o3)

    def bwd3():
        for t in pyr:
            t.grad = None
        o3.backward(g3, retain_graph=True)
    us_b = med_us(bwd3, iters=3, warm=1)
    ex["c3_bwd_us_incl_zero_fill"] = us_b
    ex["c3_fwd_bwd_rois_per_sec"] = 1024 / ((us_f + us_b) * 1e-6)
    ex["c3_fwd_output_gbs"] = o3.numel() * 4 / (us_f * 1e-6) / 1e9
    ex["c3_fwd_ncdhw_output_gbs"] = o3.numel() * 4 / (us_nc * 1e-6) / 1e9
    del pyr, o3, g3
    torch.cuda.empty_cache()
    # C4: RPN proposal path, 8 volumes of 512x512x160 (5 levels, A=1) on this GPU: top-k 2000 -> decode -> 3D NMS 0.7
    # -> 1000 per level -> top 1000 per volume.  Wall time of the public call (includes its one host read).
    from roi3d_b200 import RPNProposal3D
    Bv = 8
    dims4 = [(80, 128, 128), (40, 64, 64), (20, 32, 32), (10, 16, 16), (5, 8, 8)]
    gen.manual_seed(6)
    cls = [2 * torch.randn((Bv, 1) + d, device=dev, generator=gen) for d in dims4]
    reg = [0.1 * torch.randn((Bv, 6) + d, device=dev, generator=gen) for d in dims4]
    head = RPNProposal3D(anchor_scales=[2], anchor_depth_scales=[2], anchor_ratios=[1.0],
                         anchor_strides=[4, 8, 16, 32, 64], anchor_strides_depth=[2, 4, 8, 16, 32])
    cfg = dict(nms_pre=2000, nms_post=1000, max_num=1000, nms_thr=0.7, min_bbox_size=0, nms_across_levels=False)
    metas = [dict(img_shape=(512, 512, 3, 160), scale_factor=1.0)] * Bv
    props = head.get_proposals(cls, reg, metas, cfg)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        head.get_proposals(cls, reg, metas, cfg)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 5
    ex["c4_proposal_path_8vol_us"] = dt * 1e6
    ex["c4_volumes_per_sec"] = Bv / dt
    ex["c4_anchors_scored_per_sec"] = Bv * sum(int(np.prod(d)) for d in dims4) / dt
    ex["c4_proposals_out"] = [int(p.shape[0]) for p in props]
    head.cuda_graph = True   # same call with the launches captured once and replayed (stable activation buffers)
    for _ in range(2):
        head.get_proposals(cls, reg, metas, cfg)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        props_g = head.get_proposals(cls, reg, metas, cfg)
    torch.cuda.synchronize()
    ex["c4_proposal_path_8vol_cuda_graph_us"] = (time.perf_counter() - t0) / 5 * 1e6
    ex["c4_cuda_graph_identical"] = bool(all(torch.equal(a, b) for a, b in zip(props, props_g)))
    head.cuda_graph = False
    del props_g
    del cls, reg, props
    torch.cuda.empty_cache()
    # C5: RoI stage of configs/3d-multi-resolution-rcnn.py (proposals -> bbox extractor 7x7x3 -> FC head -> decode ->
    # multiclass NMS -> mask extractor 14x14x10 -> conv mask head), one 512x512x160 volume, 64-ch pyramids, random init.
    # Heads are plain torch layers (out of scope); wall time of the whole stage and of its hot-path part.
    import roi_stage
    stage = roi_stage.RoIStage(max_masks=100).to(dev)
    feats5, cls5, reg5, metas5 = roi_stage.synthetic_inputs(1, device=dev)
    stage(feats5, cls5, reg5, metas5)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        out5 = stage(feats5, cls5, reg5, metas5)
    torch.cuda.synchronize()
    ex["c5_roi_stage_1vol_us"] = (time.perf_counter() - t0) / 3 * 1e6
    ex["c5_detections"] = int(out5[0][0].shape[0])

    def hot_only():
        props5 = stage.rpn.get_proposals(cls5, reg5, metas5, roi_stage.TEST_CFG_RPN)
        rois5 = roi3d_b200.bbox2roi3D(props5)
        stage.bbox_ex(feats5[:4], rois5)
        stage.mask_ex(feats5[:4], rois5[:100].contiguous())
    hot_only()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        hot_only()
    torch.cuda.synchronize()
    ex["c5_hot_path_only_us"] = (time.perf_counter() - t0) / 3 * 1e6
    # N1 (SURVEY 8f): evaluation-time NMS, coco_utils.apply_nms: 64 volumes x 300 json detections, iou 0.1 -- host
    # lists in, host lists out (upload, one batched float64-IoU device NMS, read-back), beside the numpy reference
    import oracle  # CPU baseline leg of this row (the numpy reference restated), never on the measured path
    from roi3d_b200.core.evaluation import nms_3d_eval_batched
    vols = []
    for v in range(64):
        b = synth.c1_boxes(300, seed=100 + v)
        vols.append(b)
    nms_3d_eval_batched(vols, 0.1, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        kept = nms_3d_eval_batched(vols, 0.1, device=dev)
    dt = (time.perf_counter() - t0) / 5
    ex["n1_eval_nms_64vol_x300_us"] = dt * 1e6
    ex["n1_eval_nms_boxes_per_sec"] = 64 * 300 / dt
    ex["n1_eval_nms_kept"] = int(sum(len(k) for k in kept))
    t0 = time.perf_counter()
    ref_kept = [oracle.nms_3d_python(b.astype(np.float64), 0.1) for b in vols]
    ex["n1_eval_nms_numpy_reference_us"] = (time.perf_counter() - t0) * 1e6
    ex["n1_eval_nms_identical_to_numpy"] = bool(all(np.array_equal(a, b) for a, b in zip(kept, ref_kept)))
    # N2 (SURVEY 8f): MaxIoU assigner as the RPN uses it in training: all anchors of one 512x512x160 volume
    # (1 497 920, five levels) against 16 gts; pos 0.7 / neg 0.3 / min_pos 0.3.  Device-resident, CUDA events.
    from roi3d_b200.core.bbox import MaxIoUAssigner, bbox2delta3d
    from roi3d_b200 import AnchorGenerator3D
    anchors = []
    for (d_, h_, w_), st_, sd_ in zip(dims4, [4, 8, 16, 32, 64], [2, 4, 8, 16, 32]):
        gen_a = AnchorGenerator3D(st_, [2], [2], [1.0], sd_)
        anchors.append(gen_a.grid_anchors((d_, h_, w_), st_, sd_, device=dev))
    anchors = torch.cat(anchors, 0).contiguous()
    gsel = torch.randint(0, anchors.shape[0], (16,), generator=torch.Generator().manual_seed(9)).to(dev)
    gts = (anchors[gsel] + torch.from_numpy(np.random.default_rng(9).uniform(-2, 2, (16, 6)).astype(np.float32)).to(dev))
    gts = gts.contiguous()  # gts are jittered anchors so that all four rules fire
    assigner = MaxIoUAssigner(0.7, 0.3, 0.3, True)
    res = assigner.assign(anchors, gts)
    us = med_us(lambda: assigner.assign(anchors, gts), iters=10, do_flush=False)
    ex["n2_assign_anchors"] = int(anchors.shape[0])
    ex["n2_assign_1p5M_anchors_x16gt_us"] = us
    ex["n2_assign_pairs_per_sec"] = anchors.shape[0] * 16 / (us * 1e-6)
    ex["n2_assign_pos_neg"] = [int((res.gt_inds > 0).sum()), int((res.gt_inds == 0).sum())]

    def torch_way():  # the reference's formulation (dense matrix, two reductions, gt loop) with today's torch ops
        b1, b2 = gts, anchors
        xa, ya = torch.max(b1[:, None, 0], b2[:, 0]), torch.max(b1[:, None, 1], b2[:, 1])
        xb, yb = torch.min(b1[:, None, 2], b2[:, 2]), torch.min(b1[:, None, 3], b2[:, 3])
        za, zb = torch.max(b1[:, None, 4], b2[:, 4]), torch.min(b1[:, None, 5], b2[:, 5])
        inter = (xb - xa + 1).clamp(min=0) * (yb - ya + 1).clamp(min=0) * (zb - za + 1).clamp(min=0)
        a1 = (b1[:, 2] - b1[:, 0] + 1) * (b1[:, 3] - b1[:, 1] + 1) * (b1[:, 5] - b1[:, 4] + 1)
        a2 = (b2[:, 2] - b2[:, 0] + 1) * (b2[:, 3] - b2[:, 1] + 1) * (b2[:, 5] - b2[:, 4] + 1)
        ov = inter / (a1[:, None] + a2 - inter)
        out = ov.new_full((ov.size(1),), -1, dtype=torch.long)
        mo, am = ov.max(dim=0)
        gm, _ = ov.max(dim=1)
        out[(mo >= 0) & (mo < 0.3)] = 0
        pos = mo >= 0.7
        out[pos] = am[pos] + 1
        for i in range(ov.size(0)):
            if gm[i] >= 0.3:
                out[ov[i, :] == gm[i]] = i + 1
        return out
    ref_out = torch_way()
    ex["n2_assign_torch_formulation_us"] = med_us(torch_way, iters=3, warm=1, do_flush=False)
    ex["n2_assign_identical_to_torch_formulation"] = bool(torch.equal(ref_out, res.gt_inds))
    # N4 (SURVEY 8f): mask paste of 100 detections (14x14x10 mask logits -> box-sized binary masks), host lists out
    from roi3d_b200.models.mask_heads import paste_masks_compact
    rng4 = np.random.default_rng(4)
    n4 = 100
    lg4 = torch.from_numpy((3 * rng4.standard_normal((n4, 2, 10, 14, 14))).astype(np.float32)).to(dev)
    lo4 = np.stack([rng4.uniform(0, 400, n4), rng4.uniform(0, 400, n4), rng4.uniform(0, 120, n4)], 1)
    sz4 = np.stack([rng4.integers(4, 64, n4), rng4.integers(4, 64, n4), rng4.integers(2, 24, n4)], 1)
    det4 = np.stack([lo4[:, 0], lo4[:, 1], lo4[:, 0] + sz4[:, 0], lo4[:, 1] + sz4[:, 1], lo4[:, 2], lo4[:, 2] + sz4[:, 2],
                     rng4.random(n4)], 1).astype(np.float32)
    det4_t, lab4_t = torch.from_numpy(det4).to(dev), torch.zeros(n4, dtype=torch.long, device=dev)
    paste_masks_compact(lg4, det4_t, lab4_t, 0.5)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        _b4, m4, _l4 = paste_masks_compact(lg4, det4_t, lab4_t, 0.5)
    ex["n4_mask_paste_100det_us"] = (time.perf_counter() - t0) / 5 * 1e6
    t0 = time.perf_counter()
    _bo, mo4, _lo = oracle.get_seg_masks_compact(lg4.cpu().numpy(), det4, np.zeros(n4, np.int64), 0.5)
    ex["n4_mask_paste_scipy_restatement_us"] = (time.perf_counter() - t0) * 1e6
    ex["n4_mask_voxels_differing"] = int(sum(int((a != b).sum()) for a, b in zip(m4, mo4)))
    pos_idx = torch.nonzero(res.gt_inds > 0).squeeze(1)
    if pos_idx.numel():
        pa, pg = anchors[pos_idx].contiguous(), gts[res.gt_inds[pos_idx] - 1].contiguous()
        ex["n2_bbox2delta3d_us"] = med_us(lambda: bbox2delta3d(pa, pg), iters=10, do_flush=False)
    return ex


if __name__ == "__main__":
    main()

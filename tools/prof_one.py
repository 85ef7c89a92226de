"""Run one hot-path op a few times (for ncu).  usage: prof_one.py {c2fwd|c2bwd|c3fwd|c3bwd|nms|topk} [variant]

variant (roi3d_set_tuning key 0 / 1): forward 0 = auto, 50, 60 or 99; backward 0 = auto, 50 or 60."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "3d-multi-resolution-rcnn_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import synth  # noqa: E402
from roi3d_b200 import SingleRoIExtractor, _lib  # noqa: E402
from roi3d_b200.ops import RoIAlign3D, nms3d_batched  # noqa: E402

what = sys.argv[1]
variant = int(sys.argv[2]) if len(sys.argv) > 2 else 0
dev = torch.device("cuda:0")
reps = 3
if what in ("c2fwd", "c2bwd"):
    f = torch.randn(1, 256, 40, 128, 128, device=dev).contiguous(memory_format=torch.channels_last_3d)
    rois = torch.from_numpy(synth.c2_rois(512, seed=2)).to(dev)
    layer = RoIAlign3D(7, 7, 0.25, 0.5, 2)
    if what == "c2fwd":
        _lib.set_tuning(0, variant)
        for _ in range(reps):
            out = layer(f, rois)
    else:
        _lib.set_tuning(1, variant)
        f.requires_grad_(True)
        out = layer(f, rois)
        g = torch.randn_like(out)
        for _ in range(reps):
            f.grad = None
            out.backward(g, retain_graph=True)
elif what in ("c3fwd", "c3bwd"):
    dims = [(40, 128, 128), (20, 64, 64), (10, 32, 32), (5, 16, 16)]
    feats = [torch.randn((2, 256) + d, device=dev).contiguous(memory_format=torch.channels_last_3d) for d in dims]
    rois = torch.from_numpy(synth.c3_rois(512, vols=2, seed=4)).to(dev)
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=14, out_size_depth=14, sample_num=2), 256,
                            [4, 8, 16, 32], [2, 4, 8, 16])
    if what == "c3fwd":
        _lib.set_tuning(0, variant)
        for _ in range(reps):
            out = ex(feats, rois)
    else:
        _lib.set_tuning(1, variant)
        for t in feats:
            t.requires_grad_(True)
        out = ex(feats, rois)
        g = torch.randn_like(out)
        for _ in range(reps):
            for t in feats:
                t.grad = None
            out.backward(g, retain_graph=True)
elif what == "nms":
    dets = torch.from_numpy(synth.c1_boxes(2000, seed=0)).to(dev).unsqueeze(0).contiguous()
    for _ in range(reps):
        nms3d_batched(dets, None, 0.7)
torch.cuda.synchronize()
print("done", what)

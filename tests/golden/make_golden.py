"""Generates tests/golden/*.npz by running the REFERENCE's own CUDA kernels (oracle/_ref, built by
oracle/build_ref.sh from /root/reference with API-rename patches only) on a GPU.

    gpurun -- 'python tests/golden/make_golden.py gpurun_out/golden'      # then copy the .npz files here

The fixtures pin the CPU oracle (tests/test_golden.py) without needing a GPU or /root/reference at test time."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_nms_cuda  # noqa: E402
import ref_roi_align_cuda as ra  # noqa: E402
import synth  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else HERE
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda:0")

# ---- RoIAlign3D forward / backward ------------------------------------------------------------------------
# the features and the output gradients are not stored: synth.roi_align_ref_draws draws them again from a seed
cfgs = [("c7", 7, 7, 2), ("m14x10", 14, 10, 2), ("b7x3", 7, 3, 2), ("a5", 5, 5, 0)]
assert tuple(c[0] for c in cfgs) == synth.ROI_ALIGN_REF_TAGS
rois = np.concatenate([synth.c2_rois(10, seed=11, img=(48, 52, 14), batch=2),
                       synth.adversarial_rois((7, 13, 12), 0.25, 0.5, batch=2)], 0)
tag_rois = []
for tag, ps, pdp, sn in cfgs:
    ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
    tag_rois.append(rois[ok] if sn == 0 else rois)
feats, gouts = synth.roi_align_ref_draws([(r.shape[0], 6, pdp, ps, ps) for r, (_, ps, pdp, _) in zip(tag_rois, cfgs)])
shape = feats.shape
ft = torch.from_numpy(feats).to(dev)
pack = dict(rois=rois, spatial_scale=np.float32(0.25), spatial_scale_depth=np.float32(0.5),
            draws_sha256=np.array(synth.roi_align_ref_digest(feats, gouts)))
for (tag, ps, pdp, sn), r, g in zip(cfgs, tag_rois, gouts):
    rr = torch.from_numpy(r).to(dev)
    out = torch.zeros(r.shape[0], shape[1], pdp, ps, ps, device=dev)
    ra.forward3d(ft, rr, pdp, ps, ps, 0.25, 0.5, sn, out)
    grad = torch.zeros(shape, device=dev)
    ra.backward3d(torch.from_numpy(g).to(dev), rr, pdp, ps, ps, 0.25, 0.5, sn, grad)
    torch.cuda.synchronize()
    pack["%s_cfg" % tag] = np.array([ps, pdp, sn], np.int32)
    pack["%s_rois" % tag] = r
    pack["%s_out" % tag] = out.cpu().numpy()
    pack["%s_gin" % tag] = grad.cpu().numpy()     # NB: the reference's non-cubic top_diff index (bug_compat)
np.savez_compressed(os.path.join(out_dir, "roi_align3d_ref.npz"), **pack)

# ---- 3D NMS ------------------------------------------------------------------------------------------------
pack = {}
for tag, n, thr, seed in [("a", 300, 0.7, 1), ("b", 300, 0.3, 2), ("c", 65, 0.5, 3), ("d", 1000, 0.7, 4)]:
    dets = synth.c1_boxes(n, seed=seed)
    keep = ref_nms_cuda.nms_3d(torch.from_numpy(dets).to(dev), thr).cpu().numpy()
    pack["%s_dets" % tag] = dets
    pack["%s_thr" % tag] = np.float32(thr)
    pack["%s_keep" % tag] = keep
np.savez_compressed(os.path.join(out_dir, "nms3d_ref.npz"), **pack)
print("wrote", os.listdir(out_dir))

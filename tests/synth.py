"""Seeded synthetic inputs of BASELINE.md / SURVEY 8(d) (C1..C4), shared by tests and bench.py."""
import hashlib

import numpy as np


def c1_boxes(n=2000, seed=0, vol=(512, 512, 160)):
    """C1: clustered 3D boxes with DISTINCT scores. [n,7] fp32 (x1,y1,x2,y2,z1,z2,score)."""
    rng = np.random.default_rng(seed)
    per = 8
    ncl = (n + per - 1) // per
    W, H, D = vol
    cx, cy, cz = rng.uniform(0, W, ncl), rng.uniform(0, H, ncl), rng.uniform(0, D, ncl)
    w, h, d = rng.uniform(6, 40, ncl), rng.uniform(6, 40, ncl), rng.uniform(3, 20, ncl)
    idx = np.repeat(np.arange(ncl), per)[:n]
    jit = rng.uniform(-3, 3, (n, 3))
    sc = rng.uniform(0.9, 1.1, (n, 3))
    ccx, ccy, ccz = cx[idx] + jit[:, 0], cy[idx] + jit[:, 1], cz[idx] + jit[:, 2]
    ww, hh, dd = w[idx] * sc[:, 0], h[idx] * sc[:, 1], d[idx] * sc[:, 2]
    x1, x2 = np.clip(ccx - ww / 2, 0, W - 1), np.clip(ccx + ww / 2, 0, W - 1)
    y1, y2 = np.clip(ccy - hh / 2, 0, H - 1), np.clip(ccy + hh / 2, 0, H - 1)
    z1, z2 = np.clip(ccz - dd / 2, 0, D - 1), np.clip(ccz + dd / 2, 0, D - 1)
    scores = rng.permutation(np.linspace(0.05, 0.99, n))
    return np.stack([x1, y1, np.maximum(x2, x1), np.maximum(y2, y1), z1, np.maximum(z2, z1), scores],
                    axis=1).astype(np.float32)


def c2_rois(k=512, seed=2, img=(512, 512, 80), batch=1):
    """C2: RoIs for the P2 level (strides 4/4/2). [k,7] (b,x1,y1,x2,y2,z1,z2)."""
    rng = np.random.default_rng(seed)
    W, H, D = img
    x1, y1 = rng.uniform(0, max(W - 42, 1), k), rng.uniform(0, max(H - 42, 1), k)   # 470 at 512 px
    w, h = rng.uniform(8, 64, k), rng.uniform(8, 64, k)
    z1, d = rng.uniform(0, max(D - 20, 1), k), rng.uniform(4, 24, k)             # 60 at 80 slices
    b = rng.integers(0, batch, k).astype(np.float64)
    return np.stack([b, x1, y1, np.minimum(x1 + w, W - 1), np.minimum(y1 + h, H - 1), z1,
                     np.minimum(z1 + d, D - 1)], axis=1).astype(np.float32)


def c3_rois(k_per_vol=512, vols=2, seed=4, img=(512, 512, 80)):
    """C3: sqrt(w*h*d) log-uniform in [20, 900], w = h, d ~ w/2, so all four FPN levels are populated."""
    rng = np.random.default_rng(seed)
    W, H, D = img
    k = k_per_vol * vols
    s = np.exp(rng.uniform(np.log(20), np.log(900), k))
    # s^2 = w*w*d = w^3/2  ->  w = (2 s^2)^(1/3)
    w = np.minimum((2 * s * s) ** (1 / 3), W - 2)
    d = np.minimum(np.maximum(s * s / (w * w), 1.0), D - 2)
    x1, y1, z1 = rng.uniform(0, W - 1 - w), rng.uniform(0, H - 1 - w), rng.uniform(0, D - 1 - d)
    b = np.repeat(np.arange(vols), k_per_vol).astype(np.float64)
    return np.stack([b, x1, y1, x1 + w - 1, y1 + w - 1, z1, z1 + d - 1], axis=1).astype(np.float32)


ROI_ALIGN_REF_TAGS = ("c7", "m14x10", "b7x3", "a5")


def roi_align_ref_draws(out_shapes):
    """The random inputs of tests/golden/roi_align3d_ref.npz, drawn from one seeded stream in this order: the
    features, then one output gradient per shape.  The file does not store them (it would pass 1 MB)."""
    rng = np.random.default_rng(2024)
    feats = rng.standard_normal((2, 6, 7, 13, 12)).astype(np.float32)
    return feats, [rng.standard_normal(s).astype(np.float32) for s in out_shapes]


def roi_align_ref_digest(feats, gouts):
    """sha256 of the drawn arrays, stored beside the reference outputs as "draws_sha256"."""
    h = hashlib.sha256(feats.tobytes())
    for g in gouts:
        h.update(g.tobytes())
    return h.hexdigest()


def load_roi_align_ref(path):
    """tests/golden/roi_align3d_ref.npz with "feats" and "<tag>_gout" drawn again by roi_align_ref_draws."""
    z = dict(np.load(path))
    z["feats"], gouts = roi_align_ref_draws([z["%s_out" % t].shape for t in ROI_ALIGN_REF_TAGS])
    if roi_align_ref_digest(z["feats"], gouts) != str(z["draws_sha256"]):
        raise RuntimeError("numpy %s draws a different stream from default_rng(2024) than the one %s was made with: "
                           "its features and output gradients have to be stored again" % (np.__version__, path))
    z.update(("%s_gout" % t, g) for t, g in zip(ROI_ALIGN_REF_TAGS, gouts))
    return z


def adversarial_rois(feat_dhw, scale, scale_d, batch=1, seed=7):
    """RoIs outside the map, zero-size / inverted, single-voxel, border-straddling, whole-map."""
    D, H, W = feat_dhw
    iw, ih, idp = W / scale, H / scale, D / scale_d
    r = [
        [0, -50, -50, -10, -10, -20, -5],            # fully outside (negative)
        [0, iw + 10, ih + 10, iw + 40, ih + 40, idp + 5, idp + 20],  # fully outside (positive)
        [0, 10, 10, 9, 9, 4, 3],                      # x2 = x1 - 1: zero size
        [0, 10, 10, 10, 10, 4, 4],                    # one pixel
        [0, -8, -8, 12, 12, -4, 6],                   # straddles the low border
        [0, iw - 12, ih - 12, iw + 8, ih + 8, idp - 6, idp + 4],     # straddles the high border
        [0, 0, 0, iw - 1, ih - 1, 0, idp - 1],        # whole map
        [0, 3.25, 7.75, 41.5, 29.125, 2.5, 17.75],    # fractional
        [0, 20, 20, 5, 5, 10, 2],                     # inverted
    ]
    r = np.asarray(r, dtype=np.float32)
    rng = np.random.default_rng(seed)
    r[:, 0] = rng.integers(0, batch, r.shape[0])
    return r

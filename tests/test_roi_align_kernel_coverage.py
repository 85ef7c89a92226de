"""Every RoIAlign3D kernel instantiation, reached through the public API, checked against the oracle -- and checked to
be the kernel that actually ran.

`dispatch_fwd` / `dispatch_bwd` (csrc/roi_align3d.cu) and the planar launchers choose among about forty instantiations
by output width and squareness, PD / PH against 7 and 16, C modulo 64 / 4 / 2, the alignment of the level, gradient and
output pointers, the number of levels, K and the tuning variant.  COVERAGE maps each instantiation to the cases that
select it; every row runs under torch.profiler, asserts that its named kernel is the RoIAlign3D compute kernel that ran,
and compares the result with the oracle at the tolerances of test_gpu_parity.py.  The CPU test at the bottom lists the
instantiations in the built library, so a new one without a row fails on any machine.

Every row's RoI set holds C2-like RoIs, synth.adversarial_rois, a boundary lattice (samples exactly on -1, 0, size - 1
and size, and 1/16 voxel outside -1 and size, one axis at a time), RoIs whose batch index is out of range or fractional
and, where the level is wide enough, one RoI wider than the 40-voxel tables (the literal fallback inside the same
launch).  K is odd, so the last CTA of the per-warp kernels is partial.
"""
from collections import namedtuple

import numpy as np
import pytest

import synth
from kernel_inventory import built_kernels, kernel_key, launched_kernels, library_kernels
from test_gpu_parity import BWD_TOL, FWD_TOL, rel_err

SCALE, SCALE_D = 0.25, 0.5
STRIDES, STRIDES_D = [4, 8, 16, 32, 64], [2, 4, 8, 16, 32]
TABLE_VOXELS = 40         # RXMAX: widest footprint the per-warp / CTA tables hold
# Kernels of the library that run beside a RoIAlign3D compute kernel: the streamed kernels' planner, the planar RoI
# order pass, the deterministic backward's footprint boxes, the layout transposes and the level map.
HELPERS = ("roi_align3d_plan_kernel", "roi_align3d_order_kernel", "roi_align3d_det_boxes_kernel",
           "transpose_kernel", "transpose_r32c128_kernel", "transpose_r128c32_kernel", "map_roi_levels_kernel")


# ------------------------------------------------------------------------------------------------ kernel names
def compute_kernels(names):
    """The RoIAlign3D compute kernels among launched kernel names (library kernels other than the helpers)."""
    return sorted(k for k in library_kernels(names) if k.split("<")[0] not in HELPERS)


# ------------------------------------------------------------------------------------------------ the map
Row = namedtuple("Row", "kernel direction shape out sample_num layout offset levels variant bug_compat det k_total tag")


def row(kernel, direction, shape, out, tag, sample_num=2, layout="NDHWC", offset=None, levels=1, variant=0,
        bug_compat=False, det=False, k_total=None):
    """kernel: the instantiation as it appears in the demangled name; direction: "fwd" or "bwd"; shape: level 0 as
    (B, C, D, H, W); out: (PD, PH, PW); layout of the features; offset: None, ("feats", n) -- the level is `x[1:]` of
    a channels-last batch whose C*D*H*W = n mod 4 floats, so it starts 4n bytes past a 16-byte boundary -- or ("out" /
    "grad", n): the output / gradient buffer handed to the C ABI starts n floats past one; levels: > 1 runs
    SingleRoIExtractor on a pyramid with strides 4, 8, 16, ...; variant: roi3d_set_tuning key 0 (fwd) / 1 (bwd)."""
    return Row(kernel, direction, shape, out, sample_num, layout, offset, levels, variant, bug_compat, det, k_total, tag)


STREAM = "roi_align3d_fwd_stream_kernel<3, 43008>"
STREAM_NC = "roi_align3d_fwd_stream_ncdhw_kernel<3>"
RING2_7 = "roi_align3d_fwd_ring2_kernel<7, 7, 2, 3, 5, 18, 2, false>"
RING2_14 = "roi_align3d_fwd_ring2_kernel<14, 4, 2, 3, 3, 18, 0, true>"
RING_7 = "roi_align3d_fwd_ring_kernel<7, 7, 2, 3, 4, 18, 2>"
RING_14 = "roi_align3d_fwd_ring_kernel<14, 4, 2, 3, 3, 18, 0>"
CL_7_1 = "roi_align3d_fwd_cl_kernel<7, 7, 1, 3>"
CL_7_2 = "roi_align3d_fwd_cl_kernel<7, 7, 2, 3>"
CL_14_1 = "roi_align3d_fwd_cl_kernel<14, 7, 1, 3>"
CL_14_2 = "roi_align3d_fwd_cl_kernel<14, 4, 2, 3>"
GEN_F1, GEN_F2 = "roi_align3d_fwd_generic_kernel<1>", "roi_align3d_fwd_generic_kernel<2>"
BSTREAM = "roi_align3d_bwd_stream_kernel"
BWD2_7, BWD2_14 = "roi_align3d_bwd2_kernel<7, 7, 2, 0>", "roi_align3d_bwd2_kernel<14, 2, 2, 4>"
BCL_7_1, BCL_7_2 = "roi_align3d_bwd_cl_kernel<7, 7, 1, 40>", "roi_align3d_bwd_cl_kernel<7, 7, 2, 26>"
BCL_14_1, BCL_14_2 = "roi_align3d_bwd_cl_kernel<14, 7, 1, 40>", "roi_align3d_bwd_cl_kernel<14, 4, 2, 30>"
GEN_B1, GEN_B2 = "roi_align3d_bwd_generic_kernel<1>", "roi_align3d_bwd_generic_kernel<2>"
DET = "roi_align3d_bwd_det_kernel"


def PF(p, cl, pd):
    return "roi_align3d_fwd_planar_kernel<%d, %s, %d>" % (p, "true" if cl else "false", pd)


def PB(p, pd):
    return "roi_align3d_bwd_planar_kernel<%d, %d>" % (p, pd)


S44 = (2, 0, 8, 12, 44)    # (B, -, D, H, W) of the default level: 44 voxels wide, so the wide RoI leaves the tables
SODD = (1, 0, 7, 11, 45)   # odd D*H*W: x[1:] of a channels-last batch is 4- (C odd) or 8-byte (C = 2 mod 4) aligned
SPYR = (2, 0, 16, 32, 32)  # level 0 of the pyramids


def S(base, C):
    return (base[0], C) + base[2:]


COVERAGE = [
    # ---- forward: streamed (7 x 7 x PD <= 7, C % 64 == 0, channels-last, <= 4 levels, 16-byte aligned output)
    row(STREAM, "fwd", S(S44, 64), (7, 7, 7), "C64-7x7x7"),
    row(STREAM, "fwd", S(SPYR, 64), (3, 7, 7), "4-levels-C64-7x7x3", levels=4),
    row(STREAM_NC, "fwd", S(S44, 64), (3, 7, 7), "NCDHW-C64-7x7x3", layout="NCDHW"),
    # ---- ring2 7-wide: C % 4 == 0 and 16-byte aligned levels, PD and PH <= 16, streamed kernel not applicable
    row(RING2_7, "fwd", S(S44, 32), (7, 7, 7), "C32-7x7x7"),
    row(RING2_7, "fwd", S(S44, 32), (7, 7, 7), "C32-7x7x7-adaptive", sample_num=0),
    row(RING2_7, "fwd", S(S44, 64), (8, 7, 7), "C64-PD8-past-streamed"),
    row(RING2_7, "fwd", S(S44, 68), (7, 7, 7), "C68-ragged-64-chunk"),
    row(RING2_7, "fwd", S(S44, 32), (16, 7, 7), "C32-PD16"),
    row(RING2_7, "fwd", S(S44, 32), (7, 16, 7), "C32-PH16"),
    row(RING2_7, "fwd", S(S44, 64), (7, 7, 7), "out+1float-C64", offset=("out", 1)),
    row(RING2_7, "fwd", S(S44, 64), (7, 7, 7), "out+2floats-C64", offset=("out", 2)),
    row(RING2_7, "fwd", S(SPYR, 32), (7, 7, 7), "3-levels-C32", levels=3),
    row(RING2_7, "fwd", S(SPYR, 64), (3, 7, 7), "5-levels-C64-past-streamed-cap", levels=5),
    # ---- ring 7-wide: per-warp tables for PD or PH > 16
    row(RING_7, "fwd", S(S44, 32), (17, 7, 7), "C32-PD17"),
    row(RING_7, "fwd", S(S44, 32), (7, 17, 7), "C32-PH17"),
    row(RING_7, "fwd", S(SPYR, 32), (17, 7, 7), "3-levels-C32-PD17", levels=3),
    # ---- fwd_cl 7-wide: no ring (C % 4 != 0 or a level not 16-byte aligned)
    row(CL_7_1, "fwd", S(S44, 37), (3, 7, 7), "C37-7x7x3"),
    row(CL_7_1, "fwd", (1, 37, 12, 40, 40), (3, 7, 7), "C37-7x7x3-variant60-planar-not-applicable", variant=60),
    row(CL_7_1, "fwd", S(S44, 1), (7, 7, 7), "C1"),
    row(CL_7_1, "fwd", S(SODD, 5), (7, 7, 7), "slice-4byte-aligned-C5", offset=("feats", 1)),
    row(CL_7_1, "fwd", S(SPYR, 37), (3, 7, 7), "3-levels-C37", levels=3),
    row(CL_7_2, "fwd", S(S44, 66), (7, 7, 7), "C66"),
    row(CL_7_2, "fwd", S(S44, 2), (7, 7, 7), "C2"),
    row(CL_7_2, "fwd", S(SODD, 6), (3, 7, 7), "slice-8byte-aligned-C6", offset=("feats", 2)),
    # ---- generic: widths other than 7 and 14
    row(GEN_F2, "fwd", S(S44, 16), (4, 5, 5), "C16-5x5x4"),
    row(GEN_F2, "fwd", S(SPYR, 16), (4, 5, 5), "3-levels-C16-5x5x4", levels=3),
    row(GEN_F1, "fwd", S(S44, 15), (4, 5, 5), "C15-5x5x4"),
    # ---- 14-wide: planar (square, PD <= 16, C % 4 == 0, 16-byte aligned), else ring2 / ring / fwd_cl
    row(RING2_14, "fwd", S(S44, 32), (10, 12, 14), "C32-12x14x10-non-square"),
    row(RING2_14, "fwd", S(SPYR, 32), (10, 12, 14), "3-levels-C32-12x14x10", levels=3),
    row(RING_14, "fwd", S(S44, 16), (17, 14, 14), "C16-PD17"),
    row(RING_14, "fwd", S(S44, 16), (10, 17, 14), "C16-PH17"),
    row(CL_14_1, "fwd", S(S44, 37), (10, 14, 14), "C37-14x14x10"),
    row(CL_14_1, "fwd", S(SODD, 5), (10, 14, 14), "slice-4byte-aligned-C5", offset=("feats", 1)),
    row(CL_14_2, "fwd", S(S44, 66), (10, 14, 14), "C66-14x14x10"),
    row(CL_14_2, "fwd", S(S44, 2), (10, 14, 14), "C2-14x14x10"),
    row(CL_14_2, "fwd", S(SODD, 6), (10, 14, 14), "slice-8byte-aligned-C6", offset=("feats", 2)),
    # ---- planar forward, channels-last: automatic for 14-wide, tuning variant 60 for 7-wide (nothing else reaches it)
    row(PF(7, True, 7), "fwd", S(S44, 32), (7, 7, 7), "variant60-C32-7x7x7", variant=60),
    row(PF(7, True, 3), "fwd", S(S44, 32), (3, 7, 7), "variant60-C32-7x7x3", variant=60),
    row(PF(7, True, 0), "fwd", S(S44, 32), (5, 7, 7), "variant60-C32-7x7x5", variant=60),
    row(PF(14, True, 14), "fwd", S(S44, 16), (14, 14, 14), "C16-14x14x14"),
    row(PF(14, True, 10), "fwd", S(S44, 16), (10, 14, 14), "C16-14x14x10"),
    row(PF(14, True, 10), "fwd", S(S44, 16), (10, 14, 14), "C16-14x14x10-adaptive", sample_num=0),
    row(PF(14, True, 0), "fwd", S(S44, 8), (16, 14, 14), "C8-PD16"),
    # ---- planar forward, NCDHW read in place (the streamed twin takes 7 x 7 x PD <= 7 with C % 64 == 0)
    row(PF(7, False, 7), "fwd", S(S44, 32), (7, 7, 7), "NCDHW-C32-7x7x7", layout="NCDHW"),
    row(PF(7, False, 3), "fwd", S(S44, 32), (3, 7, 7), "NCDHW-C32-7x7x3", layout="NCDHW"),
    row(PF(7, False, 3), "fwd", S(S44, 8), (3, 7, 7), "NCDHW-K1-no-order-pass", layout="NCDHW", k_total=1),
    row(PF(7, False, 3), "fwd", S(S44, 8), (3, 7, 7), "NCDHW-K8193-no-order-pass", layout="NCDHW", k_total=8193),
    row(PF(7, False, 0), "fwd", S(S44, 24), (5, 7, 7), "NCDHW-C24-7x7x5", layout="NCDHW"),
    row(PF(7, False, 0), "fwd", S(S44, 64), (8, 7, 7), "NCDHW-C64-PD8-past-streamed", layout="NCDHW"),
    row(PF(14, False, 14), "fwd", S(S44, 8), (14, 14, 14), "NCDHW-C8-14x14x14", layout="NCDHW"),
    row(PF(14, False, 10), "fwd", S(S44, 12), (10, 14, 14), "NCDHW-C12-14x14x10", layout="NCDHW"),
    row(PF(14, False, 0), "fwd", S(S44, 8), (16, 14, 14), "NCDHW-C8-PD16", layout="NCDHW"),

    # ---- backward: streamed (7 x 7 x PD <= 7, C % 64 == 0, <= 4 levels, 8-byte aligned gradient, no bug_compat)
    row(BSTREAM, "bwd", S(S44, 64), (7, 7, 7), "C64-7x7x7"),
    row(BSTREAM, "bwd", S(S44, 64), (7, 7, 7), "grad+2floats-C64", offset=("grad", 2)),
    # ---- bwd2 7-wide: CTA-shared tables, PD and PH <= 16
    row(BWD2_7, "bwd", S(S44, 32), (7, 7, 7), "C32-7x7x7"),
    row(BWD2_7, "bwd", S(S44, 64), (8, 7, 7), "C64-PD8-past-streamed"),
    row(BWD2_7, "bwd", S(S44, 32), (16, 7, 7), "C32-PD16"),
    row(BWD2_7, "bwd", S(S44, 32), (7, 7, 7), "grad+2floats-C32", offset=("grad", 2)),
    row(BWD2_7, "bwd", S(S44, 64), (3, 7, 7), "bug-compat-C64-7x7x3", bug_compat=True),
    row(BWD2_7, "bwd", S(SPYR, 32), (7, 7, 7), "3-levels-C32", levels=3),
    row(BWD2_7, "bwd", S(SPYR, 64), (3, 7, 7), "5-levels-C64-past-streamed-cap", levels=5),
    # ---- bwd_cl 7-wide: one channel per lane (odd C, 4-byte aligned gradient) or per-warp tables (PD / PH > 16)
    row(BCL_7_1, "bwd", S(S44, 37), (3, 7, 7), "C37-7x7x3"),
    row(BCL_7_1, "bwd", S(S44, 1), (7, 7, 7), "C1"),
    row(BCL_7_1, "bwd", S(S44, 64), (7, 7, 7), "grad+1float-C64", offset=("grad", 1)),
    row(BCL_7_1, "bwd", S(S44, 37), (3, 7, 7), "bug-compat-C37-7x7x3", bug_compat=True),
    row(BCL_7_1, "bwd", S(SPYR, 37), (3, 7, 7), "3-levels-C37", levels=3),
    row(BCL_7_2, "bwd", S(S44, 32), (17, 7, 7), "C32-PD17"),
    row(BCL_7_2, "bwd", S(S44, 32), (7, 17, 7), "C32-PH17"),
    row(BCL_7_2, "bwd", S(S44, 32), (3, 17, 7), "bug-compat-C32-17x7x3", bug_compat=True),
    row(BCL_7_2, "bwd", S(S44, 66), (7, 7, 7), "variant60-C66-planar-not-applicable", variant=60),
    row(BCL_7_2, "bwd", S(SPYR, 32), (17, 7, 7), "3-levels-C32-PD17", levels=3),
    # ---- planar backward: automatic for 14-wide, tuning variant 60 for 7-wide (nothing else reaches it)
    row(PB(7, 7), "bwd", S(S44, 32), (7, 7, 7), "variant60-C32-7x7x7", variant=60),
    row(PB(7, 0), "bwd", S(S44, 32), (3, 7, 7), "variant60-C32-7x7x3", variant=60),
    row(PB(14, 14), "bwd", S(S44, 16), (14, 14, 14), "C16-14x14x14"),
    row(PB(14, 0), "bwd", S(S44, 16), (10, 14, 14), "C16-14x14x10"),
    row(PB(14, 0), "bwd", S(S44, 8), (16, 14, 14), "C8-PD16"),
    # ---- 14-wide where the planar backward does not apply
    row(BWD2_14, "bwd", S(S44, 66), (10, 14, 14), "C66-14x14x10"),
    row(BWD2_14, "bwd", S(S44, 32), (10, 12, 14), "C32-12x14x10-non-square"),
    row(BWD2_14, "bwd", S(S44, 32), (10, 14, 14), "grad+2floats-C32", offset=("grad", 2)),
    row(BWD2_14, "bwd", S(S44, 32), (10, 14, 14), "bug-compat-C32-14x14x10", bug_compat=True),
    row(BWD2_14, "bwd", S(SPYR, 32), (10, 12, 14), "3-levels-C32-12x14x10", levels=3),
    row(BCL_14_1, "bwd", S(S44, 37), (10, 14, 14), "C37-14x14x10"),
    row(BCL_14_1, "bwd", S(S44, 32), (10, 14, 14), "grad+1float-C32", offset=("grad", 1)),
    row(BCL_14_1, "bwd", S(S44, 37), (10, 14, 14), "bug-compat-C37-14x14x10", bug_compat=True),
    row(BCL_14_2, "bwd", S(S44, 16), (17, 14, 14), "C16-PD17"),
    row(BCL_14_2, "bwd", S(S44, 16), (10, 17, 14), "C16-PH17"),
    row(BCL_14_2, "bwd", S(S44, 16), (10, 17, 14), "bug-compat-C16-17x14x10", bug_compat=True),
    # ---- generic backward
    row(GEN_B2, "bwd", S(S44, 16), (4, 5, 5), "C16-5x5x4"),
    row(GEN_B2, "bwd", S(S44, 16), (4, 5, 5), "bug-compat-C16-5x5x4", bug_compat=True),
    row(GEN_B2, "bwd", S(SPYR, 16), (4, 5, 5), "3-levels-C16-5x5x4", levels=3),
    row(GEN_B1, "bwd", S(S44, 15), (4, 5, 5), "C15-5x5x4"),
    row(GEN_B1, "bwd", S(S44, 15), (3, 5, 5), "bug-compat-C15-5x5x3", bug_compat=True),
    # ---- deterministic backward (torch.use_deterministic_algorithms(True))
    row(DET, "bwd", S(S44, 32), (7, 7, 7), "C32-7x7x7", det=True),
    row(DET, "bwd", S(SPYR, 37), (3, 7, 7), "3-levels-C37", levels=3, det=True),
]


def _row_id(r):
    return "%s-%s-%s" % (r.direction, kernel_key(r.kernel), r.tag)


# ------------------------------------------------------------------------------------------------ RoI sets
def lattice_rois(dhw, out, scale, scale_d, sample_num, batch):
    """RoIs whose samples fall exactly on -1, 0, size - 1 and size of one axis, and 1/16 voxel outside -1 and size.
    With bin = S (the samples per bin) the scaled start, the bin and every sample coordinate start + p * S + i + 0.5
    are small dyadic numbers: each evaluation order computes them exactly.  The other two axes take the middle half
    of the map."""
    D, H, W = dhw
    PD, PH, PW = out
    S = sample_num if sample_num > 0 else 2           # adaptive: S = ceil(bin) = 2
    axes = [(W, scale, PW, (1, 3)), (H, scale, PH, (2, 4)), (D, scale_d, PD, (5, 6))]
    rois = []
    for a, (L, s, P, (lo, hi)) in enumerate(axes):
        n = P * S                                     # samples along the axis, one voxel apart
        for first in (-1.0, -1.0 - 1 / 16, L - n // 2, L + 1 / 16 - n // 2):
            r = np.zeros(7)
            r[0] = len(rois) % batch
            for b, (Lb, sb, _, (lob, hib)) in enumerate(axes):
                if b == a:
                    start = first - 0.5
                    r[lo], r[hi] = start / s, (start + n) / s - 1
                else:
                    r[lob], r[hib] = 0.25 * Lb / sb, 0.75 * Lb / sb
            rois.append(r)
    return np.asarray(rois, np.float32)


def _axis_coords(c1, c2, s, P, S):
    """Sample coordinates of one axis as the kernels compute them (common.cuh axis_setup / axis_coord), in float64,
    with a check that every intermediate is a float32 -- so that float32 arithmetic computes the same values."""
    vals = [np.float64(c1) * s]
    size = max((np.float64(c2) + 1) * s - vals[0], 0.0)
    vals += [size, size / P]
    start, b = vals[0], vals[2]
    coords = [start + p * b + (i + 0.5) * b / S for p in range(P) for i in range(S)]
    for v in vals + coords + [(i + 0.5) * b for i in range(S)]:
        assert np.float32(v) == v, v
    return coords


def roi_set(r, dhw, seed):
    B = r.shape[0]
    D, H, W = dhw
    img = (int(W / SCALE), int(H / SCALE), int(D / SCALE_D))
    if r.k_total == 1:
        return synth.c2_rois(1, seed=seed, img=img, batch=B)
    parts = [synth.adversarial_rois(dhw, SCALE, SCALE_D, batch=B),
             lattice_rois(dhw, r.out, SCALE, SCALE_D, r.sample_num, B)]
    bad = synth.c2_rois(4, seed=seed + 1, img=img, batch=B)
    bad[:, 0] = [-1, B, -0.5, B - 0.5]        # out of range below / above; (int) truncates the last two into range
    parts.append(bad)
    if W > TABLE_VOXELS + 2 and r.levels == 1:
        parts.append(np.array([[B - 1, 0, 0.25 * img[1], img[0] - 1, 0.75 * img[1], 0.25 * img[2], 0.75 * img[2]]],
                              np.float32))    # the whole width: wider than the tables, literal path in the same launch
    if r.levels > 1:                          # large enough for the coarsest level, reaching past every border
        parts.append(np.array([[0, -200, -200, img[0] + 200, img[1] + 200, -30, img[2] + 30]], np.float32))
    rest = sum(len(p) for p in parts)
    k = (r.k_total - rest) if r.k_total else 9
    if (k + rest) % 2 == 0 and not r.k_total:
        k += 1
    rois = np.concatenate([synth.c2_rois(k, seed=seed, img=img, batch=B)] + parts, 0)
    if r.sample_num == 0 and r.direction == "bwd":   # adaptive sampling of a zero-size RoI divides by 0 samples
        ok = (rois[:, 3] >= rois[:, 1]) & (rois[:, 4] >= rois[:, 2]) & (rois[:, 6] >= rois[:, 5])
        rois = rois[ok]
    return rois


def level_shapes(r):
    B, C, D, H, W = r.shape
    return [(B, C) + tuple(max(1, s >> l) for s in (D, H, W)) for l in range(r.levels)]


def level_scales(r):
    if r.levels == 1:
        return [SCALE], [SCALE_D]
    return [1 / s for s in STRIDES[:r.levels]], [1 / s for s in STRIDES_D[:r.levels]]


def in_batch(rois, B):
    b = rois[:, 0].astype(np.int64)       # (int) truncates toward zero, as every kernel and the reference do
    return (b >= 0) & (b < B)


def expected_forward(oracle, feats, rois, r):
    """The oracle per level; a RoI with an out-of-range batch index gives 0, or NaN where its sample count is 0 -- the
    oracle's value for the same RoI over an all-zero map (such rows are never fed to the oracle as they are: it would
    read outside the features)."""
    PD, PH, PW = r.out
    B, C = feats[0].shape[:2]
    sc, scd = level_scales(r)
    lv = oracle.map_roi_levels(rois, r.levels) if r.levels > 1 else np.zeros(len(rois), np.int64)
    inside = in_batch(rois, B)
    want = np.zeros((len(rois), C, PD, PH, PW), np.float32)
    for l, f in enumerate(feats):
        for sel, src in ((inside & (lv == l), f), (~inside & (lv == l), np.zeros_like(f[:1]))):
            if sel.any():
                rr = rois[sel].copy()
                if src is not f:
                    rr[:, 0] = 0
                want[sel] = oracle.roi_align3d_forward(src, rr, (PH, PW), PD, sc[l], scd[l], r.sample_num)
    return want


def expected_backward(oracle, g, rois, r):
    shapes = level_shapes(r)
    sc, scd = level_scales(r)
    lv = oracle.map_roi_levels(rois, r.levels) if r.levels > 1 else np.zeros(len(rois), np.int64)
    inside = in_batch(rois, shapes[0][0])
    return [oracle.roi_align3d_backward(g[inside & (lv == l)], rois[inside & (lv == l)], shp, sc[l], scd[l],
                                        r.sample_num, bug_compat=r.bug_compat) for l, shp in enumerate(shapes)]


def check_forward(got, want):
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), "NaN pattern differs from the oracle's"
    assert rel_err(np.where(nan, 0, got), np.where(nan, 0, want)) <= FWD_TOL


# ------------------------------------------------------------------------------------------------ GPU rows
@pytest.fixture(scope="module")
def dev():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _cl(x):
    import torch
    return x.contiguous(memory_format=torch.channels_last_3d)


def _device_levels(r, feats, dev):
    """Feature tensors in the row's layout; an ("feats", n) offset takes x[1:] of a channels-last batch of B + 1."""
    import torch
    if r.offset is not None and r.offset[0] == "feats":
        (f,) = feats
        C, D, H, W = f.shape[1:]
        assert C * D * H * W % 4 == r.offset[1]
        big = _cl(torch.zeros((f.shape[0] + 1,) + f.shape[1:], device=dev))
        big[1:] = torch.from_numpy(f).to(dev)
        x = big[1:]
        assert x.is_contiguous(memory_format=torch.channels_last_3d)
        assert x.data_ptr() % 16 == 4 * r.offset[1]
        return [x]
    xs = [torch.from_numpy(f).to(dev) for f in feats]
    return [_cl(x) for x in xs] if r.layout == "NDHWC" else xs


def _module(r):
    from roi3d_b200 import SingleRoIExtractor
    from roi3d_b200.ops import RoIAlign3D
    PD, PH, PW = r.out
    out_size = PH if PH == PW else (PH, PW)
    if r.levels == 1:
        layer = RoIAlign3D(out_size, PD, SCALE, SCALE_D, r.sample_num)
        return lambda xs, rt: layer(xs[0], rt)
    ex = SingleRoIExtractor(dict(type='RoIAlign3D', out_size=out_size, out_size_depth=PD, sample_num=r.sample_num),
                            r.shape[1], STRIDES[:r.levels], STRIDES_D[:r.levels])
    return lambda xs, rt: ex(xs, rt)


def _run_forward(r, xs, rt, dev):
    """(launched kernel names, output) of the row's forward call."""
    import torch
    import roi3d_b200
    from roi3d_b200._util import stream_ptr
    res = []
    if r.offset is not None and r.offset[0] == "out":
        (x,) = xs
        B, C, D, H, W = x.shape
        PD, PH, PW = r.out
        K, n, off = rt.shape[0], rt.shape[0] * C * PD * PH * PW, r.offset[1]
        buf = torch.full((n + 4,), float("nan"), device=dev)
        assert buf.data_ptr() % 16 == 0

        def fn():
            roi3d_b200._lib.check(roi3d_b200._lib.lib.roi3d_roi_align3d_forward(
                x.data_ptr(), roi3d_b200._lib.NDHWC, B, C, D, H, W, rt.data_ptr(), K, PD, PH, PW, SCALE, SCALE_D,
                r.sample_num, buf.data_ptr() + 4 * off, stream_ptr()))
            res.append(buf[off:off + n].view(K, C, PD, PH, PW))
    else:
        mod = _module(r)

        def fn():
            res.append(mod(xs, rt))
    roi3d_b200._lib.set_tuning(0, r.variant)
    try:
        names = launched_kernels(fn)
    finally:
        roi3d_b200._lib.set_tuning(0, 0)
    return names, res[0]


def _run_backward(r, feats, rt, g, dev):
    """(launched kernel names, per-level input gradients) of the row's backward call."""
    import torch
    import roi3d_b200
    from roi3d_b200._util import stream_ptr
    from roi3d_b200.ops import set_bug_compat
    gt = torch.from_numpy(g).to(dev)
    res = []
    if r.offset is not None and r.offset[0] == "grad":
        (f,) = feats
        B, C, D, H, W = f.shape
        PD, PH, PW = r.out
        n, off = f.size, r.offset[1]
        buf = torch.full((n + 4,), float("nan"), device=dev)      # zero_fill=1 clears exactly the gradient
        assert buf.data_ptr() % 16 == 0

        def fn():
            roi3d_b200._lib.check(roi3d_b200._lib.lib.roi3d_roi_align3d_backward(
                gt.data_ptr(), rt.data_ptr(), rt.shape[0], PD, PH, PW, SCALE, SCALE_D, r.sample_num,
                buf.data_ptr() + 4 * off, roi3d_b200._lib.NDHWC, B, C, D, H, W, 1, int(r.bug_compat), stream_ptr()))
            res.append([buf[off:off + n].view(B, D, H, W, C).permute(0, 4, 1, 2, 3)])
    else:
        xs = [_cl(torch.from_numpy(f).to(dev)).requires_grad_(True) for f in feats]
        out = _module(r)(xs, rt)

        def fn():
            out.backward(gt)
            res.append([x.grad for x in xs])
    roi3d_b200._lib.set_tuning(1, r.variant)
    set_bug_compat(r.bug_compat)
    det_before = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(r.det)
    try:
        names = launched_kernels(fn)
    finally:
        torch.use_deterministic_algorithms(det_before)
        set_bug_compat(False)
        roi3d_b200._lib.set_tuning(1, 0)
    return names, res[0]


@pytest.mark.gpu
@pytest.mark.parametrize("r", COVERAGE, ids=_row_id)
def test_roi_align_kernel_row(oracle, dev, r):
    import torch
    seed = sum(map(ord, r.tag + r.kernel)) % 1000
    rng = np.random.default_rng(seed)
    shapes = level_shapes(r)
    feats = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    rois = roi_set(r, shapes[0][2:], seed)
    if r.k_total:
        assert len(rois) == r.k_total
    rt = torch.from_numpy(rois).to(dev)
    if r.direction == "fwd":
        names, out = _run_forward(r, _device_levels(r, feats, dev), rt, dev)
        got = out.detach().cpu().numpy()
        want = expected_forward(oracle, feats, rois, r)
        assert compute_kernels(names) == [kernel_key(r.kernel)], names
        assert got.shape == want.shape
        check_forward(got, want)
    else:
        PD, PH, PW = r.out
        g = rng.standard_normal((len(rois), shapes[0][1], PD, PH, PW)).astype(np.float32)
        names, grads = _run_backward(r, feats, rt, g, dev)
        want = expected_backward(oracle, g, rois, r)
        assert compute_kernels(names) == [kernel_key(r.kernel)], names
        for got, w in zip(grads, want):
            assert tuple(got.shape) == w.shape
            assert rel_err(got.cpu().numpy(), w) <= BWD_TOL


# ------------------------------------------------------------------------------------------------ CPU checks
def test_every_roi_align_kernel_has_a_coverage_row():
    """The RoIAlign3D instantiations in the built library are exactly the COVERAGE kernels plus the helpers: a kernel
    added without a row here fails this test on any machine."""
    built = built_kernels("roi_align3d_")
    covered = {kernel_key(r.kernel) for r in COVERAGE}
    helpers = {h for h in HELPERS if h.startswith("roi_align3d_")}
    assert not covered & helpers
    assert built == covered | helpers, ("built, no row: %s; row, not built: %s"
                                        % (sorted(built - covered - helpers), sorted((covered | helpers) - built)))


def test_coverage_rows_are_well_formed():
    for r in COVERAGE:
        assert r.direction in ("fwd", "bwd") and r.layout in ("NDHWC", "NCDHW")
        assert len(r.shape) == 5 and len(r.out) == 3
        assert r.variant in (0, 50, 60, 99)
        assert not (r.bug_compat and r.direction == "fwd")
        # bug_compat rows are non-cubic with PD < PH: the reference's wrong top_diff index then stays inside the RoI's
        # own (k, c) block, so the oracle run on the in-range RoIs alone reads what the kernel reads
        assert not r.bug_compat or r.out[0] < r.out[1]
        assert r.direction == "fwd" or r.layout == "NDHWC"
    ids = [_row_id(r) for r in COVERAGE]
    assert len(ids) == len(set(ids))


@pytest.mark.parametrize("sample_num", [2, 0, 3, 1])
def test_boundary_lattice_puts_samples_on_the_edges(sample_num):
    """The lattice RoIs place samples exactly where the reference's axis_tap is discontinuous, on every axis."""
    dhw, out = (8, 12, 44), (10, 12, 14)
    rois = lattice_rois(dhw, out, SCALE, SCALE_D, sample_num, 2)
    S = sample_num if sample_num > 0 else 2
    D, H, W = dhw
    for a, (L, s, P, (lo, hi)) in enumerate([(W, SCALE, out[2], (1, 3)), (H, SCALE, out[1], (2, 4)),
                                             (D, SCALE_D, out[0], (5, 6))]):
        hits = set()
        for rr in rois[4 * a:4 * a + 4]:
            assert ((np.float64(rr[hi]) + 1) * s - np.float64(rr[lo]) * s) / P == S   # bin = S (adaptive: ceil = 2)
            hits |= set(_axis_coords(rr[lo], rr[hi], s, P, S))
        for edge in (-1.0, 0.0, L - 1.0, float(L), -1.0 - 1 / 16, L + 1 / 16):
            assert edge in hits, (a, edge)

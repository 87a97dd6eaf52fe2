"""Adversarial inputs for RPN target assignment.  TEST INFRASTRUCTURE ONLY.

Inputs that take the any-input branch of the IoU / argmax kernel (csrc/targets.cu, k2_exact_warp): boxes that are
not "nice" (a coordinate that is not 0 and not of magnitude in [2^-16, 2^8), or an extent that is not positive).
Shared by tests/test_targets_adversarial_gpu.py (kernel against the C oracle) and tests/test_oracle_cross.py (the
NumPy and C oracles against each other on the same inputs).

Every layout returns anchors (N,4), gt_boxes (B,G,4) and gt_labels (B,G), float32 / int32, [y1, x1, y2, x2].
"""
import numpy as np

F32 = np.float32
NAN, INF = float("nan"), float("inf")

FALLBACK_LAYOUTS = ("pixel", "tiny", "flip_one_axis", "flip_both_axes", "nan_inf", "line_vs_zero_area", "nan_column")


def dyadic_boxes(rng, n, lo=0, hi=64, ext=(1, 9)):
    """n boxes with corners on the 1/64 grid inside [lo/64, hi/64], extents ext[0]..ext[1]-1 steps (all nice)"""
    h = rng.integers(ext[0], ext[1], size=n)
    w = rng.integers(ext[0], ext[1], size=n)
    y1 = rng.integers(lo, hi - h + 1)
    x1 = rng.integers(lo, hi - w + 1)
    return (np.stack([y1, x1, y1 + h, x1 + w], axis=1) / 64.0).astype(F32)


def _gt(rng, B, G, n_real):
    """zero-padded GT (utils/data_utils.py:152-157): n_real dyadic boxes with labels >= 0, then padding rows"""
    gtb = np.zeros((B, G, 4), F32)
    gtl = np.full((B, G), -1, np.int32)
    for b in range(B):
        gtb[b, :n_real] = dyadic_boxes(rng, n_real, ext=(4, 30))
        gtl[b, :n_real] = rng.integers(0, 20, size=n_real)
    return gtb, gtl


def fallback_layout(name, seed=0, N=700, B=3, G=12):
    """N is not a multiple of any tile (32 * APT anchors), so every layout also has a partial last tile."""
    rng = np.random.default_rng(seed)
    anchors = dyadic_boxes(rng, N)
    gtb, gtl = _gt(rng, B, G, 8)
    if name == "pixel":
        # unnormalised pixel coordinates (up to 1333): anchors and GT; some GT boxes are copies of anchors (IoU 1)
        py = rng.integers(0, 780, size=N); px = rng.integers(0, 1300, size=N)
        ph = rng.integers(8, 300, size=N); pw = rng.integers(8, 300, size=N)
        anchors = np.stack([py, px, np.minimum(py + ph, 800), np.minimum(px + pw, 1333)], 1).astype(F32)
        anchors[N // 2] = anchors[3]                     # duplicate: the lower index wins
        for b in range(B):
            gtb[b, :8] = anchors[rng.integers(0, N, size=8)] + F32(b)      # image 0: exact copies
            gtb[b, 0] = anchors[3]
            gtb[b, 1] = [0, 0, 800, 1333]
    elif name == "tiny":
        # a coordinate in (0, 2^-16): subnormal-free but below the nice range, in anchors and GT boxes
        anchors[5, 0] = F32(3e-6)
        anchors[N - 2, 1] = F32(2.0 ** -20)
        gtb[0, 2] = [2.0 ** -18, 0.25, 0.5, 0.75]
        gtb[1, 0] = anchors[5]                           # IoU 1 with the anchor that carries the tiny coordinate
        gtb[2, 3] = [1e-7, 1e-7, 2e-7, 2e-7]             # overlaps nothing
    elif name == "flip_one_axis":
        # negative area: inter = 0 and union = anchor area + GT area < 0 for the smaller anchors, so those IoUs are -0
        # and the larger anchors' are +0.  They compare equal: the first index wins (the oracle's argmax).
        anchors[0] = [0, 0, 0.1, 0.1]
        anchors[1] = [0.5, 0.5, 1, 1]
        anchors[300] = [0.5, 0.25, 1, 0.75]              # another +0, in a later lane and CTA at every tile size
        gtb[0, 0] = [0.8, 0, 0.6, 0.1]                   # area -0.02: IoU -0 with anchor 0, +0 with anchor 1
        gtb[1, :4] = gtb[1, :4][:, [2, 1, 0, 3]]         # y flipped
        gtb[1, 0] = [0.9, 0.0, 0.1, 0.9]                 # area -0.72: -0 with every anchor
        gtb[2, :3] = gtb[2, :3][:, [0, 3, 2, 1]]         # x flipped
        gtl[2, 1] = -1                                   # a flipped box that forces nothing
    elif name == "flip_both_axes":
        # positive area without extent: every pair is disjoint, IoU +0
        gtb[0, 0] = [0.8, 0.9, 0.6, 0.7]
        gtb[1, :8] = gtb[1, :8][:, [2, 3, 0, 1]]
        gtb[2, 5] = [1.0, 1.0, 0.0, 0.0]
    elif name == "nan_inf":
        anchors[3, 0] = NAN                              # NaN area: a NaN row, max_iou -inf
        anchors[40, 3] = NAN
        anchors[41] = [-INF, -INF, INF, INF]             # area inf: IoU +0 or NaN (inf / inf)
        anchors[N - 1] = [0, 0, INF, 0.5]
        anchors[200] = [0, INF, 0.5, INF]                # extent inf - inf = NaN
        gtb[0, 0] = [0.1, 0.1, 0.4, INF]
        gtb[0, 1] = [-INF, 0.0, INF, 0.25]
        gtb[1, 0] = [0.2, NAN, 0.6, 0.6]
        gtb[1, 1] = [NAN, NAN, NAN, NAN]
        gtl[1, 1] = -1
        gtb[2, 0] = [-INF, -INF, INF, INF]
        gtb[2, 1] = [INF, INF, INF, INF]
    elif name == "line_vs_zero_area":
        # every anchor has zero area (y1 == y2); a GT with extent along x only has area 0 as well: 0 / 0 = NaN in its
        # whole column, so its key is -inf everywhere and argmax picks anchor 0.  Against boxes with area, +0.
        anchors[:, 2] = anchors[:, 0]
        gtb[0, 0] = [0.5, 0.1, 0.5, 0.9]
        gtb[1, :] = 0; gtl[1, :] = -1
        gtb[1, 0] = [0.25, 0.0, 0.25, 1.0]; gtl[1, 0] = 4
        gtb[1, 1] = [0.75, 0.5, 0.75, 0.5]; gtl[1, 1] = 2
        gtb[2, 2] = [0.3, 0.2, 0.3, 0.2]                 # a point with label >= 0
    elif name == "nan_column":
        # a valid GT whose whole column is NaN: never wins a '>', so its forced positive is anchor 0
        gtb[0, 0] = [NAN, 0.1, 0.5, 0.5]
        gtb[1, :] = NAN                                  # every column NaN: all max_iou -inf, the deltas of the
        gtl[1, :] = 3                                    # forced positive (anchor 0) are NaN
        gtb[2, 4] = [0.1, 0.1, 0.5, NAN]
        gtl[2, 4] = -1
    else:
        raise ValueError(name)
    return np.ascontiguousarray(anchors, F32), gtb, gtl

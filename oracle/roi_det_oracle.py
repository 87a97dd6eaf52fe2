"""NumPy restatement of the second stage's box-head detections (tfrpn_roi_head_detections, include/tfrpn.h).
TEST INFRASTRUCTURE, not product.

Built from the RPN oracle's pieces, every float operation rounded separately in float32:
  * the boxes: d = box_deltas * variances, dh and dw replaced by max_log_scale where greater (NaN stays NaN),
    get_bboxes_from_deltas(roi, d), clip01 when clip;
  * the candidates: rows s < clamp(valid[b], 0, S), classes 1..C-1, p > score_threshold and, when min_size > 0,
    (y2 - y1) >= min_size and (x2 - x1) >= min_size;
  * combined_non_max_suppression over the C - 1 foreground columns (non-candidates read as NaN, which never passes
    the score test), pre_nms_topn as a per-class top-n over the candidates, then class ids shifted by 1.
The softmax here is NumPy's (float32, another sum order and exp than the kernel's): the GPU tests feed the device's
own probabilities to the oracle for bit parity.
"""
from __future__ import annotations

import numpy as np

from . import rpn_oracle as O

F32 = np.float32


def softmax(x):
    """float32 softmax of the last axis; a NaN logit makes the row NaN"""
    x = np.asarray(x, F32)
    m = np.max(np.where(np.isnan(x), -np.inf, x), axis=-1, keepdims=True)
    e = np.exp(x - m)
    return (e / np.sum(e, axis=-1, keepdims=True, dtype=F32)).astype(F32)


def scale_deltas(box_deltas, variances=(0.1, 0.1, 0.2, 0.2), max_log_scale=float("inf")):
    """deltas * variances, then dh, dw = d > max ? max : d (NaN stays NaN)"""
    d = (np.asarray(box_deltas, F32) * np.asarray(variances, F32)).astype(F32)
    mx = F32(max_log_scale)
    d[..., 2:] = np.where(d[..., 2:] > mx, mx, d[..., 2:])
    return d


def decode(rois, box_deltas, variances=(0.1, 0.1, 0.2, 0.2), max_log_scale=float("inf"), clip=True):
    """(B,S,4) RoIs and (B,S,q,4) deltas -> (B,S,q,4) boxes"""
    d = scale_deltas(box_deltas, variances, max_log_scale)
    r = np.broadcast_to(np.asarray(rois, F32)[:, :, None, :], d.shape)
    b = O.get_bboxes_from_deltas(r, d)
    return O.clip01(b) if clip else b


def candidates(probs, boxes, valid=None, score_threshold=0.05, min_size=0.0):
    """(B,S,C) bool: the entries that enter the NMS"""
    p = np.asarray(probs, F32)
    B, S, Cn = p.shape
    nv = np.full(B, S) if valid is None else np.clip(np.asarray(valid, np.int64), 0, S)
    cand = (np.arange(S)[None, :] < nv[:, None])[..., None] & (p > F32(score_threshold))
    cand[..., 0] = False
    if min_size > 0:
        ms = F32(min_size)
        with np.errstate(invalid="ignore"):
            ok = ((boxes[..., 2] - boxes[..., 0]) >= ms) & ((boxes[..., 3] - boxes[..., 1]) >= ms)
        cand &= np.broadcast_to(ok, cand.shape)
    return cand


def roi_head_detections(rois, probs, box_deltas, valid=None, *, variances=(0.1, 0.1, 0.2, 0.2),
                        max_log_scale=float("inf"), clip=True, min_size=0.0, max_output_size_per_class=100,
                        max_total_size=100, iou_threshold=0.5, score_threshold=0.05, pad_per_class=False,
                        clip_boxes=True, pre_nms_topn=0, boxes=None):
    """probs (B,S,C) -> (boxes, scores, classes, valid, keep_idx).  `boxes` (B,S,q,4) replaces the decode (the GPU
    tests pass tfrpn_decode's output)."""
    p = np.asarray(probs, F32)
    B, S, Cn = p.shape
    if boxes is None:
        boxes = decode(rois, box_deltas, variances, max_log_scale, clip)
    boxes = np.asarray(boxes, F32)
    q = boxes.shape[2]
    cand = candidates(p, boxes, valid, score_threshold, min_size)
    sc = np.where(cand, p, F32(np.nan))[..., 1:]
    if pre_nms_topn > 0:
        for b in range(B):
            for c in range(Cn - 1):
                order = np.argsort(-sc[b, :, c].astype(np.float64), kind="stable")   # NaN last
                sc[b, order[pre_nms_topn:], c] = np.nan
    bx = boxes if q == 1 else boxes[:, :, 1:]
    nb, ns, nc, nv, ni = O.combined_non_max_suppression(bx, sc, max_output_size_per_class, max_total_size,
                                                        iou_threshold=iou_threshold, score_threshold=score_threshold,
                                                        pad_per_class=pad_per_class, clip_boxes=clip_boxes,
                                                        return_indices=True)
    live = np.arange(nc.shape[1])[None, :] < nv[:, None]
    nc = np.where(live, nc + F32(1), nc).astype(F32)
    return nb, ns, nc, nv, ni

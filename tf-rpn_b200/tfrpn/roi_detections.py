"""Box-head detections of a two-stage detector's second stage at inference, on the GPU (tfrpn_roi_head_detections,
include/tfrpn.h): softmax over the class logits, per-class decode of the RoIs, clip, the size filter and class-aware
NMS, i.e. torchvision's ``RoIHeads.postprocess_detections`` without the framework glue.

Only the (image, class, row) entries above the score threshold are decoded; the proposals' padding rows (``valid``
of ``generate_proposals``) never produce a detection.  No host synchronisation: the call can be captured in a CUDA
graph once the workspace is sized (one eager call, or tfrpn_reserve_roi_head_detections).
"""
import ctypes as C

import torch

from . import _lib
from ._tensor import Origin, from_device, ptr, stream_ptr, to_device

F32 = torch.float32
_SCORES = {"logits": 0, "probs": 1}


def roi_head_detections(rois, cls_scores, box_deltas, valid_detections=None, *, scores="logits",
                        variances=(0.1, 0.1, 0.2, 0.2), max_log_scale=float("inf"), clip=True, min_size=0.0,
                        max_output_size_per_class=100, max_total_size=100, iou_threshold=0.5, score_threshold=0.05,
                        pad_per_class=False, pre_nms_topn=0, return_indices=False, return_probs=False):
    """Detections from the box head's output: rois (B,S,4) and valid_detections (B,) or None as
    ``generate_proposals`` returns them, cls_scores (B,S,C) float32 (``scores="logits"``: the softmax is taken here;
    ``"probs"``: probabilities), box_deltas (B,S,C*4), (B,S,C,4), (B,S,4) or (B,S,1,4) float32 (class-specific q = C or
    class-agnostic q = 1, inferred from the shape; the reshape is a view).

    Per (image, row s, class c >= 1): the box is the RoI decoded with deltas * ``variances`` (dh, dw clamped from
    above at ``max_log_scale``), clipped to [0,1] when ``clip``; the entry is a candidate when row s < valid[b], its
    probability is > ``score_threshold`` and, with ``min_size`` > 0, both extents are >= min_size.  The candidates of
    each (image, class) then go through ``non_max_suppression``'s multi-class NMS and merge.  Class 0 is the
    background and is never detected.

    Returns (boxes (B,rows,4), scores (B,rows), classes (B,rows) float ids in 1..C-1, valid (B,) int32), the layout of
    ``non_max_suppression``, so ``DetectionMAP.update(*dets, gt_boxes, gt_labels)`` takes it as it is; rows =
    min(max_total_size, max_output_size_per_class * (C - 1)) with ``pad_per_class``, else max_total_size.
    ``return_indices`` appends keep_idx (B,rows) int32, the RoI row of each detection (-1 padded), and then
    ``return_probs`` the probabilities (B,S,C) (logits input only).  torch, NumPy and TF inputs come back in their own
    framework.  C > 1024, S > 8192 or B > 65535 raise NotImplementedError; bad arguments raise ValueError."""
    if scores not in _SCORES:
        raise ValueError("scores must be 'logits' or 'probs', got %r" % (scores,))
    if return_probs and scores != "logits":
        raise ValueError("return_probs needs scores='logits'")
    o = Origin()
    r = to_device(rois, F32, o, "rois")
    if r.dim() != 3 or r.shape[2] != 4:
        raise ValueError("rois must be (B,S,4), got %s" % (tuple(r.shape),))
    B, S = r.shape[:2]
    x = to_device(cls_scores, F32, o, "cls_scores")
    if x.dim() != 3 or x.shape[:2] != (B, S):
        raise ValueError("cls_scores must be (%d,%d,C), got %s" % (B, S, tuple(x.shape)))
    Cn = x.shape[2]
    d = to_device(box_deltas, F32, o, "box_deltas")
    if d.dim() == 3 and d.shape[:2] == (B, S) and d.shape[2] % 4 == 0:
        d4 = d.view(B, S, d.shape[2] // 4, 4)
    elif d.dim() == 4 and d.shape[:2] == (B, S) and d.shape[3] == 4:
        d4 = d
    else:
        raise ValueError("box_deltas must be (B,S,q*4) or (B,S,q,4) with (B,S) = (%d,%d), got %s"
                         % (B, S, tuple(d.shape)))
    val = None if valid_detections is None else to_device(valid_detections, torch.int32, o, "valid_detections")
    if val is not None and tuple(val.shape) != (B,):
        raise ValueError("valid_detections must be (%d,), got %s" % (B, tuple(val.shape)))
    nms = _lib.NmsCfg(int(max_output_size_per_class), int(max_total_size), _lib.iou_threshold(iou_threshold),
                      float(score_threshold), int(bool(pad_per_class)), int(bool(clip)), int(pre_nms_topn or 0))
    cfg = _lib.RoiDetCfg(int(Cn), int(d4.shape[2]), _SCORES[scores], (C.c_float * 4)(*[float(v) for v in variances]),
                         float(max_log_scale), int(bool(clip)), float(min_size), nms)
    if nms.max_output_size_per_class <= 0 or nms.max_total_size <= 0:
        raise ValueError("max_output_size_per_class and max_total_size must be > 0")
    rows = min(nms.max_total_size, nms.max_output_size_per_class * max(Cn - 1, 0)) if nms.pad_per_class \
        else nms.max_total_size
    dev = r.device
    run = B > 0 and S > 0   # the kernels write every output; without rows every output row is padding
    alloc = torch.empty if run else torch.zeros
    nb = alloc((B, rows, 4), dtype=F32, device=dev)
    ns = alloc((B, rows), dtype=F32, device=dev)
    nc = alloc((B, rows), dtype=F32, device=dev)
    nv = alloc((B,), dtype=torch.int32, device=dev)
    ni = None
    if return_indices:
        ni = torch.empty((B, rows), dtype=torch.int32, device=dev) if run else torch.full((B, rows), -1, dtype=torch.int32, device=dev)
    pr = alloc((B, S, Cn), dtype=F32, device=dev) if return_probs else None
    if run:
        _lib.check(_lib.load().tfrpn_roi_head_detections(_lib.handle(dev.index), ptr(r), ptr(val), ptr(x), ptr(d4), B,
                                                         S, C.byref(cfg), ptr(nb), ptr(ns), ptr(nc), ptr(nv), ptr(ni),
                                                         ptr(pr), stream_ptr(dev)))
    res = tuple(from_device(t, o) for t in (nb, ns, nc, nv))
    if return_indices:
        res += (from_device(ni, o),)
    if return_probs:
        res += (from_device(pr, o),)
    return res

"""RoI target assignment of a two-stage detector's second stage, on the GPU (tfrpn_roi_targets, include/tfrpn.h).

Matches every proposal (and, with ``append_gt``, every GT box) to its best GT box, samples a fixed-size minibatch
of foreground and background rows per image and writes what the box head trains on: the rows' boxes, class labels
and encoded deltas.  The rules follow Detectron (fg at IoU >= 0.5, bg in [0, 0.5), 128 fg of 512); the sampler is
the counter RNG of the RPN targets (words 2 and 3 of the same Philox counter), so a run is reproducible from
(seed, offset) and a sharded batch samples like the whole one given ``image_offset``.  One kernel launch, no
workspace, no host synchronisation: the call can be captured in a CUDA graph.
"""
import collections
import ctypes as C

import torch

from . import _lib
from ._tensor import Origin, from_device, ptr, stream_ptr, to_device
from .utils import train_utils

F32 = torch.float32
RoiTargets = collections.namedtuple("RoiTargets", "rois labels deltas src_index counts")


def roi_target_cfg(num_classes, total_pos=128, total_neg=384, fg_iou_threshold=0.5, bg_iou_high=0.5, bg_iou_low=0.0,
                   variances=(0.1, 0.1, 0.2, 0.2), append_gt=True, seed=0, offset=None, image_offset=0):
    """-> a filled tfrpn_roi_target_cfg; ``offset=None`` takes the next value of the RPN targets' auto offset."""
    var = [float(v) for v in variances]
    if len(var) != 4:
        raise ValueError("variances must have 4 values, got %d" % len(var))
    cfg = _lib.RoiTargetCfg()
    cfg.num_classes = int(num_classes)
    cfg.total_pos = int(total_pos)
    cfg.total_neg = int(total_neg)
    cfg.fg_iou_threshold = float(fg_iou_threshold)
    cfg.bg_iou_high = float(bg_iou_high)
    cfg.bg_iou_low = float(bg_iou_low)
    for i, v in enumerate(var):
        cfg.variances[i] = v
    cfg.append_gt = 1 if append_gt else 0
    cfg.image_offset = int(image_offset)
    cfg.seed = int(seed)
    cfg.offset = next(train_utils._auto_offset) if offset is None else int(offset)
    return cfg


def roi_targets(rois, gt_boxes, gt_labels, valid_detections=None, *, num_classes, total_pos=128, total_neg=384,
                fg_iou_threshold=0.5, bg_iou_high=0.5, bg_iou_low=0.0, variances=(0.1, 0.1, 0.2, 0.2),
                append_gt=True, seed=0, offset=None, image_offset=0, return_debug=False):
    """Second-stage training targets for rois (B,P,4) against gt_boxes (B,G,4) / gt_labels (B,G) int.

    rois and valid_detections (B,) are what ``generate_proposals`` returns; gt_boxes and gt_labels what
    ``pad_gt_batch(label_add=1)`` returns (class 0 is background; GT with a label outside [1, num_classes) take no
    part).  Each image gets S = total_pos + total_neg rows: its sampled fg rows in ascending row order, then its
    sampled bg rows, then padding.  Returns RoiTargets(rois (B,S,4), labels (B,S) int32 -- the GT class for fg, 0 for
    bg, -1 for padding, deltas (B,S,4) -- get_deltas_from_bboxes(row, matched GT) / variances for fg, 0 otherwise,
    src_index (B,S) int32 -- the row (n < P a proposal, P + g GT box g; -1 padding), counts (B,2) int32 -- (#fg,
    #fg + #bg)); with ``return_debug`` also a dict of max_iou (B,P') float32 and argmax (B,P') int32 (-1.0 / -1 for
    rows that take no part), P' = P + G with ``append_gt``.  Results come back in the framework of the inputs
    (device tensors stay on the device).  The full definition is in include/tfrpn.h.  P > 8192, G > 1024 or S > 8192
    raise NotImplementedError; bad arguments raise ValueError."""
    cfg = roi_target_cfg(num_classes, total_pos, total_neg, fg_iou_threshold, bg_iou_high, bg_iou_low, variances,
                         append_gt, seed, offset, image_offset)
    o = Origin()
    r = to_device(rois, F32, o, "rois")
    if r.dim() != 3 or r.shape[2] != 4:
        raise ValueError("rois must be (B,P,4), got %s" % (tuple(r.shape),))
    B, P = r.shape[:2]
    gt = to_device(gt_boxes, F32, o, "gt_boxes")
    if gt.dim() != 3 or gt.shape[2] != 4 or gt.shape[0] != B:
        raise ValueError("gt_boxes must be (B,G,4) with B = %d, got %s" % (B, tuple(gt.shape)))
    G = gt.shape[1]
    lab = to_device(gt_labels, torch.int32, o, "gt_labels")
    if tuple(lab.shape) != (B, G):
        raise ValueError("gt_labels must be (%d,%d), got %s" % (B, G, tuple(lab.shape)))
    val = None if valid_detections is None else to_device(valid_detections, torch.int32, o, "valid_detections")
    if val is not None and tuple(val.shape) != (B,):
        raise ValueError("valid_detections must be (%d,), got %s" % (B, tuple(val.shape)))
    dev = r.device
    S = max(cfg.total_pos + cfg.total_neg, 0)
    Pp = P + (G if append_gt else 0)
    i32 = torch.int32
    out = RoiTargets(torch.empty((B, S, 4), dtype=F32, device=dev), torch.empty((B, S), dtype=i32, device=dev),
                     torch.empty((B, S, 4), dtype=F32, device=dev), torch.empty((B, S), dtype=i32, device=dev),
                     torch.empty((B, 2), dtype=i32, device=dev))
    dbg = None
    if return_debug:
        dbg = dict(max_iou=torch.empty((B, Pp), dtype=F32, device=dev), argmax=torch.empty((B, Pp), dtype=i32, device=dev))
    _lib.check(_lib.load().tfrpn_roi_targets(
        _lib.handle(dev.index), ptr(r), ptr(val), ptr(gt), ptr(lab), B, P, G, C.byref(cfg), ptr(out.rois),
        ptr(out.labels), ptr(out.deltas), ptr(out.src_index), ptr(out.counts),
        ptr(dbg["max_iou"]) if dbg else None, ptr(dbg["argmax"]) if dbg else None, stream_ptr(dev)))
    res = RoiTargets(*(from_device(t, o) for t in out))
    if return_debug:
        return res, {k: from_device(v, o) for k, v in dbg.items()}
    return res

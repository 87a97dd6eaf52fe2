"""Proposal recall against ground truth, on the GPU (tfrpn_proposal_recall, include/tfrpn.h).

The standard quality measure of an RPN: the fraction of valid GT boxes that the top-k proposals of their image
cover at IoU >= t, for every limit k and threshold t, and AR@k, its mean over t (the Detectron / COCO mean, not
Hosang's integral).  A GT box is valid when its area is positive and, with labels, its label is >= 0, so the
padding rows of ``pad_gt_batch`` (zero box, label -1) do not count.  ``matching="greedy"`` is the one-to-one
matching of Detectron's ``evaluate_box_proposals`` and mmdet's ``eval_recalls`` (largest IoU first; ties to the
lowest GT index, then the lowest rank); ``"coverage"`` gives every GT its best IoU with no exclusivity.
The result is exact integer counting: it does not depend on batching or on launch order.
"""
import collections
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._tensor import Origin, default_device, from_device, ptr, stream_ptr, to_device

F32 = torch.float32
DEFAULT_THRESHOLDS = tuple(float(np.float32(x / 100)) for x in range(50, 100, 5))   # 0.50:0.05:0.95 in float32
DEFAULT_LIMITS = (100, 300, 1000)
MATCHING = {"greedy": 0, "coverage": 1}
MAX_THRESHOLDS, MAX_LIMITS = 16, 8

RecallResult = collections.namedtuple("RecallResult", "recall average_recall hits n_gt thresholds limits")
RecallResultIoU = collections.namedtuple("RecallResultIoU", RecallResult._fields + ("gt_iou",))


def recall_cfg(iou_thresholds=None, limits=DEFAULT_LIMITS, matching="greedy"):
    """-> a filled tfrpn_recall_cfg.  Values outside the supported range are rejected by the library."""
    thr = np.asarray(DEFAULT_THRESHOLDS if iou_thresholds is None else iou_thresholds, np.float32).reshape(-1)
    lim = [int(v) for v in np.asarray(limits).reshape(-1)]
    if not 1 <= thr.size <= MAX_THRESHOLDS:
        raise ValueError("iou_thresholds: 1..%d values, got %d" % (MAX_THRESHOLDS, thr.size))
    if not 1 <= len(lim) <= MAX_LIMITS:
        raise ValueError("limits: 1..%d values, got %d" % (MAX_LIMITS, len(lim)))
    if matching not in MATCHING:
        raise ValueError("matching must be one of %s, got %r" % (sorted(MATCHING), matching))
    cfg = _lib.RecallCfg()
    cfg.n_thresholds = thr.size
    for i, v in enumerate(thr):
        cfg.thresholds[i] = float(v)
    cfg.n_limits = len(lim)
    for i, v in enumerate(lim):
        cfg.limits[i] = v
    cfg.matching = MATCHING[matching]
    return cfg


def _inputs(o, proposals, gt_boxes, gt_labels, valid_detections):
    prop = to_device(proposals, F32, o, "proposals")
    gt = to_device(gt_boxes, F32, o, "gt_boxes")
    if prop.dim() != 3 or prop.shape[2] != 4:
        raise ValueError("proposals must be (B,P,4), got %s" % (tuple(prop.shape),))
    if gt.dim() != 3 or gt.shape[2] != 4 or gt.shape[0] != prop.shape[0]:
        raise ValueError("gt_boxes must be (B,G,4) with B = %d, got %s" % (prop.shape[0], tuple(gt.shape)))
    B, G = gt.shape[:2]
    lab = None if gt_labels is None else to_device(gt_labels, torch.int32, o, "gt_labels")
    if lab is not None and tuple(lab.shape) != (B, G):
        raise ValueError("gt_labels must be (%d,%d), got %s" % (B, G, tuple(lab.shape)))
    val = None if valid_detections is None else to_device(valid_detections, torch.int32, o, "valid_detections")
    if val is not None and tuple(val.shape) != (B,):
        raise ValueError("valid_detections must be (%d,), got %s" % (B, tuple(val.shape)))
    return prop, gt, lab, val


def _launch(cfg, prop, gt, lab, val, gt_iou, counts):
    dev = counts.device
    B, P = prop.shape[:2]
    _lib.check(_lib.load().tfrpn_proposal_recall(_lib.handle(dev.index), ptr(prop), ptr(val), ptr(gt), ptr(lab), B, P,
                                                 gt.shape[1], C.byref(cfg), ptr(gt_iou), ptr(counts), stream_ptr(dev)))


def _result(counts_host, cfg, o):
    L, T = cfg.n_limits, cfg.n_thresholds
    c = np.asarray(counts_host, np.int64)
    hits = c[:-1].reshape(L, T)
    with np.errstate(invalid="ignore"):
        recall = hits / np.float64(c[-1])   # NaN without valid GT
    thr = np.asarray(cfg.thresholds[:T], np.float32)
    out = [from_device(torch.from_numpy(np.ascontiguousarray(a)), o) for a in (recall, recall.mean(axis=1), hits, thr)]
    return RecallResult(out[0], out[1], out[2], int(c[-1]), out[3], tuple(cfg.limits[:L]))


def proposal_recall(proposals, gt_boxes, gt_labels=None, valid_detections=None, iou_thresholds=None,
                    limits=DEFAULT_LIMITS, matching="greedy", return_gt_iou=False):
    """Recall of proposals (B,P,4), in rank order best first, against gt_boxes (B,G,4) at every limit and threshold.

    ``gt_labels`` (B,G): GT with a label < 0 do not count.  ``valid_detections`` (B,): only the first valid[b] rows of
    image b are proposals.  Both take what ``generate_proposals`` and ``pad_gt_batch`` return.  ``iou_thresholds``:
    1..16 values in (0,1], default 0.50:0.05:0.95 in float32; ``limits``: 1..8 positive ints.
    Returns RecallResult(recall (L,T) float64 -- NaN without valid GT, average_recall (L,), hits (L,T) int64, n_gt,
    thresholds (T,) float32, limits) as NumPy arrays for NumPy inputs and as (CPU) torch tensors otherwise; with
    ``return_gt_iou`` also gt_iou (L,B,G) float32, the matched IoU of every GT box (-1 = invalid GT), which for device
    inputs stays on the device and is computed on the current stream.  Synchronises once, to read the counts.
    G > 1024 or a limit > 8192 raises NotImplementedError; bad arguments raise ValueError."""
    cfg = recall_cfg(iou_thresholds, limits, matching)
    o = Origin()
    prop, gt, lab, val = _inputs(o, proposals, gt_boxes, gt_labels, valid_detections)
    dev = prop.device
    counts = torch.zeros(cfg.n_limits * cfg.n_thresholds + 1, dtype=torch.int64, device=dev)
    gt_iou = (torch.empty((cfg.n_limits, gt.shape[0], gt.shape[1]), dtype=F32, device=dev) if return_gt_iou else None)
    _launch(cfg, prop, gt, lab, val, gt_iou, counts)
    res = _result(counts.cpu().numpy(), cfg, o)
    if return_gt_iou:
        return RecallResultIoU(*res, from_device(gt_iou, o))
    return res


class ProposalRecall:
    """Running proposal-recall meter over a validation set (same definition as ``proposal_recall``).

    ``update`` only enqueues one kernel on the current stream of the meter's device: no synchronisation and, for
    device tensors of the right dtypes, no allocation, so it can be captured in a CUDA graph.  ``compute`` synchronises
    once and returns a RecallResult; ``reset`` zeroes the counts.  ``counts`` is the raw int64 tensor
    (hits[l][t] row-major, then n_gt); all counts are integers, so an ``all_reduce(SUM)`` of it across ranks followed
    by ``compute`` gives the global result exactly."""

    def __init__(self, iou_thresholds=None, limits=DEFAULT_LIMITS, matching="greedy", device=None):
        self._cfg = recall_cfg(iou_thresholds, limits, matching)
        self.device = torch.device(device) if device is not None else default_device()
        if self.device.type != "cuda":
            raise ValueError("ProposalRecall needs a CUDA device, got %s" % self.device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.counts = torch.zeros(self._cfg.n_limits * self._cfg.n_thresholds + 1, dtype=torch.int64,
                                  device=self.device)

    def update(self, proposals, gt_boxes, gt_labels=None, valid_detections=None):
        o = Origin()
        o.device = self.device
        prop, gt, lab, val = _inputs(o, proposals, gt_boxes, gt_labels, valid_detections)
        _launch(self._cfg, prop, gt, lab, val, None, self.counts)

    def compute(self):
        o = Origin()
        o.kind = "torch"
        return _result(self.counts.cpu().numpy(), self._cfg, o)

    def reset(self):
        self.counts.zero_()

"""Proposal recall against ground truth, on the GPU (tfrpn_proposal_recall, include/tfrpn.h).

The standard quality measure of an RPN: the fraction of valid GT boxes that the top-k proposals of their image
cover at IoU >= t, for every limit k and threshold t, and AR@k, its mean over t (the Detectron / COCO mean, not
Hosang's integral).  A GT box is valid when its area is positive and, with labels, its label is >= 0, so the
padding rows of ``pad_gt_batch`` (zero box, label -1) do not count.  ``matching="greedy"`` is the one-to-one
matching of Detectron's ``evaluate_box_proposals`` and mmdet's ``eval_recalls`` (largest IoU first; ties to the
lowest GT index, then the lowest rank); ``"coverage"`` gives every GT its best IoU with no exclusivity.
The result is exact integer counting: it does not depend on batching or on launch order.

``detection_map`` / ``DetectionMAP`` (tfrpn_map_update / tfrpn_map_compute): mean average precision of multi-class
detections (``non_max_suppression`` output) under the ``coco``, ``voc`` or ``voc07`` protocol; the definition is in
include/tfrpn.h and oracle/map_oracle.py.
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


MAP_PROTOCOLS = {"coco": 0, "voc": 1, "voc07": 2}
MAX_MAP_CLASSES = 1024
MapResult = collections.namedtuple("MapResult", "ap map mean_ap recall n_gt thresholds protocol")


def map_cfg(num_classes, protocol="coco", iou_thresholds=None, max_dets=100):
    """-> a filled tfrpn_map_cfg.  Default thresholds: 0.50:0.05:0.95 (float32) for coco, 0.5 for voc / voc07."""
    if protocol not in MAP_PROTOCOLS:
        raise ValueError("protocol must be one of %s, got %r" % (sorted(MAP_PROTOCOLS), protocol))
    if iou_thresholds is None:
        iou_thresholds = DEFAULT_THRESHOLDS if protocol == "coco" else (0.5,)
    thr = np.asarray(iou_thresholds, np.float32).reshape(-1)
    if not 1 <= thr.size <= MAX_THRESHOLDS:
        raise ValueError("iou_thresholds: 1..%d values, got %d" % (MAX_THRESHOLDS, thr.size))
    cfg = _lib.MapCfg()
    cfg.protocol = MAP_PROTOCOLS[protocol]
    cfg.num_classes = int(num_classes)
    cfg.n_thresholds = thr.size
    for i, v in enumerate(thr):
        cfg.thresholds[i] = float(v)
    cfg.max_dets = int(max_dets)
    return cfg


def _map_inputs(o, det_boxes, det_scores, det_classes, valid_detections, gt_boxes, gt_labels, gt_flags):
    db = to_device(det_boxes, F32, o, "det_boxes")
    if db.dim() != 3 or db.shape[2] != 4:
        raise ValueError("det_boxes must be (B,R,4), got %s" % (tuple(db.shape),))
    B, R = db.shape[:2]
    ds = to_device(det_scores, F32, o, "det_scores")
    dc = to_device(det_classes, F32, o, "det_classes")
    for name, t in (("det_scores", ds), ("det_classes", dc)):
        if tuple(t.shape) != (B, R):
            raise ValueError("%s must be (%d,%d), got %s" % (name, B, R, tuple(t.shape)))
    val = None if valid_detections is None else to_device(valid_detections, torch.int32, o, "valid_detections")
    if val is not None and tuple(val.shape) != (B,):
        raise ValueError("valid_detections must be (%d,), got %s" % (B, tuple(val.shape)))
    gt = to_device(gt_boxes, F32, o, "gt_boxes")
    if gt.dim() != 3 or gt.shape[2] != 4 or gt.shape[0] != B:
        raise ValueError("gt_boxes must be (B,G,4) with B = %d, got %s" % (B, tuple(gt.shape)))
    G = gt.shape[1]
    lab = to_device(gt_labels, torch.int32, o, "gt_labels")
    if tuple(lab.shape) != (B, G):
        raise ValueError("gt_labels must be (%d,%d), got %s" % (B, G, tuple(lab.shape)))
    flg = None if gt_flags is None else to_device(gt_flags, torch.uint8, o, "gt_flags")
    if flg is not None and tuple(flg.shape) != (B, G):
        raise ValueError("gt_flags must be (%d,%d), got %s" % (B, G, tuple(flg.shape)))
    return db, ds, dc, val, gt, lab, flg


class _MapState:
    """Device state of tfrpn_map_state: the records and one int64 vector [cursor, n_gt (C), overflow]."""

    def __init__(self, num_classes, capacity, device):
        if capacity < 0:
            raise ValueError("capacity must be >= 0, got %d" % capacity)
        self.records = torch.empty(max(int(capacity), 1) * 16, dtype=torch.uint8, device=device)
        self.counters = torch.zeros(num_classes + 2, dtype=torch.int64, device=device)
        self.c = _lib.MapState(self.records.data_ptr(), int(capacity), self.counters.data_ptr(),
                               self.counters.data_ptr() + 8, self.counters.data_ptr() + 8 * (num_classes + 1))


def _map_update(cfg, st, dev, db, ds, dc, val, gt, lab, flg):
    B, R = db.shape[:2]
    _lib.check(_lib.load().tfrpn_map_update(_lib.handle(dev.index), ptr(db), ptr(ds), ptr(dc), ptr(val), ptr(gt),
                                            ptr(lab), ptr(flg), B, R, gt.shape[1], C.byref(cfg), C.byref(st.c),
                                            stream_ptr(dev)))


def _map_compute(cfg, st, dev, o):
    Cn, T = cfg.num_classes, cfg.n_thresholds
    out = torch.empty((2, Cn, T), dtype=torch.float64, device=dev)
    _lib.check(_lib.load().tfrpn_map_compute(_lib.handle(dev.index), C.byref(cfg), C.byref(st.c), out[0].data_ptr(),
                                             out[1].data_ptr(), stream_ptr(dev)))
    host = torch.empty(out.shape, dtype=torch.float64, pin_memory=True)
    counters = torch.empty(st.counters.shape, dtype=torch.int64, pin_memory=True)
    host.copy_(out, non_blocking=True)
    counters.copy_(st.counters, non_blocking=True)
    torch.cuda.current_stream(dev).synchronize()
    c = counters.numpy()
    if c[-1]:
        raise RuntimeError("DetectionMAP: a batch did not fit in the capacity of %d records and was not recorded; "
                           "use a larger capacity" % st.c.capacity)
    ap, recall = host[0].numpy(), host[1].numpy()
    n_gt = c[1:Cn + 1].copy()
    sel = np.flatnonzero(n_gt > 0)
    if sel.size:
        m = np.cumsum(ap[sel], axis=0)[-1] / sel.size     # classes added in class order
        mean_ap = float(np.cumsum(m)[-1] / T)
    else:
        m = np.full(T, np.nan)
        mean_ap = float("nan")
    thr = np.asarray(cfg.thresholds[:T], np.float32)
    res = [from_device(torch.from_numpy(np.ascontiguousarray(a)), o) for a in (ap, m, recall, n_gt, thr)]
    return MapResult(res[0], res[1], mean_ap, res[2], res[3], res[4],
                     {v: k for k, v in MAP_PROTOCOLS.items()}[cfg.protocol])


def detection_map(det_boxes, det_scores, det_classes, valid_detections, gt_boxes, gt_labels, gt_flags=None, *,
                  num_classes, protocol="coco", iou_thresholds=None, max_dets=100):
    """Mean average precision of detections against ground truth, on the GPU.

    det_boxes (B,R,4), det_scores (B,R), det_classes (B,R) float class ids and valid_detections (B,) or None are what
    ``non_max_suppression`` returns, so ``detection_map(*nms_out, gt_boxes, gt_labels, num_classes=C)`` works as it is.
    gt_boxes (B,G,4) and gt_labels (B,G) are what ``pad_gt_batch`` returns; gt_flags (B,G) uint8, optional: bit 0
    ignore (VOC "difficult", COCO "ignore"), bit 1 crowd (COCO iscrowd, implies ignore).  ``protocol``: "coco" (IoU >=
    t, crowd rule, 101-point AP, per (image, class) the best ``max_dets`` detections, 0 = all), "voc" (IoU > t,
    all-point AP) or "voc07" (11-point AP).  ``iou_thresholds``: 1..16 values in (0,1]; default 0.50:0.05:0.95 (coco)
    or 0.5.  Returns MapResult(ap (C,T) float64 -- NaN for classes without non-ignored GT, map (T,) -- the mean over
    the other classes, mean_ap, recall (C,T), n_gt (C,) int64, thresholds (T,) float32, protocol), NumPy for NumPy
    inputs and CPU torch tensors otherwise.  Synchronises once.  R > 4096, G > 1024 or num_classes > 1024 raise
    NotImplementedError; bad arguments raise ValueError."""
    cfg = map_cfg(num_classes, protocol, iou_thresholds, max_dets)
    o = Origin()
    db, ds, dc, val, gt, lab, flg = _map_inputs(o, det_boxes, det_scores, det_classes, valid_detections, gt_boxes,
                                                gt_labels, gt_flags)
    dev = db.device
    st = _MapState(max(cfg.num_classes, 0), db.shape[0] * db.shape[1], dev)
    _map_update(cfg, st, dev, db, ds, dc, val, gt, lab, flg)
    return _map_compute(cfg, st, dev, o)


class DetectionMAP:
    """Running mAP meter over a validation set (same definition and arguments as ``detection_map``).

    ``update`` enqueues two kernels on the current stream of the meter's device: no synchronisation and, for device
    tensors of the right dtypes, no allocation, so it can be captured in a CUDA graph.  Every update takes B*R of the
    ``capacity`` record slots (16 bytes each).  ``compute`` synchronises once and returns a MapResult of CPU torch
    tensors; it raises RuntimeError if a batch did not fit.  ``reset`` empties the meter.  The records of one meter
    cover one process's data: they do not add across ranks."""

    def __init__(self, num_classes, protocol="coco", iou_thresholds=None, max_dets=100, capacity=1 << 22, device=None):
        self._cfg = map_cfg(num_classes, protocol, iou_thresholds, max_dets)
        self.device = torch.device(device) if device is not None else default_device()
        if self.device.type != "cuda":
            raise ValueError("DetectionMAP needs a CUDA device, got %s" % self.device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if not 1 <= self._cfg.num_classes:
            raise ValueError("num_classes must be >= 1, got %d" % self._cfg.num_classes)
        if self._cfg.num_classes > MAX_MAP_CLASSES:
            raise NotImplementedError("num_classes = %d, at most %d" % (self._cfg.num_classes, MAX_MAP_CLASSES))
        self._state = _MapState(self._cfg.num_classes, int(capacity), self.device)

    def update(self, det_boxes, det_scores, det_classes, valid_detections, gt_boxes, gt_labels, gt_flags=None):
        o = Origin()
        o.device = self.device
        args = _map_inputs(o, det_boxes, det_scores, det_classes, valid_detections, gt_boxes, gt_labels, gt_flags)
        _map_update(self._cfg, self._state, self.device, *args)

    def compute(self):
        o = Origin()
        o.kind = "torch"
        return _map_compute(self._cfg, self._state, self.device, o)

    def reset(self):
        self._state.counters.zero_()

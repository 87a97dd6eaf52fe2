"""NumPy restatement of detection mAP (tfrpn_map_update / tfrpn_map_compute, include/tfrpn.h).  TEST INFRASTRUCTURE,
not product.

Three protocols, each fixed as a whole:
  * ``coco``:  match at IoU >= t, the crowd rule, 101-point AP (pycocotools ``evaluateImg`` + ``accumulate``);
  * ``voc``:   match at IoU > t, the difficult rule, all-point area AP (the VOC2010+ devkit ``voc_ap``);
  * ``voc07``: the ``voc`` matching with the 11-point AP.
Inputs of one batch: detections (B,R,4) / (B,R) scores / (B,R) float class ids / valid (B,) or None; GT (B,G,4) /
(B,G) int labels / (B,G) uint8 flags or None (bit 0 ignore -- VOC "difficult", COCO "ignore"; bit 1 crowd, which
implies ignore).  A detection takes part when its row is < clamp(valid[b], 0, R) and its class is an integer in
[0, C); a GT when its label is in [0, C).  The IoU is ``rpn_oracle.generate_iou_map`` with the detection as
``bboxes``, NaN / negative / -0 read as +0; a crowd GT under ``coco`` scores inter / area(det) (+0 when area(det) <= 0).
Inside an (image, class) detections go by score descending, compared by value (NaN on top, +0 == -0), then row;
``coco`` keeps the first ``max_dets`` (0 = all).  Across the dataset the same key orders a class's detections, ties
in insertion order (update, image, order inside the image): a stable sort.  Every sum of the AP is taken in a stated
order, so the device reproduces these numbers bit for bit; ``pycocotools_ap`` / ``devkit_ap`` restate the original
``np.mean`` / ``np.sum`` forms for comparison.
"""
from __future__ import annotations

import numpy as np

from . import rpn_oracle

F32 = np.float32
PROTOCOLS = ("coco", "voc", "voc07")
DEFAULT_THRESHOLDS = np.asarray([x / 100 for x in range(50, 100, 5)], F32)
EPS = np.float64(2.0 ** -52)   # np.spacing(1)
IGNORE, CROWD = 1, 2


def default_thresholds(protocol):
    return DEFAULT_THRESHOLDS if protocol == "coco" else np.asarray([0.5], F32)


def score_key(scores):
    """uint32 keys that sort ascending in the order 'score descending by value': NaN first, +0 and -0 equal."""
    s = np.asarray(scores, F32).copy()
    s[s == 0] = F32(0)                  # -0 -> +0
    u = s.view(np.uint32)
    k = np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)
    k[np.isnan(s)] = np.uint32(0xFFFFFFFF)
    return (~k).astype(np.uint32)


def pair_ious(det, gt, crowd, protocol):
    """(n,m) float32: the matching score of every (detection, GT) pair."""
    det = np.asarray(det, F32).reshape(-1, 4)
    gt = np.asarray(gt, F32).reshape(-1, 4)
    iou = rpn_oracle.generate_iou_map(det[None], gt[None])[0]
    if protocol == "coco" and np.any(crowd):
        x_top = np.maximum(det[:, None, 1], gt[None, :, 1])
        y_top = np.maximum(det[:, None, 0], gt[None, :, 0])
        x_bot = np.minimum(det[:, None, 3], gt[None, :, 3])
        y_bot = np.minimum(det[:, None, 2], gt[None, :, 2])
        inter = np.maximum(x_bot - x_top, F32(0)) * np.maximum(y_bot - y_top, F32(0))
        darea = ((det[:, 2] - det[:, 0]) * (det[:, 3] - det[:, 1]))[:, None]
        with np.errstate(divide="ignore", invalid="ignore"):
            ciou = np.where(darea > F32(0), inter / np.where(darea > F32(0), darea, F32(1)), F32(0)).astype(F32)
        iou = np.where(np.asarray(crowd, bool)[None, :], ciou, iou)
    return np.where(iou > F32(0), iou, F32(0)).astype(F32)


def match_image_class(iou, ignore, crowd, gidx, thresholds, protocol):
    """Sequential matching of one (image, class): iou (n,m) with the detections in order, per-GT ignore / crowd / index.
    -> tp (n,T) bool, ig (n,T) bool."""
    n, m = iou.shape
    T = len(thresholds)
    tp = np.zeros((n, T), bool)
    ig = np.zeros((n, T), bool)
    if n == 0 or m == 0:
        return tp, ig
    rows = iou.tolist()
    ign = [bool(x) for x in ignore]
    crd = [bool(x) for x in crowd]
    gi = [int(x) for x in gidx]
    for ti, t in enumerate(np.asarray(thresholds, F32)):
        t = float(t)
        matched = [False] * m
        for d in range(n):
            r = rows[d]
            if protocol == "coco":
                best, bj = None, -1
                for phase in (False, True):   # non-ignored GT first, then the ignored ones
                    for j in range(m):
                        if ign[j] != phase or r[j] < t:
                            continue
                        if matched[j] and not (phase and crd[j]):
                            continue
                        if best is None or r[j] > best or (r[j] == best and gi[j] > gi[bj]):
                            best, bj = r[j], j
                    if bj >= 0:
                        break
                if bj >= 0:
                    matched[bj] = True
                    if ign[bj]:
                        ig[d, ti] = True
                    else:
                        tp[d, ti] = True
            else:
                s = max(r)
                j = min((gi[k], k) for k in range(m) if r[k] == s)[1]
                if not s > t:
                    continue
                if ign[j]:
                    ig[d, ti] = True
                elif not matched[j]:
                    tp[d, ti] = True
                    matched[j] = True
    return tp, ig


class MapAccumulator:
    """Running restatement: ``update`` per batch, ``compute`` -> (ap (C,T), recall (C,T), n_gt (C,))."""

    def __init__(self, num_classes, protocol="coco", thresholds=None, max_dets=100):
        assert protocol in PROTOCOLS
        self.C, self.protocol = int(num_classes), protocol
        self.thr = np.asarray(default_thresholds(protocol) if thresholds is None else thresholds, F32).reshape(-1)
        self.max_dets = int(max_dets) if protocol == "coco" else 0
        self.n_gt = np.zeros(self.C, np.int64)
        self.keys = [[] for _ in range(self.C)]   # per class: lists of arrays in insertion order
        self.tp = [[] for _ in range(self.C)]
        self.ig = [[] for _ in range(self.C)]

    def update(self, det_boxes, det_scores, det_classes, valid, gt_boxes, gt_labels, gt_flags=None):
        db = np.asarray(det_boxes, F32)
        ds = np.asarray(det_scores, F32)
        dc = np.asarray(det_classes, F32)
        gb = np.asarray(gt_boxes, F32)
        gl = np.asarray(gt_labels, np.int64)
        B, R = ds.shape
        G = gl.shape[1]
        gf = np.zeros((B, G), np.uint8) if gt_flags is None else np.asarray(gt_flags, np.uint8)
        for b in range(B):
            nv = R if valid is None else min(max(int(valid[b]), 0), R)
            cls = dc[b, :nv]
            ok = (cls == np.floor(cls)) & (cls >= 0) & (cls < self.C)
            rows = np.flatnonzero(ok)
            cl = cls[rows].astype(np.int64)
            key = score_key(ds[b, rows])
            order = np.lexsort((rows, key, cl))
            rows, cl, key = rows[order], cl[order], key[order]
            gok = (gl[b] >= 0) & (gl[b] < self.C)
            crowd_all = (gf[b] & CROWD) != 0
            ign_all = ((gf[b] & IGNORE) != 0) | crowd_all
            for c in np.unique(cl):
                sel = cl == c
                r_c, k_c = rows[sel], key[sel]
                if self.max_dets:
                    r_c, k_c = r_c[:self.max_dets], k_c[:self.max_dets]
                gsel = np.flatnonzero(gok & (gl[b] == c))
                iou = pair_ious(db[b, r_c], gb[b, gsel], crowd_all[gsel], self.protocol)
                crowd = crowd_all[gsel] if self.protocol == "coco" else np.zeros(gsel.size, bool)
                tp, ig = match_image_class(iou, ign_all[gsel], crowd, gsel, self.thr, self.protocol)
                self.keys[c].append(k_c)
                self.tp[c].append(tp)
                self.ig[c].append(ig)
            for c in range(self.C):
                self.n_gt[c] += int(np.sum(gok & (gl[b] == c) & ~ign_all))

    def entries(self, c):
        """-> (tp (N,T), ig (N,T)) of class c in dataset order."""
        T = self.thr.size
        if not self.keys[c]:
            return np.zeros((0, T), bool), np.zeros((0, T), bool)
        key = np.concatenate(self.keys[c])
        order = np.argsort(key, kind="stable")
        return np.concatenate(self.tp[c])[order], np.concatenate(self.ig[c])[order]

    def compute(self):
        T = self.thr.size
        ap = np.full((self.C, T), np.nan)
        rec = np.full((self.C, T), np.nan)
        for c in range(self.C):
            if self.n_gt[c] == 0:
                continue
            tp, ig = self.entries(c)
            for t in range(T):
                keep = ~ig[:, t]
                ap[c, t], rec[c, t] = average_precision(tp[keep, t], int(self.n_gt[c]), self.protocol)
        return ap, rec, self.n_gt.copy()


def ordered_sum(v):
    v = np.asarray(v, np.float64)
    return float(np.cumsum(v)[-1]) if v.size else 0.0   # np.add.accumulate adds in index order


def curves(tp, n_gt, protocol):
    """-> rc, pr, envelope (float64) of one (class, threshold) from its non-ignored entries in dataset order."""
    tp = np.asarray(tp, bool)
    TP = np.cumsum(tp).astype(np.float64)
    FP = np.cumsum(~tp).astype(np.float64)
    rc = TP / np.float64(n_gt)
    if protocol == "coco":
        pr = TP / ((FP + TP) + EPS)
    else:
        pr = TP / np.maximum(TP + FP, EPS)
    env = np.maximum.accumulate(pr[::-1])[::-1] if pr.size else pr
    return rc, pr, env


def average_precision(tp, n_gt, protocol):
    """-> (AP, recall) of one (class, threshold), every sum in the stated order."""
    rc, _, env = curves(tp, n_gt, protocol)
    last = float(rc[-1]) if rc.size else 0.0
    if protocol == "voc":
        prev = np.concatenate([[0.0], rc[:-1]])
        i = np.flatnonzero(rc > prev)
        return ordered_sum((rc[i] - prev[i]) * env[i]), last
    npts, step = (101, 0.01) if protocol == "coco" else (11, 0.1)
    r = np.arange(npts, dtype=np.float64) * step
    idx = np.searchsorted(rc, r, side="left")
    q = np.where(idx < rc.size, env[np.minimum(idx, max(rc.size - 1, 0))] if rc.size else 0.0, 0.0)
    if protocol == "coco":
        return ordered_sum(q) / 101.0, last
    return ordered_sum(q / 11.0), last


def pycocotools_ap(tp, n_gt):
    """pycocotools ``accumulate`` for one (class, threshold, area, maxDets), as written there."""
    tps = np.asarray(tp, bool)
    fps = ~tps
    tp_sum = np.cumsum(tps).astype(dtype=float)
    fp_sum = np.cumsum(fps).astype(dtype=float)
    nd = len(tp_sum)
    rc = tp_sum / n_gt
    pr = tp_sum / (fp_sum + tp_sum + np.spacing(1))
    recThrs = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
    q = np.zeros((len(recThrs),))
    pr = pr.tolist()
    q = q.tolist()
    for i in range(nd - 1, 0, -1):
        if pr[i] > pr[i - 1]:
            pr[i - 1] = pr[i]
    inds = np.searchsorted(rc, recThrs, side="left")
    try:
        for ri, pi in enumerate(inds):
            q[ri] = pr[pi]
    except IndexError:
        pass
    return float(np.mean(np.array(q)))


def devkit_ap(tp, n_gt, use_07_metric=False):
    """The VOC devkit's ``voc_eval`` tail and ``voc_ap``, as written there."""
    tp = np.asarray(tp, bool).astype(float)
    fp = 1.0 - tp
    fp = np.cumsum(fp)
    tp = np.cumsum(tp)
    rec = tp / float(n_gt)
    prec = tp / np.maximum(tp + fp, np.finfo(np.float64).eps)
    if use_07_metric:
        ap = 0.
        for t in np.arange(0., 1.1, 0.1):
            if np.sum(rec >= t) == 0:
                p = 0
            else:
                p = np.max(prec[rec >= t])
            ap = ap + p / 11.
        return float(ap)
    mrec = np.concatenate(([0.], rec, [1.]))
    mpre = np.concatenate(([0.], prec, [0.]))
    for i in range(mpre.size - 1, 0, -1):
        mpre[i - 1] = np.maximum(mpre[i - 1], mpre[i])
    i = np.where(mrec[1:] != mrec[:-1])[0]
    return float(np.sum((mrec[i + 1] - mrec[i]) * mpre[i + 1]))


def class_mean(ap, n_gt):
    """(C,T) -> (T,) mean over the classes with n_gt > 0, added in class order; NaN when there are none."""
    ap = np.asarray(ap, np.float64)
    sel = np.flatnonzero(np.asarray(n_gt) > 0)
    if sel.size == 0:
        return np.full(ap.shape[1], np.nan)
    return np.cumsum(ap[sel], axis=0)[-1] / sel.size


def detection_map(det_boxes, det_scores, det_classes, valid, gt_boxes, gt_labels, gt_flags=None, *, num_classes,
                  protocol="coco", thresholds=None, max_dets=100):
    """One-shot -> (ap (C,T), recall (C,T), n_gt (C,), map (T,), mean_ap)."""
    acc = MapAccumulator(num_classes, protocol, thresholds, max_dets)
    acc.update(det_boxes, det_scores, det_classes, valid, gt_boxes, gt_labels, gt_flags)
    ap, rec, n_gt = acc.compute()
    m = class_mean(ap, n_gt)
    return ap, rec, n_gt, m, float(np.cumsum(m)[-1] / m.size)

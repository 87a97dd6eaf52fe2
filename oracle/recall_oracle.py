"""NumPy restatement of proposal recall (tfrpn_proposal_recall, include/tfrpn.h).  TEST INFRASTRUCTURE, not product.

The reference has no evaluation; this restates the definition Detectron's ``evaluate_box_proposals`` and mmdet's
``eval_recalls`` use, with their tie rule made explicit:
  * a GT box is valid when its float32 area (y2-y1)*(x2-x1) is > 0 and, with labels, its label is >= 0;
  * image b takes part with its first min(k, valid[b], P) proposals (rank order; valid clamped to [0, P]);
  * a pair scores the IoU of ``rpn_oracle.generate_iou_map`` (proposal = bboxes), NaN / negative / -0 read as +0;
  * greedy: repeatedly take the remaining pair of largest score, ties to the lowest GT index and then the lowest
    rank, until no remaining pair scores > 0; that score is the GT's IoU, valid GT never taken get 0;
  * coverage: a GT's IoU is its best score (a column maximum, no exclusivity);
  * hits[l][t] = #valid GT with IoU >= thr[t] (float32 compare); recall = hits / n_gt; AR = mean over t.
"""
from __future__ import annotations

import numpy as np

from . import rpn_oracle

F32 = np.float32
DEFAULT_THRESHOLDS = np.asarray([x / 100 for x in range(50, 100, 5)], F32)
DEFAULT_LIMITS = (100, 300, 1000)


def valid_gt(gt_boxes, gt_labels=None):
    """(B,G) bool: positive float32 area and, with labels, label >= 0."""
    g = np.asarray(gt_boxes, F32)
    area = (g[..., 2] - g[..., 0]) * (g[..., 3] - g[..., 1])
    ok = area > F32(0)
    if gt_labels is not None:
        ok &= np.asarray(gt_labels) >= 0
    return ok


def pair_scores(proposals, gt_boxes):
    """(k,G) scores of one image: generate_iou_map with NaN, negative and -0 read as +0."""
    iou = rpn_oracle.generate_iou_map(np.asarray(proposals, F32)[None], np.asarray(gt_boxes, F32)[None])[0]
    return np.where(iou > F32(0), iou, F32(0)).astype(F32)


def match_greedy(S):
    """Detectron's greedy loop on the (k,G) score matrix S (columns of valid GT only) -> (G,) matched IoU.

    Detectron takes max_overlaps = overlaps.max(axis=0) in every round, picks the GT of the largest one (argmax: the
    lowest GT on ties) and the row of its maximum (argmax: the lowest rank), records the score and sets that row and
    column to -1.  Removing a row changes only the columns whose maximum sat on it, so only those are recomputed here:
    the same rounds, in time proportional to the work they change."""
    S = np.array(S, F32, copy=True)
    k, G = S.shape
    out = np.zeros(G, F32)
    if k == 0 or G == 0:
        return out
    colmax = S.max(axis=0)
    colarg = S.argmax(axis=0)
    live = np.ones(G, bool)
    while True:
        cand = np.where(live, colmax, F32(-1))
        g = int(cand.argmax())
        if not cand[g] > 0:
            break
        p = int(colarg[g])
        out[g] = S[p, g]
        live[g] = False
        S[p, :] = F32(-1)
        S[:, g] = F32(-1)
        stale = np.flatnonzero(live & (colarg == p))
        if stale.size:
            colmax[stale] = S[:, stale].max(axis=0)
            colarg[stale] = S[:, stale].argmax(axis=0)
    return out


def match_coverage(S):
    """Best score per GT over the proposals (Hosang et al.; round 0 of the greedy loop)."""
    S = np.asarray(S, F32)
    if S.shape[0] == 0:
        return np.zeros(S.shape[1], F32)
    return S.max(axis=0)


def gt_ious(proposals, gt_boxes, gt_labels=None, valid=None, limits=DEFAULT_LIMITS, matching="greedy"):
    """(L,B,G) float32: the matched IoU of every GT at every limit, -1 for invalid GT."""
    prop = np.asarray(proposals, F32)
    gt = np.asarray(gt_boxes, F32)
    B, P = prop.shape[:2]
    G = gt.shape[1]
    ok = valid_gt(gt, gt_labels)
    match = {"greedy": match_greedy, "coverage": match_coverage}[matching]
    out = np.full((len(limits), B, G), -1, F32)
    for b in range(B):
        nv = P if valid is None else min(max(int(valid[b]), 0), P)
        cols = np.flatnonzero(ok[b])
        S = pair_scores(prop[b, :min(max(int(v) for v in limits), nv)], gt[b, cols])   # the limits take its first rows
        for li, lim in enumerate(limits):
            out[li, b, cols] = match(S[:min(int(lim), nv)])
    return out


def recall_counts(gt_iou, thresholds=DEFAULT_THRESHOLDS):
    """gt_iou (L,B,G) -> int64 counts (L*T + 1): hits[l][t] row-major, then the number of valid GT."""
    iou = np.asarray(gt_iou, F32)
    thr = np.asarray(thresholds, F32)
    hits = (iou[:, None] >= thr[None, :, None, None]).reshape(iou.shape[0], thr.size, -1).sum(axis=-1)
    n_gt = int((iou[0] >= 0).sum()) if iou.shape[0] else 0
    return np.concatenate([hits.reshape(-1), [n_gt]]).astype(np.int64)


def proposal_recall(proposals, gt_boxes, gt_labels=None, valid=None, thresholds=DEFAULT_THRESHOLDS,
                    limits=DEFAULT_LIMITS, matching="greedy"):
    """-> (recall (L,T) float64, AR (L,), counts (L*T+1,) int64, gt_iou (L,B,G))."""
    iou = gt_ious(proposals, gt_boxes, gt_labels, valid, limits, matching)
    counts = recall_counts(iou, thresholds)
    L, T = len(limits), len(thresholds)
    with np.errstate(invalid="ignore"):
        recall = counts[:-1].reshape(L, T) / np.float64(counts[-1])   # 0 / 0 = NaN without valid GT
    return recall, recall.mean(axis=1), counts, iou

"""NumPy restatement of the second stage's RoI target assignment (tfrpn_roi_targets, include/tfrpn.h).
TEST INFRASTRUCTURE, not product.

The reference has no second stage; the rules follow Detectron (fg at IoU >= 0.5, bg in [lo, 0.5), 25 % fg of 512,
GT boxes appended to the proposals):
  * GT g takes part iff 1 <= label < C; row n < P is proposal n (taking part iff n < clamp(valid, 0, P)), row P + g
    (append_gt) is GT box g (taking part iff GT g does);
  * a pair scores ``rpn_oracle.generate_iou_map`` (row = bboxes), NaN / negative / -0 read as +0;
  * a taking-part row matches m = its best score over the taking-part GT and j = the lowest GT with that score
    (m = +0, j = -1 without a taking-part GT);
  * fg: m >= fg_iou_threshold; bg: not fg and bg_iou_low <= m < bg_iou_high;
  * fg kept: all if at most total_pos, else the first total_pos by (Philox word 2 descending, row ascending);
    bg kept: the same with quota S - #fg kept and word 3 (``rpn_oracle.sampling_keys``);
  * outputs: kept fg rows ascending, kept bg rows ascending, padding (box 0, label -1, deltas 0, src -1); fg deltas
    are ``rpn_oracle.get_deltas_from_bboxes(row, gt[j]) / variances``.
"""
from __future__ import annotations

import numpy as np

from . import rpn_oracle

F32 = np.float32


def _sample(cand, quota, P_rows, image_index, seed, offset, stream):
    """bool mask over the rows: the kept subset of the candidate rows ``cand`` (ascending indices)."""
    keep = np.zeros(P_rows, bool)
    if quota <= 0 or cand.size == 0:
        return keep
    if cand.size <= quota:
        keep[cand] = True
        return keep
    keys = rpn_oracle.sampling_keys(P_rows, image_index, seed, offset, stream)[cand]
    order = np.lexsort((cand, -keys.astype(np.int64)))   # key descending, then row ascending
    keep[cand[order[:quota]]] = True
    return keep


def match_rows(rows, part, gt, gt_part):
    """(m (P',) float32, j (P',) int32) of one image's rows against its GT; -1.0 / -1 for rows that take no part."""
    Pp = rows.shape[0]
    m = np.full(Pp, F32(-1), F32)
    j = np.full(Pp, -1, np.int32)
    cols = np.flatnonzero(gt_part)
    if cols.size == 0:
        m[part] = F32(0)
        return m, j
    iou = rpn_oracle.generate_iou_map(rows[None], gt[cols][None])[0]          # (P', G_part)
    s = np.where(iou > F32(0), iou, F32(0)).astype(F32)
    best = s.argmax(axis=1)                                                   # the first maximum: the lowest GT
    m[part] = s[np.arange(Pp), best][part]
    j[part] = cols[best][part]
    return m, j


def roi_targets(rois, gt_boxes, gt_labels, valid=None, *, num_classes, total_pos=128, total_neg=384,
                fg_iou_threshold=0.5, bg_iou_high=0.5, bg_iou_low=0.0, variances=(0.1, 0.1, 0.2, 0.2),
                append_gt=True, seed=0, offset=0, image_offset=0):
    """-> dict of rois (B,S,4), labels (B,S), deltas (B,S,4), src (B,S), counts (B,2), max_iou (B,P'), argmax (B,P'),
    fg_cand / bg_cand / fg_keep / bg_keep (B,P') bool."""
    rois = np.asarray(rois, F32)
    gt = np.asarray(gt_boxes, F32)
    lab = np.asarray(gt_labels).astype(np.int64)
    B, P = rois.shape[:2]
    G = gt.shape[1]
    S = int(total_pos) + int(total_neg)
    Pp = P + (G if append_gt else 0)
    var = np.asarray(variances, F32)
    fg_thr, lo, hi = F32(fg_iou_threshold), F32(bg_iou_low), F32(bg_iou_high)
    out = dict(rois=np.zeros((B, S, 4), F32), labels=np.full((B, S), -1, np.int32), deltas=np.zeros((B, S, 4), F32),
               src=np.full((B, S), -1, np.int32), counts=np.zeros((B, 2), np.int32),
               max_iou=np.zeros((B, Pp), F32), argmax=np.zeros((B, Pp), np.int32))
    for k in ("fg_cand", "bg_cand", "fg_keep", "bg_keep"):
        out[k] = np.zeros((B, Pp), bool)
    for b in range(B):
        gt_part = (lab[b] >= 1) & (lab[b] < num_classes)
        nv = P if valid is None else min(max(int(valid[b]), 0), P)
        rows = np.concatenate([rois[b], gt[b]]) if append_gt else rois[b]
        part = np.concatenate([np.arange(P) < nv, gt_part]) if append_gt else np.arange(P) < nv
        m, j = match_rows(rows, part, gt[b], gt_part)
        fg = part & (m >= fg_thr)
        bg = part & ~fg & (m >= lo) & (m < hi)
        fg_keep = _sample(np.flatnonzero(fg), int(total_pos), Pp, image_offset + b, seed, offset, 2)
        nfg = int(fg_keep.sum())
        bg_keep = _sample(np.flatnonzero(bg), S - nfg, Pp, image_offset + b, seed, offset, 3)
        fr, br = np.flatnonzero(fg_keep), np.flatnonzero(bg_keep)
        kept = np.concatenate([fr, br])
        out["rois"][b, :kept.size] = rows[kept]
        out["labels"][b, :fr.size] = lab[b, j[fr]]
        out["labels"][b, fr.size:kept.size] = 0
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            out["deltas"][b, :fr.size] = rpn_oracle.get_deltas_from_bboxes(rows[fr], gt[b, j[fr]]) / var
        out["src"][b, :kept.size] = kept
        out["counts"][b] = (fr.size, kept.size)
        out["max_iou"][b], out["argmax"][b] = m, j
        out["fg_cand"][b], out["bg_cand"][b], out["fg_keep"][b], out["bg_keep"][b] = fg, bg, fg_keep, bg_keep
    return out

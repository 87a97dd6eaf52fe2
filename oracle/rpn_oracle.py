"""NumPy-float32 restatement of the tf-rpn box hot path.  TEST INFRASTRUCTURE, not product.

PARITY UNPINNED against real TensorFlow (no TF in this image; the reference has no tests).
Pinned instead against the reference's own Python source run over ``oracle/tf_numpy_shim``
(``tests/golden``) and the IEEE-exact KATs of SURVEY.md 8(c).

Every function cites the reference lines it restates (paths relative to /root/reference).
All arithmetic is explicit ``np.float32`` in the reference's op order; NumPy never
FMA-contracts, so thresholds (``> 0.7``, ``< 0.3``, NMS ``> thr``) flip exactly where an
op-by-op TensorFlow evaluation would.  Behaviour that lives inside TensorFlow (argmax /
top_k tie rules, the combined-NMS algorithm) is restated from TF's published kernels and is
marked [TF-internal].
"""
from __future__ import annotations

import numpy as np

F32 = np.float32

# --------------------------------------------------------------------------------------
# hyper params (utils/train_utils.py:5-38)
# --------------------------------------------------------------------------------------
RPN = {
    "vgg16": {"img_size": 500, "feature_map_shape": 31,
              "anchor_ratios": [1., 2., 1. / 2.], "anchor_scales": [128, 256, 512]},
    "mobilenet_v2": {"img_size": 500, "feature_map_shape": 32,
                     "anchor_ratios": [1., 2., 1. / 2.], "anchor_scales": [128, 256, 512]},
}


def get_hyper_params(backbone, **kwargs):
    """utils/train_utils.py:20-38 (returns a copy instead of mutating the module dict)."""
    hp = dict(RPN[backbone])
    hp["test_nms_topn"] = 300
    hp["total_pos_bboxes"] = 128
    hp["total_neg_bboxes"] = 128
    hp["variances"] = [0.1, 0.1, 0.2, 0.2]
    for key, value in kwargs.items():
        if key in hp and value:
            hp[key] = value
    hp["anchor_count"] = len(hp["anchor_ratios"]) * len(hp["anchor_scales"])
    return hp


def _pair(v):
    """int -> (v, v); (h, w) -> (h, w).  Square is the only case the reference expresses."""
    if isinstance(v, (tuple, list)):
        return int(v[0]), int(v[1])
    return int(v), int(v)


def clip01(x):
    """The library's clip to [0, 1] (include/tfrpn.h): min(max(x, 0), 1) with NaN-ignoring max / min, so NaN -> 0.
    np.clip would keep NaN.  TF's GPU minimum / maximum also send NaN to the other operand; its CPU kernels keep it."""
    return np.fmin(np.fmax(np.asarray(x, F32), F32(0)), F32(1))


# --------------------------------------------------------------------------------------
# anchors (utils/bbox_utils.py:3-46)
# --------------------------------------------------------------------------------------
def generate_base_anchors(hp):
    """utils/bbox_utils.py:3-21.

    dtype walk: ``scale /= img_size`` and ``scale**2/ratio`` are Python float64 (:16,:18);
    ``tf.sqrt`` converts the quotient to f32 and takes an f32 sqrt (:18); ``h = w*ratio``
    multiplies by f32(ratio) (:19); ``/2`` is exact.  Loop order scale-outer, ratio-inner.
    Non-square extension (SURVEY 8d): per-axis normalisation, identical when square.
    """
    img_h, img_w = _pair(hp["img_size"])
    out = []
    for scale in hp["anchor_scales"]:
        sw = scale / img_w
        sh = scale / img_h
        for ratio in hp["anchor_ratios"]:
            w = np.sqrt(F32(sw ** 2 / ratio))
            h = np.sqrt(F32(sh ** 2 / ratio)) * F32(ratio)
            out.append([-h / F32(2), -w / F32(2), h / F32(2), w / F32(2)])
    return np.asarray(out, dtype=F32)


def generate_anchors(hp):
    """utils/bbox_utils.py:23-46.

    ``tf.range(0,F)/F + stride/2`` is evaluated in float64 ([TF-internal]: int32 truediv
    promotes to f64) and then cast to f32 (:35-36).  meshgrid => flat cell c = i*FW + j with
    y = grid[i], x = grid[j] (:38-40); anchor index = c*A + a (:44-45); clip to [0,1] (:46).
    """
    fh, fw = _pair(hp["feature_map_shape"])
    gy = (np.arange(fh, dtype=np.int32) / fh + (1 / fh) / 2).astype(F32)
    gx = (np.arange(fw, dtype=np.int32) / fw + (1 / fw) / 2).astype(F32)
    grid_x, grid_y = np.meshgrid(gx, gy)
    fx, fy = grid_x.reshape(-1), grid_y.reshape(-1)
    grid_map = np.stack([fy, fx, fy, fx], axis=-1)
    base = generate_base_anchors(hp)
    anchors = base.reshape(1, -1, 4) + grid_map.reshape(-1, 1, 4)
    anchors = anchors.reshape(-1, 4).astype(F32)
    return clip01(anchors)


# --------------------------------------------------------------------------------------
# decode / encode / IoU (utils/bbox_utils.py:72-150)
# --------------------------------------------------------------------------------------
def get_bboxes_from_deltas(anchors, deltas):
    """utils/bbox_utils.py:72-96.  No clip, no exp clamp."""
    anchors = np.asarray(anchors, F32)
    deltas = np.asarray(deltas, F32)
    half = F32(0.5)
    aw = anchors[..., 3] - anchors[..., 1]
    ah = anchors[..., 2] - anchors[..., 0]
    acx = anchors[..., 1] + half * aw
    acy = anchors[..., 0] + half * ah
    w = np.exp(deltas[..., 3]) * aw
    h = np.exp(deltas[..., 2]) * ah
    cx = (deltas[..., 1] * aw) + acx
    cy = (deltas[..., 0] * ah) + acy
    y1 = cy - (half * h)
    x1 = cx - (half * w)
    y2 = h + y1
    x2 = w + x1
    return np.stack([y1, x1, y2, x2], axis=-1).astype(F32)


def get_deltas_from_bboxes(bboxes, gt_boxes):
    """utils/bbox_utils.py:98-124."""
    bboxes = np.asarray(bboxes, F32)
    gt_boxes = np.asarray(gt_boxes, F32)
    half = F32(0.5)
    bw = bboxes[..., 3] - bboxes[..., 1]
    bh = bboxes[..., 2] - bboxes[..., 0]
    bcx = bboxes[..., 1] + half * bw
    bcy = bboxes[..., 0] + half * bh
    gw = gt_boxes[..., 3] - gt_boxes[..., 1]
    gh = gt_boxes[..., 2] - gt_boxes[..., 0]
    gcx = gt_boxes[..., 1] + half * gw
    gcy = gt_boxes[..., 0] + half * gh
    bw = np.where(bw == 0, F32(1e-3), bw)
    bh = np.where(bh == 0, F32(1e-3), bh)
    with np.errstate(divide="ignore", invalid="ignore"):
        dx = np.where(gw == 0, F32(0), (gcx - bcx) / bw)
        dy = np.where(gh == 0, F32(0), (gcy - bcy) / bh)
        dw = np.where(gw == 0, F32(0), np.log(gw / bw))
        dh = np.where(gh == 0, F32(0), np.log(gh / bh))
    return np.stack([dy, dx, dh, dw], axis=-1).astype(F32)


def generate_iou_map(bboxes, gt_boxes):
    """utils/bbox_utils.py:126-150.  bboxes (N,4) or (B,N,4); gt (B,G,4) -> (B,N,G).

    Op order: areas (:138-139); max/min corners (:141-144); inter = max(dx,0)*max(dy,0)
    with the x factor first (:146); union = (bbox_area + gt_area) - inter (:148); divide
    (:150).  No epsilon: 0/0 -> NaN when both boxes are degenerate.
    """
    b = np.asarray(bboxes, F32)
    g = np.asarray(gt_boxes, F32)
    if b.ndim == 2:
        b = b[None]
    by1, bx1, by2, bx2 = (b[..., i:i + 1] for i in range(4))          # (B|1,N,1)
    gy1, gx1, gy2, gx2 = (g[..., i][:, None, :] for i in range(4))    # (B,1,G)
    gt_area = (gy2 - gy1) * (gx2 - gx1)
    bbox_area = (by2 - by1) * (bx2 - bx1)
    x_top = np.maximum(bx1, gx1)
    y_top = np.maximum(by1, gy1)
    x_bot = np.minimum(bx2, gx2)
    y_bot = np.minimum(by2, gy2)
    inter = np.maximum(x_bot - x_top, F32(0)) * np.maximum(y_bot - y_top, F32(0))
    union = (bbox_area + gt_area) - inter
    with np.errstate(divide="ignore", invalid="ignore"):
        return (inter / union).astype(F32)


def normalize_bboxes(bboxes, height, width):
    """utils/bbox_utils.py:152-166."""
    b = np.asarray(bboxes, F32)
    return np.stack([b[..., 0] / F32(height), b[..., 1] / F32(width),
                     b[..., 2] / F32(height), b[..., 3] / F32(width)], axis=-1)


def denormalize_bboxes(bboxes, height, width):
    """utils/bbox_utils.py:168-182 (tf.round = round-half-to-even = np.rint)."""
    b = np.asarray(bboxes, F32)
    return np.rint(np.stack([b[..., 0] * F32(height), b[..., 1] * F32(width),
                             b[..., 2] * F32(height), b[..., 3] * F32(width)], axis=-1))


# --------------------------------------------------------------------------------------
# counter-based RNG (replaces tf.random.uniform, utils/train_utils.py:60)
# --------------------------------------------------------------------------------------
PHILOX_M0 = np.uint64(0xD2511F53)
PHILOX_M1 = np.uint64(0xCD9E8D57)
PHILOX_W0 = 0x9E3779B9
PHILOX_W1 = 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11).  Counters: uint32 arrays; key: two ints."""
    c0 = np.asarray(c0, np.uint64) & _MASK32
    c1 = np.asarray(c1, np.uint64) & _MASK32
    c2 = np.asarray(c2, np.uint64) & _MASK32
    c3 = np.asarray(c3, np.uint64) & _MASK32
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = PHILOX_M0 * c0
        p1 = PHILOX_M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK32
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0)
        k0 = (k0 + PHILOX_W0) & 0xFFFFFFFF
        k1 = (k1 + PHILOX_W1) & 0xFFFFFFFF
    return (c0.astype(np.uint32), c1.astype(np.uint32), c2.astype(np.uint32), c3.astype(np.uint32))


def sampling_keys(n_items, image_index, seed, offset, stream):
    """32-bit sampling key of item n of (global) image ``image_index``.

    counter = (n, image_index, offset_lo, offset_hi); key = (seed_lo, seed_hi);
    stream 0 (positives) takes output word 0, stream 1 (negatives) word 1.
    """
    n = np.arange(n_items, dtype=np.uint64)
    out = philox4x32_10(n, np.uint64(image_index), np.uint64(offset & 0xFFFFFFFF),
                        np.uint64((offset >> 32) & 0xFFFFFFFF),
                        seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return out[stream]


def randomly_select_xyz_mask(mask, select_xyz, seed=0, offset=0, stream=0, image_offset=0):
    """Semantics of utils/train_utils.py:50-65 with a counter RNG.

    The reference ranks ``mask * r`` descending (argsort-desc => [TF-internal] ties to the
    lower index, :62-63) and keeps rank < select (:64) AND mask (:65): i.e. keep
    min(#True, select) True entries per row.  Here r is the Philox key above (not
    ``tf.random``), ranked by (key desc, index asc) among the True entries only, so the
    reference's key-collision bias (maxval = 10*max(select)) is not reproduced.
    ``select_xyz`` broadcasts over the batch like the reference's (1,) constant (:123).
    """
    mask = np.asarray(mask, bool)
    B, N = mask.shape
    select = np.broadcast_to(np.asarray(select_xyz, np.int64).reshape(-1), (B,))
    out = np.zeros_like(mask)
    for b in range(B):
        cand = np.flatnonzero(mask[b])
        q = int(select[b])
        if q <= 0 or cand.size == 0:
            continue
        if cand.size <= q:
            out[b, cand] = True
            continue
        keys = sampling_keys(N, image_offset + b, seed, offset, stream)[cand]
        order = np.lexsort((cand, -keys.astype(np.int64)))   # key desc, then index asc
        out[b, cand[order[:q]]] = True
    return out


# --------------------------------------------------------------------------------------
# target assignment (utils/train_utils.py:84-144)
# --------------------------------------------------------------------------------------
def calculate_rpn_actual_outputs(anchors, gt_boxes, gt_labels, hp, seed=0, offset=0,
                                 image_offset=0, return_debug=False):
    """utils/train_utils.py:84-144.

    [TF-internal] tf.argmax returns the FIRST maximal index and NaN never wins a '>'.
    Thresholds 0.7 / 0.3 are the reference's literals (:114,:128) unless the optional
    extension keys ``pos_iou_threshold`` / ``neg_iou_threshold`` are present.
    """
    anchors = np.asarray(anchors, F32)
    gt_boxes = np.asarray(gt_boxes, F32)
    gt_labels = np.asarray(gt_labels)
    B = gt_boxes.shape[0]
    fh, fw = _pair(hp["feature_map_shape"])
    A = hp["anchor_count"]
    total_pos = int(hp["total_pos_bboxes"])
    total_neg = int(hp["total_neg_bboxes"])
    variances = np.asarray(hp["variances"], F32)
    pos_thr = F32(hp.get("pos_iou_threshold", 0.7))
    neg_thr = F32(hp.get("neg_iou_threshold", 0.3))

    iou = generate_iou_map(anchors, gt_boxes)                       # :106
    iou_cmp = np.where(np.isnan(iou), F32(-np.inf), iou)            # NaN never wins
    argmax_row = iou_cmp.argmax(axis=2).astype(np.int32)            # :108 (per anchor)
    argmax_col = iou_cmp.argmax(axis=1).astype(np.int32)            # :110 (per GT)
    merged = iou_cmp.max(axis=2)                                    # :112
    pos_pre = merged > pos_thr                                      # :114
    valid = gt_labels != -1                                         # :116
    bb, gg = np.nonzero(valid)
    pos_pre = pos_pre.copy()
    pos_pre[bb, argmax_col[bb, gg]] = True                          # :117-122
    pos = randomly_select_xyz_mask(pos_pre, [total_pos], seed, offset, 0, image_offset)  # :123
    pos_count = pos.sum(axis=-1).astype(np.int32)                   # :125
    neg_quota = (total_pos + total_neg) - pos_count                 # :126
    neg_pre = (merged < neg_thr) & ~pos                             # :128
    neg = randomly_select_xyz_mask(neg_pre, neg_quota, seed, offset, 1, image_offset)    # :129
    labels = np.where(pos, F32(1), F32(-1)) + neg.astype(F32)       # :131-133
    gt_map = np.take_along_axis(gt_boxes, argmax_row[..., None].astype(np.int64), axis=1)  # :135
    expanded = np.where(pos[..., None], gt_map, F32(0))             # :137
    deltas = get_deltas_from_bboxes(anchors, expanded) / variances  # :139
    labels = labels.reshape(B, fh, fw, A)                           # :142
    if return_debug:
        dbg = dict(argmax_row=argmax_row, argmax_col=argmax_col, max_iou=merged.astype(F32),
                   pos_pre=pos_pre, neg_pre=neg_pre, pos=pos, neg=neg,
                   pos_count=pos_count, neg_count=neg.sum(-1).astype(np.int32))
        return deltas.astype(F32), labels.astype(F32), dbg
    return deltas.astype(F32), labels.astype(F32)


# --------------------------------------------------------------------------------------
# top-k (predictor.py:58-60) and combined NMS (utils/bbox_utils.py:48-70)
# --------------------------------------------------------------------------------------
def top_k(scores, k):
    """tf.nn.top_k [TF-internal]: values descending, equal values -> lower index first."""
    scores = np.asarray(scores, F32)
    idx = np.argsort(-scores.astype(np.float64), axis=-1, kind="stable")[..., :k].astype(np.int32)
    return np.take_along_axis(scores, idx.astype(np.int64), axis=-1), idx


def _nms_iou_vs(box, sel):
    """TF combined-NMS IOU ([TF-internal] non_max_suppression_op.cc): canonicalise corners,
    0 when either area <= 0, inter/(a_i + a_j - inter)."""
    ymin_i, ymax_i = min(box[0], box[2]), max(box[0], box[2])
    xmin_i, xmax_i = min(box[1], box[3]), max(box[1], box[3])
    ymin_j = np.minimum(sel[:, 0], sel[:, 2]); ymax_j = np.maximum(sel[:, 0], sel[:, 2])
    xmin_j = np.minimum(sel[:, 1], sel[:, 3]); xmax_j = np.maximum(sel[:, 1], sel[:, 3])
    area_i = F32(F32(ymax_i - ymin_i) * F32(xmax_i - xmin_i))
    area_j = (ymax_j - ymin_j) * (xmax_j - xmin_j)
    iy = np.maximum(np.minimum(ymax_i, ymax_j) - np.maximum(ymin_i, ymin_j), F32(0))
    ix = np.maximum(np.minimum(xmax_i, xmax_j) - np.maximum(xmin_i, xmin_j), F32(0))
    inter = iy * ix
    with np.errstate(divide="ignore", invalid="ignore"):
        iou = inter / ((area_i + area_j) - inter)
    return np.where((area_i <= 0) | (area_j <= 0), F32(0), iou)


def combined_non_max_suppression(boxes, scores, max_output_size_per_class, max_total_size,
                                 iou_threshold=0.5, score_threshold=float("-inf"),
                                 pad_per_class=False, clip_boxes=True, return_indices=False):
    """tf.image.combined_non_max_suppression [TF-internal].

    boxes (B,K,q,4) with q = 1 (boxes shared by the classes) or q = C, scores (B,K,C).  Per image and class:
    greedy in score order (equal scores: lower index first -- TF's heap order for ties is unspecified; this is
    the documented rule), suppress iff IoU > iou_threshold (strict), stop at max_output_size_per_class.  The
    per-class results are then merged by score (descending; TF uses an unstable std::sort, the documented rule
    here: equal scores -> lower class id first, then the class's own order) and truncated to max_total_size.
    Output rows: max_total_size, or with pad_per_class min(max_total_size, max_output_size_per_class * C); zero
    padded; OUTPUT boxes clipped to [0,1] when clip_boxes.  nmsed_classes holds the class ids as floats.  Also
    returns the kept box indices (-1 padded) when ``return_indices`` (TF returns none).
    """
    boxes = np.asarray(boxes, F32)
    scores = np.asarray(scores, F32)
    assert boxes.ndim == 4 and scores.ndim == 3
    B, K, C = scores.shape
    q = boxes.shape[2]
    assert q in (1, C), "boxes must be (B,K,1,4) or (B,K,C,4)"
    per_class = int(max_output_size_per_class)
    total = int(max_total_size)
    out_n = total if not pad_per_class else min(total, per_class * C)
    thr = F32(iou_threshold)
    sthr = F32(score_threshold)
    nb = np.zeros((B, out_n, 4), F32); ns = np.zeros((B, out_n), F32)
    nc = np.zeros((B, out_n), F32); nv = np.zeros((B,), np.int32)
    ni = np.full((B, out_n), -1, np.int32)
    for b in range(B):
        cand = []                                   # (score, class, position in the class's keep list, box index)
        for c in range(C):
            bx = boxes[b, :, c if q > 1 else 0, :]
            sc = scores[b, :, c]
            order = np.argsort(-sc.astype(np.float64), kind="stable")
            order = order[sc[order] > sthr]
            sel = []
            for i in order:
                if len(sel) >= per_class:
                    break
                if sel and np.any(_nms_iou_vs(bx[i], bx[sel]) > thr):
                    continue
                sel.append(int(i))
            cand.extend((float(sc[i]), c, pos, i) for pos, i in enumerate(sel))
        cand.sort(key=lambda t: (-t[0], t[1], t[2]))
        cand = cand[:min(out_n, total)]
        nv[b] = len(cand)
        for r, (_, c, _, i) in enumerate(cand):
            kept = boxes[b, i, c if q > 1 else 0, :]
            nb[b, r] = clip01(kept) if clip_boxes else kept
            ns[b, r] = scores[b, i, c]
            nc[b, r] = F32(c)
            ni[b, r] = i
    if return_indices:
        return nb, ns, nc, nv, ni
    return nb, ns, nc, nv


# --------------------------------------------------------------------------------------
# composed proposal pipeline (SURVEY 8a row P; predictor.py:52-60 + bbox_utils.py:48-70)
# --------------------------------------------------------------------------------------
def generate_proposals(rpn_reg, rpn_cls, anchors, hp, pre_nms_topn=None, post_nms_topn=None,
                       nms_iou_threshold=None):
    """deltas*variances -> decode -> clip[0,1] -> top-k(pre_nms_topn) -> gather ->
    combined NMS(post_nms_topn, thr).  Returns boxes (B,P,4), scores (B,P), valid (B,),
    keep_idx (B,P) int32 indices into N (-1 padded)."""
    rpn_reg = np.asarray(rpn_reg, F32)
    rpn_cls = np.asarray(rpn_cls, F32)
    B = rpn_reg.shape[0]
    deltas = rpn_reg.reshape(B, -1, 4)                                # predictor.py:52
    scores = rpn_cls.reshape(B, -1)                                   # predictor.py:53
    N = scores.shape[1]
    k = min(int(pre_nms_topn if pre_nms_topn is not None else hp.get("pre_nms_topn", 6000)), N)
    post = int(post_nms_topn if post_nms_topn is not None else hp["test_nms_topn"])
    thr = nms_iou_threshold if nms_iou_threshold is not None else hp.get("nms_iou_threshold", 0.7)
    deltas = deltas * np.asarray(hp["variances"], F32)                # predictor.py:55
    boxes = get_bboxes_from_deltas(anchors, deltas)                   # predictor.py:56
    boxes = clip01(boxes)
    top_scores, top_idx = top_k(scores, k)                            # predictor.py:58
    top_boxes = np.take_along_axis(boxes, top_idx[..., None].astype(np.int64), axis=1)  # :60
    nb, ns, _, nv, ni = combined_non_max_suppression(
        top_boxes.reshape(B, k, 1, 4), top_scores.reshape(B, k, 1),
        max_output_size_per_class=post, max_total_size=post, iou_threshold=thr,
        return_indices=True)
    keep = np.where(ni >= 0, np.take_along_axis(top_idx, np.maximum(ni, 0).astype(np.int64), axis=1), -1)
    return nb, ns, nv, keep.astype(np.int32)


# ---- losses (SURVEY 8f rank 1) -------------------------------------------------------------------
def _bce_terms(t, p):
    """[TF-internal] Keras backend.binary_crossentropy(from_logits=False) of TF 2.0.0, float32:
    p = clip(p, eps, 1 - eps); -(t*log(p + eps) + (1 - t)*log(1 - p + eps)), eps = 1e-7."""
    eps = F32(1e-7)
    p = np.clip(p.astype(F32), eps, F32(1) - eps)
    t = t.astype(F32)
    bce = t * np.log(p + eps)
    bce = bce + (F32(1) - t) * np.log(F32(1) - p + eps)
    return -bce


def cls_loss(y_true, y_pred):
    """utils/train_utils.py:146-161.  Entries with y_true != -1 (:156) -> BinaryCrossentropy, mean
    over them (:159-161).  The per-entry terms are float32 in TF's op order; the sum is carried
    in float64 (TF sums in float32 in an unspecified order), so compare at ~1e-6 relative."""
    t = np.asarray(y_true, F32).reshape(-1)
    p = np.asarray(y_pred, F32).reshape(-1)
    m = t != F32(-1.0)
    terms = _bce_terms(t[m], p[m])
    with np.errstate(invalid="ignore", divide="ignore"):
        return F32(np.sum(terms, dtype=np.float64) / np.float64(terms.size))     # 0/0 -> NaN, as TF


def _huber_terms(t, p, delta=1.0):
    """[TF-internal] keras huber_loss of TF 2.0.0: elementwise (no mean over the last axis)."""
    delta = F32(delta)
    ae = np.abs(p.astype(F32) - t.astype(F32))
    q = np.minimum(ae, delta)
    lin = ae - q
    return F32(0.5) * (q * q) + delta * lin


def reg_loss(y_true, y_pred, delta=1.0):
    """utils/train_utils.py:163-185.  y_pred reshaped to (B,-1,4) (:175); Huber per coordinate,
    summed over the 4 coordinates (:178); rows with any non-zero true delta (:180-181);
    sum / max(1, #rows) (:183-185)."""
    t = np.asarray(y_true, F32)
    p = np.asarray(y_pred, F32).reshape(t.shape[0], -1, 4)
    h = _huber_terms(t, p, delta)
    rows = ((h[..., 0] + h[..., 1]) + h[..., 2]) + h[..., 3]
    pos = np.any(t != F32(0.0), axis=-1)
    n = int(pos.sum())
    return F32(np.sum(rows[pos], dtype=np.float64) / np.float64(max(1, n)))


def loss_grads(true_deltas, pred_deltas, true_labels, pred_labels, delta=1.0):
    """d reg_loss / d pred_deltas and d cls_loss / d pred_labels as TF's autograd derives them from
    the ops above: Huber' = e for |e| <= delta else delta*sign(e) (minimum routes the gradient to
    its first argument on ties), masked and / max(1, #pos); BCE' = ((1-t)/(1-p+eps) - t/(p+eps)) / M
    inside the clip range [eps, 1-eps] (clip_by_value passes the gradient on its closed range)."""
    t = np.asarray(true_deltas, F32)
    p = np.asarray(pred_deltas, F32).reshape(t.shape)
    e = p - t
    pos = np.any(t != F32(0.0), axis=-1, keepdims=True)
    g = np.where(np.abs(e) <= F32(delta), e, np.where(e > 0, F32(delta), -F32(delta))).astype(F32)
    inv = F32(1.0) / F32(max(1, int(pos.sum())))
    gd = np.where(pos, g * inv, F32(0.0)).astype(F32).reshape(np.asarray(pred_deltas).shape)
    tl = np.asarray(true_labels, F32)
    pl = np.asarray(pred_labels, F32)
    eps = F32(1e-7)
    valid = tl != F32(-1.0)
    inside = (pl >= eps) & (pl <= F32(1) - eps)
    with np.errstate(invalid="ignore", divide="ignore"):
        gb = (F32(1) - tl) / ((F32(1) - pl) + eps) - tl / (pl + eps)
        invm = F32(1.0) / F32(int(valid.sum()))
        gl = np.where(valid, np.where(inside, gb, F32(0.0)) * invm, F32(0.0)).astype(F32)
    return gd, gl


# ---- the callers either side of the path (SURVEY 8f ranks 2 and 3) ----------------------------------
def predictor_top_boxes(rpn_bbox_deltas, rpn_labels, anchors, hp, k=10):
    """predictor.py:52-60: reshape (:52-53), deltas *= variances (:55), get_bboxes_from_deltas (:56),
    tf.nn.top_k(rpn_labels, k) (:58, [TF-internal] ties -> lower index first), gather (:60).
    Returns (selected_rpn_bboxes (B,k,4), top_values (B,k), top_indices (B,k) int32)."""
    reg = np.asarray(rpn_bbox_deltas, F32)
    B = reg.shape[0]
    reg = reg.reshape(B, -1, 4) * np.asarray(hp["variances"], F32)
    cls = np.asarray(rpn_labels, F32).reshape(B, -1)
    boxes = get_bboxes_from_deltas(np.asarray(anchors, F32), reg)
    vals, idx = top_k(cls, k)
    return np.take_along_axis(boxes, idx[..., None].astype(np.int64), axis=1), vals, idx


def flip_horizontally_boxes(gt_boxes):
    """utils/data_utils.py:66-69: [y1, 1 - x2, y2, 1 - x1] in float32."""
    b = np.asarray(gt_boxes, F32)
    return np.stack([b[..., 0], F32(1.0) - b[..., 3], b[..., 2], F32(1.0) - b[..., 1]], axis=-1)


def pad_gt_batch(gt_boxes_list, gt_labels_list, max_boxes=None, flip=None, label_add=0):
    """tf.data padded_batch with utils/data_utils.py:152-157's padding values (boxes 0, labels -1),
    optional per-image flip (:54-68) and the ``label + 1`` of preprocessing (:20)."""
    B = len(gt_boxes_list)
    G = int(max_boxes) if max_boxes is not None else max([len(b) for b in gt_boxes_list] + [1])
    boxes = np.zeros((B, G, 4), F32)
    labels = np.full((B, G), -1, np.int32)
    for b in range(B):
        n = min(len(gt_boxes_list[b]), G)
        if n:
            bx = np.asarray(gt_boxes_list[b], F32)[:n]
            if flip is not None and flip[b]:
                bx = flip_horizontally_boxes(bx)
            boxes[b, :n] = bx
            labels[b, :n] = np.asarray(gt_labels_list[b], np.int32)[:n] + np.int32(label_add)
    return boxes, labels

"""Drop-in for the reference's utils/bbox_utils.py, running on libtfrpn_cuda.so (sm_100a).

Same function names, positional signatures and output shapes as the reference; every function
cites the reference lines it replaces.  Inputs/outputs: see tfrpn._tensor.
"""
import collections
import ctypes as C

import torch

from .. import _lib
from .._tensor import Origin, default_device, from_device, ptr, stream_ptr, to_device

F32 = torch.float32


def _pair(v):
    if isinstance(v, (tuple, list)):
        return int(v[0]), int(v[1])
    return int(v), int(v)


def _anchor_cfg(hyper_params):
    cfg = _lib.AnchorCfg()
    cfg.img_h, cfg.img_w = _pair(hyper_params["img_size"])
    cfg.fm_h, cfg.fm_w = _pair(hyper_params["feature_map_shape"])
    scales, ratios = hyper_params["anchor_scales"], hyper_params["anchor_ratios"]
    if not (1 <= len(scales) <= 8 and 1 <= len(ratios) <= 8):
        raise ValueError("1..8 anchor_scales and anchor_ratios are supported")
    cfg.n_scales, cfg.n_ratios = len(scales), len(ratios)
    for i, s in enumerate(scales):
        cfg.scales[i] = float(s)
    for i, r in enumerate(ratios):
        cfg.ratios[i] = float(r)
    return cfg


def generate_base_anchors(hyper_params):
    """utils/bbox_utils.py:3-21 -> (anchor_count, [y1, x1, y2, x2]) float32."""
    cfg = _anchor_cfg(hyper_params)
    A = cfg.n_scales * cfg.n_ratios
    host = (C.c_float * (A * 4))()
    _lib.check(_lib.load().tfrpn_base_anchors_host(C.byref(cfg), host))
    return torch.tensor(list(host), dtype=F32).reshape(A, 4).to(default_device())


def generate_anchors(hyper_params):
    """utils/bbox_utils.py:23-46 -> (fm_h * fm_w * anchor_count, 4) float32 in [0, 1]."""
    cfg = _anchor_cfg(hyper_params)
    dev = default_device()
    N = cfg.fm_h * cfg.fm_w * cfg.n_scales * cfg.n_ratios
    out = torch.empty((N, 4), dtype=F32, device=dev)
    _lib.check(_lib.load().tfrpn_anchors(C.byref(cfg), ptr(out), stream_ptr(dev)))
    return out


NmsOutput = collections.namedtuple(
    "CombinedNonMaxSuppression", ["nmsed_boxes", "nmsed_scores", "nmsed_classes", "valid_detections"])


def non_max_suppression(pred_bboxes, pred_labels, **kwargs):
    """utils/bbox_utils.py:48-70 (tf.image.combined_non_max_suppression pass-through).

    pred_bboxes (B, K, 1, 4), pred_labels (B, K, 1); kwargs are TF's: max_output_size_per_class,
    max_total_size, iou_threshold=0.5, score_threshold=-inf, pad_per_class=False, clip_boxes=True.
    Extra kwarg ``return_indices=True`` appends the kept indices (B, rows) int32, -1 padded.
    Extra kwarg ``pre_nms_topn=k`` lets only the k best scores compete: the tf.nn.top_k + tf.gather of
    predictor.py:58-60 fused in front of the NMS (same result as calling them first, but consumed lazily).
    """
    known = {"max_output_size_per_class", "max_total_size", "iou_threshold", "score_threshold",
             "pad_per_class", "clip_boxes", "name", "return_indices", "pre_nms_topn"}
    unknown = set(kwargs) - known
    if unknown:
        raise TypeError("non_max_suppression() got unexpected keyword arguments %s" % sorted(unknown))
    if "max_output_size_per_class" not in kwargs or "max_total_size" not in kwargs:
        raise TypeError("non_max_suppression() needs max_output_size_per_class and max_total_size")
    o = Origin()
    boxes = to_device(pred_bboxes, F32, o, "pred_bboxes")
    scores = to_device(pred_labels, F32, o, "pred_labels")
    if boxes.dim() != 4 or boxes.shape[-1] != 4 or scores.dim() != 3:
        raise ValueError("pred_bboxes must be (B,K,q,4) and pred_labels (B,K,C)")
    B, K = scores.shape[0], scores.shape[1]
    if boxes.shape[0] != B or boxes.shape[1] != K:
        raise ValueError("pred_bboxes %s and pred_labels %s disagree" % (tuple(boxes.shape), tuple(scores.shape)))
    if boxes.shape[2] != 1 or scores.shape[2] != 1:
        return _multi_class_nms(boxes, scores, kwargs, o)
    cfg = _lib.NmsCfg(int(kwargs["max_output_size_per_class"]), int(kwargs["max_total_size"]),
                      float(kwargs.get("iou_threshold", 0.5)), float(kwargs.get("score_threshold", float("-inf"))),
                      int(bool(kwargs.get("pad_per_class", False))), int(bool(kwargs.get("clip_boxes", True))),
                      int(kwargs.get("pre_nms_topn") or 0))
    rows = min(cfg.max_total_size, cfg.max_output_size_per_class) if cfg.pad_per_class else cfg.max_total_size
    dev = boxes.device
    nb = torch.empty((B, rows, 4), dtype=F32, device=dev)
    ns = torch.empty((B, rows), dtype=F32, device=dev)
    nc = torch.empty((B, rows), dtype=F32, device=dev)
    nv = torch.empty((B,), dtype=torch.int32, device=dev)
    ni = torch.empty((B, rows), dtype=torch.int32, device=dev) if kwargs.get("return_indices") else None
    _lib.check(_lib.load().tfrpn_nms(_lib.handle(dev.index), ptr(boxes), ptr(scores), B, K, C.byref(cfg),
                                     ptr(nb), ptr(ns), ptr(nc), ptr(nv), ptr(ni), stream_ptr(dev)))
    res = NmsOutput(*(from_device(t, o) for t in (nb, ns, nc, nv)))
    if ni is not None:
        return tuple(res) + (from_device(ni, o),)
    return res


def _multi_class_nms(boxes, scores, kwargs, o):
    """tf.image.combined_non_max_suppression with C > 1 classes or q = C boxes per entry (the reference's wrapper allows
    ``total_labels`` > 1, utils/bbox_utils.py:53-55; the RPN itself has one), in one tfrpn_nms_multiclass call: per
    (image, class) the one-class NMS, then the merge of the C keep lists by score (equal scores -> lower class id first,
    then the class's own order -- TF leaves ties to an unstable std::sort)."""
    B, K, Cn = scores.shape
    q = boxes.shape[2]
    if q not in (1, Cn):
        raise ValueError("pred_bboxes must be (B,K,1,4) or (B,K,C,4) for pred_labels (B,K,C); got q = %d, C = %d" % (q, Cn))
    cfg = _lib.NmsCfg(int(kwargs["max_output_size_per_class"]), int(kwargs["max_total_size"]),
                      float(kwargs.get("iou_threshold", 0.5)), float(kwargs.get("score_threshold", float("-inf"))),
                      int(bool(kwargs.get("pad_per_class", False))), int(bool(kwargs.get("clip_boxes", True))),
                      int(kwargs.get("pre_nms_topn") or 0))
    if cfg.max_output_size_per_class <= 0 or cfg.max_total_size <= 0:
        raise ValueError("max_output_size_per_class and max_total_size must be > 0")
    rows = min(cfg.max_total_size, cfg.max_output_size_per_class * Cn) if cfg.pad_per_class else cfg.max_total_size
    dev = boxes.device
    run = B > 0 and K > 0 and Cn > 0   # the kernels write every output; without boxes or classes every row is padding
    alloc = torch.empty if run else torch.zeros
    nb = alloc((B, rows, 4), dtype=F32, device=dev)
    ns = alloc((B, rows), dtype=F32, device=dev)
    nc = alloc((B, rows), dtype=F32, device=dev)
    nv = alloc((B,), dtype=torch.int32, device=dev)
    ni = None
    if kwargs.get("return_indices"):
        ni = torch.empty((B, rows), dtype=torch.int32, device=dev) if run else torch.full((B, rows), -1, dtype=torch.int32, device=dev)
    if run:
        _lib.check(_lib.load().tfrpn_nms_multiclass(_lib.handle(dev.index), ptr(boxes), q, ptr(scores), B, K, Cn,
                                                    C.byref(cfg), ptr(nb), ptr(ns), ptr(nc), ptr(nv), ptr(ni),
                                                    stream_ptr(dev)))
    res = NmsOutput(*(from_device(t, o) for t in (nb, ns, nc, nv)))
    if ni is not None:
        return tuple(res) + (from_device(ni, o),)
    return res


def _broadcast_pair(first, second, o, n1, n2):
    """(N,4)|(B,N,4) x (B,N,4) | (N,4) -> tensors, batched flag of `first`, B, N, squeeze flag."""
    a = to_device(first, F32, o, n1)
    b = to_device(second, F32, o, n2)
    if a.shape[-1] != 4 or b.shape[-1] != 4 or a.dim() not in (2, 3) or b.dim() not in (2, 3):
        raise ValueError("%s and %s must be (N,4) or (B,N,4)" % (n1, n2))
    squeeze = a.dim() == 2 and b.dim() == 2
    if b.dim() == 2:
        if a.dim() == 3:                      # (B,N,4) x (N,4): expand the second operand
            b = b.unsqueeze(0).expand(a.shape[0], -1, -1).contiguous()
        else:
            b = b.unsqueeze(0)
    B, N = b.shape[0], b.shape[1]
    batched = a.dim() == 3
    if a.shape[-2] != N or (batched and a.shape[0] != B):
        raise ValueError("%s %s and %s %s do not broadcast" % (n1, tuple(a.shape), n2, tuple(b.shape)))
    return a, b, batched, B, N, squeeze


def get_bboxes_from_deltas(anchors, deltas):
    """utils/bbox_utils.py:72-96.  anchors (N,4) or (B,N,4); deltas (B,N,4) -> (B,N,4)."""
    o = Origin()
    a, d, batched, B, N, squeeze = _broadcast_pair(anchors, deltas, o, "anchors", "deltas")
    out = torch.empty((B, N, 4), dtype=F32, device=d.device)
    _lib.check(_lib.load().tfrpn_decode(ptr(a), int(batched), ptr(d), None, 0, B, N, ptr(out), stream_ptr(d.device)))
    return from_device(out[0] if squeeze else out, o)


def get_bboxes_from_hyper_params(hyper_params, deltas, variances=None, clip=False):
    """generate_anchors (utils/bbox_utils.py:23-46) fused into get_bboxes_from_deltas (:72-96): the anchors are
    regenerated in registers, no anchor tensor is read.  ``variances`` multiplies the deltas first (predictor.py:55),
    ``clip`` clips the boxes to [0,1].  deltas (B,N,4) or (B,F,F,4A) -> (B,N,4)."""
    o = Origin()
    d = to_device(deltas, F32, o, "deltas")
    B = d.shape[0]
    d = d.reshape(B, -1, 4)
    cfg = _anchor_cfg(hyper_params)
    N = cfg.fm_h * cfg.fm_w * cfg.n_scales * cfg.n_ratios
    if d.shape[1] != N:
        raise ValueError("deltas %s but hyper_params give %d anchors" % (tuple(d.shape), N))
    out = torch.empty((B, N, 4), dtype=F32, device=d.device)
    var = None if variances is None else (C.c_float * 4)(*[float(v) for v in variances])
    _lib.check(_lib.load().tfrpn_decode_anchor_cfg(C.byref(cfg), ptr(d), var, int(bool(clip)), B, ptr(out), stream_ptr(d.device)))
    return from_device(out, o)


def get_deltas_from_bboxes(bboxes, gt_boxes):
    """utils/bbox_utils.py:98-124.  bboxes (N,4) or (B,N,4); gt_boxes (B,N,4) -> (B,N,4)."""
    o = Origin()
    a, g, batched, B, N, squeeze = _broadcast_pair(bboxes, gt_boxes, o, "bboxes", "gt_boxes")
    out = torch.empty((B, N, 4), dtype=F32, device=g.device)
    _lib.check(_lib.load().tfrpn_encode_deltas(ptr(a), int(batched), ptr(g), B, N, ptr(out), stream_ptr(g.device)))
    return from_device(out[0] if squeeze else out, o)


def generate_iou_map(bboxes, gt_boxes):
    """utils/bbox_utils.py:126-150.  bboxes (N,4) or (B,N,4); gt_boxes (B,G,4) -> (B,N,G)."""
    o = Origin()
    b = to_device(bboxes, F32, o, "bboxes")
    g = to_device(gt_boxes, F32, o, "gt_boxes")
    if g.dim() != 3 or g.shape[-1] != 4 or b.shape[-1] != 4 or b.dim() not in (2, 3):
        raise ValueError("bboxes must be (N,4) or (B,N,4) and gt_boxes (B,G,4)")
    B, G = g.shape[0], g.shape[1]
    N = b.shape[-2]
    batched = b.dim() == 3
    if batched and b.shape[0] != B:
        raise ValueError("batch sizes differ: %d vs %d" % (b.shape[0], B))
    out = torch.empty((B, N, G), dtype=F32, device=g.device)
    _lib.check(_lib.load().tfrpn_iou_map(ptr(b), int(batched), ptr(g), B, N, G, ptr(out), stream_ptr(g.device)))
    return from_device(out, o)


def _scale(bboxes, height, width, denorm):
    o = Origin()
    b = to_device(bboxes, F32, o, "bboxes")
    if b.shape[-1] != 4:
        raise ValueError("bboxes must end in 4 coordinates")
    out = torch.empty_like(b)
    _lib.check(_lib.load().tfrpn_scale_boxes(ptr(b), b.numel() // 4, float(height), float(width), denorm,
                                             ptr(out), stream_ptr(b.device)))
    return from_device(out, o)


def normalize_bboxes(bboxes, height, width):
    """utils/bbox_utils.py:152-166."""
    return _scale(bboxes, height, width, 0)


def denormalize_bboxes(bboxes, height, width):
    """utils/bbox_utils.py:168-182 (multiply, then round half to even like tf.round)."""
    return _scale(bboxes, height, width, 1)


def top_k_boxes(scores, k, boxes=None):
    """tf.nn.top_k(scores, k) [+ tf.gather(boxes, indices, batch_dims=1)], predictor.py:58-60.

    scores (B,N); boxes (N,4) or (B,N,4).  Returns (values, indices[, gathered])."""
    o = Origin()
    s = to_device(scores, F32, o, "scores")
    if s.dim() != 2:
        raise ValueError("scores must be (B,N)")
    B, N = s.shape
    k = int(k)
    bx = to_device(boxes, F32, o, "boxes") if boxes is not None else None
    if bx is not None and (bx.shape[-1] != 4 or bx.shape[-2] != N):
        raise ValueError("boxes must be (N,4) or (B,N,4)")
    dev = s.device
    vals = torch.empty((B, k), dtype=F32, device=dev)
    idx = torch.empty((B, k), dtype=torch.int32, device=dev)
    gat = torch.empty((B, k, 4), dtype=F32, device=dev) if bx is not None else None
    _lib.check(_lib.load().tfrpn_topk(_lib.handle(dev.index), ptr(s), B, N, k, ptr(vals), ptr(idx), ptr(bx),
                                      int(bx is not None and bx.dim() == 3), ptr(gat), stream_ptr(dev)))
    res = (from_device(vals, o), from_device(idx, o))
    return res + ((from_device(gat, o),) if gat is not None else ())

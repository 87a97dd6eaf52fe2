"""The composed proposal stage (SURVEY.md 8a row P): what predictor.py:52-60 plus the reference's
NMS wrapper (utils/bbox_utils.py:48-70) compute, fused into one launch per batch."""
import ctypes as C

import torch

from . import _lib
from ._tensor import Origin, from_device, ptr, stream_ptr, to_device

F32 = torch.float32


def proposal_cfg(hyper_params, pre_nms_topn=None, post_nms_topn=None, nms_iou_threshold=None, clip=True):
    cfg = _lib.ProposalCfg()
    for i, v in enumerate(hyper_params["variances"]):
        cfg.variances[i] = float(v)
    cfg.pre_nms_topn = int(pre_nms_topn if pre_nms_topn is not None else hyper_params.get("pre_nms_topn", 6000))
    cfg.post_nms_topn = int(post_nms_topn if post_nms_topn is not None else hyper_params["test_nms_topn"])
    cfg.nms_iou_threshold = _lib.iou_threshold(nms_iou_threshold if nms_iou_threshold is not None
                                               else hyper_params.get("nms_iou_threshold", 0.7), "nms_iou_threshold")
    cfg.clip = int(bool(clip))
    return cfg


def generate_proposals(rpn_bbox_deltas, rpn_labels, anchors, hyper_params, pre_nms_topn=None,
                       post_nms_topn=None, nms_iou_threshold=None, clip=True):
    """rpn_bbox_deltas (B,F,F,4A) or (B,N,4); rpn_labels (B,F,F,A) or (B,N) -- the two outputs of
    ``rpn_model.predict_on_batch`` (predictor.py:50); anchors (N,4).

    reshape (:52-53) -> deltas *= variances (:55) -> get_bboxes_from_deltas (:56) -> clip [0,1]
    -> tf.nn.top_k(k = pre_nms_topn = 6000) (:58) -> gather (:60) -> combined NMS
    (max_output_size_per_class = max_total_size = test_nms_topn = 300, iou 0.7).
    Returns (boxes (B,P,4), scores (B,P), valid_detections (B,), keep_indices (B,P) into N, -1 pad).

    ``anchors=None``: the anchors of ``hyper_params`` (utils/bbox_utils.py:23-46) are regenerated in registers
    inside the kernel -- no anchor tensor is read (feature maps below 40000 anchors).
    """
    o = Origin()
    reg = to_device(rpn_bbox_deltas, F32, o, "rpn_bbox_deltas")
    cls = to_device(rpn_labels, F32, o, "rpn_labels")
    B = reg.shape[0]
    reg = reg.reshape(B, -1, 4)
    cls = cls.reshape(B, -1)
    N = cls.shape[1]
    cfg = proposal_cfg(hyper_params, pre_nms_topn, post_nms_topn, nms_iou_threshold, clip)
    if anchors is None:
        from .utils.bbox_utils import _anchor_cfg
        acfg = _anchor_cfg(hyper_params)
        n_cfg = acfg.fm_h * acfg.fm_w * acfg.n_scales * acfg.n_ratios
        if reg.shape[1] != N or N != n_cfg:
            raise ValueError("shapes disagree: deltas %s, labels %s, hyper_params give %d anchors"
                             % (tuple(reg.shape), tuple(cls.shape), n_cfg))
        dev = reg.device
        P = cfg.post_nms_topn
        boxes = torch.empty((B, P, 4), dtype=F32, device=dev)
        scores = torch.empty((B, P), dtype=F32, device=dev)
        valid = torch.empty((B,), dtype=torch.int32, device=dev)
        keep = torch.empty((B, P), dtype=torch.int32, device=dev)
        _lib.check(_lib.load().tfrpn_proposals_anchor_cfg(_lib.handle(dev.index), ptr(reg), ptr(cls), C.byref(acfg), B,
                                                          C.byref(cfg), ptr(boxes), ptr(scores), ptr(valid), ptr(keep),
                                                          stream_ptr(dev)))
        return tuple(from_device(t, o) for t in (boxes, scores, valid, keep))
    anc = to_device(anchors, F32, o, "anchors")
    if reg.shape[1] != N or anc.shape != (N, 4):
        raise ValueError("shapes disagree: deltas %s, labels %s, anchors %s"
                         % (tuple(reg.shape), tuple(cls.shape), tuple(anc.shape)))
    dev = reg.device
    P = cfg.post_nms_topn
    boxes = torch.empty((B, P, 4), dtype=F32, device=dev)
    scores = torch.empty((B, P), dtype=F32, device=dev)
    valid = torch.empty((B,), dtype=torch.int32, device=dev)
    keep = torch.empty((B, P), dtype=torch.int32, device=dev)
    _lib.check(_lib.load().tfrpn_proposals(_lib.handle(dev.index), ptr(reg), ptr(cls), ptr(anc), B, N,
                                           C.byref(cfg), ptr(boxes), ptr(scores), ptr(valid), ptr(keep),
                                           stream_ptr(dev)))
    return tuple(from_device(t, o) for t in (boxes, scores, valid, keep))


def predict_top_boxes(rpn_bbox_deltas, rpn_labels, anchors, hyper_params, k=10, clip=False):
    """The body of the reference's predictor loop, predictor.py:52-60, in one launch:

        rpn_bbox_deltas = reshape(.., (B,-1,4)); rpn_labels = reshape(.., (B,-1))      (:52-53)
        rpn_bbox_deltas *= variances; rpn_bboxes = get_bboxes_from_deltas(anchors, ..)  (:55-56)
        _, top_indices = tf.nn.top_k(rpn_labels, 10)                                    (:58)
        selected_rpn_bboxes = tf.gather(rpn_bboxes, top_indices, batch_dims=1)          (:60)

    Only the k selected rows are decoded.  Returns (selected_rpn_bboxes (B,k,4), top_values (B,k),
    top_indices (B,k) int32).  ``clip`` defaults to False because the reference never clips here.
    """
    o = Origin()
    reg = to_device(rpn_bbox_deltas, F32, o, "rpn_bbox_deltas")
    cls = to_device(rpn_labels, F32, o, "rpn_labels")
    anc = to_device(anchors, F32, o, "anchors")
    B = reg.shape[0]
    reg = reg.reshape(B, -1, 4)
    cls = cls.reshape(B, -1)
    N = cls.shape[1]
    if reg.shape[1] != N or anc.shape != (N, 4):
        raise ValueError("shapes disagree: deltas %s, labels %s, anchors %s"
                         % (tuple(reg.shape), tuple(cls.shape), tuple(anc.shape)))
    k = int(k)
    dev = reg.device
    boxes = torch.empty((B, k, 4), dtype=F32, device=dev)
    vals = torch.empty((B, k), dtype=F32, device=dev)
    idx = torch.empty((B, k), dtype=torch.int32, device=dev)
    var = (C.c_float * 4)(*[float(v) for v in hyper_params["variances"]])
    _lib.check(_lib.load().tfrpn_predict_topk(_lib.handle(dev.index), ptr(reg), ptr(cls), ptr(anc), B, N, k, var,
                                              int(bool(clip)), ptr(boxes), ptr(vals), ptr(idx), stream_ptr(dev)))
    return tuple(from_device(t, o) for t in (boxes, vals, idx))

"""Box-head losses of a two-stage detector's second stage on the GPU (tfrpn_roi_head_losses, include/tfrpn.h):
softmax cross-entropy over the rows ``roi_targets`` samples and class-specific Huber over its fg rows, with their
gradients.

Which rows count is read from ``roi_targets``' labels on the device (-1 padding, 0 background, 1..C-1 a class), so
the call needs no ``torch.where`` and no host synchronisation: one kernel launch, two with the gradients, and it can
be captured in a CUDA graph.  The loss sums have a fixed order, so the losses are the same bits on every run.
"""
import collections
import ctypes as C

import torch

from . import _lib
from ._tensor import Origin, from_device, ptr, stream_ptr, to_device

F32 = torch.float32
RoiHeadLosses = collections.namedtuple("RoiHeadLosses", "cls_loss reg_loss n_rows n_fg n_correct n_fg_correct "
                                                        "grad_logits grad_deltas", defaults=(None, None))
_NORMALIZERS = {"fg": 0, "rows": 1}


def _launch(cfg, logits, deltas, labels, targets, scale=None, with_grads=False):
    """-> (out (8,) float32 holding tfrpn_roi_loss_out, grad_logits, grad_deltas)"""
    B, S = labels.shape
    dev = logits.device
    out = torch.empty((8,), dtype=F32, device=dev)
    gl = torch.empty_like(logits) if with_grads else None
    gd = torch.empty_like(deltas) if with_grads else None
    _lib.check(_lib.load().tfrpn_roi_head_losses(_lib.handle(dev.index), ptr(logits), ptr(deltas), ptr(labels),
                                                 ptr(targets), B, S, C.byref(cfg), ptr(out), ptr(scale), ptr(gl),
                                                 ptr(gd), stream_ptr(dev)))
    return out, gl, gd


class _RoiHeadLosses(torch.autograd.Function):
    """(cls_loss, reg_loss, counts) differentiable with respect to the logits and the box deltas.  Saves its inputs
    only; the backward runs the losses again with both gradients, scaled on the device by
    grad_scale = stack([d cls, d reg]) (autograd passes a zero for a loss that is not used)."""

    @staticmethod
    def forward(ctx, logits, deltas, labels, targets, cfg):
        ctx.save_for_backward(logits, deltas, labels, targets)
        ctx.cfg = cfg
        out, _, _ = _launch(cfg, logits, deltas, labels, targets)
        counts = out.view(torch.int32)[2:6]
        ctx.mark_non_differentiable(counts)
        return out[0], out[1], counts

    @staticmethod
    def backward(ctx, g_cls, g_reg, _):
        logits, deltas, labels, targets = ctx.saved_tensors
        zero = torch.zeros((), dtype=F32, device=logits.device)
        scale = torch.stack([zero if g_cls is None else g_cls.to(F32), zero if g_reg is None else g_reg.to(F32)])
        _, gl, gd = _launch(ctx.cfg, logits, deltas, labels, targets, scale, with_grads=True)
        return (gl if ctx.needs_input_grad[0] else None), (gd if ctx.needs_input_grad[1] else None), None, None, None


def roi_head_losses(cls_logits, box_deltas, labels, target_deltas, *, huber_delta=1.0, normalize="fg",
                    with_grads=False):
    """The box head's losses over roi_targets' rows: cls_logits (B,S,C) float32, box_deltas (B,S,C*4), (B,S,C,4),
    (B,S,4) or (B,S,1,4) float32 (q = C class-specific or q = 1 class-agnostic, inferred from the shape; the reshape
    is a view), labels (B,S) int and target_deltas (B,S,4) float32 as ``roi_targets`` returns them.

    cls_loss is the softmax cross-entropy averaged over the rows with 0 <= label < C (NaN when there are none);
    reg_loss sums keras Huber(huber_delta) over the 4 coordinates of each fg row's label-class deltas (1 <= label < C),
    divided by max(1, #fg) with ``normalize="fg"`` (the rule of ``rpn_losses``) or by max(1, #rows taking part) with
    ``normalize="rows"`` (torchvision's and Detectron2's box_loss / labels.numel(); their smooth_l1(beta) equals
    Huber(delta = beta) / beta).  Returns RoiHeadLosses(cls_loss, reg_loss, n_rows, n_fg, n_correct,
    n_fg_correct) as 0-d tensors (the counts int32; n_correct counts the rows whose first argmax logit is the label).

    On torch CUDA tensors the two losses are differentiable with respect to cls_logits and box_deltas, with no host
    synchronisation in the forward or the backward.  ``with_grads=True`` instead returns the unscaled gradients
    d cls_loss / d cls_logits and d reg_loss / d box_deltas (shaped like the inputs) as grad_logits and grad_deltas,
    for callers that apply the chain rule themselves (a tf.custom_gradient).  NumPy and TF inputs come back in their
    own framework.  C > 1024, S > 8192 or B > 65535 raise NotImplementedError; bad arguments raise ValueError."""
    if normalize not in _NORMALIZERS:
        raise ValueError("normalize must be 'fg' or 'rows', got %r" % (normalize,))
    o = Origin()
    x = to_device(cls_logits, F32, o, "cls_logits")
    if x.dim() != 3:
        raise ValueError("cls_logits must be (B,S,C), got %s" % (tuple(x.shape),))
    B, S, Cn = x.shape
    d = to_device(box_deltas, F32, o, "box_deltas")
    if d.dim() == 3 and d.shape[:2] == (B, S) and d.shape[2] % 4 == 0:
        d4 = d.view(B, S, d.shape[2] // 4, 4)
    elif d.dim() == 4 and d.shape[:2] == (B, S) and d.shape[3] == 4:
        d4 = d
    else:
        raise ValueError("box_deltas must be (B,S,q*4) or (B,S,q,4) with (B,S) = (%d,%d), got %s"
                         % (B, S, tuple(d.shape)))
    lab = to_device(labels, torch.int32, o, "labels")
    if tuple(lab.shape) != (B, S):
        raise ValueError("labels must be (%d,%d), got %s" % (B, S, tuple(lab.shape)))
    t = to_device(target_deltas, F32, o, "target_deltas")
    if tuple(t.shape) != (B, S, 4):
        raise ValueError("target_deltas must be (%d,%d,4), got %s" % (B, S, tuple(t.shape)))
    cfg = _lib.RoiLossCfg(int(Cn), int(d4.shape[2]), float(huber_delta), _NORMALIZERS[normalize])
    if o.kind == "torch" and not with_grads:
        cls, reg, counts = _RoiHeadLosses.apply(x, d4, lab, t, cfg)
        return RoiHeadLosses(cls, reg, *counts.unbind())
    out, gl, gd = _launch(cfg, x, d4, lab, t, with_grads=with_grads)
    counts = out.view(torch.int32)
    res = [from_device(out[0], o), from_device(out[1], o)] + [from_device(counts[i], o) for i in range(2, 6)]
    if with_grads:
        res += [from_device(gl, o), from_device(gd.view(d.shape), o)]
    return RoiHeadLosses(*res)

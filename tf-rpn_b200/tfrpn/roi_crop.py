"""RoI feature cropping of a two-stage detector's second stage on the GPU: ``tf.image.crop_and_resize`` (bilinear)
and its image gradient (tfrpn_crop_and_resize, tfrpn_crop_and_resize_grad_image, include/tfrpn.h).

Boxes are normalised [y1, x1, y2, x2] with a batch index each, which is what ``roi_targets`` writes: its ``rois``
(B,S,4) go in as they are with ``box_indices=None``.  The samples sit on crop_and_resize's end-point grid (not on
roi_align's bin centres), every operation is TensorFlow's CPU kernel in float32, and the gradient is a gather with no
atomics that sums each element's terms in TensorFlow's loop order, so it is the same on every run.  Both calls are
one kernel launch with no host synchronisation.
"""
import torch

from . import _lib
from ._tensor import Origin, from_device, ptr, stream_ptr, to_device

F32 = torch.float32


def _launch_forward(image, boxes, index, ch, cw, extrapolation_value):
    B, H, W, C = image.shape
    M = boxes.shape[0]
    out = torch.empty((M, ch, cw, C), dtype=F32, device=image.device)
    _lib.check(_lib.load().tfrpn_crop_and_resize(ptr(image), B, H, W, C, ptr(boxes), ptr(index), M, ch, cw,
                                                 float(extrapolation_value), ptr(out), stream_ptr(image.device)))
    return out


def _launch_grad(grad, boxes, index, image_shape):
    B, H, W, C = image_shape
    M, ch, cw = grad.shape[:3]
    grad = grad.contiguous()
    out = torch.empty((B, H, W, C), dtype=F32, device=grad.device)
    _lib.check(_lib.load().tfrpn_crop_and_resize_grad_image(ptr(grad), ptr(boxes), ptr(index), M, B, H, W, C, ch, cw,
                                                            ptr(out), stream_ptr(grad.device)))
    return out


class _CropAndResize(torch.autograd.Function):
    """Gradient for the image only: the boxes and their indices get None (RoIs are stop-gradient in Faster R-CNN).
    Saves the boxes and indices, not the output."""

    @staticmethod
    def forward(ctx, image, boxes, index, ch, cw, extrapolation_value):
        ctx.save_for_backward(boxes, index)
        ctx.image_shape = tuple(image.shape)
        return _launch_forward(image, boxes, index, ch, cw, extrapolation_value)

    @staticmethod
    def backward(ctx, grad):
        boxes, index = ctx.saved_tensors
        gi = _launch_grad(grad, boxes, index, ctx.image_shape) if ctx.needs_input_grad[0] else None
        return gi, None, None, None, None, None


def crop_and_resize(image, boxes, box_indices, crop_size, method="bilinear", extrapolation_value=0.0):
    """tf.image.crop_and_resize on the GPU: image (B,H,W,C) float32, boxes (M,4) normalised [y1,x1,y2,x2] with
    box_indices (M,) int, crop_size (ch, cw) -> (M,ch,cw,C) float32.  ``box_indices=None`` is the batched layout of
    ``roi_targets``: boxes (B,S,4) and a result (B,S,ch,cw,C).

    Samples outside the image, or at a NaN coordinate, take ``extrapolation_value``; a box whose index is outside
    [0,B) gives NaN (TensorFlow raises).  For torch CUDA inputs the result is differentiable with respect to the
    image (through the deterministic tfrpn_crop_and_resize_grad_image); the boxes get no gradient.  Results come back
    in the framework of the inputs.  ``method="nearest"`` raises NotImplementedError, as do C > 4096, a crop side
    > 32, H or W > 8192; bad arguments raise ValueError."""
    if method == "nearest":
        raise NotImplementedError("crop_and_resize: only method='bilinear' is implemented")
    if method != "bilinear":
        raise ValueError("crop_and_resize: method must be 'bilinear' or 'nearest', got %r" % (method,))
    ch, cw = (int(v) for v in crop_size)
    o = Origin()
    img = to_device(image, F32, o, "image")
    if img.dim() != 4:
        raise ValueError("image must be (B,H,W,C), got %s" % (tuple(img.shape),))
    bx = to_device(boxes, F32, o, "boxes")
    B = img.shape[0]
    if box_indices is None:
        if bx.dim() != 3 or bx.shape[0] != B or bx.shape[2] != 4:
            raise ValueError("with box_indices=None, boxes must be (B,S,4) with B = %d, got %s" % (B, tuple(bx.shape)))
        lead = tuple(bx.shape[:2])
        idx = None
    else:
        if bx.dim() != 2 or bx.shape[1] != 4:
            raise ValueError("boxes must be (M,4), got %s" % (tuple(bx.shape),))
        lead = (bx.shape[0],)
        idx = to_device(box_indices, torch.int32, o, "box_indices")
        if tuple(idx.shape) != lead:
            raise ValueError("box_indices must be (%d,), got %s" % (lead[0], tuple(idx.shape)))
    bx = bx.reshape(-1, 4)
    if o.kind == "torch":
        out = _CropAndResize.apply(img, bx, idx, ch, cw, extrapolation_value)
    else:
        out = _launch_forward(img, bx, idx, ch, cw, extrapolation_value)
    return from_device(out.reshape(lead + tuple(out.shape[1:])), o)

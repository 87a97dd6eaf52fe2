"""NumPy restatement of tf.image.crop_and_resize (bilinear) and its image gradient (tfrpn_crop_and_resize,
tfrpn_crop_and_resize_grad_image, include/tfrpn.h).  TEST INFRASTRUCTURE, not product.

TensorFlow's CPU kernels CropAndResize / CropAndResizeGradImage (crop_and_resize_op.cc), every float operation
rounded separately in float32:
  * box m, output row y: in_y = y1*(H-1) + y*((y2-y1)*(H-1)/(ch-1)) when ch > 1, else 0.5*(y1+y2)*(H-1) with y1+y2 in
    float32 and the rest in float64, rounded once; columns likewise;
  * a sample outside [0, L-1] or NaN is extrapolated (forward) and adds nothing (gradient);
  * top = floor, bottom = ceil, lerp = in - top; out = t + (b - t)*y_lerp, t / b = l + (r - l)*x_lerp;
  * a box_index outside [0,B) gives NaN rows and no gradient;
  * gradient: per sample dtop = (1 - y_lerp)*g, dbot = y_lerp*g and the four terms (1 - x_lerp)*dtop -> (top,left),
    x_lerp*dtop -> (top,right), (1 - x_lerp)*dbot -> (bottom,left), x_lerp*dbot -> (bottom,right), summed from +0
    in the order (m, y, x, term): ``np.add.at`` is unbuffered and applies its terms in index order.
Vectorised over boxes and channels, in chunks of boxes so that the corner gathers stay small.
"""
from __future__ import annotations

import numpy as np

F32 = np.float32
_CHUNK_ELEMS = 1 << 22   # output elements per chunk of boxes


def batched_index(M, B):
    """box_index of the batched layout (box_index NULL / None): box m belongs to image m // (M // B)"""
    if B < 1 or M % B:
        raise ValueError("M = %d is not a multiple of B = %d" % (M, B))
    return (np.arange(M) // (M // B)).astype(np.int32)


def sample_grid(lo, hi, L, n):
    """(M,) box edges -> (M, n) float32 sample coordinates along an axis of length L"""
    lo, hi = np.asarray(lo, F32), np.asarray(hi, F32)
    lmax = F32(L - 1)
    with np.errstate(all="ignore"):
        if n > 1:
            s = (hi - lo) * lmax / F32(n - 1)
            return (lo * lmax)[:, None] + np.arange(n, dtype=F32)[None, :] * s[:, None]
        return (0.5 * (lo + hi).astype(np.float64) * float(L - 1)).astype(F32)[:, None]


def axis_terms(coord, L):
    """-> inside mask, floor index, ceil index, lerp (0 where outside)"""
    ok = (coord >= 0) & (coord <= F32(L - 1))
    c = np.where(ok, coord, F32(0))
    lo = np.floor(c).astype(np.int64)
    with np.errstate(all="ignore"):
        lerp = np.where(ok, coord - lo.astype(F32), F32(0)).astype(F32)
    return ok, lo, np.ceil(c).astype(np.int64), lerp


def _chunks(M, per_box):
    step = max(1, _CHUNK_ELEMS // max(1, per_box))
    for m0 in range(0, M, step):
        yield slice(m0, min(M, m0 + step))


def _geometry(boxes, box_index, B, H, W, ch, cw):
    bi = np.asarray(box_index, np.int64)
    bad = (bi < 0) | (bi >= B)
    y = axis_terms(sample_grid(boxes[:, 0], boxes[:, 2], H, ch), H)
    x = axis_terms(sample_grid(boxes[:, 1], boxes[:, 3], W, cw), W)
    return np.where(bad, 0, bi), bad, y, x


def crop_and_resize(image, boxes, box_index, crop_size, extrapolation_value=0.0):
    """image (B,H,W,C), boxes (M,4), box_index (M,) or None (batched layout) -> (M,ch,cw,C) float32"""
    image = np.asarray(image, F32)
    boxes = np.asarray(boxes, F32).reshape(-1, 4)
    B, H, W, C = image.shape
    M = boxes.shape[0]
    ch, cw = (int(v) for v in crop_size)
    if box_index is None:
        box_index = batched_index(M, B)
    out = np.empty((M, ch, cw, C), F32)
    for sl in _chunks(M, ch * cw * C):
        b, bad, (yok, top, bot, yl), (xok, left, right, xl) = _geometry(boxes[sl], box_index[sl], B, H, W, ch, cw)
        bI = b[:, None, None]
        t_, b_, l_, r_ = top[:, :, None], bot[:, :, None], left[:, None, :], right[:, None, :]
        tl, tr, bl, br = image[bI, t_, l_], image[bI, t_, r_], image[bI, b_, l_], image[bI, b_, r_]
        xlv, ylv = xl[:, None, :, None], yl[:, :, None, None]
        t = tl + (tr - tl) * xlv
        bo = bl + (br - bl) * xlv
        o = t + (bo - t) * ylv
        ok = yok[:, :, None] & xok[:, None, :]
        o = np.where(ok[..., None], o, F32(extrapolation_value))
        o[bad] = np.nan
        out[sl] = o
    return out


def crop_and_resize_grad_image(grad, boxes, box_index, image_shape):
    """grad (M,ch,cw,C), boxes (M,4), box_index (M,) or None, image_shape (B,H,W,C) -> (B,H,W,C) float32"""
    grad = np.asarray(grad, F32)
    boxes = np.asarray(boxes, F32).reshape(-1, 4)
    B, H, W, C = (int(v) for v in image_shape)
    M, ch, cw, _ = grad.shape
    if box_index is None:
        box_index = batched_index(M, B)
    acc = np.zeros(B * H * W * C, F32)
    lanes = np.arange(C, dtype=np.int64)
    for sl in _chunks(M, 4 * ch * cw * C):
        b, bad, (yok, top, bot, yl), (xok, left, right, xl) = _geometry(boxes[sl], box_index[sl], B, H, W, ch, cw)
        g = grad[sl]
        dtop = (F32(1) - yl)[:, :, None, None] * g
        dbot = yl[:, :, None, None] * g
        wl, wr = (F32(1) - xl)[:, None, :, None], xl[:, None, :, None]
        terms = np.stack([wl * dtop, wr * dtop, wl * dbot, wr * dbot], axis=3)               # (m, ch, cw, 4, C)
        rows = np.stack([top, top, bot, bot], axis=-1)[:, :, None, :]                         # (m, ch, 1, 4)
        cols = np.stack([left, right, left, right], axis=-1)[:, None, :, :]                   # (m, 1, cw, 4)
        pix = (b[:, None, None, None] * H + rows) * W + cols                                 # (m, ch, cw, 4)
        live = yok[:, :, None] & xok[:, None, :] & ~bad[:, None, None]
        idx = pix[live][..., None] * C + lanes                                                # (k, 4, C)
        np.add.at(acc, idx.reshape(-1), terms[live].reshape(-1))
    return acc.reshape(B, H, W, C)

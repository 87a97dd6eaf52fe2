"""NumPy restatement of the second stage's box-head losses and their gradients (tfrpn_roi_head_losses,
include/tfrpn.h).  TEST INFRASTRUCTURE, not product.

Per row, every float operation rounded separately in float32:
  * a row takes part iff 0 <= label < C, and is fg iff 1 <= label < C;
  * m = max_c x_c (NaN ignored), e_c = exp(x_c - m), s = sum of e_c, term = log(s) - (x[label] - m); a NaN logit makes
    s, and so the term and the row's gradient, NaN;
  * the fg row's Huber: e = pred - target, a = |e|, q = min(a, delta) (NaN ignored), 0.5*(q*q) + delta*(a - q),
    summed over the 4 coordinates in order; pred is the label's slice (q = C) or slice 0 (q = 1);
  * the loss sums in float64: cls = sum / #rows (NaN for none), reg = sum / max(1, #fg or #rows), each rounded to
    float32 once;
  * argmax: the first index of the maximum; a row with a NaN logit is never correct;
  * gradients: (e_c / s - [c == label]) * inv_rows * scale[0] and huber_grad * inv_reg * scale[1], inv = 1 / count
    in float32, 0 elsewhere.
The kernel sums s in another order, and CUDA's expf / logf are not NumPy's, so cls_loss and grad_logits agree to
float32 accuracy; reg_loss agrees to float64-sum accuracy and grad_deltas bit for bit.
"""
from __future__ import annotations

import numpy as np

F32 = np.float32
NORMALIZERS = ("fg", "rows")


def huber_term(t, p, delta):
    """keras huber_loss elementwise in float32 (csrc/losses.cu huber_term)"""
    delta = F32(delta)
    a = np.abs(p - t)
    q = np.fmin(a, delta)
    return F32(0.5) * (q * q) + delta * (a - q)


def huber_grad(t, p, delta):
    """d huber / d pred: e where |e| <= delta, else +-delta (NaN e gives -delta, as the kernel's branches)"""
    delta = F32(delta)
    e = p - t
    return np.where(np.abs(e) <= delta, e, np.where(e > 0, delta, -delta)).astype(F32)


def roi_head_losses(logits, deltas, labels, targets, huber_delta=1.0, normalize="fg", scale=None):
    """logits (B,S,C), deltas (B,S,q,4), labels (B,S), targets (B,S,4) -> dict of cls_loss, reg_loss (float32),
    n_rows, n_fg, n_correct, n_fg_correct (int) and grad_logits, grad_deltas (float32, shaped like the inputs);
    scale: None or the two upstream gradients"""
    x = np.asarray(logits, F32)
    B, S, C = x.shape
    x = x.reshape(-1, C)
    d = np.asarray(deltas, F32)
    q = d.shape[2]
    d = d.reshape(-1, q, 4)
    lab = np.asarray(labels).reshape(-1).astype(np.int64)
    t = np.asarray(targets, F32).reshape(-1, 4)
    s0, s1 = (F32(1), F32(1)) if scale is None else (F32(scale[0]), F32(scale[1]))
    part = (lab >= 0) & (lab < C)
    fg = (lab >= 1) & (lab < C)
    rows, fgr = np.flatnonzero(part), np.flatnonzero(fg)

    xp, lp = x[rows], lab[rows]
    nan = np.isnan(xp).any(axis=1)
    m = np.fmax.reduce(xp, axis=1, initial=-np.inf).astype(F32)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        e = np.exp(xp - m[:, None])
        s = e.sum(axis=1, dtype=F32)
        term = np.log(s) - (xp[np.arange(len(rows)), lp] - m)
    ok = ~nan & (np.argmax(np.where(np.isnan(xp), -np.inf, xp), axis=1) == lp)

    sel = lab[fgr] if q == C else np.zeros(len(fgr), np.int64)
    p, tt = d[fgr, sel], t[fgr]
    h = huber_term(tt, p, huber_delta)
    row = ((h[:, 0] + h[:, 1]) + h[:, 2]) + h[:, 3]

    n_rows, n_fg = len(rows), len(fgr)
    norm = max(1, n_rows if normalize == "rows" else n_fg)
    cls = F32(term.astype(np.float64).sum() / n_rows) if n_rows else F32(np.nan)
    reg = F32(row.astype(np.float64).sum() / norm)

    with np.errstate(divide="ignore"):
        inv_rows = F32(1) / F32(n_rows)
    inv_reg = F32(1) / F32(norm)
    gl = np.zeros_like(x)
    with np.errstate(invalid="ignore"):
        pr = e / s[:, None]
        onehot = np.zeros_like(pr)
        onehot[np.arange(len(rows)), lp] = 1
        gl[rows] = ((pr - onehot) * inv_rows) * s0
    gd = np.zeros_like(d)
    gd[fgr, sel] = (huber_grad(tt, p, huber_delta) * inv_reg) * s1
    return dict(cls_loss=cls, reg_loss=reg, n_rows=n_rows, n_fg=n_fg, n_correct=int(ok.sum()),
                n_fg_correct=int(ok[fg[rows]].sum()), grad_logits=gl.reshape(B, S, C), grad_deltas=gd.reshape(B, S, q, 4))

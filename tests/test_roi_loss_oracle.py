"""CPU checks of the box-head loss restatement (oracle/roi_loss_oracle.py, tfrpn_roi_head_losses): hand-derived cases,
torchvision's fastrcnn_loss on the rows without padding, torch autograd of the same composition for the gradients,
and the ctypes mirrors of the new structs against what gcc makes of include/tfrpn.h."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import roi_loss_oracle as L

F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def case(B, S, Cn, q, rng, fg_frac=0.3, pad_frac=0.2):
    """random logits / deltas / targets; labels: fg, background and -1 padding"""
    x = rng.normal(0, 2, size=(B, S, Cn)).astype(F32)
    d = rng.normal(0, 1, size=(B, S, q, 4)).astype(F32)
    t = rng.normal(0, 1, size=(B, S, 4)).astype(F32)
    u = rng.uniform(size=(B, S))
    lab = np.where(u < fg_frac, rng.integers(1, Cn, size=(B, S)), 0)
    lab = np.where(u > 1 - pad_frac, -1, lab).astype(np.int32)
    t[lab <= 0] = 0
    return x, d, lab, t


def test_uniform_logits_give_log_c():
    for Cn in (2, 21, 81, 1024):
        x = np.full((2, 5, Cn), 3.5, F32)
        lab = np.array([[0, 1, Cn - 1, -1, 0], [1, 1, -1, -1, 0]], np.int32)
        r = L.roi_head_losses(x, np.zeros((2, 5, 1, 4), F32), lab, np.zeros((2, 5, 4), F32))
        assert r["n_rows"] == 7 and r["n_fg"] == 4
        assert float(r["cls_loss"]) == pytest.approx(math.log(Cn), rel=1e-6)
        # uniform: every row's argmax is class 0, so only the background rows are correct
        assert r["n_correct"] == 3 and r["n_fg_correct"] == 0
        g = r["grad_logits"]
        assert np.all(g[lab < 0] == 0)
        assert float(g[0, 0, 1]) == pytest.approx(1.0 / Cn / 7, rel=1e-6)
        assert float(g[0, 0, 0]) == pytest.approx((1.0 / Cn - 1) / 7, rel=1e-6)


def test_huber_kink_and_zero_target_fg_row():
    """|e| == delta is on the quadratic side (term 0.5 delta^2, gradient e); just above it the linear side; an fg
    row whose target deltas are all zero (an appended GT row) still counts"""
    delta = F32(0.5)
    x = np.zeros((1, 3, 4), F32)
    lab = np.array([[2, 3, 0]], np.int32)
    t = np.zeros((1, 3, 4), F32)
    d = np.zeros((1, 3, 4, 4), F32)
    d[0, 0, 2] = [0.5, -0.5, 0.0, np.nextafter(F32(0.5), F32(1))]
    d[0, 1, 3] = [1.0, 0, 0, 0]
    d[0, 1, 2] = [9, 9, 9, 9]                          # not row 1's class: not read
    d[0, 2, 0] = [9, 9, 9, 9]                          # background: no box loss
    r = L.roi_head_losses(x, d, lab, t, huber_delta=delta)
    above = np.nextafter(F32(0.5), F32(1))
    row0 = F32(0.125) + F32(0.125) + F32(0) + (F32(0.125) + F32(0.5) * (above - F32(0.5)))
    row1 = F32(0.125) + F32(0.5) * F32(0.5)
    assert r["n_fg"] == 2
    assert float(r["reg_loss"]) == pytest.approx((float(row0) + float(row1)) / 2, rel=1e-7)
    gd = r["grad_deltas"]
    inv = F32(0.5)
    assert gd[0, 0, 2].tolist() == [0.5 * inv, -0.5 * inv, 0.0, 0.5 * inv]
    assert gd[0, 1, 3].tolist() == [0.5 * inv, 0, 0, 0]
    assert np.count_nonzero(gd) == 4


def test_rows_that_take_no_part_and_no_rows():
    rng = np.random.default_rng(1)
    x, d, _, t = case(1, 6, 5, 5, rng)
    lab = np.array([[-1, 5, -5, 2, 0, 7]], np.int32)
    r = L.roi_head_losses(x, d, lab, t)
    assert r["n_rows"] == 2 and r["n_fg"] == 1
    only = L.roi_head_losses(x[:, [3, 4]], d[:, [3, 4]], lab[:, [3, 4]], t[:, [3, 4]])
    assert r["cls_loss"] == only["cls_loss"] and r["reg_loss"] == only["reg_loss"]
    g = r["grad_logits"]
    assert np.all(g[0, [0, 1, 2, 5]] == 0) and np.all(r["grad_deltas"][0, [0, 1, 2, 4, 5]] == 0)
    none = L.roi_head_losses(x, d, np.full((1, 6), -1, np.int32), t)
    assert np.isnan(none["cls_loss"]) and none["reg_loss"] == 0 and none["n_rows"] == 0 and none["n_fg"] == 0
    assert np.all(none["grad_logits"] == 0) and np.all(none["grad_deltas"] == 0)


def test_normalizers():
    rng = np.random.default_rng(2)
    x, d, lab, t = case(3, 40, 7, 1, rng)
    fg = L.roi_head_losses(x, d, lab, t, normalize="fg")
    rows = L.roi_head_losses(x, d, lab, t, normalize="rows")
    assert fg["cls_loss"] == rows["cls_loss"]
    assert float(fg["reg_loss"]) * fg["n_fg"] == pytest.approx(float(rows["reg_loss"]) * rows["n_rows"], rel=1e-6)
    ratio = F32(1) / F32(rows["n_rows"]) / (F32(1) / F32(fg["n_fg"]))
    nz = fg["grad_deltas"] != 0
    assert np.allclose(rows["grad_deltas"][nz] / fg["grad_deltas"][nz], ratio, rtol=1e-6)


def test_argmax_ties_and_nan_rows():
    x = np.array([[[1, 3, 3, 0], [5, 5, 5, 5], [0, 2, np.nan, 1], [np.nan] * 4, [2, 1, 2, 1]]], F32)
    lab = np.array([[2, 0, 1, 0, 0]], np.int32)
    r = L.roi_head_losses(x, np.zeros((1, 5, 1, 4), F32), lab, np.zeros((1, 5, 4), F32))
    assert r["n_correct"] == 2 and r["n_fg_correct"] == 0          # rows 1 and 4: ties go to the lower index
    assert np.isnan(r["cls_loss"])                                   # NaN rows make the mean NaN
    g = r["grad_logits"]
    assert np.all(np.isnan(g[0, 2])) and np.all(np.isnan(g[0, 3])) and np.all(np.isfinite(g[0, [0, 1, 4]]))
    ok = L.roi_head_losses(x[:, [0, 1, 4]], np.zeros((1, 3, 1, 4), F32), lab[:, [0, 1, 4]], np.zeros((1, 3, 4), F32))
    assert np.isfinite(ok["cls_loss"])


@pytest.mark.parametrize("q", ["C", 1])
def test_against_torchvision_fastrcnn_loss(q):
    """fastrcnn_loss (F.cross_entropy + smooth_l1(beta = 1/9, sum) / labels.numel()) in float64 on the rows
    without padding: cls equal, reg(delta = 1/9, normalize='rows') * 9 equal to its box_loss"""
    torch = pytest.importorskip("torch")
    roi_heads = pytest.importorskip("torchvision.models.detection.roi_heads")
    rng = np.random.default_rng(3)
    B, S, Cn = 4, 64, 21
    qq = Cn if q == "C" else 1
    x, d, lab, t = case(B, S, Cn, qq, rng)
    keep = lab >= 0
    beta = 1.0 / 9
    r = L.roi_head_losses(x, d, lab, t, huber_delta=beta, normalize="rows")
    lx = torch.from_numpy(x[keep]).double()
    ld = torch.from_numpy(np.broadcast_to(d, (B, S, Cn, 4)).copy()[keep].reshape(-1, Cn * 4)).double()
    cls, box = roi_heads.fastrcnn_loss(lx, ld, [torch.from_numpy(lab[keep].astype(np.int64))],
                                       [torch.from_numpy(t[keep]).double()])
    assert float(r["cls_loss"]) == pytest.approx(float(cls), rel=2e-6)
    assert float(r["reg_loss"]) * 9 == pytest.approx(float(box), rel=2e-6)


@pytest.mark.parametrize("normalize,q", [("fg", "C"), ("rows", "C"), ("fg", 1), ("rows", 1)])
def test_gradients_against_torch_autograd(normalize, q):
    """the oracle's gradients, with upstream scales, against torch CPU autograd of the same composition in float64"""
    torch = pytest.importorskip("torch")
    F = torch.nn.functional
    rng = np.random.default_rng(4)
    B, S, Cn = 3, 50, 9
    qq = Cn if q == "C" else 1
    x, d, lab, t = case(B, S, Cn, qq, rng)
    delta, scale = 0.7, (F32(1.5), F32(-0.25))
    r = L.roi_head_losses(x, d, lab, t, huber_delta=delta, normalize=normalize, scale=scale)
    X = torch.from_numpy(x).double().requires_grad_(True)
    D = torch.from_numpy(d).double().requires_grad_(True)
    lab_t = torch.from_numpy(lab.astype(np.int64))
    part = (lab_t >= 0) & (lab_t < Cn)
    fg = (lab_t >= 1) & (lab_t < Cn)
    cls = F.cross_entropy(X[part], lab_t[part])
    sel = lab_t[fg] if qq == Cn else torch.zeros_like(lab_t[fg])
    pred = D[fg.nonzero(as_tuple=True) + (sel,)]
    hub = F.huber_loss(pred, torch.from_numpy(t).double()[fg], reduction="sum", delta=delta)
    reg = hub / max(1, int(part.sum() if normalize == "rows" else fg.sum()))
    (float(scale[0]) * cls + float(scale[1]) * reg).backward()
    assert float(r["cls_loss"]) == pytest.approx(cls.item(), rel=2e-6)
    assert float(r["reg_loss"]) == pytest.approx(reg.item(), rel=2e-6)
    np.testing.assert_allclose(r["grad_logits"], X.grad.numpy(), rtol=2e-6, atol=1e-8)
    np.testing.assert_allclose(r["grad_deltas"], D.grad.numpy(), rtol=1e-6, atol=0)


def test_ctypes_structs_match_header_layout(tmp_path):
    from tfrpn import _lib
    pairs = {"tfrpn_roi_loss_cfg": _lib.RoiLossCfg, "tfrpn_roi_loss_out": _lib.RoiLossOut}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tfrpn.h"', 'int main(void) {']
    for cname, cls in pairs.items():
        lines.append('printf("%s size %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ['return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    got = {tuple(l.split()[:2]): int(l.split()[2]) for l in out.splitlines()}
    for cname, cls in pairs.items():
        assert got[(cname, "size")] == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, (cname, fname)
    assert C.sizeof(_lib.RoiLossOut) == 32

"""CPU checks of the box-head detections restatement (oracle/roi_det_oracle.py, tfrpn_roi_head_detections):
hand-derived cases, agreement with an independent torch-CPU composition (softmax, the same decode op order, clip,
torchvision's remove_small_boxes rule and a per-class torchvision.ops.nms), and the ctypes mirror of
tfrpn_roi_det_cfg against what gcc makes of include/tfrpn.h."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import roi_det_oracle as D

F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VAR = (0.1, 0.1, 0.2, 0.2)


def run(rois, probs, deltas, valid=None, **kw):
    kw.setdefault("score_threshold", 0.05)
    return D.roi_head_detections(rois, probs, deltas, valid, **kw)


def one_image(S, Cn, q, rng):
    rois = np.sort(rng.uniform(0.05, 0.95, size=(1, S, 2, 2)), axis=2).transpose(0, 1, 3, 2).reshape(1, S, 4)
    return rois.astype(F32), np.zeros((1, S, q, 4), F32)


def test_class_zero_is_never_detected():
    rng = np.random.default_rng(0)
    rois, d = one_image(6, 3, 3, rng)
    p = np.tile(np.array([0.9, 0.06, 0.04], F32), (1, 6, 1))   # background wins every row
    nb, ns, nc, nv, ni = run(rois, p, d, iou_threshold=1.0, max_total_size=20)
    assert nv[0] == 6 and np.all(nc[0, :6] == 1) and np.all(ns[0, :6] == F32(0.06))
    assert sorted(ni[0, :6]) == list(range(6)) and np.all(ni[0, 6:] == -1) and np.all(nc[0, 6:] == 0)


def test_rows_beyond_valid_are_never_detected():
    rng = np.random.default_rng(1)
    rois, d = one_image(8, 2, 1, rng)
    rois = np.concatenate([rois, rois])
    d = np.concatenate([d, d])
    p = np.tile(np.array([0.1, 0.9], F32), (2, 8, 1))
    for valid, want in (([3, 0], [3, 0]), ([-5, 100], [0, 8])):
        nb, ns, nc, nv, ni = run(rois, p, d, np.array(valid, np.int32), iou_threshold=1.0, max_total_size=10)
        assert nv.tolist() == want
        for b in range(2):
            assert sorted(ni[b, :nv[b]]) == list(range(want[b]))


def test_min_size_drops_clipped_and_nan_boxes():
    rois = np.array([[[0.2, 0.2, 0.4, 0.4], [1.2, 0.2, 1.5, 0.4], [0.2, 0.2, 0.4, 0.4], [0.5, 0.5, 0.6, 0.6]]], F32)
    d = np.zeros((1, 4, 1, 4), F32)
    d[0, 2, 0, 2] = np.nan                          # NaN height
    p = np.tile(np.array([0.0, 1.0], F32), (1, 4, 1))
    kw = dict(iou_threshold=1.0, max_total_size=10)
    assert run(rois, p, d, **kw)[3][0] == 4         # no size filter: NaN clips to 0, the outside box to a line
    nb, ns, nc, nv, ni = run(rois, p, d, min_size=0.05, **kw)
    assert nv[0] == 2 and sorted(ni[0, :2]) == [0, 3]   # row 1 clips to zero height, row 2 has a NaN extent
    assert run(rois, p, d, min_size=0.15, **kw)[3][0] == 1   # row 3 is 0.1 high


def test_clamp_keeps_nan_and_caps_log_scale():
    d = np.array([[[[0.0, 0.0, np.nan, 1000.0], [0.0, 0.0, -np.inf, np.inf]]]], F32)
    s = D.scale_deltas(d, VAR, max_log_scale=4.0)
    assert np.isnan(s[0, 0, 0, 2]) and s[0, 0, 0, 3] == F32(4.0)
    assert s[0, 0, 1, 2] == -np.inf and s[0, 0, 1, 3] == F32(4.0)
    s = D.scale_deltas(d, VAR)                       # +inf: no clamp
    assert s[0, 0, 0, 3] == F32(1000.0) * F32(0.2) and s[0, 0, 1, 3] == np.inf


@pytest.mark.parametrize("Cn,per_class,total,want", [(2, 5, 100, 5), (5, 3, 100, 12), (5, 3, 7, 7), (21, 100, 100, 100)])
def test_row_count_rule_with_pad_per_class(Cn, per_class, total, want):
    rng = np.random.default_rng(Cn)
    rois, d = one_image(4, Cn, 1, rng)
    p = np.full((1, 4, Cn), 1.0 / Cn, F32)
    nb, ns, nc, nv, ni = run(rois, p, d, max_output_size_per_class=per_class, max_total_size=total,
                             pad_per_class=True, score_threshold=0.0)
    assert nb.shape == (1, want, 4) and ni.shape == (1, want)
    assert run(rois, p, d, max_output_size_per_class=per_class, max_total_size=total)[0].shape == (1, total, 4)


def test_class_agnostic_deltas_share_one_box():
    rng = np.random.default_rng(3)
    rois, _ = one_image(5, 4, 1, rng)
    d = rng.normal(0, 1, size=(1, 5, 1, 4)).astype(F32)
    p = np.tile(np.array([0.1, 0.3, 0.3, 0.3], F32), (1, 5, 1))
    nb, ns, nc, nv, ni = run(rois, p, d, iou_threshold=1.0, max_total_size=15)
    boxes = D.decode(rois, d, VAR)
    assert nv[0] == 15
    for r in range(15):
        assert np.array_equal(nb[0, r], boxes[0, ni[0, r], 0])
    assert sorted(nc[0].tolist()) == [1.0] * 5 + [2.0] * 5 + [3.0] * 5


def test_softmax_nan_row():
    x = np.array([[[1.0, np.nan, 0.5], [1.0, 2.0, 3.0]]], F32)
    p = D.softmax(x)
    assert np.all(np.isnan(p[0, 0])) and abs(float(p[0, 1].sum()) - 1) < 1e-6


def torch_composition(rois, x, d, valid, clip, min_size, mls, per_class, total, iou, sthr):
    """softmax, decode in the reference's op order, clip, remove_small_boxes, per-class torchvision nms, merge"""
    torch = pytest.importorskip("torch")
    tv = pytest.importorskip("torchvision")
    P = torch.softmax(torch.from_numpy(x), -1)
    dd = torch.from_numpy(d) * torch.tensor(VAR, dtype=torch.float32)
    dd = torch.cat([dd[..., :2], torch.clamp(dd[..., 2:], max=mls)], -1)
    r = torch.from_numpy(rois)[:, :, None, :]
    aw, ah = r[..., 3] - r[..., 1], r[..., 2] - r[..., 0]
    acx, acy = r[..., 1] + 0.5 * aw, r[..., 0] + 0.5 * ah
    w, h = torch.exp(dd[..., 3]) * aw, torch.exp(dd[..., 2]) * ah
    cx, cy = dd[..., 1] * aw + acx, dd[..., 0] * ah + acy
    y1, x1 = cy - 0.5 * h, cx - 0.5 * w
    boxes = torch.stack([y1, x1, h + y1, w + x1], -1)
    if clip:
        boxes = boxes.clamp(0, 1)
    B, S, Cn = x.shape
    q = d.shape[2]
    out = []
    for b in range(B):
        rows = torch.arange(S) < min(max(int(valid[b]), 0), S)
        dets = []
        for c in range(1, Cn):
            bx = boxes[b, :, c if q > 1 else 0]
            keep = rows & (P[b, :, c] > sthr)
            if min_size > 0:   # torchvision.ops.remove_small_boxes' rule
                keep &= ((bx[:, 2] - bx[:, 0]) >= min_size) & ((bx[:, 3] - bx[:, 1]) >= min_size)
            idx = torch.nonzero(keep).flatten()
            k = tv.ops.nms(bx[idx], P[b, idx, c], iou)[:per_class]   # IoU does not care that boxes are (y, x)
            dets += [(float(P[b, i, c]), c, pos, int(i)) for pos, i in enumerate(idx[k])]
        dets.sort(key=lambda t: (-t[0], t[1], t[2]))
        out.append(dets[:total])
    return out, boxes.numpy(), P.numpy()


@pytest.mark.parametrize("Cn,q,min_size,mls", [(5, 5, 0.0, float("inf")), (5, 1, 0.02, float("inf")),
                                               (21, 21, 0.01, 1.0), (3, 1, 0.0, 0.5)])
def test_agrees_with_torch_composition(Cn, q, min_size, mls):
    rng = np.random.default_rng(Cn * 10 + q)
    B, S = 3, 120
    ctr = rng.uniform(0.1, 0.9, size=(B, S, 2))
    sz = rng.uniform(0.05, 0.4, size=(B, S, 2))
    rois = np.concatenate([ctr - sz / 2, ctr + sz / 2], -1).astype(F32)
    x = rng.normal(0, 2, size=(B, S, Cn)).astype(F32)
    d = rng.normal(0, 2, size=(B, S, q, 4)).astype(F32)
    valid = np.array([S, 70, 0], np.int32)
    per_class, total, iou, sthr = 20, 60, 0.5, 0.05
    want, boxes, P = torch_composition(rois, x, d, valid, True, min_size, mls, per_class, total, iou, sthr)
    p = D.softmax(x)
    np.testing.assert_allclose(p, P, rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(D.decode(rois, d, VAR, mls, True), boxes, rtol=0, atol=2e-6)
    nb, ns, nc, nv, ni = run(rois, p, d, valid, max_log_scale=mls, min_size=min_size, max_output_size_per_class=per_class,
                             max_total_size=total, iou_threshold=iou, score_threshold=sthr)
    for b in range(B):
        assert nv[b] == len(want[b])
        assert [int(c) for c in nc[b, :nv[b]]] == [t[1] for t in want[b]]
        assert ni[b, :nv[b]].tolist() == [t[3] for t in want[b]]
        np.testing.assert_allclose(ns[b, :nv[b]], [t[0] for t in want[b]], rtol=2e-6)
    assert nv[2] == 0


def test_ctypes_struct_matches_header_layout(tmp_path):
    from tfrpn import _lib
    cls = _lib.RoiDetCfg
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tfrpn.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(tfrpn_roi_det_cfg));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(tfrpn_roi_det_cfg, %s));' % (fname, fname))
    lines += ['return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    got = {l.split()[0]: int(l.split()[1]) for l in out.splitlines()}
    assert got["size"] == C.sizeof(cls)
    for fname, _ in cls._fields_:
        assert got[fname] == getattr(cls, fname).offset, fname

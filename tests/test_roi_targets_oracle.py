"""The NumPy restatement of the second stage's RoI target assignment (oracle/roi_oracle.py): one hand-derived case per
rule of include/tfrpn.h, the sampler's invariants, a cross-check of the matching against torchvision's Matcher, and
the ctypes layout of tfrpn_roi_target_cfg.  CPU only; tests/test_roi_targets_gpu.py holds the kernel to these."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import roi_oracle as R
from oracle import rpn_oracle as O

F32 = np.float32
NAN = float("nan")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
UNIT = [0.0, 0.0, 1.0, 1.0]


def run(rois, gt, labels, valid=None, **kw):
    kw.setdefault("num_classes", 5)
    return R.roi_targets(np.asarray(rois, F32), np.asarray(gt, F32), np.asarray(labels, np.int32), valid, **kw)


def random_boxes(rng, shape, lo=0.05, hi=0.5):
    """boxes with positive extent inside [0, 1]"""
    c = rng.uniform(0.0, 1.0, size=shape + (2,))
    s = rng.uniform(lo, hi, size=shape + (2,))
    return np.clip(np.concatenate([c - s / 2, c + s / 2], axis=-1), 0, 1).astype(F32)


# ---- hand-derived cases --------------------------------------------------------------------------------------------
def strip_rows():
    """rows [0, 0, 1, w] against the unit GT: IoU exactly w (dyadic)"""
    ws = [1.0, 0.75, 0.5, 0.25, 0.125]
    return np.asarray([[0.0, 0.0, 1.0, w] for w in ws], F32)[None], np.asarray([[UNIT]], F32), np.asarray([[3]])


def test_iou_exactly_at_each_threshold():
    rois, gt, lab = strip_rows()
    o = run(rois, gt, lab, append_gt=False, fg_iou_threshold=0.75, bg_iou_high=0.5, bg_iou_low=0.25,
            total_pos=8, total_neg=8)
    assert o["max_iou"][0].tolist() == [1.0, 0.75, 0.5, 0.25, 0.125]
    assert o["fg_cand"][0].tolist() == [True, True, False, False, False]     # >= fg_iou_threshold
    assert o["bg_cand"][0].tolist() == [False, False, False, True, False]    # 0.5 = bg_iou_high: neither; 0.25 = low: bg
    assert o["src"][0, :3].tolist() == [0, 1, 3] and o["labels"][0, :3].tolist() == [3, 3, 0]
    assert o["counts"][0].tolist() == [2, 3]
    d = run(rois, gt, lab, append_gt=False, total_pos=8, total_neg=8)       # defaults: 0.5 is fg
    assert d["fg_cand"][0].tolist() == [True, True, True, False, False]
    assert d["bg_cand"][0].tolist() == [False, False, False, True, True]


def test_overlapping_intervals_fg_wins():
    rois, gt, lab = strip_rows()
    o = run(rois, gt, lab, append_gt=False, fg_iou_threshold=0.5, bg_iou_high=1.0, bg_iou_low=0.0)
    assert o["fg_cand"][0].tolist() == [True, True, True, False, False]
    assert not (o["fg_cand"] & o["bg_cand"]).any() and o["bg_cand"][0, 3:].all()


def test_equal_iou_lower_gt_wins():
    rois = [[UNIT]]
    # two different GT boxes at IoU 0.5 each, and two copies of one box with different labels
    o = run(rois, [[[0, 0.5, 1, 1], [0, 0, 1, 0.5]]], [[4, 2]], append_gt=False)
    assert o["argmax"][0, 0] == 0 and o["labels"][0, 0] == 4
    o = run(rois, [[[0, 0, 1, 0.5], [0, 0.5, 1, 1]]], [[4, 2]], append_gt=False)
    assert o["argmax"][0, 0] == 0 and o["labels"][0, 0] == 4
    o = run(rois, [[[0, 0.5, 1, 1], UNIT, UNIT]], [[1, 3, 2]], append_gt=True)
    assert o["argmax"][0].tolist() == [1, 0, 1, 1]        # duplicate GT rows match the first copy
    assert o["labels"][0, :4].tolist() == [3, 1, 3, 3]


@pytest.mark.parametrize("label", [-1, 0, 5, 10])
def test_labels_outside_classes_take_no_part(label):
    o = run([[UNIT, [0, 0, 1, 0.5]]], [[UNIT, UNIT]], [[label, 2]], num_classes=5, total_pos=4, total_neg=4)
    assert o["argmax"][0].tolist() == [1, 1, -1, 1]       # GT 0 never matches; its appended row takes no part
    assert o["max_iou"][0].tolist() == [1.0, 0.5, -1.0, 1.0]
    assert o["src"][0, :3].tolist() == [0, 1, 3] and o["labels"][0, :3].tolist() == [2, 2, 2]
    assert o["counts"][0].tolist() == [3, 3]


@pytest.mark.parametrize("valid,n_part", [(-3, 0), (0, 0), (4, 4), (9, 4)])
def test_valid_is_clamped(valid, n_part):
    rois = np.asarray([[UNIT, [0, 0, 1, 0.75], [0, 0, 1, 0.125], [0, 0, 0.5, 0.5]]], F32)
    o = run(rois, [[UNIT]], [[1]], valid=[valid], total_pos=8, total_neg=8)
    assert (o["max_iou"][0, :4] >= 0).sum() == n_part and o["max_iou"][0, 4] == 1.0
    assert o["counts"][0, 1] == n_part + 1 and (o["argmax"][0, n_part:4] == -1).all()


def test_proposals_all_miss_only_gt_rows_are_fg():
    rois = np.tile(np.asarray([[0.75, 0.75, 1, 1]], F32), (1, 6, 1))
    gt = np.asarray([[[0, 0, 0.5, 0.5], [0, 0, 0.25, 0.5], [0, 0, 0, 0]]], F32)
    o = run(rois, gt, [[1, 2, -1]], total_pos=4, total_neg=12)
    assert o["fg_cand"][0].tolist() == [False] * 6 + [True, True, False]
    assert o["src"][0, :2].tolist() == [6, 7] and o["labels"][0, :2].tolist() == [1, 2]
    assert np.array_equal(o["rois"][0, :2], gt[0, :2]) and (o["deltas"][0, :2] == 0).all()   # a GT row encodes to 0
    assert o["argmax"][0, 7] == 1 and o["max_iou"][0, 7] == 1.0   # GT 1's row: 0.5 against GT 0, 1.0 against itself
    assert o["counts"][0].tolist() == [2, 8] and o["src"][0, 2:8].tolist() == list(range(6))


def test_nan_inverted_and_zero_area_boxes():
    rois = np.asarray([[[NAN, 0, 1, 1], [1, 1, 0, 0], [0.5, 0, 0.5, 1], [0, 0, 1, 0.5]]], F32)
    gt = np.asarray([[UNIT, [0.5, 0.5, 0.5, 0.5], [1, 0, 0, 1], [0, NAN, 1, 1]]], F32)
    o = run(rois, gt, [[1, 2, 3, 4]], total_pos=8, total_neg=8)
    # NaN row: NaN scores -> +0; inverted (positive area, no extent): +0; zero-area line: +0; the strip: 0.5 with GT 0
    assert o["max_iou"][0, :4].tolist() == [0.0, 0.0, 0.0, 0.5] and o["argmax"][0, :4].tolist() == [0, 0, 0, 0]
    # GT rows: unit box 1.0; the point vs itself 0/0 = NaN -> +0; the inverted box vs itself scores -0 or NaN -> +0
    assert o["max_iou"][0, 4:].tolist() == [1.0, 0.0, 0.0, 0.0]
    assert o["fg_cand"][0].tolist() == [False, False, False, True, True, False, False, False]
    assert o["counts"][0].tolist() == [2, 8]


def test_no_gt_takes_part_every_row_is_bg():
    rois = random_boxes(np.random.default_rng(1), (1, 7))
    o = run(rois, [[UNIT, UNIT]], [[0, -1]], total_pos=2, total_neg=14)
    assert (o["max_iou"][0, :7] == 0).all() and (o["argmax"][0] == -1).all() and (o["max_iou"][0, 7:] == -1).all()
    assert o["bg_cand"][0, :7].all() and o["counts"][0].tolist() == [0, 7]
    assert o["labels"][0, :7].tolist() == [0] * 7 and o["labels"][0, 7:].tolist() == [-1] * 9
    assert (o["src"][0, 7:] == -1).all() and (o["rois"][0, 7:] == 0).all()
    assert run(rois, [[UNIT]], [[0]], bg_iou_low=0.25)["counts"][0].tolist() == [0, 0]   # +0 is below bg_iou_low


def quota_case(n_fg, n_bg, total_pos, total_neg, seed=0):
    rows = [[0, 0, 1, 1]] * n_fg + [[0, 0, 1, 0.25]] * n_bg
    return run(np.asarray([rows], F32), [[UNIT]], [[1]], append_gt=False, total_pos=total_pos, total_neg=total_neg,
               seed=seed, offset=5)


@pytest.mark.parametrize("n_fg", [3, 4, 9])
def test_fg_below_at_and_above_total_pos(n_fg):
    o = quota_case(n_fg, 40, 4, 12)
    kept = o["fg_keep"][0]
    assert kept.sum() == min(n_fg, 4) and not (kept & ~o["fg_cand"][0]).any()
    assert o["counts"][0].tolist() == [min(n_fg, 4), 16]
    assert o["src"][0, :min(n_fg, 4)].tolist() == np.flatnonzero(kept).tolist()   # ascending row order


@pytest.mark.parametrize("n_bg", [5, 12, 30])
def test_bg_below_at_and_above_quota(n_bg):
    o = quota_case(4, n_bg, 4, 12)                        # quota 16 - 4 = 12
    assert o["bg_keep"][0].sum() == min(n_bg, 12) and o["counts"][0].tolist() == [4, 4 + min(n_bg, 12)]
    assert o["src"][0, 4:4 + min(n_bg, 12)].tolist() == np.flatnonzero(o["bg_keep"][0]).tolist()
    o = quota_case(2, n_bg, 4, 12)                        # fewer fg: the bg quota grows to 14
    assert o["bg_keep"][0].sum() == min(n_bg, 14)


def test_zero_quotas():
    o = quota_case(6, 20, 0, 8)
    assert o["counts"][0].tolist() == [0, 8] and (o["labels"][0] == 0).all() and (o["src"][0] >= 6).all()
    o = quota_case(6, 20, 4, 0)
    assert o["counts"][0].tolist() == [4, 4] and (o["labels"][0] == 1).all()
    o = quota_case(2, 20, 4, 0)
    assert o["counts"][0].tolist() == [2, 4] and o["labels"][0].tolist() == [1, 1, 0, 0]


def test_fg_deltas_are_the_rpn_encoding():
    rng = np.random.default_rng(2)
    rois = random_boxes(rng, (1, 30))
    gt = rois[:, :3] + F32(0.01)
    o = run(rois, gt, [[1, 2, 3]], total_pos=8, total_neg=8, variances=(0.1, 0.1, 0.2, 0.2))
    nfg = o["counts"][0, 0]
    assert nfg >= 3
    src, j = o["src"][0, :nfg], o["argmax"][0, o["src"][0, :nfg]]
    rows = np.concatenate([rois[0], gt[0]])
    want = O.get_deltas_from_bboxes(rows[src], gt[0, j]) / np.asarray([0.1, 0.1, 0.2, 0.2], F32)
    assert np.array_equal(o["deltas"][0, :nfg], want) and (o["deltas"][0, nfg:] == 0).all()


# ---- sampler ---------------------------------------------------------------------------------------------------------
def test_sampler_invariants():
    rng = np.random.default_rng(3)
    B, P, G = 6, 400, 12
    rois = random_boxes(rng, (B, P))
    gt = rois[:, rng.integers(0, P, size=G)] + rng.normal(0, 0.02, size=(B, G, 4)).astype(F32)
    lab = rng.integers(-1, 6, size=(B, G))
    valid = rng.integers(-5, P + 5, size=B)
    for tp, tn in ((16, 48), (64, 64), (1, 3)):
        o = run(rois, gt, lab, valid, num_classes=5, total_pos=tp, total_neg=tn, seed=9, offset=2 ** 40 + 3)
        for b in range(B):
            nf, nb = o["fg_cand"][b].sum(), o["bg_cand"][b].sum()
            assert o["fg_keep"][b].sum() == min(nf, tp)
            assert o["bg_keep"][b].sum() == min(nb, tp + tn - min(nf, tp))
            assert not (o["fg_keep"][b] & ~o["fg_cand"][b]).any() and not (o["bg_keep"][b] & ~o["bg_cand"][b]).any()
    a = run(rois, gt, lab, valid, total_pos=8, total_neg=24, seed=1, offset=0)
    b = run(rois, gt, lab, valid, total_pos=8, total_neg=24, seed=1, offset=1)
    assert not np.array_equal(a["src"], b["src"])            # another offset, another sample


def test_words_2_and_3_differ_from_words_0_and_1():
    w = [O.sampling_keys(4096, 7, 123, 45, s) for s in range(4)]
    for i in range(4):
        for k in range(i + 1, 4):
            assert (w[i] != w[k]).mean() > 0.99


def test_shards_with_image_offset_equal_one_call():
    rng = np.random.default_rng(4)
    rois = random_boxes(rng, (5, 200))
    gt = rois[:, :6] + F32(0.01)
    lab = np.ones((5, 6), np.int32)
    kw = dict(total_pos=8, total_neg=24, seed=3, offset=11)
    whole = run(rois, gt, lab, **kw)
    for s in (slice(0, 2), slice(2, 5)):
        part = run(rois[s], gt[s], lab[s], image_offset=s.start, **kw)
        assert np.array_equal(part["src"], whole["src"][s])


# ---- an independent implementation of the matching --------------------------------------------------------------------
def test_matching_equals_torchvision_matcher():
    torch = pytest.importorskip("torch")
    pytest.importorskip("torchvision")
    from torchvision.models.detection._utils import Matcher
    from torchvision.ops import box_iou
    rng = np.random.default_rng(5)
    B, P, G = 4, 500, 20
    rois = random_boxes(rng, (B, P))
    gt = random_boxes(rng, (B, G), 0.1, 0.4)
    src = rng.integers(0, P, size=(B, G))
    rois[np.arange(B)[:, None], src] = np.clip(gt + rng.normal(0, 0.02, size=gt.shape), 0, 1).astype(F32)
    lab = rng.integers(1, 21, size=(B, G))
    o = run(rois, gt, lab, num_classes=21, total_pos=128, total_neg=384)
    matcher = Matcher(0.5, 0.5, allow_low_quality_matches=False)
    n_fg = 0
    for b in range(B):
        rows = np.concatenate([rois[b], gt[b]])
        xyxy = lambda a: torch.from_numpy(np.ascontiguousarray(a[:, [1, 0, 3, 2]]))  # noqa: E731
        q = box_iou(xyxy(gt[b]), xyxy(rows))                 # (G, P')
        top = q.topk(2, dim=0).values
        assert bool(((top[0] > top[1]) | (top[0] < 0.5)).all()), "inputs must be tie-free"
        m = matcher(q).numpy()
        assert np.array_equal(o["fg_cand"][b], m >= 0)
        assert np.array_equal(o["bg_cand"][b], m == Matcher.BELOW_LOW_THRESHOLD)
        assert np.array_equal(o["argmax"][b][m >= 0], m[m >= 0])
        assert np.array_equal(o["max_iou"][b], q.max(dim=0).values.numpy())
        n_fg += int((m >= 0).sum())
    assert n_fg > B * G


# ---- ABI ---------------------------------------------------------------------------------------------------------------
def test_ctypes_roi_target_cfg_matches_header_layout(tmp_path):
    from tfrpn import _lib
    cls = _lib.RoiTargetCfg
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tfrpn.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(tfrpn_roi_target_cfg));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(tfrpn_roi_target_cfg, %s));' % (fname, fname))
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

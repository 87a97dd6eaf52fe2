"""oracle/map_oracle.py on hand-derived cases: every matching rule of the three protocols, the crowd IoU, max_dets,
the score order (NaN, +-0, ties across images and updates), classes without GT or without detections, and the
ordered sums against the literal restatements of pycocotools' ``accumulate`` and the devkit's ``voc_ap``.  Also the
ctypes layout of tfrpn_map_cfg / tfrpn_map_state."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import map_oracle as M

F32 = np.float32
UNIT = [0.0, 0.0, 1.0, 1.0]


def one(det, scores, gt, labels=None, flags=None, classes=None, valid=None, **kw):
    """One image -> MapAccumulator after one update."""
    det = np.asarray(det, F32).reshape(1, -1, 4)
    R = det.shape[1]
    gt = np.asarray(gt, F32).reshape(1, -1, 4)
    G = gt.shape[1]
    acc = M.MapAccumulator(kw.pop("num_classes", 1), **kw)
    acc.update(det, np.asarray(scores, F32).reshape(1, R),
               np.zeros((1, R), F32) if classes is None else np.asarray(classes, F32).reshape(1, R),
               valid, gt, np.zeros((1, G), np.int32) if labels is None else np.asarray(labels, np.int32).reshape(1, G),
               None if flags is None else np.asarray(flags, np.uint8).reshape(1, G))
    return acc


def tp_ig(acc, c=0, t=0):
    tp, ig = acc.entries(c)
    return tp[:, t].astype(int).tolist(), ig[:, t].astype(int).tolist()


def test_iou_exactly_at_threshold():
    # the detection covers half of the unit GT: IoU = 0.5 exactly (dyadic)
    kw = dict(det=[[0, 0, 0.5, 1]], scores=[0.9], gt=[UNIT], thresholds=[0.5])
    assert tp_ig(one(protocol="coco", **kw)) == ([1], [0])
    assert tp_ig(one(protocol="voc", **kw)) == ([0], [0])
    assert tp_ig(one(protocol="voc07", **kw)) == ([0], [0])


@pytest.mark.parametrize("protocol", M.PROTOCOLS)
def test_second_detection_on_a_matched_gt(protocol):
    acc = one([UNIT, UNIT], [0.9, 0.8], [UNIT], protocol=protocol, thresholds=[0.5])
    assert tp_ig(acc) == ([1, 0], [0, 0])


def test_best_gt_difficult_other_gt_overlaps():
    # GT 0 equals the detection (difficult); GT 1 overlaps it at 0.75 (non-difficult)
    kw = dict(det=[UNIT], scores=[0.9], gt=[UNIT, [0, 0, 0.75, 1]], flags=[1, 0], thresholds=[0.5])
    assert tp_ig(one(protocol="voc", **kw)) == ([0], [1])
    assert tp_ig(one(protocol="voc07", **kw)) == ([0], [1])
    assert tp_ig(one(protocol="coco", **kw)) == ([1], [0])


def test_best_gt_already_matched_other_gt_overlaps():
    # det 0 takes GT 0; det 1 has IoU 0.75 with GT 0 and 0.5625 with GT 1
    det = [UNIT, [0, 0, 0.75, 1]]
    gt = [UNIT, [0, 0, 0.75, 0.75]]
    kw = dict(det=det, scores=[0.9, 0.8], gt=gt, thresholds=[0.5])
    assert tp_ig(one(protocol="voc", **kw)) == ([1, 0], [0, 0])    # the devkit does not fall back
    assert tp_ig(one(protocol="coco", **kw)) == ([1, 1], [0, 0])


def test_iou_ties_between_gt():
    # the detection [0,0.25,1,0.75] overlaps GT 0 = [0,0,1,0.5] and GT 1 = [0,0.5,1,1] at 1/3 each
    det = [[0, 0.25, 1, 0.75]]
    gt = [[0, 0, 1, 0.5], [0, 0.5, 1, 1]]
    iou = M.pair_ious(np.asarray(det, F32), np.asarray(gt, F32), np.zeros(2, bool), "voc")
    assert iou[0, 0] == iou[0, 1]
    # voc: GT 0 (lowest index) is taken first; for the second detection the best is still GT 0: FP
    assert tp_ig(one(det * 2, [0.9, 0.8], gt, protocol="voc", thresholds=[0.25]))[0] == [1, 0]
    # coco: GT 1 (highest index) first, then GT 0; with GT 1 difficult, only the second detection is TP
    assert tp_ig(one(det * 2, [0.9, 0.8], gt, protocol="coco", thresholds=[0.25])) == ([1, 1], [0, 0])
    assert tp_ig(one(det * 2, [0.9, 0.8], gt, flags=[0, 1], protocol="coco", thresholds=[0.25])) == ([1, 0], [0, 1])
    assert tp_ig(one(det * 2, [0.9, 0.8], gt, flags=[1, 0], protocol="voc", thresholds=[0.25])) == ([0, 0], [1, 1])


def test_crowd_absorbs_detections():
    det = [[0, 0, 0.25, 0.25], [0.5, 0.5, 1, 1], [0.25, 0.25, 0.5, 0.5]]
    kw = dict(det=det, scores=[0.9, 0.8, 0.7], gt=[UNIT], flags=[2], thresholds=[0.5])
    iou = M.pair_ious(np.asarray(det, F32), np.asarray([UNIT], F32), np.ones(1, bool), "coco")
    assert iou[:, 0].tolist() == [1.0, 1.0, 1.0]   # inter / area(det)
    acc = one(protocol="coco", **kw)
    assert tp_ig(acc) == ([0, 0, 0], [1, 1, 1]) and acc.n_gt[0] == 0
    acc = one(protocol="voc", **kw)                 # a difficult GT there: plain IoU 1/16, 1/4, 1/16
    assert tp_ig(acc) == ([0, 0, 0], [0, 0, 0])
    # a detection with no area scores +0 against a crowd
    z = M.pair_ious(np.asarray([[0.5, 0.5, 0.5, 0.9]], F32), np.asarray([UNIT], F32), np.ones(1, bool), "coco")
    assert z[0, 0] == 0 and not np.signbit(z[0, 0])


def test_ignored_gt_matched_once_unless_crowd():
    # two detections on one ignored (non-crowd) GT: the first is ignored, the second FP
    acc = one([UNIT, UNIT], [0.9, 0.8], [UNIT], flags=[1], protocol="coco", thresholds=[0.5])
    assert tp_ig(acc) == ([0, 0], [1, 0])


def test_max_dets_truncation():
    gt = [[0, 0, 0.25, 0.25], [0.5, 0.5, 0.75, 0.75], [0.25, 0.25, 0.5, 0.5]]
    acc = one(gt, [0.9, 0.8, 0.7], gt, protocol="coco", thresholds=[0.5], max_dets=2)
    assert tp_ig(acc) == ([1, 1], [0, 0])
    ap, rec, n_gt = acc.compute()
    assert n_gt[0] == 3 and rec[0, 0] == 2 / 3
    acc = one(gt, [0.9, 0.8, 0.7], gt, protocol="coco", thresholds=[0.5], max_dets=0)
    assert tp_ig(acc) == ([1, 1, 1], [0, 0, 0])
    acc = one(gt, [0.9, 0.8, 0.7], gt, protocol="voc", thresholds=[0.5], max_dets=2)   # voc ignores max_dets
    assert tp_ig(acc) == ([1, 1, 1], [0, 0, 0])


def test_classes_without_gt_or_without_detections():
    # class 0: detections, no GT; class 1: GT, no detections; class 2: one TP
    det = [UNIT, [0, 0, 0.5, 0.5]]
    gt = [[0.5, 0.5, 1, 1], [0, 0, 0.5, 0.5]]
    acc = one(det, [0.9, 0.8], gt, labels=[1, 2], classes=[0, 2], num_classes=3, protocol="voc")
    ap, rec, n_gt = acc.compute()
    assert n_gt.tolist() == [0, 1, 1]
    assert math.isnan(ap[0, 0]) and math.isnan(rec[0, 0])
    assert ap[1, 0] == 0.0 and rec[1, 0] == 0.0
    assert ap[2, 0] == 1.0 and rec[2, 0] == 1.0
    assert M.class_mean(ap, n_gt).tolist() == [0.5]


def test_participation_rules():
    # rows past valid, non-integer / out-of-range / NaN classes take no part; labels outside [0, C) neither
    det = [UNIT] * 5
    acc = one(det, [0.9] * 5, [UNIT, UNIT], labels=[0, 7], classes=[0.5, 3, np.nan, -1, 0], num_classes=2,
              protocol="voc", valid=np.asarray([5], np.int32))
    assert tp_ig(acc) == ([1], [0]) and acc.n_gt.tolist() == [1, 0]
    acc = one(det, [0.9] * 5, [UNIT], classes=[0] * 5, protocol="voc", valid=np.asarray([-3], np.int32))
    assert acc.entries(0)[0].shape[0] == 0
    acc = one(det, [0.9] * 5, [UNIT], classes=[0] * 5, protocol="voc", valid=np.asarray([99], np.int32))
    assert acc.entries(0)[0].shape[0] == 5


def test_nan_and_signed_zero_scores():
    far = [0.5, 0.5, 0.75, 0.75]
    # NaN ranks above 0.9: the FP with a NaN score comes first
    acc = one([UNIT, far], [0.9, np.nan], [UNIT], protocol="voc")
    assert tp_ig(acc)[0] == [0, 1]
    assert acc.compute()[0][0, 0] == 0.5
    # -0 and +0 tie: row order decides
    acc = one([UNIT, far], [-0.0, 0.0], [UNIT], protocol="voc")
    assert tp_ig(acc)[0] == [1, 0] and acc.compute()[0][0, 0] == 1.0
    acc = one([far, UNIT], [-0.0, 0.0], [UNIT], protocol="voc")
    assert tp_ig(acc)[0] == [0, 1] and acc.compute()[0][0, 0] == 0.5
    assert M.score_key(np.asarray([np.nan, -np.nan, np.inf, 1.0, 0.0, -0.0, -np.inf], F32)).tolist() == \
        sorted(M.score_key(np.asarray([np.nan, -np.nan, np.inf, 1.0, 0.0, -0.0, -np.inf], F32)).tolist())


def test_score_ties_across_images_and_updates():
    far = [0.5, 0.5, 0.75, 0.75]
    boxes = np.asarray([[far], [UNIT]], F32)           # image 0: FP, image 1: TP, equal scores
    gt = np.asarray([[far[:2] + [0.5, 0.5]], [UNIT]], F32)
    gt[0, 0] = [0.0, 0.0, 0.0, 0.0]
    args = (np.full((2, 1), 0.5, F32), np.zeros((2, 1), F32), None)
    labels = np.asarray([[-1], [0]], np.int32)
    acc = M.MapAccumulator(1, "voc")
    acc.update(boxes, *args, gt, labels)
    assert tp_ig(acc)[0] == [0, 1] and acc.compute()[0][0, 0] == 0.5
    acc = M.MapAccumulator(1, "voc")
    acc.update(boxes[::-1].copy(), *args, gt[::-1].copy(), labels[::-1].copy())
    assert tp_ig(acc)[0] == [1, 0] and acc.compute()[0][0, 0] == 1.0
    acc = M.MapAccumulator(1, "voc")   # across updates: the earlier update first
    acc.update(boxes[:1], args[0][:1], args[1][:1], None, gt[:1], labels[:1])
    acc.update(boxes[1:], args[0][1:], args[1][1:], None, gt[1:], labels[1:])
    assert tp_ig(acc)[0] == [0, 1]


def test_known_ap_values():
    tp = np.asarray([1, 0, 1, 1, 0, 0, 1], bool)
    # VOC all-point with n_gt = 5: rc 0.2 .. 0.8, envelope 1, 2/3, 2/3, 3/4 (pr at the TP entries: 1, 2/3, 3/4, 4/7)
    ap, rec = M.average_precision(tp, 5, "voc")
    assert rec == 0.8
    assert abs(ap - (0.2 * 1 + 0.2 * 0.75 + 0.2 * 0.75 + 0.2 * 4 / 7)) < 1e-15
    ap07, _ = M.average_precision(tp, 5, "voc07")
    # points 0, .1, .2 -> 1; .3, .4, .5 -> 3/4; .6, .7, .8 -> 4/7 (6 * 0.1 = 0.6000000000000001 > 3/5); .9, 1 -> 0
    assert 6 * 0.1 > 3 / 5
    assert abs(ap07 - (3 * 1 + 3 * 0.75 + 3 * 4 / 7) / 11) < 1e-15
    assert ap07 == M.devkit_ap(tp, 5, use_07_metric=True)


@pytest.mark.parametrize("seed", range(6))
def test_ordered_sums_match_pycocotools_and_devkit(seed):
    rng = np.random.default_rng(seed)
    for n, p, n_gt in ((1, 1.0, 1), (50, 0.3, 40), (997, 0.5, 600), (3000, 0.1, 2000)):
        tp = rng.uniform(size=n) < p
        tp_count = int(tp.sum())
        n_gt = max(n_gt, tp_count, 1)
        for protocol, ref in (("coco", lambda: M.pycocotools_ap(tp, n_gt)), ("voc", lambda: M.devkit_ap(tp, n_gt)),
                              ("voc07", lambda: M.devkit_ap(tp, n_gt, use_07_metric=True))):
            ap, rec = M.average_precision(tp, n_gt, protocol)
            r = ref()
            assert abs(ap - r) <= 1e-12 * max(abs(r), 1e-300) or ap == r, (protocol, n, ap, r)
            assert rec == (tp_count / n_gt if n else 0.0)


def test_recall_points_equal_numpy_grids():
    assert np.array_equal(np.arange(101, dtype=np.float64) * 0.01, np.linspace(0, 1, 101))
    assert np.array_equal(np.arange(11, dtype=np.float64) * 0.1, np.arange(0, 1.1, 0.1))


def test_ctypes_layout():
    from tfrpn import _lib
    assert C.sizeof(_lib.MapCfg) == 4 * 3 + 64 + 8
    assert _lib.MapCfg.max_dets.offset == 76
    assert C.sizeof(_lib.MapState) == 40 and _lib.MapState.overflow.offset == 32
    assert _lib.KERNEL_IDS == 13
    for name in ("tfrpn_map_update", "tfrpn_map_compute", "tfrpn_map_workspace_bytes"):
        assert name in _lib.PROTOTYPES

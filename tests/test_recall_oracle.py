"""Known answers of the proposal-recall oracle (oracle/recall_oracle.py), worked out by hand, its greedy matching
against a plain restatement of Detectron's loop, and the ctypes mirror of tfrpn_recall_cfg.  CPU only."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import recall_oracle as R

F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(prop, gt, labels=None, valid=None, limits=(100,), thresholds=(0.5,), matching="greedy"):
    prop = np.asarray(prop, F32).reshape(1, -1, 4) if np.ndim(prop) < 3 else np.asarray(prop, F32)
    gt = np.asarray(gt, F32).reshape(1, -1, 4) if np.ndim(gt) < 3 else np.asarray(gt, F32)
    return R.proposal_recall(prop, gt, labels, valid, np.asarray(thresholds, F32), limits, matching)


def detectron_loop(S):
    """evaluate_box_proposals' loop as written there (overlaps = proposals x GT)."""
    S = np.array(S, F32, copy=True)
    out = np.zeros(S.shape[1], F32)
    for _ in range(min(S.shape)):
        argmax_overlaps = S.argmax(axis=0)
        max_overlaps = S.max(axis=0)
        gt_ind = max_overlaps.argmax()
        if not max_overlaps[gt_ind] > 0:
            break
        box_ind = argmax_overlaps[gt_ind]
        out[gt_ind] = S[box_ind, gt_ind]
        S[box_ind, :] = -1
        S[:, gt_ind] = -1
    return out


def test_iou_equal_to_threshold_is_a_hit():
    rec, ar, counts, iou = run([[0, 0, 1, 1]], [[0, 0, 1, 0.5]])
    assert iou[0, 0, 0] == F32(0.5)
    assert counts.tolist() == [1, 1] and rec[0, 0] == 1.0 and ar[0] == 1.0
    _, _, counts, _ = run([[0, 0, 1, 1]], [[0, 0, 1, 0.5]], thresholds=(np.nextafter(F32(0.5), F32(1)),))
    assert counts.tolist() == [0, 1]


def test_shared_best_proposal_greedy_vs_coverage():
    # GT 0 = [0,0,1,1] and GT 1 = [0,0,1,0.75] both prefer proposal 0 = [0,0,1,1] (IoU 1 and 0.75); proposal 1 =
    # [0,0,1,0.5] covers them at 0.5 and 0.5/0.75.  Greedy: GT 0 takes proposal 0, GT 1 falls back to proposal 1.
    prop = [[0, 0, 1, 1], [0, 0, 1, 0.5]]
    gt = [[0, 0, 1, 1], [0, 0, 1, 0.75]]
    _, _, _, g = run(prop, gt)
    _, _, _, c = run(prop, gt, matching="coverage")
    assert g[0, 0].tolist() == [1.0, float(F32(0.5) / F32(0.75))]
    assert c[0, 0].tolist() == [1.0, 0.75]


def test_identical_gt_lower_index_wins():
    prop = [[0, 0, 1, 1], [0, 0, 0.5, 1]]
    gt = [[0, 0, 1, 1], [0, 0, 1, 1]]
    _, _, _, g = run(prop, gt)
    assert g[0, 0].tolist() == [1.0, 0.5]


def test_identical_proposals_lower_rank_taken():
    prop = [[0, 0, 1, 1], [0, 0, 1, 1], [0, 0, 0.5, 1]]
    gt = [[0, 0, 1, 1], [0, 0, 1, 1]]
    _, _, _, g = run(prop, gt)
    assert g[0, 0].tolist() == [1.0, 1.0]
    S = R.pair_scores(np.asarray(prop, F32), np.asarray(gt, F32))
    assert detectron_loop(S).tolist() == [1.0, 1.0]
    # with one copy the second GT gets the half box, and with the limit 1 nothing
    _, _, _, g = run(prop, gt, limits=(1, 2))
    assert g[:, 0].tolist() == [[1.0, 0.0], [1.0, 1.0]]


def test_fewer_proposals_than_gt():
    gt = [[0, 0, 0.5, 0.5], [0.5, 0.5, 1, 1], [0, 0.5, 0.5, 1]]
    rec, _, counts, g = run([[0.5, 0.5, 1, 1]], gt, thresholds=(0.5, 1.0))
    assert g[0, 0].tolist() == [0.0, 1.0, 0.0]
    assert counts.tolist() == [1, 1, 3] and np.allclose(rec, [[1 / 3, 1 / 3]])


def test_valid_zero_and_limit_larger_than_p():
    prop = [[[0, 0, 1, 1]], [[0, 0, 1, 1]]]
    gt = [[[0, 0, 1, 1]], [[0, 0, 1, 1]]]
    _, _, counts, g = run(prop, gt, valid=[0, 5], limits=(1, 1000))
    assert g[:, :, 0].tolist() == [[0.0, 1.0], [0.0, 1.0]]
    assert counts.tolist() == [1, 1, 2]


def test_all_padding_image_adds_no_gt():
    prop = [[[0, 0, 1, 1]], [[0, 0, 1, 1]]]
    gt = [[[0, 0, 1, 1], [0, 0, 0, 0]], [[0, 0, 0, 0], [0, 0, 0, 0]]]
    labels = [[3, -1], [-1, -1]]
    _, _, counts, g = run(prop, gt, labels=labels)
    assert counts.tolist() == [1, 1]
    assert g[0].tolist() == [[1.0, -1.0], [-1.0, -1.0]]
    # a label < 0 excludes a real box too; without any valid GT the recall is NaN
    rec, ar, counts, _ = run(prop[:1], [[[0, 0, 1, 1]]], labels=[[-1]])
    assert counts.tolist() == [0, 0] and np.isnan(rec).all() and np.isnan(ar).all()


def test_nan_and_inverted_boxes_score_zero():
    nan = float("nan")
    prop = [[nan, 0, 1, 1], [1, 1, 0, 0], [0, 0, 1, 0.25]]
    gt = [[0, 0, 1, 1]]
    S = R.pair_scores(np.asarray(prop, F32), np.asarray(gt, F32))
    assert S[:, 0].tolist() == [0.0, 0.0, 0.25]
    _, _, _, g = run(prop, gt, thresholds=(0.25,))
    assert g[0, 0].tolist() == [0.25]
    # an inverted GT box has positive area, so it is valid; it scores 0 against everything here
    _, _, counts, g = run([[0, 0, 1, 1]], [[1, 1, 0, 0]], thresholds=(0.01,))
    assert counts.tolist() == [0, 1] and g[0, 0].tolist() == [0.0]


def test_coverage_recall_at_least_greedy():
    rng = np.random.default_rng(4)
    for _ in range(5):
        B, P, G = 3, 60, 12
        c = rng.uniform(0.2, 0.8, size=(B, G, 2))
        s = rng.uniform(0.1, 0.3, size=(B, G, 2))
        gt = np.concatenate([c - s / 2, c + s / 2], axis=-1).astype(F32)
        j = gt[np.arange(B)[:, None], rng.integers(0, G, size=(B, P))]   # jittered copies of the GT
        prop = (j + rng.normal(0, 0.04, size=j.shape)).astype(F32)
        thr = np.asarray([x / 100 for x in range(50, 100, 5)], F32)
        rg, _, _, _ = R.proposal_recall(prop, gt, thresholds=thr, limits=(5, 20, 60))
        rc, _, _, _ = R.proposal_recall(prop, gt, thresholds=thr, limits=(5, 20, 60), matching="coverage")
        assert np.all(rc >= rg)


@pytest.mark.parametrize("seed", range(6))
def test_greedy_equals_detectron_loop(seed):
    """Tie-heavy score matrices (few distinct values, zeros, more rows or more columns)."""
    rng = np.random.default_rng(seed)
    for _ in range(40):
        k, G = int(rng.integers(0, 12)), int(rng.integers(1, 12))
        S = (rng.integers(0, 4, size=(k, G)) / F32(4)).astype(F32)
        assert np.array_equal(R.match_greedy(S), detectron_loop(S))


def test_default_thresholds():
    assert R.DEFAULT_THRESHOLDS.dtype == F32 and R.DEFAULT_THRESHOLDS.size == 10
    assert R.DEFAULT_THRESHOLDS[1] == F32(0.55) and R.DEFAULT_THRESHOLDS[-1] == F32(0.95)
    from tfrpn import evaluation
    assert np.array_equal(np.asarray(evaluation.DEFAULT_THRESHOLDS, F32), R.DEFAULT_THRESHOLDS)


def test_recall_cfg_rejects_bad_arguments():
    from tfrpn import evaluation
    with pytest.raises(ValueError):
        evaluation.recall_cfg(iou_thresholds=[0.5] * 17)
    with pytest.raises(ValueError):
        evaluation.recall_cfg(limits=[])
    with pytest.raises(ValueError):
        evaluation.recall_cfg(matching="hungarian")
    cfg = evaluation.recall_cfg([0.5, 0.75], (1, 10), "coverage")
    assert (cfg.n_thresholds, cfg.n_limits, cfg.matching) == (2, 2, 1)
    assert list(cfg.limits[:2]) == [1, 10] and cfg.thresholds[1] == 0.75


def test_recall_cfg_layout_matches_header(tmp_path):
    from tfrpn import _lib
    cls = _lib.RecallCfg
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "tfrpn.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(tfrpn_recall_cfg));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(tfrpn_recall_cfg, %s));' % (fname, fname))
    lines += ['return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    got = {l.split()[0]: int(l.split()[1]) for l in out.splitlines()}
    assert got["size"] == C.sizeof(cls) == 112
    for fname, _ in cls._fields_:
        assert got[fname] == getattr(cls, fname).offset, fname

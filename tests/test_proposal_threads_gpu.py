"""The two builds of the one-CTA proposal_kernel, 512 and 1024 threads per CTA (TFRPN_PROP_THREADS), on the layouts
that exercise the parts whose mapping to threads differs between them: the histogram scans (4 or 2 bins per thread),
the candidate list and the batch (4 or 2 list entries, 2 or 1 ranks per thread), the counting sort and its bitonic
fall-back for long bins, the kept-list test (4 or 8 parts per candidate) and the folded triangle (32 or 64 teams).
Each case runs on both builds; every output must match the oracle as in test_proposal_front_end_gpu.py, and the two
builds must agree bit for bit.  TFRPN_PROP_CLUSTER=0 keeps every batch size on the one-CTA kernel."""
import numpy as np
import pytest

import test_nms_multiclass_gpu as MC
import test_proposal_front_end_gpu as FE

pytestmark = pytest.mark.gpu
F32 = np.float32
NINF = float("-inf")
BUILDS = {"t512": {"TFRPN_PROP_CLUSTER": 0, "TFRPN_PROP_THREADS": 512},
          "t1024": {"TFRPN_PROP_CLUSTER": 0, "TFRPN_PROP_THREADS": 1024}}
FE.CONFIGS.update(BUILDS)   # FE.open_handle reads the environment of a configuration from there


@pytest.fixture(scope="module")
def builds(cuda_device):
    hs = {}
    try:
        for name in BUILDS:
            hs[name] = FE.open_handle(cuda_device, name)
        yield hs
    finally:
        for ns in hs.values():
            ns.lib.load().tfrpn_destroy(ns.h)


def same(a, b):
    return all(FE.bits_equal(x, y) if x.dtype == F32 else np.array_equal(x, y) for x, y in zip(a, b))


def on_both(builds, run):
    """run(ns) on both builds -> the outputs of the 512-thread build, after checking that the other one agrees"""
    got = {name: run(ns) for name, ns in builds.items()}
    assert same(got["t512"], got["t1024"])
    return got["t512"]


SHAPES_NK = [(1025, 1025), (8649, 127), (8649, 1025), (8649, 6000), (37800, 6000)]
LAYOUTS = ["equal", "three", "one_bin_ulps", "one_bin", "sigmoid"]


@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES_NK)
def test_topk(builds, name, N, k):
    """tie groups across the batch floor, rank 1024 and rank k ("three"), one 11-bit bin, one tie group ("equal":
    the bitonic fall-back)"""
    scores, boxes, wv, wi = FE.topk_case(name, N, k)
    v, i, g = on_both(builds, lambda ns: FE.run_topk(ns, scores, k, boxes))
    assert np.array_equal(i, wi) and FE.bits_equal(v, wv)
    assert FE.bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(FE.B)]))


@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES_NK)
def test_nms(builds, name, N, k):
    """near-duplicate boxes: NMS runs through several batches"""
    scores, boxes, want = FE.nms_case(name, N, k)
    FE.assert_nms_equal(on_both(builds, lambda ns: FE.run_nms(ns, boxes, scores, k, NINF)), want)


@pytest.mark.parametrize("name", ["three", "one_bin", "sigmoid"])
@pytest.mark.parametrize("k", [127, 6000])
def test_proposals(builds, name, k):
    """the fused decode + NMS mode at the C2 shape"""
    hp, anchors, reg, cls, (wb, ws, wv, wk) = FE.c2_case(name, k)
    ob, os_, ov, ok = on_both(builds, lambda ns: FE.run_proposals(ns, reg, cls, anchors, hp, k))
    assert np.array_equal(ov, wv) and np.array_equal(ok, wk)
    assert FE.bits_equal(os_, ws) and FE.within_ulps(ob, wb, 4)


@pytest.mark.parametrize("M", [0, 1, 1030])
@pytest.mark.parametrize("N,k", [(1025, 0), (8649, 6000), (37800, 0)])
def test_score_threshold_leaves(builds, M, N, k):
    """a score threshold leaving 0, 1 or 1030 entries above it"""
    scores, boxes, want = FE.threshold_case(M, N, k)
    FE.assert_nms_equal(on_both(builds, lambda ns: FE.run_nms(ns, boxes, scores, k, 0.05)), want)


def test_unstaged_keys(builds):
    """N above the shared-memory staging limit: every select sweep re-reads the scores (top-k, then NMS that walks
    every rank)"""
    N = FE.first_unstaged_n("one_cta", 0) + 37
    k = N // 4 + 1                                # k > N / 4: the prefilter does not apply
    rng = np.random.default_rng(N)
    scores = FE.layout("three", rng, N, Bn=2)
    boxes = rng.uniform(0, 1, size=(2, N, 4)).astype(F32)
    v, i, g = on_both(builds, lambda ns: FE.run_topk(ns, scores, k, boxes))
    wv, wi = FE.composite_topk(scores, k)
    assert np.array_equal(i, wi) and FE.bits_equal(v, wv)
    N = FE.first_unstaged_n("one_cta", 500) + 37
    scores = FE.layout("sigmoid", rng, N, Bn=2)
    boxes = FE.near_dup_boxes(rng, N, Bn=2)
    got = on_both(builds, lambda ns: FE.run_nms(ns, boxes, scores, 0, NINF, rows=500))
    FE.assert_nms_equal(got, FE.oracle_nms(boxes, scores, 0, NINF, rows=500))


def test_prefilter_flagged_redo(builds):
    """NMS over all 90 000 boxes: the prefilter keeps the top ~6144 ranks for the compact launch; images 0 and 2
    (boxes that all overlap each other) run out of candidates before 300 are kept, raise their flags and are redone
    over every box by the unfiltered launch; image 1 (disjoint boxes) finishes inside its candidates"""
    N = 90000
    rng = np.random.default_rng(N)
    scores = FE.layout("sigmoid", rng, N, Bn=3)
    c = rng.uniform(0.49, 0.51, size=(3, N, 2))
    sz = rng.uniform(0.3, 0.31, size=(3, N, 2))
    boxes = np.concatenate([c - sz / 2, c + sz / 2], -1).astype(F32)
    g = np.arange(N)
    y, x = (g // 300) / F32(300), (g % 300) / F32(300)
    boxes[1] = np.stack([y, x, y + F32(0.002), x + F32(0.002)], -1).astype(F32)
    got = on_both(builds, lambda ns: FE.run_nms(ns, boxes, scores, 0, NINF))
    FE.assert_nms_equal(got, FE.oracle_nms(boxes, scores, 0, NINF))
    assert got[2][0] < 300 and got[2][1] == 300 and got[2][2] < 300


def test_nms_multiclass(builds):
    """tfrpn_nms_multiclass: per-(image, class) launches of proposal_kernel on the staged segments"""
    import torch
    from tfrpn import _lib

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.lib, ns.L, ns.dev = torch, _lib.load(), _lib, builds["t512"].dev
    ns.cu = builds["t512"].cu
    rng = np.random.default_rng(8732)
    boxes, scores = MC.layout(rng, 2, 8732, 21, 1)
    cfg = MC.cfg_of(ns, 100, 200, 0.45, 0.05, False, True, 0)
    got = on_both(builds, lambda b: MC.native(ns, boxes, scores, cfg, h=b.h))
    MC.assert_same(got, MC.oracle(boxes, scores, cfg))

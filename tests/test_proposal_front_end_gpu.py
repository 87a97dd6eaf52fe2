"""Adversarial score layouts for the front end of the one-CTA proposal kernel (threshold batches, 11-bit histogram
select, counting sort with a bitonic fall-back), forced with TFRPN_PROP_CLUSTER=0, in TOPK, NMS and fused-proposal
modes, against the C restatement of the reference.  Keep lists, valid counts, indices and scores bit-exact; decoded
boxes within the 4-ulp bar of the other parity tests.

The kernels order scores by their orderable bit pattern, so +0.0 ranks above -0.0; the C oracle compares float values,
so there the two tie and the lower index goes first.  Top-k is therefore checked against a NumPy restatement of the
kernels' order (equal to the C oracle whenever the zeros do not mix).  tfrpn_nms reads a -inf score threshold as no
threshold, while the C oracle keeps only scores > -inf.  The NMS layouts therefore use one sign of zero and no -inf."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32
EPS = float(np.finfo(F32).eps)


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(np.all(a.view(np.uint32) == b.view(np.uint32)))


def within_ulps(a, b, ulps=4, scale=1.0):
    a64, b64 = np.asarray(a, np.float64), np.asarray(b, np.float64)
    mag = np.maximum(np.abs(b64), scale)
    return a64.shape == b64.shape and bool(np.all(np.abs(a64 - b64) <= ulps * EPS * mag))


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    from tfrpn import _lib, synthetic
    if not CO.available():
        pytest.skip("oracle/_build/librpn_oracle.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    old = os.environ.get("TFRPN_PROP_CLUSTER")
    os.environ["TFRPN_PROP_CLUSTER"] = "0"   # read once, by tfrpn_create
    try:
        h = C.c_void_p()
        _lib.check(_lib.load().tfrpn_create(C.byref(h), cuda_device.index or 0))
    finally:
        if old is None:
            os.environ.pop("TFRPN_PROP_CLUSTER")
        else:
            os.environ["TFRPN_PROP_CLUSTER"] = old

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.lib, ns.syn, ns.dev, ns.h = torch, _lib, synthetic, cuda_device, h
    ns.cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.np = lambda t: t.detach().cpu().numpy()
    ns.st = lambda: torch.cuda.current_stream(cuda_device).cuda_stream
    yield ns
    _lib.load().tfrpn_destroy(h)


B = 9   # > 8 images: the one-CTA kernel is also what the launcher picks


def layout(name, rng, N, for_nms=False):
    """(B, N) float32 scores"""
    if name == "equal":                       # one tie group
        return np.full((B, N), 0.5, F32)
    if name == "three":                       # tie groups straddling the batch floor, rank 1024 and rank k
        s = np.full((B, N), 0.25, F32)
        s[:, : min(N, 700)] = 0.75
        s[:, 700: min(N, 1100)] = 0.5
        for b in range(B):
            s[b] = s[b][rng.permutation(N)]
        return s
    if name == "one_bin_ulps":                # every score inside one 11-bit bin, 16 distinct values
        return (1.0 - 2.0 ** -20 * rng.uniform(0, 1, size=(B, N))).astype(F32)
    if name == "one_bin":                     # every score inside [0.8, 0.85): the first histogram separates nothing
        return (0.8 + 0.05 * rng.uniform(0, 1, size=(B, N))).astype(F32)
    if name == "special":                     # negatives, +-0, +-inf, denormals among sigmoid-like scores
        s = (rng.normal(0, 3, size=(B, N))).astype(F32)
        pool = np.array([0.0, 0.0 if for_nms else -0.0, np.inf, -3e38 if for_nms else -np.inf, 1e-45, -1e-45, 1e-40, -3e-39,
                         1.0, -1.0], F32)
        m = rng.uniform(size=(B, N)) < 0.3
        s[m] = rng.choice(pool, size=int(m.sum()))
        return s
    if name == "sigmoid":
        return (1.0 / (1.0 + np.exp(-rng.normal(0, 2, size=(B, N))))).astype(F32)
    raise ValueError(name)


LAYOUTS = ["equal", "three", "one_bin_ulps", "one_bin", "special", "sigmoid"]
SHAPES = [(37, 1), (37, 127), (1023, 127), (1023, 1025), (1024, 1025), (1025, 1025), (1025, 6000),
          (8649, 127), (8649, 1025), (8649, 6000), (37800, 6000)]


def near_dup_boxes(rng, N):
    """(B, N, 4) boxes around a few centres with jitter: most candidates are suppressed, so NMS runs through
    several batches"""
    centres = rng.uniform(0.2, 0.8, size=(B, 40, 2))
    pick = rng.integers(0, 40, size=(B, N))
    c = np.take_along_axis(centres, pick[..., None].repeat(2, -1), axis=1) + rng.normal(0, 0.002, size=(B, N, 2))
    sz = rng.uniform(0.1, 0.12, size=(B, N, 2))
    return np.clip(np.concatenate([c - sz / 2, c + sz / 2], -1), 0, 1).astype(F32)


def composite_topk(scores, k):
    """higher orderable key first, then the lower index: the order of the proposal kernels"""
    u = np.ascontiguousarray(scores, F32).view(np.uint32)
    key = np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)
    idx = np.argsort(~key, axis=1, kind="stable")[:, :k].astype(np.int32)
    return np.take_along_axis(scores, idx, axis=1), idx


def run_topk(T, scores, k, boxes):
    torch, lib = T.torch, T.lib.load()
    Bn, N = scores.shape
    v = torch.empty((Bn, k), device=T.dev); i = torch.empty((Bn, k), dtype=torch.int32, device=T.dev)
    g = torch.empty((Bn, k, 4), device=T.dev)
    s_t, b_t = T.cu(scores), T.cu(boxes)
    T.lib.check(lib.tfrpn_topk(T.h, s_t.data_ptr(), Bn, N, k, v.data_ptr(), i.data_ptr(), b_t.data_ptr(), 1, g.data_ptr(), T.st()))
    torch.cuda.synchronize()
    return T.np(v), T.np(i), T.np(g)


def run_nms(T, boxes, scores, k, sthr, iou=0.7, rows=300):
    torch, lib = T.torch, T.lib.load()
    Bn, N = scores.shape
    nc = T.lib.NmsCfg(rows, rows, iou, sthr, 0, 1, k)
    nb = torch.empty((Bn, rows, 4), device=T.dev); ns = torch.empty((Bn, rows), device=T.dev)
    ncl = torch.empty((Bn, rows), device=T.dev)
    nv = torch.empty((Bn,), dtype=torch.int32, device=T.dev); nk = torch.empty((Bn, rows), dtype=torch.int32, device=T.dev)
    b_t, s_t = T.cu(boxes), T.cu(scores)
    T.lib.check(lib.tfrpn_nms(T.h, b_t.data_ptr(), s_t.data_ptr(), Bn, N, C.byref(nc), nb.data_ptr(), ns.data_ptr(),
                              ncl.data_ptr(), nv.data_ptr(), nk.data_ptr(), T.st()))
    torch.cuda.synchronize()
    return T.np(nb), T.np(ns), T.np(nv), T.np(nk)


def oracle_nms(boxes, scores, k, sthr, iou=0.7, rows=300):
    """NMS over the top-k entries (pre_nms_topn = k; 0 = all), keep indices in the caller's numbering"""
    Bn, N = scores.shape
    k = N if k == 0 else min(k, N)
    v, idx = CO.top_k(scores, k)
    sub = np.stack([boxes[b][idx[b]] for b in range(Bn)])
    wb, ws, _, wv, wk = CO.nms(sub, v, rows, rows, iou, sthr)
    wk = np.where(wk >= 0, np.take_along_axis(idx, np.maximum(wk, 0), axis=1), -1).astype(np.int32)
    return wb, ws, wv, wk


@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES)
def test_topk_layouts(T, name, N, k):
    if k > N:
        k = N
    rng = np.random.default_rng(N * 7 + k)
    scores = layout(name, rng, N)
    boxes = rng.uniform(0, 1, size=(B, N, 4)).astype(F32)
    v, i, g = run_topk(T, scores, k, boxes)
    wv, wi = composite_topk(scores, k)
    if name != "special":
        assert np.array_equal(wi, CO.top_k(scores, k)[1])
    assert np.array_equal(i, wi)
    assert bits_equal(v, wv)
    assert bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(B)]))


@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES)
def test_nms_layouts_near_duplicates(T, name, N, k):
    rng = np.random.default_rng(N * 11 + k)
    scores = layout(name, rng, N, for_nms=True)
    boxes = near_dup_boxes(rng, N)
    got = run_nms(T, boxes, scores, k, float("-inf"))
    want = oracle_nms(boxes, scores, k, float("-inf"))
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    assert bits_equal(got[1], want[1]) and bits_equal(got[0], want[0])


@pytest.mark.parametrize("M", [0, 100, 1030])
@pytest.mark.parametrize("N,k", [(1025, 0), (8649, 6000), (8649, 127), (37800, 0)])
def test_nms_score_threshold(T, M, N, k):
    """a score threshold leaving M entries: key 0 is never consumed"""
    rng = np.random.default_rng(M + N)
    scores = np.full((B, N), 0.01, F32)
    for b in range(B):
        m = min(M, N)
        scores[b, rng.permutation(N)[:m]] = rng.uniform(0.2, 0.9, size=m).astype(F32)
    scores[1, :5] = 0.05                       # exactly at the threshold: not above it
    boxes = T.syn.nms_boxes(rng, B, N)[0]
    got = run_nms(T, boxes, scores, k, 0.05)
    want = oracle_nms(boxes, scores, k, 0.05)
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    assert bits_equal(got[1], want[1]) and bits_equal(got[0], want[0])


@pytest.mark.parametrize("name", ["three", "one_bin", "sigmoid", "special"])
@pytest.mark.parametrize("k", [127, 1025, 6000])
def test_proposals_layouts(T, name, k):
    """the fused decode + NMS mode at the C2 shape"""
    hp = dict(O.get_hyper_params("vgg16"))
    anchors = O.generate_anchors(hp)
    N = anchors.shape[0]
    rng = np.random.default_rng(k)
    reg = rng.normal(0, 0.5, size=(B, N, 4)).astype(F32)
    cls = layout(name, rng, N, for_nms=True)
    from tfrpn.proposals import proposal_cfg
    torch, lib = T.torch, T.lib.load()
    pc = proposal_cfg(hp, pre_nms_topn=k)
    P = int(hp["test_nms_topn"])
    ob = torch.empty((B, P, 4), device=T.dev); os_ = torch.empty((B, P), device=T.dev)
    ov = torch.empty((B,), dtype=torch.int32, device=T.dev); ok = torch.empty((B, P), dtype=torch.int32, device=T.dev)
    r_t, c_t, a_t = T.cu(reg), T.cu(cls), T.cu(anchors)
    T.lib.check(lib.tfrpn_proposals(T.h, r_t.data_ptr(), c_t.data_ptr(), a_t.data_ptr(), B, N, C.byref(pc), ob.data_ptr(),
                                    os_.data_ptr(), ov.data_ptr(), ok.data_ptr(), T.st()))
    torch.cuda.synchronize()
    wb, ws, wv, wk = CO.proposals(reg, cls, anchors, hp, k)
    assert np.array_equal(T.np(ov), wv) and np.array_equal(T.np(ok), wk)
    assert bits_equal(T.np(os_), ws) and within_ulps(T.np(ob), wb, 4)


@pytest.mark.parametrize("name", ["sigmoid", "three"])
def test_nms_prefilter_path(T, name):
    """N >= 40 000 and 4k <= N: the large-N prefilter feeds the one-CTA kernel compacted candidates"""
    N, k = 50000, 6000
    rng = np.random.default_rng(50000)
    scores = layout(name, rng, N)
    boxes = near_dup_boxes(rng, N)
    got = run_nms(T, boxes, scores, k, float("-inf"))
    want = oracle_nms(boxes, scores, k, float("-inf"))
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    assert bits_equal(got[1], want[1]) and bits_equal(got[0], want[0])

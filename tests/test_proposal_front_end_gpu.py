"""Adversarial score layouts for the front ends of the proposal kernels, in TOPK, NMS and fused-proposal modes, against
the C restatement of the reference.  Keep lists, valid counts, indices and scores bit-exact; decoded boxes within the
4-ulp bar of the other parity tests.  Every output is filled with a sentinel (NaN, or -7 for int32) before a launch, so
a slot the kernel never wrote fails.

The proposal stage has three implementations of one algorithm, and each is run here on the same layouts:
- the one-CTA proposal_kernel (threshold batches, 11-bit histogram select, counting sort with a bitonic fall-back),
  forced with TFRPN_PROP_CLUSTER=0 (fixture T) -- also what the launcher picks for B > 8;
- proposal_cluster_kernel<CL, threads> on each of its seven compiled shapes (fixture TS): a local select per CTA
  with a 7S/8..S floor (S = 1024 / CL), a DSMEM merge with tau = max of the CTAs' thresholds, ranks by binary search
  in the peers' lists.  It is the default for B <= 8 and the only kernel of the rank / presorted launches;
- matrix NMS (TFRPN_NMS_PATH=matrix): rank launch, mask, sweep, and the lazy kernel for the images that run out of
  matrix rows.
The launch shape is read by tfrpn_create, so every configuration has its own handle.

The kernels order scores by their orderable bit pattern, so +0.0 ranks above -0.0; the C oracle compares float values,
so there the two tie and the lower index goes first.  Top-k is therefore checked against a NumPy restatement of the
kernels' order (equal to the C oracle whenever the zeros do not mix).  tfrpn_nms reads a -inf score threshold as no
threshold, while the C oracle keeps only scores > -inf.  The oracle NMS layouts therefore use one sign of zero and no
-inf; the mixed layouts are checked against the oracle fed in the kernels' order, and all shapes must agree bit for
bit on them."""
import ctypes as C
import functools
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


# Launch shapes, TFRPN_PROP_CLUSTER = 10 * t + cl (pick_cluster in csrc/proposals.cu): 0 is the one-CTA kernel
SHAPES = {"one_cta": 0, "1x1024": 1, "2x1024": 2, "2x512": 12, "4x512": 4, "4x256": 14, "8x256": 8, "8x512": 28}
CLUSTER_SHAPES = [s for s in SHAPES if SHAPES[s]]
CONFIGS = {s: {"TFRPN_PROP_CLUSTER": c} for s, c in SHAPES.items()}
# Matrix NMS with the default shape policy (B = 9: rank launch on 2 x 512, redo on the one-CTA kernel), and once with
# every launch on 8 x 256
MATRIX = ["matrix64", "matrix640", "matrix1024", "matrix640_8x256"]
CONFIGS.update({"matrix%d" % r: {"TFRPN_NMS_PATH": "matrix", "TFRPN_NMS_ROWS": r} for r in (64, 640, 1024)})
CONFIGS["matrix640_8x256"] = {"TFRPN_NMS_PATH": "matrix", "TFRPN_NMS_ROWS": 640, "TFRPN_PROP_CLUSTER": 8}


def ctas_of(config):
    """CTAs per image of the kernel that selects the batches (1 for the one-CTA kernel)"""
    env = CONFIGS[config]
    if "TFRPN_PROP_CLUSTER" in env:
        return max(env["TFRPN_PROP_CLUSTER"] % 10, 1)
    return 2   # matrix, default policy: B > 8 ranks on 2 x 512


def open_handle(cuda_device, config):
    import torch
    from tfrpn import _lib, synthetic
    if not CO.available():
        pytest.skip("oracle/_build/librpn_oracle.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    env = {k: str(v) for k, v in CONFIGS[config].items()}
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)   # read once, by tfrpn_create
    try:
        h = C.c_void_p()
        _lib.check(_lib.load().tfrpn_create(C.byref(h), cuda_device.index or 0))
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.lib, ns.syn, ns.dev, ns.h = torch, _lib, synthetic, cuda_device, h
    ns.config, ns.cl = config, ctas_of(config)
    ns.S = 1024 // ns.cl                      # composites per CTA in a batch
    ns.cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.np = lambda t: t.detach().cpu().numpy()
    ns.st = lambda: torch.cuda.current_stream(cuda_device).cuda_stream
    return ns


@pytest.fixture(scope="module")
def T(cuda_device):
    ns = open_handle(cuda_device, "one_cta")
    yield ns
    ns.lib.load().tfrpn_destroy(ns.h)


@pytest.fixture(scope="module")
def TS(request, cuda_device):
    """one handle per configuration named by the test's (indirect) parameter"""
    ns = open_handle(cuda_device, request.param)
    yield ns
    ns.lib.load().tfrpn_destroy(ns.h)


on_clusters = pytest.mark.parametrize("TS", CLUSTER_SHAPES, indirect=True)
on_nms_paths = pytest.mark.parametrize("TS", CLUSTER_SHAPES + MATRIX, indirect=True)
on_every_shape = pytest.mark.parametrize("TS", list(SHAPES), indirect=True)


B = 9   # > 8 images: the one-CTA kernel is also what the launcher picks


def layout(name, rng, N, for_nms=False, Bn=B):
    """(Bn, N) float32 scores"""
    if name == "equal":                       # one tie group
        return np.full((Bn, N), 0.5, F32)
    if name == "three":                       # tie groups straddling the batch floor, rank 1024 and rank k
        s = np.full((Bn, N), 0.25, F32)
        s[:, : min(N, 700)] = 0.75
        s[:, 700: min(N, 1100)] = 0.5
        for b in range(Bn):
            s[b] = s[b][rng.permutation(N)]
        return s
    if name == "one_bin_ulps":                # every score inside one 11-bit bin, 16 distinct values
        return (1.0 - 2.0 ** -20 * rng.uniform(0, 1, size=(Bn, N))).astype(F32)
    if name == "one_bin":                     # every score inside [0.8, 0.85): the first histogram separates nothing
        return (0.8 + 0.05 * rng.uniform(0, 1, size=(Bn, N))).astype(F32)
    if name == "special":                     # negatives, +-0, +-inf, denormals among sigmoid-like scores
        s = (rng.normal(0, 3, size=(Bn, N))).astype(F32)
        pool = np.array([0.0, 0.0 if for_nms else -0.0, np.inf, -3e38 if for_nms else -np.inf, 1e-45, -1e-45, 1e-40, -3e-39,
                         1.0, -1.0], F32)
        m = rng.uniform(size=(Bn, N)) < 0.3
        s[m] = rng.choice(pool, size=int(m.sum()))
        return s
    if name == "zeros":                       # +0, -0 and -inf only: three tie groups the C oracle cannot order
        return rng.choice(np.array([0.0, -0.0, -np.inf], F32), size=(Bn, N))
    if name == "sigmoid":
        return (1.0 / (1.0 + np.exp(-rng.normal(0, 2, size=(Bn, N))))).astype(F32)
    raise ValueError(name)


LAYOUTS = ["equal", "three", "one_bin_ulps", "one_bin", "special", "sigmoid"]
SHAPES_NK = [(37, 1), (37, 127), (1023, 127), (1023, 1025), (1024, 1025), (1025, 1025), (1025, 6000),
             (8649, 127), (8649, 1025), (8649, 6000), (37800, 6000)]


def near_dup_boxes(rng, N, Bn=B):
    """(Bn, N, 4) boxes around a few centres with jitter: most candidates are suppressed, so NMS runs through
    several batches"""
    centres = rng.uniform(0.2, 0.8, size=(Bn, 40, 2))
    pick = rng.integers(0, 40, size=(Bn, N))
    c = np.take_along_axis(centres, pick[..., None].repeat(2, -1), axis=1) + rng.normal(0, 0.002, size=(Bn, N, 2))
    sz = rng.uniform(0.1, 0.12, size=(Bn, N, 2))
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
    v = torch.full((Bn, k), float("nan"), device=T.dev)
    i = torch.full((Bn, k), -7, dtype=torch.int32, device=T.dev)
    g = torch.full((Bn, k, 4), float("nan"), device=T.dev)
    s_t, b_t = T.cu(scores), T.cu(boxes)
    T.lib.check(lib.tfrpn_topk(T.h, s_t.data_ptr(), Bn, N, k, v.data_ptr(), i.data_ptr(), b_t.data_ptr(), 1, g.data_ptr(), T.st()))
    torch.cuda.synchronize()
    return T.np(v), T.np(i), T.np(g)


def run_nms(T, boxes, scores, k, sthr, iou=0.7, rows=300):
    torch, lib = T.torch, T.lib.load()
    Bn, N = scores.shape
    nan = float("nan")
    nc = T.lib.NmsCfg(rows, rows, iou, sthr, 0, 1, k)
    nb = torch.full((Bn, rows, 4), nan, device=T.dev); ns = torch.full((Bn, rows), nan, device=T.dev)
    ncl = torch.full((Bn, rows), nan, device=T.dev)
    nv = torch.full((Bn,), -7, dtype=torch.int32, device=T.dev)
    nk = torch.full((Bn, rows), -7, dtype=torch.int32, device=T.dev)
    b_t, s_t = T.cu(boxes), T.cu(scores)
    T.lib.check(lib.tfrpn_nms(T.h, b_t.data_ptr(), s_t.data_ptr(), Bn, N, C.byref(nc), nb.data_ptr(), ns.data_ptr(),
                              ncl.data_ptr(), nv.data_ptr(), nk.data_ptr(), T.st()))
    torch.cuda.synchronize()
    assert bits_equal(T.np(ncl), np.zeros((Bn, rows), F32))
    return T.np(nb), T.np(ns), T.np(nv), T.np(nk)


def run_proposals(T, reg, cls, anchors, hp, k):
    from tfrpn.proposals import proposal_cfg
    torch, lib = T.torch, T.lib.load()
    Bn, N = cls.shape
    pc = proposal_cfg(hp, pre_nms_topn=k)
    P = int(hp["test_nms_topn"])
    ob = torch.full((Bn, P, 4), float("nan"), device=T.dev); os_ = torch.full((Bn, P), float("nan"), device=T.dev)
    ov = torch.full((Bn,), -7, dtype=torch.int32, device=T.dev); ok = torch.full((Bn, P), -7, dtype=torch.int32, device=T.dev)
    r_t, c_t, a_t = T.cu(reg), T.cu(cls), T.cu(anchors)
    T.lib.check(lib.tfrpn_proposals(T.h, r_t.data_ptr(), c_t.data_ptr(), a_t.data_ptr(), Bn, N, C.byref(pc), ob.data_ptr(),
                                    os_.data_ptr(), ov.data_ptr(), ok.data_ptr(), T.st()))
    torch.cuda.synchronize()
    return T.np(ob), T.np(os_), T.np(ov), T.np(ok)


def oracle_nms(boxes, scores, k, sthr, iou=0.7, rows=300):
    """NMS over the top-k entries (pre_nms_topn = k; 0 = all), keep indices in the caller's numbering"""
    Bn, N = scores.shape
    k = N if k == 0 else min(k, N)
    v, idx = CO.top_k(scores, k)
    sub = np.stack([boxes[b][idx[b]] for b in range(Bn)])
    wb, ws, _, wv, wk = CO.nms(sub, v, rows, rows, iou, sthr)
    wk = np.where(wk >= 0, np.take_along_axis(idx, np.maximum(wk, 0), axis=1), -1).astype(np.int32)
    return wb, ws, wv, wk


def composite_oracle_nms(boxes, scores, k, iou=0.7, rows=300):
    """NMS without a score threshold in the kernels' order (+0 above -0, -inf included): the oracle NMS fed the top-k
    entries in that order with stand-in scores that fall strictly, its outputs mapped back"""
    Bn, N = scores.shape
    k = N if k == 0 else min(k, N)
    _, idx = composite_topk(scores, k)
    sub = np.stack([boxes[b][idx[b]] for b in range(Bn)])
    stand_in = np.broadcast_to(np.arange(k, 0, -1, dtype=F32), (Bn, k))
    wb, _, _, wv, wk = CO.nms(sub, stand_in, rows, rows, iou)
    keep = np.where(wk >= 0, np.take_along_axis(idx, np.maximum(wk, 0), axis=1), -1).astype(np.int32)
    ws = np.where(keep >= 0, np.take_along_axis(scores, np.maximum(keep, 0), axis=1), F32(0)).astype(F32)
    return wb, ws, wv, keep


def assert_nms_equal(got, want):
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[3], want[3])
    assert bits_equal(got[1], want[1]) and bits_equal(got[0], want[0])


# ---- the layouts on every launch shape (inputs and oracle results are shared by the shapes) -------------------------

@functools.lru_cache(maxsize=None)
def topk_case(name, N, k):
    rng = np.random.default_rng(N * 7 + k)
    scores = layout(name, rng, N)
    boxes = rng.uniform(0, 1, size=(B, N, 4)).astype(F32)
    wv, wi = composite_topk(scores, k)
    if name != "special":
        assert np.array_equal(wi, CO.top_k(scores, k)[1])
    return scores, boxes, wv, wi


def check_topk_layout(T, name, N, k):
    scores, boxes, wv, wi = topk_case(name, N, min(k, N))
    v, i, g = run_topk(T, scores, min(k, N), boxes)
    assert np.array_equal(i, wi)
    assert bits_equal(v, wv)
    assert bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(B)]))


@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES_NK)
def test_topk_layouts(T, name, N, k):
    check_topk_layout(T, name, N, k)


@on_clusters
@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES_NK)
def test_topk_layouts_cluster(TS, name, N, k):
    check_topk_layout(TS, name, N, k)


@functools.lru_cache(maxsize=None)
def nms_case(name, N, k):
    rng = np.random.default_rng(N * 11 + k)
    scores = layout(name, rng, N, for_nms=True)
    boxes = near_dup_boxes(rng, N)
    return scores, boxes, oracle_nms(boxes, scores, k, float("-inf"))


def check_nms_layout(T, name, N, k):
    scores, boxes, want = nms_case(name, N, k)
    assert_nms_equal(run_nms(T, boxes, scores, k, float("-inf")), want)


@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES_NK)
def test_nms_layouts_near_duplicates(T, name, N, k):
    check_nms_layout(T, name, N, k)


@on_nms_paths
@pytest.mark.parametrize("name", LAYOUTS)
@pytest.mark.parametrize("N,k", SHAPES_NK)
def test_nms_layouts_near_duplicates_paths(TS, name, N, k):
    check_nms_layout(TS, name, N, k)


@functools.lru_cache(maxsize=None)
def threshold_case(M, N, k):
    rng = np.random.default_rng(M + N)
    scores = np.full((B, N), 0.01, F32)
    for b in range(B):
        m = min(M, N)
        scores[b, rng.permutation(N)[:m]] = rng.uniform(0.2, 0.9, size=m).astype(F32)
    scores[1, :5] = 0.05                       # exactly at the threshold: not above it
    boxes = random_boxes(rng, B, N)
    return scores, boxes, oracle_nms(boxes, scores, k, 0.05)


def random_boxes(rng, Bn, N):
    """(Bn, N, 4) boxes drawn like GT boxes: NMS keeps many"""
    from tfrpn import synthetic
    return synthetic.nms_boxes(rng, Bn, N)[0]


def check_nms_score_threshold(T, M, N, k):
    scores, boxes, want = threshold_case(M, N, k)
    assert_nms_equal(run_nms(T, boxes, scores, k, 0.05), want)


@pytest.mark.parametrize("M", [0, 100, 1030])
@pytest.mark.parametrize("N,k", [(1025, 0), (8649, 6000), (8649, 127), (37800, 0)])
def test_nms_score_threshold(T, M, N, k):
    """a score threshold leaving M entries: key 0 is never consumed"""
    check_nms_score_threshold(T, M, N, k)


@on_nms_paths
@pytest.mark.parametrize("M", [0, 100, 1030])
@pytest.mark.parametrize("N,k", [(1025, 0), (8649, 6000), (8649, 127), (37800, 0)])
def test_nms_score_threshold_paths(TS, M, N, k):
    """the cluster kernel keeps entries at or below the threshold in its batches as nonzero composites: K = the count
    above it must end the consumption"""
    check_nms_score_threshold(TS, M, N, k)


@functools.lru_cache(maxsize=None)
def c2_case(name, k):
    hp = dict(O.get_hyper_params("vgg16"))
    anchors = O.generate_anchors(hp)
    N = anchors.shape[0]
    rng = np.random.default_rng(k)
    reg = rng.normal(0, 0.5, size=(B, N, 4)).astype(F32)
    cls = layout(name, rng, N, for_nms=True)
    return hp, anchors, reg, cls, CO.proposals(reg, cls, anchors, hp, k)


def check_proposals_layout(T, name, k):
    hp, anchors, reg, cls, (wb, ws, wv, wk) = c2_case(name, k)
    ob, os_, ov, ok = run_proposals(T, reg, cls, anchors, hp, k)
    assert np.array_equal(ov, wv) and np.array_equal(ok, wk)
    assert bits_equal(os_, ws) and within_ulps(ob, wb, 4)


@pytest.mark.parametrize("name", ["three", "one_bin", "sigmoid", "special"])
@pytest.mark.parametrize("k", [127, 1025, 6000])
def test_proposals_layouts(T, name, k):
    """the fused decode + NMS mode at the C2 shape"""
    check_proposals_layout(T, name, k)


@on_nms_paths
@pytest.mark.parametrize("name", ["three", "one_bin", "sigmoid", "special"])
@pytest.mark.parametrize("k", [127, 1025, 6000])
def test_proposals_layouts_paths(TS, name, k):
    check_proposals_layout(TS, name, k)


@functools.lru_cache(maxsize=None)
def prefilter_case(name):
    N, k = 50000, 6000
    rng = np.random.default_rng(50000)
    scores = layout(name, rng, N)
    boxes = near_dup_boxes(rng, N)
    return scores, boxes, oracle_nms(boxes, scores, k, float("-inf"))


def check_prefilter(T, name):
    scores, boxes, want = prefilter_case(name)
    assert_nms_equal(run_nms(T, boxes, scores, 6000, float("-inf")), want)


@pytest.mark.parametrize("name", ["sigmoid", "three"])
def test_nms_prefilter_path(T, name):
    """N >= 40 000 and 4k <= N: the large-N prefilter feeds the one-CTA kernel compacted candidates"""
    check_prefilter(T, name)


@on_clusters
@pytest.mark.parametrize("name", ["sigmoid", "three"])
def test_nms_prefilter_path_cluster(TS, name):
    """the prefilter's compacted candidates (counts + remap) through the cluster kernel"""
    check_prefilter(TS, name)


# ---- cases of the cluster kernel's own front end --------------------------------------------------------------------

def owner_of(N, cl):
    """CTA of the cluster that owns each entry: 32-entry chunk c belongs to CTA c % CL"""
    return (np.arange(N) // 32) % cl


@on_every_shape
@pytest.mark.parametrize("name", ["equal", "three", "special", "sigmoid"])
@pytest.mark.parametrize("n", ["1", "31", "33", "37", "32cl-1", "32cl+1"])
def test_small_n(TS, name, n):
    """N below a chunk per CTA (some CTAs own no chunk at all), and N = 32 * CL +- 1 (the last chunk partial or
    alone): top-k of every entry, NMS over every entry"""
    N = int(n) if n.isdigit() else 32 * TS.cl + (1 if n.endswith("+1") else -1)
    rng = np.random.default_rng(N + len(name))
    scores = layout(name, rng, N)
    boxes = rng.uniform(0, 1, size=(B, N, 4)).astype(F32)
    v, i, g = run_topk(TS, scores, N, boxes)
    wv, wi = composite_topk(scores, N)
    assert np.array_equal(i, wi) and bits_equal(v, wv)
    assert bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(B)]))
    ns = layout(name, rng, N, for_nms=True)
    for bx in (near_dup_boxes(rng, N), random_boxes(rng, B, N)):
        assert_nms_equal(run_nms(TS, bx, ns, 0, float("-inf")), oracle_nms(bx, ns, 0, float("-inf")))


@on_every_shape
@pytest.mark.parametrize("N", [8649, 37800])
def test_skewed_ownership(TS, N):
    """every high score lies in the chunks of one CTA: its list alone sets tau, batches shrink to about 7S/8, and
    k = 6000 takes dozens of batches (top-k, and NMS over near-duplicates that keeps few)"""
    rng = np.random.default_rng(N)
    own = owner_of(N, TS.cl) == TS.cl - 1
    scores = rng.uniform(0.0, 0.4, size=(B, N)).astype(F32)
    scores[:, own] = rng.uniform(0.5, 1.0, size=(B, int(own.sum()))).astype(F32)
    scores[:, own & (np.arange(N) % 5 == 0)] = 0.75           # a tie group inside the favoured CTA
    k = 6000
    boxes = rng.uniform(0, 1, size=(B, N, 4)).astype(F32)
    v, i, g = run_topk(TS, scores, k, boxes)
    wv, wi = CO.top_k(scores, k)
    assert np.array_equal(i, wi) and bits_equal(v, wv)
    assert bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(B)]))
    nb = near_dup_boxes(rng, N)
    assert_nms_equal(run_nms(TS, nb, scores, k, float("-inf")), oracle_nms(nb, scores, k, float("-inf")))


@on_every_shape
@pytest.mark.parametrize("quantized", [False, True])
@pytest.mark.parametrize("N", [8649, 37800])
def test_every_list_cut(TS, quantized, N):
    """every CTA's list is full, and CTA r's scores sit r steps lower: tau (the first CTA's threshold) cuts most of
    the later CTAs' lists, which must offer the cut entries again in the next batch.  Quantized: tie groups across
    tau and across CTAs"""
    rng = np.random.default_rng(N + quantized)
    r = owner_of(N, TS.cl)
    L = N / TS.cl                                           # entries per CTA
    step = 0.8 * (TS.S / L) / max(TS.cl - 1, 1)
    scores = (rng.uniform(0, 1, size=(B, N)) - r * step).astype(F32)
    if quantized:
        scores = (np.round(scores * 256) / 256 + 0.0).astype(F32)   # (+ 0.0: no -0 beside +0)
    k = 6000
    boxes = rng.uniform(0, 1, size=(B, N, 4)).astype(F32)
    v, i, g = run_topk(TS, scores, k, boxes)
    wv, wi = CO.top_k(scores, k)
    assert np.array_equal(i, wi) and bits_equal(v, wv)
    assert bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(B)]))
    nb = near_dup_boxes(rng, N)
    assert_nms_equal(run_nms(TS, nb, scores, k, float("-inf")), oracle_nms(nb, scores, k, float("-inf")))


@pytest.mark.parametrize("TS", list(SHAPES) + MATRIX, indirect=True)
@pytest.mark.parametrize("left", ["0", "1", "S-1", "S+1", "1030"])
@pytest.mark.parametrize("N,k", [(1025, 0), (8649, 0), (8649, 6000), (8649, 700)])
def test_score_threshold_leaves(TS, left, N, k):
    """a score threshold leaving 0, 1, S - 1, S + 1 or 1030 entries above it (S: composites per CTA and batch);
    entries exactly at the threshold and tie groups on both sides of it"""
    M = {"0": 0, "1": 1, "S-1": TS.S - 1, "S+1": TS.S + 1, "1030": 1030}[left]
    rng = np.random.default_rng(M * 3 + N + k)
    thr = F32(0.05)
    scores = rng.uniform(-1.0, 0.05, size=(B, N)).astype(F32)
    scores[rng.uniform(size=(B, N)) < 0.2] = thr             # at the threshold: not above it
    for b in range(B):
        m = min(M, N)
        hi = (np.round(rng.uniform(0.06, 0.9, size=m) * 64) / 64).astype(F32)   # ties among the kept candidates
        scores[b, rng.permutation(N)[:m]] = hi
    boxes = random_boxes(rng, B, N)
    got = run_nms(TS, boxes, scores, k, float(thr))
    assert_nms_equal(got, oracle_nms(boxes, scores, k, float(thr)))
    assert np.all(got[2] <= min(M, N))


# ---- inputs the C oracle cannot order: all launch shapes must agree -------------------------------------------------

@pytest.fixture(scope="module")
def every_shape(cuda_device):
    hs = {}
    try:
        for s in SHAPES:
            hs[s] = open_handle(cuda_device, s)
        yield hs
    finally:
        for ns in hs.values():
            ns.lib.load().tfrpn_destroy(ns.h)


@pytest.mark.parametrize("name", ["special", "zeros"])
@pytest.mark.parametrize("N,k", [(37, 0), (1025, 1025), (8649, 6000), (37800, 6000), (50000, 6000)])
def test_mixed_zeros_nms_all_shapes_agree(every_shape, name, N, k):
    """+0 / -0 / -inf mixed, no score threshold: every shape gives the same bits, and the oracle NMS run in the
    kernels' order agrees"""
    rng = np.random.default_rng(N + k + len(name))
    scores = layout(name, rng, N)
    boxes = near_dup_boxes(rng, N)
    ref = run_nms(every_shape["one_cta"], boxes, scores, k, float("-inf"))
    assert_nms_equal(ref, composite_oracle_nms(boxes, scores, k))
    for s, ns in every_shape.items():
        got = run_nms(ns, boxes, scores, k, float("-inf"))
        assert all(bits_equal(a, b) if a.dtype == F32 else np.array_equal(a, b) for a, b in zip(got, ref)), s


@pytest.mark.parametrize("name", ["special", "zeros"])
@pytest.mark.parametrize("k", [127, 6000])
def test_mixed_zeros_proposals_all_shapes_agree(every_shape, name, k):
    """the fused mode at the C2 shape on +0 / -0 / -inf scores: every shape gives the same bits"""
    hp = dict(O.get_hyper_params("vgg16"))
    anchors = O.generate_anchors(hp)
    N = anchors.shape[0]
    rng = np.random.default_rng(k + len(name))
    reg = rng.normal(0, 0.5, size=(B, N, 4)).astype(F32)
    cls = layout(name, rng, N)
    ref = run_proposals(every_shape["one_cta"], reg, cls, anchors, hp, k)
    assert np.all(ref[2] > 0)
    for s, ns in every_shape.items():
        got = run_proposals(ns, reg, cls, anchors, hp, k)
        assert all(bits_equal(a, b) if a.dtype == F32 else np.array_equal(a, b) for a, b in zip(got, ref)), s


# ---- keys re-read from global memory: N above the shared-memory staging limit, k > N / 4 (no prefilter) ---------

PROP_SMEM_LIMIT = 227 * 1024 - 4096
BATCH, NMS_CHUNK, SEL_NB, CL_NB = 1024, 128, 2048, 2048


def smem_bytes(config, n_staged, max_out):
    """prop_smem_bytes / cluster_smem_bytes of csrc/proposals.cu"""
    mo = (max_out + 3) & ~3
    cl = SHAPES[config] % 10
    if cl == 0:
        return 2 * BATCH * 8 + BATCH * 4 + (mo + NMS_CHUNK) * 20 + NMS_CHUNK * 24 + SEL_NB * 4 + n_staged * 4 + 16
    S = BATCH // cl
    nchunks = (n_staged + 31) // 32
    lmax = (nchunks + cl - 1) // cl * 32
    return CL_NB * 4 + BATCH * 8 + 2 * S * 8 + (BATCH + mo) * 20 + NMS_CHUNK * 36 + lmax * 4 + 16


def first_unstaged_n(config, max_out):
    lo, hi = 1, 1 << 22                           # smem_bytes(lo) fits, smem_bytes(hi) does not
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if smem_bytes(config, mid, max_out) <= PROP_SMEM_LIMIT else (lo, mid)
    return hi


@on_every_shape
@pytest.mark.parametrize("name", ["sigmoid", "three"])
def test_unstaged_keys_topk(TS, name):
    N = first_unstaged_n(TS.config, 0) + 37
    k = N // 4 + 1                                # k > N / 4: the prefilter does not apply
    assert smem_bytes(TS.config, N, 0) > PROP_SMEM_LIMIT and 4 * k > N
    rng = np.random.default_rng(N)
    scores = layout(name, rng, N, Bn=2)
    boxes = rng.uniform(0, 1, size=(2, N, 4)).astype(F32)
    v, i, g = run_topk(TS, scores, k, boxes)
    wv, wi = composite_topk(scores, k)
    assert np.array_equal(i, wi) and bits_equal(v, wv)
    assert bits_equal(g, np.stack([boxes[b][wi[b]] for b in range(2)]))


@on_every_shape
def test_unstaged_keys_nms(TS):
    """pre_nms_topn = 0 with max_out = 500 (above the prefilter's NMS cap): NMS over near-duplicates walks every rank"""
    N = first_unstaged_n(TS.config, 500) + 37
    assert smem_bytes(TS.config, N, 500) > PROP_SMEM_LIMIT
    rng = np.random.default_rng(N + 1)
    scores = layout("sigmoid", rng, N, Bn=2)
    boxes = near_dup_boxes(rng, N, Bn=2)
    got = run_nms(TS, boxes, scores, 0, float("-inf"), rows=500)
    assert_nms_equal(got, oracle_nms(boxes, scores, 0, float("-inf"), rows=500))

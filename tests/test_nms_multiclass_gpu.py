"""tfrpn_nms_multiclass (nms_mc_stage_kernel -> proposal_kernel per class -> nms_mc_merge_kernel) against
oracle/rpn_oracle.py:combined_non_max_suppression, bit for bit, over class counts, box layouts, K, output sizes,
score thresholds, pre_nms_topn and clipping; against tfrpn_nms for one class; and against the per-class composition
the Python drop-in used before (restated below) on score layouts the oracle cannot order.  Then the C ABI: the
caller's stream, CUDA-graph capture, error codes, determinism.  Every output is prefilled with NaN or -7."""
import ctypes as C

import numpy as np
import pytest

from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32
NINF = float("-inf")


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    import tfrpn
    from tfrpn import _lib
    from tfrpn.utils import bbox_utils

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.tfrpn, ns.lib, ns.L, ns.bbox, ns.dev = torch, tfrpn, _lib.load(), _lib, bbox_utils, cuda_device
    ns.cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.h = _lib.handle(cuda_device.index)
    return ns


def cfg_of(T, per_class, total, iou=0.5, sthr=NINF, pad=False, clip=True, topn=0):
    return T.L.NmsCfg(per_class, total, iou, sthr, int(pad), int(clip), topn)


def rows_of(cfg, Cn):
    return min(cfg.max_total_size, cfg.max_output_size_per_class * Cn) if cfg.pad_per_class else cfg.max_total_size


def outputs(T, B, rows):
    t = T.torch
    return (t.full((B, rows, 4), float("nan"), device=T.dev), t.full((B, rows), float("nan"), device=T.dev),
            t.full((B, rows), float("nan"), device=T.dev), t.full((B,), -7, dtype=t.int32, device=T.dev),
            t.full((B, rows), -7, dtype=t.int32, device=T.dev))


def call(T, bx, sc, cfg, outs, h=None, stream=None):
    B, K, q, _ = bx.shape
    Cn = sc.shape[2]
    st = stream if stream is not None else T.torch.cuda.current_stream(T.dev).cuda_stream
    return T.lib.tfrpn_nms_multiclass(h or T.h, bx.data_ptr(), q, sc.data_ptr(), B, K, Cn, C.byref(cfg),
                                      *[o.data_ptr() for o in outs], st)


def native(T, boxes, scores, cfg, h=None):
    """host arrays in -> (boxes, scores, classes, valid, keep_idx) host arrays"""
    bx, sc = T.cu(boxes), T.cu(scores)
    outs = outputs(T, boxes.shape[0], rows_of(cfg, scores.shape[2]))
    assert call(T, bx, sc, cfg, outs, h=h) == 0, T.lib.tfrpn_last_error()
    return [o.cpu().numpy() for o in outs]


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32 if a.dtype == F32 else np.int32)


def assert_same(got, want):
    for g, w, name in zip(got, want, ("boxes", "scores", "classes", "valid", "keep_idx")):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape, name
        assert np.array_equal(bits(g.astype(w.dtype)), bits(w)), "%s differ at %s" % (name, np.argwhere(bits(g) != bits(w))[:5])


def layout(rng, B, K, Cn, q, tie_every=7):
    """clustered boxes (so NMS suppresses; some reach outside [0,1]), SSD-like scores sigmoid(N(-3, 2^2)) with every
    tie_every-th row quantised to 1/16 (equal scores inside a class and across classes)"""
    ncl = max(1, K // 16)
    cen = rng.uniform(0.05, 0.95, size=(B, ncl, 2))
    pick = rng.integers(0, ncl, size=(B, K, q))
    ctr = np.take_along_axis(cen[:, :, None, :], pick.reshape(B, K * q, 1, 1).repeat(2, -1), 1).reshape(B, K, q, 2)
    ctr = ctr + rng.normal(0, 0.02, size=ctr.shape)
    sz = rng.uniform(0.04, 0.3, size=(B, K, q, 2))
    boxes = np.concatenate([ctr - sz / 2, ctr + sz / 2], -1).astype(F32)
    scores = (1.0 / (1.0 + np.exp(-rng.normal(-3.0, 2.0, size=(B, K, Cn))))).astype(F32)
    if tie_every:
        scores[:, ::tie_every, :] = np.round(scores[:, ::tie_every, :] * 16) / 16
    return boxes, scores


def oracle(boxes, scores, cfg):
    """the oracle, with pre_nms_topn as per-class tf.nn.top_k: entries outside a class's top n never compete"""
    sc = scores
    if cfg.pre_nms_topn > 0:
        sc = scores.copy()
        B, K, Cn = scores.shape
        for b in range(B):
            for c in range(Cn):
                order = np.argsort(-scores[b, :, c].astype(np.float64), kind="stable")
                sc[b, order[cfg.pre_nms_topn:], c] = np.nan     # NaN > threshold is false
    return O.combined_non_max_suppression(boxes, sc, cfg.max_output_size_per_class, cfg.max_total_size,
                                          iou_threshold=cfg.iou_threshold, score_threshold=cfg.score_threshold,
                                          pad_per_class=bool(cfg.pad_per_class), clip_boxes=bool(cfg.clip_boxes),
                                          return_indices=True)


# C, q, K, per_class, total, pad, score_threshold, pre_nms_topn, clip
CASES = [
    (1, 1, 1, 5, 5, False, NINF, 0, True),
    (1, 1, 8732, 100, 50, True, 0.05, 0, True),
    (2, 1, 1, 3, 5, False, NINF, 0, False),
    (2, 2, 37, 10, 30, True, 0.05, 0, True),
    (2, 1, 50000, 100, 150, False, 0.05, 0, True),      # K past the large-N prefilter's threshold
    (2, 2, 50000, 50, 300, True, NINF, 0, False),
    (5, 1, 1000, 30, 20, False, 0.3, 100, False),       # total < per_class; pre_nms_topn below the candidates
    (5, 5, 8732, 100, 200, True, 0.5, 20000, True),     # pre_nms_topn above K
    (5, 5, 1, 4, 10, True, NINF, 0, True),
    (5, 1, 37, 8, 100, False, 0.05, 3, True),           # total > per_class * C
    (21, 1, 8732, 100, 200, False, 0.05, 0, True),
    (21, 21, 1000, 20, 1000, False, NINF, 0, False),
    (21, 1, 37, 5, 200, True, 0.1, 3, True),
    (91, 1, 1000, 10, 100, True, 0.6, 50, True),
    (91, 91, 37, 5, 600, True, NINF, 0, False),
    (91, 91, 1000, 100, 100, False, 0.05, 0, True),
]


@pytest.mark.parametrize("Cn,q,K,per_class,total,pad,sthr,topn,clip", CASES)
def test_vs_oracle(T, Cn, q, K, per_class, total, pad, sthr, topn, clip):
    rng = np.random.default_rng(K * 131 + Cn * 7 + q)
    B = 2
    boxes, scores = layout(rng, B, K, Cn, q)
    cfg = cfg_of(T, per_class, total, 0.45, sthr, pad, clip, topn)
    assert_same(native(T, boxes, scores, cfg), oracle(boxes, scores, cfg))


@pytest.fixture(scope="module", params=["column", "rows"])
def stage_handle(T, request):
    """a handle with the staging layout forced by TFRPN_NMS_MC_STAGE (read when the handle is created)"""
    import os
    old = os.environ.get("TFRPN_NMS_MC_STAGE")
    os.environ["TFRPN_NMS_MC_STAGE"] = request.param
    h = T.L.P()
    try:
        assert T.lib.tfrpn_create(C.byref(h), T.dev.index) == 0
    finally:
        if old is None:
            del os.environ["TFRPN_NMS_MC_STAGE"]
        else:
            os.environ["TFRPN_NMS_MC_STAGE"] = old
    yield h
    T.torch.cuda.synchronize()
    T.lib.tfrpn_destroy(h)


@pytest.mark.parametrize("Cn,q,K,per_class,total,pad,sthr,topn,clip", CASES)
def test_vs_oracle_each_staging_layout(T, stage_handle, Cn, q, K, per_class, total, pad, sthr, topn, clip):
    rng = np.random.default_rng(K * 131 + Cn * 7 + q)
    boxes, scores = layout(rng, 2, K, Cn, q)
    cfg = cfg_of(T, per_class, total, 0.45, sthr, pad, clip, topn)
    assert_same(native(T, boxes, scores, cfg, h=stage_handle), oracle(boxes, scores, cfg))


@pytest.mark.parametrize("q1", [True, False])
def test_merge_scratch_in_global_memory(T, stage_handle, q1):
    """C * min(P, rows) = 60000 keys: the merge's per-CTA scratch (16 C + 4 C min(P, rows) bytes) is past the
    shared-memory limit and lives in the workspace"""
    rng = np.random.default_rng(600)
    Cn, K = 600, 37
    assert 16 * Cn + 4 * Cn * 100 > 227 * 1024 - 4096
    boxes, scores = layout(rng, 2, K, Cn, 1 if q1 else Cn)
    for sthr in (NINF, 0.05):
        cfg = cfg_of(T, 100, 100, 0.45, sthr, False, True)
        assert_same(native(T, boxes, scores, cfg, h=stage_handle), oracle(boxes, scores, cfg))


@pytest.mark.parametrize("K", [37, 1000])
@pytest.mark.parametrize("qc", [False, True])
def test_score_threshold_leaves(T, K, qc):
    """class 0: nothing above the threshold (half exactly at it); class 1: one entry; class 2: every entry;
    class 3: a third exactly at the threshold, the rest just above or below"""
    rng = np.random.default_rng(K)
    B, Cn, thr = 2, 4, F32(0.25)
    boxes, _ = layout(rng, B, K, Cn, Cn if qc else 1)
    s = np.empty((B, K, Cn), F32)
    s[:, :, 0] = np.where(rng.random((B, K)) < 0.5, thr, rng.uniform(0, 0.25, (B, K)).astype(F32))
    s[:, :, 1] = rng.uniform(0, 0.25, (B, K)).astype(F32)
    s[:, K // 2, 1] = np.nextafter(thr, F32(1))
    s[:, :, 2] = rng.uniform(0.2500001, 1, (B, K)).astype(F32)
    r = rng.random((B, K))
    s[:, :, 3] = np.where(r < 1 / 3, thr, np.where(r < 2 / 3, np.nextafter(thr, F32(1)), np.nextafter(thr, F32(0))))
    for per_class, total, pad in ((5, 12, False), (50, 400, True)):
        cfg = cfg_of(T, per_class, total, 0.5, float(thr), pad)
        got = native(T, boxes, s, cfg)
        assert_same(got, oracle(boxes, s, cfg))
        assert not np.any(got[2][:, :got[3].min()] == 0)   # class 0 keeps nothing


@pytest.mark.parametrize("K,sthr,topn", [(1000, NINF, 0), (8732, 0.05, 0), (50000, 0.05, 300)])
def test_one_class_equals_tfrpn_nms(T, K, sthr, topn):
    rng = np.random.default_rng(3)
    B = 3
    boxes, scores = layout(rng, B, K, 1, 1)
    for per_class, total, pad in ((100, 100, False), (100, 40, True), (50, 80, False)):
        cfg = cfg_of(T, per_class, total, 0.5, sthr, pad, True, topn)
        got = native(T, boxes, scores, cfg)
        bx, sc = T.cu(boxes), T.cu(scores)
        outs = outputs(T, B, rows_of(cfg, 1))
        rc = T.lib.tfrpn_nms(T.h, bx.data_ptr(), sc.data_ptr(), B, K, C.byref(cfg), *[o.data_ptr() for o in outs],
                             T.torch.cuda.current_stream(T.dev).cuda_stream)
        assert rc == 0
        assert_same(got, [o.cpu().numpy() for o in outs])


# ---- the per-class composition the Python drop-in ran before (B*C one-class NMS launches + a stable torch.sort
# merge), restated as the reference.  One correction: it masked unused keep-list slots with -inf, which ties with a
# kept score of -inf (kept when the score threshold is -inf), so an unused slot of a lower class could take an output
# row ahead of it.  Here unused slots sort after every kept entry.
def composed(T, boxes, scores, cfg):
    t = T.torch
    bx, sc = T.cu(boxes), T.cu(scores)
    B, K, Cn = sc.shape
    q = bx.shape[2]
    P, total = cfg.max_output_size_per_class, cfg.max_total_size
    rows = rows_of(cfg, Cn)
    dev = T.dev
    sc_t = sc.permute(0, 2, 1).contiguous().reshape(B * Cn, K)
    bx_t = (bx.expand(B, K, Cn, 4) if q == 1 else bx).permute(0, 2, 1, 3).contiguous().reshape(B * Cn, K, 4)
    c1 = cfg_of(T, P, P, cfg.iou_threshold, cfg.score_threshold, False, bool(cfg.clip_boxes), cfg.pre_nms_topn)
    nb, ns, nc, nv, ni = outputs(T, B * Cn, P)
    assert T.lib.tfrpn_nms(T.h, bx_t.data_ptr(), sc_t.data_ptr(), B * Cn, K, C.byref(c1), nb.data_ptr(), ns.data_ptr(),
                           nc.data_ptr(), nv.data_ptr(), ni.data_ptr(), t.cuda.current_stream(dev).cuda_stream) == 0
    slot = t.arange(P, device=dev)
    live = (slot[None, :] < nv[:, None]).reshape(B, Cn * P)
    key = t.where(live, ns.reshape(B, Cn * P), t.full((B, Cn * P), float("-inf"), device=dev))
    order = t.sort(key, dim=1, descending=True, stable=True).indices
    order = t.gather(order, 1, t.sort(t.gather(live, 1, order).to(t.int8), dim=1, descending=True, stable=True).indices)
    n_live = live.sum(dim=1)
    take = min(rows, Cn * P)
    order = order[:, :take]
    valid = t.clamp(n_live, max=min(rows, total)).to(t.int32)
    keep = t.arange(take, device=dev)[None, :] < valid[:, None]
    ob = t.zeros((B, rows, 4), dtype=t.float32, device=dev)
    os_ = t.zeros((B, rows), dtype=t.float32, device=dev)
    oc = t.zeros((B, rows), dtype=t.float32, device=dev)
    oi = t.full((B, rows), -1, dtype=t.int32, device=dev)
    gb = t.gather(nb.reshape(B, Cn * P, 4), 1, order[..., None].expand(-1, -1, 4))
    gs = t.gather(ns.reshape(B, Cn * P), 1, order)
    gi = t.gather(ni.reshape(B, Cn * P), 1, order)
    ob[:, :take] = t.where(keep[..., None], gb, t.zeros_like(gb))
    os_[:, :take] = t.where(keep, gs, t.zeros_like(gs))
    oc[:, :take] = t.where(keep, (order // P).to(t.float32), t.zeros_like(gs))
    oi[:, :take] = t.where(keep, gi, t.full_like(gi, -1))
    return [x.cpu().numpy() for x in (ob, os_, oc, valid, oi)]


NEG_NAN = np.array([0xFFC00000], np.uint32).view(F32)[0]


@pytest.mark.parametrize("q1", [True, False])
@pytest.mark.parametrize("kind", ["ties", "specials", "specials_thr"])
def test_vs_composition_on_unordered_layouts(T, stage_handle, kind, q1):
    rng = np.random.default_rng(11)
    B, K, Cn = 3, 300, 5
    boxes, scores = layout(rng, B, K, Cn, 1 if q1 else Cn, tie_every=0)
    if kind == "ties":        # few distinct values: long tie groups inside every class and across classes
        scores = rng.choice(np.array([0.9, 0.5, 0.25, 0.125], F32), size=(B, K, Cn))
        sthr = NINF
    else:                     # +0 / -0, +-inf, +-NaN and a few ordinary values
        vals = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, NEG_NAN, 0.5, -0.5], F32)
        scores = vals[rng.integers(0, len(vals), size=(B, K, Cn))]
        scores[2, :, 1] = -np.inf   # one class of only -inf scores
        sthr = NINF if kind == "specials" else -1.0
    for per_class, total, pad, topn in ((10, 25, False, 0), (40, 500, True, 0), (20, 60, False, 30)):
        cfg = cfg_of(T, per_class, total, 0.5, sthr, pad, True, topn)
        assert_same(native(T, boxes, scores, cfg, h=stage_handle), composed(T, boxes, scores, cfg))


@pytest.mark.parametrize("Cn,q", [(3, 1), (4, 4)])
def test_vs_composition_on_random_layouts(T, Cn, q):
    rng = np.random.default_rng(5)
    boxes, scores = layout(rng, 4, 2000, Cn, q)
    cfg = cfg_of(T, 50, 120, 0.5, 0.05, True, True, 0)
    assert_same(native(T, boxes, scores, cfg), composed(T, boxes, scores, cfg))


def test_python_drop_in(T):
    """non_max_suppression with C > 1 runs the native call: NumPy in -> NumPy out, torch in -> torch out,
    return_indices and pre_nms_topn as keyword arguments"""
    rng = np.random.default_rng(9)
    boxes, scores = layout(rng, 2, 500, 6, 1)
    kw = dict(max_output_size_per_class=20, max_total_size=50, iou_threshold=0.45, score_threshold=0.05, pre_nms_topn=100)
    cfg = cfg_of(T, 20, 50, 0.45, 0.05, False, True, 100)
    want = native(T, boxes, scores, cfg)
    got = T.bbox.non_max_suppression(boxes, scores, return_indices=True, **kw)
    assert all(isinstance(x, np.ndarray) for x in got)
    assert_same(got, want)
    res = T.bbox.non_max_suppression(T.cu(boxes), T.cu(scores), **kw)
    assert len(res) == 4 and all(isinstance(x, T.torch.Tensor) and x.is_cuda for x in res)
    assert_same([x.cpu().numpy() for x in res], want[:4])
    with pytest.raises(ValueError):
        T.bbox.non_max_suppression(np.zeros((2, 500, 3, 4), F32), scores, **kw)
    # no classes: every row is padding, as for no boxes
    for bx0, sc0 in ((np.zeros((2, 500, 1, 4), F32), np.zeros((2, 500, 0), F32)),
                     (np.zeros((2, 0, 6, 4), F32), np.zeros((2, 0, 6), F32))):
        nb, ns, nc, nv, ni = T.bbox.non_max_suppression(bx0, sc0, return_indices=True, **kw)
        assert nb.shape == (2, 50, 4) and not nb.any() and not ns.any() and not nc.any()
        assert not nv.any() and np.all(ni == -1)


# ---- C ABI ---------------------------------------------------------------------------------------------------------
def test_callers_stream_and_determinism(T):
    rng = np.random.default_rng(21)
    boxes, scores = layout(rng, 4, 8732, 20, 1)
    cfg = cfg_of(T, 100, 200, 0.45, 0.05, False, True)
    want = oracle(boxes, scores, cfg)
    bx, sc = T.cu(boxes), T.cu(scores)
    s = T.torch.cuda.Stream(T.dev)
    s.wait_stream(T.torch.cuda.current_stream(T.dev))
    runs = []
    for _ in range(2):
        outs = outputs(T, 4, 200)
        s.wait_stream(T.torch.cuda.current_stream(T.dev))
        assert call(T, bx, sc, cfg, outs, stream=s.cuda_stream) == 0
        s.synchronize()
        runs.append([o.cpu().numpy() for o in outs])
    assert_same(runs[0], want)
    assert_same(runs[1], runs[0])


def test_graph_capture(T):
    t = T.torch
    rng = np.random.default_rng(4)
    B, K, Cn = 8, 3000, 10
    boxes, scores = layout(rng, B, K, Cn, Cn)
    cfg = cfg_of(T, 50, 100, 0.5, 0.1, True, True, 500)
    eager = native(T, boxes, scores, cfg)
    bx, sc = T.cu(boxes), T.cu(scores)
    handles = []
    try:
        for _ in range(2):
            h = T.L.P()
            assert T.lib.tfrpn_create(C.byref(h), T.dev.index) == 0
            handles.append(h)
        reserved, bare = handles
        assert T.lib.tfrpn_reserve_nms_multiclass(reserved, B, K, Cn, C.byref(cfg)) == 0
        assert T.lib.tfrpn_nms_multiclass_workspace_bytes(B, K, Cn, C.byref(cfg)) > 0
        outs = outputs(T, B, rows_of(cfg, Cn))
        g = t.cuda.CUDAGraph()
        with t.cuda.graph(g):
            rc = call(T, bx, sc, cfg, outs, h=reserved)
        assert rc == 0, T.lib.tfrpn_last_error()
        for o in outs:
            o.fill_(-7)
        g.replay()
        t.cuda.synchronize()
        assert_same([o.cpu().numpy() for o in outs], eager)
        g2 = t.cuda.CUDAGraph()
        with t.cuda.graph(g2):
            rc = call(T, bx, sc, cfg, outs, h=bare)
        assert rc == -4   # TFRPN_ERR_WORKSPACE: the workspace must grow while the stream is capturing
    finally:
        t.cuda.synchronize()
        for h in handles:
            T.lib.tfrpn_destroy(h)


def test_error_codes(T):
    t = T.torch
    B, K, Cn = 2, 64, 5
    bx = t.zeros((B, K, Cn, 4), device=T.dev)
    sc = t.zeros((B, K, Cn), device=T.dev)
    outs = outputs(T, B, 10)
    cfg = cfg_of(T, 5, 10)
    st = t.cuda.current_stream(T.dev).cuda_stream
    p = [o.data_ptr() for o in outs]
    f = T.lib.tfrpn_nms_multiclass
    assert f(T.h, bx.data_ptr(), 3, sc.data_ptr(), B, K, Cn, C.byref(cfg), *p, st) == -1     # q not in {1, C}
    assert f(T.h, bx.data_ptr(), 1, sc.data_ptr(), B, K, 0, C.byref(cfg), *p, st) == -1     # C = 0
    assert f(T.h, bx.data_ptr(), 1, sc.data_ptr(), 0, K, Cn, C.byref(cfg), *p, st) == -1    # B = 0
    assert f(T.h, bx.data_ptr(), 1, sc.data_ptr(), B, 0, Cn, C.byref(cfg), *p, st) == -1    # K = 0
    assert f(T.h, None, 1, sc.data_ptr(), B, K, Cn, C.byref(cfg), *p, st) == -1             # null boxes
    assert f(T.h, bx.data_ptr() + 4, Cn, sc.data_ptr(), B, K, Cn, C.byref(cfg), *p, st) == -2   # misaligned
    big = cfg_of(T, 100000, 100000)
    assert f(T.h, bx.data_ptr(), Cn, sc.data_ptr(), B, K, Cn, C.byref(big), *p, st) == -5   # like tfrpn_nms
    assert T.lib.tfrpn_reserve_nms_multiclass(T.h, B, K, 0, C.byref(cfg)) == -1
    t.cuda.synchronize()
    assert np.all(outs[3].cpu().numpy() == -7)   # nothing was launched

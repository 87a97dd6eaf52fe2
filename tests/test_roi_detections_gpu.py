"""tfrpn_roi_head_detections (roi_det_score_kernel -> the multi-class NMS's stage / proposal_kernel / merge) bit for
bit against oracle/roi_det_oracle.py fed the device's own probabilities and boxes from tfrpn_decode of the RoIs
repeated q times, at the C2 chain, the two-stage decoder and Detectron-like shapes, C from 2 to 1024, q = 1 and q = C,
with and without valid, min_size, the dh / dw clamp and pad_per_class, under both staging layouts.  Then the
probabilities input, the softmax bits against numpy and against tfrpn_roi_head_losses, the equivalence with
tfrpn_nms_multiclass on the materialised boxes, edge cases, run-to-run bits, handles, streams, graph capture, launch
counts, errors, the Python wrapper and a whole validation step captured in one CUDA graph.  Every output is prefilled
with a sentinel."""
import ctypes as C

import numpy as np
import pytest

from oracle import roi_det_oracle as D

pytestmark = pytest.mark.gpu
F32 = np.float32
INF = float("inf")
VAR = (0.1, 0.1, 0.2, 0.2)
SENT = -7.25


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    import tfrpn
    from tfrpn import _lib

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.tfrpn, ns.L, ns.lib, ns.dev = torch, tfrpn, _lib, _lib.load(), cuda_device
    ns.cu = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.h = _lib.handle(cuda_device.index or 0)
    return ns


def cfg_of(T, Cn, q, score_input=0, mls=INF, clip=True, min_size=0.0, per_class=100, total=100, iou=0.5, sthr=0.05,
           pad=False, topn=0, var=VAR):
    nms = T.L.NmsCfg(per_class, total, iou, sthr, int(pad), int(clip), topn)
    return T.L.RoiDetCfg(Cn, q, score_input, (C.c_float * 4)(*var), mls, int(clip), min_size, nms)


def rows_of(cfg):
    n = cfg.nms
    return min(n.max_total_size, n.max_output_size_per_class * (cfg.num_classes - 1)) if n.pad_per_class else n.max_total_size


def workload(rng, B, S, Cn, q, pad_rows=True):
    """proposal-like RoIs, valid with padding rows, trained-looking logits (most rows background, a confident class
    on the others) and box deltas ~ N(0, 1)"""
    ctr = rng.uniform(0.05, 0.95, size=(B, S, 2))
    sz = rng.uniform(0.02, 0.5, size=(B, S, 2))
    rois = np.concatenate([ctr - sz / 2, ctr + sz / 2], -1).astype(F32)
    valid = (S - rng.integers(0, S // 4 + 1, size=B)).astype(np.int32) if pad_rows else np.full(B, S, np.int32)
    x = rng.normal(0, 1, size=(B, S, Cn)).astype(F32)
    k = np.where(rng.uniform(size=(B, S)) < 0.6, 0, rng.integers(1, Cn, size=(B, S)))
    np.put_along_axis(x, k[..., None], np.take_along_axis(x, k[..., None], -1) + rng.uniform(1, 6, size=(B, S, 1)).astype(F32), -1)
    rois[np.arange(S)[None, :] >= valid[:, None]] = 0   # the proposals' padding rows
    d = rng.normal(0, 1, size=(B, S, q, 4)).astype(F32)
    return rois, valid, x, d


def outputs(T, B, rows):
    t = T.torch
    return (t.full((B, rows, 4), SENT, device=T.dev), t.full((B, rows), SENT, device=T.dev),
            t.full((B, rows), SENT, device=T.dev), t.full((B,), -7, dtype=t.int32, device=T.dev),
            t.full((B, rows), -7, dtype=t.int32, device=T.dev))


def call(T, r, v, x, d, cfg, outs, probs=None, h=None, stream=None, shape=None):
    p = lambda a: None if a is None else a.data_ptr()  # noqa: E731
    B, S = shape or (r.shape[0], r.shape[1])
    st = stream if stream is not None else T.torch.cuda.current_stream(T.dev).cuda_stream
    return T.lib.tfrpn_roi_head_detections(h or T.h, p(r), p(v), p(x), p(d), B, S, C.byref(cfg),
                                           *[o.data_ptr() for o in outs], p(probs), st)


def native(T, rois, valid, x, d, cfg, h=None, with_probs=True):
    """host arrays in -> ([boxes, scores, classes, valid, keep_idx], probs) host arrays"""
    B, S, Cn = x.shape
    outs = outputs(T, B, rows_of(cfg))
    pr = T.torch.full((B, S, Cn), SENT, device=T.dev) if with_probs and cfg.score_input == 0 else None
    rc = call(T, T.cu(rois), T.cu(valid), T.cu(x), T.cu(d), cfg, outs, pr, h=h)
    assert rc == 0, T.lib.tfrpn_last_error()
    return [o.cpu().numpy() for o in outs], (None if pr is None else pr.cpu().numpy())


def decoded(T, rois, d, cfg):
    """tfrpn_decode of the RoIs repeated q times; the deltas pre-scaled and pre-clamped in NumPy for a finite clamp"""
    B, S, q, _ = d.shape
    anchors = np.repeat(rois[:, :, None, :], q, axis=2).reshape(B, S * q, 4)
    var = np.asarray(cfg.variances[:], F32)
    if np.isinf(cfg.max_log_scale) and cfg.max_log_scale > 0:
        dd, vh = d, var
    else:
        dd, vh = D.scale_deltas(d, var, cfg.max_log_scale), None
    out = T.torch.full((B, S * q, 4), SENT, device=T.dev)
    vptr = None if vh is None else vh.ctypes.data_as(C.c_void_p)
    a_dev, d_dev = T.cu(anchors), T.cu(dd.reshape(B, S * q, 4))   # alive until the call has been enqueued
    rc = T.lib.tfrpn_decode(a_dev.data_ptr(), 1, d_dev.data_ptr(), vptr, int(cfg.clip), B, S * q, out.data_ptr(),
                            T.torch.cuda.current_stream(T.dev).cuda_stream)
    assert rc == 0, T.lib.tfrpn_last_error()
    return out.cpu().numpy().reshape(B, S, q, 4)


def oracle(T, rois, valid, probs, d, cfg):
    n = cfg.nms
    return D.roi_head_detections(rois, probs, d, valid, boxes=decoded(T, rois, d, cfg), min_size=cfg.min_size,
                                 max_output_size_per_class=n.max_output_size_per_class, max_total_size=n.max_total_size,
                                 iou_threshold=n.iou_threshold, score_threshold=n.score_threshold,
                                 pad_per_class=bool(n.pad_per_class), clip_boxes=bool(n.clip_boxes),
                                 pre_nms_topn=n.pre_nms_topn)


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == F32 else np.int32)


def assert_same(got, want):
    for g, w, name in zip(got, want, ("boxes", "scores", "classes", "valid", "keep_idx")):
        g, w = np.asarray(g), np.asarray(w).astype(np.asarray(g).dtype)
        assert g.shape == w.shape, (name, g.shape, w.shape)
        bad = np.argwhere(bits(g) != bits(w))
        assert bad.size == 0, "%s differ at %s: %s vs %s" % (name, bad[:5].tolist(), g[tuple(bad[:5].T)], w[tuple(bad[:5].T)])


def parity(T, rois, valid, x, d, cfg, h=None):
    got, probs = native(T, rois, valid, x, d, cfg, h=h)
    p = probs if cfg.score_input == 0 else x
    assert_same(got, oracle(T, rois, valid, p, d, cfg))
    return got, probs


# B, S, C, q, valid, min_size, max_log_scale, pad_per_class, pre_nms_topn
CASES = [
    (64, 300, 21, 21, True, 0.0, INF, False, 0),          # the C2 chain at inference
    (64, 300, 21, 1, True, 0.0, INF, False, 0),
    (16, 300, 21, 21, True, 0.01, 4.135, False, 0),       # the two-stage decoder
    (16, 300, 21, 1, False, 0.01, INF, True, 0),
    (16, 1000, 81, 81, True, 0.0, 4.135, False, 0),       # Detectron-like
    (16, 1000, 81, 1, True, 0.02, INF, True, 50),
    (3, 64, 2, 2, True, 0.0, INF, True, 0),
    (3, 64, 2, 1, False, 0.05, 0.5, False, 0),
    (4, 50, 3, 3, True, 0.0, 0.5, True, 0),
    (4, 50, 3, 1, True, 0.03, INF, False, 5),
    (2, 24, 1024, 1024, True, 0.01, 1.0, False, 0),
    (2, 24, 1024, 1, False, 0.0, INF, True, 0),
]


@pytest.mark.parametrize("B,S,Cn,q,use_valid,min_size,mls,pad,topn", CASES)
def test_chain_parity(T, B, S, Cn, q, use_valid, min_size, mls, pad, topn):
    rng = np.random.default_rng(B * 1000 + S + Cn * 7 + q)
    rois, valid, x, d = workload(rng, B, S, Cn, q, use_valid)
    cfg = cfg_of(T, Cn, q, mls=mls, min_size=min_size, pad=pad, topn=topn, per_class=100, total=100)
    got, _ = parity(T, rois, valid if use_valid else None, x, d, cfg)
    assert got[3].sum() > 0
    if use_valid:
        for b in range(B):
            assert np.all(got[4][b, :got[3][b]] < valid[b])
    assert np.all(got[2][got[2] != 0] >= 1)


@pytest.fixture(scope="module", params=["column", "rows"])
def stage_handle(T, request):
    """a handle with the NMS staging layout forced by TFRPN_NMS_MC_STAGE (read when the handle is created)"""
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


@pytest.mark.parametrize("B,S,Cn,q,use_valid,min_size,mls,pad,topn", [CASES[i] for i in (1, 2, 5, 6, 9, 10)])
def test_chain_parity_each_staging_layout(T, stage_handle, B, S, Cn, q, use_valid, min_size, mls, pad, topn):
    rng = np.random.default_rng(B * 1000 + S + Cn * 7 + q)
    rois, valid, x, d = workload(rng, B, S, Cn, q, use_valid)
    cfg = cfg_of(T, Cn, q, mls=mls, min_size=min_size, pad=pad, topn=topn)
    parity(T, rois, valid if use_valid else None, x, d, cfg, h=stage_handle)


@pytest.mark.parametrize("Cn,q", [(21, 21), (21, 1), (81, 1), (2, 2)])
def test_probabilities_input(T, Cn, q):
    rng = np.random.default_rng(Cn + q)
    rois, valid, x, d = workload(rng, 8, 300, Cn, q)
    p = D.softmax(x)
    p[0, 5] = np.nan                           # a NaN probability is never a candidate
    cfg = cfg_of(T, Cn, q, score_input=1, min_size=0.01)
    got, probs = parity(T, rois, valid, p, d, cfg)
    assert probs is None and got[3].sum() > 0


@pytest.mark.parametrize("Cn", [2, 3, 20, 21, 81, 1024])
def test_probs_close_to_numpy_softmax(T, Cn):
    rng = np.random.default_rng(Cn)
    rois, valid, x, d = workload(rng, 4, 64, Cn, 1)
    _, probs = native(T, rois, valid, x, d, cfg_of(T, Cn, 1))
    np.testing.assert_allclose(probs, D.softmax(x), rtol=4e-6, atol=1e-9)


@pytest.mark.parametrize("Cn,q", [(21, 21), (20, 1), (81, 81), (1024, 1), (3, 3)])
def test_probs_are_roi_head_losses_softmax_bits(T, Cn, q):
    """B*S a power of two, every label 0, grad_scale (B*S, 0): grad_logits[..., c >= 1] = p * 2^-k * 2^k = p exactly"""
    torch = T.torch
    rng = np.random.default_rng(Cn * 3 + q)
    B, S = 4, 64
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    x = np.clip(x, -8, 8)                      # no subnormal intermediate
    _, probs = native(T, rois, valid, x, d, cfg_of(T, Cn, q))
    gl = torch.full((B, S, Cn), SENT, device=T.dev)
    out = torch.empty((8,), device=T.dev)
    zeros4 = T.cu(np.zeros((B, S, 4), F32))
    xd, dd, lab, scale = T.cu(x), T.cu(d), T.cu(np.zeros((B, S), np.int32)), T.cu(np.array([B * S, 0], F32))
    rc = T.lib.tfrpn_roi_head_losses(T.h, xd.data_ptr(), dd.data_ptr(), lab.data_ptr(), zeros4.data_ptr(), B, S,
                                     C.byref(T.L.RoiLossCfg(Cn, q, 1.0, 0)), out.data_ptr(), scale.data_ptr(),
                                     gl.data_ptr(), None,
                                     torch.cuda.current_stream(T.dev).cuda_stream)
    assert rc == 0, T.lib.tfrpn_last_error()
    assert np.array_equal(bits(gl.cpu().numpy()[..., 1:]), bits(probs[..., 1:]))


def test_misaligned_logits_same_bits(T):
    """C % 4 == 0: float4 rows on an aligned tensor, scalar loads and stores 4 bytes off; the same bits"""
    torch = T.torch
    rng = np.random.default_rng(77)
    B, S, Cn, q = 8, 300, 20, 20
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    cfg = cfg_of(T, Cn, q, min_size=0.01)
    want, wprobs = native(T, rois, valid, x, d, cfg)
    buf = torch.full((B * S * Cn + 1,), SENT, device=T.dev)
    buf[1:] = T.cu(x).reshape(-1)
    pbuf = torch.full((B * S * Cn + 1,), SENT, device=T.dev)
    outs = outputs(T, B, rows_of(cfg))
    assert call(T, T.cu(rois), T.cu(valid), buf[1:], T.cu(d), cfg, outs, pbuf[1:], shape=(B, S)) == 0
    assert_same([o.cpu().numpy() for o in outs], want)
    assert np.array_equal(bits(pbuf[1:].cpu().numpy().reshape(B, S, Cn)), bits(wprobs))


def composition(T, rois, valid, d, cfg, probs):
    """what the call replaces: the boxes decoded for every (row, class), the masked scores, tfrpn_nms_multiclass"""
    B, S, Cn = probs.shape
    boxes = decoded(T, rois, d, cfg)
    cand = D.candidates(probs, boxes, valid, cfg.nms.score_threshold, cfg.min_size)
    scores = np.where(cand, probs, F32(-np.inf)).astype(F32)
    full = np.ascontiguousarray(np.broadcast_to(boxes, (B, S, Cn, 4)))
    outs = outputs(T, B, rows_of(cfg))
    full_dev, scores_dev = T.cu(full), T.cu(scores)
    rc = T.lib.tfrpn_nms_multiclass(T.h, full_dev.data_ptr(), Cn, scores_dev.data_ptr(), B, S, Cn,
                                    C.byref(cfg.nms), *[o.data_ptr() for o in outs],
                                    T.torch.cuda.current_stream(T.dev).cuda_stream)
    assert rc == 0, T.lib.tfrpn_last_error()
    return [o.cpu().numpy() for o in outs]


@pytest.mark.parametrize("q", [1, 21])
def test_equals_nms_multiclass_on_materialised_inputs(T, q):
    rng = np.random.default_rng(q)
    B, S, Cn = 16, 300, 21
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    cfg = cfg_of(T, Cn, q, min_size=0.01)
    got, probs = native(T, rois, valid, x, d, cfg)
    assert_same(got, composition(T, rois, valid, d, cfg, probs))


def test_edge_cases(T):
    rng = np.random.default_rng(5)
    B, S, Cn, q = 4, 100, 5, 5
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    cfg = cfg_of(T, Cn, q, total=30)
    # every image with valid = 0: padding only, probs still written for every row
    got, probs = native(T, rois, np.zeros(B, np.int32), x, d, cfg)
    assert np.all(got[3] == 0) and not got[0].any() and not got[1].any() and not got[2].any() and np.all(got[4] == -1)
    assert np.all(np.isfinite(probs)) and np.allclose(probs.sum(-1), 1, atol=1e-5)
    # every score below the threshold
    got, _ = native(T, rois, valid, x, d, cfg_of(T, Cn, q, sthr=0.9999999, total=30))
    assert np.all(got[3] == 0)
    # a NaN logit row: no detection from it, its probs NaN
    x2 = x.copy()
    x2[1, 3, 2] = np.nan
    got, probs = parity(T, rois, valid, x2, d, cfg)
    assert np.all(np.isnan(probs[1, 3])) and not np.any(got[4][1, :got[3][1]] == 3)
    # +-inf deltas with and without the clamp and the clip
    d2 = d.copy()
    d2[:, ::7, :, 2] = np.inf
    d2[:, 3::7, :, 3] = -np.inf
    d2[:, 5::11, :, 0] = np.inf
    for mls in (INF, 2.0):
        for clip in (True, False):
            for ms in (0.0, 0.01):
                cfg = cfg_of(T, Cn, q, mls=mls, clip=clip, min_size=ms, total=30)
                if clip or ms > 0:   # every box that reaches the NMS is finite
                    parity(T, rois, valid, x, d2, cfg)
                else:                # unclipped inf / NaN boxes reach the NMS: the same bits as the composition
                    got, probs = native(T, rois, valid, x, d2, cfg)
                    assert_same(got, composition(T, rois, valid, d2, cfg, probs))


def test_run_to_run_bits_handles_and_streams(T):
    torch = T.torch
    rng = np.random.default_rng(8)
    B, S, Cn, q = 16, 1000, 81, 81
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    cfg = cfg_of(T, Cn, q)
    want, wp = native(T, rois, valid, x, d, cfg)
    h2 = T.L.P()
    assert T.lib.tfrpn_create(C.byref(h2), T.dev.index) == 0
    try:
        assert_same(native(T, rois, valid, x, d, cfg, h=h2)[0], want)
        assert_same(native(T, rois, valid, x, d, cfg)[0], want)
        s = torch.cuda.Stream(T.dev)
        r, v, xx, dd = T.cu(rois), T.cu(valid), T.cu(x), T.cu(d)
        outs = outputs(T, B, rows_of(cfg))
        pr = torch.full((B, S, Cn), SENT, device=T.dev)
        s.wait_stream(torch.cuda.current_stream(T.dev))
        assert call(T, r, v, xx, dd, cfg, outs, pr, h=h2, stream=s.cuda_stream) == 0
        s.synchronize()
        assert_same([o.cpu().numpy() for o in outs], want)
        assert np.array_equal(bits(pr.cpu().numpy()), bits(wp))
    finally:
        torch.cuda.synchronize()
        T.lib.tfrpn_destroy(h2)


def test_graph_capture(T):
    torch = T.torch
    rng = np.random.default_rng(12)
    B, S, Cn, q = 16, 300, 21, 21
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    cfg = cfg_of(T, Cn, q, min_size=0.01, pad=True)
    r, v, xx, dd = T.cu(rois), T.cu(valid), T.cu(x), T.cu(d)
    handles = []
    try:
        for _ in range(2):
            h = T.L.P()
            assert T.lib.tfrpn_create(C.byref(h), T.dev.index) == 0
            handles.append(h)
        reserved, bare = handles
        assert T.lib.tfrpn_roi_head_detections_workspace_bytes(B, S, C.byref(cfg)) == \
            T.lib.tfrpn_nms_multiclass_workspace_bytes(B, S, Cn, C.byref(cfg.nms)) + \
            -(-B * S * Cn * 4 // 256) * 256 + -(-B * S * q * 16 // 256) * 256
        assert T.lib.tfrpn_reserve_roi_head_detections(reserved, B, S, C.byref(cfg)) == 0
        x2 = x.copy()
        x2[:, :, 0] += 1.0
        want = [native(T, rois, valid, a, d, cfg, h=reserved) for a in (x, x2)]
        outs = outputs(T, B, rows_of(cfg))
        pr = torch.full((B, S, Cn), SENT, device=T.dev)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            rc = call(T, r, v, xx, dd, cfg, outs, pr, h=reserved)
        assert rc == 0, T.lib.tfrpn_last_error()
        for a, (w, wp) in zip((x, x2), want):
            xx.copy_(T.cu(a))
            for o in outs:
                o.fill_(-7)
            g.replay()
            torch.cuda.synchronize()
            assert_same([o.cpu().numpy() for o in outs], w)
            assert np.array_equal(bits(pr.cpu().numpy()), bits(wp))
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2):
            rc = call(T, r, v, xx, dd, cfg, outs, pr, h=bare)
        assert rc == -4   # TFRPN_ERR_WORKSPACE: it would have to grow while the stream is capturing
    finally:
        torch.cuda.synchronize()
        for h in handles:
            T.lib.tfrpn_destroy(h)


def test_launch_counts(T, stage_handle):
    """one score kernel in front of exactly the launches tfrpn_nms_multiclass makes on the staged shapes"""
    rng = np.random.default_rng(2)
    for B, S, Cn, q in ((2, 100, 5, 5), (16, 1000, 81, 1)):
        rois, valid, x, d = workload(rng, B, S, Cn, q)
        cfg = cfg_of(T, Cn, q)
        native(T, rois, valid, x, d, cfg, h=stage_handle)
        n0 = T.L.launch_count()
        native(T, rois, valid, x, d, cfg, h=stage_handle)
        n_det = T.L.launch_count() - n0
        bx = T.cu(np.zeros((B, S, q, 4), F32))
        sc = T.cu(np.zeros((B, S, Cn), F32))
        outs = outputs(T, B, rows_of(cfg))
        st = T.torch.cuda.current_stream(T.dev).cuda_stream
        n0 = T.L.launch_count()
        assert T.lib.tfrpn_nms_multiclass(stage_handle, bx.data_ptr(), q, sc.data_ptr(), B, S, Cn, C.byref(cfg.nms),
                                          *[o.data_ptr() for o in outs], st) == 0
        n_mc = T.L.launch_count() - n0
        assert n_mc in (3, 4) and n_det == n_mc + 1


def test_errors_and_limits(T):
    torch = T.torch
    B, S, Cn, q = 2, 16, 5, 5
    r = torch.zeros((B, S, 4), device=T.dev)
    x = torch.zeros((B, S, Cn), device=T.dev)
    d = torch.zeros((B, S, q, 4), device=T.dev)
    pr = torch.zeros((B, S, Cn), device=T.dev)
    outs = outputs(T, B, 100)
    f = lambda cfg, **kw: call(T, kw.get("r", r), None, kw.get("x", x), kw.get("d", d), cfg,  # noqa: E731
                               kw.get("outs", outs), kw.get("pr"), shape=kw.get("shape", (B, S)))
    ok = cfg_of(T, Cn, q)
    assert f(ok) == 0
    torch.cuda.synchronize()
    outs[3].fill_(-7)
    st = torch.cuda.current_stream(T.dev).cuda_stream
    p = [o.data_ptr() for o in outs]
    L = T.lib.tfrpn_roi_head_detections
    assert L(None, r.data_ptr(), None, x.data_ptr(), d.data_ptr(), B, S, C.byref(ok), *p, None, st) == -1
    assert L(T.h, None, None, x.data_ptr(), d.data_ptr(), B, S, C.byref(ok), *p, None, st) == -1
    assert L(T.h, r.data_ptr(), None, None, d.data_ptr(), B, S, C.byref(ok), *p, None, st) == -1
    assert L(T.h, r.data_ptr(), None, x.data_ptr(), None, B, S, C.byref(ok), *p, None, st) == -1
    assert L(T.h, r.data_ptr(), None, x.data_ptr(), d.data_ptr(), B, S, None, *p, None, st) == -1
    assert L(T.h, r.data_ptr(), None, x.data_ptr(), d.data_ptr(), B, S, C.byref(ok), p[0], p[1], p[2], None, p[4],
             None, st) == -1                                                       # null valid output
    assert f(ok, shape=(0, S)) == -1 and f(ok, shape=(B, 0)) == -1
    assert f(cfg_of(T, 1, 1)) == -1                                               # C < 2
    assert f(cfg_of(T, Cn, 3)) == -1                                              # q not in {1, C}
    assert f(cfg_of(T, Cn, q, var=(0.1, INF, 0.2, 0.2))) == -1
    assert f(cfg_of(T, Cn, q, var=(0.1, 0.1, float("nan"), 0.2))) == -1
    assert f(cfg_of(T, Cn, q, mls=float("nan"))) == -1
    assert f(cfg_of(T, Cn, q, score_input=2)) == -1
    assert f(cfg_of(T, Cn, q, score_input=1), pr=pr) == -1                        # probs with probabilities input
    assert f(cfg_of(T, Cn, q, per_class=0)) == -1 and f(cfg_of(T, Cn, q, total=0)) == -1
    assert f(cfg_of(T, Cn, q, topn=-1)) == -1                                     # as tfrpn_nms_multiclass
    assert f(cfg_of(T, 1025, 1), shape=(B, S)) == -5                              # C > 1024
    assert f(ok, shape=(B, 8193)) == -5 and f(ok, shape=(65536, S)) == -5
    assert f(cfg_of(T, Cn, q, per_class=100000, total=100000)) == -5              # beyond the NMS kernel's smem
    assert f(ok, r=r.view(-1)[1:]) == -2 and f(ok, d=d.view(-1)[1:]) == -2
    assert f(ok, outs=(outs[0].view(-1)[2:],) + outs[1:]) == -2
    xb = x.view(torch.uint8).view(-1)[1:]
    assert L(T.h, r.data_ptr(), None, xb.data_ptr(), d.data_ptr(), B, S, C.byref(ok), *p, None, st) == -2
    assert L(T.h, r.data_ptr(), None, x.data_ptr(), d.data_ptr(), B, S, C.byref(ok), *p, pr.data_ptr() + 2, st) == -2
    assert T.lib.tfrpn_reserve_roi_head_detections(T.h, B, S, C.byref(cfg_of(T, Cn, 3))) == -1
    assert T.lib.tfrpn_reserve_roi_head_detections(T.h, B, 9000, C.byref(ok)) == -5
    assert T.lib.tfrpn_roi_head_detections_workspace_bytes(B, S, None) == 0
    torch.cuda.synchronize()
    assert np.all(outs[3].cpu().numpy() == -7)   # nothing was launched


def test_python_wrapper(T):
    torch = T.torch
    rng = np.random.default_rng(31)
    B, S, Cn = 4, 300, 21
    rois, valid, x, d = workload(rng, B, S, Cn, Cn)
    kw = dict(max_output_size_per_class=50, max_total_size=80, score_threshold=0.05, min_size=0.01,
              max_log_scale=3.0, pad_per_class=True)
    cfg = cfg_of(T, Cn, Cn, mls=3.0, min_size=0.01, per_class=50, total=80, pad=True)
    want, wp = native(T, rois, valid, x, d, cfg)
    for layout in (d, d.reshape(B, S, Cn * 4)):
        got = T.tfrpn.roi_head_detections(rois, x, layout, valid, return_indices=True, return_probs=True, **kw)
        assert len(got) == 6 and all(isinstance(a, np.ndarray) for a in got)
        assert_same(got[:5], want)
        assert np.array_equal(bits(got[5]), bits(wp))
    res = T.tfrpn.roi_head_detections(T.cu(rois), T.cu(x), T.cu(d), T.cu(valid), **kw)
    assert len(res) == 4 and all(isinstance(a, torch.Tensor) and a.is_cuda for a in res)
    assert_same([a.cpu().numpy() for a in res], want[:4])
    d1 = d[:, :, :1]
    cfg1 = cfg_of(T, Cn, 1, mls=3.0, min_size=0.01, per_class=50, total=80, pad=True)
    want1, _ = native(T, rois, valid, x, d1, cfg1)
    for layout in (d1, d1.reshape(B, S, 4)):
        res = T.tfrpn.roi_head_detections(T.cu(rois), T.cu(x), T.cu(layout), T.cu(valid), return_indices=True, **kw)
        assert_same([a.cpu().numpy() for a in res], want1)
    p = D.softmax(x)
    cfgp = cfg_of(T, Cn, Cn, score_input=1, mls=3.0, min_size=0.01, per_class=50, total=80, pad=True)
    assert_same(T.tfrpn.roi_head_detections(rois, p, d, valid, scores="probs", return_indices=True, **kw),
                native(T, rois, valid, p, d, cfgp)[0])
    nb, ns, nc, nv, ni = T.tfrpn.roi_head_detections(np.zeros((0, S, 4), F32), np.zeros((0, S, Cn), F32),
                                                     np.zeros((0, S, Cn, 4), F32), return_indices=True)
    assert nb.shape == (0, 100, 4) and nv.shape == (0,)
    nb, ns, nc, nv, ni = T.tfrpn.roi_head_detections(np.zeros((2, 0, 4), F32), np.zeros((2, 0, Cn), F32),
                                                     np.zeros((2, 0, Cn, 4), F32), return_indices=True)
    assert nb.shape == (2, 100, 4) and not nb.any() and not nv.any() and np.all(ni == -1)
    with pytest.raises(ValueError):
        T.tfrpn.roi_head_detections(rois, x, d[:, :, :3], valid)
    with pytest.raises(ValueError):
        T.tfrpn.roi_head_detections(rois, x, d, valid, scores="probs", return_probs=True)
    with pytest.raises(NotImplementedError):
        T.tfrpn.roi_head_detections(rois[:, :1], np.zeros((B, 1, 1025), F32), np.zeros((B, 1, 4), F32))


def test_validation_step_in_one_graph(T):
    """generate_proposals -> crop_and_resize -> a fixed linear head -> roi_head_detections -> DetectionMAP.update, one
    CUDA graph replayed over three batches: the AP equals eager calls' and oracle/map_oracle.py's on the same
    detections"""
    torch = T.torch
    from oracle import map_oracle as M
    from oracle import rpn_oracle as O
    from tfrpn import synthetic
    from tfrpn.utils import data_utils
    rng = np.random.default_rng(40)
    hp = O.get_hyper_params("vgg16")
    B, G, Cn, Fc = 4, 20, 21, 16
    fh, fw = O._pair(hp["feature_map_shape"])
    anchors = T.cu(O.generate_anchors(hp))
    torch.manual_seed(0)
    head = torch.nn.Linear(7 * 7 * Fc, Cn * 5).to(T.dev)
    batches = []
    for _ in range(3):
        reg, cls = synthetic.head_outputs(rng, B, fh, fw, hp["anchor_count"])
        gtb, gtl = synthetic.gt_batch(rng, B, G)
        n = (gtl >= 0).sum(axis=1)
        gb, gl = data_utils.pad_gt_batch([gtb[b, :n[b]] for b in range(B)], [gtl[b, :n[b]] % (Cn - 1) for b in range(B)],
                                         max_boxes=G, label_add=1)
        feats = rng.normal(size=(B, fh, fw, Fc)).astype(F32)
        gb, gl = [a.to(T.dev) if isinstance(a, torch.Tensor) else T.cu(a) for a in (gb, gl)]
        batches.append([T.cu(reg), T.cu(cls), gb.float(), gl.to(torch.int32), T.cu(feats)])
    inp = [torch.empty_like(t) for t in batches[0]]

    def step(meter):
        reg, cls, gb, gl, feats = inp
        rois, _, valid, _ = T.tfrpn.generate_proposals(reg, cls, anchors, hp)
        pooled = T.tfrpn.crop_and_resize(feats, rois, None, (7, 7))
        y = head(pooled.reshape(B, rois.shape[1], -1))
        dets = T.tfrpn.roi_head_detections(rois, y[..., :Cn].contiguous(), y[..., Cn:].contiguous(), valid,
                                           score_threshold=0.02)
        meter.update(*dets, gb, gl)
        return dets

    with torch.no_grad():
        eager = T.tfrpn.DetectionMAP(Cn, device=T.dev)
        host_dets = []
        for bt in batches:
            for a, b in zip(inp, bt):
                a.copy_(b)
            host_dets.append([t.cpu().numpy() for t in step(eager)])
        want = eager.compute()
        graphed = T.tfrpn.DetectionMAP(Cn, device=T.dev)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream(T.dev)
        s.wait_stream(torch.cuda.current_stream(T.dev))
        with torch.cuda.stream(s):
            for a, b in zip(inp, batches[0]):   # a warm-up on the capture stream
                a.copy_(b)
            step(T.tfrpn.DetectionMAP(Cn, device=T.dev))
        torch.cuda.current_stream(T.dev).wait_stream(s)
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            gdets = step(graphed)
        for i, bt in enumerate(batches):
            for a, b in zip(inp, bt):
                a.copy_(b)
            g.replay()
            torch.cuda.synchronize()
            assert_same([t.cpu().numpy() for t in gdets], host_dets[i])
        got = graphed.compute()
    assert sum(int(h[3].sum()) for h in host_dets) > 0
    assert np.array_equal(got.ap.numpy().view(np.uint64), want.ap.numpy().view(np.uint64))
    cat = [np.concatenate([h[i] for h in host_dets]) for i in range(4)]
    gts = [np.concatenate([bt[i].cpu().numpy() for bt in batches]) for i in (2, 3)]
    ap, rec, n_gt, m, mean_ap = M.detection_map(*cat, *gts, None, num_classes=Cn, protocol="coco")
    assert np.array_equal(want.ap.numpy().view(np.uint64), ap.view(np.uint64))

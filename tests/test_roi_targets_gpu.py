"""tfrpn_roi_targets (roi_target_kernel) against oracle/roi_oracle.py: rois, labels, src, counts and argmax exact,
max_iou bit-exact, deltas dy/dx bit-exact and dh/dw within 4 ulp (the RPN targets' bar), at this library's own chain
(generate_proposals -> pad_gt_batch), at Detectron-like shapes, on the CPU hand cases, tie-heavy, pixel, NaN/inf and
flipped layouts, and at the limits.  Then the properties: sharding, determinism, graph replay, streams, errors."""
import ctypes as C

import numpy as np
import pytest

from oracle import roi_oracle as R
from oracle import rpn_oracle as O
from oracle import target_layouts as L

pytestmark = pytest.mark.gpu
F32 = np.float32
NAN, INF = float("nan"), float("inf")
SENT_F, SENT_I = F32(-7.25), -77


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    import tfrpn

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.tfrpn, ns.dev = torch, tfrpn, cuda_device
    ns.cu = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    return ns


def launch(T, rois, gt, labels, valid=None, stream=None, **kw):
    """Direct C call with every output prefilled with a sentinel -> dict of host arrays."""
    torch = T.torch
    from tfrpn import _lib, roi_target_cfg
    cfg = roi_target_cfg(**kw)
    r, g, l = T.cu(np.asarray(rois, F32)), T.cu(np.asarray(gt, F32)), T.cu(np.asarray(labels, np.int32))
    v = T.cu(None if valid is None else np.asarray(valid, np.int32))
    B, P, G = r.shape[0], r.shape[1], g.shape[1]
    S = cfg.total_pos + cfg.total_neg
    Pp = P + (G if cfg.append_gt else 0)
    f = lambda *s: torch.full(s, float(SENT_F), dtype=torch.float32, device=T.dev)   # noqa: E731
    i = lambda *s: torch.full(s, SENT_I, dtype=torch.int32, device=T.dev)             # noqa: E731
    out = dict(rois=f(B, S, 4), labels=i(B, S), deltas=f(B, S, 4), src=i(B, S), counts=i(B, 2), max_iou=f(B, Pp),
               argmax=i(B, Pp))
    st = (stream or torch.cuda.current_stream(T.dev)).cuda_stream
    _lib.check(_lib.load().tfrpn_roi_targets(
        _lib.handle(T.dev.index or 0), r.data_ptr(), None if v is None else v.data_ptr(), g.data_ptr(), l.data_ptr(),
        B, P, G, C.byref(cfg), *(out[k].data_ptr() for k in ("rois", "labels", "deltas", "src", "counts", "max_iou",
                                                             "argmax")), st))
    (stream or torch.cuda.current_stream(T.dev)).synchronize()
    return {k: t.cpu().numpy() for k, t in out.items()}


def ulp_diff(a, b):
    ia = a.view(np.int32).astype(np.int64)
    ib = b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


def check(T, rois, gt, labels, valid=None, **kw):
    kw.setdefault("num_classes", 21)
    kw.setdefault("offset", 17)
    got = launch(T, rois, gt, labels, valid, **kw)
    want = R.roi_targets(np.asarray(rois, F32), np.asarray(gt, F32), np.asarray(labels, np.int32), valid, **kw)
    for k in ("labels", "src", "counts", "argmax"):
        assert np.array_equal(got[k], want[k]), (k, np.argwhere(got[k] != want[k])[:8])
    for k in ("rois", "max_iou"):
        bad = np.argwhere(got[k].view(np.uint32) != want[k].view(np.uint32))
        assert bad.size == 0, (k, bad[:8])
    gd, wd = got["deltas"], want["deltas"]
    nan_g, nan_w = np.isnan(gd), np.isnan(wd)
    assert np.array_equal(nan_g, nan_w), "deltas NaN"           # NaN payloads are not compared
    same = (gd.view(np.uint32) == wd.view(np.uint32)) | nan_g
    assert same[..., :2].all(), ("dy/dx", np.argwhere(~same[..., :2])[:8])
    fin = ~nan_g[..., 2:]
    assert (ulp_diff(gd[..., 2:][fin], wd[..., 2:][fin]) <= 4).all(), "dh/dw"
    return got, want


def chain_inputs(T, rng, B, G, hp):
    """generate_proposals output of the C2 shapes and pad_gt_batch(label_add=1) ground truth"""
    from tfrpn import synthetic
    from tfrpn.utils import data_utils
    fh, fw = O._pair(hp["feature_map_shape"])
    reg, cls = synthetic.head_outputs(rng, B, fh, fw, hp["anchor_count"])
    boxes, _, valid, _ = T.tfrpn.generate_proposals(T.cu(reg), T.cu(cls), T.cu(O.generate_anchors(hp)), hp)
    gtb, gtl = synthetic.gt_batch(rng, B, G)
    n = (gtl >= 0).sum(axis=1)
    gb, gl = data_utils.pad_gt_batch([gtb[b, :n[b]] for b in range(B)], [gtl[b, :n[b]] - 1 for b in range(B)],
                                     max_boxes=G, label_add=1)
    return boxes.cpu().numpy(), valid.cpu().numpy(), gb.cpu().numpy(), gl.cpu().numpy()


@pytest.mark.parametrize("append_gt", [True, False])
def test_c2_chain(T, append_gt):
    rng = np.random.default_rng(40)
    prop, valid, gt, lab = chain_inputs(T, rng, 64, 50, O.get_hyper_params("vgg16"))
    got, _ = check(T, prop, gt, lab, valid, num_classes=21, total_pos=32, total_neg=96, append_gt=append_gt)
    assert got["counts"][:, 0].sum() > 0


def detectron_like(rng, B, P, G):
    gt = np.zeros((B, G, 4), F32)
    lab = np.full((B, G), -1, np.int32)
    rois = np.zeros((B, P, 4), F32)
    for b in range(B):
        n = int(rng.integers(G // 2, G + 1))
        gt[b, :n] = R_boxes(rng, n, 0.05, 0.4)
        lab[b, :n] = rng.integers(1, 81, size=n)
        near = gt[b, rng.integers(0, n, size=P // 4)] + rng.normal(0, 0.03, size=(P // 4, 4)).astype(F32)
        rois[b] = np.concatenate([np.clip(near, 0, 1), R_boxes(rng, P - P // 4, 0.02, 0.5)]).astype(F32)
    return rois, gt, lab


def R_boxes(rng, n, lo, hi):
    c = rng.uniform(0, 1, size=(n, 2))
    s = rng.uniform(lo, hi, size=(n, 2))
    return np.clip(np.concatenate([c - s / 2, c + s / 2], axis=1), 0, 1).astype(F32)


@pytest.mark.parametrize("B", [2, 16])
@pytest.mark.parametrize("append_gt", [True, False])
def test_detectron_like(T, B, append_gt):
    rng = np.random.default_rng(41 + B)
    rois, gt, lab = detectron_like(rng, B, 2000, 100)
    valid = rng.integers(1500, 2001, size=B).astype(np.int32)
    got, _ = check(T, rois, gt, lab, valid, num_classes=81, total_pos=128, total_neg=384, append_gt=append_gt)
    assert (got["counts"][:, 1] == 512).all() and (got["counts"][:, 0] > 0).all()


HAND = [
    # (rois, gt, labels, valid, kw): the rules of the CPU hand cases
    ([[[0, 0, 1, w] for w in (1.0, 0.75, 0.5, 0.25, 0.125)]], [[[0, 0, 1, 1]]], [[3]], None,
     dict(append_gt=False, fg_iou_threshold=0.75, bg_iou_high=0.5, bg_iou_low=0.25, total_pos=8, total_neg=8)),
    ([[[0, 0, 1, 1]]], [[[0, 0.5, 1, 1], [0, 0, 1, 1], [0, 0, 1, 1]]], [[1, 3, 2]], None, dict(total_pos=4, total_neg=4)),
    ([[[0, 0, 1, 1], [0, 0, 1, 0.5]]] * 4, [[[0, 0, 1, 1], [0, 0, 1, 1]]] * 4, [[-1, 2], [0, 2], [21, 2], [26, 2]], None,
     dict(total_pos=4, total_neg=4)),
    ([[[0, 0, 1, 1], [0, 0, 1, 0.75], [0, 0, 1, 0.125], [0, 0, 0.5, 0.5]]] * 4, [[[0, 0, 1, 1]]] * 4, [[1]] * 4,
     [-3, 0, 4, 9], dict(total_pos=8, total_neg=8)),
    ([[[0.75, 0.75, 1, 1]] * 6], [[[0, 0, 0.5, 0.5], [0, 0, 0.25, 0.5], [0, 0, 0, 0]]], [[1, 2, -1]], None,
     dict(total_pos=4, total_neg=12)),
    ([[[NAN, 0, 1, 1], [1, 1, 0, 0], [0.5, 0, 0.5, 1], [0, 0, 1, 0.5]]],
     [[[0, 0, 1, 1], [0.5, 0.5, 0.5, 0.5], [1, 0, 0, 1], [0, NAN, 1, 1]]], [[1, 2, 3, 4]], None,
     dict(total_pos=8, total_neg=8)),
    ([[[0.1, 0.1, 0.3, 0.4]] * 7], [[[0, 0, 1, 1], [0, 0, 1, 1]]], [[0, -1]], None, dict(total_pos=2, total_neg=14)),
    ([[[0, 0, 1, 1]] * 9 + [[0, 0, 1, 0.25]] * 30], [[[0, 0, 1, 1]]], [[1]], None,
     dict(append_gt=False, total_pos=4, total_neg=12)),
    ([[[0, 0, 1, 1]] * 3 + [[0, 0, 1, 0.25]] * 5], [[[0, 0, 1, 1]]], [[1]], None,
     dict(append_gt=False, total_pos=4, total_neg=12)),
    ([[[0, 0, 1, 1]] * 6 + [[0, 0, 1, 0.25]] * 20], [[[0, 0, 1, 1]]], [[1]], None,
     dict(append_gt=False, total_pos=0, total_neg=8)),
    ([[[0, 0, 1, 1]] * 6 + [[0, 0, 1, 0.25]] * 20], [[[0, 0, 1, 1]]], [[1]], None,
     dict(append_gt=False, total_pos=4, total_neg=0)),
]


@pytest.mark.parametrize("case", range(len(HAND)))
def test_hand_cases(T, case):
    rois, gt, lab, valid, kw = HAND[case]
    check(T, rois, gt, lab, valid, num_classes=21, **kw)


def test_tie_heavy_dyadic(T):
    rng = np.random.default_rng(42)
    B, P, G = 6, 1500, 40
    rois = np.stack([L.dyadic_boxes(rng, P, ext=(2, 12)) for _ in range(B)])
    gt = np.stack([L.dyadic_boxes(rng, G, ext=(2, 12)) for _ in range(B)])
    gt[:, 1::3] = gt[:, ::3][:, :gt[:, 1::3].shape[1]]          # duplicate GT boxes
    lab = rng.integers(-1, 8, size=(B, G)).astype(np.int32)
    for tp, tn in ((64, 192), (8, 24)):
        check(T, rois, gt, lab, num_classes=6, total_pos=tp, total_neg=tn, fg_iou_threshold=0.25, bg_iou_high=0.25,
              bg_iou_low=0.0625)


@pytest.mark.parametrize("name", ["pixel", "nan_inf", "flip_one_axis", "flip_both_axes", "tiny"])
def test_exact_path_layouts(T, name):
    anchors, gt, lab = L.fallback_layout(name, seed=3, N=900, B=3, G=12)
    rois = np.stack([np.roll(anchors, 37 * b, axis=0) for b in range(3)])
    rois[1, :5] = gt[1, :5]
    lab = np.where(lab >= 0, lab % 20 + 1, lab).astype(np.int32)
    for append_gt in (True, False):
        check(T, rois, gt, lab, num_classes=21, total_pos=32, total_neg=96, append_gt=append_gt, bg_iou_low=0.0,
              fg_iou_threshold=0.5)


def test_limits(T):
    """P = 8192, G = 1024 and S = 8192: P' = 9216 rows, the largest shared-memory plan"""
    rng = np.random.default_rng(43)
    rois, gt, lab = detectron_like(rng, 2, 8192, 1024)
    check(T, rois, gt, lab, num_classes=81, total_pos=2048, total_neg=6144, append_gt=True)
    check(T, rois, gt, lab, np.asarray([8000, 9000], np.int32), num_classes=81, total_pos=100, total_neg=8092)
    torch = T.torch
    z = lambda *s: torch.zeros(s, device=T.dev)   # noqa: E731
    zl = lambda *s: torch.ones(s, dtype=torch.int32, device=T.dev)   # noqa: E731
    with pytest.raises(NotImplementedError):
        T.tfrpn.roi_targets(z(1, 8193, 4), z(1, 4, 4), zl(1, 4), num_classes=3)
    with pytest.raises(NotImplementedError):
        T.tfrpn.roi_targets(z(1, 16, 4), z(1, 1025, 4), zl(1, 1025), num_classes=3)
    with pytest.raises(NotImplementedError):
        T.tfrpn.roi_targets(z(1, 16, 4), z(1, 4, 4), zl(1, 4), num_classes=3, total_pos=1, total_neg=8192)


def test_shards_equal_one_call_and_runs_repeat(T):
    torch = T.torch
    rng = np.random.default_rng(44)
    rois, gt, lab = detectron_like(rng, 8, 1000, 40)
    r, g, l = T.cu(rois), T.cu(gt), T.cu(lab)
    kw = dict(num_classes=81, total_pos=64, total_neg=192, seed=5, offset=9)
    whole = T.tfrpn.roi_targets(r, g, l, **kw)
    again = T.tfrpn.roi_targets(r, g, l, **kw)
    parts = [T.tfrpn.roi_targets(r[s], g[s], l[s], image_offset=s.start, **kw) for s in (slice(0, 3), slice(3, 8))]
    for k in range(5):
        a = whole[k].view(torch.int32) if whole[k].dtype == torch.float32 else whole[k]
        b = again[k].view(torch.int32) if again[k].dtype == torch.float32 else again[k]
        assert torch.equal(a, b)
        cat = torch.cat([p[k] for p in parts])
        cat = cat.view(torch.int32) if cat.dtype == torch.float32 else cat
        assert torch.equal(cat, a)
    other = T.tfrpn.roi_targets(r, g, l, **dict(kw, offset=10))
    assert not torch.equal(other.src_index, whole.src_index)


def test_graph_replay_and_stream(T):
    torch = T.torch
    rng = np.random.default_rng(45)
    rois, gt, lab = detectron_like(rng, 4, 1200, 30)
    r, g, l = T.cu(rois), T.cu(gt), T.cu(lab)
    kw = dict(num_classes=81, total_pos=32, total_neg=96, seed=2, offset=3)
    eager, dbg = T.tfrpn.roi_targets(r, g, l, return_debug=True, **kw)
    s = torch.cuda.Stream(T.dev)
    s.wait_stream(torch.cuda.current_stream(T.dev))
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        on_s = T.tfrpn.roi_targets(r, g, l, **kw)
    s.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cap = T.tfrpn.roi_targets(r, g, l, **kw)
    for t in cap:
        t.fill_(-5)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize(T.dev)
    for a, b, c in zip(eager, on_s, cap):
        assert torch.equal(a, b) and torch.equal(a, c)
    want = R.roi_targets(rois, gt, lab, **kw)
    assert np.array_equal(dbg["argmax"].cpu().numpy(), want["argmax"])
    res = T.tfrpn.roi_targets(rois, gt, lab, **kw)       # NumPy in, NumPy out
    assert isinstance(res.rois, np.ndarray) and np.array_equal(res.src_index, want["src"])


def test_errors(T):
    torch = T.torch
    from tfrpn import _lib, roi_target_cfg
    lib = _lib.load()
    h = _lib.handle(T.dev.index or 0)
    st = torch.cuda.current_stream(T.dev).cuda_stream
    B, P, G, S = 1, 16, 4, 8
    rois = torch.zeros((B, P + 1, 4), device=T.dev)
    gt = torch.zeros((B, G, 4), device=T.dev)
    lab = torch.ones((B, G), dtype=torch.int32, device=T.dev)
    o4 = torch.zeros((B, S + 1, 4), device=T.dev)
    oi = torch.zeros((B, S), dtype=torch.int32, device=T.dev)
    cnt = torch.zeros((B, 2), dtype=torch.int32, device=T.dev)
    d4 = torch.zeros((B, S, 4), device=T.dev)

    def call(cfg, r=rois.data_ptr(), g=gt.data_ptr(), orr=o4.data_ptr(), od=d4.data_ptr(), c=cnt.data_ptr(), l=lab.data_ptr()):
        return lib.tfrpn_roi_targets(h, r, None, g, l, B, P, G, C.byref(cfg), orr, oi.data_ptr(), od, None, c,
                                     None, None, st)
    good = roi_target_cfg(5, total_pos=2, total_neg=6, offset=0)
    assert call(good) == 0
    assert call(good, r=None) == -1 and call(good, c=None) == -1 and call(good, l=None) == -1
    assert call(good, r=rois.data_ptr() + 4) == -2 and call(good, orr=o4.data_ptr() + 4) == -2
    assert call(good, od=d4.data_ptr() + 8) == -2 and call(good, g=gt.data_ptr() + 4) == -2
    for kw in (dict(num_classes=1), dict(total_pos=-1), dict(total_pos=0, total_neg=0), dict(fg_iou_threshold=0.0),
               dict(fg_iou_threshold=1.5), dict(fg_iou_threshold=NAN), dict(bg_iou_low=-0.1), dict(bg_iou_high=NAN),
               dict(bg_iou_low=0.6, bg_iou_high=0.5), dict(bg_iou_high=1.5)):
        a = dict(num_classes=5, total_pos=2, total_neg=6, offset=0)
        a.update(kw)
        assert call(roi_target_cfg(**a)) == -1, kw
    host = np.zeros((B, G, 4), F32)
    assert call(good, g=host.ctypes.data) == -1                 # not a device pointer
    with pytest.raises(ValueError):
        T.tfrpn.roi_targets(rois, gt, lab[:, :3], num_classes=5)
    with pytest.raises(ValueError):
        T.tfrpn.roi_targets(rois, gt, lab, num_classes=5, bg_iou_low=0.7)

"""tfrpn_map_update / tfrpn_map_compute (map_match_kernel, the radix sort, map_ap_kernel) against the NumPy
restatement of oracle/map_oracle.py: ap and recall bit-equal and n_gt exactly equal, under all three protocols, on
multi-class NMS output at the SSD-VOC and decoder shapes, on unsorted rows with tie groups across warp and sort-tile
boundaries, crowd / difficult flags, invalid class values and valid counts outside [0, R], the edge shapes, more than
2^20 records in one tie group, and through the running meter: accumulation, CUDA-graph capture, the caller's stream,
overflow, determinism and the raw C ABI with sentinel-filled outputs."""
import ctypes as C

import numpy as np
import pytest

from oracle import map_oracle as M

pytestmark = pytest.mark.gpu
F32 = np.float32
PROTOCOLS = M.PROTOCOLS


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


def same_bits(a, b):
    a = np.ascontiguousarray(a, np.float64)
    b = np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def check(T, inputs, num_classes, protocol, thresholds=None, max_dets=100):
    """tfrpn.detection_map on device tensors against the oracle; returns the result."""
    db, ds, dc, val, gb, gl, gf = inputs
    r = T.tfrpn.detection_map(*[T.cu(x) for x in inputs], num_classes=num_classes, protocol=protocol,
                              iou_thresholds=thresholds, max_dets=max_dets)
    ap, rec, n_gt, m, mean_ap = M.detection_map(db, ds, dc, val, gb, gl, gf, num_classes=num_classes,
                                                protocol=protocol, thresholds=thresholds, max_dets=max_dets)
    assert np.array_equal(r.n_gt.numpy(), n_gt), protocol
    bad = np.argwhere(r.ap.numpy().view(np.uint64) != ap.view(np.uint64))
    assert same_bits(r.ap.numpy(), ap), (protocol, bad[:5], r.ap.numpy()[tuple(bad[:5].T)], ap[tuple(bad[:5].T)])
    assert same_bits(r.recall.numpy(), rec), protocol
    assert same_bits(r.map.numpy(), m) and (r.mean_ap == mean_ap or (np.isnan(r.mean_ap) and np.isnan(mean_ap)))
    return r


def synthetic(rng, B, R, G, Cn, ties=0, frac_gt=0.7, flags=True, shuffle=True):
    """Detections around the GT of their image (jittered copies, classes mostly right), random extras, scores
    quantised to `ties` levels when ties > 0; GT with labels in [0, Cn), -1 padding, random difficult / crowd flags."""
    gt = np.zeros((B, G, 4), F32)
    gl = np.full((B, G), -1, np.int32)
    for b in range(B):
        n = int(rng.integers(max(1, G // 2), G + 1))
        c = rng.uniform(0.15, 0.85, size=(n, 2))
        s = rng.uniform(0.05, 0.3, size=(n, 2))
        gt[b, :n] = np.clip(np.concatenate([c - s / 2, c + s / 2], 1), 0, 1)
        gl[b, :n] = rng.integers(0, Cn, size=n)
    src = rng.integers(0, G, size=(B, R))
    db = gt[np.arange(B)[:, None], src] + rng.normal(0, 0.03, size=(B, R, 4)).astype(F32)
    rand = rng.uniform(size=(B, R)) > frac_gt
    c = rng.uniform(0.1, 0.9, size=(B, R, 2))
    s = rng.uniform(0.05, 0.4, size=(B, R, 2))
    db[rand] = np.concatenate([c - s / 2, c + s / 2], -1)[rand]
    db = np.clip(db, 0, 1).astype(F32)
    dc = np.where(rng.uniform(size=(B, R)) < 0.85, np.maximum(gl[np.arange(B)[:, None], src], 0),
                  rng.integers(0, Cn, size=(B, R))).astype(F32)
    ds = rng.uniform(size=(B, R)).astype(F32)
    if ties:
        ds = (np.floor(ds * ties) / ties).astype(F32)
    if not shuffle:
        order = np.argsort(-ds, axis=1, kind="stable")
        db, ds, dc = (np.take_along_axis(x, order[..., None] if x.ndim == 3 else order, 1) for x in (db, ds, dc))
    gf = None
    if flags:
        u = rng.uniform(size=(B, G))
        gf = np.where(u < 0.1, 1, np.where(u < 0.15, 2, np.where(u < 0.17, 3, 0))).astype(np.uint8)
    val = rng.integers(0, R + 1, size=B).astype(np.int32)
    return db, ds, dc, val, gt, gl, gf


def nms_inputs(T, rng, B, K, Cn, q, per_class, total, sthr):
    """non_max_suppression output for clustered boxes, and GT drawn from the kept boxes (labels = their classes)."""
    from tfrpn.utils import bbox_utils
    ncl = max(1, K // 16)
    cen = rng.uniform(0.05, 0.95, size=(B, ncl, 1, 2))
    ctr = cen[np.arange(B)[:, None, None], rng.integers(0, ncl, size=(B, K, q)), 0] + rng.normal(0, 0.02, (B, K, q, 2))
    sz = rng.uniform(0.04, 0.3, size=(B, K, q, 2))
    boxes = np.clip(np.concatenate([ctr - sz / 2, ctr + sz / 2], -1), 0, 1).astype(F32)
    scores = (1.0 / (1.0 + np.exp(-rng.normal(-3.0, 2.0, size=(B, K, Cn))))).astype(F32)
    ob, os_, oc, ov = [x.cpu().numpy() for x in bbox_utils.non_max_suppression(
        T.cu(boxes), T.cu(scores), max_output_size_per_class=per_class, max_total_size=total, iou_threshold=0.45,
        score_threshold=sthr)]
    G = 24
    gt = np.zeros((B, G, 4), F32)
    gl = np.full((B, G), -1, np.int32)
    for b in range(B):
        n = min(G, int(ov[b]))
        pick = rng.choice(max(int(ov[b]), 1), size=n, replace=False)
        gt[b, :n] = np.clip(ob[b, pick] + rng.normal(0, 0.02, size=(n, 4)), 0, 1)
        gl[b, :n] = oc[b, pick].astype(np.int32)
    gl[gl == 0] = -1   # class 0 is background: no GT
    gf = (rng.uniform(size=(B, G)) < 0.1).astype(np.uint8) | ((rng.uniform(size=(B, G)) < 0.05) * 2).astype(np.uint8)
    return ob, os_, oc, ov, gt, gl, gf


@pytest.mark.parametrize("protocol", PROTOCOLS)
def test_ssd_voc_nms_output(T, protocol):
    rng = np.random.default_rng(1)
    inputs = nms_inputs(T, rng, 32, 8732, 21, 1, 100, 200, 0.05)
    r = check(T, inputs, 21, protocol)
    assert np.isnan(r.ap.numpy()[0]).all() and 0 < r.mean_ap <= 1   # background class 0 has no GT


@pytest.mark.parametrize("protocol", PROTOCOLS)
def test_decoder_nms_output_c80(T, protocol):
    rng = np.random.default_rng(2)
    inputs = nms_inputs(T, rng, 16, 300, 80, 1, 100, 100, 0.05)
    check(T, inputs, 80, protocol, thresholds=np.linspace(0.3, 0.9, 16).astype(F32) if protocol == "coco" else None)


@pytest.mark.parametrize("protocol", PROTOCOLS)
@pytest.mark.parametrize("ties", [0, 3, 40])
def test_unsorted_rows_ties_flags(T, protocol, ties):
    rng = np.random.default_rng(3 + ties)
    db, ds, dc, val, gb, gl, gf = synthetic(rng, 12, 700, 40, 5, ties=ties)
    dc[0, :50] = 0.5            # non-integer classes
    dc[1, :50] = -1.0
    dc[2, :50] = 5.0             # = C
    dc[3, :50] = np.nan
    dc[4, :50] = -0.0
    ds[5, :20] = np.nan
    ds[5, 20:40] = -0.0
    ds[5, 40:60] = 0.0
    ds[6, :30] = np.inf
    ds[6, 30:60] = -np.inf
    val[7], val[8], val[9] = -5, 701, 0
    check(T, (db, ds, dc, val, gb, gl, gf), 5, protocol, max_dets=60)


def test_crowd_and_difficult_heavy(T):
    rng = np.random.default_rng(4)
    db, ds, dc, val, gb, gl, _ = synthetic(rng, 8, 300, 30, 3, ties=5)
    gf = rng.integers(0, 4, size=gl.shape).astype(np.uint8)
    for protocol in PROTOCOLS:
        check(T, (db, ds, dc, val, gb, gl, gf), 3, protocol, max_dets=0)


def test_non_nice_boxes(T):
    """Pixel coordinates, tiny coordinates, NaN / inf / inverted boxes: the exact IoU path and the crowd rule's guards."""
    rng = np.random.default_rng(5)
    db, ds, dc, val, gb, gl, gf = synthetic(rng, 6, 200, 20, 3)
    db2, gb2 = db * F32(640), gb * F32(640)
    check(T, (db2, ds, dc, val, gb2, gl, gf), 3, "coco")
    db[0, :5] = np.nan
    db[1, :5, 0] = np.inf
    db[2, :5] = db[2, :5][:, [2, 3, 0, 1]]
    gb[3, :3] = np.nan
    gb[4, :3, 2:] = np.inf
    gb[5, :3] = gb[5, :3][:, [2, 3, 0, 1]]
    gf = np.full(gl.shape, 2, np.uint8)   # crowds everywhere
    for protocol in PROTOCOLS:
        check(T, (db, ds, dc, val, gb, gl, gf), 3, protocol)


@pytest.mark.parametrize("B,R,G,Cn", [(3, 50, 1, 2), (2, 64, 1024, 7), (2, 4096, 16, 1), (4, 100, 20, 1),
                                      (3, 300, 30, 1024), (2, 1, 1, 3), (2, 0, 5, 3), (2, 5, 0, 3)])
def test_edge_shapes(T, B, R, G, Cn):
    rng = np.random.default_rng(B * 7 + R + G + Cn)
    db, ds, dc, val, gb, gl, gf = synthetic(rng, B, R, max(G, 1), Cn, ties=7)
    gb, gl, gf = gb[:, :G], gl[:, :G], gf[:, :G]
    for protocol in ("coco", "voc"):
        check(T, (db, ds, dc, val, gb, gl, gf), Cn, protocol, max_dets=0 if R == 4096 else 100)


def test_limits(T):
    torch = T.torch
    z = lambda *s: torch.zeros(s, device=T.dev)
    zi = lambda *s: torch.zeros(s, dtype=torch.int32, device=T.dev)
    with pytest.raises(NotImplementedError):
        T.tfrpn.detection_map(z(1, 4097, 4), z(1, 4097), z(1, 4097), None, z(1, 2, 4), zi(1, 2), num_classes=2)
    with pytest.raises(NotImplementedError):
        T.tfrpn.detection_map(z(1, 8, 4), z(1, 8), z(1, 8), None, z(1, 1025, 4), zi(1, 1025), num_classes=2)
    with pytest.raises(NotImplementedError):
        T.tfrpn.detection_map(z(1, 8, 4), z(1, 8), z(1, 8), None, z(1, 2, 4), zi(1, 2), num_classes=1025)
    with pytest.raises(NotImplementedError):
        T.tfrpn.DetectionMAP(1025, device=T.dev)
    args = (z(1, 8, 4), z(1, 8), z(1, 8), None, z(1, 2, 4), zi(1, 2))
    for kw in (dict(num_classes=0), dict(num_classes=2, protocol="pascal"), dict(num_classes=2, iou_thresholds=[0.0]),
               dict(num_classes=2, iou_thresholds=[1.5]), dict(num_classes=2, iou_thresholds=[0.5] * 17),
               dict(num_classes=2, max_dets=-1)):
        with pytest.raises(ValueError):
            T.tfrpn.detection_map(*args, **kw)
    with pytest.raises(ValueError):
        T.tfrpn.detection_map(z(1, 8, 4), z(1, 8), torch.zeros((1, 8), dtype=torch.int32, device=T.dev), None,
                              z(1, 2, 4), zi(1, 2), num_classes=2)   # classes must be float32
    # at the limits themselves
    T.tfrpn.detection_map(z(1, 4096, 4), z(1, 4096), z(1, 4096), None, z(1, 1024, 4), zi(1, 1024), num_classes=1024)


@pytest.mark.parametrize("protocol", ["voc", "coco"])
def test_one_tie_group_over_2e20_records(T, protocol):
    """257 images x 4096 detections of one class, all with the same score: one tie group over ~500 sort tiles.  Each
    image has one GT, covered by the detection at a different row, so the AP depends on the insertion order."""
    B, R = 257, 4096
    db = np.tile(np.asarray([0.6, 0.6, 0.9, 0.9], F32), (B, R, 1))
    hit = (np.arange(B) * 1031) % R
    db[np.arange(B), hit] = [0.1, 0.1, 0.4, 0.4]
    ds = np.full((B, R), 0.25, F32)
    dc = np.zeros((B, R), F32)
    gb = np.tile(np.asarray([0.1, 0.1, 0.4, 0.4], F32), (B, 1, 1))
    gl = np.zeros((B, 1), np.int32)
    assert B * R > 1 << 20
    r = check(T, (db, ds, dc, None, gb, gl, None), 1, protocol, thresholds=[0.5], max_dets=0)
    assert r.n_gt[0] == B and r.recall.numpy()[0, 0] == 1.0


def test_batches_accumulate_like_one_shot(T):
    rng = np.random.default_rng(7)
    inputs = synthetic(rng, 20, 400, 30, 6, ties=4)
    for protocol in PROTOCOLS:
        whole = T.tfrpn.detection_map(*[T.cu(x) for x in inputs], num_classes=6, protocol=protocol)
        meter = T.tfrpn.DetectionMAP(6, protocol=protocol, capacity=20 * 400, device=T.dev)
        for s in (slice(0, 3), slice(3, 4), slice(4, 20)):
            meter.update(*[T.cu(x[s]) for x in inputs])
        part = meter.compute()
        assert same_bits(part.ap.numpy(), whole.ap.numpy()) and same_bits(part.recall.numpy(), whole.recall.numpy())
        assert np.array_equal(part.n_gt.numpy(), whole.n_gt.numpy())
        meter.reset()
        meter.update(*[T.cu(x) for x in inputs])
        again = meter.compute()
        assert same_bits(again.ap.numpy(), whole.ap.numpy())
    # NumPy in, NumPy out
    rn = T.tfrpn.detection_map(*inputs, num_classes=6, protocol="voc")
    assert all(isinstance(x, np.ndarray) for x in (rn.ap, rn.map, rn.recall, rn.n_gt, rn.thresholds))
    assert rn.protocol == "voc" and rn.ap.shape == (6, 1)


def test_update_in_cuda_graph_and_callers_stream(T):
    torch = T.torch
    rng = np.random.default_rng(8)
    inputs = [T.cu(x) for x in synthetic(rng, 8, 256, 20, 4, ties=6)]
    eager = T.tfrpn.DetectionMAP(4, capacity=8 * 256 * 3, device=T.dev)
    for _ in range(2):
        eager.update(*inputs)
    ref = eager.compute()
    meter = T.tfrpn.DetectionMAP(4, capacity=8 * 256 * 3, device=T.dev)
    s = torch.cuda.Stream(T.dev)
    s.wait_stream(torch.cuda.current_stream(T.dev))
    torch.cuda.synchronize(T.dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        meter.update(*inputs)
    torch.cuda.synchronize(T.dev)
    assert int(meter._state.counters.abs().sum()) == 0
    graph.replay()
    graph.replay()
    got = meter.compute()
    assert same_bits(got.ap.numpy(), ref.ap.numpy()) and np.array_equal(got.n_gt.numpy(), ref.n_gt.numpy())
    # the caller's stream: an update queued behind a long kernel on s has not run when the default stream looks
    side = T.tfrpn.DetectionMAP(4, capacity=8 * 256, device=T.dev)
    torch.cuda.synchronize(T.dev)
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)
        side.update(*inputs)
    before = side._state.counters.clone()
    s.synchronize()
    assert int(before.abs().sum()) == 0 and int(side._state.counters[0]) == 8 * 256


def test_overflow_and_determinism(T):
    rng = np.random.default_rng(9)
    inputs = [T.cu(x) for x in synthetic(rng, 6, 300, 20, 3, ties=5)]
    meter = T.tfrpn.DetectionMAP(3, capacity=6 * 300 + 10, device=T.dev)
    meter.update(*inputs)
    first = meter.compute()
    meter.update(*inputs)          # does not fit: records nothing, n_gt included
    assert int(meter._state.counters[0]) == 6 * 300
    assert np.array_equal(meter._state.counters[1:4].cpu().numpy(), first.n_gt.numpy())
    with pytest.raises(RuntimeError):
        meter.compute()
    meter.reset()
    meter.update(*inputs)
    second = meter.compute()
    assert same_bits(first.ap.numpy(), second.ap.numpy()) and same_bits(first.recall.numpy(), second.recall.numpy())


def test_c_abi_sentinel_outputs_and_errors(T):
    torch = T.torch
    from tfrpn import _lib, evaluation
    rng = np.random.default_rng(10)
    db, ds, dc, val, gb, gl, gf = synthetic(rng, 5, 200, 16, 4, ties=3)
    d = [T.cu(x) for x in (db, ds, dc, val, gb, gl, gf)]
    lib = _lib.load()
    h = _lib.handle(T.dev.index or 0)
    st = torch.cuda.current_stream(T.dev).cuda_stream
    for protocol in PROTOCOLS:
        cfg = evaluation.map_cfg(4, protocol)
        state = evaluation._MapState(4, 5 * 200, T.dev)
        state.records.fill_(0xA5)          # record contents before the first update do not matter
        args = [x.data_ptr() for x in d]
        assert lib.tfrpn_map_update(h, *args, 5, 200, 16, C.byref(cfg), C.byref(state.c), st) == 0
        ap = torch.full((4, cfg.n_thresholds), -7.0, dtype=torch.float64, device=T.dev)
        rc = torch.full((4, cfg.n_thresholds), -7.0, dtype=torch.float64, device=T.dev)
        assert lib.tfrpn_map_compute(h, C.byref(cfg), C.byref(state.c), ap.data_ptr(), rc.data_ptr(), st) == 0
        o = M.detection_map(db, ds, dc, val, gb, gl, gf, num_classes=4, protocol=protocol)
        assert same_bits(ap.cpu().numpy(), o[0]) and same_bits(rc.cpu().numpy(), o[1]), protocol
        assert int(state.counters[-1]) == 0 and int(state.counters[0]) == 5 * 200   # exactly full
        assert np.array_equal(state.counters[1:5].cpu().numpy(), o[2])
    cfg = evaluation.map_cfg(4, "coco")
    state = evaluation._MapState(4, 1000, T.dev)
    args = [x.data_ptr() for x in d]
    bad = _lib.MapCfg.from_buffer_copy(cfg)
    bad.protocol = 3
    assert lib.tfrpn_map_update(h, *args, 5, 200, 16, C.byref(bad), C.byref(state.c), st) == -1
    assert lib.tfrpn_map_update(h, args[0] + 4, *args[1:], 5, 200, 16, C.byref(cfg), C.byref(state.c), st) == -2
    assert lib.tfrpn_map_update(h, None, *args[1:], 5, 200, 16, C.byref(cfg), C.byref(state.c), st) == -1
    assert lib.tfrpn_map_update(h, *args, 5, 4097, 16, C.byref(cfg), C.byref(state.c), st) == -5
    assert lib.tfrpn_map_compute(h, C.byref(cfg), C.byref(state.c), None, None, st) == -1
    # under capture the workspace cannot grow
    big = evaluation._MapState(4, 1 << 26, T.dev)
    ap = torch.empty((4, 10), dtype=torch.float64, device=T.dev)
    s = torch.cuda.Stream(T.dev)
    torch.cuda.synchronize(T.dev)
    rc = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        rc = lib.tfrpn_map_compute(h, C.byref(cfg), C.byref(big.c), ap.data_ptr(), ap.data_ptr(), s.cuda_stream)
    assert rc == -4

"""tfrpn_proposal_recall (recall_kernel) against the NumPy restatement of oracle/recall_oracle.py: matched IoUs
bit-equal and counts exactly equal, in both matching modes, on real proposals at the C2 and C4 shapes, on a
conflict-heavy layout, at the edges of the supported range, and on boxes that take the exact-division path.  Then
the Python interface: accumulation, framework in = framework out, the caller's stream, CUDA-graph capture, errors."""
import ctypes as C

import numpy as np
import pytest

from oracle import recall_oracle as R
from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32
THR16 = np.linspace(0.2, 0.95, 16).astype(F32)


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


def check(T, prop, gt, labels=None, valid=None, thresholds=R.DEFAULT_THRESHOLDS, limits=R.DEFAULT_LIMITS):
    """Both matching modes through tfrpn.proposal_recall against the oracle; returns the greedy result."""
    out = None
    for matching in ("greedy", "coverage"):
        r = T.tfrpn.proposal_recall(T.cu(prop), T.cu(gt), T.cu(labels), T.cu(valid), iou_thresholds=thresholds,
                                    limits=limits, matching=matching, return_gt_iou=True)
        _, _, counts, iou = R.proposal_recall(prop, gt, labels, valid, np.asarray(thresholds, F32), limits, matching)
        got = r.gt_iou.cpu().numpy()
        assert got.shape == iou.shape
        bad = np.flatnonzero(got.view(np.uint32) != iou.view(np.uint32))
        assert bad.size == 0, (matching, bad[:8], got.reshape(-1)[bad[:8]], iou.reshape(-1)[bad[:8]])
        assert np.array_equal(r.hits.numpy(), counts[:-1].reshape(len(limits), -1)) and r.n_gt == counts[-1], matching
        out = out or r
    return out


def proposals_for(T, rng, B, G, hp):
    from tfrpn import synthetic
    fh, fw = O._pair(hp["feature_map_shape"])
    reg, cls = synthetic.head_outputs(rng, B, fh, fw, hp["anchor_count"])
    anchors = O.generate_anchors(hp)
    boxes, _, valid, _ = T.tfrpn.generate_proposals(T.cu(reg), T.cu(cls), T.cu(anchors), hp)
    gt, labels = synthetic.gt_batch(rng, B, G)
    return boxes.cpu().numpy(), valid.cpu().numpy(), gt, labels


def test_c2_generate_proposals_output(T):
    rng = np.random.default_rng(20)
    prop, valid, gt, labels = proposals_for(T, rng, 64, 50, O.get_hyper_params("vgg16"))
    r = check(T, prop, gt, labels, valid)
    assert r.n_gt == int((labels >= 0).sum()) and 0 < r.average_recall[0] <= 1


def test_c4_generate_proposals_output(T):
    rng = np.random.default_rng(21)
    hp = O.get_hyper_params("vgg16", img_size=(800, 1333), feature_map_shape=(50, 84))
    prop, valid, gt, labels = proposals_for(T, rng, 32, 200, hp)
    check(T, prop, gt, labels, valid)


def clustered(rng, B, n_clusters, per_cluster, P, jitter):
    """GT boxes that overlap in clusters, and proposals that are jittered copies of them (most GT share their best
    proposals with their neighbours, so most greedy rounds recompute rows)."""
    G = n_clusters * per_cluster
    c = rng.uniform(0.25, 0.75, size=(B, n_clusters, 1, 2)) + rng.normal(0, 0.02, size=(B, n_clusters, per_cluster, 2))
    s = rng.uniform(0.1, 0.3, size=(B, n_clusters, per_cluster, 2))
    gt = np.clip(np.concatenate([c - s / 2, c + s / 2], axis=-1), 0, 1).reshape(B, G, 4).astype(F32)
    src = gt[np.arange(B)[:, None], rng.integers(0, G, size=(B, P))]
    prop = np.clip(src + rng.normal(0, jitter, size=src.shape), 0, 1).astype(F32)
    return prop, gt


def test_conflict_heavy_layout(T):
    rng = np.random.default_rng(22)
    prop, gt = clustered(rng, 6, 6, 24, 1500, 0.03)
    r = check(T, prop, gt, thresholds=THR16, limits=(50, 144, 300, 1500))
    assert r.hits[0, 0] > 0


@pytest.mark.parametrize("P,valid", [(2000, 0), (2000, 1500), (2000, 2000), (8192, 5000), (8192, 8192)])
def test_range_edges_one_image(T, P, valid):
    rng = np.random.default_rng(P + valid)
    prop, gt = clustered(rng, 1, 64, 16, P, 0.05)
    gt[0, ::7] = 0   # padding rows between real ones
    v = np.asarray([valid], np.int32)
    if P == 8192:
        check(T, prop, gt, valid=v, thresholds=THR16, limits=(1, 10, 100, 300, 1000, 2000, 4096, 8192))
    else:
        check(T, prop, gt, valid=v, thresholds=(0.5,), limits=(100, 1000, 2000))


def test_exact_division_path(T):
    """Boxes outside the nice range (pixel coordinates, tiny coordinates) and NaN / inverted / degenerate boxes send
    the CTA to the exact IoU; the same boxes in [0,1] use the range-check-free division."""
    rng = np.random.default_rng(23)
    prop, gt = clustered(rng, 4, 5, 8, 400, 0.04)
    labels = np.ones(gt.shape[:2], np.int32)
    r_unit = check(T, prop, gt, labels)
    r_px = check(T, prop * F32(640), gt * F32(640), labels)            # coordinates >= 2^8
    assert r_px.n_gt == r_unit.n_gt
    check(T, prop * F32(2.0 ** -20), gt * F32(2.0 ** -20), labels)     # coordinates < 2^-16
    odd = prop.copy()
    odd[0, 0] = np.nan
    odd[1, 1] = odd[1, 1][[2, 3, 0, 1]]       # inverted
    odd[2, 2, 2] = odd[2, 2, 0]               # no height
    g2 = gt.copy()
    g2[3, 0] = g2[3, 0][[2, 3, 0, 1]]          # inverted GT: positive area, valid
    check(T, odd, g2, labels, np.asarray([400, 3, 2, 400], np.int32))


def test_update_accumulates_and_meters_sum(T):
    torch = T.torch
    rng = np.random.default_rng(24)
    prop, gt = clustered(rng, 12, 4, 6, 300, 0.04)
    labels = np.where(rng.uniform(size=gt.shape[:2]) < 0.2, -1, 1).astype(np.int32)
    valid = rng.integers(0, 301, size=12).astype(np.int32)
    whole = T.tfrpn.ProposalRecall(device=T.dev)
    whole.update(T.cu(prop), T.cu(gt), T.cu(labels), T.cu(valid))
    three = T.tfrpn.ProposalRecall(device=T.dev)
    for s in (slice(0, 5), slice(5, 6), slice(6, 12)):
        three.update(T.cu(prop[s]), T.cu(gt[s]), T.cu(labels[s]), T.cu(valid[s]))
    assert torch.equal(three.counts, whole.counts)
    a, b = T.tfrpn.ProposalRecall(device=T.dev), T.tfrpn.ProposalRecall(device=T.dev)
    a.update(prop[:7], gt[:7], labels[:7], valid[:7])
    b.update(prop[7:], gt[7:], labels[7:], valid[7:])
    assert torch.equal(a.counts + b.counts, whole.counts)
    res = whole.compute()
    ref = R.proposal_recall(prop, gt, labels, valid)
    assert np.array_equal(res.hits.numpy(), ref[2][:-1].reshape(3, 10)) and res.n_gt == ref[2][-1]
    assert np.allclose(res.recall.numpy(), ref[0]) and np.allclose(res.average_recall.numpy(), ref[1])
    whole.reset()
    assert int(whole.counts.sum()) == 0


def test_numpy_in_numpy_out_and_torch_on_callers_stream(T):
    torch = T.torch
    rng = np.random.default_rng(25)
    prop, gt = clustered(rng, 3, 3, 5, 200, 0.04)
    rn = T.tfrpn.proposal_recall(prop, gt, return_gt_iou=True)
    assert all(isinstance(x, np.ndarray) for x in (rn.recall, rn.average_recall, rn.hits, rn.thresholds, rn.gt_iou))
    assert rn.limits == (100, 300, 1000) and rn.recall.shape == (3, 10) and rn.gt_iou.shape == (3, 3, 15)
    s = torch.cuda.Stream(T.dev)
    meter = T.tfrpn.ProposalRecall(device=T.dev)
    p, g = T.cu(prop), T.cu(gt)
    torch.cuda.synchronize(T.dev)
    with torch.cuda.stream(s):
        rt = T.tfrpn.proposal_recall(p, g, return_gt_iou=True)
        meter.update(p, g)
        once = meter.counts.clone()
    assert torch.is_tensor(rt.recall) and rt.gt_iou.is_cuda
    s.synchronize()
    assert int(once[-1]) == 45
    before = torch.zeros_like(meter.counts)
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)
        meter.update(p, g)
    before.copy_(meter.counts)   # on the default stream, which does not wait for s: the update has not run yet
    s.synchronize()
    assert torch.equal(before, once) and torch.equal(meter.counts, 2 * once)
    assert np.array_equal(rt.gt_iou.cpu().numpy(), rn.gt_iou) and np.array_equal(rt.hits.numpy(), rn.hits)


def test_update_in_cuda_graph(T):
    torch = T.torch
    rng = np.random.default_rng(26)
    prop, gt = clustered(rng, 8, 4, 8, 300, 0.04)
    p, g = T.cu(prop), T.cu(gt)
    meter = T.tfrpn.ProposalRecall(limits=(10, 100), matching="greedy", device=T.dev)
    s = torch.cuda.Stream(T.dev)
    s.wait_stream(torch.cuda.current_stream(T.dev))
    with torch.cuda.stream(s):
        meter.update(p, g)     # warm-up outside the capture
    torch.cuda.current_stream(T.dev).wait_stream(s)
    torch.cuda.synchronize(T.dev)
    once = meter.counts.clone()
    meter.reset()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        meter.update(p, g)
    torch.cuda.synchronize(T.dev)
    assert int(meter.counts.sum()) == 0
    graph.replay()
    graph.replay()
    torch.cuda.synchronize(T.dev)
    assert torch.equal(meter.counts, 2 * once)


def test_errors(T):
    torch = T.torch
    from tfrpn import _lib
    prop = torch.zeros((1, 16, 4), device=T.dev)
    with pytest.raises(NotImplementedError):
        T.tfrpn.proposal_recall(prop, torch.zeros((1, 1025, 4), device=T.dev))
    with pytest.raises(NotImplementedError):
        T.tfrpn.proposal_recall(prop, torch.zeros((1, 4, 4), device=T.dev), limits=(8193,))
    gt = torch.zeros((1, 4, 4), device=T.dev)
    for kw in (dict(iou_thresholds=[0.0]), dict(iou_thresholds=[1.5]), dict(iou_thresholds=[float("nan")]),
               dict(limits=[0]), dict(limits=[1] * 9), dict(matching="hungarian")):
        with pytest.raises(ValueError):
            T.tfrpn.proposal_recall(prop, gt, **kw)
    with pytest.raises(ValueError):
        T.tfrpn.proposal_recall(prop, gt, gt_labels=torch.zeros((1, 5), dtype=torch.int32, device=T.dev))
    counts = torch.zeros(11, dtype=torch.int64, device=T.dev)
    cfg = T.tfrpn.evaluation.recall_cfg(limits=(16,))
    buf = torch.zeros(17 * 4, device=T.dev)
    lib = _lib.load()
    st = torch.cuda.current_stream(T.dev).cuda_stream
    h = _lib.handle(T.dev.index or 0)
    rc = lib.tfrpn_proposal_recall(h, buf.data_ptr() + 4, None, gt.data_ptr(), None, 1, 16, 4, C.byref(cfg), None,
                                   counts.data_ptr(), st)
    assert rc == -2   # TFRPN_ERR_MISALIGNED
    assert lib.tfrpn_proposal_recall(h, buf.data_ptr(), None, gt.data_ptr(), None, 1, 16, 4, C.byref(cfg), None,
                                     counts.data_ptr(), st) == 0


def test_two_runs_bit_identical(T):
    rng = np.random.default_rng(27)
    prop, gt = clustered(rng, 16, 6, 10, 1000, 0.03)
    a = T.tfrpn.proposal_recall(T.cu(prop), T.cu(gt), return_gt_iou=True)
    b = T.tfrpn.proposal_recall(T.cu(prop), T.cu(gt), return_gt_iou=True)
    assert T.torch.equal(a.gt_iou.view(T.torch.int32), b.gt_iou.view(T.torch.int32))
    assert T.torch.equal(a.hits, b.hits) and a.n_gt == b.n_gt

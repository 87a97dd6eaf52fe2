"""The host pipeline's two-phase proposal transfer (csrc/pipeline.cu): rank launch over the scores, host gather of
the candidate rows of rpn_reg, NMS over the gathered rows; images that need more rows than were gathered are redone
by the unfiltered kernel (page-locked tensor: on the device, pulling rows; pageable tensor: when the step is
retired).  Every variant must give the oracle's keep lists bit for bit."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(np.all(a.view(np.uint32) == b.view(np.uint32)))


def close(a, b, rtol=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= rtol * np.maximum(1.0, np.abs(b))))


class Env:
    """A/B switches are read when a handle is created: set them around the constructor."""

    def __init__(self, **kv):
        self.kv = {k: str(v) for k, v in kv.items()}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        os.environ.update(self.kv)

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def want_for(anchors_np, hp, gtb, gtl, reg, cls, seed, offset, image_offset, pre_nms_topn=6000):
    B = gtb.shape[0]
    if CO.available():
        od, ol = CO.rpn_targets(anchors_np, gtb, gtl, hp, seed=seed, offset=offset, image_offset=image_offset)
        wb, ws, wv, wk = CO.proposals(reg.reshape(B, -1, 4), cls.reshape(B, -1), anchors_np, hp, pre_nms_topn)
    else:
        od, ol = O.calculate_rpn_actual_outputs(anchors_np, gtb, gtl, hp, seed=seed, offset=offset, image_offset=image_offset)
        wb, ws, wv, wk = O.generate_proposals(reg, cls, anchors_np, hp, pre_nms_topn=pre_nms_topn)
    return od, ol.reshape(B, -1), wb, ws, wv, wk


def synthetic_head(i, B):
    from tfrpn import synthetic
    return synthetic.head_outputs(np.random.default_rng(800 + i), B, 31, 31, 9)


def run_acquired(cuda_device, B, G, depth, steps, env, pre_nms_topn=6000, head=synthetic_head):
    """`steps` steps through acquired slots; head(i, B) gives step i's (rpn_reg, rpn_cls)"""
    from tfrpn import HostPipeline, synthetic
    hp = dict(O.get_hyper_params("vgg16"))
    anchors_np = O.generate_anchors(hp)
    with Env(**env):
        pipe = HostPipeline(hp, depth=depth, device=cuda_device, pre_nms_topn=pre_nms_topn)
    # the slot views live apart from the pending items: a failure report shows check()'s argument, and the views'
    # page-locked memory is freed by pipe.close() before the report is written
    pending, copied, views = [], [], {}
    try:
        def check(item):
            t, i, gtb, gtl, reg, cls = item
            pipe.wait(t)
            v = views.pop(t)
            od, ol, wb, ws, wv, wk = want_for(anchors_np, hp, gtb, gtl, reg, cls, 21, i, 5 * i, pre_nms_topn)
            assert bits_equal(v.labels.reshape(B, -1), ol) and close(v.deltas, od)
            assert np.array_equal(v.deltas != 0, od != 0)
            assert np.array_equal(v.valid, wv) and np.array_equal(v.keep_idx, wk)
            assert bits_equal(v.out_scores, ws) and close(v.out_boxes, wb)
            copied.append(pipe.last_copy_bytes())
        for i in range(steps):
            gtb, gtl = synthetic.gt_batch(np.random.default_rng(700 + i), B, G)
            reg, cls = head(i, B)
            if len(pending) == depth - 1:
                check(pending.pop(0))
            v = pipe.acquire(B, G)
            v.gt_boxes[...] = gtb; v.gt_labels[...] = gtl; v.rpn_reg[...] = reg; v.rpn_cls[...] = cls
            v.out_boxes[...] = np.nan; v.out_scores[...] = np.nan; v.valid[...] = -7; v.keep_idx[...] = -7
            t = pipe.submit(seed=21, offset=i, image_offset=5 * i)
            views[t] = v
            pending.append((t, i, gtb, gtl, reg, cls))
        while pending:
            check(pending.pop(0))
    finally:
        pipe.close()
    return copied


def test_acquired_c2_full_batch_depth4(cuda_device):
    """BASELINE config 2 through the pipeline as bench.py drives it: B = 64, four steps in flight"""
    copied = run_acquired(cuda_device, 64, 50, 4, 9, {})
    h2d, d2h = copied[-1]
    dense_in = 64 * 8649 * 20 + 64 * 50 * 20
    assert h2d < 0.4 * dense_in, "the two-phase transfer should move well under half of the dense input bytes"
    assert d2h < 0.4 * 64 * 8649 * 20


@pytest.mark.parametrize("threads", [1, 3, 8])
def test_acquired_host_thread_counts(cuda_device, threads):
    run_acquired(cuda_device, 13, 17, 3, 5, {"TFRPN_HOST_THREADS": threads})


def test_acquired_few_gathered_rows_redone_on_device(cuda_device):
    """128 gathered rows per image cannot yield 300 proposals: every image is redone by the unfiltered kernel,
    which pulls its rows from the slot's page-locked tensor"""
    copied = run_acquired(cuda_device, 6, 9, 2, 4, {"TFRPN_PIPE_GATHER_ROWS": 128})
    assert copied[-1][0] > 6 * 8649 * 4 + 6 * 128 * 16     # scores + gathered rows + pulled rows


def test_acquired_device_side_gather(cuda_device):
    """TFRPN_PIPE_GATHER=device: a kernel reads the candidate rows from the page-locked tensor (no host stage);
    with few rows per image the flagged images are redone as well"""
    copied = run_acquired(cuda_device, 64, 50, 4, 6, {"TFRPN_PIPE_GATHER": "device"})
    assert copied[-1][0] < 0.4 * (64 * 8649 * 20 + 64 * 50 * 20)
    run_acquired(cuda_device, 5, 9, 3, 4, {"TFRPN_PIPE_GATHER": "device", "TFRPN_PIPE_GATHER_ROWS": 200})
    run_acquired(cuda_device, 5, 9, 3, 4, {"TFRPN_PIPE_GATHER": "host", "TFRPN_HOST_THREADS": 2})


def test_acquired_sparse_labels(cuda_device):
    """TFRPN_PIPE_SPARSE_LABELS=1: bbox_labels returns as codes of its <= 256 entries != -1 per image and the host threads
    keep the slot's dense array consistent from step to step (slots are reused: depth 2, 6 steps)"""
    copied = run_acquired(cuda_device, 64, 50, 4, 9, {"TFRPN_PIPE_SPARSE_LABELS": 1})
    assert copied[-1][1] < 64 * 8649 * 4 // 2
    run_acquired(cuda_device, 6, 9, 2, 6, {"TFRPN_PIPE_SPARSE_LABELS": 1, "TFRPN_PIPE_GATHER": "device", "TFRPN_HOST_THREADS": 2})
    run_acquired(cuda_device, 6, 9, 2, 6, {"TFRPN_PIPE_SPARSE_LABELS": 0})


def test_acquired_device_side_expansion(cuda_device):
    """TFRPN_PIPE_EXPAND=device: a kernel keeps the slot's dense bbox_deltas array (page-locked host memory) up to date --
    zeroes the previous step's rows, writes this step's -- and the host scatters nothing (slots reused: depth 2)"""
    run_acquired(cuda_device, 64, 50, 4, 9, {"TFRPN_PIPE_EXPAND": "device"})
    run_acquired(cuda_device, 6, 9, 2, 7, {"TFRPN_PIPE_EXPAND": "device", "TFRPN_PIPE_GATHER": "device", "TFRPN_HOST_THREADS": 1})


def test_acquired_dense_input_switch_equals_two_phase(cuda_device):
    run_acquired(cuda_device, 7, 5, 3, 4, {"TFRPN_PIPE_DENSE_IN": 1})
    run_acquired(cuda_device, 7, 5, 3, 4, {"TFRPN_PIPE_DENSE": 1})


@pytest.mark.parametrize("gather_rows", [0, 96, -1])
@pytest.mark.parametrize("pinned", [False, True])
def test_submit_caller_buffers_two_phase(cuda_device, gather_rows, pinned):
    """tfrpn_pipeline_submit with the caller's own arrays (pageable: the gather reads them in place, flagged images
    are redone when the step is retired; page-locked: redone on the device)"""
    import torch
    from tfrpn import _lib, synthetic
    from tfrpn.proposals import proposal_cfg
    from tfrpn.utils.train_utils import _target_cfg
    hp = dict(O.get_hyper_params("vgg16"))
    anchors_np = O.generate_anchors(hp)
    anchors = torch.from_numpy(anchors_np).to(cuda_device)
    B, G, N, P = 5, 8, 8649, 300
    lib = _lib.load()
    env = {"TFRPN_PIPE_GATHER_ROWS": gather_rows} if gather_rows > 0 else ({"TFRPN_PIPE_SPARSE_LABELS": 1} if gather_rows else {})
    h = C.c_void_p()
    with Env(**env):
        _lib.check(lib.tfrpn_create(C.byref(h), cuda_device.index or 0))
    pipe = C.c_void_p()
    _lib.check(lib.tfrpn_pipeline_create(h, 3, C.byref(pipe)))
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    ptrs = []

    def buf(shape, dtype):
        if not pinned:
            return np.empty(shape, dtype)
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _lib.check(lib.tfrpn_host_alloc(C.byref(p), n))
        ptrs.append(p)
        return np.frombuffer((C.c_char * n).from_address(p.value), dtype=dtype).reshape(shape)

    pc = proposal_cfg(hp, pre_nms_topn=6000)
    steps = []
    try:
        for i in range(5):
            gtb0, gtl0 = synthetic.gt_batch(np.random.default_rng(900 + i), B, G)
            reg0, cls0 = synthetic.head_outputs(np.random.default_rng(950 + i), B, 31, 31, 9)
            st = dict(tc=_target_cfg(hp, 8, i, 2 * i))
            for k, (a, dt) in dict(gtb=(gtb0, F32), gtl=(gtl0, np.int32), reg=(reg0, F32), cls=(cls0, F32)).items():
                st[k] = buf(a.shape, dt)
                st[k][...] = a
            for k, (sh, dt) in dict(d=((B, N, 4), F32), l=((B, N), F32), ob=((B, P, 4), F32), os=((B, P), F32),
                                    ov=((B,), np.int32), ok=((B, P), np.int32)).items():
                st[k] = buf(sh, dt)
                st[k][...] = 55
            t = C.c_int64(-1)
            _lib.check(lib.tfrpn_pipeline_submit(pipe, anchors.data_ptr(), B, N, vp(st["gtb"]), vp(st["gtl"]), G, C.byref(st["tc"]),
                                                 vp(st["d"]), vp(st["l"]), vp(st["reg"]), vp(st["cls"]), C.byref(pc),
                                                 vp(st["ob"]), vp(st["os"]), vp(st["ov"]), vp(st["ok"]), C.byref(t)))
            st["t"] = t.value
            steps.append(st)
        _lib.check(lib.tfrpn_pipeline_drain(pipe))
        for i, st in enumerate(steps):
            od, ol, wb, ws, wv, wk = want_for(anchors_np, hp, st["gtb"], st["gtl"], st["reg"], st["cls"], 8, i, 2 * i)
            assert bits_equal(st["l"], ol) and close(st["d"], od) and np.array_equal(st["d"] != 0, od != 0)
            assert np.array_equal(st["ov"], wv) and np.array_equal(st["ok"], wk)
            assert bits_equal(st["os"], ws) and close(st["ob"], wb)
    finally:
        _lib.check(lib.tfrpn_pipeline_destroy(pipe))
        lib.tfrpn_destroy(h)
        for p in ptrs:
            lib.tfrpn_host_free(p)


def test_submit_arrays_stable_outputs_ring(cuda_device):
    """HostPipeline.submit_arrays on a ring of pageable output dicts with TFRPN_PIPE_OPT_STABLE_OUTPUTS: the dense
    bbox_deltas of every step equals the oracle although only the previously written rows are reset"""
    from tfrpn import HostPipeline, synthetic
    hp = dict(O.get_hyper_params("vgg16"))
    anchors_np = O.generate_anchors(hp)
    B, G, depth = 6, 9, 3
    pipe = HostPipeline(hp, depth=depth, device=cuda_device, pre_nms_topn=6000)
    pipe.set_stable_outputs(True)
    outs = [dict() for _ in range(depth)]
    pending = []
    try:
        def check(item):
            t, i, out, gtb, gtl, reg, cls = item
            pipe.wait(t)
            od, ol, wb, ws, wv, wk = want_for(anchors_np, hp, gtb, gtl, reg, cls, 4, i, 0)
            assert bits_equal(out["bbox_labels"], ol) and close(out["bbox_deltas"], od)
            assert np.array_equal(out["bbox_deltas"] != 0, od != 0)
            assert np.array_equal(out["valid"], wv) and np.array_equal(out["keep_idx"], wk)
        for i in range(8):
            gtb, gtl = synthetic.gt_batch(np.random.default_rng(40 + i), B, G)
            reg, cls = synthetic.head_outputs(np.random.default_rng(60 + i), B, 31, 31, 9)
            if len(pending) == depth - 1:
                check(pending.pop(0))
            t, out = pipe.submit_arrays(gtb, gtl, reg, cls, out=outs[i % depth], seed=4, offset=i)
            pending.append((t, i, out, gtb, gtl, reg, cls))
        while pending:
            check(pending.pop(0))
    finally:
        pipe.close()


# ---- adversarial scores and regressions ---------------------------------------------------------------------------

def tie_scores(rng, B, name, N=8649):
    """(B, N) scores made of tie groups (no -0 beside +0, no -inf: the oracle orders them like the kernels)"""
    if name == "equal":
        return np.full((B, N), 0.5, F32)
    if name == "three":                       # tie groups across the batch floor, rank 1024 and the pre-NMS cap
        s = np.full((B, N), 0.25, F32)
        s[:, :700] = 0.75
        s[:, 700:1100] = 0.5
        return np.stack([r[rng.permutation(N)] for r in s])
    if name == "one_bin_ulps":                # 16 distinct values inside one 11-bit bin
        return (1.0 - 2.0 ** -20 * rng.uniform(0, 1, size=(B, N))).astype(F32)
    if name == "coarse":                      # 65 values: tie groups of ~130 entries everywhere
        return (np.round(rng.uniform(0, 1, size=(B, N)) * 64) / 64).astype(F32)
    raise ValueError(name)


TIE_LAYOUTS = ["three", "equal", "one_bin_ulps", "coarse"]


def collapsed_head(i, B):
    """Step i: rpn_cls from a tie layout, and rpn_reg that decodes a share of the anchors (all, 90 %, half or none,
    by image) onto five boxes per image.  NMS then suppresses nearly everything, runs out of the gathered rows and
    the image is redone; the other images finish inside them."""
    hp = O.get_hyper_params("vgg16")
    anchors = O.generate_anchors(hp)
    N = anchors.shape[0]
    rng = np.random.default_rng(300 + i)
    cls = tie_scores(rng, B, TIE_LAYOUTS[i % len(TIE_LAYOUTS)])
    reg = rng.normal(0, 0.5, size=(B, N, 4)).astype(F32)
    c = rng.uniform(0.2, 0.8, size=(B, 5, 2))
    sz = rng.uniform(0.1, 0.4, size=(B, 5, 2))
    targets = np.clip(np.concatenate([c - sz / 2, c + sz / 2], -1), 0, 1).astype(F32)
    onto = np.take_along_axis(targets, rng.integers(0, 5, size=(B, N, 1)).repeat(4, -1), axis=1)
    deltas = CO.encode(anchors, onto) / np.asarray(hp["variances"], F32) + rng.normal(0, 0.002, size=(B, N, 4))
    share = np.array([1.0, 0.9, 0.5, 0.0])[np.arange(B) % 4]
    m = rng.uniform(size=(B, N)) < share[:, None]
    reg[m] = deltas[m]
    return reg.astype(F32).reshape(B, 31, 31, 36), cls.reshape(B, 31, 31, 9)


TWO_PHASE_PATHS = {
    "host": {},
    "host_rows128": {"TFRPN_PIPE_GATHER_ROWS": 128},
    "device": {"TFRPN_PIPE_GATHER": "device"},
    "device_rows128": {"TFRPN_PIPE_GATHER": "device", "TFRPN_PIPE_GATHER_ROWS": 128},
    "matrix": {"TFRPN_NMS_PATH": "matrix"},
    "matrix_rows128": {"TFRPN_NMS_PATH": "matrix", "TFRPN_PIPE_GATHER_ROWS": 128},
}


@pytest.mark.parametrize("path", list(TWO_PHASE_PATHS))
@pytest.mark.parametrize("topn", [300, 1000, 6000])
def test_acquired_tie_scores_collapsed_boxes(cuda_device, path, topn):
    """Tie-group scores and collapsed regressions through acquired slots.  pre_nms_topn = 300: the rank launch holds
    every rank (rank_more = 0), and with 128 gathered rows the presorted launch must still send its images to the
    redo because it could not serve all their ranks.  1000: the rank batch may or may not hold them all.  Six steps:
    the adaptive gathered-row count grows while images are redone.  B = 6 ranks on 8 x 256, B = 12 on 2 x 512."""
    if not CO.available():
        pytest.skip("oracle/_build/librpn_oracle.so not built")
    B = 12 if path == "host" else 6
    run_acquired(cuda_device, B, 9, 3, 6, TWO_PHASE_PATHS[path], pre_nms_topn=topn, head=collapsed_head)


@pytest.mark.parametrize("rows", [0, 128])
@pytest.mark.parametrize("topn", [300, 1000, 6000])
def test_submit_arrays_tie_scores_collapsed_boxes(cuda_device, rows, topn):
    """the same inputs through submit_arrays on pageable arrays: flagged images are redone when the step is retired"""
    from tfrpn import HostPipeline
    if not CO.available():
        pytest.skip("oracle/_build/librpn_oracle.so not built")
    hp = dict(O.get_hyper_params("vgg16"))
    anchors_np = O.generate_anchors(hp)
    B, depth, P = 6, 3, int(hp["test_nms_topn"])
    with Env(**({"TFRPN_PIPE_GATHER_ROWS": rows} if rows else {})):
        pipe = HostPipeline(hp, depth=depth, device=cuda_device, pre_nms_topn=topn)
    pending = []
    try:
        def check(item):
            t, out, reg, cls = item
            pipe.wait(t)
            wb, ws, wv, wk = CO.proposals(reg.reshape(B, -1, 4), cls.reshape(B, -1), anchors_np, hp, topn)
            assert np.array_equal(out["valid"], wv) and np.array_equal(out["keep_idx"], wk)
            assert bits_equal(out["scores"], ws) and close(out["boxes"], wb)
        for i in range(6):
            reg, cls = collapsed_head(i, B)
            if len(pending) == depth - 1:
                check(pending.pop(0))
            out = dict(boxes=np.full((B, P, 4), np.nan, F32), scores=np.full((B, P), np.nan, F32),
                       valid=np.full((B,), -7, np.int32), keep_idx=np.full((B, P), -7, np.int32))
            t, out = pipe.submit_arrays(rpn_reg=reg, rpn_cls=cls, out=out)
            pending.append((t, out, reg, cls))
        while pending:
            check(pending.pop(0))
    finally:
        pipe.close()

"""Boundary behaviour on the GPU (SURVEY 8b): DLPack producers other than torch, the stream contract,
device selection from the handle / the pointers, pipelines next to drop-in calls."""
import ctypes as C

import numpy as np
import pytest

from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(np.all(a.view(np.uint32) == b.view(np.uint32)))


def close(a, b, rtol=1e-6):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= rtol * np.maximum(1.0, np.abs(b))))


def rand_boxes(rng, *shape):
    a = np.sort(rng.uniform(0, 1, size=shape + (2, 2)), axis=-2).astype(F32)
    return np.stack([a[..., 0, 0], a[..., 0, 1], a[..., 1, 0], a[..., 1, 1]], axis=-1)


class FakeCudaProducer:
    """A third-party GPU array: nothing but the DLPack protocol (neither torch nor TensorFlow on the outside)."""

    def __init__(self, t):
        self._t = t
        self.streams = []

    def __dlpack__(self, *args, **kw):
        self.streams.append(kw.get("stream"))
        return self._t.__dlpack__(**kw)

    def __dlpack_device__(self):
        return self._t.__dlpack_device__()


def test_dlpack_cuda_producer_zero_copy_and_stream_contract(cuda_device):
    import torch
    from tfrpn import _tensor
    from tfrpn.utils import bbox_utils
    rng = np.random.default_rng(1)
    boxes, gt = rand_boxes(rng, 300), rand_boxes(rng, 2, 10)
    tb, tg = torch.from_numpy(boxes).to(cuda_device), torch.from_numpy(gt).to(cuda_device)
    pb, pg = FakeCudaProducer(tb), FakeCudaProducer(tg)
    o = _tensor.Origin()
    t = _tensor.ingest(pb, o, "boxes")
    assert o.kind == "dlpack" and t.data_ptr() == tb.data_ptr()          # zero copy
    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        got = bbox_utils.generate_iou_map(pb, pg)
        # the producer was told which stream the consumer enqueues on: the one our kernels are launched on
        assert pb.streams[-1] == side.cuda_stream and pg.streams[-1] == side.cuda_stream
        assert _tensor.stream_ptr(cuda_device) == side.cuda_stream
    side.synchronize()
    assert isinstance(got, torch.Tensor) and got.is_cuda
    assert bits_equal(got.cpu().numpy(), O.generate_iou_map(boxes, gt))
    # on the default stream torch announces the legacy default stream (1) or the per-thread one (2)
    bbox_utils.generate_iou_map(pb, pg)
    assert pb.streams[-1] in (1, 2, None)


def two_gpus():
    import torch
    return torch.cuda.is_available() and torch.cuda.device_count() >= 2


def test_two_devices_driven_from_one_thread(cuda_device):
    """One thread, handle(0) then handle(1): launches, workspaces and >48 KB shared-memory attributes must
    follow the handle's device, and the caller's current device must not change."""
    if not two_gpus():
        pytest.skip("needs 2 GPUs")
    import torch
    import tfrpn
    from tfrpn import synthetic
    from tfrpn.utils import bbox_utils, train_utils
    hp = dict(O.get_hyper_params("vgg16"))
    a_np = O.generate_anchors(hp)
    rng = np.random.default_rng(4)
    gtb, gtl = synthetic.gt_batch(rng, 3, 20)
    reg, cls = synthetic.head_outputs(rng, 3, 31, 31, 9)
    od, ol = O.calculate_rpn_actual_outputs(a_np, gtb, gtl, hp, seed=3, offset=1)
    wb, ws, wv, wk = O.generate_proposals(reg, cls, a_np, hp)
    torch.cuda.set_device(0)
    for rep in range(2):
        for d in (0, 1, 1, 0):
            dev = torch.device("cuda", d)
            cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
            anchors = cu(a_np)
            deltas, labels = train_utils.calculate_rpn_actual_outputs(anchors, cu(gtb), cu(gtl), hp, seed=3, offset=1)
            assert deltas.device == dev and torch.cuda.current_device() == 0
            assert bits_equal(labels.cpu().numpy(), ol) and close(deltas.cpu().numpy(), od)
            pb, ps, pv, pk = tfrpn.generate_proposals(cu(reg), cu(cls), anchors, hp)
            assert np.array_equal(pv.cpu().numpy(), wv) and np.array_equal(pk.cpu().numpy(), wk)
            assert bits_equal(ps.cpu().numpy(), ws) and torch.cuda.current_device() == 0
            iou = bbox_utils.generate_iou_map(anchors, cu(gtb))          # handle-less: device from the pointers
            assert iou.device == dev and bits_equal(iou.cpu().numpy(), O.generate_iou_map(a_np, gtb))
    # a tensor on the wrong device for the handle is refused, not silently read across devices
    from tfrpn import _lib
    lib, h0 = _lib.load(), _lib.handle(0)
    dev1 = torch.device("cuda", 1)
    s1 = torch.zeros((2, 100), device=dev1)
    v = torch.empty((2, 5), device=dev1)
    i = torch.empty((2, 5), dtype=torch.int32, device=dev1)
    assert lib.tfrpn_topk(h0, s1.data_ptr(), 2, 100, 5, v.data_ptr(), i.data_ptr(), None, 0, None, None) == -1
    assert b"device" in lib.tfrpn_last_error()


def test_pipeline_in_flight_next_to_dropin_calls(cuda_device):
    """A training loop that pulls targets from the prefetching generator and calls the drop-in functions
    (losses, target assignment, sampling) in the same thread while steps are in flight: the pipeline owns its
    own handle, so the shared per-thread workspace is never raced."""
    import torch
    from tfrpn import synthetic
    from tfrpn.utils import bbox_utils, train_utils
    hp = dict(O.get_hyper_params("vgg16"), seed=9)
    a_np = O.generate_anchors(hp)
    data = []
    for i in range(4):
        gtb, gtl = synthetic.gt_batch(np.random.default_rng(700 + i), 8, 25)
        data.append(("img%d" % i, gtb, gtl))
    reg, cls = synthetic.head_outputs(np.random.default_rng(7), 8, 31, 31, 9)
    treg, tcls = torch.from_numpy(reg).to(cuda_device), torch.from_numpy(cls).to(cuda_device)
    gen = train_utils.rpn_generator(data, a_np, hp, prefetch=3)          # NumPy anchors are accepted here too
    anchors = bbox_utils.generate_anchors(hp)
    for step in range(10):
        img, (deltas, labels) = next(gen)
        name, gtb, gtl = data[step % 4]
        od, ol = O.calculate_rpn_actual_outputs(a_np, gtb, gtl, hp, seed=9, offset=step)
        assert bits_equal(labels, ol) and close(deltas, od)
        # drop-in calls on torch's stream, the thread's shared handle, while 3 generator steps are in flight
        r = train_utils.rpn_losses(torch.from_numpy(np.ascontiguousarray(deltas)).to(cuda_device), treg,
                                   torch.from_numpy(np.ascontiguousarray(labels)).to(cuda_device), tcls)
        d2, l2 = train_utils.calculate_rpn_actual_outputs(anchors, torch.from_numpy(gtb).to(cuda_device),
                                                          torch.from_numpy(gtl).to(cuda_device), hp, seed=9, offset=step)
        want_reg, want_cls = O.reg_loss(deltas, reg), O.cls_loss(labels, cls)
        assert abs(float(r["reg_loss"]) - want_reg) <= 2e-6 * max(abs(want_reg), 1e-30)
        assert abs(float(r["cls_loss"]) - want_cls) <= 2e-6 * max(abs(want_cls), 1e-30)
        assert bits_equal(l2.cpu().numpy(), ol)
    gen.close()


def test_pipeline_rejects_foreign_anchors(cuda_device):
    from tfrpn import HostPipeline
    hp = dict(O.get_hyper_params("vgg16"))
    with pytest.raises(ValueError):
        HostPipeline(hp, depth=1, anchors=np.zeros((10, 3), F32))
    with pytest.raises(ValueError):
        HostPipeline(hp, depth=1, anchors=np.zeros((10, 4), np.float64))


def test_pipeline_dense_deltas_survive_a_layout_change(cuda_device):
    """Compact step, then a proposals-only step with ANOTHER (B,G) layout in the same slot (its inputs land inside
    the old dense deltas region), then the first layout again: the dense bbox_deltas view must be rebuilt from
    scratch, not patched incrementally over garbage."""
    from tfrpn import HostPipeline, synthetic
    hp = dict(O.get_hyper_params("vgg16"))
    a_np = O.generate_anchors(hp)
    pipe = HostPipeline(hp, depth=1)
    try:
        for i, (B, G, mode) in enumerate([(9, 9, "targets"), (9, 9, "targets"), (4, 40, "proposals"), (3, 2, "both"),
                                          (9, 9, "targets"), (9, 9, "both")]):
            gtb, gtl = synthetic.gt_batch(np.random.default_rng(900 + i), B, G)
            reg, cls = synthetic.head_outputs(np.random.default_rng(950 + i), B, 31, 31, 9)
            v = pipe.acquire(B, G)
            v.gt_boxes[...] = gtb; v.gt_labels[...] = gtl
            v.rpn_reg[...] = reg if mode != "proposals" else 1e3   # garbage that must never show up as a delta
            v.rpn_cls[...] = cls
            if mode == "proposals":
                v.rpn_reg[...] = reg
            t = pipe.submit(targets=mode != "proposals", proposals=mode != "targets", seed=2, offset=i)
            pipe.wait(t)
            if mode != "proposals":
                od, ol = O.calculate_rpn_actual_outputs(a_np, gtb, gtl, hp, seed=2, offset=i)
                assert bits_equal(v.labels, ol) and close(v.deltas, od)
                assert np.array_equal(v.deltas != 0, od != 0)
    finally:
        pipe.close()

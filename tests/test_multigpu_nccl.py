"""The optional final gather on real hardware (north star: "NCCL over NVLink is used only for an optional
final gather of proposals and targets"): world_size 2 over NCCL, one process per GPU, the CUDA path on each
shard, `sharding.gather_rows` == the unsharded run bit for bit.  Skipped below 2 GPUs."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    for p in (ROOT, os.path.join(ROOT, "tf-rpn_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import tfrpn
        from tfrpn import sharding, synthetic
        from tfrpn.utils import bbox_utils, train_utils
        hp = dict(train_utils.get_hyper_params("vgg16"))
        anchors = bbox_utils.generate_anchors(hp)
        B, G = 13, 30                                   # ragged split: 7 + 6
        rng = np.random.default_rng(12)                 # every rank generates the same global batch
        gtb, gtl = synthetic.gt_batch(rng, B, G)
        reg, cls = synthetic.head_outputs(rng, B, 31, 31, 9)
        cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
        d, l = sharding.sharded_rpn_targets(anchors, cu(gtb), cu(gtl), hp, rank, world, seed=5, offset=2)
        pb, ps, pv, pk = sharding.sharded_proposals(cu(reg), cu(cls), anchors, hp, rank, world)
        torch.cuda.synchronize()
        parts = [d, l, pb, ps, pv, pk]
        gathered = [sharding.gather_rows(t, B) for t in parts]
        # timing of the gather alone (latency-bound: 20*N*B/R bytes of targets + ~28*300*B/R of proposals per rank)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(20):
            for t in parts:
                sharding.gather_rows(t, B)
        e1.record()
        torch.cuda.synchronize()
        ok = True
        if rank == 0:
            fd, fl = train_utils.calculate_rpn_actual_outputs(anchors, cu(gtb), cu(gtl), hp, seed=5, offset=2)
            fb, fs, fv, fk = tfrpn.generate_proposals(cu(reg), cu(cls), anchors, hp)
            for got, want in zip(gathered, (fd, fl, fb, fs, fv, fk)):
                ok = ok and got.shape == want.shape and bool(torch.equal(got, want))
        q.put((rank, ok, e0.elapsed_time(e1) / 20, dist.get_backend()))
    finally:
        dist.destroy_process_group()


def test_nccl_gather_equals_unsharded():
    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok, _, _ in res) and all(b == "nccl" for *_, b in res)
    print("NCCL gather of targets + proposals (B=13, world 2): %.3f ms per step" % max(ms for _, _, ms, _ in res))

#!/usr/bin/env python
"""Time of the detection mAP: tfrpn_map_update (map_match_kernel + map_cursor_kernel) per batch and tfrpn_map_compute
(the radix sort + map_ap_kernel) per call.  CUDA events around `reps` calls after 3 warm-up calls, inputs resident on
the device.  Update workloads (seeded, synthetic detections around the GT, 20 GT per image): the SSD-VOC shape
(B = 32 images x R = 200 detections, C = 21) and a decoder shape (B = 16 x R = 100, C = 80), each with T = 1 (voc,
0.5) and T = 10 (coco, 0.50:0.05:0.95).  Compute workloads: 10^5 and 10^6 records (SSD-VOC batches accumulated), T = 1
and T = 10.  Beside them, labelled CPU, the host time of the NumPy oracle (oracle/map_oracle.py) for one update batch
and for the compute of 10^5 records.
Usage: map_time.py [reps]"""
import ctypes as C
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tf-rpn_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import tfrpn  # noqa: E402
from oracle import map_oracle as M  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
dev = torch.device("cuda:0")
F32 = np.float32


def batch(rng, B, R, G, Cn):
    gt = np.zeros((B, G, 4), F32)
    c = rng.uniform(0.15, 0.85, size=(B, G, 2))
    s = rng.uniform(0.05, 0.3, size=(B, G, 2))
    gt[:] = np.clip(np.concatenate([c - s / 2, c + s / 2], -1), 0, 1)
    gl = rng.integers(1, Cn, size=(B, G)).astype(np.int32)
    src = rng.integers(0, G, size=(B, R))
    db = np.clip(gt[np.arange(B)[:, None], src] + rng.normal(0, 0.03, size=(B, R, 4)), 0, 1).astype(F32)
    dc = np.where(rng.uniform(size=(B, R)) < 0.8, gl[np.arange(B)[:, None], src], rng.integers(1, Cn, size=(B, R)))
    ds = np.sort(rng.uniform(size=(B, R)).astype(F32), axis=1)[:, ::-1].copy()
    valid = np.full(B, R, np.int32)
    gf = (rng.uniform(size=(B, G)) < 0.05).astype(np.uint8)
    return db, ds, dc.astype(F32), valid, gt, gl, gf


def timed(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


SETUPS = [("T=1 voc", dict(protocol="voc")), ("T=10 coco", dict(protocol="coco"))]


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
print("CUDA events around %d calls after 3 warm-up calls, inputs resident on the device" % reps)
rng = np.random.default_rng(0)
for name, B, R, Cn in (("SSD-VOC", 32, 200, 21), ("decoder", 16, 100, 80)):
    host = batch(rng, B, R, 20, Cn)
    d = [torch.from_numpy(x).to(dev) for x in host]
    for label, kw in SETUPS:
        meter = tfrpn.DetectionMAP(Cn, capacity=(reps + 3) * B * R, device=dev, **kw)
        t = timed(lambda: meter.update(*d))
        acc = M.MapAccumulator(Cn, kw["protocol"])
        t0 = time.perf_counter()
        acc.update(*host)
        cpu = time.perf_counter() - t0
        print("update %-8s B=%-3d R=%-4d C=%-3d %-9s GPU %8.1f us per batch   (CPU oracle %8.1f ms)" % (
            name, B, R, Cn, label, 1e3 * t, 1e3 * cpu), flush=True)

host = batch(rng, 32, 200, 20, 21)
d = [torch.from_numpy(x).to(dev) for x in host]
for n_rec in (100_000, 1_000_000):
    nb = (n_rec + 32 * 200 - 1) // (32 * 200)
    for label, kw in SETUPS:
        meter = tfrpn.DetectionMAP(21, capacity=nb * 32 * 200, device=dev, **kw)
        for _ in range(nb):
            meter.update(*d)
        st = meter._state
        cfg = meter._cfg
        out = torch.empty((2, 21, cfg.n_thresholds), dtype=torch.float64, device=dev)
        lib = tfrpn._lib.load()
        h = tfrpn._lib.handle(0)
        def run():
            tfrpn._lib.check(lib.tfrpn_map_compute(h, C.byref(cfg), C.byref(st.c), out[0].data_ptr(),
                                                   out[1].data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
        t = timed(run)
        line = "compute %8d records (%d batches) C=21 %-9s GPU %8.1f us" % (nb * 32 * 200, nb, label, 1e3 * t)
        if n_rec == 100_000:
            acc = M.MapAccumulator(21, kw["protocol"])
            for _ in range(nb):
                acc.update(*host)
            t0 = time.perf_counter()
            ap, _, _ = acc.compute()
            line += "   (CPU oracle %8.1f ms)" % (1e3 * (time.perf_counter() - t0))
            got = meter.compute()
            line += "  bit-equal=%s" % np.array_equal(got.ap.numpy().view(np.uint64), ap.view(np.uint64))
        print(line, flush=True)

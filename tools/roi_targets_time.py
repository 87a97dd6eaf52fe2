#!/usr/bin/env python
"""Time of the second stage's RoI target assignment: tfrpn_roi_targets (roi_target_kernel, one launch) per batch,
inputs resident on the device, CUDA events after 3 warm-up calls.  "kernel": 20 calls captured in one CUDA graph,
replayed reps times (device time alone); "Python call": `reps` eager calls of tfrpn.roi_targets (the device timeline,
including any gap while the host prepares the next call).  Workloads (seeded, synthetic):
this library's chain at C2 (B = 64 images x P = 300 proposals, G = 50 GT, S = 128 rows with 32 fg) and two
Detectron-like batches (B = 2 and 16, P = 2000, G = 100, S = 512 with 128 fg), each with and without the GT rows
appended; at the Detectron shape also pixel coordinates (the exact-division IoU instead of the range-check-free one).
Beside them, on the same GPU, torchvision's RoIHeads.select_training_samples configured alike (same S, fg fraction,
thresholds; it always appends the GT) on the same boxes in (x1,y1,x2,y2) order, and, labelled CPU, the host time of
the NumPy oracle (oracle/roi_oracle.py) for one batch.
Usage: roi_targets_time.py [reps]"""
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
from oracle import roi_oracle as R  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
dev = torch.device("cuda:0")
F32 = np.float32


def boxes(rng, n, lo, hi):
    c = rng.uniform(0, 1, size=(n, 2))
    s = rng.uniform(lo, hi, size=(n, 2))
    return np.clip(np.concatenate([c - s / 2, c + s / 2], axis=1), 0, 1).astype(F32)


def batch(rng, B, P, G, C):
    """a quarter of the proposals jittered around GT boxes, the rest anywhere; 50..100 % of the GT rows real"""
    gt = np.zeros((B, G, 4), F32)
    lab = np.full((B, G), -1, np.int32)
    rois = np.zeros((B, P, 4), F32)
    for b in range(B):
        n = int(rng.integers(G // 2, G + 1))
        gt[b, :n] = boxes(rng, n, 0.05, 0.4)
        lab[b, :n] = rng.integers(1, C, size=n)
        near = gt[b, rng.integers(0, n, size=P // 4)] + rng.normal(0, 0.03, size=(P // 4, 4)).astype(F32)
        rois[b] = np.concatenate([np.clip(near, 0, 1), boxes(rng, P - P // 4, 0.02, 0.5)])
    return rois, gt, lab


def events(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize(dev)
    return a.elapsed_time(b) * 1e3 / reps


def graph_events(fn, per_graph=20):
    """device time of fn alone: `per_graph` calls captured in one CUDA graph, replayed; no host work in the window"""
    s = torch.cuda.Stream(dev)
    s.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream(dev).wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            fn()
    return events(g.replay) / per_graph


def torchvision_fn(rois, gt, lab, tp, tn, fg_thr, bg_hi):
    from torchvision.models.detection.roi_heads import RoIHeads
    S = tp + tn
    heads = RoIHeads(None, None, None, fg_thr, bg_hi, S, tp / S, (10.0, 10.0, 5.0, 5.0), 0.05, 0.5, 100)
    xy = [1, 0, 3, 2]
    props = [torch.from_numpy(np.ascontiguousarray(r[:, xy])).to(dev) for r in rois]
    targets = []
    for b in range(gt.shape[0]):
        keep = lab[b] >= 1
        targets.append({"boxes": torch.from_numpy(np.ascontiguousarray(gt[b][keep][:, xy])).to(dev),
                        "labels": torch.from_numpy(lab[b][keep].astype(np.int64)).to(dev)})
    return lambda: heads.select_training_samples(props, targets)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
print("CUDA events around %d calls after 3 warm-up calls, inputs resident on the device" % reps)
rng = np.random.default_rng(0)
for name, B, P, G, C, tp, tn, scale in (("C2 chain", 64, 300, 50, 21, 32, 96, 1.0),
                                       ("Detectron", 2, 2000, 100, 81, 128, 384, 1.0),
                                       ("Detectron", 16, 2000, 100, 81, 128, 384, 1.0),
                                       ("Detectron px", 16, 2000, 100, 81, 128, 384, 1333.0)):
    rois, gt, lab = batch(rng, B, P, G, C)
    rois, gt = (rois * F32(scale)).astype(F32), (gt * F32(scale)).astype(F32)
    r, g, l = (torch.from_numpy(x).to(dev) for x in (rois, gt, lab))
    for append_gt in (True, False):
        call = lambda: tfrpn.roi_targets(r, g, l, num_classes=C, total_pos=tp, total_neg=tn,  # noqa: E731
                                         append_gt=append_gt, offset=0)
        us = events(call)
        kern = graph_events(call)
        t0 = time.perf_counter()
        R.roi_targets(rois, gt, lab, num_classes=C, total_pos=tp, total_neg=tn, append_gt=append_gt)
        cpu_ms = (time.perf_counter() - t0) * 1e3
        line = ("%-12s B=%-3d P=%-5d G=%-4d S=%-4d append_gt=%d  kernel %7.1f us   Python call %7.1f us"
                "   (CPU oracle %7.1f ms)") % (name, B, P, G, tp + tn, append_gt, kern, us, cpu_ms)
        if append_gt:
            tv = events(torchvision_fn(rois, gt, lab, tp, tn, 0.5, 0.5))
            line += "   torchvision select_training_samples %8.1f us" % tv
        print(line, flush=True)

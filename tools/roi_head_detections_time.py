#!/usr/bin/env python
"""Time of the second stage's box-head detections: tfrpn_roi_head_detections (roi_det_score_kernel, then the
multi-class NMS's stage, proposal_kernel and merge launches), inputs resident on the device, CUDA events around `reps`
calls after 5 warm-up calls.
  (a) kernel       the C entry point alone, 20 calls captured in one CUDA graph and replayed (device time only)
  (b) python       tfrpn.roi_head_detections (the same launches plus the Python call)
  (c) composition  what the call replaces: torch.softmax, tfrpn_decode on the RoIs repeated q times, the masking
                   (rows < valid, classes >= 1, score > threshold; min_size is 0 here) in torch ops, then
                   tfrpn_nms_multiclass.
                   Checked in the same run: with the call's own probabilities in place of torch.softmax its five
                   outputs are bit-identical to (a)'s; with torch.softmax the number of images whose outputs differ
                   in any bit is printed.
  (d) torchvision  RoIHeads.postprocess_detections on the same tensors in pixel coordinates (the valid rows of each
                   image as its proposal list, box_coder weights (10, 10, 5, 5)); a timing reference only.
Then one torch.profiler pass over (a)'s calls gives the device time of each kernel.
Workloads (seeded): proposal-like RoIs with padding rows at the end of every image, trained-looking logits (60 % of the
rows background, the others one class raised by U(1, 6)), deltas ~ N(0, 1), score threshold 0.05, 100 detections:
  C2 chain     B = 64, S = 300, C = 21, q = 21 and q = 1
  two-stage    B = 16, S = 300, C = 21, q = 21 (tools/nms_multiclass_time.py's "two-stage decoder")
  Detectron    B = 16, S = 1000, C = 81, q = 81
Usage: roi_head_detections_time.py [reps] [output file]"""
import collections
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tf-rpn_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import tfrpn  # noqa: E402
from tfrpn import _lib  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
out_path = sys.argv[2] if len(sys.argv) > 2 else None
dev = torch.device("cuda:0")
F32 = np.float32
VAR = (0.1, 0.1, 0.2, 0.2)
THR, PER_CLASS, TOTAL, IOU = 0.05, 100, 100, 0.5
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def events(fn):
    for _ in range(5):
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


def workload(rng, B, S, Cn, q):
    ctr = rng.uniform(0.05, 0.95, size=(B, S, 2))
    sz = rng.uniform(0.02, 0.5, size=(B, S, 2))
    rois = np.concatenate([ctr - sz / 2, ctr + sz / 2], -1).astype(F32)
    valid = (S - rng.integers(0, S // 4 + 1, size=B)).astype(np.int32)
    rois[np.arange(S)[None, :] >= valid[:, None]] = 0
    x = rng.normal(0, 1, size=(B, S, Cn)).astype(F32)
    k = np.where(rng.uniform(size=(B, S)) < 0.6, 0, rng.integers(1, Cn, size=(B, S)))
    np.put_along_axis(x, k[..., None], np.take_along_axis(x, k[..., None], -1)
                      + rng.uniform(1, 6, size=(B, S, 1)).astype(F32), -1)
    d = rng.normal(0, 1, size=(B, S, q, 4)).astype(F32)
    return [torch.from_numpy(a).to(dev) for a in (rois, valid, x, d)]


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
say("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
say("CUDA events around %d calls after 5 warm-up calls, inputs resident on the device; times per call" % reps)
try:
    from torchvision.models.detection.roi_heads import RoIHeads
except ImportError:
    RoIHeads = None
lib, h = _lib.load(), _lib.handle(0)
rng = np.random.default_rng(0)
for name, B, S, Cn, q in (("C2 chain", 64, 300, 21, 21), ("C2 chain", 64, 300, 21, 1), ("two-stage", 16, 300, 21, 21),
                          ("Detectron", 16, 1000, 81, 81)):
    rois, valid, x, d = workload(rng, B, S, Cn, q)
    st = lambda: torch.cuda.current_stream(dev).cuda_stream  # noqa: E731
    nms = _lib.NmsCfg(PER_CLASS, TOTAL, IOU, THR, 0, 1, 0)
    cfg = _lib.RoiDetCfg(Cn, q, 0, (_lib.C.c_float * 4)(*VAR), float("inf"), 1, 0.0, nms)
    outs = [torch.empty((B, TOTAL, 4), device=dev), torch.empty((B, TOTAL), device=dev),
            torch.empty((B, TOTAL), device=dev), torch.empty((B,), dtype=torch.int32, device=dev),
            torch.empty((B, TOTAL), dtype=torch.int32, device=dev)]
    probs = torch.empty((B, S, Cn), device=dev)

    def kernel(with_probs=False):
        return lambda: _lib.check(lib.tfrpn_roi_head_detections(
            h, rois.data_ptr(), valid.data_ptr(), x.data_ptr(), d.data_ptr(), B, S, _lib.C.byref(cfg),
            *[o.data_ptr() for o in outs], probs.data_ptr() if with_probs else None, st()))

    def python():
        tfrpn.roi_head_detections(rois, x, d, valid, score_threshold=THR, return_indices=True)

    anchors = rois[:, :, None, :].expand(B, S, q, 4).reshape(B, S * q, 4).contiguous()
    var_host = (_lib.C.c_float * 4)(*VAR)
    boxes = torch.empty((B, S, q, 4), device=dev)
    c_outs = [torch.empty_like(o) for o in outs]
    row_ok = (torch.arange(S, device=dev)[None, :] < valid[:, None])[..., None]
    cls_ok = torch.arange(Cn, device=dev) >= 1

    def composition(p=None):
        def run():
            pr = torch.softmax(x, -1) if p is None else p
            _lib.check(lib.tfrpn_decode(anchors.data_ptr(), 1, d.data_ptr(), var_host, 1, B, S * q, boxes.data_ptr(),
                                        st()))
            sc = torch.where(row_ok & cls_ok & (pr > THR), pr, torch.full_like(pr, float("-inf")))
            _lib.check(lib.tfrpn_nms_multiclass(h, boxes.data_ptr(), q, sc.data_ptr(), B, S, Cn, _lib.C.byref(nms),
                                                *[o.data_ptr() for o in c_outs], st()))
        return run

    kernel(True)()
    composition(probs)()
    torch.cuda.synchronize(dev)
    same = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(outs, c_outs))
    composition()()
    torch.cuda.synchronize(dev)
    diff_img = torch.zeros(B, dtype=torch.bool, device=dev)
    for a, b in zip(outs, c_outs):
        diff_img |= (a.view(torch.int32) != b.view(torch.int32)).reshape(B, -1).any(1)
    n_det = int(outs[3].sum())
    t_a, t_b, t_c = graph_events(kernel()), events(python), events(composition())
    say("%-10s B=%-3d S=%-4d C=%-3d q=%-3d  %5d detections | (a) kernel %7.1f us | (b) Python %7.1f us | (c) composition "
        "%7.1f us | (a) == (c) on the call's probs: %s, with torch.softmax: %d of %d images differ"
        % (name, B, S, Cn, q, n_det, t_a, t_b, t_c, "bit-identical" if same else "DIFFERENT", int(diff_img.sum()), B))
    if RoIHeads is not None:
        heads = RoIHeads(None, None, None, 0.5, 0.5, 512, 0.25, (10.0, 10.0, 5.0, 5.0), THR, IOU, TOTAL)
        px = rois * 512.0
        props = [px[b, :int(valid[b]), [1, 0, 3, 2]] for b in range(B)]
        logits = torch.cat([x[b, :int(valid[b])] for b in range(B)])
        reg = torch.cat([d[b, :int(valid[b])] for b in range(B)]).reshape(logits.shape[0], -1)
        if q == 1:
            reg = reg.repeat(1, Cn)
        shapes = [(512, 512)] * B

        def tv():
            heads.postprocess_detections(logits, reg, props, shapes)

        say("%-10s (d) torchvision RoIHeads.postprocess_detections: %7.1f us" % ("", events(tv)))
    else:
        say("%-10s (d) torchvision not installed: not measured" % "")
    f = kernel()
    for _ in range(3):
        f()
    torch.cuda.synchronize(dev)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            f()
        torch.cuda.synchronize(dev)
    per = collections.OrderedDict()
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            k = e.name.split("(")[0].replace("void ", "").replace("tfrpn::", "")
            per[k] = per.get(k, 0.0) + e.device_time / 20
    say("%-10s (a) per kernel, torch.profiler: %s" % ("", ", ".join("%s %.1f us" % kv for kv in per.items())))

if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write("\n".join(lines) + "\n")

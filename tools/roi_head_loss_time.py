#!/usr/bin/env python
"""Time of the second stage's box-head losses: tfrpn_roi_head_losses (roi_loss_partial_kernel, and with the gradients
roi_loss_grad_kernel), inputs resident on the device, CUDA events around `reps` calls after 5 warm-up calls.
  kernel            the C entry point alone, 20 calls captured in one CUDA graph and replayed (device time only):
                    without the gradients (one launch) and with both gradients and a device scale (two launches)
  forward           tfrpn.roi_head_losses without the gradients (one launch, plus the Python call)
  forward+backward  tfrpn.roi_head_losses on tensors that require grad, then (cls + reg).backward() (three launches,
                    plus the Python call and autograd)
Beside them, on the same GPU and tensors, torchvision's roi_heads.fastrcnn_loss (F.cross_entropy, torch.where on the
labels, smooth_l1 with beta = 1/9) forward, and forward + autograd backward.  Its torch.where synchronises the host on
every call, which the timing includes: that is what a training step pays for it.
Workloads (seeded; labels like roi_targets' rows: 25 % fg, the rest background, padding at the end of some images):
  C2 chain   B = 64, S = 128, C = 21, q = 21 and q = 1
  Detectron  B = 2 and B = 16, S = 512, C = 81, q = 81
Usage: roi_head_loss_time.py [reps] [output file]"""
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


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
say("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
say("CUDA events around %d calls after 5 warm-up calls, inputs resident on the device; times per call" % reps)
try:
    from torchvision.models.detection.roi_heads import fastrcnn_loss
except ImportError:
    fastrcnn_loss = None
rng = np.random.default_rng(0)
for name, B, S, C, q in (("C2 chain", 64, 128, 21, 21), ("C2 chain", 64, 128, 21, 1), ("Detectron", 2, 512, 81, 81),
                         ("Detectron", 16, 512, 81, 81)):
    u = rng.uniform(size=(B, S))
    lab = np.where(u < 0.25, rng.integers(1, C, size=(B, S)), 0).astype(np.int32)
    lab[::3, S - S // 8:] = -1
    logits = torch.from_numpy(rng.normal(0, 2, size=(B, S, C)).astype(F32)).to(dev)
    deltas = torch.from_numpy(rng.normal(0, 1, size=(B, S, q * 4)).astype(F32)).to(dev)
    tgt_np = rng.normal(0, 1, size=(B, S, 4)).astype(F32)
    tgt_np[lab <= 0] = 0
    labels, targets = torch.from_numpy(lab).to(dev), torch.from_numpy(tgt_np).to(dev)
    lg, dg = logits.clone().requires_grad_(True), deltas.clone().requires_grad_(True)

    def ours_fwd():
        tfrpn.roi_head_losses(logits, deltas, labels, targets, huber_delta=1.0 / 9, normalize="rows")

    def ours_bwd():
        r = tfrpn.roi_head_losses(lg, dg, labels, targets, huber_delta=1.0 / 9, normalize="rows")
        (r.cls_loss + r.reg_loss).backward()

    cfg = _lib.RoiLossCfg(C, q, 1.0 / 9, 1)
    out, scale = torch.empty(8, device=dev), torch.ones(2, device=dev)
    g_l, g_d = torch.empty_like(logits), torch.empty_like(deltas)
    lib, h = _lib.load(), _lib.handle(0)

    def kernel(grads):
        return lambda: _lib.check(lib.tfrpn_roi_head_losses(
            h, logits.data_ptr(), deltas.data_ptr(), labels.data_ptr(), targets.data_ptr(), B, S, _lib.C.byref(cfg),
            out.data_ptr(), scale.data_ptr() if grads else None, g_l.data_ptr() if grads else None,
            g_d.data_ptr() if grads else None, torch.cuda.current_stream(dev).cuda_stream))

    k_f, k_b = graph_events(kernel(False)), graph_events(kernel(True))
    t_f, t_b = events(ours_fwd), events(ours_bwd)
    say("%-10s B=%-3d S=%-4d C=%-3d q=%-3d  tfrpn kernel %6.1f us, with gradients %6.1f us | Python forward %6.1f us,"
        " forward+backward %6.1f us" % (name, B, S, C, q, k_f, k_b, t_f, t_b))
    if fastrcnn_loss is None:
        say("%-10s torchvision not installed: fastrcnn_loss not measured" % "")
        continue
    keep = labels >= 0                                  # fastrcnn_loss has no padding rule: it gets the real rows
    tv_l, tv_d = logits[keep], deltas[keep].reshape(-1, q * 4)
    if q == 1:
        tv_d = tv_d.repeat(1, C)                        # class-agnostic deltas shared by every class
    tv_lab, tv_t = [labels[keep].long()], [targets[keep]]
    tv_lg, tv_dg = tv_l.clone().requires_grad_(True), tv_d.clone().requires_grad_(True)

    def tv_fwd():
        fastrcnn_loss(tv_l, tv_d, tv_lab, tv_t)

    def tv_bwd():
        c, b = fastrcnn_loss(tv_lg, tv_dg, tv_lab, tv_t)
        (c + b).backward()

    say("%-10s torchvision fastrcnn_loss + autograd: forward %6.1f us, forward+backward %6.1f us"
        % ("", events(tv_fwd), events(tv_bwd)))

if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write("\n".join(lines) + "\n")

#!/usr/bin/env python
"""Time of RoI feature cropping: tfrpn_crop_and_resize (crop_kernel) and tfrpn_crop_and_resize_grad_image
(crop_grad_kernel), inputs resident on the device, CUDA events around `reps` calls after 5 warm-up calls.
Workloads (seeded, synthetic boxes like roi_targets' rows, NULL box_index layout):
  C2 chain      B = 64, S = 128, VGG16 features 31 x 31 x 512, 7 x 7 crops
  B16 VGG16     B = 16, S = 512, 31 x 31 x 512, 7 x 7
  Detectron     B = 2,  S = 512, 50 x 50 x 256, 14 x 14
Bytes from shapes: forward = crops written once + feature map read once; gradient = grad_out read once + grad_image
written once; achieved bytes/s against 7.7 TB/s (HBM3e of one B200 on its data sheet).  The feature map (at most
31 MB here) fits in L2, so the corner reads mostly come from there.
Beside each, on the same GPU, torchvision.ops.roi_align (aligned=True, sampling_ratio=2) forward and its backward op
on the same features in NCHW and the same boxes in pixels: a different sampling rule (bin centres, 2 x 2 samples
averaged per bin) doing the same job; its backward scatters with atomics.
Usage: crop_and_resize_time.py [reps] [output file]"""
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
HBM = 7.7e12
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


def rand_boxes(rng, n):
    c = rng.uniform(0, 1, size=(n, 2))
    s = rng.uniform(0.02, 0.6, size=(n, 2))
    return np.clip(np.concatenate([c - s / 2, c + s / 2], axis=1), 0, 1).astype(F32)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
say("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
say("CUDA events around %d calls after 5 warm-up calls, inputs resident on the device; GB/s from shapes" % reps)
lib = _lib.load()
st = torch.cuda.current_stream(dev).cuda_stream
rng = np.random.default_rng(0)
for name, B, S, H, W, C, ch, cw in (("C2 chain", 64, 128, 31, 31, 512, 7, 7),
                                    ("B16 VGG16", 16, 512, 31, 31, 512, 7, 7),
                                    ("Detectron", 2, 512, 50, 50, 256, 14, 14)):
    M = B * S
    feats = torch.from_numpy(rng.normal(size=(B, H, W, C)).astype(F32)).to(dev)
    boxes_np = rand_boxes(rng, M)
    boxes = torch.from_numpy(boxes_np).to(dev)
    out = torch.empty((M, ch, cw, C), device=dev)
    grad = torch.randn((M, ch, cw, C), device=dev)
    gimg = torch.empty_like(feats)
    fwd = lambda: _lib.check(lib.tfrpn_crop_and_resize(  # noqa: E731
        feats.data_ptr(), B, H, W, C, boxes.data_ptr(), None, M, ch, cw, 0.0, out.data_ptr(), st))
    bwd = lambda: _lib.check(lib.tfrpn_crop_and_resize_grad_image(  # noqa: E731
        grad.data_ptr(), boxes.data_ptr(), None, M, B, H, W, C, ch, cw, gimg.data_ptr(), st))
    t_f, t_b = events(fwd), events(bwd)
    crop_bytes, map_bytes = 4.0 * M * ch * cw * C, 4.0 * B * H * W * C
    gbs = lambda t: (crop_bytes + map_bytes) / (t * 1e-6) / 1e9  # noqa: E731
    say("%-10s B=%-3d S=%-4d %dx%dx%-4d crop %dx%-2d  crops %6.1f MB | forward %8.1f us %6.0f GB/s (%.2f of 7.7 TB/s)"
        " | gradient %8.1f us %6.0f GB/s (%.2f)" % (name, B, S, H, W, C, ch, cw, crop_bytes / 1e6, t_f, gbs(t_f),
                                                   gbs(t_f) * 1e9 / HBM, t_b, gbs(t_b), gbs(t_b) * 1e9 / HBM))
    try:
        import torchvision  # noqa: F401
        nchw = feats.permute(0, 3, 1, 2).contiguous()
        bi = torch.arange(M, device=dev, dtype=torch.float32).div_(S).floor_()
        px = boxes[:, [1, 0, 3, 2]] * torch.tensor([W - 1, H - 1, W - 1, H - 1], device=dev, dtype=torch.float32)
        rois = torch.cat([bi[:, None], px], dim=1).contiguous()
        g_nchw = torch.randn((M, C, ch, cw), device=dev)
        tv_f = events(lambda: torch.ops.torchvision.roi_align(nchw, rois, 1.0, ch, cw, 2, True))
        tv_b = events(lambda: torch.ops.torchvision._roi_align_backward(g_nchw, rois, 1.0, ch, cw, B, C, H, W, 2, True))
        say("%-10s torchvision roi_align (aligned, sampling_ratio 2): forward %8.1f us | backward %8.1f us"
            % ("", tv_f, tv_b))
    except ImportError:
        say("%-10s torchvision not installed: roi_align not measured" % "")
    del feats, out, grad, gimg
    torch.cuda.empty_cache()

if out_path:
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        f.write("\n".join(lines) + "\n")

#!/usr/bin/env python
"""Time of tfrpn_proposal_recall (recall_kernel), greedy against coverage matching, with CUDA events around `reps`
calls after 3 warm-up calls.  Coverage matching is round 0 alone, so greedy - coverage is what the greedy rounds cost.
Workloads: real generate_proposals output at the C2 shape (64 images, 300 proposals, 50 GT slots) and at the C4 shape
(32 images, 200 GT slots, 1000 proposals kept so that AR@1000 sees 1000 ranks), limits (100, 300, 1000); and one
image of 1024 clustered GT boxes against 2000 / 8192 jittered copies.  `pairs` is the number of round-0 IoUs: the
sum over limits and images of k_eff x valid GT.  Usage: recall_time.py [reps]"""
import ctypes as C, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tf-rpn_b200"))
import numpy as np, torch
import tfrpn
from tfrpn import _lib, evaluation, synthetic
from oracle import rpn_oracle as O

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
dev = torch.device("cuda:0")
lib = _lib.load(); h = _lib.handle(0)
st = torch.cuda.current_stream(dev).cuda_stream
F32 = np.float32


def rpn_case(rng, hp, B, G, post):
    fh, fw = O._pair(hp["feature_map_shape"])
    reg, cls = synthetic.head_outputs(rng, B, fh, fw, hp["anchor_count"])
    anchors = torch.from_numpy(O.generate_anchors(hp)).to(dev)
    boxes, _, valid, _ = tfrpn.generate_proposals(torch.from_numpy(reg).to(dev), torch.from_numpy(cls).to(dev),
                                                  anchors, hp, post_nms_topn=post)
    gt, labels = synthetic.gt_batch(rng, B, G)
    return boxes, valid, torch.from_numpy(gt).to(dev), torch.from_numpy(labels).to(dev)


def clustered_case(rng, P, n_clusters=64, per=16):
    G = n_clusters * per
    c = rng.uniform(0.25, 0.75, size=(n_clusters, 1, 2)) + rng.normal(0, 0.02, size=(n_clusters, per, 2))
    s = rng.uniform(0.05, 0.2, size=(n_clusters, per, 2))
    gt = np.clip(np.concatenate([c - s / 2, c + s / 2], axis=-1), 0, 1).reshape(1, G, 4).astype(F32)
    src = gt[:, rng.integers(0, G, size=P)]
    prop = np.clip(src + rng.normal(0, 0.05, size=src.shape), 0, 1).astype(F32)
    return torch.from_numpy(prop).to(dev), None, torch.from_numpy(gt).to(dev), None


def time_case(name, case, limits):
    prop, valid, gt, labels = case
    B, P = prop.shape[:2]
    G = gt.shape[1]
    nv = (valid.clamp(0, P) if valid is not None else torch.full((B,), P, device=dev)).cpu().numpy()
    area = (gt[..., 2] - gt[..., 0]) * (gt[..., 3] - gt[..., 1])
    ngt = ((area > 0) & (labels >= 0 if labels is not None else True)).sum(dim=1).cpu().numpy()
    pairs = sum(int((np.minimum(nv, k) * ngt).sum()) for k in limits)
    line = "%-34s B=%-3d P=%-5d G=%-5d limits=%-20s pairs=%9d" % (name, B, P, G, ",".join(map(str, limits)), pairs)
    ms = {}
    for matching in ("coverage", "greedy"):
        cfg = evaluation.recall_cfg(None, limits, matching)
        counts = torch.zeros(len(limits) * 10 + 1, dtype=torch.int64, device=dev)
        call = lambda: _lib.check(lib.tfrpn_proposal_recall(
            h, prop.data_ptr(), valid.data_ptr() if valid is not None else None, gt.data_ptr(),
            labels.data_ptr() if labels is not None else None, B, P, G, C.byref(cfg), None, counts.data_ptr(), st))
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms[matching] = e0.elapsed_time(e1) / reps
        if matching == "greedy":
            c = counts.cpu().numpy() // (reps + 3)
            ar = (c[:-1].reshape(len(limits), 10).mean(axis=1) / max(c[-1], 1)).round(3).tolist()
    cov, gr = ms["coverage"], ms["greedy"]
    print("%s  coverage %9.1f us  greedy %9.1f us  greedy rounds %+9.1f us (%4.2fx round 0)  AR %s"
          % (line, 1e3 * cov, 1e3 * gr, 1e3 * (gr - cov), (gr - cov) / cov, ar), flush=True)


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                      "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
print("recall_kernel, CUDA events around %d calls after 3 warm-up calls, inputs resident on the device" % reps)
rng = np.random.default_rng(0)
time_case("C2 generate_proposals", rpn_case(rng, O.get_hyper_params("vgg16"), 64, 50, 300), (100, 300, 1000))
hp4 = O.get_hyper_params("vgg16", img_size=(800, 1333), feature_map_shape=(50, 84))
time_case("C4 generate_proposals (post 1000)", rpn_case(rng, hp4, 32, 200, 1000), (100, 300, 1000))
time_case("1 image, 1024 clustered GT", clustered_case(rng, 2000), (100, 300, 1000, 2000))
time_case("1 image, 1024 clustered GT", clustered_case(rng, 8192), (100, 300, 1000, 8192))

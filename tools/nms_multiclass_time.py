#!/usr/bin/env python
"""Time of the multi-class combined NMS: tfrpn_nms_multiclass (nms_mc_stage_kernel -> proposal_kernel per class ->
nms_mc_merge_kernel) against the composition the Python drop-in ran before it (restated below: a (B*C, K) copy of
the scores and a (B*C, K, 4) copy of the boxes, one tfrpn_nms launch over B*C "images", a stable torch.sort merge).
CUDA events around `reps` calls of each after 3 warm-up calls, inputs resident on the device; both paths' outputs are
compared bit for bit in the same run; per-kernel times of the native path come from tfrpn_profile_* in a separate
pass.  The native path is timed with each staging layout (TFRPN_NMS_MC_STAGE=column | rows, one handle each; its
outputs are compared too).  Workloads (seeded): SSD-VOC (32 x 8732 anchors, 20 classes, shared boxes) at score
thresholds 0.05 and 0.5, a two-stage decoder (16 x 300 RoIs, 20 classes, class-specific boxes), 4 x 20000 boxes,
8 classes, no threshold, and 4 x 100000 boxes, 4 classes (past the one-class NMS's large-N prefilter threshold).
Usage: nms_multiclass_time.py [reps]"""
import ctypes as C, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tf-rpn_b200"))
import numpy as np, torch
from tfrpn import _lib

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
dev = torch.device("cuda:0")
lib = _lib.load(); h = _lib.handle(0)


def stage_handle(mode):
    os.environ["TFRPN_NMS_MC_STAGE"] = mode   # read once, when the handle is created
    hh = _lib.P()
    _lib.check(lib.tfrpn_create(C.byref(hh), 0))
    del os.environ["TFRPN_NMS_MC_STAGE"]
    return hh


LAYOUTS = {"column": stage_handle("column"), "rows": stage_handle("rows")}
st = torch.cuda.current_stream(dev).cuda_stream
F32 = np.float32


def rows_of(cfg, Cn):
    return min(cfg.max_total_size, cfg.max_output_size_per_class * Cn) if cfg.pad_per_class else cfg.max_total_size


def native(bx, sc, cfg, hh=None):
    B, K, q, _ = bx.shape
    Cn = sc.shape[2]
    rows = rows_of(cfg, Cn)
    outs = (torch.empty((B, rows, 4), device=dev), torch.empty((B, rows), device=dev), torch.empty((B, rows), device=dev),
            torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B, rows), dtype=torch.int32, device=dev))
    _lib.check(lib.tfrpn_nms_multiclass(hh or h, bx.data_ptr(), q, sc.data_ptr(), B, K, Cn, C.byref(cfg),
                                        *[o.data_ptr() for o in outs], st))
    return outs


def composed(bx, sc, cfg):
    """the replaced torch composition (tfrpn/utils/bbox_utils.py before tfrpn_nms_multiclass)"""
    B, K, Cn = sc.shape
    q = bx.shape[2]
    P, total = cfg.max_output_size_per_class, cfg.max_total_size
    rows = rows_of(cfg, Cn)
    sc_t = sc.permute(0, 2, 1).contiguous().reshape(B * Cn, K)
    bx_t = (bx.expand(B, K, Cn, 4) if q == 1 else bx).permute(0, 2, 1, 3).contiguous().reshape(B * Cn, K, 4)
    c1 = _lib.NmsCfg(P, P, cfg.iou_threshold, cfg.score_threshold, 0, cfg.clip_boxes, cfg.pre_nms_topn)
    nb = torch.empty((B * Cn, P, 4), device=dev)
    ns = torch.empty((B * Cn, P), device=dev)
    nc = torch.empty((B * Cn, P), device=dev)
    nv = torch.empty((B * Cn,), dtype=torch.int32, device=dev)
    ni = torch.empty((B * Cn, P), dtype=torch.int32, device=dev)
    _lib.check(lib.tfrpn_nms(h, bx_t.data_ptr(), sc_t.data_ptr(), B * Cn, K, C.byref(c1), nb.data_ptr(), ns.data_ptr(),
                             nc.data_ptr(), nv.data_ptr(), ni.data_ptr(), st))
    slot = torch.arange(P, device=dev)
    live = slot[None, :] < nv[:, None]
    key = torch.where(live, ns, torch.full_like(ns, float("-inf"))).reshape(B, Cn * P)
    order = torch.sort(key, dim=1, descending=True, stable=True).indices
    n_live = live.reshape(B, -1).sum(dim=1)
    take = min(rows, Cn * P)
    order = order[:, :take]
    valid = torch.clamp(n_live, max=min(rows, total)).to(torch.int32)
    keep = torch.arange(take, device=dev)[None, :] < valid[:, None]
    ob = torch.zeros((B, rows, 4), device=dev)
    os_ = torch.zeros((B, rows), device=dev)
    oc = torch.zeros((B, rows), device=dev)
    oi = torch.full((B, rows), -1, dtype=torch.int32, device=dev)
    gb = torch.gather(nb.reshape(B, Cn * P, 4), 1, order[..., None].expand(-1, -1, 4))
    gs = torch.gather(ns.reshape(B, Cn * P), 1, order)
    gi = torch.gather(ni.reshape(B, Cn * P), 1, order)
    ob[:, :take] = torch.where(keep[..., None], gb, torch.zeros_like(gb))
    os_[:, :take] = torch.where(keep, gs, torch.zeros_like(gs))
    oc[:, :take] = torch.where(keep, (order // P).to(torch.float32), torch.zeros_like(gs))
    oi[:, :take] = torch.where(keep, gi, torch.full_like(gi, -1))
    return ob, os_, oc, valid, oi


def workload(rng, B, K, Cn, q, uniform):
    ncl = max(1, K // 16)   # clustered boxes, so the NMS suppresses
    cen = rng.uniform(0.05, 0.95, size=(B, ncl, 1, 2))
    ctr = cen[np.arange(B)[:, None, None], rng.integers(0, ncl, size=(B, K, q)), 0] + rng.normal(0, 0.02, size=(B, K, q, 2))
    sz = rng.uniform(0.04, 0.3, size=(B, K, q, 2))
    boxes = np.clip(np.concatenate([ctr - sz / 2, ctr + sz / 2], -1), 0, 1).astype(F32)
    if uniform:
        scores = rng.uniform(0, 1, size=(B, K, Cn)).astype(F32)
    else:
        scores = (1.0 / (1.0 + np.exp(-rng.normal(-3.0, 2.0, size=(B, K, Cn))))).astype(F32)
    return torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev)


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


def kernel_times(bx, sc, cfg, hh):
    _lib.check(lib.tfrpn_profile_enable(hh, 1))
    for _ in range(reps):
        native(bx, sc, cfg, hh)
    out = []
    for kid in range(_lib.KERNEL_IDS):
        ms, n = C.c_double(), C.c_int()
        _lib.check(lib.tfrpn_profile_read(hh, kid, C.byref(ms), C.byref(n)))
        if n.value:
            out.append("%s %.1f us" % (lib.tfrpn_kernel_name(kid).decode(), 1e3 * ms.value / n.value))
    _lib.check(lib.tfrpn_profile_enable(hh, 0))
    return ", ".join(out)


def run(name, B, K, Cn, q, per_class, total, iou, sthr, uniform, seed):
    bx, sc = workload(np.random.default_rng(seed), B, K, Cn, q, uniform)
    cfg = _lib.NmsCfg(per_class, total, iou, sthr, 0, 1, 0)
    b = composed(bx, sc, cfg)
    same = True
    for hh in [h] + list(LAYOUTS.values()):
        a = native(bx, sc, cfg, hh)
        torch.cuda.synchronize()
        same = same and all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(a, b))
    cand = int((sc > sthr).sum()) if sthr != float("-inf") else sc.numel()
    t_comp = timed(lambda: composed(bx, sc, cfg))
    t_nat = timed(lambda: native(bx, sc, cfg))
    line = "%-20s B=%-3d K=%-6d C=%-3d q=%-3d %d/%d iou=%.2f sthr=%-5s candidates=%-8d" % (
        name, B, K, Cn, q, per_class, total, iou, sthr, cand)
    print("%s composed %9.1f us  native %9.1f us  (%.2fx)  identical=%s" % (line, 1e3 * t_comp, 1e3 * t_nat,
                                                                           t_comp / t_nat, same), flush=True)
    for mode, hh in LAYOUTS.items():
        print("    staging %-6s native %9.1f us; per kernel: %s" % (mode, 1e3 * timed(lambda: native(bx, sc, cfg, hh)),
                                                                  kernel_times(bx, sc, cfg, hh)), flush=True)
    if not same:
        raise SystemExit("native and composed outputs differ")


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                      "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("GPU: %s (name, power limit, max SM clock, SM clock at start)" % smi)
print("CUDA events around %d calls after 3 warm-up calls, inputs resident on the device" % reps)
run("SSD-VOC", 32, 8732, 20, 1, 100, 200, 0.45, 0.05, False, 1)
run("SSD-VOC", 32, 8732, 20, 1, 100, 200, 0.45, 0.5, False, 1)
run("two-stage decoder", 16, 300, 20, 20, 100, 100, 0.5, 0.05, False, 2)
run("no threshold", 4, 20000, 8, 1, 300, 300, 0.7, float("-inf"), True, 3)
run("large K", 4, 100000, 4, 1, 100, 100, 0.5, 0.05, False, 4)
for hh in LAYOUTS.values():
    lib.tfrpn_destroy(hh)

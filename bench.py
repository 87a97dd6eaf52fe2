#!/usr/bin/env python
"""bench.py -- RPN target + proposal images/sec on B200 (BASELINE.json's metric; default config C2).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores
    python bench.py --config C1|C2|C3|C4|C5 [--c5-k 100000] [--c5-mode topk_nms|nms_all]
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs (.npy)

A "step" is one pass of the hot path over one synthetic batch: calculate_rpn_actual_outputs
(target assignment) + generate_proposals (decode, clip, top-6000, NMS 300 @ 0.7) for the batch one
GPU owns (C2: 64 VGG16-RPN 500x500 images); C5 is the NMS / top-k stress (8 images of K boxes per GPU).
`value` = images/s with inputs resident in HBM (device timed, CUDA events, max over ranks); `e2e` = the
same through the host-buffer C-ABI entry points with the H2D / D2H copies inside the timed region.
One JSON line on stdout (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tf-rpn_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "rpn_target+proposal_images_per_sec"
PRE_NMS = 6000
L2_BYTES = 126e6
MAX_SETS = 512


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class Workload:
    """One BASELINE.json config.  kind "rpn": target assignment + proposals (C1-C4); kind "nms": C5."""

    def __init__(self, name, c5_k=100000, c5_mode="topk_nms"):
        from tfrpn import synthetic
        self.name, self.kind = name, ("nms" if name == "C5" else "rpn")
        if self.kind == "rpn":
            bb, B, G, over = synthetic.CONFIGS[name]
            self.backbone, self.B, self.G, self.over = bb, B, G, over
            fm = over.get("feature_map_shape", 31 if bb == "vgg16" else 32)
            self.fm_h, self.fm_w = (fm, fm) if isinstance(fm, int) else fm
            self.A = 9
            self.N = self.fm_h * self.fm_w * self.A
            img = over.get("img_size", 500)
            img = "%dx%d" % ((img, img) if isinstance(img, int) else (img[1], img[0]))
            self.desc = ("%s: %s-RPN %s (%dx%dx9 = %d anchors), batch %d per GPU, <=%d GT boxes/image, "
                         "pre-NMS top-%d / post-NMS 300 @ IoU 0.7"
                         % (name, {"vgg16": "VGG16", "mobilenet_v2": "MobileNetV2"}[bb], img, self.fm_h, self.fm_w,
                            self.N, B, G, PRE_NMS))
            if name == "C2":   # the driver compares this string between the two arms: keep round 1's text
                self.desc = ("C2: VGG16-RPN 500x500 (31x31x9 = 8649 anchors), batch 64 per GPU, <=50 GT boxes/image, "
                             "pre-NMS top-6000 / post-NMS 300 @ IoU 0.7")
        else:
            self.B, self.G, self.N, self.mode = 8, 0, int(c5_k), c5_mode
            self.pre = min(PRE_NMS, self.N) if c5_mode == "topk_nms" else 0
            self.desc = ("C5: NMS / top-k stress, %d boxes per image, batch 8 per GPU, %s, 300 @ IoU 0.7"
                         % (self.N, "top-6000 then NMS" if self.pre else "NMS over all boxes"))
        self.P = 300

    def hyper_params(self, get_hyper_params):
        return dict(get_hyper_params(self.backbone), **self.over)

    def set_bytes(self):
        if self.kind == "rpn":
            return self.B * (self.G * 20 + self.N * 40 + self.P * 28)
        return self.B * (self.N * 20 + self.P * 32)

    def n_sets(self, lanes):
        s = int(np.ceil(2.1 * L2_BYTES / self.set_bytes()))
        s = max(lanes, min(MAX_SETS, s))
        return (s + lanes - 1) // lanes * lanes

    def make_inputs(self, rank, n_sets):
        """SURVEY 8d synthetic inputs; seed = 1000*config + rank.  Two generated sets, the rest are
        batch-rolled copies (distinct memory is what matters for the L2 rotation)."""
        from tfrpn import synthetic
        rng = np.random.default_rng(1000 * int(self.name[1]) + rank)
        base = []
        for _ in range(2):
            if self.kind == "rpn":
                gtb, gtl = synthetic.gt_batch(rng, self.B, self.G)
                reg, cls = synthetic.head_outputs(rng, self.B, self.fm_h, self.fm_w, self.A)
                base.append((gtb, gtl, reg, cls))
            else:
                base.append(synthetic.nms_boxes(rng, self.B, self.N))
        sets = []
        for s in range(n_sets):
            sh = s // 2
            if sh == 0 or self.B == 1:
                sets.append(base[s % 2])
            else:
                sets.append(tuple(np.ascontiguousarray(np.roll(a, sh, axis=0)) for a in base[s % 2]))
        return sets


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons through NVML.  The thread samples every 5 ms while it runs (it is
    started before the barrier, so its start-up is not inside the timed region); sample() is also called
    from the main thread right after the timed steps have been enqueued, while the GPU is still busy."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz, self.stop_flag = [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def sample(self):
        nv = self.nv
        if nv is None:
            return
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for name in ("HwSlowdown", "HwThermalSlowdown", "SwThermalSlowdown", "SwPowerCap", "HwPowerBrakeSlowdown"):
                bit = getattr(nv, "nvmlClocksEventReason" + name, getattr(nv, "nvmlClocksThrottleReason" + name, 0))
                if bit and (r & bit):
                    self.reasons.add(name)
        except Exception:  # noqa: BLE001
            pass

    def run(self):
        while not self.stop_flag:
            time.sleep(0.005)
            if not self.stop_flag:
                self.sample()

    def result(self):
        self.stop_flag = True
        if self.is_alive():
            self.join(timeout=1)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def cpu_path(wl, sets, anchors_np, hp, threads, n_images):
    """The CPU restatement of one step on `n_images` images (C oracle, OpenMP over images; NumPy
    oracle if the C library is missing).  Returns (seconds, kind-description)."""
    from oracle import c_oracle, rpn_oracle
    t0 = time.perf_counter()
    if wl.kind == "nms":
        boxes, scores = (a[:n_images] for a in sets[0])
        if not c_oracle.available():
            raise SystemExit("C5 needs the C oracle (make -C oracle)")
        if wl.pre:
            v, i = c_oracle.top_k(scores, wl.pre)
            boxes = np.take_along_axis(boxes, i[..., None].astype(np.int64), axis=1)
            scores = v
        c_oracle.nms(boxes, scores, wl.P, wl.P, 0.7)
        return time.perf_counter() - t0, "oracle/rpn_oracle.c (gcc -O2, top_k + nms, 1 thread)"
    gtb, gtl, reg, cls = (a[:n_images] for a in sets[0])
    if c_oracle.available():
        c_oracle.rpn_targets(anchors_np, gtb, gtl, hp, seed=1, offset=0, threads=threads)
        c_oracle.proposals(reg.reshape(n_images, -1, 4), cls.reshape(n_images, -1), anchors_np, hp, PRE_NMS,
                           threads=threads)
        what = "oracle/rpn_oracle.c (gcc -O2, OpenMP over images)"
    else:
        rpn_oracle.calculate_rpn_actual_outputs(anchors_np, gtb, gtl, hp, seed=1)
        rpn_oracle.generate_proposals(reg, cls, anchors_np, hp, pre_nms_topn=PRE_NMS)
        what = "oracle/rpn_oracle.py (NumPy, 1 thread)"
    return time.perf_counter() - t0, what


def cpu_threads(wl):
    from oracle import c_oracle
    # every host thread this process may use (torchrun exports OMP_NUM_THREADS=1: the oracle overrides it)
    return len(os.sched_getaffinity(0)) if (c_oracle.available() and wl.kind == "rpn") else 1


def run_reference(args):
    """--impl reference: the reference algorithm on the host cores.  The reference itself (TF 2.0
    eager Python) cannot be installed in this image, so this arm times the oracle port with every
    host thread it can use (kind = "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import rpn_oracle
    wl = Workload(args.config, args.c5_k, args.c5_mode)
    hp = anchors = None
    if wl.kind == "rpn":
        hp = wl.hyper_params(rpn_oracle.get_hyper_params)
        anchors = rpn_oracle.generate_anchors(hp)
    cores = os.cpu_count() or 1
    threads = cpu_threads(wl)
    sets = wl.make_inputs(0, 2)
    W, K = max(args.warmup, 1), max(args.steps, 1)
    dt, _ = cpu_path(wl, sets, anchors, hp, threads, wl.B)
    K = max(1, min(K, 20, int(60.0 / max(dt, 1e-3))))   # bounded: each step is a full batch on the CPU
    W = min(W, 2)
    for _ in range(W - 1):
        cpu_path(wl, sets, anchors, hp, threads, wl.B)
    t = 0.0
    what = ""
    for _ in range(K):
        dt, what = cpu_path(wl, sets, anchors, hp, threads, wl.B)
        t += dt
    value = wl.B * K / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * t / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl.desc, "global_batch": wl.B,
                       "note": "CPU arm runs one %d-image batch per step on rank 0" % wl.B},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
                             "sample": "%d steps x %d images, %s; host has %d cores" % (K, wl.B, what, cores)},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def k2_apt(B, N, sms=148):
    """anchors per thread the target kernel picks (targets.cu: pick_apt)"""
    ctas = lambda apt: B * ((N + 32 * apt - 1) // (32 * apt))  # noqa: E731
    return 4 if ctas(4) >= 16 * sms else (2 if ctas(2) >= 16 * sms else 1)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tfrpn import _lib
    from tfrpn.proposals import proposal_cfg
    from tfrpn.utils import bbox_utils, train_utils

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # keep stdout clean for the ONE JSON line: libraries (NCCL prints its version) go to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; tfrpn has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    h = _lib.handle(local)

    wl = Workload(args.config, args.c5_k, args.c5_mode)
    rpn = wl.kind == "rpn"
    B, G, N, P = wl.B, wl.G, wl.N, wl.P
    hp = anchors = None
    if rpn:
        hp = wl.hyper_params(train_utils.get_hyper_params)
        anchors = bbox_utils.generate_anchors(hp)
        assert anchors.shape[0] == N
    # LANES independent steps are in flight at a time (consecutive batches do not depend on each other): each
    # lane has its own library handle (= its own workspace), a stream for the target half and a high-priority
    # stream for the proposal half.
    LANES = max(1, min(6, int(os.environ.get("TFRPN_BENCH_LANES", "4"))))
    SETS = wl.n_sets(LANES)
    np_sets = wl.make_inputs(rank, SETS)
    cu = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    sets = []
    for tup in np_sets:
        out = dict(pb=torch.empty((B, P, 4), device=dev), ps=torch.empty((B, P), device=dev),
                   pv=torch.empty((B,), dtype=torch.int32, device=dev),
                   pk=torch.empty((B, P), dtype=torch.int32, device=dev))
        if rpn:
            gtb, gtl, reg, cls = tup
            out.update(gtb=cu(gtb), gtl=cu(gtl), reg=cu(reg), cls=cu(cls),
                       deltas=torch.empty((B, N, 4), device=dev), labels=torch.empty((B, N), device=dev))
        else:
            out.update(boxes=cu(tup[0]), scores=cu(tup[1]), pc=torch.empty((B, P), device=dev))
        sets.append(out)
    set_bytes = sum(t.numel() * t.element_size() for t in sets[0].values())
    reserve_k = PRE_NMS if rpn else (wl.pre or N)
    _lib.check(lib.tfrpn_reserve(h, B, N, max(G, 1), reserve_k))
    pcfg = proposal_cfg(hp, pre_nms_topn=PRE_NMS) if rpn else None
    ncfg = None if rpn else _lib.NmsCfg(P, P, 0.7, float("-inf"), 0, 1, wl.pre)
    handles, mains, sides = [h], [], []
    for _ in range(1, LANES):
        hh = C.c_void_p()
        _lib.check(lib.tfrpn_create(C.byref(hh), local))
        _lib.check(lib.tfrpn_reserve(hh, B, N, max(G, 1), reserve_k))
        handles.append(hh)
    for _ in range(LANES):
        mains.append(torch.cuda.Stream(dev))
        sides.append(torch.cuda.Stream(dev, priority=-1))

    def tcfg(step):
        return train_utils._target_cfg(hp, 2026, step, rank * B)

    def targets(s, step, stream, hh=h):
        _lib.check(lib.tfrpn_rpn_targets(hh, anchors.data_ptr(), s["gtb"].data_ptr(), s["gtl"].data_ptr(), B, N, G,
                                         C.byref(tcfg(step)), s["deltas"].data_ptr(), s["labels"].data_ptr(), None,
                                         stream.cuda_stream))

    def proposals(s, stream, hh=h):
        _lib.check(lib.tfrpn_proposals(hh, s["reg"].data_ptr(), s["cls"].data_ptr(), anchors.data_ptr(), B, N,
                                       C.byref(pcfg), s["pb"].data_ptr(), s["ps"].data_ptr(), s["pv"].data_ptr(),
                                       s["pk"].data_ptr(), stream.cuda_stream))

    def nms(s, stream, hh=h):
        _lib.check(lib.tfrpn_nms(hh, s["boxes"].data_ptr(), s["scores"].data_ptr(), B, N, C.byref(ncfg),
                                 s["pb"].data_ptr(), s["ps"].data_ptr(), s["pc"].data_ptr(), s["pv"].data_ptr(),
                                 s["pk"].data_ptr(), stream.cuda_stream))

    def step_eager(i):
        """One step on lane i % LANES: targets on the lane's stream, proposals concurrently on its side stream."""
        lane = i % LANES
        cur, side, s = mains[lane], sides[lane], sets[i % SETS]
        if not rpn:
            nms(s, cur, handles[lane])
            return
        side.wait_stream(cur)
        targets(s, i, cur, handles[lane])
        proposals(s, side, handles[lane])
        cur.wait_stream(side)

    # eager warm-up (also sets kernel attributes before any capture)
    n0 = _lib.launch_count()
    step_eager(0)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - n0
    for i in range(1, LANES):
        step_eager(i)
    torch.cuda.synchronize()

    graphs = None
    if not args.no_graph:
        graphs = []
        for i in range(SETS):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=mains[i % LANES]):
                step_eager(i)
            graphs.append(g)

    def run_step(i):
        if graphs is not None:
            with torch.cuda.stream(mains[i % LANES]):
                graphs[i % SETS].replay()
        else:
            step_eager(i)
        return mains[i % LANES]

    # EVERY graph is launched before the timed region, whatever --warmup says: the first replay of a graph
    # pays its upload to the device, and a timed step must never be a graph's first launch
    if graphs is not None:
        for _ in range(2):
            for i in range(SETS):
                run_step(i)
            torch.cuda.synchronize()
    W, K = max(args.warmup, 3), max(args.steps, 1)
    for i in range(W):
        run_step(i)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cur0 = torch.cuda.current_stream(dev)
    sampler.start()
    barrier()
    # The first steps are enqueued while the GPU spins in a gate kernel that precedes the start event, so the
    # device never waits for the host inside the timed region (a 20-step region lasts ~1 ms: one scheduling
    # hiccup of the enqueueing thread would otherwise be the measurement).  Exactly K steps lie between e0 and e1.
    torch.cuda._sleep(int(min(K, 100) * 60e-6 * 1.9e9))
    e0.record(cur0)
    for m in mains:
        m.wait_stream(cur0)
    t_host = time.perf_counter()
    for i in range(W, W + K):
        run_step(i)
    t_host = time.perf_counter() - t_host   # host time to ENQUEUE the K steps (no synchronisation inside)
    for m in mains:
        cur0.wait_stream(m)
    e1.record(cur0)
    sampler.sample()                        # the GPU is still working through the queue
    barrier()
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        # the buffers of the last timed step, read now: the passes below write into the same sets
        dump_outputs(args.dump_outputs, sets[(W + K - 1) % SETS], rpn)
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = world * B * K / (ms * 1e-3)

    # ---- p50 single-step latency (device time of ONE step, the GPU idle before and after) ----------
    lat = []
    for i in range(min(K, 200)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        st = mains[i % LANES]
        a.record(st)
        run_step(i)
        b.record(st)
        torch.cuda.synchronize()
        lat.append(a.elapsed_time(b))
    p50 = float(np.median(lat))
    p90 = float(np.percentile(lat, 90))

    # ---- per-kernel device time, live (library tracing hooks, eager launches, rotating sets) ----
    hbm_peak, peak_src = peaks()
    _lib.check(lib.tfrpn_profile_enable(h, 1))
    n_prof = max(8, min(4 * SETS, 96))
    cur_s = torch.cuda.current_stream(dev)
    for i in range(n_prof):          # one stream: kernels are timed without overlapping each other
        if rpn:
            targets(sets[i % SETS], i, cur_s)
            proposals(sets[i % SETS], cur_s)
        else:
            nms(sets[i % SETS], cur_s)
    kern = {}
    for kid in range(_lib.KERNEL_IDS):   # the kernels of the step (ids of include/tfrpn.h)
        tot, n = C.c_double(), C.c_int()
        _lib.check(lib.tfrpn_profile_read(h, kid, C.byref(tot), C.byref(n)))
        if n.value:
            kern[lib.tfrpn_kernel_name(kid).decode()] = 1e3 * tot.value / n.value   # us per launch
    _lib.check(lib.tfrpn_profile_enable(h, 0))
    # algorithmic bytes per launch (DESIGN.md "Kernels"): what each kernel must read and write once
    k_cand = min(PRE_NMS if rpn else (wl.pre or N), N)
    alg = {"proposal_kernel": 4 * B * N + 16 * B * k_cand + 24 * B * P,
           "proposal_cluster_kernel": 4 * B * N + 16 * B * k_cand + 24 * B * P}
    if rpn:
        nparts = (N + 32 * k2_apt(B, N) - 1) // (32 * k2_apt(B, N))   # K2 tiles per image
        alg.update({"rpn_iou_argmax_kernel": 16 * N + 16 * B * G + 4 * B * N + 16 * B * N + 8 * B * nparts * G,
                    "rpn_label_encode_kernel": 4 * B * N + 8 * B * nparts * G + 20 * B * G + 4 * B * N + 16 * B * 128})
    # measured DRAM traffic and warp instructions per launch (one `ncu --set full` capture, summarised by
    # tools/summarize_profiles.py into profiles/traffic.json); null if not captured
    traffic, winstr = {}, {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and args.config == "C2":
        with open(tpath) as f:
            tj = json.load(f)
        traffic = dict(tj.get("dram_bytes_per_launch", {}))
        winstr = dict(tj.get("warp_instr_per_launch", {}))
        # one kernel name covers several launch shapes / modes: take the captured group whose duration is
        # closest to the launch timed here
        for k, us in kern.items():
            gs = tj.get("groups", {}).get(k)
            if gs:
                best = min(gs.values(), key=lambda g: abs(g["avg_us"] - us))
                traffic[k] = best["dram_bytes"]
                if "warp_instr" in best:
                    winstr[k] = best["warp_instr"]
    issue_peak = 148 * 4 * 1.965e9          # warp instructions / s: one per cycle per SM sub-partition
    kernels = []
    for k, v in kern.items():
        row = {"kernel": k, "us_per_launch": v}
        if k in alg:
            row.update({"algorithmic_bytes": alg[k], "achieved_gbs": alg[k] / (v * 1e-6) / 1e9,
                        "frac_hbm": alg[k] / (v * 1e-6) / 1e9 / hbm_peak, "traffic": traffic.get(k)})
        if k in winstr:
            row.update({"warp_instr": winstr[k], "frac_issue": winstr[k] / (v * 1e-6) / issue_peak})
        kernels.append(row)
    dominant = max(kern, key=kern.get)
    dom_us = kern[dominant]
    if dominant in alg:
        achieved = alg[dominant] / (dom_us * 1e-6) / 1e9
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": traffic.get(dominant), "us_per_launch": dom_us,
                    "algorithmic_bytes": alg[dominant], "peak_source": peak_src}
    else:
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s",
                    "frac": None, "traffic": traffic.get(dominant), "us_per_launch": dom_us, "peak_source": peak_src}
    if dominant.startswith("proposal") or dominant == "rpn_label_encode_kernel":
        # SURVEY 8d: these kernels are bound by work (select / sort / greedy NMS per image), not by HBM: the
        # HBM figures above are kept for the contract, the binding roof is instruction issue on the SMs the
        # launch occupies (one CTA, or one cluster of CTAs, per image)
        roofline["note"] = ("not HBM-bound: per-image select / sort / sequential greedy NMS; see `work` for the "
                            "issue-capacity view (warp instructions from the committed ncu capture)")
        cl = 1 if dominant != "proposal_cluster_kernel" else (8 if B <= 8 else 2)      # proposals.cu: pick_cluster
        sms_used = min(148, B * cl)
        work = {"us_per_image_batch": dom_us, "images": B, "us_per_image": dom_us / B, "ctas": B * cl, "sms_used": sms_used}
        if dominant.startswith("proposal") and rpn:
            # NMS work actually scheduled: every round tests its <= 128 candidates against the kept list so far and
            # against each other (sizes from the launch's own results: rank of every kept box)
            s0 = sets[0]
            proposals(s0, cur_s)
            torch.cuda.synchronize()
            keep, valid = s0["pk"].cpu().numpy(), s0["pv"].cpu().numpy()
            sc = s0["cls"].reshape(B, -1).cpu().numpy()
            order = np.argsort(-sc, axis=1, kind="stable")
            rk = np.empty_like(order)
            np.put_along_axis(rk, order, np.arange(N)[None, :].repeat(B, 0), axis=1)
            pairs, examined = 0, []
            for b_ in range(B):
                kr = np.sort(rk[b_][keep[b_][:valid[b_]]])
                last = int(kr[-1]) + 1 if len(kr) else 0
                examined.append(last)
                for lo_ in range(0, last, 128):   # a round tests all of its 128 candidates before it is resolved
                    c_ = min(128, min(N, PRE_NMS) - lo_)
                    pairs += c_ * int(np.searchsorted(kr, lo_)) + c_ * (c_ - 1) // 2
            work.update({"pair_tests_per_launch": int(pairs), "pair_tests_per_s": pairs / (dom_us * 1e-6),
                         "candidates_examined_per_image": float(np.mean(examined))})
        if dominant in winstr:
            floor_us = winstr[dominant] / (sms_used * 4 * 1.965e9) * 1e6
            work.update({"bound": "issue", "warp_instr_per_launch": winstr[dominant],
                         "issue_floor_us_on_sms_used": floor_us, "frac_issue_on_sms_used": floor_us / dom_us,
                         "achieved_gwarp_instr_per_s": winstr[dominant] / (dom_us * 1e-6) / 1e9,
                         "peak_gwarp_instr_per_s": issue_peak / 1e9, "frac": winstr[dominant] / (dom_us * 1e-6) / issue_peak})
        roofline["work"] = work
    # the IoU/argmax kernel is bound by instruction issue, not by HBM.  Two views: SURVEY 8d's model (B*N*G
    # pairs x ~22 lane-instr vs 148 SM x 128 lanes) and the pairs the kernel really evaluates (the zero
    # padding of the GT lists is compacted away before the loop)
    if "rpn_iou_argmax_kernel" in kern:
        alu_peak = 148 * 128 * 1.965e9
        pairs = B * N * G
        real = int(sum(int((s_[1] != -1).sum()) for s_ in np_sets)) / len(np_sets) * N   # anchors x real GT boxes, per step
        t = kern["rpn_iou_argmax_kernel"] * 1e-6
        kernels.append({"kernel": "rpn_iou_argmax_kernel", "bound": "fp32-alu", "pairs": pairs,
                        "achieved_lane_instr_per_s": pairs * 22 / t, "peak_lane_instr_per_s": alu_peak,
                        "frac_alu": pairs * 22 / t / alu_peak,
                        "pairs_evaluated": real, "frac_alu_evaluated": real * 22 / t / alu_peak})

    # ---- the two HBM-bound drop-in kernels (materialised IoU map K1, decode K3), timed alone ----
    def timed_loop(fn, reps):
        """us per launch of `reps` back-to-back launches replayed from ONE CUDA graph (no host launch gaps)."""
        cs = torch.cuda.Stream(dev)
        with torch.cuda.stream(cs):
            for r in range(3):
                fn(r, cs.cuda_stream)
            cs.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=cs):
                for r in range(reps):
                    fn(r, cs.cuda_stream)
            g.replay()
            cs.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(cs)
            for _ in range(3):
                g.replay()
            b.record(cs)
            cs.synchronize()
        return 1e3 * a.elapsed_time(b) / (3 * reps)

    if rpn:
        n_iou = max(3, int(np.ceil(2.1 * L2_BYTES / (4.0 * B * N * G))))       # rotating outputs > L2
        iou_out = [torch.empty((B, N, G), device=dev) for _ in range(n_iou)]
        us = timed_loop(lambda r, cur: _lib.check(lib.tfrpn_iou_map(anchors.data_ptr(), 0, sets[r % SETS]["gtb"].data_ptr(), B, N, G,
                                                                    iou_out[r % n_iou].data_ptr(), cur)), 10 * n_iou)
        by = 4 * B * N * G + 16 * (N + B * G)
        k1_name = "iou_map_pairs_kernel" if G % 2 == 0 else "iou_map_kernel"
        kernels.append({"kernel": k1_name, "us_per_launch": us, "algorithmic_bytes": by, "traffic": traffic.get(k1_name),
                        "achieved_gbs": by / (us * 1e-6) / 1e9, "frac_hbm": by / (us * 1e-6) / 1e9 / hbm_peak})
        del iou_out
        var = (C.c_float * 4)(*hp["variances"])
        reps = max(20, min(10 * SETS, 120))
        us = timed_loop(lambda r, cur: _lib.check(lib.tfrpn_decode(anchors.data_ptr(), 0, sets[r % SETS]["reg"].data_ptr(), var, 1, B, N,
                                                                   sets[r % SETS]["deltas"].data_ptr(), cur)), reps)
        by = 32 * B * N + 16 * N
        kernels.append({"kernel": "decode_kernel", "us_per_launch": us, "algorithmic_bytes": by, "traffic": traffic.get("decode_kernel"),
                        "achieved_gbs": by / (us * 1e-6) / 1e9, "frac_hbm": by / (us * 1e-6) / 1e9 / hbm_peak})
        # the losses that consume the targets (SURVEY 8f rank 1): reads labels + true deltas, predictions only
        # where a term exists; one launch (the last CTA sums the per-CTA partials)
        lout = torch.empty((4,), device=dev)
        us = timed_loop(lambda r, cur: _lib.check(lib.tfrpn_rpn_losses(h, sets[r % SETS]["deltas"].data_ptr(), sets[r % SETS]["reg"].data_ptr(),
                                                                       sets[r % SETS]["labels"].data_ptr(), sets[r % SETS]["cls"].data_ptr(),
                                                                       B, N, 1.0, lout.data_ptr(), None, None, cur)), reps)
        by = 20 * B * N
        kernels.append({"kernel": "rpn_loss_partial_kernel", "traffic": traffic.get("rpn_loss_partial_kernel"), "us_per_launch": us, "algorithmic_bytes": by,
                        "achieved_gbs": by / (us * 1e-6) / 1e9, "frac_hbm": by / (us * 1e-6) / 1e9 / hbm_peak})

    # ---- e2e: host buffers through the public host-buffer API, copies inside the timed region ----
    def wall(fn, n):
        barrier()
        t0 = time.perf_counter()
        fn(n)
        torch.cuda.synchronize()
        t = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([t], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t = float(tt.item())
        return t

    # ---- the optional final gather of targets and proposals (north star: the only NCCL traffic; NOT part of `value`) ----
    final_gather = None
    if world > 1 and rpn:
        from tfrpn import sharding
        s0 = sets[0]
        parts = [s0["deltas"], s0["labels"], s0["pb"], s0["ps"], s0["pv"], s0["pk"]]
        outs_g = [torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=dev) for t in parts]
        for t, o in zip(parts, outs_g):
            sharding.gather_equal(t, o)
        barrier()
        ga, gb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ga.record()
        for _ in range(20):
            for t, o in zip(parts, outs_g):
                sharding.gather_equal(t, o)
        gb.record()
        torch.cuda.synchronize()
        gms = torch.tensor([ga.elapsed_time(gb) / 20], device=dev)
        dist.all_reduce(gms, op=dist.ReduceOp.MAX)
        by = sum(t.numel() * t.element_size() for t in parts)
        final_gather = {"ms_per_step": float(gms.item()), "bytes_per_rank": by, "tensors": 6,
                        "algbw_gbs_per_rank": by * (world - 1) / (float(gms.item()) * 1e-3) / 1e9,
                        "api": "tfrpn.sharding.gather_equal (torch.distributed all_gather_into_tensor, NCCL): dense bbox_deltas, "
                               "bbox_labels and the four proposal tensors of one step; optional, outside `value`"}
        del outs_g

    if rpn:
        e2e = e2e_rpn(args, wl, lib, _lib, h, hp, anchors, np_sets, tcfg, pcfg, wall, world, rank, dev, K)
    else:
        e2e = e2e_nms(wl, np_sets, wall, world, K)

    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": wl.desc, "global_batch": world * B, "parallelism": "images sharded, no collective",
                       "l2": "rotating %d input/output sets (%.0f MB) > 126 MB L2" % (SETS, SETS * set_bytes / 1e6),
                       "launch": ("eager" if graphs is None else "one CUDA graph per step, every graph launched before "
                                  "the timed region; the first timed steps are enqueued behind a gate kernel") +
                                 "; targets || proposals on two streams (proposals high priority); %d independent steps "
                                 "in flight, one library handle each" % LANES},
            "p50_ms": p50, "p90_ms": p90, "host_enqueue_ms_per_step": t_host * 1e3 / K, "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches_per_step * K),
            "roofline": roofline, "kernels": kernels}
    if final_gather is not None:
        line["final_gather"] = final_gather

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import rpn_oracle
        threads = cpu_threads(wl)
        a_np = rpn_oracle.generate_anchors(hp) if rpn else None
        t_cpu, n_img, what = 0.0, 0, ""
        while t_cpu < 10.0 and n_img < 64 * 2000:
            dt, what = cpu_path(wl, np_sets, a_np, hp, threads, B)
            t_cpu += dt
            n_img += B
        line["cpu_baseline"] = {"value": n_img / t_cpu, "unit": "images/s", "cores": threads, "kind": "port",
                                "sample": "%d images (batches of %d) in %.1f s, %s; host has %d cores"
                                          % (n_img, B, t_cpu, what, os.cpu_count() or 1)}
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, s, rpn):
    """Write the arrays a caller of the timed path receives, one DIR/<name>.npy each (float32, integer
    outputs as float64, which holds every int32 exactly).  Every config's outputs fit in 64 MB whole."""
    names = ({"deltas": "bbox_deltas", "labels": "bbox_labels", "pb": "proposal_boxes", "ps": "proposal_scores",
              "pv": "proposal_valid", "pk": "proposal_keep"} if rpn else
             {"pb": "nmsed_boxes", "ps": "nmsed_scores", "pc": "nmsed_classes", "pv": "valid_detections",
              "pk": "keep_indices"})
    os.makedirs(out_dir, exist_ok=True)
    for key, name in names.items():
        a = s[key].cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def e2e_rpn(args, wl, lib, _lib, h, hp, anchors, np_sets, tcfg, pcfg, wall, world, rank, dev, K):
    """HostPipeline (tfrpn_pipeline_* C ABI) with the slots' page-locked blocks as the caller's buffers."""
    import torch
    import tfrpn
    B, G, N, P = wl.B, wl.G, wl.N, wl.P

    def pinned(shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _lib.check(lib.tfrpn_host_alloc(C.byref(p), n))
        buf = (C.c_char * n).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    DEPTH = max(2, min(16, int(os.environ.get("TFRPN_BENCH_DEPTH", "8"))))   # host steps in flight (tfrpn.HostPipeline)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    st = torch.cuda.current_stream(dev).cuda_stream
    pipe = tfrpn.HostPipeline(hp, depth=DEPTH, device=dev, anchors=anchors, pre_nms_topn=PRE_NMS)
    # every slot's page-locked input block holds one synthetic batch (written by the "data loader" once;
    # the H2D copy of those inputs and the D2H copy of the results happen inside every timed step)
    for i in range(DEPTH):
        v = pipe.acquire(B, G)
        gtb, gtl, reg, cls = np_sets[i % len(np_sets)]
        v.gt_boxes[...] = gtb; v.gt_labels[...] = gtl; v.rpn_reg[...] = reg; v.rpn_cls[...] = cls
        pipe.submit(seed=2026, offset=i, image_offset=rank * B)
    pipe.drain()
    hsets = []
    for gtb, gtl, reg, cls in np_sets[:2]:
        d = dict(gtb=pinned(gtb.shape, np.float32), gtl=pinned(gtl.shape, np.int32), reg=pinned(reg.shape, np.float32),
                 cls=pinned(cls.shape, np.float32), deltas=pinned((B, N, 4), np.float32),
                 labels=pinned((B, N), np.float32), pb=pinned((B, P, 4), np.float32), ps=pinned((B, P), np.float32),
                 pv=pinned((B,), np.int32), pk=pinned((B, P), np.int32))
        d["gtb"][...] = gtb; d["gtl"][...] = gtl; d["reg"][...] = reg; d["cls"][...] = cls
        hsets.append(d)

    def sync_step(i):
        s = hsets[i % 2]
        _lib.check(lib.tfrpn_rpn_step_host(h, anchors.data_ptr(), vp(s["gtb"]), vp(s["gtl"]), B, N, G,
                                           C.byref(tcfg(i)), vp(s["deltas"]), vp(s["labels"]), vp(s["reg"]),
                                           vp(s["cls"]), C.byref(pcfg), vp(s["pb"]), vp(s["ps"]), vp(s["pv"]),
                                           vp(s["pk"]), st))

    sink = []

    def pipelined(n, fill=False):
        """n steps: acquire the next slot (its inputs are resident in pinned host memory; with `fill` the
        producer's pageable arrays are copied into the slot inside the loop), submit, and consume the results
        of the step submitted DEPTH-1 steps earlier (a device->host read per step)."""
        tickets = []
        views = []
        for i in range(n):
            if i >= DEPTH - 1:
                pipe.wait(tickets[i - (DEPTH - 1)])
                sink.append(int(views[i - (DEPTH - 1)].valid[0]))
            v = pipe.acquire(B, G)
            if fill:
                gtb, gtl, reg, cls = np_sets[i % len(np_sets)]
                v.gt_boxes[...] = gtb; v.gt_labels[...] = gtl; v.rpn_reg[...] = reg; v.rpn_cls[...] = cls
            views.append(v)
            tickets.append(pipe.submit(seed=2026, offset=i, image_offset=rank * B))
        pipe.drain()

    outs = [dict() for _ in range(DEPTH)]

    def pageable(n):
        """n steps on the producer's own pageable NumPy arrays (HostPipeline.submit_arrays -> tfrpn_pipeline_submit):
        nothing is copied by the caller; results land in pageable arrays too."""
        tickets = []
        for i in range(n):
            if i >= DEPTH - 1:
                pipe.wait(tickets[i - (DEPTH - 1)])
                sink.append(int(outs[(i - (DEPTH - 1)) % DEPTH]["valid"][0]))
            gtb, gtl, reg, cls = np_sets[i % len(np_sets)]
            t, _ = pipe.submit_arrays(gtb, gtl, reg, cls, out=outs[i % DEPTH], seed=2026, offset=i, image_offset=rank * B)
            tickets.append(t)
        pipe.drain()

    # e2e is wall-clock over a pipeline DEPTH steps deep: a 20-step run would mostly measure its fill and drain, so the
    # loop is at least 200 steps long whatever --steps says (the count is reported as e2e.steps)
    Ke = min(max(K, 200), 400)
    pipelined(2 * DEPTH)
    t_e2e = wall(pipelined, Ke)
    h2d_pipe, d2h_pipe = pipe.last_copy_bytes()
    t_fill = wall(lambda n: pipelined(n, True), Ke)
    pipe.set_stable_outputs(True)   # the ring `outs` is written by the pipeline only: no per-step memset of the dense deltas
    pageable(2 * DEPTH)
    t_page = wall(pageable, Ke)
    h2d_page, d2h_page = pipe.last_copy_bytes()
    for i in range(3):
        sync_step(i)
    Ks = min(K, 100)
    t_sync = wall(lambda n: [sync_step(i) for i in range(n)], Ks)
    pipe.close()
    h2d = B * G * 16 + B * G * 4 + B * N * 16 + B * N * 4
    d2h = B * N * 16 + B * N * 4 + B * P * 16 + B * P * 4 + B * 4 + B * P * 4
    return {"value": world * B * Ke / t_e2e, "unit": "images/s", "h2d_bytes_per_step": h2d_pipe, "d2h_bytes_per_step": d2h_pipe,
            "steps": Ke, "ms_per_step": 1e3 * t_e2e / Ke,
            "pcie_gbs_each_way": [h2d_pipe * Ke / t_e2e / 1e9, d2h_pipe * Ke / t_e2e / 1e9],
            "dense_result_bytes_per_step": d2h,
            "api": "tfrpn.HostPipeline acquire/submit/wait (tfrpn_pipeline_* C ABI), %d host steps in flight, inputs and "
                   "results in the slots' page-locked host blocks.  Two-phase input: scores H2D, ranks D2H, the library's "
                   "host threads gather the candidate rows of rpn_reg, rows H2D; bbox_deltas crosses PCIe in compact form "
                   "(its <=128 non-zero rows per image) and wait() scatters it into the dense (B,N,4) host array -- all "
                   "inside the timed region; h2d/d2h bytes are what crossed the link per step" % DEPTH,
            "pageable_arrays": {"value": world * B * Ke / t_page, "ms_per_step": 1e3 * t_page / Ke,
                                "h2d_bytes_per_step": h2d_page, "d2h_bytes_per_step": d2h_page,
                                "api": "HostPipeline.submit_arrays (tfrpn_pipeline_submit): the producer's pageable NumPy "
                                       "arrays in, a ring of pageable dense arrays out (TFRPN_PIPE_OPT_STABLE_OUTPUTS), no copy "
                                       "by the caller"},
            "with_producer_fill": {"value": world * B * Ke / t_fill, "ms_per_step": 1e3 * t_fill / Ke,
                                   "note": "the same loop with the producer's pageable NumPy batch copied into the slot's "
                                           "pinned block inside every step (single-threaded memcpy)"},
            "one_step_at_a_time": {"value": world * B * Ks / t_sync, "ms_per_step": 1e3 * t_sync / Ks,
                                   "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                   "api": "tfrpn_rpn_step_host (synchronous: returns with the dense results in host memory)"}}


def e2e_nms(wl, np_sets, wall, world, K):
    """C5: the drop-in non_max_suppression with NumPy host buffers in and out (copies inside the call)."""
    from tfrpn.utils import bbox_utils
    B, N, P = wl.B, wl.N, wl.P
    ins = [(b.reshape(B, N, 1, 4), s.reshape(B, N, 1)) for b, s in np_sets[:2]]
    kw = dict(max_output_size_per_class=P, max_total_size=P, iou_threshold=0.7)
    if wl.pre:
        kw["pre_nms_topn"] = wl.pre
    sink = []

    def loop(n):
        for i in range(n):
            r = bbox_utils.non_max_suppression(ins[i % 2][0], ins[i % 2][1], **kw)
            sink.append(int(r[3][0]))

    loop(3)
    Ke = min(K, 100)
    t = wall(loop, Ke)
    return {"value": world * B * Ke / t, "unit": "images/s", "h2d_bytes_per_step": B * N * 20,
            "d2h_bytes_per_step": B * P * 24 + B * 4, "steps": Ke, "ms_per_step": 1e3 * t / Ke,
            "api": "tfrpn.utils.bbox_utils.non_max_suppression with NumPy host arrays (pageable): H2D, kernels, D2H "
                   "inside every call"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C4", "C5"])
    ap.add_argument("--c5-k", type=int, default=100000, help="boxes per image of config C5")
    ap.add_argument("--c5-mode", default="topk_nms", choices=["topk_nms", "nms_all"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

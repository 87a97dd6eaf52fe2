"""The box-math kernels (csrc/boxmath.cu) and the loss kernels (csrc/losses.cu) in every launch variant their
launchers select, against the NumPy oracle (oracle/rpn_oracle.py).

tfrpn_iou_map picks iou_map_pairs_kernel<W, 512 or 256>, iou_map_kernel<true> (one column per thread) or
iou_map_kernel<false> (generic) from G, the output pointer's alignment and the grid size; tfrpn_decode picks
decode_kernel<SCALE, CLIP, PT> from the variances, the clip flag and TFRPN_DECODE_PT; tfrpn_scale_boxes runs a
grid-stride loop once n_boxes exceeds its capped grid; tfrpn_rpn_losses reduces one partial per CTA in its last CTA.
Each test first asserts the dispatch condition it is written for (restated from the launchers below), so a policy
change cannot make it silently test another variant.

Bars: IoU, labels, counts and indices bit for bit; decoded boxes within 4 ulp of the magnitude of the operands of
their final add / sub (exp, then a cancelling difference), with NaN and inf exactly where the oracle has them;
scalar losses within 2e-6 relative of the float64 sum of the oracle's float32 terms; gradients bit for bit.  Every
output starts filled with a NaN or -7 sentinel."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32
EPS = float(np.finfo(F32).eps)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMS = 148
EW_GRID_CAP = SMS * 32 * 256          # boxes one pass of scale_boxes_kernel's capped grid covers
LOSS_RTOL = 2e-6
VAR = [0.1, 0.15, 0.2, 0.25]          # every component distinct: a swapped component changes the result


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    from tfrpn import _lib

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.L, ns.lib, ns.dev = torch, _lib, _lib.load(), cuda_device
    ns.cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.np = lambda t: t.detach().cpu().numpy()
    ns.st = lambda: torch.cuda.current_stream(cuda_device).cuda_stream
    return ns


def bits_equal(a, b):
    """same float32 bits, any NaN equal to any NaN"""
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def decoded_close(got, want, scale):
    """NaN / inf exactly where the oracle has them; finite values within 4 ulp of max(|want|, scale)"""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    if got.shape != want.shape or not np.array_equal(np.isnan(got), np.isnan(want)):
        return False
    fin = np.isfinite(want)
    if not np.array_equal(got[~fin & ~np.isnan(want)], want[~fin & ~np.isnan(want)]):
        return False
    mag = np.maximum(np.abs(want), np.nan_to_num(np.asarray(scale, np.float64), nan=0.0, posinf=np.inf))[fin]
    return bool(np.all(np.abs(got[fin] - want[fin]) <= 4 * EPS * np.maximum(mag, 1e-30)))


def rand_boxes(rng, *shape):
    a = np.sort(rng.uniform(0, 1, size=shape + (2, 2)), axis=-2).astype(F32)
    return np.stack([a[..., 0, 0], a[..., 0, 1], a[..., 1, 0], a[..., 1, 1]], axis=-1)


# ------------------------------------------------------------------------------------------------ K1 IoU map
def iou_variant(B, N, G, out_addr, max_w=4):
    """tfrpn_iou_map's launch policy (boxmath.cu), restated"""
    tile = 512 if -(-N // 512) * B >= 8 * SMS else 256
    if max_w >= 4 and G % 4 == 0 and G <= 1024 and out_addr % 16 == 0:
        return "pairs<4,%d>" % tile
    if max_w >= 2 and G % 2 == 0 and G <= 512 and out_addr % 8 == 0:
        return "pairs<2,%d>" % tile
    return "cols" if G <= 128 else "generic"


def oracle_iou(boxes, gt):
    """O.generate_iou_map a few images at a time (bounded temporaries)"""
    B, G = gt.shape[:2]
    N = boxes.shape[-2]
    out = np.empty((B, N, G), F32)
    step = max(1, (1 << 24) // max(1, N * G))
    with np.errstate(invalid="ignore", over="ignore"):
        for b0 in range(0, B, step):
            bx = boxes[b0:b0 + step] if boxes.ndim == 3 else boxes
            out[b0:b0 + step] = O.generate_iou_map(bx, gt[b0:b0 + step])
    return out


def run_iou(T, boxes, gt, offset_floats=0, guard=64, max_w=4):
    """tfrpn_iou_map through the C ABI; out sits offset_floats floats into a -7-filled buffer with guard floats
    after it.  Returns (map, variant, guard bytes intact)."""
    B, G = gt.shape[:2]
    N = boxes.shape[-2]
    b_t, g_t = T.cu(boxes), T.cu(gt)
    n = B * N * G
    buf = T.torch.full((offset_floats + n + guard,), -7.0, device=T.dev)
    ptr = buf.data_ptr() + 4 * offset_floats
    variant = iou_variant(B, N, G, ptr, max_w)
    assert T.lib.tfrpn_iou_map(b_t.data_ptr(), int(boxes.ndim == 3), g_t.data_ptr(), B, N, G, ptr, T.st()) == 0, \
        T.lib.tfrpn_last_error()
    host = T.np(buf)
    intact = bool(np.all(host[:offset_floats] == -7.0) and np.all(host[offset_floats + n:] == -7.0))
    return host[offset_floats:offset_floats + n].reshape(B, N, G), variant, intact


def adversarial_rows(boxes, gt, tile=512):
    """non-nice entries in the second half of 512-row tiles (rows a 256-row staging would miss): a coordinate
    below 2^-16, a zero-area box, NaN, +-inf; a flipped GT box and a GT coordinate below 2^-16"""
    bx = boxes if boxes.ndim == 3 else boxes[None]
    N = bx.shape[1]
    rows = [r for r in (tile + 300, 3 * tile + 450, 5 * tile + 511, 7 * tile + 257, 2 * tile + 256) if r < N]
    vals = [[1e-7, 0.1, 0.3, 0.4], [0.2, 0.2, 0.2, 0.6], [0.1, np.nan, 0.5, 0.6], [0.0, 0.0, np.inf, 0.5],
            [-np.inf, 0.2, 0.3, 0.4]]
    for r, v in zip(rows, vals):
        bx[-1, r] = v
    gt[min(1, gt.shape[0] - 1), 0] = [0.5, 0.5, 0.2, 0.2]
    gt[-1, gt.shape[1] - 1] = [1e-7, 0.1, 0.3, 0.4]


# (id, B, N, G, boxes batched, expected variant): shapes that just meet / just miss ceil(N/512) * B >= 8 * 148, and
# tails N % 512 in {1, 255, 256, 511} at ceil(N/512) * B == 1184
K1_CASES = [
    ("pairs4_512_meets", 74, 7681, 4, False, "pairs<4,512>"),
    ("pairs4_256_misses", 74, 7680, 4, True, "pairs<4,256>"),
    ("pairs2_512_meets", 74, 7681, 6, True, "pairs<2,512>"),
    ("pairs2_256_misses", 74, 7680, 6, False, "pairs<2,256>"),
    ("pairs4_512_tail1", 37, 15873, 8, True, "pairs<4,512>"),
    ("pairs2_512_tail255", 37, 16127, 6, False, "pairs<2,512>"),
    ("pairs4_512_tail256", 37, 16128, 12, False, "pairs<4,512>"),
    ("pairs2_512_tail511", 37, 16383, 10, True, "pairs<2,512>"),
]


@pytest.mark.parametrize("name,B,N,G,batched,variant", K1_CASES, ids=[c[0] for c in K1_CASES])
def test_iou_map_pairs_tiles(T, name, B, N, G, batched, variant):
    """iou_map_pairs_kernel<W, 512> and <W, 256> either side of the grid-size switch, nice and non-nice tiles"""
    rng = np.random.default_rng(B * N + G)
    boxes = rand_boxes(rng, B, N) if batched else rand_boxes(rng, N)
    gt = rand_boxes(rng, B, G)
    gt[0, 0] = 0                                   # padded GT row
    adversarial_rows(boxes, gt)
    got, v, intact = run_iou(T, boxes, gt)
    assert v == variant and intact
    assert bits_equal(got, oracle_iou(boxes, gt))


@pytest.mark.parametrize("cfg,variant", [("C3", "pairs<2,512>"), ("C4", "pairs<4,512>")])
def test_iou_map_bench_shapes(T, cfg, variant):
    """K1 at the shapes bench.py times: C3 (128 x 9216 x 50) and C4 (32 x 37800 x 200), anchors broadcast"""
    from tfrpn import synthetic
    bb, B, G, over = synthetic.CONFIGS[cfg]
    anchors = O.generate_anchors(dict(O.get_hyper_params(bb), **over))
    rng = np.random.default_rng(91)
    gt, _ = synthetic.gt_batch(rng, B, G)
    for b in range(0, B, 2):                       # every other image full
        gt[b] = rand_boxes(rng, G)
    got, v, intact = run_iou(T, anchors, gt)
    assert v == variant and intact
    assert bits_equal(got, oracle_iou(anchors, gt))


# (G, out offset in bytes, N, expected variant): out only 4- or 8-byte aligned
ALIGN_CASES = [(G, off, N, None) for G in (4, 52, 128, 132, 200, 1024, 50, 510) for off in (4, 8) for N in (600,)]
ALIGN_CASES += [(52, 8, 7681, None), (50, 4, 7681, None)]


@pytest.mark.parametrize("G,off,N,_", ALIGN_CASES, ids=["G%d_off%d_N%d" % c[:3] for c in ALIGN_CASES])
def test_iou_map_misaligned_out(T, G, off, N, _):
    """tfrpn_iou_map does not require a 16-byte-aligned out: W = 2 at 8 bytes (G even, G <= 512), else one column
    per thread (G <= 128) or the generic kernel.  The bytes just before and after the map stay untouched."""
    B = 74 if N > 1000 else 3
    rng = np.random.default_rng(G * 10 + off)
    boxes = rand_boxes(rng, B, N) if G % 3 else rand_boxes(rng, N)
    gt = rand_boxes(rng, B, G)
    gt[-1, 1] = 0
    adversarial_rows(boxes, gt)
    got, v, intact = run_iou(T, boxes, gt, offset_floats=off // 4)
    want_v = iou_variant(B, N, G, 256 + off)
    assert v == want_v
    assert v.startswith("pairs<2") if (off == 8 and G <= 512) else v in ("cols", "generic")
    assert intact
    assert bits_equal(got, oracle_iou(boxes, gt))


# ------------------------------------------------------------------------------------------------ K3 decode
def decode_inputs(rng, B, N, batched):
    """anchors (incl. a zero-extent one), deltas ~ N(0, 0.5^2) with NaN, +-inf and exp-overflowing entries"""
    anchors = rand_boxes(rng, B, N) if batched else rand_boxes(rng, N)
    deltas = rng.normal(0, 0.5, size=(B, N, 4)).astype(F32)
    a = anchors if batched else anchors[None]
    a[..., 0, :] = [0.4, 0.4, 0.4, 0.4]
    deltas[:, 0, 2:] = [1000.0, 1000.0]             # 0 * exp(overflow) = NaN, then clip -> 0
    if N > 5:
        deltas[0, 1, 3] = 500.0                     # exp overflows: -inf / inf / NaN corners
        deltas[-1, 2, 2] = -500.0                   # exp underflows to 0
        deltas[0, 3] = [np.nan, 0.1, 0.1, 0.1]
        deltas[-1, 4] = [0.1, np.inf, -np.inf, 0.1]
        deltas[-1, N - 1] = [0.3, np.nan, 0.2, np.nan]
    return anchors, deltas


def oracle_decode(anchors, deltas, var, clip):
    """variances multiplied in float32 first (predictor.py:55), then the decode, then the NaN -> 0 clip"""
    with np.errstate(invalid="ignore", over="ignore"):
        d = (deltas * np.asarray(var, F32)).astype(F32) if var is not None else deltas
        want = O.get_bboxes_from_deltas(anchors, d)
        h = want[..., 2] - want[..., 0]
        w = want[..., 3] - want[..., 1]
        scale = np.stack([np.abs(want[..., 0]) + h, np.abs(want[..., 1]) + w] * 2, -1)
        if clip:
            want = O.clip01(want)
    return want, scale


def run_decode(T, anchors, deltas, var, clip):
    B, N = deltas.shape[:2]
    out = T.torch.full((B, N, 4), float("nan"), device=T.dev)
    a_t, d_t = T.cu(anchors), T.cu(deltas)
    v = (C.c_float * 4)(*var) if var is not None else None
    assert T.lib.tfrpn_decode(a_t.data_ptr(), int(anchors.ndim == 3), d_t.data_ptr(), v, int(clip), B, N,
                              out.data_ptr(), T.st()) == 0, T.lib.tfrpn_last_error()
    return T.np(out)


@pytest.mark.parametrize("batched", [False, True], ids=["anchors_broadcast", "anchors_batched"])
@pytest.mark.parametrize("scale,clip", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["decode_kernel<false,false>", "decode_kernel<true,false>", "decode_kernel<false,true>",
                              "decode_kernel<true,true>"])
def test_decode_variants(T, scale, clip, batched):
    """the four decode_kernel<SCALE, CLIP, 2> variants of tfrpn_decode, N % 512 and N % 1024 tails"""
    assert os.environ.get("TFRPN_DECODE_PT") in (None, "", "2")       # the default PT = 2 build
    rng = np.random.default_rng(int(scale) * 2 + int(clip) + 4 * int(batched))
    var = VAR if scale else None
    for N in (1, 511, 513, 1023, 1025, 1537):
        anchors, deltas = decode_inputs(rng, 3, N, batched)
        got = run_decode(T, anchors, deltas, var, clip)
        want, sc = oracle_decode(anchors, deltas, var, clip)
        assert decoded_close(got, want, sc), N
        if clip:                                  # NaN -> 0, inf -> 1, -inf -> 0
            assert not np.isnan(got).any() and np.array_equal(got[:, 0], np.zeros((3, 4), F32))


@pytest.mark.parametrize("scale,clip", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["decode_gen_kernel<false,false>", "decode_gen_kernel<true,false>",
                              "decode_gen_kernel<false,true>", "decode_gen_kernel<true,true>"])
def test_decode_anchor_cfg_variants(T, scale, clip):
    """the four decode_gen_kernel<SCALE, CLIP, 2> variants of tfrpn_decode_anchor_cfg against the oracle"""
    from tfrpn.utils import bbox_utils
    var = VAR if scale else None
    for hp in (O.get_hyper_params("vgg16"),                                  # N = 8649: N % 512 = N % 1024 = 457
               dict(O.get_hyper_params("vgg16"), feature_map_shape=(13, 17), anchor_scales=[64, 300],
                    anchor_ratios=[1., 3., 0.25], anchor_count=6)):           # N = 1326: tail 302
        anchors = O.generate_anchors(hp)
        rng = np.random.default_rng(anchors.shape[0] + int(scale) + 2 * int(clip))
        B, N = 3, anchors.shape[0]
        _, deltas = decode_inputs(rng, B, N, False)
        deltas[:, 0, 2:] = 1000.0
        out = T.torch.full((B, N, 4), float("nan"), device=T.dev)
        d_t = T.cu(deltas)
        cfg = bbox_utils._anchor_cfg(hp)
        v = (C.c_float * 4)(*var) if var is not None else None
        assert T.lib.tfrpn_decode_anchor_cfg(C.byref(cfg), d_t.data_ptr(), v, int(clip), B, out.data_ptr(), T.st()) == 0
        want, sc = oracle_decode(anchors, deltas, var, clip)
        assert decoded_close(T.np(out), want, sc), N


@pytest.mark.parametrize("cfg", ["C2", "C3", "C4"])
def test_decode_bench_shapes(T, cfg):
    """decode_kernel<true, true, 2> as bench.py times it: broadcast anchors, the config's variances, clip"""
    from tfrpn import synthetic
    bb, B, _, over = synthetic.CONFIGS[cfg]
    hp = dict(O.get_hyper_params(bb), **over)
    anchors = O.generate_anchors(hp)
    N = anchors.shape[0]
    rng = np.random.default_rng(int(cfg[1]))
    reg = rng.normal(0, 2.0, size=(B, N, 4)).astype(F32)
    reg[::7, ::13] = np.nan
    got = run_decode(T, anchors, reg, hp["variances"], True)
    want, sc = oracle_decode(anchors, reg, hp["variances"], True)
    assert not np.isnan(got).any() and decoded_close(got, want, sc)


# ------------------------------------------------------------------------------------------------ per-process switches
def switch_workload(T, max_w, pt):
    """IoU maps and decodes whose variant TFRPN_IOU_W / TFRPN_DECODE_PT change; returns their outputs"""
    rng = np.random.default_rng(2024)
    out = {}
    expect = {(74, 7681, 52): {4: "pairs<4,512>", 2: "pairs<2,512>", 1: "cols"},
              (3, 600, 200): {4: "pairs<4,256>", 2: "pairs<2,256>", 1: "generic"},
              (4, 1000, 50): {4: "pairs<2,256>", 2: "pairs<2,256>", 1: "cols"},
              (2, 300, 4): {4: "pairs<4,256>", 2: "pairs<2,256>", 1: "cols"}}
    for (B, N, G), batched in zip(expect, (False, True, False, True)):
        boxes = rand_boxes(rng, B, N) if batched else rand_boxes(rng, N)
        gt = rand_boxes(rng, B, G)
        adversarial_rows(boxes, gt)
        got, v, intact = run_iou(T, boxes, gt, max_w=max_w)
        assert intact and v == expect[(B, N, G)][max_w]
        out["iou_%d_%d_%d" % (B, N, G)] = got
    assert pt in (1, 2, 4)
    for batched in (False, True):
        for var in (None, VAR):
            for clip in (False, True):
                for N in (1025, 1537, 3):           # N % (256 * PT) tails for PT = 1, 2, 4
                    anchors, deltas = decode_inputs(rng, 2, N, batched)
                    out["dec_%d_%d_%d_%d" % (batched, var is None, clip, N)] = run_decode(T, anchors, deltas, var, clip)
    return out


def child_main(path):
    """entry point of the child process (python -c): the switch workload under the child's environment"""
    import torch
    from tfrpn import _lib

    class Ns:
        pass
    ns = Ns()
    dev = torch.device("cuda:0")
    ns.torch, ns.L, ns.lib, ns.dev = torch, _lib, _lib.load(), dev
    ns.cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ns.np = lambda t: t.detach().cpu().numpy()
    ns.st = lambda: torch.cuda.current_stream(dev).cuda_stream
    pt = int(os.environ.get("TFRPN_DECODE_PT", "2"))
    np.savez(path, **switch_workload(ns, int(os.environ.get("TFRPN_IOU_W", "4")), pt))


@pytest.mark.parametrize("env", [{"TFRPN_IOU_W": "1", "TFRPN_DECODE_PT": "1"}, {"TFRPN_IOU_W": "2", "TFRPN_DECODE_PT": "4"}],
                         ids=["iou_w1_decode_pt1", "iou_w2_decode_pt4"])
def test_ab_switches_bit_identical(T, env, tmp_path):
    """TFRPN_IOU_W and TFRPN_DECODE_PT are read once per process, so a child process runs the other builds
    (iou_map_kernel<true> / <false> and iou_map_pairs_kernel<2, *> for W = 1 / 2; decode_kernel<*, *, 1> and
    <*, *, 4>).  Their outputs must be bit-identical to the default builds' in this process."""
    assert not os.environ.get("TFRPN_IOU_W") and not os.environ.get("TFRPN_DECODE_PT")
    want = switch_workload(T, 4, 2)
    path = str(tmp_path / "child.npz")
    code = ("import sys; sys.path[:0] = %r; import test_boxmath_losses_variants_gpu as m; m.child_main(%r)"
            % ([ROOT, os.path.join(ROOT, "tf-rpn_b200"), os.path.join(ROOT, "tests")], path))
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable] + flags + ["-c", code], env=dict(os.environ, **env), capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    got = dict(np.load(path))
    assert sorted(got) == sorted(want)
    for k in want:
        assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), k


# ------------------------------------------------------------------------------------------------ scale_boxes
def run_scale(T, boxes_t, h, w, denorm):
    out = T.torch.full_like(boxes_t, float("nan"))
    n = boxes_t.numel() // 4
    assert T.lib.tfrpn_scale_boxes(boxes_t.data_ptr(), n, h, w, int(denorm), out.data_ptr(), T.st()) == 0
    return T.np(out)


@pytest.mark.parametrize("n", [1, EW_GRID_CAP - 1, EW_GRID_CAP, EW_GRID_CAP + 1, 5_000_000])
def test_scale_boxes_grid_stride(T, n):
    """scale_boxes_kernel's grid is capped at 148 * 32 CTAs of 256 threads: beyond 1 212 416 boxes its grid-stride
    loop runs a second pass (and a fourth at ~5e6)"""
    assert EW_GRID_CAP == 1212416
    rng = np.random.default_rng(n)
    norm = rng.uniform(-0.1, 1.1, size=(n, 4)).astype(F32)
    pix = (norm * F32(700)).astype(F32)
    for h, w in ((375.0, 500.0), (375.5, 499.25)):
        assert bits_equal(run_scale(T, T.cu(pix), h, w, False), O.normalize_bboxes(pix, h, w))
        assert bits_equal(run_scale(T, T.cu(norm), h, w, True), O.denormalize_bboxes(norm, h, w))


def tie_inputs(h, ks):
    """float32 b with fl(b * h) == k + 0.5 exactly, plus b one ulp either side"""
    out = []
    for k in ks:
        t = k + 0.5
        b0 = F32(t / h)
        for s in range(-4, 5):
            b = b0
            for _ in range(abs(s)):
                b = np.nextafter(b, F32(np.inf if s > 0 else -np.inf), dtype=F32)
            if F32(b * F32(h)) == F32(t):
                out += [np.nextafter(b, F32(-np.inf), dtype=F32), b, np.nextafter(b, F32(np.inf), dtype=F32)]
                break
    return np.asarray(out, F32)


@pytest.mark.parametrize("h,w", [(512.0, 256.0), (375.0, 500.0), (375.5, 499.25)])
def test_denormalize_ties_to_even(T, h, w):
    """denormalize rounds half to even (tf.round, rintf): products landing exactly on k + 0.5, and one ulp either side"""
    ks = list(range(-3, 12)) + [100, 101, 254, 255, 372, 373]
    ty, tx = tie_inputs(h, ks), tie_inputs(w, ks)
    m = min(ty.size, tx.size)
    assert m >= 3 * 15                               # most k have an exact tie at these scales
    boxes = np.stack([ty[:m], tx[:m], ty[:m][::-1], tx[:m][::-1]], -1)
    got = run_scale(T, T.cu(boxes), h, w, True)
    want = O.denormalize_bboxes(boxes, h, w)
    assert bits_equal(got, want)
    prod = (boxes[:, 0] * F32(h)).astype(F32)
    tie = prod == np.floor(prod) + F32(0.5)
    assert tie.sum() >= 15 and np.all(np.fmod(got[tie, 0], 2) == 0)      # ties went to the even neighbour


# ------------------------------------------------------------------------------------------------ NaN through the clip
def test_proposals_clip_nan_regressions(T):
    """the fused proposal stage clips with the NaN -> 0 rule: NaN regressions on top-scoring rows and a zero-extent
    anchor whose exp overflows give the oracle's keep list and boxes"""
    import tfrpn
    from tfrpn import synthetic
    hp = O.get_hyper_params("vgg16")
    anchors = O.generate_anchors(hp)
    anchors[7] = [0.4, 0.4, 0.4, 0.4]
    rng = np.random.default_rng(3)
    B = 4
    reg, cls = synthetic.head_outputs(rng, B, 31, 31, 9)
    reg, cls = reg.reshape(B, -1, 4), cls.reshape(B, -1)
    top = np.argsort(-cls, axis=1)[:, :60]
    for b in range(B):
        reg[b, top[b, b::4], b % 4] = np.nan
    reg[1, top[1, :10]] = np.nan
    reg[:, 7, 2:] = 1000.0
    cls[:, 7] = 1.0
    pb, ps, pv, pk = tfrpn.generate_proposals(T.cu(reg), T.cu(cls), T.cu(anchors), hp, pre_nms_topn=6000)
    with np.errstate(invalid="ignore", over="ignore"):
        ob, os_, ov, ok = O.generate_proposals(reg, cls, anchors, hp, pre_nms_topn=6000)
    assert np.array_equal(T.np(pv), ov) and np.array_equal(T.np(pk), ok)
    assert bits_equal(T.np(ps), os_)
    assert not np.isnan(T.np(pb)).any() and decoded_close(T.np(pb), ob, 1.0)
    assert np.all(ok[:, 0] == 7) and np.array_equal(T.np(pb)[:, 0], np.zeros((B, 4), F32))


@pytest.mark.parametrize("q", [1, 3])
def test_nms_multiclass_clip_boxes_nan(T, q):
    """tfrpn_nms_multiclass and tfrpn_nms with clip_boxes on NaN boxes: a NaN coordinate leaves as 0, bit for bit"""
    rng = np.random.default_rng(q)
    B, K, Cn = 3, 400, 3
    boxes = rand_boxes(rng, B, K, q) * F32(1.2) - F32(0.1)
    boxes = boxes.astype(F32)
    boxes[0, ::5, :, 0] = np.nan
    boxes[1, ::7] = np.nan
    boxes[2, 1::3, :, 3] = np.nan
    scores = rng.uniform(size=(B, K, Cn)).astype(F32)
    cfg = T.L.NmsCfg(50, 100, 0.5, float("-inf"), 0, 1, 0)
    outs = [T.torch.full((B, 100, 4), float("nan"), device=T.dev), T.torch.full((B, 100), float("nan"), device=T.dev),
            T.torch.full((B, 100), float("nan"), device=T.dev), T.torch.full((B,), -7, dtype=T.torch.int32, device=T.dev),
            T.torch.full((B, 100), -7, dtype=T.torch.int32, device=T.dev)]
    b_t, s_t = T.cu(boxes), T.cu(scores)
    h = T.L.handle(T.dev.index)
    assert T.lib.tfrpn_nms_multiclass(h, b_t.data_ptr(), q, s_t.data_ptr(), B, K, Cn, C.byref(cfg),
                                      *[o.data_ptr() for o in outs], T.st()) == 0, T.lib.tfrpn_last_error()
    got = [T.np(o) for o in outs]
    with np.errstate(invalid="ignore"):
        want = O.combined_non_max_suppression(boxes, scores, 50, 100, 0.5, return_indices=True)
    assert not np.isnan(got[0]).any()
    assert np.array_equal(got[3], want[3]) and np.array_equal(got[4], want[4])
    for g, w in zip(got[:3], want[:3]):
        assert np.array_equal(np.ascontiguousarray(g).view(np.uint32), np.ascontiguousarray(w).view(np.uint32))
    if q == 1:                                     # the single-class entry point, same rule
        b1, s1 = T.cu(boxes[:, :, 0]), T.cu(scores[:, :, :1])
        outs1 = [o.clone().fill_(-7) for o in outs]
        assert T.lib.tfrpn_nms(h, b1.data_ptr(), s1.data_ptr(), B, K, C.byref(cfg), *[o.data_ptr() for o in outs1],
                               T.st()) == 0
        with np.errstate(invalid="ignore"):
            w1 = O.combined_non_max_suppression(boxes, scores[:, :, :1], 50, 100, 0.5, return_indices=True)
        assert np.array_equal(T.np(outs1[4]), w1[4]) and np.array_equal(T.np(outs1[0]).view(np.uint32), w1[0].view(np.uint32))


# ------------------------------------------------------------------------------------------------ losses
def loss_close(got, want, rtol=LOSS_RTOL):
    got, want = float(got), float(want)
    return (np.isnan(got) and np.isnan(want)) or abs(got - want) <= rtol * max(abs(want), 1e-30)


def new_handle(T):
    h = C.c_void_p()
    T.L.check(T.lib.tfrpn_create(C.byref(h), T.dev.index or 0))
    return h


def run_losses(T, h, td, pd, tl, ps, B, N, delta, grads, stream=None):
    """tfrpn_rpn_losses on device tensors (None = not passed); out and the gradients prefilled with NaN.
    Returns (reg, cls, n_pos, n_cls, out bytes, grad_deltas, grad_scores)."""
    torch = T.torch
    out = torch.full((4,), float("nan"), device=T.dev)
    gd = torch.full_like(pd, float("nan")) if (grads and td is not None) else None
    gl = torch.full_like(ps, float("nan")) if (grads and tl is not None) else None
    p = lambda t: t.data_ptr() if t is not None else None
    rc = T.lib.tfrpn_rpn_losses(h, p(td), p(pd), p(tl), p(ps), B, N, delta, out.data_ptr(), p(gd), p(gl),
                                stream if stream is not None else T.st())
    assert rc == 0, T.lib.tfrpn_last_error()
    o = T.np(out)
    cnt = o.view(np.int32)
    return (o[0], o[1], int(cnt[2]), int(cnt[3]), o.tobytes(), None if gd is None else T.np(gd),
            None if gl is None else T.np(gl))


def loss_inputs(rng, B, N, delta):
    """RPN-like targets (~3 % labelled, ~1.5 % positive rows) plus the edges: p at eps, 1 - eps and their
    neighbours, 0 and 1; |e| == delta exactly and e == +-0 inside positive rows"""
    tl = np.full((B, N), -1.0, F32)
    lab = rng.uniform(size=(B, N)) < 0.03
    tl[lab] = rng.integers(0, 2, size=int(lab.sum())).astype(F32)
    ps = rng.uniform(size=(B, N)).astype(F32)
    td = np.zeros((B, N, 4), F32)
    pos = rng.uniform(size=(B, N)) < 0.015
    td[pos] = rng.normal(0, 1, size=(int(pos.sum()), 4)).astype(F32)
    pd = rng.normal(0, 1.5, size=(B, N, 4)).astype(F32)
    eps = F32(1e-7)
    hi = F32(1) - eps
    edge = [eps, np.nextafter(eps, F32(0)), np.nextafter(eps, F32(1)), hi, np.nextafter(hi, F32(0)),
            np.nextafter(hi, F32(2)), F32(0), F32(1)]
    flat_t, flat_p = tl.reshape(-1), ps.reshape(-1)
    n = min(flat_t.size, 2 * len(edge))
    flat_p[:n] = np.resize(np.asarray(edge, F32), n)
    flat_t[:n] = np.resize(np.asarray([1, 0], F32), n)
    d = F32(delta)
    rows = td.reshape(-1, 4)
    prd = pd.reshape(-1, 4)
    m = min(rows.shape[0], 6)
    rows[:m] = F32(0.25)
    rows[:m, 3] = F32(0)                           # e == 0 - 0 with pred -0: e == -0; pred +0: e == +0
    prd[:m] = [F32(0.25) + d, F32(0.25) - d, F32(0.25), F32(-0.0)]
    prd[:m:2, 3] = F32(0.0)
    prd[1:m:3, 0] = F32(0.25) + np.nextafter(d, F32(0))
    return td, pd, tl, ps


def oracle_losses(td, pd, tl, ps, delta):
    with np.errstate(invalid="ignore", divide="ignore"):
        gd, gl = O.loss_grads(td, pd, tl, ps, delta)
        return O.reg_loss(td, pd, delta), O.cls_loss(tl, ps), gd, gl


@pytest.mark.parametrize("grads", [False, True], ids=["no_grads", "grads"])
@pytest.mark.parametrize("mode", ["both", "labels_only", "deltas_only"])
@pytest.mark.parametrize("delta", [0.5, 1.0, 3.0])
def test_losses_delta_and_partial_calls(T, delta, mode, grads):
    """rpn_loss_partial_kernel / rpn_loss_grad_kernel with huber_delta passed through, each loss alone or both"""
    rng = np.random.default_rng(int(delta * 10) + len(mode))
    B, N = 3, 5003
    td, pd, tl, ps = loss_inputs(rng, B, N, delta)
    reg, cls, gd, gl = oracle_losses(td, pd, tl, ps, delta)
    use_d, use_l = mode != "labels_only", mode != "deltas_only"
    t = [T.cu(x) if u else None for x, u in ((td, use_d), (pd, use_d), (tl, use_l), (ps, use_l))]
    r_reg, r_cls, npos, ncls, _, r_gd, r_gl = run_losses(T, T.L.handle(T.dev.index), *t, B, N, delta, grads)
    if use_d:
        assert loss_close(r_reg, reg) and npos == int(np.any(td != 0, axis=-1).sum())
    else:
        assert r_reg == 0.0 and npos == 0
    if use_l:
        assert loss_close(r_cls, cls) and ncls == int((tl != -1).sum())
    else:
        assert r_cls == 0.0 and ncls == 0
    if grads:
        assert (r_gd is not None) == use_d and (r_gl is not None) == use_l
        if use_d:
            assert bits_equal(r_gd, gd)
            e = (pd - td)[np.any(td != 0, axis=-1)]
            assert (np.abs(e) > delta).any() and (np.abs(e) == F32(delta)).any() and (e == 0).any()
        if use_l:
            assert bits_equal(r_gl, gl)


def test_losses_nan_labels_and_true_deltas(T):
    """a NaN label is != -1, so it counts as a labelled entry (NaN loss, NaN gradient inside the clip range); a row
    with a NaN true delta is != 0, so it counts as positive (NaN loss); its NaN error takes the -delta branch of the
    Huber gradient, since both |e| <= delta and e > 0 are false"""
    rng = np.random.default_rng(8)
    B, N = 2, 3000
    td, pd, tl, ps = loss_inputs(rng, B, N, 1.0)
    tl[0, 100] = np.nan
    ps[0, 100] = 0.5
    tl[1, 7] = np.nan
    ps[1, 7] = 0.0                                  # outside the clip range: gradient 0
    td[1, 200] = [np.nan, 0, 0, 0]
    reg, cls, gd, gl = oracle_losses(td, pd, tl, ps, 1.0)
    r_reg, r_cls, npos, ncls, _, r_gd, r_gl = run_losses(T, T.L.handle(T.dev.index), T.cu(td), T.cu(pd), T.cu(tl),
                                                         T.cu(ps), B, N, 1.0, True)
    assert np.isnan(r_reg) and np.isnan(r_cls) and np.isnan(reg) and np.isnan(cls)
    assert npos == int(np.any(td != 0, axis=-1).sum()) and ncls == int((tl != -1).sum())
    assert bits_equal(r_gd, gd) and bits_equal(r_gl, gl)
    assert np.isnan(r_gl[0, 100]) and r_gl[1, 7] == 0 and r_gd[1, 200, 0] == -(F32(1) / F32(npos))


@pytest.mark.parametrize("total", [1, 255, 1023, 1024, 1025, 262145, 1 << 27])
def test_losses_sizes_and_reduction(T, total):
    """B * N from 1 up to 2^27 entries (131 072 per-CTA partials summed by the last CTA); at the largest size the
    result is bit-identical over three runs and over two handles"""
    torch = T.torch
    B = 4 if total % 4 == 0 and total >= 1024 else 1
    N = total // B
    g = torch.Generator(device=T.dev)
    g.manual_seed(total)
    tl = torch.full((B, N), -1.0, device=T.dev)
    lab = torch.rand((B, N), generator=g, device=T.dev) < 0.03
    tl[lab] = (torch.rand((B, N), generator=g, device=T.dev)[lab] < 0.5).float()
    ps = torch.rand((B, N), generator=g, device=T.dev)
    td = torch.zeros((B, N, 4), device=T.dev)
    pos = torch.rand((B, N), generator=g, device=T.dev) < 0.015
    if total <= 1025:
        lab[0, 0] = pos[0, 0] = True
        tl[0, 0] = 1.0
    td[pos] = torch.randn((int(pos.sum()), 4), generator=g, device=T.dev)
    pd = torch.randn((B, N, 4), generator=g, device=T.dev) * 1.5
    ctas = -(-total // 1024)
    assert ctas == max(1, total // 1024 + (total % 1024 > 0))
    h = T.L.handle(T.dev.index)
    r = run_losses(T, h, td, pd, tl, ps, B, N, 1.0, False)
    tl_h, ps_h = T.np(tl).reshape(-1), T.np(ps).reshape(-1)
    m = tl_h != -1
    pos_h = T.np(pos)
    td_p, pd_p = T.np(td[pos]), T.np(pd[pos])
    assert loss_close(r[0], O.reg_loss(td_p[None], pd_p[None])) and r[2] == int(pos_h.sum())
    assert loss_close(r[1], O.cls_loss(tl_h[m], ps_h[m])) and r[3] == int(m.sum())
    if total == 1 << 27:
        assert ctas == 131072
        h2 = new_handle(T)
        try:
            runs = [run_losses(T, h, td, pd, tl, ps, B, N, 1.0, False)[4] for _ in range(2)]
            runs.append(run_losses(T, h2, td, pd, tl, ps, B, N, 1.0, False)[4])
        finally:
            T.lib.tfrpn_destroy(h2)
        assert all(x == r[4] for x in runs)


def test_losses_ticket_reset_over_50_calls(T):
    """the last CTA resets the handle's ticket: 50 back-to-back calls on one handle, with grid sizes changing from
    call to call and out refilled with NaN each time, all give the oracle's results"""
    rng = np.random.default_rng(50)
    sets = []
    for N in (1000, 300000, 7, 70000, 1):
        td, pd, tl, ps = loss_inputs(rng, 1, N, 1.0)
        tl[0, 0], ps[0, 0] = 1.0, 0.25
        td[0, 0] = [0.5, 0, 0, 0]
        sets.append(([T.cu(x) for x in (td, pd, tl, ps)], N, oracle_losses(td, pd, tl, ps, 1.0)))
    h = new_handle(T)
    try:
        for i in range(50):
            t, N, (reg, cls, _, _) = sets[i % len(sets)]
            r = run_losses(T, h, *t, 1, N, 1.0, False)
            assert loss_close(r[0], reg) and loss_close(r[1], cls), i
    finally:
        T.lib.tfrpn_destroy(h)


def test_losses_graph_capture_and_replay(T):
    """a captured tfrpn_rpn_losses (with gradients) replayed 5 times over changing inputs equals 5 direct calls"""
    torch = T.torch
    rng = np.random.default_rng(77)
    B, N = 4, 20000
    data = [loss_inputs(rng, B, N, 0.5) for _ in range(5)]
    h = new_handle(T)
    try:
        td, pd, tl, ps = [T.cu(x) for x in data[0]]
        out = torch.empty((4,), device=T.dev)
        gd, gl = torch.empty_like(pd), torch.empty_like(ps)
        s = torch.cuda.Stream(T.dev)
        call = lambda st: T.lib.tfrpn_rpn_losses(h, td.data_ptr(), pd.data_ptr(), tl.data_ptr(), ps.data_ptr(), B, N,
                                                 0.5, out.data_ptr(), gd.data_ptr(), gl.data_ptr(), st)
        assert call(T.st()) == 0                     # sizes the workspace before the capture
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            assert call(s.cuda_stream) == 0
        replayed = []
        for x in data:
            for dst, src in zip((td, pd, tl, ps), x):
                dst.copy_(T.cu(src))
            out.fill_(float("nan")); gd.fill_(float("nan")); gl.fill_(float("nan"))
            graph.replay()
            torch.cuda.synchronize()
            replayed.append((T.np(out).tobytes(), T.np(gd), T.np(gl)))
        for x, (ob, g1, g2) in zip(data, replayed):
            r = run_losses(T, h, *[T.cu(v) for v in x], B, N, 0.5, True)
            assert r[4] == ob and bits_equal(r[5], g1) and bits_equal(r[6], g2)
            reg, cls, wgd, wgl = oracle_losses(*x, 0.5)
            assert loss_close(r[0], reg) and loss_close(r[1], cls) and bits_equal(g1, wgd) and bits_equal(g2, wgl)
        del graph
    finally:
        torch.cuda.synchronize()
        T.lib.tfrpn_destroy(h)


def test_losses_empty_batch(T):
    """B = 0: reg_loss 0 / max(1, 0) = 0, cls_loss 0 / 0 = NaN, no rows counted, gradients untouched"""
    torch = T.torch
    buf = torch.zeros((64,), device=T.dev)
    gbuf = torch.full((64,), -7.0, device=T.dev)
    out = torch.full((4,), -7.0, device=T.dev)
    p = buf.data_ptr()
    assert T.lib.tfrpn_rpn_losses(T.L.handle(T.dev.index), p, p, p, p, 0, 100, 1.0, out.data_ptr(), gbuf.data_ptr(),
                                  gbuf.data_ptr(), T.st()) == 0
    o = T.np(out)
    assert o[0] == 0.0 and np.isnan(o[1]) and o.view(np.int32)[2] == 0 and o.view(np.int32)[3] == 0
    assert np.isnan(O.cls_loss(np.zeros(0, F32), np.zeros(0, F32)))
    assert np.all(T.np(gbuf) == -7.0)


# ------------------------------------------------------------------------------------------------ 64-bit offsets
def need_free(T, nbytes):
    free, _ = T.torch.cuda.mem_get_info(T.dev)
    if free < nbytes:
        pytest.skip("needs %.1f GB of free device memory, %.1f GB free" % (nbytes / 1e9, free / 1e9))


def test_iou_map_past_2_pow_32_elements(T):
    """an IoU map of B * N * G > 2^32 elements (17 GB): the images past element 2^31 and across 2^32 against the
    oracle, rows around each boundary and at the ends; no element left unwritten"""
    B, N, G = 4, 1_050_000, 1024
    n = B * N * G
    assert n > 1 << 32
    need_free(T, 5 * n + (2 << 30))                 # the map and isnan's mask
    torch = T.torch
    rng = np.random.default_rng(64)
    boxes = rand_boxes(rng, B, N)
    gt = rand_boxes(rng, B, G)
    b_t, g_t = T.cu(boxes), T.cu(gt)
    out = torch.full((B, N, G), float("nan"), device=T.dev)
    assert iou_variant(B, N, G, out.data_ptr()) == "pairs<4,512>"
    assert T.lib.tfrpn_iou_map(b_t.data_ptr(), 1, g_t.data_ptr(), B, N, G, out.data_ptr(), T.st()) == 0
    assert not bool(torch.isnan(out).any())
    for b in (2, 3):                                 # image 2 starts past 2^31, image 3 crosses 2^32
        rows = {0, N - 1}
        for bound in (1 << 31, 1 << 32):
            r = (bound - b * N * G) // G
            if 0 <= r < N:
                rows.update(range(max(0, r - 600), min(N, r + 600)))
        rows.update(range(N - 600, N))
        rows.update(rng.integers(0, N, size=2000).tolist())
        idx = np.asarray(sorted(rows))
        got = T.np(out[b, torch.from_numpy(idx).to(T.dev)])
        assert bits_equal(got, O.generate_iou_map(boxes[b, idx][None], gt[b:b + 1])[0]), b
    del out
    torch.cuda.empty_cache()


def test_losses_labels_only_past_2_pow_31_entries(T):
    """a labels-only loss (with its gradient) over 2^31 + 2^20 entries: every labelled entry lies past 2^31 - 2^20,
    so the oracle sums only those"""
    B, N = 2049, 1 << 20
    total = B * N
    assert total == (1 << 31) + (1 << 20)
    need_free(T, 3 * 4 * total + (1 << 30))
    torch = T.torch
    g = torch.Generator(device=T.dev)
    g.manual_seed(31)
    tl = torch.full((B, N), -1.0, device=T.dev)
    ps = torch.rand((B, N), generator=g, device=T.dev)
    tail = 2 * N                                     # the last two images: elements from 2^31 - 2^20 on
    lab = torch.rand((tail,), generator=g, device=T.dev) < 0.25
    tl.view(-1)[-tail:] = torch.where(lab, (torch.rand((tail,), generator=g, device=T.dev) < 0.5).float(),
                                      torch.full((tail,), -1.0, device=T.dev))
    tl.view(-1)[-1] = 1.0
    gl = torch.full((B, N), float("nan"), device=T.dev)
    out = torch.full((4,), float("nan"), device=T.dev)
    assert T.lib.tfrpn_rpn_losses(T.L.handle(T.dev.index), None, None, tl.data_ptr(), ps.data_ptr(), B, N, 1.0,
                                  out.data_ptr(), None, gl.data_ptr(), T.st()) == 0
    o = T.np(out)
    tl_h, ps_h = T.np(tl.view(-1)[-tail:]), T.np(ps.view(-1)[-tail:])
    m = tl_h != -1
    assert o.view(np.int32)[3] == int(m.sum()) and o[0] == 0.0
    assert loss_close(o[1], O.cls_loss(tl_h[m], ps_h[m]))
    assert not bool(gl.view(-1)[:-tail].any()) and not bool(torch.isnan(gl).any())
    with np.errstate(invalid="ignore", divide="ignore"):
        _, want = O.loss_grads(np.zeros((1, 1, 4), F32), np.zeros((1, 1, 4), F32), tl_h, ps_h)
    # loss_grads divides by the count of ITS labelled entries, which are all the labelled entries
    assert bits_equal(T.np(gl.view(-1)[-tail:]), want)
    del tl, ps, gl
    torch.cuda.empty_cache()

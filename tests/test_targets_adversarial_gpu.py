"""RPN target assignment (tfrpn_rpn_targets, _compact, _sparse) on the inputs where its kernels branch, against the C
oracle (oracle/rpn_oracle.c) and, where the IoU map is small, the NumPy oracle.

  * rpn_iou_argmax_kernel's any-input warp (k2_exact_warp): pixel coordinates, tiny coordinates, flipped boxes,
    NaN / inf, zero-area anchors, NaN columns (oracle/target_layouts.py), at every APT, packed and scalar;
  * images whose tiles mix the nice path and the any-input warp, so the label kernel merges partial keys of both;
  * per-GT ties placed across CTA boundaries, lane boundaries and inside one lane's slots, at IoU 1, at an interior
    value and at 0, on both paths: the lowest anchor index wins;
  * every rpn_label_encode_kernel variant (<9>, <12>, <0>), the candidate list either side of its shared-memory
    limit, the per-GT partial grouping GR = min(1024 / G, 32) and the G > 1024 shared-atomic path up to the largest
    G the plan supports;
  * sampling extremes: zero quotas, every anchor a candidate (multi-trip encode loop, radix select over a full-N
    list), quotas around the candidate count, thresholds an IoU attains exactly, offsets above 2^32;
  * run-to-run determinism of the atomics path and of the full-N selection.

Bars: labels, argmax_row, argmax_col, max_iou (bits, including the sign of zero), pos_pre / neg_pre and the counts
bit-exact; deltas dy / dx bit-exact, dh / dw within 4 ulp (one logf), NaN where the oracle has NaN.  Every output is
filled with a sentinel (NaN or -7) before the launch, so an entry the kernels never write fails too.
"""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import rpn_oracle as O
from oracle import target_layouts as TL

pytestmark = pytest.mark.gpu
F32 = np.float32
EPS = float(np.finfo(F32).eps)
SENT = -7
ERR_UNSUPPORTED = -5
LBL_THREADS = 1024
NUMPY_MAX_PAIRS = 1_000_000
VARIANTS = [(1, False), (1, True), (2, False), (2, True), (4, False), (4, True), (8, False), (8, True)]
VARIANT_IDS = ["apt%d%s" % (a, "_scalar" if s else "") for a, s in VARIANTS]


def bits(a):
    return np.ascontiguousarray(a, F32).view(np.uint32)


def within_ulps(a, b, ulps=4):
    a64, b64 = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return bool(np.all(np.abs(a64 - b64) <= ulps * EPS * np.maximum(np.abs(b64), 1e-30)))


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    from tfrpn import _lib, synthetic
    from tfrpn.utils import train_utils
    if not CO.available():
        pytest.skip("oracle/_build/librpn_oracle.so not built (python -c 'import __graft_entry__ as g; g.build()')")

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.train, ns.dev, ns.lib, ns.syn = torch, train_utils, cuda_device, _lib, synthetic
    ns.cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.handles = {}
    yield ns
    for h in ns.handles.values():
        _lib.load().tfrpn_destroy(h)


def fresh_handle(T, **env):
    """a library handle created with A/B switches set (they are read once, by tfrpn_create)"""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        h = C.c_void_p()
        T.lib.check(T.lib.load().tfrpn_create(C.byref(h), T.dev.index or 0))
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return h


def handle(T, apt=None, scalar=False):
    """one handle per A/B switch for the whole module; apt None = the launcher's own choice"""
    key = (apt, scalar)
    if key not in T.handles:
        env = {}
        if apt is not None:
            env["TFRPN_K2_APT"] = apt
        if scalar:
            env["TFRPN_K2_SCALAR"] = 1
        T.handles[key] = fresh_handle(T, **env)
    return T.handles[key]


def make_hp(N, pos_thr=0.7, neg_thr=0.3, total_pos=128, total_neg=128):
    hp = dict(O.get_hyper_params("vgg16"), feature_map_shape=(1, N), pos_iou_threshold=pos_thr,
              neg_iou_threshold=neg_thr)
    hp["anchor_count"] = 1
    hp["total_pos_bboxes"], hp["total_neg_bboxes"] = total_pos, total_neg
    return hp


def launch(T, h, anchors, gtb, gtl, hp, seed, offset, image_offset=0, form="dense"):
    """one call of the C ABI on sentinel-filled outputs; returns (rc, numpy outputs)"""
    torch = T.torch
    B, G = gtl.shape
    N = anchors.shape[0]
    TP, Q = int(hp["total_pos_bboxes"]), int(hp["total_pos_bboxes"]) + int(hp["total_neg_bboxes"])
    cfg = T.train._target_cfg(hp, seed, offset, image_offset)
    a_t, g_t, l_t = T.cu(anchors), T.cu(gtb), T.cu(gtl)
    dev, nan = T.dev, float("nan")
    i32 = dict(dtype=torch.int32, device=dev)
    lib = T.lib.load()
    st = torch.cuda.current_stream(dev).cuda_stream
    out = {}
    if form == "dense":
        out["deltas"] = torch.full((B, N, 4), nan, device=dev)
        out["labels"] = torch.full((B, N), nan, device=dev)
        out.update(argmax_row=torch.full((B, N), SENT, **i32), argmax_col=torch.full((B, G), SENT, **i32),
                   max_iou=torch.full((B, N), nan, device=dev),
                   pos_pre=torch.full((B, N), SENT & 0xFF, dtype=torch.uint8, device=dev),
                   neg_pre=torch.full((B, N), SENT & 0xFF, dtype=torch.uint8, device=dev),
                   pos_count=torch.full((B,), SENT, **i32), neg_count=torch.full((B,), SENT, **i32))
        dbg = T.lib.TargetDebug(*[out[k].data_ptr() for k in ("argmax_row", "argmax_col", "max_iou", "pos_pre",
                                                               "neg_pre", "pos_count", "neg_count")])
        rc = lib.tfrpn_rpn_targets(h, a_t.data_ptr(), g_t.data_ptr(), l_t.data_ptr(), B, N, G, C.byref(cfg),
                                   out["deltas"].data_ptr(), out["labels"].data_ptr(), C.byref(dbg), st)
    else:
        out["pos_idx"] = torch.full((B, max(TP, 1)), SENT, **i32)
        out["pos_deltas"] = torch.full((B, max(TP, 1), 4), nan, device=dev)
        if form == "compact":
            out["labels"] = torch.full((B, N), nan, device=dev)
            rc = lib.tfrpn_rpn_targets_compact(h, a_t.data_ptr(), g_t.data_ptr(), l_t.data_ptr(), B, N, G, C.byref(cfg),
                                               out["labels"].data_ptr(), out["pos_idx"].data_ptr(),
                                               out["pos_deltas"].data_ptr(), st)
        else:
            out["codes"] = torch.full((B, max(Q, 1)), SENT, **i32)
            rc = lib.tfrpn_rpn_targets_sparse(h, a_t.data_ptr(), g_t.data_ptr(), l_t.data_ptr(), B, N, G, C.byref(cfg),
                                              out["codes"].data_ptr(), out["pos_idx"].data_ptr(),
                                              out["pos_deltas"].data_ptr(), st)
        out["pos_idx"], out["pos_deltas"] = out["pos_idx"][:, :TP], out["pos_deltas"][:, :TP]
        if "codes" in out:
            out["codes"] = out["codes"][:, :Q]
    torch.cuda.synchronize()
    return rc, {k: v.cpu().numpy() for k, v in out.items()}


def assert_deltas(d, od):
    """dy / dx bit-exact, dh / dw within 4 ulp, NaN exactly where the oracle has NaN"""
    nan = np.isnan(od)
    assert np.array_equal(np.isnan(d), nan)
    dd, oo = d[..., :2][~nan[..., :2]], od[..., :2][~nan[..., :2]]
    assert np.array_equal(bits(dd), bits(oo))
    dd, oo = d[..., 2:][~nan[..., 2:]], od[..., 2:][~nan[..., 2:]]
    same = dd == oo
    assert within_ulps(dd[~same], oo[~same], 4)


def check_dense(got, ref, npref=None):
    od, ol, odbg = ref
    assert np.array_equal(bits(got["labels"]), bits(ol))
    assert np.array_equal(got["argmax_col"], odbg["argmax_col"])
    assert np.array_equal(got["argmax_row"], odbg["argmax_row"])
    assert np.array_equal(bits(got["max_iou"]), bits(odbg["max_iou"]))
    assert np.array_equal(got["pos_pre"], odbg["pos_pre"]) and np.array_equal(got["neg_pre"], odbg["neg_pre"])
    assert np.array_equal(got["pos_count"], (ol == 1).sum(-1)) and np.array_equal(got["neg_count"], (ol == 0).sum(-1))
    assert_deltas(got["deltas"], od)
    if npref is not None:   # NumPy oracle: its max reduction may pick either zero (test_oracle_cross.py), compare values
        nd, nl, ndbg = npref
        assert np.array_equal(got["labels"], nl.reshape(ol.shape))
        assert np.array_equal(got["argmax_col"], ndbg["argmax_col"]) and np.array_equal(got["argmax_row"], ndbg["argmax_row"])
        assert np.array_equal(got["max_iou"], ndbg["max_iou"])
        assert np.array_equal(got["pos_pre"].astype(bool), ndbg["pos_pre"])
        assert np.array_equal(got["neg_pre"].astype(bool), ndbg["neg_pre"])


def check_compact(got, ref, TP):
    od, ol = ref[0], ref[1]
    assert np.array_equal(bits(got["labels"]), bits(ol))
    check_rows(got, od, ol, TP)


def check_rows(got, od, ol, TP):
    """pos_idx / pos_deltas: the sampled positives' rows in any order, then -1"""
    for b in range(ol.shape[0]):
        pos = np.flatnonzero(ol[b] == 1)
        idx = got["pos_idx"][b]
        assert np.all(idx[pos.size:] == -1) and pos.size <= TP
        order = np.argsort(idx[:pos.size], kind="stable")
        assert np.array_equal(idx[:pos.size][order], pos)
        assert_deltas(got["pos_deltas"][b, :pos.size][order], od[b, pos])


def check_sparse(got, ref, TP, Q):
    od, ol = ref[0], ref[1]
    for b in range(ol.shape[0]):
        want = np.flatnonzero(ol[b] != -1)
        want = 2 * want + (ol[b, want] == 1)
        codes = got["codes"][b]
        assert np.all(codes[want.size:] == -1) and want.size <= Q
        assert np.array_equal(np.sort(codes[:want.size]), np.sort(want))
    check_rows(got, od, ol, TP)


def oracle(anchors, gtb, gtl, hp, seed, offset, image_offset=0, numpy_too=None):
    ref = CO.rpn_targets(anchors, gtb, gtl, hp, seed=seed, offset=offset, image_offset=image_offset, debug=True)
    B, G = gtl.shape
    if numpy_too is None:
        numpy_too = B * anchors.shape[0] * G <= NUMPY_MAX_PAIRS
    npref = None
    if numpy_too:
        with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
            npref = O.calculate_rpn_actual_outputs(anchors, gtb, gtl, hp, seed=seed, offset=offset,
                                                   image_offset=image_offset, return_debug=True)
    return ref, npref


def run_and_check(T, h, anchors, gtb, gtl, hp, seed=5, offset=11, image_offset=0, forms=("dense",), ref=None):
    if ref is None:
        ref = oracle(anchors, gtb, gtl, hp, seed, offset, image_offset)
    TP = int(hp["total_pos_bboxes"]); Q = TP + int(hp["total_neg_bboxes"])
    for form in forms:
        rc, got = launch(T, h, anchors, gtb, gtl, hp, seed, offset, image_offset, form)
        T.lib.check(rc)
        if form == "dense":
            check_dense(got, ref[0], ref[1])
        elif form == "compact":
            check_compact(got, ref[0], TP)
        else:
            check_sparse(got, ref[0], TP, Q)
    return ref[0]


def nice(b):
    """csrc/common.cuh nice_box: every coordinate 0 or of magnitude in [2^-16, 2^8), positive extents"""
    b = np.asarray(b, np.float64)
    a = np.abs(b)
    ok = np.all((a == 0) | ((a >= 2.0 ** -16) & (a < 2.0 ** 8)), axis=-1)
    return ok & (b[..., 2] > b[..., 0]) & (b[..., 3] > b[..., 1])


# ---- 1. inputs that take the any-input warp ----------------------------------------------------------------------
@pytest.mark.parametrize("apt,scalar", VARIANTS, ids=VARIANT_IDS)
@pytest.mark.parametrize("name", TL.FALLBACK_LAYOUTS)
def test_fallback_layouts(T, name, apt, scalar):
    anchors, gtb, gtl = TL.fallback_layout(name, seed=apt)
    hp = make_hp(anchors.shape[0])
    ref = run_and_check(T, handle(T, apt, scalar), anchors, gtb, gtl, hp, seed=apt, offset=7)
    if name == "flip_one_axis":   # the worked case: IoUs (-0, +0) with anchors 0 and 1, the first index wins
        assert ref[2]["argmax_col"][0, 0] == 0 and ref[1][0, 0] == 1


def test_fallback_layouts_compact_and_sparse(T):
    for name in TL.FALLBACK_LAYOUTS:
        anchors, gtb, gtl = TL.fallback_layout(name, seed=11)
        run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(anchors.shape[0], total_pos=16, total_neg=40),
                      forms=("compact", "sparse"))


# ---- 2. images mixing nice tiles and any-input tiles -------------------------------------------------------------
def special(k):
    """box k of a grid of disjoint 3/64 x 3/64 boxes in [1/2, 1]^2 (background anchors stay in [0, 1/2)^2)"""
    y, x = 32 + 4 * (k // 8), 32 + 4 * (k % 8)
    return np.array([y, x, y + 3, x + 3], F32) / 64


def shifted(b):
    return (b + F32(1 / 64)).astype(F32)


def mixed_layout(apt, seed):
    """every third CTA carries one non-nice anchor (zero area or pixel coordinates); GT winners placed in both kinds"""
    tile = 32 * apt
    N = tile * 9 + 17
    rng = np.random.default_rng(seed)
    anchors = TL.dyadic_boxes(rng, N, hi=32, ext=(1, 5))
    slow = [t for t in range(N // tile + 1) if t % 3 == 1]
    for i, t in enumerate(slow):
        n = min(t * tile + 5 + i, N - 1)
        if i % 2:
            anchors[n, 2] = anchors[n, 0]                  # zero area
        else:
            anchors[n] = anchors[n] * F32(64) + F32(300)    # pixel coordinates
    fast_t, slow_t = 3, 4                                   # tile 4 is slow for every APT (4 % 3 == 1)
    places = {0: [slow_t * tile + 9], 1: [fast_t * tile + 9], 2: [fast_t * tile + 2, slow_t * tile + 2],
              3: [tile + 20, 2 * tile + 20], 4: [slow_t * tile + 30, 6 * tile + 1]}
    for k, idx in places.items():
        for n in idx:
            anchors[n] = special(k)
    tile_of = np.arange(N) // tile
    for t in range(tile_of[-1] + 1):
        assert nice(anchors[tile_of == t]).all() == (t not in slow)
    gtb = np.zeros((2, 8, 4), F32)
    gtl = np.full((2, 8), -1, np.int32)
    for k in places:
        gtb[0, k] = special(k); gtb[1, k] = shifted(special(k))
        gtl[:, k] = k
    gtb[:, 5] = TL.dyadic_boxes(rng, 2, hi=32, ext=(4, 12)); gtl[:, 5] = 9
    winners = {k: min(idx) for k, idx in places.items()}
    return anchors, gtb, gtl, winners, slow


@pytest.mark.parametrize("apt,scalar", VARIANTS, ids=VARIANT_IDS)
def test_mixed_fast_and_fallback_tiles(T, apt, scalar):
    anchors, gtb, gtl, winners, slow = mixed_layout(apt, seed=20 + apt)
    ref = run_and_check(T, handle(T, apt, scalar), anchors, gtb, gtl, make_hp(anchors.shape[0]))
    col = ref[2]["argmax_col"]
    tile = 32 * apt
    for k, n in winners.items():
        assert col[0, k] == n
    assert col[0, 0] // tile in slow and col[0, 1] // tile not in slow     # winner in a fallback / a fast tile
    assert col[0, 2] // tile not in slow and col[0, 4] // tile in slow     # ties between the two kinds


# ---- 3. per-GT ties at tile boundaries ---------------------------------------------------------------------------
def tie_layout(apt, seed, fallback):
    tile = 32 * apt
    N = tile * 5 + tile // 2 + 3                            # the last tile is partial
    rng = np.random.default_rng(seed)
    anchors = TL.dyadic_boxes(rng, N, hi=32, ext=(1, 5))
    lane_pair = (2 * tile + 7 * apt, 2 * tile + 8 * apt - 1) if apt > 1 else (2 * tile + 1, 2 * tile + 30)
    places = [(tile - 1, tile),                             # across the CTA boundary
              (2 * tile - 1, 2 * tile, 3 * tile),
              (apt - 1, apt),                               # across the lane boundary
              (3 * tile + 5 * apt - 1, 3 * tile + 5 * apt),
              lane_pair,                                    # inside one lane's slots (APT 1: lanes 1 and 30)
              (3 * tile + 1, 4 * tile + 1, 4 * tile + 2),
              (5 * tile + 1, 5 * tile + 4)]                 # only in the last, partial tile
    flat = [n for p in places for n in p]
    assert len(set(flat)) == len(flat) and max(flat) < N
    for k, p in enumerate(places):
        for n in p:
            anchors[n] = special(k)
    G = len(places) + 3
    gtb = np.zeros((3, G, 4), F32)
    gtl = np.full((3, G), -1, np.int32)
    for k in range(len(places)):
        gtb[0, k] = special(k)                             # IoU 1
        gtb[1, k] = shifted(special(k))                    # an interior IoU (4/14), the same for every copy
        gtl[:2, k] = k
    gtb[2, 0] = [40 / 64, 2 / 64, 50 / 64, 20 / 64]         # overlaps nothing: every IoU +0, anchor 0 wins
    gtb[2, 1] = shifted(special(len(places) - 1))          # overlaps only the partial tile's copies
    gtl[2, :2] = 1
    if fallback:   # a box with no extent and positive area: every CTA of every image takes the any-input warp
        gtb[:, G - 1] = [0.9, 0.9, 0.8, 0.8]
    return anchors, gtb, gtl, places


@pytest.mark.parametrize("path", ["fast", "fallback"])
@pytest.mark.parametrize("apt,scalar", VARIANTS, ids=VARIANT_IDS)
def test_ties_at_tile_boundaries(T, apt, scalar, path):
    anchors, gtb, gtl, places = tie_layout(apt, seed=30 + apt, fallback=path == "fallback")
    ref = run_and_check(T, handle(T, apt, scalar), anchors, gtb, gtl, make_hp(anchors.shape[0]))
    col = ref[2]["argmax_col"]
    for k, p in enumerate(places):
        assert col[0, k] == min(p) and col[1, k] == min(p)
    assert col[2, 0] == 0 and col[2, 1] == min(places[-1])


# ---- 4. label-kernel variants ------------------------------------------------------------------------------------
def random_layout(N, B, G, seed, n_real=None):
    """dyadic anchors over [0,1] (many exact duplicates: ties everywhere); GT boxes, one a copy of the last anchor
    (its winner lies in the last tile) and one of anchor 0"""
    rng = np.random.default_rng(seed)
    anchors = TL.dyadic_boxes(rng, N, ext=(2, 20))
    n_real = G if n_real is None else n_real
    gtb = np.zeros((B, G, 4), F32)
    gtl = np.full((B, G), -1, np.int32)
    for b in range(B):
        gtb[b, :n_real] = TL.dyadic_boxes(rng, n_real, ext=(2, 30))
        gtl[b, :n_real] = rng.integers(0, 20, size=n_real)
        gtb[b, 0] = anchors[N - 1]
        gtb[b, n_real - 1] = anchors[0]
    return anchors, gtb, gtl


def lbl_iters(N):
    """the rpn_label_encode_kernel<ITERS> launch_targets picks"""
    return 9 if N <= 9 * LBL_THREADS else 12 if N <= 12 * LBL_THREADS else 0


SELECT_SCRATCH = 256 * 4 + 3 * 4                            # sizeof(SelectScratch)


def smem_lbl(N, G):
    """launch_targets' shared-memory plan of the label kernel: (bytes without the list, list fits in shared memory)"""
    words = (N + 31) // 32
    base = (G * (16 + 8 + 4) + 3 * words * 4 + SELECT_SCRATCH + 15) & ~15
    return base, base + N * 8 <= 160 * 1024


def smem_k2(G):
    return G * (2 * 16 + 4 + 4 + 4 + 8 + 1) + 4 * 8 * 40 * 4 + 16


def list_limit(G):
    """the largest N whose candidate list still lives in shared memory"""
    lo, hi = 1, 1 << 16
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if smem_lbl(mid, G)[1] else (lo, mid)
    return lo


@pytest.mark.parametrize("N,iters", [(9216, 9), (9217, 12), (12288, 12), (12289, 0)])
def test_label_kernel_iters(T, N, iters):
    assert lbl_iters(N) == iters
    anchors, gtb, gtl = random_layout(N, 2, 20, seed=N)
    gtb[1, 3] = anchors[N - 1] + F32(1 / 64)
    run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(N), forms=("dense", "sparse"))


@pytest.mark.parametrize("side", ["smem", "workspace"])
def test_candidate_list_shared_memory_limit(T, side):
    G = 50
    N = list_limit(G) + (side == "workspace")
    assert 19000 < N < 19500 and smem_lbl(N, G)[1] == (side == "smem")
    anchors, gtb, gtl = random_layout(N, 2, G, seed=N)
    # a low positive threshold: several thousand positive candidates, so the list is long on both passes
    run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(N, pos_thr=0.05, total_pos=300, total_neg=2000),
                  forms=("dense", "compact"))


@pytest.mark.parametrize("apt", [None, 1])
@pytest.mark.parametrize("G,GR", [(1, 32), (32, 32), (33, 31), (200, 5), (341, 3), (1000, 1), (1024, 1)])
def test_label_kernel_gt_grouping(T, G, GR, apt):
    assert min(LBL_THREADS // G, 32) == GR
    N = 4003
    anchors, gtb, gtl = random_layout(N, 2, G, seed=G, n_real=max(1, G - 7))
    run_and_check(T, handle(T, apt), anchors, gtb, gtl, make_hp(N))


@pytest.mark.parametrize("apt", [None, 1])
@pytest.mark.parametrize("G", [1025, 2000, 3767])
def test_label_kernel_many_gt_atomics(T, G, apt):
    assert G > LBL_THREADS and smem_k2(G) <= 200 * 1024
    N = 3001
    anchors, gtb, gtl = random_layout(N, 2, G, seed=G, n_real=G - 5)
    run_and_check(T, handle(T, apt), anchors, gtb, gtl, make_hp(N, total_pos=64), forms=("dense", "compact"))


def test_many_gt_workspace_list(T):
    G, N = 3000, 12288
    assert smem_k2(G) <= 200 * 1024 and not smem_lbl(N, G)[1] and lbl_iters(N) == 12
    anchors, gtb, gtl = random_layout(N, 1, G, seed=3)
    run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(N, pos_thr=0.3, total_pos=200))


def test_gt_beyond_shared_memory_plan(T):
    G, N = 3768, 512
    assert smem_k2(G) > 200 * 1024 and smem_k2(G - 1) <= 200 * 1024
    anchors, gtb, gtl = random_layout(N, 1, G, seed=4)
    rc, got = launch(T, handle(T), anchors, gtb, gtl, make_hp(N), 1, 1)
    assert rc == ERR_UNSUPPORTED
    assert np.all(np.isnan(got["labels"])) and np.all(got["argmax_col"] == SENT)   # nothing was launched


# ---- 5. sampling extremes ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c4(T):
    bb, _, G, over = T.syn.CONFIGS["C4"]
    hp = dict(O.get_hyper_params(bb), **over)
    anchors = O.generate_anchors(hp)
    gtb, gtl = T.syn.gt_batch(np.random.default_rng(77), 2, G)
    return hp, anchors, gtb, gtl


def c4_hp(hp, **kw):
    out = dict(hp)
    for k, v in kw.items():
        out[k] = v
    return out


@pytest.mark.parametrize("total_pos", [512, 1000])
def test_every_anchor_a_candidate(T, c4, total_pos):
    """pos threshold -1: the positive list holds all N anchors (workspace list, radix select over it), and the
    8-lanes-per-positive encode loop takes total_pos / 128 trips"""
    hp, anchors, gtb, gtl = c4
    N = anchors.shape[0]
    assert N == 37800 and not smem_lbl(N, gtl.shape[1])[1]
    h = c4_hp(hp, pos_iou_threshold=-1.0, total_pos_bboxes=total_pos, total_neg_bboxes=256)
    ref = run_and_check(T, handle(T), anchors, gtb, gtl, h, seed=9, offset=(1 << 40) + 3, image_offset=5,
                        forms=("dense", "compact", "sparse"))
    assert np.all(ref[2]["pos_pre"]) and np.all((ref[1] == 1).sum(-1) == total_pos)


@pytest.mark.parametrize("tp,tn", [(0, 128), (128, 0), (0, 0)])
def test_zero_quotas(T, tp, tn):
    N = 2500
    anchors, gtb, gtl = random_layout(N, 3, 30, seed=tp + tn)
    run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(N, total_pos=tp, total_neg=tn),
                  forms=("dense", "compact", "sparse"))


@pytest.mark.parametrize("d", [-1, 0, 1])
def test_quota_around_candidate_count(T, d):
    N = 3000
    anchors, gtb, gtl = random_layout(N, 1, 40, seed=8)
    hp = make_hp(N, pos_thr=0.4)
    _, _, dbg = CO.rpn_targets(anchors, gtb, gtl, hp, debug=True)
    M = int(dbg["pos_pre"].sum())
    assert M > 2
    hp = make_hp(N, pos_thr=0.4, total_pos=M + d, total_neg=0)
    run_and_check(T, handle(T), anchors, gtb, gtl, hp, forms=("dense", "sparse"))
    # negatives: neg_quota = total_pos + total_neg - pos_count lands on the negative candidate count -1 / 0 / +1
    hp = make_hp(N, pos_thr=0.4, total_pos=M, total_neg=0)
    _, _, dbg = CO.rpn_targets(anchors, gtb, gtl, hp, debug=True)
    Mn = int(dbg["neg_pre"].sum())
    run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(N, pos_thr=0.4, total_pos=M, total_neg=Mn + d),
                  forms=("dense", "sparse"))


def test_thresholds_attained_exactly(T):
    N = 3000
    anchors, gtb, gtl = random_layout(N, 2, 40, seed=12)
    _, _, dbg = CO.rpn_targets(anchors, gtb, gtl, make_hp(N), debug=True)
    vals = np.unique(dbg["max_iou"][dbg["max_iou"] > 0])
    hi, lo = vals[int(0.9 * vals.size)], vals[int(0.2 * vals.size)]
    for pos_thr, neg_thr in [(hi, lo), (lo, hi)]:           # (lo, hi): the negative threshold above the positive
        ref = run_and_check(T, handle(T), anchors, gtb, gtl, make_hp(N, pos_thr=float(pos_thr), neg_thr=float(neg_thr)))
        m = ref[2]["max_iou"]
        assert np.any(m == pos_thr) and np.any(m == neg_thr)


def test_labels_and_forcing(T):
    """GT boxes with extent labelled -1 force nothing; zero-padding rows labelled >= 0 force anchor 0 (their
    column is +0 everywhere); several GT boxes force the same anchor; an offset with its high 32 bits set"""
    N = 2000
    anchors, gtb, gtl = random_layout(N, 3, 24, seed=13)
    gtl[0, :6] = -1
    gtb[1, 10:] = 0; gtl[1, 10:] = 4
    gtb[2, 5:12] = gtb[2, 4]; gtl[2, 5:12] = 1
    hp = make_hp(N, total_pos=40, total_neg=60)
    ref = run_and_check(T, handle(T), anchors, gtb, gtl, hp, seed=(3 << 33) + 1, offset=(0xABCD << 32) | 17,
                        image_offset=2, forms=("dense", "compact", "sparse"))
    col = ref[2]["argmax_col"]
    assert np.all(col[1, 10:] == 0) and np.all(col[2, 5:12] == col[2, 4])


# ---- 6. determinism ----------------------------------------------------------------------------------------------
def test_deterministic_atomics_and_full_n_select(T, c4):
    hp, anchors, gtb, gtl = c4
    cases = [(random_layout(3001, 2, 2000, seed=2000), make_hp(3001, total_pos=64)),
             ((anchors, gtb, gtl), c4_hp(hp, pos_iou_threshold=-1.0, total_pos_bboxes=1000))]
    h = handle(T)
    for (a, g, l), p in cases:
        outs = []
        for _ in range(2):
            rc, got = launch(T, h, a, g, l, p, 21, 1 << 35)
            T.lib.check(rc)
            outs.append(got)
        for k in outs[0]:
            assert np.array_equal(outs[0][k].view(np.uint8), outs[1][k].view(np.uint8)), k

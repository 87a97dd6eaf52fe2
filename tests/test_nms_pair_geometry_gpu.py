"""The NMS pair decision, the round resolution and the output cap on constructed box geometry, in every NMS kernel.

Every output of the library ends in one NMS core (csrc/proposals.cu): canonical_box, the pre-test nms_maybe(2) with its
2^-10 margin on lo_s, nms_suppresses_fast (float pre-filters at thr * (1 -+ 2^-12), then the float64 midpoint test),
the slow nms_suppresses (thresholds outside [1e-30, 1e30], zero-area boxes unsanitised), kept_list_suppresses<2|4>
and resolve_round.  Random boxes reach these branches by chance; here every pair is built for one branch:

- CPU part (no GPU needed): a case generator and a plain reference.  For each pair it computes TF's float32 decision
  with the oracle's op order (rpn_oracle._nms_iou_vs) and the band the pair lies in, from the exact rational values of
  inter / (ai + aj) and inter / uni against a restatement of make_threshold.  Each case must land in the band it was
  built for, and the decision must follow from the band (RN(q) > thr  <=>  q > mid, mid = thr + ulp(thr) / 2).
- GPU part: the pairs (adjacent, and with the suppressor in the kept list of the round before), round structures
  (suppression chains across 128-candidate rounds, kept-list residues and part tails, max_out cuts), on every launch
  path: both proposal_kernel builds, the seven cluster shapes, the matrix NMS, the large-N prefilter with a redo
  image, tfrpn_nms_multiclass (q = 1 and q = C, both staging layouts) and tfrpn_proposals (the boxes as anchors, zero
  deltas).  Outputs are filled with a sentinel first; valid counts, keep indices, boxes and scores must equal the
  oracle bit for bit.
- IoU thresholds outside [0, 1] (and NaN) are refused by every entry point, as TF refuses them; 0 and 1 are accepted
  and their behaviour is pinned.

Each launch configuration is read by tfrpn_create, so every configuration has its own handle."""
import ctypes as C
import functools
import os
from fractions import Fraction

import numpy as np
import pytest

from oracle import rpn_oracle as O

F32 = np.float32
INF = float("inf")
NMS_CHUNK = 128
THRS = [0.05, 0.3, 0.45, 0.5, 0.6, 0.7, 0.9, 1.0]
SLOW_THRS = [0.0, -0.0, 1e-31, 2.0 ** -126, 1e-40]     # make_threshold: fast = 0 (nms_suppresses)
SENT_F = np.array([0x7FC0DEAD], np.uint32).view(F32)[0]   # sentinel NaN payload no kernel writes
SENT_I = -7


# ---------------------------------------------------------------------------------------------------------------------
# plain reference: make_threshold, the kernels' float32 terms of a pair, TF's decision, the band
# ---------------------------------------------------------------------------------------------------------------------
def host_threshold(thr):
    """make_threshold (csrc/proposals.cu) restated: double arithmetic, rounded to float where the C code does"""
    t = F32(thr)
    nxt = np.nextafter(t, F32(INF))
    d = float(t)
    return dict(thr=t, nxt=nxt, mid=Fraction(float(t)) / 2 + Fraction(float(nxt)) / 2,
                lo_f=F32(d * (1.0 - 1.0 / 4096.0)), hi_f=F32(d * (1.0 + 1.0 / 4096.0)),
                lo_s=F32(d / (1.0 + d) * (1.0 - 1.0 / 1024.0)),
                fast=bool(t >= F32(1e-30) and t <= F32(1e30)),
                tie_up=int(nxt.view(np.uint32)) & 1 == 0)


def canon(b):
    """canonical_box: fminf / fmaxf (NaN-ignoring) and the float32 area"""
    b = np.asarray(b, F32)
    c = np.array([np.fmin(b[0], b[2]), np.fmin(b[1], b[3]), np.fmax(b[0], b[2]), np.fmax(b[1], b[3])], F32)
    return c, F32(F32(c[2] - c[0]) * F32(c[3] - c[1]))


def pair_terms(bi, bj):
    """(ai, aj, inter, S = RN(ai + aj), U = RN(S - inter)) as the kernels compute them"""
    with np.errstate(all="ignore"):
        ci, ai = canon(bi)
        cj, aj = canon(bj)
        h = F32(np.fmin(ci[2], cj[2]) - np.fmax(ci[0], cj[0]))
        w = F32(np.fmin(ci[3], cj[3]) - np.fmax(ci[1], cj[1]))
        inter = F32(np.fmax(h, F32(0)) * np.fmax(w, F32(0)))
        S = F32(ai + aj)
        return ai, aj, inter, S, F32(S - inter)


def tf_decision(bi, bj, thr):
    """TF's float32 decision, RN(inter / RN(RN(ai + aj) - inter)) > thr, in the oracle's op order"""
    with np.errstate(all="ignore"):
        return bool(O._nms_iou_vs(np.asarray(bi, F32), np.asarray(bj, F32)[None])[0] > F32(thr))


def band(bi, bj, t):
    """(pre, q) bands of a pair with finite positive areas and terms: pre = 'in' | 'out' of the lo_s pre-test
    (exact I >= lo_s * S), q = 'below' (q < lo_f), 'above' (q > hi_f) or 'mid_lo' / 'mid_hi' (the float64 midpoint
    test, q below or above mid), from the exact quotient q = I / U"""
    ai, aj, inter, S, U = pair_terms(bi, bj)
    if not all(np.isfinite(v) for v in (ai, aj, inter, S, U)) or not (ai > 0 and aj > 0 and inter > 0):
        return None
    I = Fraction(float(inter))
    pre = "in" if I >= Fraction(float(t["lo_s"])) * Fraction(float(S)) else "out"
    q = I / Fraction(float(U))
    if q < Fraction(float(t["lo_f"])):
        qb = "below"
    elif q > Fraction(float(t["hi_f"])):
        qb = "above"
    else:
        qb = "mid_hi" if q > t["mid"] else "mid_lo"
    return pre, qb


def quotient(bi, bj):
    _, _, inter, _, U = pair_terms(bi, bj)
    return Fraction(float(inter)) / Fraction(float(U))


def rn32(fr):
    """round-to-nearest-even float32 of a Fraction"""
    x = F32(float(fr))
    cands = [np.nextafter(x, F32(-INF)), x, np.nextafter(x, F32(INF))]
    best = min(cands, key=lambda c: (abs(Fraction(float(c)) - fr), int(c.view(np.uint32)) & 1))
    return F32(best)


def ulp(t):
    return Fraction(float(np.nextafter(F32(t), F32(INF)))) - Fraction(float(F32(t)))


# ---------------------------------------------------------------------------------------------------------------------
# case generator
# ---------------------------------------------------------------------------------------------------------------------
def strips(p, u, sy=1.0, sx=1.0, oy=0.0, ox=0.0):
    """two boxes sharing their top-left corner: i is sy x (u sx), j is sy x (p sx) (p <= u): inter = area j"""
    i = [oy, ox, oy + sy, ox + u * sx]
    j = [oy, ox, oy + sy, ox + p * sx]
    return np.array(i, F32), np.array(j, F32)


def search(target, pred, n=1 << 13):
    """first width pair (p, u) whose real float32 terms satisfy pred: u drawn from [2^22, 2^23) with its fraction bit,
    p one of the five floats nearest target * u (seeded, so the cases are the same on every machine; consecutive
    integer u would give quotients on a lattice that can miss a target next to a simple ratio)"""
    us = np.random.default_rng(int(target * 2 ** 30)).integers(1 << 23, 1 << 24, size=n) * 0.5
    for u in us:
        pc = F32(target * u)
        lo, hi = pc, pc
        cands = [pc]
        for _ in range(2):
            lo, hi = np.nextafter(lo, F32(-INF)), np.nextafter(hi, F32(INF))
            cands += [lo, hi]
        for p in cands:
            if 0 < p <= u:
                bi, bj = strips(p, u)
                if pred(bi, bj):
                    return p, u
    return None


@functools.lru_cache(maxsize=None)
def quotient_cases(thr):
    """(name, box i, box j, expected band) at one fast threshold: strips of height 1 and widths below 2^23"""
    t = host_threshold(thr)
    T, mid, eps = Fraction(float(t["thr"])), t["mid"], ulp(thr)
    pred_t, succ_t = np.nextafter(t["thr"], F32(-INF)), t["nxt"]
    out = []

    def add(name, pu, want):
        if pu is not None:
            out.append((name,) + strips(*pu) + (want,))

    # next to a power of two (0.5, 1.0) inter and uni cannot be such floats: they have the same relative spacing
    add("rn_pred", search(float(pred_t), lambda a, b: rn32(quotient(a, b)) == pred_t), None)
    add("rn_thr", search(float(T), lambda a, b: rn32(quotient(a, b)) == t["thr"] and quotient(a, b) != T), None)
    if thr < 1.0:
        add("rn_succ", search(float(succ_t), lambda a, b: rn32(quotient(a, b)) == succ_t), None)
        add("mid_above", search(float(mid), lambda a, b: mid < quotient(a, b) < mid + eps / 8), ("in", "mid_hi"))
        add("mid_below", search(float(mid), lambda a, b: mid - eps / 8 < quotient(a, b) < mid), ("in", "mid_lo"))
        # thr < q < mid with inter > RN(thr * uni): only the midpoint test keeps it (a float test at thr says "above");
        # none exists when thr * uni is always a float (thr = 0.5)
        trap = search(float(mid), lambda a, b: T < quotient(a, b) < mid
                      and pair_terms(a, b)[2] > F32(t["thr"] * pair_terms(a, b)[4]))
        if trap is not None:
            add("float_thr_trap", trap, ("in", "mid_lo"))
    else:
        add("equal", (5123457.5, 5123457.5), ("in", "mid_lo"))     # identical boxes: q = 1, not > 1
    lo_s = Fraction(float(t["lo_s"]))

    def pre_ratio(a, b):
        _, _, inter, S, _ = pair_terms(a, b)
        return Fraction(float(inter)) / Fraction(float(S))
    r = float(lo_s / (1 - lo_s))                             # I / U with I / S = lo_s
    add("pre_inside", search(r, lambda a, b: lo_s <= pre_ratio(a, b) < lo_s * (1 + Fraction(1, 1 << 20))),
        ("in", "below"))
    add("pre_outside", search(r, lambda a, b: lo_s * (1 - Fraction(1, 1 << 20)) < pre_ratio(a, b) < lo_s),
        ("out", "below"))
    return out


def scaled(bi, bj, sy, sx, oy=0.0, ox=0.0):
    f = lambda b: np.array([oy + b[0] * sy, ox + b[1] * sx, oy + b[2] * sy, ox + b[3] * sx], F32)  # noqa: E731
    return f(bi), f(bj)


# magnitudes of the quotient cases: coordinates are scaled by powers of two, so the float32 terms scale exactly
MAGNITUDES = {
    "unit": (1.0, 2.0 ** -23),              # x in [0, 1)
    "pixel1333": (1.0, 2.0 ** -8, 1333.0),  # x in [0, 2^15), y in [1333, 1334]
    "pixel2e20": (1.0, 2.0 ** -8, 2.0 ** 20),
    "tiny": (2.0 ** -20, 2.0 ** -43),       # coordinates below 2^-20, areas ~2^-41
}


def magnitude_cases(thr):
    out = []
    for name, bi, bj, want in quotient_cases(thr):
        for mname, m in MAGNITUDES.items():
            a, b = scaled(bi, bj, *m)
            out.append(("%s/%s" % (name, mname), a, b, want))
    return out


def special_pairs():
    """(name, box i, box j, property): magnitudes, the far coordinates and degenerate boxes.  Properties are checked
    on the kernels' float32 terms (area_subnormal, area_inf, sum_inf) or are None"""
    u = np.array([0.25, 0.25, 0.75, 0.75], F32)
    out = []
    d = 2.0 ** -149
    for p, q in ((1, 1), (1, 2), (2, 3), (3, 5), (7, 8), (9, 10), (5, 9)):   # areas q * 2^-149 and p * 2^-149: exact
        out.append(("subnormal_%d_%d" % (p, q), np.array([0, 0, 2.0 ** -74, q * 2.0 ** -75], F32),
                    np.array([0, 0, 2.0 ** -74, p * 2.0 ** -75], F32), "area_subnormal"))
    out.append(("subnormal_vs_unit", np.array([0, 0, 2.0 ** -74, 2.0 ** -75], F32), u, "area_subnormal"))
    out.append(("quotient_underflow", np.array([0, 0, 2.0 ** 50, 2.0 ** 50], F32),
                np.array([0, 0, 2.0 ** -74, 2.0 ** -75], F32), "area_subnormal"))
    big = np.array([0, 0, 2.0 ** 64, 1.5 * 2.0 ** 63], F32)              # area 1.5 * 2^127: finite, the sum is not
    out.append(("sum_inf_identical", big, big.copy(), "sum_inf"))
    out.append(("sum_inf_shifted", big, np.array([0, 2.0 ** 60, 2.0 ** 64, 1.5 * 2.0 ** 63 + 2.0 ** 60], F32), "sum_inf"))
    huge = np.array([0, 0, 2.0 ** 100, 2.0 ** 100], F32)                 # area overflows
    out.append(("area_inf_identical", huge, huge.copy(), "area_inf"))
    out.append(("area_inf_vs_unit", huge, u, "area_inf"))
    fmax = float(np.finfo(F32).max)
    far = np.array([3.0e38, 3.0e38, -3.0e38, -3.0e38], F32)             # a real box equal to FAR_BOX
    out.append(("far_box_vs_unit", far, u, "area_inf"))
    out.append(("far_box_identical", far, far.copy(), "area_inf"))
    out.append(("flt_max_box", np.array([-fmax, -fmax, fmax, fmax], F32), u, "area_inf"))
    e1 = np.array([3.0e38, 3.0e38, fmax, fmax], F32)                     # extents ~4e37: area overflows
    out.append(("flt_max_corner", e1, e1.copy(), "area_inf"))
    e2 = np.array([-3.0e38, 0.0, -3.0e38 + 2.0 ** 104, 2.0 ** -100], F32)   # one ulp high at -3e38: area 16
    out.append(("far_finite_identical", e2, e2.copy(), None))
    out.append(("far_finite_flipped", e2, e2[[2, 3, 0, 1]].copy(), None))
    # degenerate boxes against a unit box and against a copy of themselves
    degs = {"zero_w": [0.25, 0.5, 0.75, 0.5], "zero_h": [0.5, 0.25, 0.5, 0.75], "point": [0.5, 0.5, 0.5, 0.5],
            "flip_y": [0.75, 0.25, 0.25, 0.75], "flip_x": [0.25, 0.75, 0.75, 0.25], "flip_xy": [0.75, 0.75, 0.25, 0.25],
            "neg_zero": [-0.0, -0.0, 0.5, 0.5], "inf_y": [-INF, 0.25, INF, 0.75], "inf_all": [-INF, -INF, INF, INF],
            "inf_ymin": [INF, 0.25, 0.75, 0.75], "inf_flip": [INF, INF, -INF, -INF]}
    for k in range(4):
        b = [0.25, 0.25, 0.75, 0.75]
        b[k] = float("nan")
        degs["nan_%d" % k] = b
    degs["nan_y"] = [float("nan"), 0.25, float("nan"), 0.75]
    degs["nan_all"] = [float("nan")] * 4
    for name, b in degs.items():
        b = np.array(b, F32)
        out.append(("deg_%s_vs_unit" % name, u, b, None))
        out.append(("unit_vs_deg_%s" % name, b, u, None))
        out.append(("deg_%s_self" % name, b, b.copy(), None))
    return out


def check_property(prop, bi, bj):
    ai, aj, inter, S, U = pair_terms(bi, bj)
    tiny = np.finfo(F32).tiny
    if prop == "area_subnormal":
        return (0 < ai < tiny) or (0 < aj < tiny)
    if prop == "area_inf":
        return np.isinf(ai) or np.isinf(aj)
    if prop == "sum_inf":
        return np.isfinite(ai) and np.isfinite(aj) and np.isinf(S)
    return prop is None


@functools.lru_cache(maxsize=None)
def pair_cases(thr):
    """every pair run at thr: (name, box i (higher score), box j)"""
    cases = []
    if host_threshold(thr)["fast"]:
        cases += [(n, a, b) for n, a, b, _ in quotient_cases(thr) + magnitude_cases(thr)]
    else:   # the quotient cases of 0.5 and 0.05 still make positive-area pairs for the slow path
        cases += [(n, a, b) for n, a, b, _ in quotient_cases(0.5)[:4] + quotient_cases(0.05)[:4]]
    cases += [(n, a, b) for n, a, b, _ in special_pairs()]
    return cases


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests of the generator
# ---------------------------------------------------------------------------------------------------------------------
TRAP_THRS = (0.05, 0.3, 0.6, 0.7)   # thresholds whose float_thr_trap the seeded search finds


@pytest.mark.parametrize("thr", THRS)
def test_quotient_cases_land_in_their_bands(thr):
    t = host_threshold(thr)
    assert t["fast"]
    names = set()
    for name, bi, bj, want in quotient_cases(thr) + magnitude_cases(thr):
        names.add(name.split("/")[0])
        got = band(bi, bj, t)
        assert got is not None, name
        pre, qb = got
        if want is not None:
            assert got == want, (name, got, want)
        # the decision follows from the band: the float64 midpoint test is exact, the pre-test and the float
        # pre-filters never reject a suppression
        q = quotient(bi, bj)
        dec = tf_decision(bi, bj, thr)
        assert dec == (rn32(q) > t["thr"]), name
        assert dec == (q > t["mid"] or (q == t["mid"] and t["tie_up"])), name
        if pre == "out" or qb == "below":
            assert not dec, name
        if qb == "above":
            assert dec, name
    base = {"pre_inside", "pre_outside"}
    base |= {"rn_succ", "mid_above"} if thr < 1.0 else {"equal"}
    base |= {"mid_below"} if thr not in (0.5, 1.0) else set()
    base |= {"rn_pred"} if thr < 1.0 else set()
    base |= {"rn_thr"} if thr not in (0.5, 1.0) else set()
    base |= {"float_thr_trap"} if thr in TRAP_THRS else set()
    assert base <= names, base - names


def test_rounding_targets_and_decisions():
    """rn_pred / rn_thr never suppress, rn_succ always does: the 1-ulp quotient cases cover both decisions"""
    for thr in THRS:
        for name, bi, bj, _ in quotient_cases(thr):
            if name in ("rn_pred", "rn_thr", "mid_below", "float_thr_trap", "equal", "pre_inside", "pre_outside"):
                assert not tf_decision(bi, bj, thr), (thr, name)
            if name in ("rn_succ", "mid_above"):
                assert tf_decision(bi, bj, thr), (thr, name)


def test_special_pairs_have_their_magnitudes():
    for name, bi, bj, prop in special_pairs():
        assert check_property(prop, bi, bj), name
    names = {n for n, _, _, _ in special_pairs()}
    for k in range(4):
        assert "deg_nan_%d_vs_unit" % k in names
    # the sum-overflow pair is a suppression in exact arithmetic (IoU 1) and none in TF's float32 one
    big = dict((n, (a, b)) for n, a, b, _ in special_pairs())["sum_inf_identical"]
    assert not tf_decision(*big, 0.5)
    # a real box far from the origin with a finite area suppresses its copy
    assert tf_decision(*dict((n, (a, b)) for n, a, b, _ in special_pairs())["far_finite_identical"], 0.5)


def test_slow_thresholds_are_slow():
    for thr in SLOW_THRS:
        t = host_threshold(thr)
        assert not t["fast"] and 0 <= t["thr"] <= 1


def test_thr_zero_and_one_decisions():
    """thr = 0 suppresses a pair exactly when RN(inter / uni) > 0, so a quotient that underflows does not; thr = 1
    suppresses nothing, RN(inter / uni) <= 1"""
    sp = dict((n, (a, b)) for n, a, b, _ in special_pairs())
    a, b = sp["quotient_underflow"]
    assert pair_terms(a, b)[2] > 0 and not tf_decision(a, b, 0.0)
    a, b = sp["subnormal_1_2"]
    assert tf_decision(a, b, 0.0) and tf_decision(a, b, -0.0)
    a, b = sp["deg_zero_w_vs_unit"]
    assert not tf_decision(a, b, 0.0)
    for name, a, b in pair_cases(1.0):
        assert not tf_decision(a, b, 1.0), name


# ---------------------------------------------------------------------------------------------------------------------
# round and cap structures (NMS_CHUNK = 128 candidates a round)
# ---------------------------------------------------------------------------------------------------------------------
W = 2.0 ** -10   # unit-coordinate boxes with dyadic corners: decoding them with zero deltas is exact


def chain(L, offset=0):
    """box i overlaps i + 1 with IoU 0.6 and i + 2 with IoU 1/3: at 0.45 / 0.5 box i suppresses only i + 1"""
    b = [[0.5, 0.5, 0.5 + W, 0.5 + W]] * offset   # a disjoint first box shifts the chain by one candidate
    b += [[0.0, i * W / 4, W, i * W / 4 + W] for i in range(L)]
    return np.array(b, F32)


def grid(n, size=W):
    """n disjoint boxes"""
    return np.array([[(i // 32) * 2 * size + 0.125, (i % 32) * 2 * size, (i // 32) * 2 * size + 0.125 + size,
                      (i % 32) * 2 * size + size] for i in range(n)], F32)


def kept_list_image(n):
    """round 1: n disjoint boxes and 128 - n copies of box 0 (suppressed inside the round), then copies of every box,
    last first: each copy is suppressed by the kept box it copies, at kept-list position n - 1 ... 0"""
    g = grid(n)
    return np.concatenate([g, np.repeat(g[:1], NMS_CHUNK - n, 0), g[::-1]], 0)


STRUCT_K = 300


@functools.lru_cache(maxsize=None)
def structures():
    """(names, boxes (B, K, 4), scores (B, K)): images padded with entries below the score threshold 0"""
    imgs = {}
    for L in (2, 127, 128, 129, 255, 256, 257, 300):
        imgs["chain%d" % L] = chain(L)
    for L in (128, 255, 299):
        imgs["chain%d_off1" % L] = chain(L, 1)
    imgs["all_survive"] = grid(STRUCT_K)
    imgs["first_removes_all"] = np.repeat(grid(1), STRUCT_K, 0)
    for n in list(range(97, 129)) + [1, 2, 3, 5, 9, 17, 33, 65]:
        imgs["kept%d" % n] = kept_list_image(n)
    names = sorted(imgs)
    B = len(names)
    boxes = np.zeros((B, STRUCT_K, 4), F32)
    scores = np.full((B, STRUCT_K), -1.0, F32)
    for b, nm in enumerate(names):
        x = imgs[nm]
        boxes[b, :len(x)] = x
        scores[b, :len(x)] = 1.0 - np.arange(len(x), dtype=np.float64) * 2.0 ** -12
    return names, boxes, scores


def test_structures_are_what_they_claim():
    names, boxes, scores = structures()
    d = dict(zip(names, range(len(names))))
    for thr in (0.45, 0.5):
        b = d["chain300"]
        bx = boxes[b, :300]
        assert all(tf_decision(bx[i], bx[i + 1], thr) for i in range(299))
        assert not any(tf_decision(bx[i], bx[i + 2], thr) for i in range(298))
        nb, ns, nc, nv, ni = oracle_nms(boxes[b:b + 1], scores[b:b + 1], thr, 300, 300, False)
        assert nv[0] == 150 and np.array_equal(ni[0, :150], np.arange(0, 300, 2))
    nb, ns, nc, nv, ni = oracle_nms(boxes, scores, 0.5, 256, 256, False)
    for n in (97, 101, 128, 1, 65):
        assert nv[d["kept%d" % n]] == n
    assert nv[d["all_survive"]] == 256 and nv[d["first_removes_all"]] == 1


# ---------------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------------
def oracle_nms(boxes, scores, thr, per_class, total, pad, sthr=0.0):
    with np.errstate(all="ignore"):
        return O.combined_non_max_suppression(boxes[:, :, None, :], scores[:, :, None], per_class, total,
                                              iou_threshold=thr, score_threshold=sthr, pad_per_class=pad,
                                              clip_boxes=False, return_indices=True)


FILL = NMS_CHUNK - 1


@functools.lru_cache(maxsize=None)
def pair_batch(thr, layout):
    """(names, boxes, scores): one image per pair.  'adjacent': [i, j], decided inside one round; 'kept': [i, 127
    zero-area boxes, j], so j meets i in the kept list of the round before"""
    cases = pair_cases(thr)
    K = 2 if layout == "adjacent" else FILL + 2
    boxes = np.zeros((len(cases), K, 4), F32)
    for b, (_, bi, bj) in enumerate(cases):
        boxes[b, 0], boxes[b, K - 1] = bi, bj
        if K > 2:
            boxes[b, 1:K - 1] = np.array([[2.0, 2.0 + k, 2.0, 3.0 + k] for k in range(FILL)], F32)   # zero height
    scores = np.broadcast_to((1.0 - np.arange(K) * 2.0 ** -12).astype(F32), (len(cases), K)).copy()
    return [c[0] for c in cases], boxes, scores


@functools.lru_cache(maxsize=None)
def pair_oracle(thr, layout):
    _, boxes, scores = pair_batch(thr, layout)
    K = boxes.shape[1]
    return oracle_nms(boxes, scores, thr, K, K, False, sthr=-INF)


def test_pair_oracle_is_the_pair_decision():
    """the images' expected outputs are the pair decisions: j is kept iff TF's test says i does not suppress it"""
    for thr in (0.05, 0.7, 1.0, 0.0):
        names, boxes, _ = pair_batch(thr, "kept")
        nv = pair_oracle(thr, "kept")[3]
        for b, nm in enumerate(names):
            dec = tf_decision(boxes[b, 0], boxes[b, -1], thr)
            assert nv[b] == FILL + 1 + (0 if dec else 1), (thr, nm)


# ---------------------------------------------------------------------------------------------------------------------
# the threshold range: CPU side (the checks come before the handle's)
# ---------------------------------------------------------------------------------------------------------------------
BAD_THRS = [-0.1, float(np.nextafter(F32(1), F32(2))), float("nan"), INF, -INF]
GOOD_THRS = [0.0, -0.0, 1.0]


def test_oracle_refuses_thresholds_outside_unit_interval():
    b = np.zeros((1, 1, 1, 4), F32)
    s = np.ones((1, 1, 1), F32)
    for thr in BAD_THRS:
        with pytest.raises(AssertionError):
            O.combined_non_max_suppression(b, s, 1, 1, iou_threshold=thr)
    for thr in GOOD_THRS:
        O.combined_non_max_suppression(b, s, 1, 1, iou_threshold=thr)


def test_python_cfg_refuses_thresholds_outside_unit_interval():
    from tfrpn import _lib
    from tfrpn.proposals import proposal_cfg
    hp = O.get_hyper_params("vgg16")
    for thr in BAD_THRS:
        with pytest.raises(ValueError, match=r"\[0, 1\]"):
            _lib.iou_threshold(thr)
        with pytest.raises(ValueError, match=r"\[0, 1\]"):
            proposal_cfg(hp, nms_iou_threshold=thr)
    for thr in GOOD_THRS:
        assert _lib.iou_threshold(thr) == thr
        assert proposal_cfg(hp, nms_iou_threshold=thr).nms_iou_threshold == thr


def test_c_entry_points_refuse_thresholds_before_anything_else():
    from tfrpn import _lib
    lib = _lib.load()
    buf = (C.c_float * 64)()
    p = C.c_void_p((C.addressof(buf) + 15) & ~15)
    from tfrpn.utils import bbox_utils
    acfg = bbox_utils._anchor_cfg(O.get_hyper_params("vgg16"))

    def calls(thr):
        nms = _lib.NmsCfg(4, 4, thr, -INF, 0, 1, 0)
        pc = _lib.ProposalCfg((C.c_float * 4)(0.1, 0.1, 0.2, 0.2), 8, 4, thr, 1)
        yield "nms", lambda: lib.tfrpn_nms(None, p, p, 1, 1, C.byref(nms), p, p, p, p, p, None)
        yield "nms_multiclass", lambda: lib.tfrpn_nms_multiclass(None, p, 1, p, 1, 1, 1, C.byref(nms), p, p, p, p, p,
                                                                 None)
        yield "proposals", lambda: lib.tfrpn_proposals(None, p, p, p, 1, 1, C.byref(pc), p, p, p, p, None)
        yield "proposals_anchor_cfg", lambda: lib.tfrpn_proposals_anchor_cfg(None, p, p, C.byref(acfg), 1, C.byref(pc),
                                                                             p, p, p, p, None)
    for thr in BAD_THRS:
        for name, call in calls(thr):
            assert call() == -1, (name, thr)
            assert b"iou_threshold" in lib.tfrpn_last_error(), (name, thr, lib.tfrpn_last_error())
    for thr in GOOD_THRS:
        for name, call in calls(thr):
            assert call() == -1, (name, thr)
            assert b"null handle" in lib.tfrpn_last_error(), (name, thr, lib.tfrpn_last_error())


# ---------------------------------------------------------------------------------------------------------------------
# GPU: launch paths
# ---------------------------------------------------------------------------------------------------------------------
PATHS = {
    "default": {},
    "threads512": {"TFRPN_PROP_CLUSTER": 0, "TFRPN_PROP_THREADS": 512},
    "threads1024": {"TFRPN_PROP_CLUSTER": 0, "TFRPN_PROP_THREADS": 1024},
    "cl1x1024": {"TFRPN_PROP_CLUSTER": 1}, "cl2x1024": {"TFRPN_PROP_CLUSTER": 2},
    "cl2x512": {"TFRPN_PROP_CLUSTER": 12}, "cl4x512": {"TFRPN_PROP_CLUSTER": 4},
    "cl4x256": {"TFRPN_PROP_CLUSTER": 14}, "cl8x256": {"TFRPN_PROP_CLUSTER": 8},
    "cl8x512": {"TFRPN_PROP_CLUSTER": 28},
    "matrix64": {"TFRPN_NMS_PATH": "matrix", "TFRPN_NMS_ROWS": 64},
    "matrix640": {"TFRPN_NMS_PATH": "matrix", "TFRPN_NMS_ROWS": 640},
    "matrix1024": {"TFRPN_NMS_PATH": "matrix", "TFRPN_NMS_ROWS": 1024},
}
MC_PATHS = {"mc_column": {"TFRPN_NMS_MC_STAGE": "column"}, "mc_rows": {"TFRPN_NMS_MC_STAGE": "rows"}}


class Handles:
    def __init__(self, dev):
        import torch
        from tfrpn import _lib
        self.torch, self.lib, self.dev, self.h = torch, _lib, dev, {}

    def get(self, path):
        if path not in self.h:
            env = {k: str(v) for k, v in dict(PATHS, **MC_PATHS)[path].items()}
            old = {k: os.environ.get(k) for k in env}
            os.environ.update(env)   # read once, by tfrpn_create
            try:
                h = C.c_void_p()
                self.lib.check(self.lib.load().tfrpn_create(C.byref(h), self.dev.index or 0))
            finally:
                for k, v in old.items():
                    if v is None:
                        os.environ.pop(k)
                    else:
                        os.environ[k] = v
            self.h[path] = h
        return self.h[path]

    def close(self):
        for h in self.h.values():
            self.lib.load().tfrpn_destroy(h)

    def cu(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)

    def full(self, shape, v, dtype=None):
        return self.torch.full(shape, v, dtype=dtype or self.torch.float32, device=self.dev)

    def st(self):
        return self.torch.cuda.current_stream(self.dev).cuda_stream


@pytest.fixture(scope="module")
def H(cuda_device):
    hs = Handles(cuda_device)
    yield hs
    hs.close()


def out_tensors(H, B, rows):
    import torch
    return (H.full((B, rows, 4), float(SENT_F)), H.full((B, rows), float(SENT_F)), H.full((B, rows), float(SENT_F)),
            H.full((B,), SENT_I, torch.int32), H.full((B, rows), SENT_I, torch.int32))


def fetch(H, outs):
    H.torch.cuda.synchronize()
    return [t.cpu().numpy() for t in outs]


def run_nms(H, path, boxes, scores, thr, per_class, total, pad, sthr=0.0):
    B, K = scores.shape
    rows = min(total, per_class) if pad else total
    cfg = H.lib.NmsCfg(per_class, total, float(thr), float(sthr), int(pad), 0, 0)
    outs = out_tensors(H, B, rows)
    b_t, s_t = H.cu(boxes), H.cu(scores)
    H.lib.check(H.lib.load().tfrpn_nms(H.get(path), b_t.data_ptr(), s_t.data_ptr(), B, K, C.byref(cfg),
                                       *[t.data_ptr() for t in outs], H.st()))
    return fetch(H, outs)


def assert_same(got, want, what):
    nb, ns, nc, nv, ni = got
    ob, os_, oc, ov, oi = want
    assert np.array_equal(nv, ov), (what, np.flatnonzero(nv != ov)[:8])
    assert np.array_equal(ni, oi), (what, np.flatnonzero((ni != oi).any(-1))[:8])
    for g, w, nm in ((nb, ob, "boxes"), (ns, os_, "scores"), (nc, oc, "classes")):
        g, w = np.ascontiguousarray(g, F32), np.ascontiguousarray(w, F32)
        assert g.shape == w.shape and np.array_equal(g.view(np.uint32), w.view(np.uint32)), (what, nm)


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_pairs_every_path(H, path):
    """every constructed pair, adjacent and through the kept list, at every threshold"""
    for thr in THRS + SLOW_THRS:
        for layout in ("adjacent", "kept"):
            names, boxes, scores = pair_batch(thr, layout)
            K = boxes.shape[1]
            got = run_nms(H, path, boxes, scores, thr, K, K, False, sthr=-INF)
            want = pair_oracle(thr, layout)
            bad = np.flatnonzero(got[3] != want[3])
            assert not len(bad), (path, thr, layout, [names[b] for b in bad[:8]])
            assert_same(got, want, (path, thr, layout))


MAX_OUTS = [1, 127, 128, 129, 200, 255, 256, 300, 305]


@functools.lru_cache(maxsize=None)
def structure_oracle(thr, max_out, pad):
    _, boxes, scores = structures()
    return oracle_nms(boxes, scores, thr, max_out, max_out + 7, pad)


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_round_structures_every_path(H, path):
    """chains across rounds, kept-list residues and part tails, max_out cuts, pad_per_class on and off"""
    names, boxes, scores = structures()
    for thr in (0.45, 0.5, 0.0):
        for max_out in MAX_OUTS:
            for pad in (False, True):
                got = run_nms(H, path, boxes, scores, thr, max_out, max_out + 7, pad)
                want = structure_oracle(thr, max_out, pad)
                bad = np.flatnonzero(got[3] != want[3])
                assert not len(bad), (path, thr, max_out, pad, [names[b] for b in bad[:8]])
                assert_same(got, want, (path, thr, max_out, pad))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["default", "threads512", "threads1024"])
def test_prefilter_with_redo_image(H, path):
    """K = 40000: the large-N prefilter keeps the top 6144 ranks; image 0 fills max_out from a chain, image 1 (every
    box a copy of one) runs out of candidates after keeping one box and is redone by the unfiltered kernel"""
    K, max_out = 40000, 300
    boxes = np.zeros((2, K, 4), F32)
    boxes[0, :600] = chain(600)
    boxes[0, 600:] = np.array([0.9, 0.9, 0.9, 0.95], F32)                  # zero height, never reached
    boxes[1] = grid(1)[0]
    scores = np.broadcast_to((1.0 - np.arange(K) * 2.0 ** -17).astype(F32), (2, K)).copy()
    for thr in (0.5, 0.0):
        got = run_nms(H, path, boxes, scores, thr, max_out, max_out, False, sthr=-INF)
        want = oracle_nms(boxes, scores, thr, max_out, max_out, False, sthr=-INF)
        assert list(want[3]) == ([300, 1] if thr == 0.5 else list(want[3]))
        assert_same(got, want, (path, thr))


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(MC_PATHS))
@pytest.mark.parametrize("q", ["1", "C"])
def test_multiclass_pairs_and_structures(H, path, q):
    """tfrpn_nms_multiclass: class 0 holds the pairs (or structures), class 1 the same boxes flipped in both axes
    (q = C) or shared (q = 1) with the scores in reverse order"""
    import torch
    sets = [("pairs%g" % thr, thr) + pair_batch(thr, "kept")[1:] for thr in (0.05, 0.45, 0.7, 1.0, 0.0, 1e-40)]
    names, sb, ss = structures()
    sets += [("structures", 0.5, sb, ss)]
    for what, thr, boxes, scores in sets:
        B, K = scores.shape
        Cn = 2
        s2 = np.stack([scores, scores[:, ::-1]], -1).astype(F32)
        if q == "1":
            b2 = boxes[:, :, None, :]
        else:
            b2 = np.stack([boxes, boxes[..., [2, 3, 0, 1]]], 2).astype(F32)
        P, total = 129, 2 * 129 + 5    # every kept row of both classes reaches the output: no pair hides behind the cut
        for pad in (False, True):
            cfg = H.lib.NmsCfg(P, total, float(thr), 0.0 if what == "structures" else -INF, int(pad), 0, 0)
            rows = min(total, P * Cn) if pad else total
            outs = out_tensors(H, B, rows)
            b_t, s_t = H.cu(b2), H.cu(s2)
            H.lib.check(H.lib.load().tfrpn_nms_multiclass(H.get(path), b_t.data_ptr(), b2.shape[2], s_t.data_ptr(), B,
                                                          K, Cn, C.byref(cfg), *[t.data_ptr() for t in outs], H.st()))
            got = fetch(H, outs)
            with np.errstate(all="ignore"):
                want = O.combined_non_max_suppression(b2, s2, P, total, iou_threshold=thr,
                                                      score_threshold=cfg.score_threshold, pad_per_class=pad,
                                                      clip_boxes=False, return_indices=True)
            assert_same(got, want, (path, q, what, pad))


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_proposals_on_the_same_boxes(H, path):
    """tfrpn_proposals with the boxes as anchors and zero deltas against the oracle fed the decoded boxes: the chain
    (every candidate of a round depends on the one before) and the unit-coordinate pairs"""
    import torch
    hp = O.get_hyper_params("vgg16")
    unit = [(n, a, b) for n, a, b in pair_cases(0.7) if n.endswith("/unit") or n.startswith("deg_")]
    anchors_pairs = np.concatenate([np.stack([a, b]) for _, a, b in unit], 0)
    Np = len(anchors_pairs)
    cls_pairs = np.full((len(unit), Np), 0.25, F32)
    for b in range(len(unit)):
        cls_pairs[b] = (0.5 - np.arange(Np) * 2.0 ** -14).astype(F32)[np.roll(np.arange(Np), 2 * b)]
        cls_pairs[b, 2 * b], cls_pairs[b, 2 * b + 1] = 0.9, 0.8
    ch = chain(300)
    cls_chain = np.stack([(1.0 - np.arange(300) * 2.0 ** -12).astype(F32), (0.5 + np.arange(300) * 2.0 ** -12)
                          .astype(F32)] * 5)
    for anchors, cls, P, thrs in ((anchors_pairs, cls_pairs, 2, (0.7, 0.05, 1.0, 0.0)),
                                  (ch, cls_chain, 129, (0.5, 0.0))):
        B, N = cls.shape
        reg = np.zeros((B, N, 4), F32)
        for thr in thrs:
            cfg = H.lib.ProposalCfg((C.c_float * 4)(*hp["variances"]), N, P, float(thr), 1)
            ob, os_ = H.full((B, P, 4), float(SENT_F)), H.full((B, P), float(SENT_F))
            ov, ok = H.full((B,), SENT_I, torch.int32), H.full((B, P), SENT_I, torch.int32)
            r_t, c_t, a_t = H.cu(reg), H.cu(cls), H.cu(anchors)
            H.lib.check(H.lib.load().tfrpn_proposals(H.get(path), r_t.data_ptr(), c_t.data_ptr(), a_t.data_ptr(), B, N,
                                                     C.byref(cfg), ob.data_ptr(), os_.data_ptr(), ov.data_ptr(),
                                                     ok.data_ptr(), H.st()))
            gb, gs, gv, gk = fetch(H, (ob, os_, ov, ok))
            with np.errstate(all="ignore"):
                wb, ws, wv, wk = O.generate_proposals(reg, cls, anchors, hp, pre_nms_topn=N, post_nms_topn=P,
                                                      nms_iou_threshold=thr)
            assert np.array_equal(gv, wv) and np.array_equal(gk, wk), (path, thr, N)
            assert np.array_equal(gb.view(np.uint32), np.ascontiguousarray(wb, F32).view(np.uint32)), (path, thr, N)
            assert np.array_equal(gs.view(np.uint32), np.ascontiguousarray(ws, F32).view(np.uint32)), (path, thr, N)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the threshold range through every entry point and wrapper
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_every_entry_point_refuses_thresholds_outside_unit_interval(H):
    import torch
    from tfrpn import _lib, roi_detections
    from tfrpn.proposals import generate_proposals
    from tfrpn.utils import bbox_utils
    lib = _lib.load()
    h = H.get("default")
    hp = O.get_hyper_params("vgg16")
    dev = H.dev
    B, N, P = 1, 64, 8
    anchors = H.cu(grid(N))
    reg, cls = H.cu(np.zeros((B, N, 4), F32)), H.cu(np.linspace(1, 0, N, dtype=F32)[None])
    ob, os_ = H.full((B, P, 4), 0.0), H.full((B, P), 0.0)
    ov, ok = H.full((B,), 0, torch.int32), H.full((B, P), 0, torch.int32)
    oc = H.full((B, P), 0.0)
    hb = [np.zeros(s, F32) for s in ((B, N, 4), (B, N), (B, P, 4), (B, P))]
    hv, hk = np.zeros(B, np.int32), np.zeros((B, P), np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    acfg = bbox_utils._anchor_cfg(hp)
    n_cfg = acfg.fm_h * acfg.fm_w * acfg.n_scales * acfg.n_ratios
    reg_a, cls_a = H.cu(np.zeros((B, n_cfg, 4), F32)), H.cu(np.linspace(1, 0, n_cfg, dtype=F32)[None])
    rois = H.cu(grid(N)[None])
    logits = H.cu(np.zeros((B, N, 3), F32))
    deltas = H.cu(np.zeros((B, N, 3, 4), F32))
    tcfg = _lib.TargetCfg(0.7, 0.3, 4, 4, (C.c_float * 4)(0.1, 0.1, 0.2, 0.2), 1, 0, 0, 0)
    gtb, gtl = np.zeros((B, 1, 4), F32), np.zeros((B, 1), np.int32)
    gtb[0, 0] = [0.1, 0.1, 0.4, 0.4]

    def calls(thr):
        nms = _lib.NmsCfg(P, P, thr, -INF, 0, 1, 0)
        det = _lib.RoiDetCfg(3, 3, 0, (C.c_float * 4)(0.1, 0.1, 0.2, 0.2), INF, 1, 0.0, nms)
        pc = _lib.ProposalCfg((C.c_float * 4)(0.1, 0.1, 0.2, 0.2), N, P, thr, 1)
        b4 = anchors.reshape(B, N, 4)
        yield "nms", lambda: lib.tfrpn_nms(h, b4.data_ptr(), cls.data_ptr(), B, N, C.byref(nms), ob.data_ptr(),
                                           os_.data_ptr(), oc.data_ptr(), ov.data_ptr(), ok.data_ptr(), H.st())
        yield "nms_multiclass", lambda: lib.tfrpn_nms_multiclass(h, b4.data_ptr(), 1, cls.data_ptr(), B, N, 1,
                                                                 C.byref(nms), ob.data_ptr(), os_.data_ptr(),
                                                                 oc.data_ptr(), ov.data_ptr(), ok.data_ptr(), H.st())
        yield "reserve_nms_multiclass", lambda: lib.tfrpn_reserve_nms_multiclass(h, B, N, 1, C.byref(nms))
        yield "roi_head_detections", lambda: lib.tfrpn_roi_head_detections(
            h, rois.data_ptr(), None, logits.data_ptr(), deltas.data_ptr(), B, N, C.byref(det), ob.data_ptr(),
            os_.data_ptr(), oc.data_ptr(), ov.data_ptr(), ok.data_ptr(), None, H.st())
        yield "reserve_roi_head_detections", lambda: lib.tfrpn_reserve_roi_head_detections(h, B, N, C.byref(det))
        yield "proposals", lambda: lib.tfrpn_proposals(h, reg.data_ptr(), cls.data_ptr(), anchors.data_ptr(), B, N,
                                                       C.byref(pc), ob.data_ptr(), os_.data_ptr(), ov.data_ptr(),
                                                       ok.data_ptr(), H.st())
        yield "proposals_anchor_cfg", lambda: lib.tfrpn_proposals_anchor_cfg(h, reg_a.data_ptr(), cls_a.data_ptr(),
                                                                             C.byref(acfg), B, C.byref(pc), ob.data_ptr(),
                                                                             os_.data_ptr(), ov.data_ptr(), ok.data_ptr(),
                                                                             H.st())
        yield "proposals_host", lambda: lib.tfrpn_proposals_host(h, vp(hb[0]), vp(hb[1]), anchors.data_ptr(), B, N,
                                                                 C.byref(pc), vp(hb[2]), vp(hb[3]), vp(hv), vp(hk),
                                                                 H.st())
        yield "rpn_step_host", lambda: lib.tfrpn_rpn_step_host(
            h, anchors.data_ptr(), vp(gtb), vp(gtl), B, N, 1, C.byref(tcfg), vp(np.zeros((B, N, 4), F32)),
            vp(np.zeros((B, N), F32)), vp(hb[0]), vp(hb[1]), C.byref(pc), vp(hb[2]), vp(hb[3]), vp(hv), vp(hk), H.st())

        def pipe():
            pl = C.c_void_p()
            _lib.check(lib.tfrpn_pipeline_create(h, 1, C.byref(pl)))
            try:
                t = C.c_int64()
                return lib.tfrpn_pipeline_submit(pl, anchors.data_ptr(), B, N, None, None, 0, None, None, None,
                                                 vp(hb[0]), vp(hb[1]), C.byref(pc), vp(hb[2]), vp(hb[3]), vp(hv),
                                                 vp(hk), C.byref(t))
            finally:
                lib.tfrpn_pipeline_drain(pl)
                lib.tfrpn_pipeline_destroy(pl)
        yield "pipeline_submit", pipe

    torch.cuda.synchronize()
    for thr in BAD_THRS:
        for name, call in calls(thr):
            before = _lib.launch_count()
            assert call() == -1, (name, thr)
            assert b"iou_threshold" in lib.tfrpn_last_error(), (name, thr, lib.tfrpn_last_error())
            assert _lib.launch_count() == before, (name, thr)
    # the wrappers raise ValueError before they launch anything
    for thr in BAD_THRS:
        before = _lib.launch_count()
        with pytest.raises(ValueError):
            generate_proposals(reg, cls, anchors, hp, pre_nms_topn=N, post_nms_topn=P, nms_iou_threshold=thr)
        with pytest.raises(ValueError):
            bbox_utils.non_max_suppression(anchors.reshape(B, N, 1, 4), cls.reshape(B, N, 1), max_output_size_per_class=P,
                                           max_total_size=P, iou_threshold=thr)
        with pytest.raises(ValueError):
            bbox_utils.non_max_suppression(anchors.reshape(B, N, 1, 4), cls.reshape(B, N, 1).repeat(1, 1, 2),
                                           max_output_size_per_class=P, max_total_size=P, iou_threshold=thr)
        with pytest.raises(ValueError):
            roi_detections.roi_head_detections(rois, logits, deltas, iou_threshold=thr)
        assert _lib.launch_count() == before, thr
    # 0, -0 and 1 are accepted by every entry point
    for thr in GOOD_THRS:
        for name, call in calls(thr):
            assert call() == 0, (name, thr, lib.tfrpn_last_error())
        torch.cuda.synchronize()


@pytest.mark.gpu
def test_thresholds_zero_and_one_are_pinned(H):
    """thr = 0 suppresses exactly when RN(inter / uni) > 0 (an underflowing quotient does not suppress); thr = 1
    suppresses nothing (RN(inter / uni) <= 1, identical boxes included)"""
    sp = dict((n, (a, b)) for n, a, b, _ in special_pairs())
    boxes = np.stack([np.stack(sp[k]) for k in ("quotient_underflow", "subnormal_1_2", "deg_zero_w_vs_unit",
                                                "sum_inf_identical", "far_finite_identical")])
    scores = np.broadcast_to(np.array([0.9, 0.8], F32), (len(boxes), 2)).copy()
    for thr, kept in ((0.0, [2, 1, 2, 2, 1]), (-0.0, [2, 1, 2, 2, 1]), (1.0, [2, 2, 2, 2, 2])):
        for path in ("default", "cl8x256", "matrix64"):
            got = run_nms(H, path, boxes, scores, thr, 2, 2, False, sthr=-INF)
            assert list(got[3]) == kept, (thr, path)
            assert_same(got, oracle_nms(boxes, scores, thr, 2, 2, False, sthr=-INF), (thr, path))

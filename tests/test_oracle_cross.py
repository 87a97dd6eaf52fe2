"""The two restatements (NumPy and C) must agree: integer outputs bit-exact, IEEE-only floats
bit-exact, exp/log floats within 1e-6 relative (glibc vs NumPy SIMD differ by <= 1 ulp)."""
import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import rpn_oracle as O
from oracle import target_layouts as TL

F32 = np.float32
pytestmark = pytest.mark.skipif(not CO.available(), reason="C oracle not built (make -C oracle)")


def close(a, b):
    return np.all(np.abs(a.astype(np.float64) - b) <= 1e-6 * np.maximum(1, np.abs(b)))


def bits(a):
    return np.ascontiguousarray(a, F32).view(np.uint32)


def test_c_oracle_matches_golden(golden):
    assert np.array_equal(bits(CO.iou_map(golden["iou_boxes"], golden["iou_gt"])), bits(golden["iou_map_batched"]))
    assert close(CO.decode(golden["iou_boxes"], golden["dec_deltas"]), golden["dec_boxes_batched"])
    assert close(CO.encode(golden["enc_boxes"], golden["enc_gt"]), golden["enc_deltas"])
    r = CO.nms(golden["nms_in_boxes"], golden["nms_in_scores"], 50, 60, 0.3, 0.25)
    assert np.array_equal(bits(r[0]), bits(golden["nms_out_boxes"])) and np.array_equal(r[3], golden["nms_out_valid"])
    assert np.array_equal(bits(r[1]), bits(golden["nms_out_scores"]))


@pytest.mark.parametrize("bb,B,G", [("vgg16", 3, 20), ("mobilenet_v2", 2, 50)])
def test_targets_numpy_vs_c(bb, B, G):
    from tfrpn import synthetic
    hp = O.get_hyper_params(bb)
    anchors = O.generate_anchors(hp)
    gtb, gtl = synthetic.gt_batch(np.random.default_rng(B + G), B, G)
    d, l, dbg = O.calculate_rpn_actual_outputs(anchors, gtb, gtl, hp, seed=7, offset=9, image_offset=2, return_debug=True)
    cd, cl, cdbg = CO.rpn_targets(anchors, gtb, gtl, hp, seed=7, offset=9, image_offset=2, debug=True)
    assert np.array_equal(cl, l.reshape(B, -1))
    assert np.array_equal(cdbg["argmax_row"], dbg["argmax_row"]) and np.array_equal(cdbg["argmax_col"], dbg["argmax_col"])
    assert np.array_equal(cdbg["pos_pre"].astype(bool), dbg["pos_pre"])
    assert np.array_equal(cdbg["neg_pre"].astype(bool), dbg["neg_pre"])
    assert np.array_equal(cd != 0, d != 0) and close(cd, d)


@pytest.mark.parametrize("name", TL.FALLBACK_LAYOUTS)
def test_targets_numpy_vs_c_fallback_layouts(name):
    """Pixel coordinates, tiny coordinates, flipped boxes, NaN / inf, zero-area anchors, NaN columns
    (oracle/target_layouts.py).  The NumPy oracle takes np.maximum / np.minimum (NaN-propagating), the C oracle
    fmaxf / fminf (NaN-ignoring): a NaN coordinate still gives a NaN area, hence a NaN union and IoU, on both
    sides, and inf - inf inside the intersection only arises with an infinite extent, whose area is NaN too.
    So the two agree on every output, bit for bit, except one: max_iou where an anchor's best IoU is a zero of
    both signs (a flipped GT box of negative area gives -0).  The C oracle keeps the first maximal value (its
    `v > best` scan), as the kernel does; NumPy's max reduction may return the other zero.  The values are equal,
    so no threshold sees the difference."""
    anchors, gtb, gtl = TL.fallback_layout(name)
    B, N = gtl.shape[0], anchors.shape[0]
    hp = dict(O.get_hyper_params("vgg16"), feature_map_shape=(1, N))
    hp["anchor_count"] = 1
    with np.errstate(invalid="ignore", over="ignore"):
        d, l, dbg = O.calculate_rpn_actual_outputs(anchors, gtb, gtl, hp, seed=3, offset=5, image_offset=1,
                                                   return_debug=True)
    cd, cl, cdbg = CO.rpn_targets(anchors, gtb, gtl, hp, seed=3, offset=5, image_offset=1, debug=True)
    assert np.array_equal(bits(cl), bits(l.reshape(B, -1)))
    assert np.array_equal(cdbg["argmax_row"], dbg["argmax_row"]) and np.array_equal(cdbg["argmax_col"], dbg["argmax_col"])
    assert np.array_equal(cdbg["max_iou"], dbg["max_iou"])
    zero = cdbg["max_iou"] == 0
    assert np.array_equal(bits(cdbg["max_iou"])[~zero], bits(dbg["max_iou"])[~zero])
    assert np.array_equal(cdbg["pos_pre"].astype(bool), dbg["pos_pre"])
    assert np.array_equal(cdbg["neg_pre"].astype(bool), dbg["neg_pre"])
    assert np.array_equal(np.isnan(cd), np.isnan(d))
    fin = ~np.isnan(d)
    assert np.array_equal(cd[fin] != 0, d[fin] != 0) and close(cd[fin], d[fin])


def test_select_topk_proposals_numpy_vs_c():
    from tfrpn import synthetic
    rng = np.random.default_rng(4)
    mask = rng.uniform(size=(3, 3000)) < 0.4
    assert np.array_equal(CO.select_mask(mask, [100, 5, 0], seed=3, offset=1, stream=1, image_offset=5),
                          O.randomly_select_xyz_mask(mask, [100, 5, 0], seed=3, offset=1, stream=1, image_offset=5))
    s = (rng.integers(0, 50, size=(2, 700)) / 50).astype(F32)
    v, i = CO.top_k(s, 300)
    ov, oi = O.top_k(s, 300)
    assert np.array_equal(i, oi) and np.array_equal(v, ov)
    hp = O.get_hyper_params("vgg16")
    anchors = O.generate_anchors(hp)
    reg, cls = synthetic.head_outputs(rng, 2, 31, 31, 9)
    cb, cs, cv, ck = CO.proposals(reg, cls, anchors, hp)
    ob, os_, ov, ok = O.generate_proposals(reg, cls, anchors, hp)
    assert np.array_equal(cv, ov) and np.array_equal(ck, ok) and np.array_equal(cs, os_) and close(cb, ob)


def test_clip_sends_nan_to_zero_numpy_vs_c():
    """Both restatements clip to [0, 1] with NaN-ignoring max / min (include/tfrpn.h): a NaN coordinate becomes 0.
    NaN regressions on the best-scoring rows and a zero-extent anchor whose exp overflows (0 * inf = NaN) reach the
    proposal stage's clip; NaN boxes among the NMS inputs reach its clip_boxes.  A NaN box neither suppresses nor is
    suppressed on either side, so the keep lists agree too."""
    from tfrpn import synthetic
    rng = np.random.default_rng(12)
    hp = O.get_hyper_params("vgg16")
    anchors = O.generate_anchors(hp)
    anchors[7] = [0.4, 0.4, 0.4, 0.4]                       # zero extent
    reg, cls = synthetic.head_outputs(rng, 2, 31, 31, 9)
    reg = reg.reshape(2, -1, 4)
    cls = cls.reshape(2, -1)
    top = np.argsort(-cls, axis=1)[:, :40]
    reg[0, top[0, ::3], 1] = np.nan
    reg[1, top[1, ::2]] = np.nan
    reg[:, 7, 2:] = 1000.0
    cls[:, 7] = 1.0
    with np.errstate(invalid="ignore", over="ignore"):
        ob, os_, ov, ok = O.generate_proposals(reg, cls, anchors, hp)
    cb, cs, cv, ck = CO.proposals(reg, cls, anchors, hp)
    assert not np.isnan(ob).any() and np.array_equal(ok[:, 0], [7, 7])
    assert np.array_equal(cv, ov) and np.array_equal(ck, ok) and np.array_equal(cs, os_) and close(cb, ob)
    boxes, scores = synthetic.nms_boxes(rng, 2, 300)
    boxes[0, ::5, 0] = np.nan
    boxes[1, ::7] = np.nan
    boxes[1, 1::7, 3] = np.nan
    r = CO.nms(boxes, scores, 100, 120, 0.5)
    with np.errstate(invalid="ignore"):
        w = O.combined_non_max_suppression(boxes[:, :, None], scores[:, :, None], 100, 120, 0.5, return_indices=True)
    assert not np.isnan(w[0]).any()
    assert np.array_equal(r[3], w[3]) and np.array_equal(r[4], w[4])
    assert np.array_equal(bits(r[0]), bits(w[0])) and np.array_equal(bits(r[1]), bits(w[1]))

"""oracle/crop_oracle.py (tf.image.crop_and_resize, bilinear, and its image gradient) on the CPU: hand-derived cases,
a literal float32 restatement of TensorFlow's CPU loops (bit-exact), a float64 direct evaluation and the float64
adjoint (the inner-product identity <crop(x), g> == <x, grad(g)>)."""
import math

import numpy as np
import pytest

from oracle import crop_oracle as K

F32 = np.float32
NAN, INF = float("nan"), float("inf")


def tf_loops(image, boxes, box_index, ch, cw, extrap, grad=None):
    """CropAndResize / CropAndResizeGradImage as TensorFlow's CPU kernels loop, one np.float32 scalar op at a time.
    -> crops, or grad_image when ``grad`` is given."""
    B, H, W, C = image.shape
    M = len(boxes)
    f = F32
    out = np.zeros((M, ch, cw, C), F32)
    gi = np.zeros((B, H, W, C), F32)

    def coord(lo, hi, L, n, i):
        if n > 1:
            scale = (hi - lo) * f(L - 1) / f(n - 1)
            return lo * f(L - 1) + f(i) * scale
        return f(0.5 * float(lo + hi) * (L - 1))

    with np.errstate(all="ignore"):
        for m in range(M):
            y1, x1, y2, x2 = (f(v) for v in boxes[m])
            b = int(box_index[m])
            bad = not 0 <= b < B
            for y in range(ch):
                in_y = coord(y1, y2, H, ch, y)
                for x in range(cw):
                    in_x = coord(x1, x2, W, cw, x)
                    if bad:
                        out[m, y, x] = np.nan
                        continue
                    if not (in_y >= 0 and in_y <= f(H - 1) and in_x >= 0 and in_x <= f(W - 1)):
                        out[m, y, x] = f(extrap)
                        continue
                    t, bo = int(math.floor(in_y)), int(math.ceil(in_y))
                    le, r = int(math.floor(in_x)), int(math.ceil(in_x))
                    yl, xl = in_y - f(t), in_x - f(le)
                    for c in range(C):
                        tl, tr, bl, br = image[b, t, le, c], image[b, t, r, c], image[b, bo, le, c], image[b, bo, r, c]
                        top = tl + (tr - tl) * xl
                        bot = bl + (br - bl) * xl
                        out[m, y, x, c] = top + (bot - top) * yl
                        if grad is not None:
                            g = grad[m, y, x, c]
                            dtop = (f(1) - yl) * g
                            gi[b, t, le, c] += (f(1) - xl) * dtop
                            gi[b, t, r, c] += xl * dtop
                            dbot = yl * g
                            gi[b, bo, le, c] += (f(1) - xl) * dbot
                            gi[b, bo, r, c] += xl * dbot
    return out if grad is None else gi


def same_bits(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def image_of(rng, B, H, W, C):
    return rng.normal(size=(B, H, W, C)).astype(F32)


def test_integer_samples_copy_pixels():
    """H = W = 5, crop 3 x 3 of the whole image: in_y, in_x = 0, 2, 4 -- top == bottom, left == right, lerps 0"""
    img = image_of(np.random.default_rng(0), 1, 5, 5, 3)
    boxes = np.array([[0, 0, 1, 1]], F32)
    out = K.crop_and_resize(img, boxes, [0], (3, 3))
    assert same_bits(out[0], img[0][::2, ::2])
    g = np.random.default_rng(1).normal(size=out.shape).astype(F32)
    gi = K.crop_and_resize_grad_image(g, boxes, [0], img.shape)
    want = np.zeros_like(img)
    want[0, ::2, ::2] = g[0]           # term 1 is g, terms 2-4 are +-0
    assert same_bits(gi, want)


def test_single_row_and_column_use_the_centre_in_float64():
    """ch == cw == 1: in = 0.5*(lo+hi)*(L-1) with lo+hi in float32 and the rest in float64, rounded once"""
    H, W = 1000, 777
    rng = np.random.default_rng(2)
    boxes = rng.uniform(0, 1, size=(200, 4)).astype(F32)
    got = K.sample_grid(boxes[:, 0], boxes[:, 2], H, 1)[:, 0]
    want = [F32(0.5 * float(F32(a) + F32(b)) * (H - 1)) for a, b in boxes[:, [0, 2]]]
    assert same_bits(got, want)
    # the float32 sum is part of the rule: a float64 sum gives other bits for some boxes
    wide = [F32(0.5 * (float(a) + float(b)) * (H - 1)) for a, b in boxes[:, [0, 2]]]
    assert not same_bits(got, wide)
    img = image_of(rng, 1, H, W, 2)
    assert same_bits(K.crop_and_resize(img, boxes[:20], np.zeros(20, np.int32), (1, 1)),
                     tf_loops(img, boxes[:20], np.zeros(20), 1, 1, 0.0))


def test_single_pixel_image_height():
    """H == 1: every finite row samples row 0 (scale (y2-y1)*0 = 0); an infinite y1 gives NaN, extrapolated"""
    img = image_of(np.random.default_rng(3), 1, 1, 6, 2)
    boxes = np.array([[0.2, 0.0, 0.9, 1.0], [-3.0, 0.0, 5.0, 1.0], [INF, 0.0, 0.5, 1.0]], F32)
    out = K.crop_and_resize(img, boxes, [0, 0, 0], (3, 6), extrapolation_value=-1.0)
    assert same_bits(out[0], np.broadcast_to(img[0, 0], (3, 6, 2)))
    assert same_bits(out[1], out[0])
    assert (out[2] == -1).all()


def test_partly_and_wholly_outside_boxes():
    img = image_of(np.random.default_rng(4), 1, 5, 5, 2)
    # rows: in_y = -2, -1, 0, 1, 2; columns 0..4
    boxes = np.array([[-0.5, 0.0, 0.5, 1.0], [1.5, 0.0, 2.0, 1.0]], F32)
    out = K.crop_and_resize(img, boxes, [0, 0], (5, 5), extrapolation_value=7.5)
    assert (out[0, :2] == 7.5).all() and same_bits(out[0, 2:], img[0, :3])
    assert (out[1] == 7.5).all()
    g = np.ones(out.shape, F32)
    gi = K.crop_and_resize_grad_image(g, boxes, [0, 0], img.shape)
    want = np.zeros_like(img)
    want[0, :3] = 1
    assert same_bits(gi, want)


def test_flipped_boxes_reverse_the_samples():
    img = image_of(np.random.default_rng(5), 1, 5, 9, 3)
    up = K.crop_and_resize(img, np.array([[0, 0, 1, 1]], F32), [0], (5, 9))
    down = K.crop_and_resize(img, np.array([[1, 1, 0, 0]], F32), [0], (5, 9))
    assert same_bits(down[0], up[0, ::-1, ::-1])
    rng = np.random.default_rng(6)
    boxes = rng.uniform(0, 1, size=(6, 4)).astype(F32)
    boxes[:, :2], boxes[:, 2:] = np.maximum(boxes[:, :2], boxes[:, 2:]), np.minimum(boxes[:, :2], boxes[:, 2:])
    g = rng.normal(size=(6, 4, 3, 3)).astype(F32)
    assert same_bits(K.crop_and_resize_grad_image(g, boxes, np.zeros(6, np.int32), img.shape),
                     tf_loops(img, boxes, np.zeros(6), 4, 3, 0.0, grad=g))


def test_nan_and_infinite_coordinates_are_extrapolated():
    img = image_of(np.random.default_rng(7), 1, 4, 4, 2)
    boxes = np.array([[NAN, 0, 1, 1], [0, NAN, 1, 1], [0, 0, INF, 1], [0, -INF, 1, 1], [-INF, 0, INF, 1],
                      [0, 0, 1, 1]], F32)
    out = K.crop_and_resize(img, boxes, np.zeros(6, np.int32), (3, 3), extrapolation_value=0.25)
    assert (out[:5] == F32(0.25)).all()
    # y2 = inf: row 0 is y1*(H-1) + 0*inf = NaN, the others +inf -- all extrapolated, no gradient
    gi = K.crop_and_resize_grad_image(np.ones(out[:5].shape, F32), boxes[:5], np.zeros(5, np.int32), img.shape)
    assert same_bits(gi, np.zeros_like(img))


def test_bad_box_index_writes_nan_and_adds_no_gradient():
    img = image_of(np.random.default_rng(8), 2, 4, 4, 3)
    boxes = np.array([[0, 0, 1, 1]] * 4, F32)
    idx = np.array([-1, 2, 1, 1 << 30], np.int32)
    out = K.crop_and_resize(img, boxes, idx, (2, 2))
    assert np.isnan(out[[0, 1, 3]]).all() and not np.isnan(out[2]).any()
    gi = K.crop_and_resize_grad_image(np.ones(out.shape, F32), boxes, idx, img.shape)
    assert (gi[0] == 0).all() and gi[1].sum() == 2 * 2 * 3


def test_batched_layout_is_an_index_of_m_over_s():
    assert np.array_equal(K.batched_index(6, 3), [0, 0, 1, 1, 2, 2])
    with pytest.raises(ValueError):
        K.batched_index(7, 3)


@pytest.mark.parametrize("ch,cw", [(3, 4), (1, 5), (7, 1), (2, 2)])
def test_oracle_is_tensorflows_loop_bit_for_bit(ch, cw):
    """forward and gradient against the literal float32 loops, on layouts with shared pixels, tiny and degenerate
    boxes (many terms per pixel), boxes beyond the image, flipped boxes and an explicit unsorted box_index"""
    rng = np.random.default_rng(10 + ch * 7 + cw)
    B, H, W, C = 3, 6, 7, 3
    img = image_of(rng, B, H, W, C)
    M = 14
    boxes = rng.uniform(-0.2, 1.2, size=(M, 4)).astype(F32)
    boxes[3] = [0.5, 0.5, 0.5, 0.5]                   # zero size: every sample on one point
    boxes[4] = [0.41, 0.37, 0.43, 0.39]               # tiny
    boxes[5] = [0.0, 0.0, 1.0, 1.0]
    idx = rng.integers(0, B, size=M).astype(np.int32)
    idx[6] = -2
    g = rng.normal(size=(M, ch, cw, C)).astype(F32)
    assert same_bits(K.crop_and_resize(img, boxes, idx, (ch, cw), 0.5), tf_loops(img, boxes, idx, ch, cw, 0.5))
    assert same_bits(K.crop_and_resize_grad_image(g, boxes, idx, img.shape), tf_loops(img, boxes, idx, ch, cw, 0, g))


def direct64(image, boxes, box_index, ch, cw, extrap, grad=None):
    """float64 evaluation of the same sampling (coordinates in float64 too); with ``grad`` the adjoint"""
    B, H, W, C = image.shape
    image = image.astype(np.float64)
    out = np.zeros((len(boxes), ch, cw, C))
    gi = np.zeros((B, H, W, C))

    def coord(lo, hi, L, n, i):
        return lo * (L - 1) + i * (hi - lo) * (L - 1) / (n - 1) if n > 1 else 0.5 * (lo + hi) * (L - 1)

    for m, (y1, x1, y2, x2) in enumerate(boxes.astype(np.float64)):
        b = int(box_index[m])
        for y in range(ch):
            in_y = coord(y1, y2, H, ch, y)
            for x in range(cw):
                in_x = coord(x1, x2, W, cw, x)
                if not (0 <= in_y <= H - 1 and 0 <= in_x <= W - 1):
                    out[m, y, x] = extrap
                    continue
                t, bo, le, r = math.floor(in_y), math.ceil(in_y), math.floor(in_x), math.ceil(in_x)
                yl, xl = in_y - t, in_x - le
                w = ((t, le, (1 - yl) * (1 - xl)), (t, r, (1 - yl) * xl), (bo, le, yl * (1 - xl)), (bo, r, yl * xl))
                for row, col, wt in w:
                    out[m, y, x] += wt * image[b, row, col]
                    if grad is not None:
                        gi[b, row, col] += wt * grad[m, y, x]
    return out if grad is None else gi


def random_case(seed, B=2, H=9, W=11, C=5, M=12, ch=4, cw=6):
    rng = np.random.default_rng(seed)
    img = image_of(rng, B, H, W, C)
    lo = rng.uniform(0.02, 0.6, size=(M, 2))
    boxes = np.concatenate([lo, lo + rng.uniform(0.05, 0.38, size=(M, 2))], axis=1).astype(F32)
    idx = rng.integers(0, B, size=M).astype(np.int32)
    g = rng.normal(size=(M, ch, cw, C)).astype(F32)
    return img, boxes, idx, g, (ch, cw)


@pytest.mark.parametrize("seed,crop", [(20, (4, 6)), (21, (7, 7)), (22, (1, 3))])
def test_forward_against_float64(seed, crop):
    img, boxes, idx, _, _ = random_case(seed, ch=crop[0], cw=crop[1])
    got = K.crop_and_resize(img, boxes, idx, crop)
    want = direct64(img, boxes, idx, *crop, 0.0)
    assert np.abs(got - want).max() <= 1e-5 * (1 + np.abs(img).max())


@pytest.mark.parametrize("seed,crop", [(30, (4, 6)), (31, (7, 7)), (32, (3, 1))])
def test_gradient_against_the_float64_adjoint(seed, crop):
    img, boxes, idx, g, _ = random_case(seed, ch=crop[0], cw=crop[1])
    adj = direct64(img, boxes, idx, *crop, 0.0, grad=g.astype(np.float64))
    fwd = direct64(img, boxes, idx, *crop, 0.0)
    lhs, rhs = float((fwd * g).sum()), float((img.astype(np.float64) * adj).sum())
    assert abs(lhs - rhs) <= 1e-12 * (abs(lhs) + abs(rhs) + 1)        # the float64 pair is an adjoint pair
    got = K.crop_and_resize_grad_image(g, boxes, idx, img.shape)
    assert np.abs(got - adj).max() <= 1e-5 * (1 + np.abs(adj).max())
    # and the float32 oracle pair satisfies the identity to float32 accuracy
    lhs32 = float((K.crop_and_resize(img, boxes, idx, crop).astype(np.float64) * g).sum())
    rhs32 = float((img.astype(np.float64) * got).sum())
    assert abs(lhs32 - rhs32) <= 1e-5 * (abs(lhs32) + 1)


def test_chunked_evaluation_is_the_whole_evaluation(monkeypatch):
    """the oracle walks boxes in chunks; a pixel's terms must still add in ascending box order across chunks"""
    img, boxes, idx, g, crop = random_case(40, M=40)
    boxes[::3] = [0.3, 0.3, 0.31, 0.31]             # many boxes on the same pixels
    whole = K.crop_and_resize_grad_image(g, boxes, idx, img.shape), K.crop_and_resize(img, boxes, idx, crop)
    monkeypatch.setattr(K, "_CHUNK_ELEMS", 1)
    assert same_bits(K.crop_and_resize_grad_image(g, boxes, idx, img.shape), whole[0])
    assert same_bits(K.crop_and_resize(img, boxes, idx, crop), whole[1])

"""tfrpn_crop_and_resize / tfrpn_crop_and_resize_grad_image (crop_kernel, crop_grad_kernel) against
oracle/crop_oracle.py, bit for bit with NaN compared as NaN: at this library's chain (generate_proposals ->
roi_targets at C2), at a Detectron-like shape, at odd channel counts and crop sizes, with explicit unsorted and
duplicate box indices, and on adversarial layouts.  Then the properties: run-to-run and batching identity of the
gradient, graph replay, the autograd Function, streams, errors and limits."""

import numpy as np
import pytest

from oracle import crop_oracle as K
from oracle import rpn_oracle as O

pytestmark = pytest.mark.gpu
F32 = np.float32
NAN, INF = float("nan"), float("inf")
SENT = -7.25


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    import tfrpn

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.tfrpn, ns.dev = torch, tfrpn, cuda_device
    ns.cu = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    return ns


def forward(T, image, boxes, index, crop, extrap=0.0, stream=None):
    """direct C call, output prefilled with a sentinel -> device tensor"""
    from tfrpn import _lib
    torch = T.torch
    B, H, W, Cc = image.shape
    M = boxes.shape[0]
    out = torch.full((M, crop[0], crop[1], Cc), SENT, dtype=torch.float32, device=T.dev)
    st = stream or torch.cuda.current_stream(T.dev)
    _lib.check(_lib.load().tfrpn_crop_and_resize(image.data_ptr(), B, H, W, Cc, boxes.data_ptr(),
                                                 None if index is None else index.data_ptr(), M, crop[0], crop[1],
                                                 float(extrap), out.data_ptr(), st.cuda_stream))
    return out


def backward(T, grad, boxes, index, shape, stream=None):
    """direct C call, grad_image prefilled with a sentinel (it must be overwritten) -> device tensor"""
    from tfrpn import _lib
    torch = T.torch
    B, H, W, Cc = shape
    M, ch, cw = grad.shape[:3]
    gi = torch.full((B, H, W, Cc), SENT, dtype=torch.float32, device=T.dev)
    st = stream or torch.cuda.current_stream(T.dev)
    _lib.check(_lib.load().tfrpn_crop_and_resize_grad_image(grad.data_ptr(), boxes.data_ptr(),
                                                            None if index is None else index.data_ptr(), M, B, H, W,
                                                            Cc, ch, cw, gi.data_ptr(), st.cuda_stream))
    return gi


def same_bits(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    assert a.shape == b.shape, (a.shape, b.shape)
    bad = np.argwhere(~((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))
    assert bad.size == 0, (len(bad), bad[:8], a[tuple(bad[0])], b[tuple(bad[0])])


def check(T, image, boxes, index, crop, extrap=0.0, seed=0):
    """forward and gradient of the kernels against the oracle; -> (out, grad_image) host arrays"""
    image, boxes = np.asarray(image, F32), np.asarray(boxes, F32).reshape(-1, 4)
    idx = None if index is None else np.asarray(index, np.int32)
    img_d, box_d, idx_d = T.cu(image), T.cu(boxes), T.cu(idx)
    out = forward(T, img_d, box_d, idx_d, crop, extrap).cpu().numpy()
    same_bits(out, K.crop_and_resize(image, boxes, idx, crop, extrap))
    g = np.random.default_rng(seed).normal(size=out.shape).astype(F32)
    gi = backward(T, T.cu(g), box_d, idx_d, image.shape).cpu().numpy()
    same_bits(gi, K.crop_and_resize_grad_image(g, boxes, idx, image.shape))
    return out, gi


def rand_boxes(rng, shape, lo=0.02, hi=0.6):
    c = rng.uniform(0, 1, size=shape + (2,))
    s = rng.uniform(lo, hi, size=shape + (2,))
    return np.clip(np.concatenate([c - s / 2, c + s / 2], axis=-1), 0, 1).astype(F32)


def test_c2_chain(T):
    """generate_proposals -> roi_targets at C2 (B = 64, S = 128), VGG16 features 31 x 31 x 512, 7 x 7 crops"""
    from tfrpn import synthetic
    from tfrpn.utils import data_utils
    rng = np.random.default_rng(50)
    hp = O.get_hyper_params("vgg16")
    B, G = 64, 50
    fh, fw = O._pair(hp["feature_map_shape"])
    reg, cls = synthetic.head_outputs(rng, B, fh, fw, hp["anchor_count"])
    rois, _, valid, _ = T.tfrpn.generate_proposals(T.cu(reg), T.cu(cls), T.cu(O.generate_anchors(hp)), hp)
    gtb, gtl = synthetic.gt_batch(rng, B, G)
    n = (gtl >= 0).sum(axis=1)
    gb, gl = data_utils.pad_gt_batch([gtb[b, :n[b]] for b in range(B)], [gtl[b, :n[b]] - 1 for b in range(B)],
                                     max_boxes=G, label_add=1)
    t = T.tfrpn.roi_targets(rois, gb, gl, valid, num_classes=21, total_pos=32, total_neg=96, offset=3)
    feats = rng.normal(size=(B, fh, fw, 512)).astype(F32)
    boxes = t.rois.cpu().numpy()
    assert boxes.shape == (B, 128, 4)
    check(T, feats, boxes, None, (7, 7), seed=51)


def test_detectron_like(T):
    rng = np.random.default_rng(52)
    feats = rng.normal(size=(2, 50, 50, 256)).astype(F32)
    check(T, feats, rand_boxes(rng, (2, 512)), None, (14, 14), seed=53)


@pytest.mark.parametrize("Cc,crop", [(3, (7, 7)), (1, (5, 3)), (130, (7, 7)), (256, (1, 1)), (20, (32, 32)),
                                     (4096, (2, 3)), (516, (4, 4))])
def test_channels_and_crop_sizes(T, Cc, crop):
    rng = np.random.default_rng(54 + Cc)
    feats = rng.normal(size=(3, 13, 11, Cc)).astype(F32)
    check(T, feats, rand_boxes(rng, (3, 24)), None, crop, extrap=0.5, seed=55)


def test_unaligned_rows_take_the_scalar_path(T):
    """C % 4 == 0 but image and out 4 bytes off a 16-byte boundary: the same bits through scalar channels"""
    rng = np.random.default_rng(56)
    image = rng.normal(size=(2, 9, 9, 8)).astype(F32)
    boxes = rand_boxes(rng, (2, 10)).reshape(-1, 4)
    torch = T.torch
    flat = torch.zeros(image.size + 1, dtype=torch.float32, device=T.dev)
    flat[1:] = T.cu(image.reshape(-1))
    img_d = flat[1:].view(image.shape)
    out = forward(T, img_d, T.cu(boxes), None, (5, 5))
    same_bits(out.cpu().numpy(), K.crop_and_resize(image, boxes, None, (5, 5)))


def test_explicit_index_unsorted_and_duplicate(T):
    """explicit box_index: the NULL layout after a permutation (with duplicated boxes); an order that keeps each
    image's boxes in order gives the same gradient bits as the NULL layout"""
    rng = np.random.default_rng(57)
    B, S, Cc = 4, 48, 64
    feats = rng.normal(size=(B, 17, 19, Cc)).astype(F32)
    boxes = rand_boxes(rng, (B, S)).reshape(-1, 4)
    null_idx = K.batched_index(B * S, B)
    perm = np.concatenate([rng.permutation(B * S), rng.integers(0, B * S, size=40)])
    out, _ = check(T, feats, boxes[perm], null_idx[perm], (7, 7), seed=58)
    ref, gref = check(T, feats, boxes, None, (7, 7), seed=59)
    same_bits(out, ref[perm])
    inter = np.argsort(np.arange(B * S) % S, kind="stable")     # round robin over images, each in its own order
    g = np.random.default_rng(59).normal(size=ref.shape).astype(F32)
    gi = backward(T, T.cu(g[inter]), T.cu(boxes[inter]), T.cu(null_idx[inter]), feats.shape).cpu().numpy()
    same_bits(gi, gref)


def adversarial_boxes():
    b = [[0, 0, 1, 1], [1, 1, 0, 0], [-0.5, -0.5, 0.5, 0.5], [1.5, 0, 2, 1], [0.5, 0.5, 0.5, 0.5],
         [0.3, 0.3, 0.3001, 0.3001], [NAN, 0, 1, 1], [0, NAN, 1, 1], [0, 0, INF, 1], [-INF, 0, INF, 1],
         [0, 0, 1e30, 1], [-0.0, -0.0, 0.25, 0.25], [-0.0, -0.0, -0.25, -0.25], [0.25, 0.25, 0.75, 0.75],
         [0.999999, 0.999999, 1.0, 1.0], [0, 0.25, 1, 0.25]]
    return np.array(b, F32)


@pytest.mark.parametrize("crop", [(7, 7), (1, 1), (2, 9), (32, 32)])
def test_adversarial_layouts(T, crop):
    """integer samples (top == bottom), flipped, partly / wholly outside, zero-size boxes (every sample on one
    point: long term sequences on one pixel), NaN / inf, -0 corners, boxes on tile edges, bad indices"""
    rng = np.random.default_rng(60)
    B, H, W, Cc = 3, 9, 13, 12
    feats = rng.normal(size=(B, H, W, Cc)).astype(F32)
    boxes = np.concatenate([adversarial_boxes()] * 3)
    idx = np.repeat(np.arange(3), len(adversarial_boxes())).astype(np.int32)
    idx[[5, 20, 33]] = [-1, 3, 1 << 30]
    check(T, feats, boxes, idx, crop, extrap=-3.0, seed=61)
    one = np.ones((1, 1, 1, Cc), F32)
    check(T, one * feats[:1, :1, :1], boxes, np.zeros(len(boxes), np.int32), crop, seed=62)         # H == W == 1
    check(T, feats[:, :1], boxes, idx.clip(0, 2), crop, seed=63)                               # H == 1


def test_gradient_is_run_and_batching_invariant(T):
    """the same bits twice, and one batched call equals one call per image (a pixel's terms come from its own
    image's boxes only)"""
    torch = T.torch
    rng = np.random.default_rng(64)
    B, S, Cc = 5, 64, 128
    feats_shape = (B, 21, 23, Cc)
    boxes = rand_boxes(rng, (B, S)).reshape(-1, 4)
    g = rng.normal(size=(B * S, 7, 7, Cc)).astype(F32)
    bd, gd = T.cu(boxes), T.cu(g)
    a = backward(T, gd, bd, None, feats_shape)
    b = backward(T, gd, bd, None, feats_shape)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    for i in range(B):
        one = backward(T, gd[i * S:(i + 1) * S].contiguous(), bd[i * S:(i + 1) * S].contiguous(), None,
                       (1,) + feats_shape[1:])
        assert torch.equal(one[0].view(torch.int32), a[i].view(torch.int32)), i


def test_graph_replay(T):
    torch = T.torch
    rng = np.random.default_rng(65)
    feats = T.cu(rng.normal(size=(4, 31, 31, 256)).astype(F32))
    boxes = T.cu(rand_boxes(rng, (4, 128)).reshape(-1, 4))
    g = T.cu(rng.normal(size=(512, 7, 7, 256)).astype(F32))
    ref_out, ref_gi = forward(T, feats, boxes, None, (7, 7)), backward(T, g, boxes, None, feats.shape)
    s = torch.cuda.Stream(T.dev)
    s.wait_stream(torch.cuda.current_stream(T.dev))
    with torch.cuda.stream(s):
        forward(T, feats, boxes, None, (7, 7), stream=s)
    torch.cuda.current_stream(T.dev).wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = forward(T, feats, boxes, None, (7, 7))
        gi = backward(T, g, boxes, None, feats.shape)
    for _ in range(3):
        out.fill_(SENT)
        gi.fill_(SENT)
        graph.replay()
        torch.cuda.synchronize(T.dev)
        assert torch.equal(out.view(torch.int32), ref_out.view(torch.int32))
        assert torch.equal(gi.view(torch.int32), ref_gi.view(torch.int32))


def test_autograd_function(T):
    """tfrpn.crop_and_resize: the Function's image gradient is the oracle's; the crop is linear in the image, so
    <crop(x + v) - crop(x), g> == <v, grad(g)> up to float32 rounding; boxes get no gradient"""
    torch = T.torch
    rng = np.random.default_rng(66)
    B, S, Cc = 3, 40, 36
    x = rng.normal(size=(B, 15, 16, Cc)).astype(F32)
    boxes = rand_boxes(rng, (B, S))
    g = rng.normal(size=(B, S, 6, 5, Cc)).astype(F32)
    xd = T.cu(x).requires_grad_(True)
    bd = T.cu(boxes).requires_grad_(True)
    out = T.tfrpn.crop_and_resize(xd, bd, None, (6, 5))
    assert out.shape == (B, S, 6, 5, Cc) and out.grad_fn is not None
    same_bits(out.detach().cpu().numpy().reshape(-1, 6, 5, Cc), K.crop_and_resize(x, boxes.reshape(-1, 4), None, (6, 5)))
    out.backward(T.cu(g))
    want = K.crop_and_resize_grad_image(g.reshape(-1, 6, 5, Cc), boxes.reshape(-1, 4), None, x.shape)
    same_bits(xd.grad.cpu().numpy(), want)
    assert bd.grad is None
    v = rng.normal(size=x.shape).astype(F32)
    with torch.no_grad():
        d = T.tfrpn.crop_and_resize(T.cu(x + v), T.cu(boxes), None, (6, 5)) - out
    lhs = float((d.double() * T.cu(g).double()).sum())
    rhs = float((T.cu(v).double() * xd.grad.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * (abs(lhs) + 1)
    # explicit indices, a NumPy round trip (no autograd there), the output is not retained by the graph
    idx = rng.integers(0, B, size=17).astype(np.int32)
    flat = boxes.reshape(-1, 4)[:17]
    got = T.tfrpn.crop_and_resize(x, flat, idx, (3, 3), extrapolation_value=1.0)
    assert isinstance(got, np.ndarray)
    same_bits(got, K.crop_and_resize(x, flat, idx, (3, 3), 1.0))


def test_non_default_stream(T):
    torch = T.torch
    rng = np.random.default_rng(67)
    feats = rng.normal(size=(2, 20, 20, 64)).astype(F32)
    boxes = rand_boxes(rng, (2, 32)).reshape(-1, 4)
    g = rng.normal(size=(64, 7, 7, 64)).astype(F32)
    s = torch.cuda.Stream(T.dev)
    fd, bd, gd = T.cu(feats), T.cu(boxes), T.cu(g)
    s.wait_stream(torch.cuda.current_stream(T.dev))
    with torch.cuda.stream(s):
        out = forward(T, fd, bd, None, (7, 7), stream=s)
        gi = backward(T, gd, bd, None, feats.shape, stream=s)
        via_py = T.tfrpn.crop_and_resize(fd, bd.view(2, 32, 4), None, (7, 7))
    s.synchronize()
    same_bits(out.cpu().numpy(), K.crop_and_resize(feats, boxes, None, (7, 7)))
    same_bits(via_py.cpu().numpy().reshape(out.shape), out.cpu().numpy())
    same_bits(gi.cpu().numpy(), K.crop_and_resize_grad_image(g, boxes, None, feats.shape))


def test_argument_errors_and_limits(T):
    from tfrpn import _lib
    torch = T.torch
    lib = _lib.load()
    buf = torch.zeros(1 << 16, dtype=torch.float32, device=T.dev)
    idx = torch.zeros(64, dtype=torch.int32, device=T.dev)
    p = buf.data_ptr()
    o = p + (1 << 15)        # outputs of the accepted calls: at most 128 floats
    st = torch.cuda.current_stream(T.dev).cuda_stream

    def fwd(image=p, B=2, H=4, W=4, Cc=4, boxes=p, index=None, M=4, ch=2, cw=2, out=o):
        return lib.tfrpn_crop_and_resize(image, B, H, W, Cc, boxes, index, M, ch, cw, 0.0, out, st)

    def bwd(grad=p, boxes=p, index=None, M=4, B=2, H=4, W=4, Cc=4, ch=2, cw=2, out=o):
        return lib.tfrpn_crop_and_resize_grad_image(grad, boxes, index, M, B, H, W, Cc, ch, cw, out, st)

    for call in (fwd, bwd):
        assert call() == 0
        for kw in (dict(image=None) if call is fwd else dict(grad=None), dict(boxes=None), dict(out=None), dict(B=0),
                   dict(H=0), dict(W=-1), dict(Cc=0), dict(M=0), dict(ch=0), dict(cw=0), dict(M=3)):
            assert call(**kw) == -1, (call.__name__, kw)
        assert call(M=3, index=idx.data_ptr()) == 0                    # an explicit index lifts M % B
        assert call(boxes=p + 4) == -2
        for kw in (dict(Cc=4097), dict(ch=33), dict(cw=33), dict(H=8193), dict(W=8193), dict(B=65536, M=65536),
                   dict(M=(1 << 24) + 2)):
            assert call(**kw) == -5, (call.__name__, kw)
    torch.cuda.synchronize(T.dev)
    feats = torch.zeros((1, 4, 4, 4), device=T.dev)
    boxes = torch.zeros((1, 2, 4), device=T.dev)
    with pytest.raises(NotImplementedError):
        T.tfrpn.crop_and_resize(feats, boxes, None, (2, 2), method="nearest")
    with pytest.raises(ValueError):
        T.tfrpn.crop_and_resize(feats, boxes, None, (2, 2), method="bicubic")
    with pytest.raises(NotImplementedError):
        T.tfrpn.crop_and_resize(torch.zeros((1, 2, 2, 4100), device=T.dev), boxes, None, (2, 2))
    with pytest.raises(NotImplementedError):
        T.tfrpn.crop_and_resize(feats, boxes, None, (33, 2))
    with pytest.raises(ValueError):
        T.tfrpn.crop_and_resize(feats, boxes.view(2, 4), None, (2, 2))                  # (M,4) needs indices
    with pytest.raises(ValueError):
        T.tfrpn.crop_and_resize(feats, boxes.view(2, 4), torch.zeros(3, dtype=torch.int32, device=T.dev), (2, 2))
    with pytest.raises(ValueError):
        T.tfrpn.crop_and_resize(feats.double(), boxes, None, (2, 2))

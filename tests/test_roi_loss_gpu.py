"""tfrpn_roi_head_losses (roi_loss_partial_kernel, roi_loss_grad_kernel) against oracle/roi_loss_oracle.py: losses to
1e-6 relative, counts exact, grad_deltas bit for bit, grad_logits to 1e-6 * inv_rows * |scale|, with every output
prefilled with a sentinel.  Shapes: the C2 chain, Detectron-like, C from 2 to 1024, q = 1 and q = C, misaligned
logits, all-padding images, and the real chain roi_targets -> crop_and_resize -> a linear head -> the losses ->
backward.  Then the properties: run-to-run bits, graph replay, a non-default stream, the autograd Function, launch
counts, errors and limits."""
import ctypes as C

import numpy as np
import pytest

from oracle import roi_loss_oracle as L

pytestmark = pytest.mark.gpu
F32 = np.float32
SENT = -7.25
LOSS_RTOL = 1e-6


@pytest.fixture(scope="module")
def T(cuda_device):
    import torch
    import tfrpn
    from tfrpn import _lib

    class Ns:
        pass
    ns = Ns()
    ns.torch, ns.tfrpn, ns.L, ns.lib, ns.dev = torch, tfrpn, _lib, _lib.load(), cuda_device
    ns.cu = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    ns.h = _lib.handle(cuda_device.index or 0)
    return ns


def case(rng, B, S, Cn, q, fg_frac=0.25, pad_frac=0.2, scale=2.0):
    x = rng.normal(0, scale, size=(B, S, Cn)).astype(F32)
    d = rng.normal(0, 1, size=(B, S, q, 4)).astype(F32)
    t = rng.normal(0, 1, size=(B, S, 4)).astype(F32)
    u = rng.uniform(size=(B, S))
    lab = np.where(u < fg_frac, rng.integers(1, Cn, size=(B, S)), 0)
    lab = np.where(u > 1 - pad_frac, -1, lab).astype(np.int32)
    t[lab <= 0] = 0
    return x, d, lab, t


def cfg_of(Cn, q, delta=1.0, norm=0):
    from tfrpn import _lib
    return _lib.RoiLossCfg(Cn, q, delta, norm)


def call(T, x, d, lab, t, cfg, out, scale=None, gl=None, gd=None, stream=None, h=None, shape=None):
    """the C entry point on device tensors -> status"""
    p = lambda a: None if a is None else a.data_ptr()  # noqa: E731
    B, S = shape or lab.shape
    st = stream.cuda_stream if stream is not None else T.torch.cuda.current_stream(T.dev).cuda_stream
    return T.lib.tfrpn_roi_head_losses(h or T.h, p(x), p(d), p(lab), p(t), B, S, C.byref(cfg), p(out), p(scale),
                                       p(gl), p(gd), st)


def run(T, x, d, lab, t, delta=1.0, norm=0, scale=None, grads=True, stream=None):
    """direct call on host arrays, outputs prefilled with a sentinel -> dict like the oracle's"""
    torch = T.torch
    xd, dd, ld, td = T.cu(x), T.cu(d), T.cu(lab), T.cu(t)
    out = torch.full((8,), SENT, dtype=torch.float32, device=T.dev)
    gl = torch.full_like(xd, SENT) if grads else None
    gd = torch.full_like(dd, SENT) if grads else None
    sd = None if scale is None else T.cu(np.asarray(scale, F32))
    T.L.check(call(T, xd, dd, ld, td, cfg_of(x.shape[2], d.shape[2], delta, norm), out, sd, gl, gd, stream))
    torch.cuda.synchronize(T.dev)
    o = out.cpu().numpy()
    n = o.view(np.int32)
    r = dict(cls_loss=o[0], reg_loss=o[1], n_rows=int(n[2]), n_fg=int(n[3]), n_correct=int(n[4]),
             n_fg_correct=int(n[5]), reserved=n[6:8].tolist(), raw=o.tobytes())
    if grads:
        r["grad_logits"], r["grad_deltas"] = gl.cpu().numpy(), gd.cpu().numpy()
    return r


def loss_close(got, want, rtol=LOSS_RTOL):
    got, want = float(got), float(want)
    return (np.isnan(got) and np.isnan(want)) or abs(got - want) <= rtol * max(abs(want), 1e-30)


def same_bits(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    assert a.shape == b.shape, (a.shape, b.shape)
    bad = np.argwhere(~((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))
    assert bad.size == 0, (len(bad), bad[:8], a[tuple(bad[0])], b[tuple(bad[0])])


def check(T, x, d, lab, t, delta=1.0, norm=0, scale=None):
    """kernel against the oracle -> the kernel's result"""
    r = run(T, x, d, lab, t, delta, norm, scale)
    w = L.roi_head_losses(x, d, lab, t, delta, ("fg", "rows")[norm], scale)
    assert loss_close(r["cls_loss"], w["cls_loss"]), (r["cls_loss"], w["cls_loss"])
    assert loss_close(r["reg_loss"], w["reg_loss"]), (r["reg_loss"], w["reg_loss"])
    for k in ("n_rows", "n_fg", "n_correct", "n_fg_correct"):
        assert r[k] == w[k], (k, r[k], w[k])
    assert r["reserved"] == [0, 0]
    same_bits(r["grad_deltas"], w["grad_deltas"])
    s0 = 1.0 if scale is None else abs(float(scale[0]))
    tol = 1e-6 * (1.0 / max(w["n_rows"], 1)) * s0
    g, wg = r["grad_logits"], w["grad_logits"]
    assert np.array_equal(np.isnan(g), np.isnan(wg))
    ok = ~np.isnan(wg)
    assert np.all(np.abs(g[ok] - wg[ok]) <= tol), float(np.max(np.abs(g[ok] - wg[ok])))
    assert np.all(g[lab < 0] == 0)
    return r


@pytest.mark.parametrize("B,S,Cn,q", [(64, 128, 21, 21), (64, 128, 21, 1), (2, 512, 81, 81), (16, 512, 81, 81),
                                      (16, 512, 81, 1)])
def test_c2_and_detectron_shapes(T, B, S, Cn, q):
    rng = np.random.default_rng(B * 1000 + Cn + q)
    x, d, lab, t = case(rng, B, S, Cn, q)
    check(T, x, d, lab, t)
    check(T, x, d, lab, t, delta=1.0 / 9, norm=1, scale=(0.75, -3.0))


@pytest.mark.parametrize("Cn", [2, 3, 33, 1000, 1024])
@pytest.mark.parametrize("q", ["C", 1])
def test_class_counts(T, Cn, q):
    rng = np.random.default_rng(Cn)
    qq = Cn if q == "C" else 1
    x, d, lab, t = case(rng, 3, 200 if Cn < 1000 else 40, Cn, qq)
    check(T, x, d, lab, t, delta=0.5, norm=Cn % 2)
    check(T, x, d, lab, t, scale=(2.0, 0.0))


def test_misaligned_logits_same_bits(T):
    """logits and grad_logits 4 bytes off a 16-byte boundary (C % 4 == 0): the scalar path gives the float4 path's
    bits"""
    torch = T.torch
    rng = np.random.default_rng(7)
    B, S, Cn = 4, 96, 1000
    x, d, lab, t = case(rng, B, S, Cn, Cn)
    ref = check(T, x, d, lab, t)
    flat = torch.zeros(x.size + 1, dtype=torch.float32, device=T.dev)
    flat[1:] = T.cu(x.reshape(-1))
    xm = flat[1:].view(x.shape)
    gflat = torch.full((x.size + 1,), SENT, dtype=torch.float32, device=T.dev)
    glm = gflat[1:].view(x.shape)
    dd, ld, td = T.cu(d), T.cu(lab), T.cu(t)
    out = torch.full((8,), SENT, dtype=torch.float32, device=T.dev)
    gd = torch.full_like(dd, SENT)
    T.L.check(call(T, xm, dd, ld, td, cfg_of(Cn, Cn), out, None, glm, gd))
    torch.cuda.synchronize(T.dev)
    assert out.cpu().numpy().tobytes() == ref["raw"]
    same_bits(glm.cpu().numpy(), ref["grad_logits"])
    same_bits(gd.cpu().numpy(), ref["grad_deltas"])


def test_all_padding_images_and_empty_batch(T):
    rng = np.random.default_rng(8)
    x, d, lab, t = case(rng, 6, 64, 21, 21)
    lab[[1, 4]] = -1
    lab[2, :] = np.where(lab[2] > 0, 0, lab[2])           # an image without fg rows
    check(T, x, d, lab, t)
    none = check(T, x, d, np.full_like(lab, -1), t)
    assert np.isnan(none["cls_loss"]) and none["reg_loss"] == 0 and none["n_rows"] == 0
    # B * S = 0: cls NaN, reg 0, zero counts, one launch, gradients untouched
    torch = T.torch
    for B, S in ((0, 64), (3, 0)):
        xd = torch.zeros((max(B, 1), max(S, 1), 21), device=T.dev)
        dd = torch.zeros((max(B, 1), max(S, 1), 21, 4), device=T.dev)
        ld = torch.zeros((max(B, 1), max(S, 1)), dtype=torch.int32, device=T.dev)
        td = torch.zeros((max(B, 1), max(S, 1), 4), device=T.dev)
        out = torch.full((8,), SENT, device=T.dev)
        gl, gd = torch.full_like(xd, SENT), torch.full_like(dd, SENT)
        n0 = T.L.launch_count()
        T.L.check(call(T, xd, dd, ld, td, cfg_of(21, 21), out, None, gl, gd, shape=(B, S)))
        assert T.L.launch_count() - n0 == 1
        o = out.cpu().numpy()
        assert np.isnan(o[0]) and o[1] == 0 and o.view(np.int32)[2:].tolist() == [0] * 6
        assert bool((gl == SENT).all()) and bool((gd == SENT).all())


def test_run_to_run_bits_and_handles(T):
    """the loss bits of a large batch on several calls and on two handles"""
    rng = np.random.default_rng(9)
    x, d, lab, t = case(rng, 64, 512, 81, 81)
    a = run(T, x, d, lab, t, grads=False)
    b = run(T, x, d, lab, t)
    assert a["raw"] == b["raw"]
    h = C.c_void_p()
    T.L.check(T.lib.tfrpn_create(C.byref(h), T.dev.index or 0))
    try:
        torch = T.torch
        out = torch.empty(8, device=T.dev)
        for _ in range(3):
            T.L.check(call(T, T.cu(x), T.cu(d), T.cu(lab), T.cu(t), cfg_of(81, 81), out, h=h))
            torch.cuda.synchronize(T.dev)
            assert out.cpu().numpy().tobytes() == a["raw"]
    finally:
        T.lib.tfrpn_destroy(h)


def test_graph_replay_equals_direct_calls(T):
    """a captured call with gradients and a device scale, replayed 5 times over changing inputs, equals 5 direct
    calls; a fresh handle under capture cannot size its workspace"""
    torch = T.torch
    rng = np.random.default_rng(10)
    B, S, Cn = 8, 256, 21
    data = [case(rng, B, S, Cn, Cn) for _ in range(5)]
    scales = [np.array([1.0 + i, 0.5 - i], F32) for i in range(5)]
    xd, dd, ld, td = (T.cu(a) for a in data[0])
    sd = T.cu(scales[0])
    out = torch.empty(8, device=T.dev)
    gl, gd = torch.empty_like(xd), torch.empty_like(dd)
    cfg = cfg_of(Cn, Cn, 0.5, 1)
    T.L.check(call(T, xd, dd, ld, td, cfg, out, sd, gl, gd))       # sizes the workspace before the capture
    torch.cuda.synchronize(T.dev)
    s = torch.cuda.Stream(T.dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        T.L.check(call(T, xd, dd, ld, td, cfg, out, sd, gl, gd, stream=s))
    replayed = []
    for x, sc in zip(data, scales):
        for dst, src in zip((xd, dd, ld, td), x):
            dst.copy_(T.cu(src))
        sd.copy_(T.cu(sc))
        out.fill_(SENT); gl.fill_(SENT); gd.fill_(SENT)
        graph.replay()
        torch.cuda.synchronize(T.dev)
        replayed.append((out.cpu().numpy().tobytes(), gl.cpu().numpy(), gd.cpu().numpy()))
    del graph
    for x, sc, (ob, g1, g2) in zip(data, scales, replayed):
        r = check(T, *x, delta=0.5, norm=1, scale=sc)
        assert r["raw"] == ob
        same_bits(g1, r["grad_logits"])
        same_bits(g2, r["grad_deltas"])
    h = C.c_void_p()
    T.L.check(T.lib.tfrpn_create(C.byref(h), T.dev.index or 0))
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            rc = call(T, xd, dd, ld, td, cfg, out, stream=s, h=h)     # refused before anything is enqueued
        assert rc == -4, rc                                           # TFRPN_ERR_WORKSPACE
        del g
        torch.cuda.synchronize(T.dev)
    finally:
        T.lib.tfrpn_destroy(h)


def test_non_default_stream(T):
    torch = T.torch
    rng = np.random.default_rng(11)
    x, d, lab, t = case(rng, 4, 128, 33, 1)
    ref = run(T, x, d, lab, t)
    s = torch.cuda.Stream(T.dev)
    s.wait_stream(torch.cuda.current_stream(T.dev))
    with torch.cuda.stream(s):
        r = run(T, x, d, lab, t, stream=s)
        py = T.tfrpn.roi_head_losses(T.cu(x), T.cu(d).view(4, 128, 4), T.cu(lab), T.cu(t), with_grads=True)
    s.synchronize()
    assert r["raw"] == ref["raw"]
    same_bits(r["grad_logits"], ref["grad_logits"])
    same_bits(py.grad_deltas.cpu().numpy().reshape(d.shape), ref["grad_deltas"])
    assert py.cls_loss.cpu().numpy().tobytes() == ref["raw"][:4] and int(py.n_fg) == ref["n_fg"]


@pytest.mark.parametrize("use", ["both", "cls", "reg"])
def test_autograd_function_matches_with_grads(T, use):
    """the Function's gradients are with_grads' gradients times the upstream gradients (a zero for an unused loss),
    computed on the device; (B,S,C*4) box deltas get a gradient of their own shape.  (The backward runs on autograd's
    device thread, so its two launches are not on this thread's tfrpn_launch_count.)"""
    torch = T.torch
    rng = np.random.default_rng(12)
    B, S, Cn = 8, 128, 21
    x, d, lab, t = case(rng, B, S, Cn, Cn)
    xd = T.cu(x).requires_grad_(True)
    dd = T.cu(d.reshape(B, S, Cn * 4)).requires_grad_(True)
    r = T.tfrpn.roi_head_losses(xd, dd, T.cu(lab), T.cu(t), huber_delta=0.5, normalize="rows")
    assert r.grad_logits is None and r.cls_loss.requires_grad and not r.n_rows.requires_grad
    ref = T.tfrpn.roi_head_losses(T.cu(x), T.cu(d), T.cu(lab), T.cu(t), huber_delta=0.5, normalize="rows",
                                  with_grads=True)
    assert r.cls_loss.item() == ref.cls_loss.item() and r.reg_loss.item() == ref.reg_loss.item()
    gc, gr = {"both": (1.5, -0.25), "cls": (1.5, 0.0), "reg": (0.0, -0.25)}[use]
    loss = {"both": gc * r.cls_loss + gr * r.reg_loss, "cls": gc * r.cls_loss, "reg": gr * r.reg_loss}[use]
    loss.backward()
    wl = (ref.grad_logits * torch.tensor(gc, dtype=torch.float32, device=T.dev))
    wd = (ref.grad_deltas * torch.tensor(gr, dtype=torch.float32, device=T.dev))
    assert dd.grad.shape == (B, S, Cn * 4)
    # the kernel writes +0 outside the selected slices, where 0 * gr is -0 for gr < 0: compare with zeros unsigned
    same_bits(dd.grad.cpu().numpy().reshape(d.shape) + F32(0), wd.cpu().numpy() + F32(0))
    g, w = xd.grad.cpu().numpy(), wl.cpu().numpy()
    assert np.all(np.abs(g - w) <= 1e-6 / max(int(ref.n_rows), 1) * abs(gc) + 0.0)
    # NumPy in, NumPy out
    npr = T.tfrpn.roi_head_losses(x, d, lab, t, huber_delta=0.5, normalize="rows")
    assert isinstance(npr.cls_loss, np.ndarray) and npr.cls_loss.tobytes() == ref.cls_loss.cpu().numpy().tobytes()


def test_launch_counts(T):
    rng = np.random.default_rng(13)
    x, d, lab, t = case(rng, 2, 64, 21, 21)
    for grads, want in ((False, 1), (True, 2)):
        n0 = T.L.launch_count()
        run(T, x, d, lab, t, grads=grads)
        assert T.L.launch_count() - n0 == want
    n0 = T.L.launch_count()
    T.tfrpn.roi_head_losses(T.cu(x), T.cu(d), T.cu(lab), T.cu(t))
    assert T.L.launch_count() - n0 == 1


def test_argument_errors_and_limits(T):
    torch = T.torch
    buf = torch.zeros(1 << 22, dtype=torch.float32, device=T.dev)      # 16 MB: inputs at 0, out at 2 MB, grads at 4 / 8 MB
    p = buf.data_ptr()
    o = p + (1 << 21)
    st = torch.cuda.current_stream(T.dev).cuda_stream
    lib = T.lib

    def go(h=T.h, x=p, d=p, lab=p, t=p, B=2, S=4, Cn=4, q=4, delta=1.0, norm=0, out=o, sc=None, gl=None, gd=None,
           cfg=True):
        c = cfg_of(Cn, q, delta, norm)
        return lib.tfrpn_roi_head_losses(h, x, d, lab, t, B, S, C.byref(c) if cfg else None, out, sc, gl, gd, st)

    assert go() == 0
    assert go(gl=p + (1 << 22), gd=p + (1 << 23), sc=p) == 0
    for kw in (dict(h=None), dict(x=None), dict(d=None), dict(lab=None), dict(t=None), dict(out=None),
               dict(cfg=False), dict(B=-1), dict(S=-1), dict(Cn=1, q=1), dict(q=3), dict(q=0), dict(delta=0.0),
               dict(delta=-1.0), dict(delta=float("nan")), dict(norm=2), dict(norm=-1)):
        assert go(**kw) == -1, kw
    for kw in (dict(Cn=1025, q=1), dict(S=8193), dict(B=65536)):
        assert go(**kw) == -5, kw
    for kw in (dict(d=p + 4), dict(t=p + 8), dict(gd=p + (1 << 23) + 4), dict(x=p + 2), dict(gl=p + 2)):
        assert go(**kw) == -2, kw
    assert go(Cn=1024, q=1, S=1) == 0 and go(S=8192, B=1, Cn=2, q=2) == 0
    assert go(x=p + 4, gl=p + (1 << 22) + 4) == 0                   # logits need only 4-byte alignment
    torch.cuda.synchronize(T.dev)
    x = torch.zeros((1, 2, 4), device=T.dev)
    with pytest.raises(ValueError):
        T.tfrpn.roi_head_losses(x, torch.zeros((1, 2, 3), device=T.dev), torch.zeros((1, 2), dtype=torch.int32,
                                                                                    device=T.dev),
                                torch.zeros((1, 2, 4), device=T.dev))
    with pytest.raises(ValueError):                                  # q = 2 is neither 1 nor C
        T.tfrpn.roi_head_losses(x, torch.zeros((1, 2, 8), device=T.dev),
                                torch.zeros((1, 2), dtype=torch.int32, device=T.dev), torch.zeros((1, 2, 4), device=T.dev))
    with pytest.raises(ValueError):
        T.tfrpn.roi_head_losses(x, torch.zeros((1, 2, 16), device=T.dev),
                                torch.zeros((1, 2), dtype=torch.int32, device=T.dev), torch.zeros((1, 2, 4), device=T.dev),
                                normalize="all")
    with pytest.raises(NotImplementedError):
        T.tfrpn.roi_head_losses(torch.zeros((1, 2, 1025), device=T.dev), torch.zeros((1, 2, 4), device=T.dev),
                                torch.zeros((1, 2), dtype=torch.int32, device=T.dev), torch.zeros((1, 2, 4), device=T.dev))


def test_real_chain_backward_reaches_features(T):
    """generate_proposals -> roi_targets -> crop_and_resize -> a linear box head -> roi_head_losses -> backward: the
    losses are the oracle's on the head's outputs, the gradient reaches the features, and two runs give the same
    bits"""
    torch = T.torch
    from oracle import rpn_oracle as O
    from tfrpn import synthetic
    from tfrpn.utils import data_utils
    rng = np.random.default_rng(14)
    hp = O.get_hyper_params("vgg16")
    B, G, Cn, Fc = 4, 20, 21, 32
    fh, fw = O._pair(hp["feature_map_shape"])
    reg, cls = synthetic.head_outputs(rng, B, fh, fw, hp["anchor_count"])
    rois, _, valid, _ = T.tfrpn.generate_proposals(T.cu(reg), T.cu(cls), T.cu(O.generate_anchors(hp)), hp)
    gtb, gtl = synthetic.gt_batch(rng, B, G)
    n = (gtl >= 0).sum(axis=1)
    gb, gl = data_utils.pad_gt_batch([gtb[b, :n[b]] for b in range(B)], [gtl[b, :n[b]] - 1 for b in range(B)],
                                     max_boxes=G, label_add=1)
    t = T.tfrpn.roi_targets(rois, gb, gl, valid, num_classes=Cn, total_pos=32, total_neg=96, offset=5)
    feats0 = T.cu(rng.normal(size=(B, fh, fw, Fc)).astype(F32))
    torch.manual_seed(0)
    head = torch.nn.Linear(7 * 7 * Fc, Cn * 5).to(T.dev)

    def step():
        feats = feats0.clone().requires_grad_(True)
        head.zero_grad(set_to_none=True)
        pooled = T.tfrpn.crop_and_resize(feats, t.rois, None, (7, 7))
        y = head(pooled.reshape(B, 128, -1))
        logits, deltas = y[..., :Cn], y[..., Cn:]
        r = T.tfrpn.roi_head_losses(logits, deltas, t.labels, t.deltas)
        (r.cls_loss + r.reg_loss).backward()
        torch.cuda.synchronize(T.dev)
        return r, logits.detach(), deltas.detach(), feats.grad, head.weight.grad.clone()

    r1, lg, dl, f1, w1 = step()
    r2, _, _, f2, w2 = step()
    w = L.roi_head_losses(lg.cpu().numpy(), dl.cpu().numpy().reshape(B, 128, Cn, 4), t.labels.cpu().numpy(),
                          t.deltas.cpu().numpy())
    assert loss_close(r1.cls_loss.item(), w["cls_loss"]) and loss_close(r1.reg_loss.item(), w["reg_loss"])
    assert int(r1.n_fg) == w["n_fg"] > 0 and int(r1.n_rows) == w["n_rows"]
    assert bool(torch.isfinite(f1).all()) and float(f1.abs().sum()) > 0
    assert torch.equal(f1.view(torch.int32), f2.view(torch.int32))
    assert torch.equal(w1.view(torch.int32), w2.view(torch.int32))
    assert r1.cls_loss.item() == r2.cls_loss.item() and r1.reg_loss.item() == r2.reg_loss.item()

"""Segment AdaIN gradients (rpst_seg_adain_bwd and `differentiable=True`): content, style and prev gradients
against torch autograd of the reference's op sequence in fp64, the exact pass-through / zero cases,
bit-identical repeats, plane maps, the other entry points, a masked training step, `install(segment_grad=True)`
and CUDA-graph capture.  The last test checks the raw entry point's argument validation without a GPU."""
import copy
import sys
import types

import numpy as np
import pytest
import torch
from torch import nn

from oracle import restate as R
from oracle.gen_golden import decode_inputs, decode_stub

GRAD_TOL = 1e-4


@pytest.fixture(scope="module")
def rpst():
    import rpst as m
    return m


def seg_adain64(content, style, c_labels, s_labels, eps=1e-5):
    """`oracle.restate.seg_adain_batch` op for op (per-sample loop; mean, unbiased var, masked copy-back), kept
    differentiable: the truth the gradients are compared with when run in fp64."""
    outs = []
    ch = content.shape[1]
    for i in range(content.shape[0]):
        cf, sf = content[i].reshape(ch, -1), style[i].reshape(ch, -1)
        cl, sl = c_labels[i].reshape(-1).long().cpu(), s_labels[i].reshape(-1).long().cpu()
        out = cf.clone()
        for lab, ok in R.segment_label_validity(cl, sl).items():
            if not ok:
                continue
            ci = torch.nonzero(cl == lab).reshape(-1).to(cf.device)
            si = torch.nonzero(sl == lab).reshape(-1).to(cf.device)
            mc, ms = cf[:, ci], sf[:, si]
            mu_c, sd_c = mc.mean(1, keepdim=True), torch.sqrt(mc.var(1, keepdim=True) + eps)
            mu_s, sd_s = ms.mean(1, keepdim=True), torch.sqrt(ms.var(1, keepdim=True) + eps)
            out = out.index_copy(1, ci, (mc - mu_c) / sd_c * sd_s + mu_s)
        outs.append(out.reshape(content.shape[1:]))
    return torch.stack(outs)


def _inputs(shape_c, shape_s, block, classes=6):
    n = shape_c[0]
    c = torch.relu(torch.randn(shape_c, generator=torch.Generator().manual_seed(1)) + 0.5)
    s = torch.relu(torch.randn(shape_s, generator=torch.Generator().manual_seed(2)) * 2 + 1)
    cl = R.synth_labels(n, shape_c[2], shape_c[3], classes=classes, block=block, seed=4000)
    sl = R.synth_labels(n, shape_s[2], shape_s[3], classes=classes, block=block, seed=5000)
    cl[:, :2, :3] = 255                        # ignore label, tiny region -> unusable
    cl[:, 5:, :][cl[:, 5:, :] == 4] = 17       # a label absent from the style map
    sl[:, -2:, -3:] = 201                      # a label absent from the content map: zero style gradient
    return c, s, cl, sl


def _grads64(c, s, cl, sl, prev, g):
    """fp64 (out, d content, d style, d prev) of `prev + seg_adain(c, s)` for upstream gradient g."""
    c64, s64, p64 = (t.double().cpu().requires_grad_() for t in (c, s, prev))
    out = seg_adain64(c64, s64, cl.cpu(), sl.cpu()) + p64
    return (out.detach(),) + torch.autograd.grad(out, (c64, s64, p64), g.double().cpu())


def _raw_bwd(rpst, g, c, s, cl, sl, want_c=True, want_s=True):
    n, ch, hc, wc = c.shape
    hs, ws_ = s.shape[2:]
    dc = torch.empty_like(c) if want_c else None
    ds = torch.empty_like(s) if want_s else None
    L = rpst._lib.lib()
    ws = torch.empty(L.rpst_seg_adain_bwd_workspace_bytes(n, ch, hc * wc, hs * ws_), dtype=torch.uint8, device=c.device)
    rpst._lib.check(L.rpst_seg_adain_bwd(g.data_ptr(), c.data_ptr(), s.data_ptr(), cl.data_ptr(), sl.data_ptr(),
                                         None if dc is None else dc.data_ptr(), None if ds is None else ds.data_ptr(),
                                         n, ch, hc * wc, hs * ws_, 1e-5, ws.data_ptr(), ws.numel(),
                                         torch.cuda.current_stream().cuda_stream))
    return dc, ds


SHAPES = [((1, 4, 64, 64), (1, 4, 64, 64), 16), ((2, 3, 96, 128), (2, 3, 80, 60), 8),
          ((1, 2, 37, 41), (1, 2, 50, 33), 5), ((2, 2, 256, 512), (2, 2, 256, 512), 32),
          ((1, 2, 128, 128), (1, 2, 128, 128), 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("wrt", ["all", "content", "style", "prev"])
@pytest.mark.parametrize("shape_c,shape_s,block", SHAPES)
def test_gradients_vs_fp64(rpst, shape_c, shape_s, block, wrt):
    c, s, cl, sl = _inputs(shape_c, shape_s, block)
    prev = torch.randn(shape_c, generator=torch.Generator().manual_seed(3))
    g = torch.randn(shape_c, generator=torch.Generator().manual_seed(4))
    want_out, want_dc, want_ds, want_dp = _grads64(c, s, cl, sl, prev, g)
    cc, sc, pc = (t.cuda().requires_grad_(wrt in ("all", name)) for t, name in ((c, "content"), (s, "style"), (prev, "prev")))
    out = rpst.seg_adain_batch(cc, sc, cl.cuda(), sl.cuda(), pc, differentiable=True)
    assert R.rel_l2(out.detach(), want_out) < 5e-6
    out.backward(g.cuda())
    for t, want, name in ((cc, want_dc, "content"), (sc, want_ds, "style"), (pc, want_dp, "prev")):
        if wrt in ("all", name):
            assert R.rel_l2(t.grad, want) < GRAD_TOL, name
        else:
            assert t.grad is None, name


@pytest.mark.gpu
@pytest.mark.parametrize("shape_c,shape_s,block", [SHAPES[1], SHAPES[2], SHAPES[4]])
def test_pass_through_and_zero_gradients_are_exact(rpst, shape_c, shape_s, block):
    c, s, cl, sl = (t.cuda() for t in _inputs(shape_c, shape_s, block))
    prev = torch.randn(shape_c, device="cuda").requires_grad_()
    cc, sc = c.clone().requires_grad_(), s.clone().requires_grad_()
    g = torch.randn(shape_c, device="cuda")
    rpst.seg_adain_batch(cc, sc, cl, sl, prev, differentiable=True).backward(g)
    assert torch.equal(prev.grad, g)
    n, ch = shape_c[:2]
    for i in range(n):
        valid = R.segment_label_validity(cl[i].cpu(), sl[i].cpu())
        usable = [lab for lab, ok in valid.items() if ok]
        assert usable and any(not ok for ok in valid.values())
        cmask = ~torch.isin(cl[i].reshape(-1), torch.tensor(usable, device="cuda", dtype=torch.uint8))
        smask = ~torch.isin(sl[i].reshape(-1), torch.tensor(usable, device="cuda", dtype=torch.uint8))
        assert cmask.any() and smask.any()
        assert torch.equal(cc.grad[i].reshape(ch, -1)[:, cmask], g[i].reshape(ch, -1)[:, cmask])
        assert (sc.grad[i].reshape(ch, -1)[:, smask] == 0).all()
        assert (sc.grad[i].reshape(ch, -1)[:, ~smask] != 0).any()


@pytest.mark.gpu
def test_large_offsets_per_label(rpst):
    c = torch.zeros(1, 1, 64, 64)
    cl = torch.zeros(1, 64, 64, dtype=torch.uint8)
    cl[:, :, 32:] = 1
    gen = torch.Generator().manual_seed(0)
    c[..., :32] = 1000.0 + 0.5 * torch.randn(64, 32, generator=gen)
    c[..., 32:] = 0.01 * torch.randn(64, 32, generator=gen)
    s = torch.randn(1, 1, 64, 64, generator=gen)
    g = torch.randn(1, 1, 64, 64, generator=gen)
    _, want_dc, want_ds, _ = _grads64(c, s, cl, cl, torch.zeros_like(c), g)
    dc, ds = _raw_bwd(rpst, g.cuda(), c.cuda(), s.cuda(), cl.cuda(), cl.cuda())
    assert R.rel_l2(dc, want_dc) < 1e-3
    assert R.rel_l2(ds, want_ds) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("classes", [19, 40, 80, 200])
def test_many_labels(rpst, classes):
    """More than 64 usable labels: the backward's per-warp tables cover all 256 label values."""
    shape = (1, 3, 256, 256)
    c = torch.relu(torch.randn(shape, generator=torch.Generator().manual_seed(11)) + 0.5)
    s = torch.relu(torch.randn(shape, generator=torch.Generator().manual_seed(12)) * 2 + 1)
    cl = R.synth_labels(1, 256, 256, classes=classes, block=4, seed=4100 + classes)
    sl = R.synth_labels(1, 256, 256, classes=classes, block=4, seed=5100 + classes)
    g = torch.randn(shape, generator=torch.Generator().manual_seed(13))
    usable = sum(R.segment_label_validity(cl[0], sl[0]).values())
    assert usable >= min(classes, 150) - 5, usable
    _, want_dc, want_ds, _ = _grads64(c, s, cl, sl, torch.zeros_like(c), g)
    dc, ds = _raw_bwd(rpst, g.cuda(), c.cuda(), s.cuda(), cl.cuda(), sl.cuda())
    assert R.rel_l2(dc, want_dc) < GRAD_TOL
    assert R.rel_l2(ds, want_ds) < GRAD_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("shape,block", [((2, 3, 128, 128), 1), ((2, 3, 96, 128), 4), ((1, 4, 256, 512), 32),
                                         ((1, 2, 37, 41), 5)])
def test_repeat_is_bit_identical(rpst, shape, block):
    c, s, cl, sl = (t.cuda() for t in _inputs(shape, shape, block))
    g = torch.randn(shape, device="cuda")
    dc, ds = _raw_bwd(rpst, g, c, s, cl, sl)
    for _ in range(2):
        dc2, ds2 = _raw_bwd(rpst, g, c, s, cl, sl)
        assert torch.equal(dc, dc2) and torch.equal(ds, ds2)
    # each half alone is the same computation
    assert torch.equal(_raw_bwd(rpst, g, c, s, cl, sl, want_s=False)[0], dc)
    assert torch.equal(_raw_bwd(rpst, g, c, s, cl, sl, want_c=False)[1], ds)


@pytest.mark.gpu
def test_config5_planes(rpst):
    """1024x2048 planes (BASELINE configs[4]), 19 classes in 32x32 tiles: fp64 agreement on channel 0 and a
    bit-identical repeat."""
    n, ch, h, w = 1, 8, 1024, 2048
    c, s = R.synth_features((n, ch, h, w), cfg=5, device="cuda")
    cl = R.synth_labels(n, h, w, classes=19, block=32, seed=4000, device="cuda")
    sl = R.synth_labels(n, h, w, classes=19, block=32, seed=5000, device="cuda")
    cl[:, :3, :3] = 255
    g = torch.randn((n, ch, h, w), device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
    dc, ds = _raw_bwd(rpst, g, c, s, cl, sl)
    _, want_dc, want_ds, _ = _grads64(c[:, :1], s[:, :1], cl, sl, torch.zeros_like(c[:, :1]), g[:, :1])
    assert R.rel_l2(dc[:, :1], want_dc) < GRAD_TOL
    assert R.rel_l2(ds[:, :1], want_ds) < GRAD_TOL
    dc2, ds2 = _raw_bwd(rpst, g, c, s, cl, sl)
    assert torch.equal(dc, dc2) and torch.equal(ds, ds2)


@pytest.mark.gpu
def test_plane_maps_equal_gather_then_differentiate(rpst):
    n, ch, h, w = 2, 4, 64, 96
    c, s, cl, sl = (t.cuda() for t in _inputs((n, ch, h, w), (n, ch, 48, 80), 8))
    cm = rpst.shuffle_map(n, ch, 2, "cuda")
    sm = rpst.sort_map(torch.rand(n, ch, 1, 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5)))
    g = torch.randn((n, ch, h, w), device="cuda")
    prev = torch.randn((n, ch, h, w), device="cuda")
    c1, s1, p1 = c.clone().requires_grad_(), s.clone().requires_grad_(), prev.clone().requires_grad_()
    out1 = rpst.seg_adain_batch(c1, s1, cl, sl, p1, content_map=cm, style_map=sm, differentiable=True)
    out1.backward(g)
    c2, s2, p2 = c.clone().requires_grad_(), s.clone().requires_grad_(), prev.clone().requires_grad_()
    cg = c2.flatten(0, 1)[cm.long()].view_as(c2)
    sg = s2.flatten(0, 1)[sm.long()].view_as(s2)
    out2 = rpst.seg_adain_batch(cg, sg, cl, sl, p2, differentiable=True)
    out2.backward(g)
    # the forward reproduces to rounding on 8-pixel blocks (test_seg_mapped_gpu.py); the backward is exact
    assert R.rel_l2(out1, out2) < 1e-6
    assert torch.equal(c1.grad, c2.grad) and torch.equal(s1.grad, s2.grad) and torch.equal(p1.grad, p2.grad)
    with torch.no_grad():   # the differentiable forward is the mapped kernel's result
        assert R.rel_l2(out1, rpst.seg_adain_batch(c, s, cl, sl, prev, content_map=cm, style_map=sm)) < 1e-6


def _labels_as(kind, lab, tmp_path, tag):
    if kind == "tensor":
        return lab.cuda()
    if kind == "array":
        return [m.numpy() for m in lab]
    from PIL import Image
    paths = []
    for i, m in enumerate(lab):
        p = tmp_path / f"{tag}{i}.png"
        Image.fromarray(m.numpy()).save(p)
        paths.append(str(p))
    return paths


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["path", "array", "tensor"])
def test_do_mask_stylized_and_concat_entry_points(rpst, kind, tmp_path):
    n, ch, h, w = 2, 3, 40, 48
    c, s, cl, sl = _inputs((n, ch, h, w), (n, ch, 36, 44), 4, classes=4)
    g = torch.randn((n, ch, h, w), generator=torch.Generator().manual_seed(8))
    prev = torch.randn((n, 2, h, w), generator=torch.Generator().manual_seed(9))
    c64, s64 = c.double().requires_grad_(), s.double().requires_grad_()
    out64 = seg_adain64(c64, s64, cl, sl)
    want_dc, want_ds = torch.autograd.grad(out64, (c64, s64), g.double())
    cm, sm = _labels_as(kind, cl, tmp_path, "c"), _labels_as(kind, sl, tmp_path, "s")

    cc, sc = c.cuda().requires_grad_(), s.cuda().requires_grad_()
    out = rpst.do_mask_stylized(cc, sc, cm, sm, differentiable=True)
    out.backward(g.cuda())
    assert R.rel_l2(out.detach(), out64.detach()) < 5e-6
    assert R.rel_l2(cc.grad, want_dc) < GRAD_TOL and R.rel_l2(sc.grad, want_ds) < GRAD_TOL

    cc, sc, pc = c.cuda().requires_grad_(), s.cuda().requires_grad_(), prev.cuda().requires_grad_()
    from rpst.segment import stack_label_maps
    tc = cm if kind == "tensor" else stack_label_maps(cm, w, h, "cuda")
    ts = sm if kind == "tensor" else stack_label_maps(sm, 44, 36, "cuda")
    out = rpst.seg_adain_concat(pc, cc, sc, tc, ts, differentiable=True)
    gp = torch.randn(out.shape, device="cuda")
    gp[:, 2:] = g.cuda()
    out.backward(gp)
    assert torch.equal(pc.grad, gp[:, :2])
    assert R.rel_l2(cc.grad, want_dc) < GRAD_TOL and R.rel_l2(sc.grad, want_ds) < GRAD_TOL


class TinyRP(nn.Module):
    """Two-level resolution-preserving encoder/decoder in the shape of MultiScaleAdaINRPNet (test_training_gpu.py)
    with segment AdaIN at both levels; the lower level adds the decoder state as `prev`."""

    def __init__(self):
        super().__init__()
        self.enc = nn.ModuleList([nn.Sequential(nn.Conv2d(3, 8, 3, padding=1), nn.ReLU()),
                                  nn.Sequential(nn.Conv2d(8, 16, 3, padding=1), nn.ReLU())])
        self.dec = nn.ModuleList([nn.Sequential(nn.Conv2d(16, 8, 3, padding=1), nn.ReLU()),
                                  nn.Sequential(nn.Conv2d(8, 3, 3, padding=1))])

    def feats(self, x):
        out = []
        for m in self.enc:
            x = m(x)
            out.append(x)
        return out

    def forward(self, content, style, seg, stats):
        cf, sf = self.feats(content), self.feats(style)
        y = self.dec[0](seg(cf[1], sf[1], None))
        y = self.dec[1](seg(cf[0], sf[0], y))
        yf = self.feats(y)
        loss = ((yf[1] - cf[1].detach()) ** 2).mean()
        for a, b in zip(yf, sf):
            ma, sa = stats(a)
            mb, sb = stats(b.detach())
            loss = loss + ((ma - mb) ** 2).mean() + ((sa - sb) ** 2).mean()
        return loss


def _stats64(x):
    n, c = x.shape[:2]
    f = x.reshape(n, c, -1)
    return f.mean(2).view(n, c, 1, 1), (f.var(2) + 1e-5).sqrt().view(n, c, 1, 1)


@pytest.mark.gpu
def test_masked_training_step_matches_fp64(rpst):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    hw = 48
    net = TinyRP().cuda()
    ref = TinyRP().double().cuda()
    ref.load_state_dict({k: v.double() for k, v in net.state_dict().items()})
    g = torch.Generator(device="cuda").manual_seed(1)
    content = torch.rand(2, 3, hw, hw, device="cuda", generator=g)
    style = torch.rand(2, 3, hw, hw, device="cuda", generator=g)
    cl = R.synth_labels(2, hw, hw, classes=4, block=8, seed=4300).cuda()
    sl = R.synth_labels(2, hw, hw, classes=4, block=8, seed=5300).cuda()

    loss = net(content, style, lambda c, s, p: rpst.seg_adain_batch(c, s, cl, sl, p, differentiable=True),
               rpst.calc_mean_std)
    loss.backward()
    loss64 = ref(content.double(), style.double(),
                 lambda c, s, p: seg_adain64(c, s, cl, sl) + (0 if p is None else p), _stats64)
    loss64.backward()
    assert abs(float(loss) - float(loss64)) / abs(float(loss64)) < 2e-4
    for (name, p), q in zip(net.named_parameters(), ref.parameters()):
        err = float((p.grad.double() - q.grad).norm() / q.grad.norm().clamp_min(1e-30))
        assert err < 2e-3, (name, err)


@pytest.mark.gpu
def test_install_segment_grad_on_a_stub_tree(rpst):
    """`install(segment_grad=True)` makes the patched masked decode train; plain `install()` keeps refusing, and
    `uninstall()` restores the stub's own decode."""
    from rpst import decode as D

    class MultiScaleAdaINRPNet(nn.Module):
        def __init__(self):
            super().__init__()
            stub = decode_stub("multiscale")
            self.rp_decoder = stub.rp_decoder
            self.rp_shared_encoder = stub.rp_shared_encoder
            self._sort, self._shuffle, self._shuffle_layers = False, False, 1
            self.config = {"use_mask": True}

        def decode(self, *args, **kwargs):
            raise AssertionError("the stub's own decode is never called while rpst is installed")

    orig = MultiScaleAdaINRPNet.decode
    pkg = types.ModuleType("segstub")
    pkg.MultiScaleAdaINRPNet = MultiScaleAdaINRPNet
    sys.modules["segstub"] = pkg
    try:
        m = MultiScaleAdaINRPNet().cuda()
        cs, ss, _ = decode_inputs("multiscale")
        n, _, h, w = cs[0].shape
        cl = R.synth_labels(n, h, w, classes=3, block=4, seed=4401)
        sl = R.synth_labels(n, h, w, classes=3, block=4, seed=5401)
        counts = rpst.install("segstub", segment_grad=True)
        try:
            assert counts["MultiScaleAdaINRPNet.decode"] == 1
            feats = [t.cuda().requires_grad_() for t in cs + ss]
            out = m.decode(feats[:3], feats[3:], use_mask=True, c_mask_path=cl.cuda(), s_mask_path=sl.cuda())
            gout = torch.randn_like(out)
            grads = torch.autograd.grad(out, feats + list(m.parameters()), gout)
        finally:
            rpst.uninstall()
        m64 = copy.deepcopy(m).double()
        f64 = [t.double().cuda().requires_grad_() for t in cs + ss]
        st = m64.rp_decoder[0](seg_adain64(f64[2], f64[5], cl, sl))
        for i, l in enumerate((1, 0)):
            st = m64.rp_decoder[i + 1](st + seg_adain64(f64[l], f64[3 + l], cl, sl))
        want = torch.autograd.grad(st, f64 + list(m64.parameters()), gout.double())
        assert R.rel_l2(out.detach(), st.detach()) < 1e-5
        for k, (a, b) in enumerate(zip(grads, want)):
            assert R.rel_l2(a, b) < 2e-3, k

        rpst.install("segstub")
        try:
            feats = [t.cuda().requires_grad_() for t in cs + ss]
            with pytest.raises(NotImplementedError):
                m.decode(feats[:3], feats[3:], use_mask=True, c_mask_path=cl.cuda(), s_mask_path=sl.cuda())
        finally:
            rpst.uninstall()
        assert MultiScaleAdaINRPNet.decode is orig
        assert D.SEGMENT_GRAD_DECODES["MultiScaleAdaINRPNet"].__wrapped__ is D.decode_multiscale
    finally:
        del sys.modules["segstub"]


@pytest.mark.gpu
def test_backward_replays_in_a_cuda_graph(rpst):
    n, ch, h, w = 2, 4, 64, 128
    c, s, cl, sl = (t.cuda() for t in _inputs((n, ch, h, w), (n, ch, 48, 96), 4))
    g = torch.randn((n, ch, h, w), device="cuda")
    eager_dc, eager_ds = _raw_bwd(rpst, g, c, s, cl, sl)
    L = rpst._lib.lib()
    ws = torch.empty(L.rpst_seg_adain_bwd_workspace_bytes(n, ch, h * w, 48 * 96), dtype=torch.uint8, device="cuda")
    dc, ds = torch.empty_like(c), torch.empty_like(s)

    def call():
        rpst._lib.check(L.rpst_seg_adain_bwd(g.data_ptr(), c.data_ptr(), s.data_ptr(), cl.data_ptr(), sl.data_ptr(),
                                             dc.data_ptr(), ds.data_ptr(), n, ch, h * w, 48 * 96, 1e-5, ws.data_ptr(),
                                             ws.numel(), torch.cuda.current_stream().cuda_stream))

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        call()
    dc.zero_()
    ds.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(dc, eager_dc) and torch.equal(ds, eager_ds)


def test_raw_backward_validates_without_gpu(rpst):
    """Invalid arguments are rejected before any CUDA call (runs on a GPU-less box)."""
    L = rpst._lib.lib()
    hw = 64
    g, c, s, cl, sl, dc, ds = (1 << 20) * np.arange(1, 8)   # distinct, never dereferenced
    g, c, s, cl, sl, dc, ds = (int(x) for x in (g, c, s, cl, sl, dc, ds))
    need = L.rpst_seg_adain_bwd_workspace_bytes(2, 3, hw, hw)
    assert need >= 2 * 3 * 2 * 256 * 16

    def call(*, n=2, ch=3, hw_c=hw, hw_s=hw, ptrs=None, outs=(dc, ds), ws=1 << 30, ws_bytes=need):
        p = ptrs or (g, c, s, cl, sl)
        return L.rpst_seg_adain_bwd(*p, *outs, n, ch, hw_c, hw_s, 1e-5, ws, ws_bytes, None)

    assert call(ptrs=(g, None, s, cl, sl)) == -1 and b"null" in L.rpst_last_error()
    assert call(ptrs=(g, c, s, cl, None)) == -1 and b"null" in L.rpst_last_error()
    assert call(n=-1) == -1 and b"negative" in L.rpst_last_error()
    assert call(hw_s=-4) == -1
    assert call(n=1 << 16, ch=1 << 15) == -1
    assert call(hw_c=1 << 31) == -1
    assert call(outs=(g, ds)) == -1 and b"alias" in L.rpst_last_error()
    assert call(outs=(dc, c + 16)) == -1 and b"alias" in L.rpst_last_error()    # overlap, not just equality
    assert call(outs=(dc, dc)) == -1
    assert call(ws_bytes=need - 1) == -3 and b"workspace" in L.rpst_last_error()
    assert call(ws=0) == -3
    assert call(ws=(1 << 30) + 16) == -1 and b"aligned" in L.rpst_last_error()
    assert call(n=0, ptrs=(None,) * 5, outs=(None, None), ws=None, ws_bytes=0) == 0     # empty batch
    assert call(ch=0) == 0
    assert call(outs=(None, None)) == 0     # nothing requested: no work

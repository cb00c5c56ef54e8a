"""Segment AdaIN through plane maps and into a channel slice (rpst_seg_adain_fwd_mapped): the mapped call equals
segment AdaIN on the gathered tensors, the concat form writes only its slice, no gathered copy is allocated, and
the masked decodes that use it match the reference's loops restated in fp64."""
import ctypes

import pytest
import torch

from oracle import restate as R
from oracle.gen_golden import decode_inputs, decode_stub

TIGHT = 5e-6
DECODE_TOL = 1e-5
REPRO = 1e-6    # run-to-run agreement of the segment kernel on label runs shorter than a lane's 32 pixels


@pytest.fixture(scope="module")
def rpst():
    import rpst as m
    return m


def _gather(x, plane_map):
    return x if plane_map is None else x.flatten(0, 1)[plane_map.long().cpu()].view_as(x)


def _maps(n, c, seed):
    """(name, content_map, style_map) on the CPU: within-sample permutations, then a map that crosses samples."""
    g = torch.Generator().manual_seed(seed)
    from rpst import shuffle_map, sort_map
    sort_c = sort_map(torch.rand(n, c, 1, 1, generator=g))
    shuf_s = shuffle_map(n, c, 2) if c % 2 == 0 else sort_map(torch.rand(n, c, 1, 1, generator=g))
    cross_c = torch.randint(0, n * c, (n * c,), generator=g, dtype=torch.int32)
    cross_s = torch.randperm(n * c, generator=g).to(torch.int32)
    return [("sort/shuffle", sort_c, shuf_s), ("cross-sample", cross_c, cross_s), ("content only", sort_c, None)]


def _inputs(shape_c, shape_s, block, classes=6):
    n = shape_c[0]
    c = torch.relu(torch.randn(shape_c, generator=torch.Generator().manual_seed(1)) + 0.5)
    s = torch.relu(torch.randn(shape_s, generator=torch.Generator().manual_seed(2)) * 2 + 1)
    cl = R.synth_labels(n, shape_c[2], shape_c[3], classes=classes, block=block, seed=4000)
    sl = R.synth_labels(n, shape_s[2], shape_s[3], classes=classes, block=block, seed=5000)
    cl[:, :2, :3] = 255
    return c, s, cl, sl


def _cuda(m):
    return None if m is None else m.cuda()


SHAPES = [((1, 4, 64, 64), (1, 4, 64, 64), 16, 0), ((2, 3, 96, 128), (2, 3, 80, 60), 8, 0),
          ((1, 2, 37, 41), (1, 2, 50, 33), 5, 0), ((2, 2, 256, 512), (2, 2, 256, 512), 32, 0),
          ((1, 2, 128, 128), (1, 2, 128, 128), 1, 0), ((2, 3, 96, 128), (2, 3, 80, 60), 8, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape_c,shape_s,block,adain_path", SHAPES)
def test_mapped_equals_gathered(rpst, shape_c, shape_s, block, adain_path):
    """TMA kernel (16-byte aligned planes), register-staged kernel (adain_path = 1: vectorised; 37x41: scalar),
    content and style of different H*W.  Block-32 maps on a width that is a multiple of 32 keep every lane's label
    run whole, so there the TMA kernel is bit-identical to the gathered call."""
    n, ch = shape_c[:2]
    c, s, cl, sl = _inputs(shape_c, shape_s, block)
    prev = torch.randn(shape_c, generator=torch.Generator().manual_seed(3))
    exact = block == 32 and shape_c[3] % 32 == 0 and adain_path == 0
    old = rpst.get_tuning("adain_path")
    rpst.set_tuning("adain_path", adain_path)
    try:
        for name, cm, sm in _maps(n, ch, seed=sum(shape_c) + block):
            cg, sg = _gather(c, cm), _gather(s, sm)
            want = R.seg_adain_batch(cg, sg, cl, sl, dtype=torch.float64)
            for p in (None, prev):
                pc = None if p is None else p.cuda()
                got, info = rpst.seg_adain_batch(c.cuda(), s.cuda(), cl.cuda(), sl.cuda(), pc, return_info=True,
                                                 content_map=_cuda(cm), style_map=_cuda(sm))
                dense, dinfo = rpst.seg_adain_batch(cg.cuda(), sg.cuda(), cl.cuda(), sl.cuda(), pc, return_info=True)
                assert torch.equal(info, dinfo), name
                ref = want if p is None else want + p.double()
                assert R.rel_l2(got, ref) < TIGHT, (name, p is None)
                if exact:
                    assert torch.equal(got, dense), (name, p is None)
                else:
                    assert R.rel_l2(got, dense) < REPRO, (name, p is None)
    finally:
        rpst.set_tuning("adain_path", old)


@pytest.mark.gpu
@pytest.mark.parametrize("classes", [80, 200])
def test_mapped_fallback_beyond_64_labels(rpst, classes):
    """More than 64 usable labels: the slot kernel bows out and the register-staged kernel reads through the maps."""
    shape = (2, 3, 256, 256)
    c = torch.relu(torch.randn(shape, generator=torch.Generator().manual_seed(11)) + 0.5)
    s = torch.relu(torch.randn(shape, generator=torch.Generator().manual_seed(12)) * 2 + 1)
    cl = R.synth_labels(2, 256, 256, classes=classes, block=4, seed=4100 + classes)
    sl = R.synth_labels(2, 256, 256, classes=classes, block=4, seed=5100 + classes)
    for name, cm, sm in _maps(2, 3, seed=classes)[:2]:
        got, info = rpst.seg_adain_batch(c.cuda(), s.cuda(), cl.cuda(), sl.cuda(), return_info=True,
                                         content_map=cm.cuda(), style_map=sm.cuda())
        assert int(info[0, :, 2].sum()) > 64
        want = R.seg_adain_batch(_gather(c, cm), _gather(s, sm), cl, sl, dtype=torch.float64)
        assert R.rel_l2(got, want) < TIGHT, name


def _raw_into(rpst, wide, c0, content, style, cl, sl, cm, sm):
    """rpst_seg_adain_fwd_mapped straight into channels c0.. of `wide` [N, Cw, H, W]."""
    L = rpst._lib.lib()
    n, ch, hc, wc = content.shape
    hw_s = style.shape[2] * style.shape[3]
    ws = torch.empty(max(L.rpst_seg_adain_workspace_bytes(n, ch, hc * wc, hw_s), 256), dtype=torch.uint8,
                     device=content.device)
    rpst._lib.check(L.rpst_seg_adain_fwd_mapped(
        content.data_ptr(), style.data_ptr(), cl.data_ptr(), sl.data_ptr(), None, wide[:, c0:].data_ptr(), n, ch,
        hc * wc, hw_s, wide.shape[1] * hc * wc, 1e-5, None if cm is None else cm.data_ptr(),
        None if sm is None else sm.data_ptr(), None, ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream))


@pytest.mark.gpu
@pytest.mark.parametrize("shape,cp,block", [((2, 4, 64, 128), 3, 32), ((2, 3, 37, 41), 2, 5)])
def test_concat_writes_only_its_slice(rpst, shape, cp, block):
    """Concat-write: aligned block-32 planes (TMA kernel, bit-identical to the dense call) and an odd H*W (scalar
    kernel, whatever the stride)."""
    n, ch, h, w = shape
    c, s, cl, sl = _inputs(shape, shape, block)
    c, s, cl, sl = c.cuda(), s.cuda(), cl.cuda(), sl.cuda()
    prev = torch.randn((n, cp, h, w), device="cuda")
    exact = block == 32
    for name, cm, sm in _maps(n, ch, seed=7 + cp):
        cm, sm = _cuda(cm), _cuda(sm)
        dense = rpst.seg_adain_batch(c, s, cl, sl, content_map=cm, style_map=sm)
        out = rpst.seg_adain_concat(prev, c, s, cl, sl, content_map=cm, style_map=sm)
        assert out.shape == (n, cp + ch, h, w)
        assert torch.equal(out[:, :cp], prev)
        want = R.seg_adain_batch(_gather(c.cpu(), cm), _gather(s.cpu(), sm), cl.cpu(), sl.cpu(), dtype=torch.float64)
        assert R.rel_l2(out[:, cp:], want) < TIGHT, name
        # a NaN-filled tensor wider than the concat on both sides: only the slice is written
        wide = torch.full((n, cp + ch + 1, h, w), float("nan"), device="cuda")
        _raw_into(rpst, wide, cp, c, s, cl, sl, cm, sm)
        torch.cuda.synchronize()
        assert torch.isnan(wide[:, :cp]).all() and torch.isnan(wide[:, cp + ch:]).all(), name
        for got in (out[:, cp:], wide[:, cp:cp + ch]):
            if exact:
                assert torch.equal(got, dense), name
            else:
                assert R.rel_l2(got, dense) < REPRO, name


@pytest.mark.gpu
def test_mapped_call_allocates_no_gathered_copy(rpst):
    n, ch, h, w = 1, 64, 512, 1024
    c, s = R.synth_features((n, ch, h, w), cfg=5, device="cuda")
    cl = R.synth_labels(n, h, w, classes=19, block=32, seed=4000, device="cuda")
    sl = R.synth_labels(n, h, w, classes=19, block=32, seed=5000, device="cuda")
    cm = rpst.shuffle_map(n, ch, 4, "cuda")
    sm = rpst.sort_map(torch.rand(n, ch, 1, 1, device="cuda"))
    with torch.no_grad():
        rpst.seg_adain_batch(c, s, cl, sl, content_map=cm, style_map=sm)   # warm-up: module load, kernel attributes
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = rpst.seg_adain_batch(c, s, cl, sl, content_map=cm, style_map=sm)
        torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    ws = rpst._lib.lib().rpst_seg_adain_workspace_bytes(n, ch, h * w, h * w)
    slack = 1 << 20    # allocator rounding
    assert extra <= out.numel() * 4 + ws + slack, (extra, out.numel() * 4, ws)
    assert extra < out.numel() * 4 * 2     # one gathered copy would already double it


def _stub(golden, kind):
    g = golden("decode")
    m = decode_stub(kind)
    m.load_state_dict({k[len(kind) + 1:]: v for k, v in g.items() if k.startswith(kind + ".") and
                       k[len(kind) + 1:] in m.state_dict()})
    cs, ss, atts = decode_inputs(kind)
    return m.cuda(), [c.cuda() for c in cs], [s.cuda() for s in ss], atts


@pytest.mark.gpu
def test_masked_multiscale_test_with_shuffle_and_sort(golden):
    """MultiScaleAdaINRPNet.test with use_mask, the channel shuffle and sort_by_weights: the masked levels read the
    features through plane maps.  Restated in fp64 as the reference runs it: shuffle (levels <= _shuffle_layers),
    sort, then do_mask_stylized with the decoder state added (network/adain_rp.py:251-319)."""
    from rpst import decode as D
    m, cs, ss, atts = _stub(golden, "multiscale")
    n, _, h, w = cs[0].shape
    cl = R.synth_labels(n, h, w, classes=3, block=4, seed=4401)
    sl = R.synth_labels(n, h, w, classes=3, block=4, seed=5401)
    for enc, a in zip(m.rp_shared_encoder, atts):
        enc.attention_map = a.cuda()
    m._sort, m._shuffle = True, True
    m.config["use_mask"] = True
    feats = {"c": cs, "s": ss}
    m.encode_rp_intermediate = lambda x: feats[x]
    got = D.test_multiscale(m, "c", "s", c_mask_path=cl.cuda(), s_mask_path=sl.cuda())
    with torch.no_grad():
        m64 = m.double().cpu()

        def prep(x, idx):
            x = x.cpu().double()
            if idx <= m._shuffle_layers:
                x = R.channel_shuffle(x, 4)
            return R.sort_by_weights(x, atts[idx].double())

        csd = [prep(c, i) for i, c in enumerate(cs)]
        ssd = [prep(s, i) for i, s in enumerate(ss)]
        st = m64.rp_decoder[0](R.seg_adain_batch(csd[-1], ssd[-1], cl, sl, dtype=torch.float64))
        for i, l in enumerate((1, 0)):
            st = m64.rp_decoder[i + 1](st + R.seg_adain_batch(csd[l], ssd[l], cl, sl, dtype=torch.float64))
    assert R.rel_l2(got, st) < DECODE_TOL


@pytest.mark.gpu
def test_masked_ld_concat_decode(golden):
    from rpst import decode as D
    m, cs, ss, _ = _stub(golden, "ldcat")
    n, _, h, w = cs[0].shape
    cl = R.synth_labels(n, h, w, classes=3, block=4, seed=4402)
    sl = R.synth_labels(n, h, w, classes=3, block=4, seed=5402)
    with torch.no_grad():
        got = D.decode_ld_concat(m, cs, ss, use_mask=True, c_mask_path=cl.cuda(), s_mask_path=[x.numpy() for x in sl])
        m64 = m.double().cpu()
        csd, ssd = [c.cpu().double() for c in cs], [s.cpu().double() for s in ss]
        st = m64.rp_dec0(R.seg_adain_batch(csd[-1], ssd[-1], cl, sl, dtype=torch.float64))
        for i, l in enumerate((1, 0)):
            st = getattr(m64, f"rp_dec{i + 1}")(torch.cat([st, R.seg_adain_batch(csd[l], ssd[l], cl, sl,
                                                                                   dtype=torch.float64)], dim=1))
    assert R.rel_l2(got, st) < DECODE_TOL


@pytest.mark.gpu
def test_bad_maps_stride_and_gradients_are_refused(rpst):
    n, ch, h, w = 2, 4, 32, 32
    c, s, cl, sl = (t.cuda() for t in _inputs((n, ch, h, w), (n, ch, h, w), 8))
    good = rpst.shuffle_map(n, ch, 2, "cuda")
    for bad in (good.long(), good[:-1], good.cpu()):
        with pytest.raises(TypeError):
            rpst.seg_adain_batch(c, s, cl, sl, content_map=bad)
        with pytest.raises(TypeError):
            rpst.seg_adain_concat(c, c, s, cl, sl, style_map=bad)
    out = torch.empty_like(c)
    L = rpst._lib.lib()
    ws = torch.empty(L.rpst_seg_adain_workspace_bytes(n, ch, h * w, h * w), dtype=torch.uint8, device="cuda")
    with pytest.raises(rpst.RpstError, match="out_batch_stride"):
        rpst._lib.check(L.rpst_seg_adain_fwd_mapped(c.data_ptr(), s.data_ptr(), cl.data_ptr(), sl.data_ptr(), None,
                                                    out.data_ptr(), n, ch, h * w, h * w, ch * h * w - 1, 1e-5,
                                                    good.data_ptr(), None, None, ws.data_ptr(), ws.numel(),
                                                    torch.cuda.current_stream().cuda_stream))
    cg = c.clone().requires_grad_()
    with pytest.raises(NotImplementedError):
        rpst.seg_adain_batch(cg, s, cl, sl, content_map=good)
    with pytest.raises(NotImplementedError):
        rpst.seg_adain_concat(c, cg, s, cl, sl, content_map=good)
    with pytest.raises(NotImplementedError):
        rpst.do_mask_stylized(cg, s, cl, sl, content_map=good)


@pytest.mark.gpu
def test_mapped_concat_replays_in_a_cuda_graph(rpst):
    n, ch, cp, h, w = 2, 4, 3, 64, 128
    c, s, cl, sl = (t.cuda() for t in _inputs((n, ch, h, w), (n, ch, h, w), 32))
    prev = torch.randn((n, cp, h, w), device="cuda")
    cm = rpst.shuffle_map(n, ch, 2, "cuda")
    sm = rpst.sort_map(torch.rand(n, ch, 1, 1, device="cuda"))
    eager = rpst.seg_adain_concat(prev, c, s, cl, sl, content_map=cm, style_map=sm)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            rpst.seg_adain_concat(prev, c, s, cl, sl, content_map=cm, style_map=sm)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = rpst.seg_adain_concat(prev, c, s, cl, sl, content_map=cm, style_map=sm)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


def test_raw_entry_point_validates_without_gpu(rpst):
    """Invalid arguments are rejected before any CUDA call (runs on a GPU-less box)."""
    L = rpst._lib.lib()
    fake = 256   # never dereferenced: every check below fails on the host first
    args = lambda n, c, hw, stride, ptr: (ptr, ptr, ptr, ptr, None, ptr, n, c, hw, hw, stride, 1e-5, None, None, None,
                                          ptr, 1 << 20, None)
    assert L.rpst_seg_adain_fwd_mapped(*args(1, 2, 64, 128, None)) == -1
    assert b"null" in L.rpst_last_error()
    assert L.rpst_seg_adain_fwd_mapped(*args(-1, 2, 64, 128, fake)) == -1
    assert L.rpst_seg_adain_fwd_mapped(*args(1, 2, -64, 128, fake)) == -1
    assert L.rpst_seg_adain_fwd_mapped(*args(1, 2, 64, 127, fake)) == -1
    assert b"out_batch_stride" in L.rpst_last_error()
    assert L.rpst_seg_adain_fwd_mapped(*args(1 << 16, 1 << 15, 64, 1 << 21, fake)) == -1
    assert L.rpst_seg_adain_fwd_mapped(*args(0, 2, 64, 0, None)) == 0     # empty batch

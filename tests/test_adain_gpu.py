"""GPU parity tests for the AdaIN family through the C ABI (rpst -> librpst.so) against the oracle
and the reference-generated golden vectors.  Tolerance: rel-L2 <= 1e-3 is the contract
(BASELINE.json north_star, fp32); these kernels are expected to sit at ~1e-6."""
import pytest
import torch

from oracle import restate as R

pytestmark = pytest.mark.gpu
TOL = 1e-3      # contract
TIGHT = 2e-6    # what an fp32 kernel with pairwise moments should reach


@pytest.fixture(scope="module")
def rpst():
    import rpst as m
    return m


def dev(t):
    return t.cuda()


@pytest.mark.parametrize("tag", ["odd", "sq", "signed"])
def test_golden(rpst, golden, tag):
    g = golden(f"adain_{tag}")
    c, s, p = dev(g["content"]), dev(g["style"]), dev(g["prev"])
    mean, std = rpst.calc_mean_std(c)
    assert mean.shape == g["mean"].shape and std.shape == g["std"].shape
    assert R.rel_l2(mean, g["mean"]) < TIGHT and R.rel_l2(std, g["std"]) < TIGHT
    assert R.rel_l2(rpst.adaptive_instance_normalization(c, s), g["out"]) < TIGHT
    assert R.rel_l2(rpst.adain_blend(p, c, s), g["blend"]) < TIGHT
    assert R.rel_l2(rpst.mean_variance_norm(c), g["mvn"]) < TIGHT


def test_golden_hw2(rpst, golden):
    g = golden("adain_hw2")
    out = rpst.adaptive_instance_normalization(dev(g["content"]), dev(g["style"]))
    assert R.rel_l2(out, g["out"]) < 1e-5


def test_hw1_is_nan_like_torch(rpst):
    c = torch.randn(1, 2, 1, 1).cuda()
    mean, std = rpst.calc_mean_std(c)
    assert torch.isnan(std).all() and torch.equal(mean.cpu(), c.cpu())


# direct kernel (register resident), pipelined kernel (vector + tail chunk), scalar paths, big plane
SHAPES = [(2, 3, 8, 8), (1, 512, 64, 64), (2, 5, 128, 128), (1, 3, 300, 300), (2, 4, 512, 512),
          (1, 2, 301, 301), (1, 3, 33, 31), (1, 2, 1024, 2048), (3, 2, 130, 130)]


@pytest.mark.parametrize("shape", SHAPES)
def test_vs_oracle(rpst, shape):
    c, s = R.synth_features(shape, cfg=sum(shape) % 7)
    prev = torch.randn(shape, generator=torch.Generator().manual_seed(9))
    cd, sd, pd = dev(c), dev(s), dev(prev)
    want = R.adain(c, s, dtype=torch.float64)
    assert R.rel_l2(rpst.adaptive_instance_normalization(cd, sd), want) < TIGHT
    assert R.rel_l2(rpst.adain_blend(pd, cd, sd), want + prev.double()) < TIGHT
    mu, sd_ = R.plane_stats(c, dtype=torch.float64)
    gm, gs = rpst.calc_mean_std(cd)
    assert R.rel_l2(gm, mu) < TIGHT and R.rel_l2(gs, sd_) < TIGHT
    assert R.rel_l2(rpst.mean_variance_norm(cd), R.mean_variance_norm(c, dtype=torch.float64)) < TIGHT


def test_large_mean_small_std_is_stable(rpst):
    # sum/sum-of-squares would lose everything here; (count, mean, M2) merging must not
    g = torch.Generator().manual_seed(3)
    c = 1000.0 + 0.01 * torch.randn(1, 2, 512, 512, generator=g)
    s = torch.randn(1, 2, 512, 512, generator=g)
    want = R.adain(c, s, dtype=torch.float64)
    got = rpst.adaptive_instance_normalization(dev(c), dev(s))
    # the reference's own fp32 path cannot represent the mean of such a plane better than ulp(1000);
    # the kernel carries the mean as hi+lo and must do at least as well as eager fp32, and < 1e-3
    eager_err = R.rel_l2(R.adain(c, s), want)
    err = R.rel_l2(got, want)
    assert err < 1e-3 and err <= max(eager_err, 1e-4), (err, eager_err)


def test_concat_write_and_alias(rpst):
    c, s = R.synth_features((2, 6, 96, 96), cfg=2)
    prev = torch.randn(2, 10, 96, 96)
    got = rpst.adain_concat(dev(prev), dev(c), dev(s))
    want = torch.cat([prev.double(), R.adain(c, s, dtype=torch.float64)], dim=1)
    assert got.shape == want.shape and R.rel_l2(got, want) < TIGHT
    # LDMS variant: prev aliases content (network/adain_rp.py:543-552)
    cd, sdv = dev(c), dev(s)
    got = rpst.adain_blend(cd, cd, sdv)
    assert R.rel_l2(got, c.double() + R.adain(c, s, dtype=torch.float64)) < TIGHT


def test_shape_mismatch_asserts_like_reference(rpst):
    c = torch.zeros(1, 2, 8, 8).cuda()
    with pytest.raises(AssertionError):
        rpst.adaptive_instance_normalization(c, c[:, :, :4])


def test_non_contiguous_and_unaligned_inputs(rpst):
    c, s = R.synth_features((2, 4, 40, 44), cfg=1)
    cd = dev(c).transpose(2, 3).contiguous().transpose(2, 3)        # non-contiguous view
    got = rpst.adaptive_instance_normalization(cd, dev(s))
    assert R.rel_l2(got, R.adain(c, s, dtype=torch.float64)) < TIGHT
    buf = torch.zeros(c.numel() + 1, device="cuda")
    buf[1:] = dev(c).reshape(-1)
    cu = buf[1:].view(c.shape)                                      # 4-byte aligned only -> scalar path
    got = rpst.adaptive_instance_normalization(cu, dev(s))
    assert R.rel_l2(got, R.adain(c, s, dtype=torch.float64)) < TIGHT


@pytest.mark.parametrize("shape", [(2, 3, 16, 16), (1, 2, 300, 300), (2, 2, 512, 512)])
def test_backward_matches_autograd_of_the_reference_formula(rpst, shape):
    c, s = R.synth_features(shape, cfg=5, signed=True)
    prev = torch.randn(shape)
    w = torch.randn(shape, generator=torch.Generator().manual_seed(4))

    def ref(c, s, p):
        n, ch = c.shape[:2]
        def ms(x):
            f = x.reshape(n, ch, -1)
            return f.mean(2).view(n, ch, 1, 1), (f.var(2) + 1e-5).sqrt().view(n, ch, 1, 1)
        mc, sc = ms(c)
        m_s, ss = ms(s)
        return (c - mc) / sc * ss + m_s + p

    c64, s64, p64 = (t.double().requires_grad_() for t in (c, s, prev))
    (ref(c64, s64, p64) * w.double()).sum().backward()
    cd, sd, pd = (dev(t).requires_grad_() for t in (c, s, prev))
    (rpst.adain_blend(pd, cd, sd) * dev(w)).sum().backward()
    assert R.rel_l2(cd.grad, c64.grad) < 1e-4
    assert R.rel_l2(sd.grad, s64.grad) < 1e-4
    assert R.rel_l2(pd.grad, p64.grad) < 1e-6
    # statistics with autograd (style loss path, network/adain_rp.py:84-88)
    x64 = c.double().requires_grad_()
    f = x64.reshape(shape[0], shape[1], -1)
    (f.mean(2).sum() * 0.3 + ((f.var(2) + 1e-5).sqrt() * 1.7).sum()).backward()
    xd = dev(c).requires_grad_()
    m, sdev = rpst.calc_mean_std(xd)
    (m.sum() * 0.3 + (sdev * 1.7).sum()).backward()
    assert R.rel_l2(xd.grad, x64.grad) < 1e-4


def test_properties_at_full_plane_size(rpst):
    """Size-independent properties at BASELINE config #2's plane size (512x512), C=256, N=2:
    statistics of AdaIN(c,s) equal those of s; AdaIN is invariant to an affine map of the content;
    blend - plain == prev."""
    shape = (2, 256, 512, 512)
    c, s = R.synth_features(shape, cfg=2, device="cuda")
    out = rpst.adaptive_instance_normalization(c, s)
    mo, so = rpst.calc_mean_std(out)
    ms_, ss = rpst.calc_mean_std(s)
    assert R.rel_l2(mo, ms_) < 1e-5 and R.rel_l2(so, ss) < 1e-5
    out2 = rpst.adaptive_instance_normalization(c * 3.0 + 2.0, s)
    assert R.rel_l2(out2, out) < 1e-5
    prev = torch.randn(shape, device="cuda")
    assert R.rel_l2(rpst.adain_blend(prev, c, s) - out, prev) < 1e-5
    # and one sample slice against the oracle
    want = R.adain(c[:1, :8].cpu(), s[:1, :8].cpu(), dtype=torch.float64)
    assert R.rel_l2(out[:1, :8], want) < TIGHT


def test_tuning_variants_agree(rpst):
    """Scheduling knobs must not change results: bit-identical within a kernel path (the reduction
    tree is fixed), and to fp32 rounding between the TMA-staged and the register-staged path."""
    c, s = R.synth_features((2, 8, 512, 512), cfg=3, device="cuda")
    keys = ("adain_lag_bytes", "adain_hints", "adain_path")
    old = {k: rpst.get_tuning(k) for k in keys}
    try:
        ref = {}
        for lag, hints, path in [(16 << 20, 1, 1), (1 << 20, 0, 1), (64 << 20, 1, 1), (1, 1, 1), (16 << 20, 1, 0),
                                 (8 << 20, 1, 0), (32 << 20, 0, 0), (1, 1, 0)]:
            for k, v in zip(keys, (lag, hints, path)):
                rpst.set_tuning(k, v)
            out = rpst.adaptive_instance_normalization(c, s)
            if path in ref:
                assert torch.equal(out, ref[path]), (lag, hints, path)
            else:
                ref[path] = out
        assert R.rel_l2(ref[0], ref[1]) < 1e-6
    finally:
        for k, v in old.items():
            rpst.set_tuning(k, v)


# channel shuffle / sort folded into the loads (SURVEY.md §8f rank 3): direct, scalar-pipelined and TMA paths
@pytest.mark.parametrize("shape", [(2, 8, 16, 16), (2, 8, 150, 151), (2, 16, 256, 256), (1, 8, 512, 512)])
@pytest.mark.parametrize("blend", [False, True])
def test_mapped_matches_materialised_permutation(rpst, shape, blend):
    n, ch = shape[:2]
    c, s = R.synth_features(shape, cfg=50)
    prev = torch.randn(shape, generator=torch.Generator().manual_seed(9)) if blend else None
    g = torch.Generator().manual_seed(51)
    att_c, att_s = torch.rand(n, ch, 1, 1, generator=g), torch.rand(n, ch, 1, 1, generator=g)
    shuf = rpst.shuffle_map(n, ch, 4, "cuda")
    cm = rpst.compose_maps(shuf, rpst.sort_map(att_c.cuda()))
    sm = rpst.sort_map(att_s.cuda())
    # reference spelling: shuffle (network/adain_rp.py:304-311), then sort_by_weights (:230-249), then AdaIN
    def shuffle(f):
        N, C, H, W = f.size()
        return f.view(N, 4, C // 4, H, W).permute(0, 2, 1, 3, 4).contiguous().view(N, C, H, W)
    def sort(f, att):
        _, idx = att.sort(dim=1, descending=True)
        return torch.cat([torch.index_select(f[b].unsqueeze(0), 1, idx[b].view(-1)) for b in range(f.shape[0])], 0)
    want = R.adain(sort(shuffle(c), att_c), sort(s, att_s), dtype=torch.float64)
    if blend:
        want = want + prev.double()
    got = rpst.adain_mapped(c.cuda(), s.cuda(), cm, sm, prev=None if prev is None else prev.cuda())
    assert R.rel_l2(got, want) < TIGHT
    # identity maps reproduce the unmapped call bit for bit
    ident = torch.arange(n * ch, dtype=torch.int32, device="cuda")
    a = rpst.adain_mapped(c.cuda(), s.cuda(), ident, ident)
    b = rpst.adaptive_instance_normalization(c.cuda(), s.cuda())
    assert torch.equal(a, b)


def test_mapped_autograd_matches_gather(rpst):
    c, s = R.synth_features((2, 8, 20, 20), cfg=52, signed=True)
    m = rpst.shuffle_map(2, 8, 4, "cuda")
    cg, sg = c.cuda().requires_grad_(), s.cuda().requires_grad_()
    w = torch.randn(c.shape, generator=torch.Generator().manual_seed(53))   # sum(out^2) alone is ~constant in c
    out = rpst.adain_mapped(cg, sg, m, m)
    (out * w.cuda()).sum().backward()
    cd, sd = c.double().requires_grad_(), s.double().requires_grad_()
    ml = m.long().cpu()
    cp, sp = cd.flatten(0, 1)[ml].view_as(cd), sd.flatten(0, 1)[ml].view_as(sd)
    mu_c, sd_c = cp.mean((2, 3), keepdim=True), (cp.var((2, 3), keepdim=True) + 1e-5).sqrt()
    mu_s, sd_s = sp.mean((2, 3), keepdim=True), (sp.var((2, 3), keepdim=True) + 1e-5).sqrt()
    (((cp - mu_c) / sd_c * sd_s + mu_s) * w.double()).sum().backward()
    assert R.rel_l2(cg.grad, cd.grad) < 1e-4 and R.rel_l2(sg.grad, sd.grad) < 1e-4


def test_random_shapes_and_misaligned_views(rpst):
    """Seeded fuzz over the dispatch space: tiny / ragged / multi-chunk planes, pointers that are only 4-byte
    aligned (views at an element offset -> scalar kernels), odd chunk tails on the TMA path (twin apply items
    with an odd number of chunks), blend and plain, against the fp64 oracle."""
    rng = torch.Generator().manual_seed(1234)
    hws = [(1, 2), (3, 5), (17, 19), (64, 64), (100, 164), (128, 129), (160, 160), (192, 256), (257, 255), (384, 300)]
    for i, (h, w) in enumerate(hws):
        n = int(torch.randint(1, 3, (1,), generator=rng))
        ch = int(torch.randint(1, 6, (1,), generator=rng))
        numel = n * ch * h * w
        for offset in (0, 1):
            base_c = torch.randn(numel + 4, generator=rng) * 1.5 + 0.3
            base_s = torch.randn(numel + 4, generator=rng) * 0.7 - 0.2
            base_p = torch.randn(numel + 4, generator=rng)
            cg, sg, pg = (b.cuda()[offset:offset + numel].view(n, ch, h, w) for b in (base_c, base_s, base_p))
            c, s, p = (b[offset:offset + numel].view(n, ch, h, w) for b in (base_c, base_s, base_p))
            assert cg.is_contiguous() and (cg.data_ptr() % 16 != 0) == (offset == 1)
            want = R.adain(c, s, dtype=torch.float64)
            tol = 1e-5 if h * w < 8 else TIGHT
            assert R.rel_l2(rpst.adaptive_instance_normalization(cg, sg), want) < tol, (h, w, offset)
            assert R.rel_l2(rpst.adain_blend(pg, cg, sg), want + p.double()) < tol, (h, w, offset)
            assert R.rel_l2(rpst.mean_variance_norm(cg), R.mean_variance_norm(c, dtype=torch.float64)) < tol, (h, w, offset)
            mu, sd = rpst.calc_mean_std(cg)
            wmu, wsd = R.plane_stats(c, dtype=torch.float64)
            assert R.rel_l2(mu, wmu) < tol and R.rel_l2(sd, wsd) < tol


def test_twin_apply_matches_single_chunk_items(rpst):
    """The twin-chunk apply items (no prev) must give the single-chunk result bit for bit."""
    c, s = R.synth_features((2, 3, 300, 300), cfg=60)    # 90000 px = 21.97 chunks: odd tail, partial last chunk
    cg, sg = c.cuda(), s.cuda()
    rpst.set_tuning("adain_twin_apply", 0)
    a = rpst.adaptive_instance_normalization(cg, sg)
    rpst.set_tuning("adain_twin_apply", 1)
    b = rpst.adaptive_instance_normalization(cg, sg)
    assert torch.equal(a, b)
    assert R.rel_l2(b, R.adain(c, s, dtype=torch.float64)) < TIGHT


def test_golden_channel_maps(rpst, golden):
    """shuffle / sort_by_weights outputs of the reference's own methods (tests/golden/channel_maps.npz)."""
    g = golden("channel_maps")
    c, s, att = g["content"].cuda(), g["style"].cuda(), g["attention"].cuda()
    sm = rpst.sort_map(att)
    assert R.rel_l2(rpst.adain_mapped(c, s, sm, sm), g["adain_sorted"]) < TIGHT
    hm = rpst.shuffle_map(2, 8, 4, "cuda")
    assert R.rel_l2(rpst.adain_mapped(c, s, hm, hm), g["adain_shuffled"]) < TIGHT
    assert torch.equal(c.flatten(0, 1)[hm.long()].view_as(c).cpu(), g["shuffled"])
    assert torch.equal(c.flatten(0, 1)[sm.long()].view_as(c).cpu(), g["sorted_content"])


def test_cuda_graph_capture_and_replay(rpst):
    """The C-ABI calls only enqueue stream work (memsets + kernels, no host synchronisation, no allocation of
    their own), so a whole multiscale transform step can be captured once and replayed on new data."""
    levels = [(2, 4, 160, 160), (2, 8, 160, 160), (2, 16, 64, 64)]      # TMA kernel x2, direct kernel (top level)
    cs = [torch.zeros(sh, device="cuda") for sh in levels]
    ss = [torch.zeros(sh, device="cuda") for sh in levels]
    ps = [torch.zeros(sh, device="cuda") for sh in levels[:-1]]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        rpst.multiscale_transform(cs, ss, ps)                             # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = rpst.multiscale_transform(cs, ss, ps)
    for seed in (1, 2):
        g = torch.Generator().manual_seed(seed)
        hc = [torch.randn(sh, generator=g) + 0.3 for sh in levels]
        hs = [torch.randn(sh, generator=g) * 2 - 0.5 for sh in levels]
        hp = [torch.randn(sh, generator=g) for sh in levels[:-1]]
        for d, h in zip(cs + ss + ps, hc + hs + hp):
            d.copy_(h)
        graph.replay()
        torch.cuda.synchronize()
        want = R.multiscale_transform(hc, hs, hp, dtype=torch.float64)
        for o, w in zip(outs, want):
            assert R.rel_l2(o, w) < TIGHT


@pytest.mark.parametrize("shape", [(1, 5, 1024, 2048), (2, 3, 1100, 1000)])
def test_big_planes_group_merge_kernel(rpst, shape):
    """Planes >= 4 MiB take the GROUP_MERGE instantiation (whole-group single-pass fp64 merge, 128 MiB lag):
    plain / blend / mean_variance_norm / statistics saved for the backward pass, incl. a ragged last chunk."""
    c, s = R.synth_features(shape, cfg=80, signed=True)
    prev = torch.randn(shape, generator=torch.Generator().manual_seed(81))
    cg, sg, pg = c.cuda(), s.cuda(), prev.cuda()
    want = R.adain(c, s, dtype=torch.float64)
    assert R.rel_l2(rpst.adaptive_instance_normalization(cg, sg), want) < TIGHT
    assert R.rel_l2(rpst.adain_blend(pg, cg, sg), want + prev.double()) < TIGHT
    assert R.rel_l2(rpst.mean_variance_norm(cg), R.mean_variance_norm(c, dtype=torch.float64)) < TIGHT
    # autograd: forward saves (mu_c, sd_c, mu_s, sd_s) from the group merge, backward consumes them
    w = torch.randn(shape, generator=torch.Generator().manual_seed(82))
    cd, sd = c[:, :2].double().requires_grad_(), s[:, :2].double().requires_grad_()
    mu_c, sd_c = cd.mean((2, 3), keepdim=True), (cd.var((2, 3), keepdim=True) + 1e-5).sqrt()
    mu_s, sd_s = sd.mean((2, 3), keepdim=True), (sd.var((2, 3), keepdim=True) + 1e-5).sqrt()
    (((cd - mu_c) / sd_c * sd_s + mu_s) * w[:, :2].double()).sum().backward()
    cr, sr = cg[:, :2].contiguous().requires_grad_(), sg[:, :2].contiguous().requires_grad_()
    (rpst.adaptive_instance_normalization(cr, sr) * w[:, :2].cuda()).sum().backward()
    assert R.rel_l2(cr.grad, cd.grad) < 1e-4 and R.rel_l2(sr.grad, sd.grad) < 1e-4


# ---- round-2 regressions (ADVICE.md) --------------------------------------------------------------
def _ref_adain_autograd(c, s):
    """the reference formula (network/base.py:399-418) on tensors that keep their autograd graph"""
    mu_c, sd_c = c.mean((2, 3), keepdim=True), (c.var((2, 3), keepdim=True) + 1e-5).sqrt()
    mu_s, sd_s = s.mean((2, 3), keepdim=True), (s.var((2, 3), keepdim=True) + 1e-5).sqrt()
    return (c - mu_c) / sd_c * sd_s + mu_s


# planes with 4096 < hw <= 16384 that cannot take the vectorised direct kernel (odd sizes, 4-byte aligned views)
# go to the pipelined kernels and need the real workspace, forward and backward
@pytest.mark.parametrize("shape", [(1, 2, 75, 75), (1, 2, 127, 127), (2, 3, 65, 65), (1, 2, 101, 101)])
def test_mid_size_odd_planes_forward_backward(rpst, shape):
    c, s = R.synth_features(shape, cfg=11)
    prev = torch.randn(shape, generator=torch.Generator().manual_seed(3))
    w = torch.randn(shape, generator=torch.Generator().manual_seed(4))
    want = R.adain(c, s, dtype=torch.float64)
    assert R.rel_l2(rpst.adaptive_instance_normalization(dev(c), dev(s)), want) < TIGHT
    assert R.rel_l2(rpst.adain_blend(dev(prev), dev(c), dev(s)), want + prev.double()) < TIGHT
    assert R.rel_l2(rpst.mean_variance_norm(dev(c)), R.mean_variance_norm(c, dtype=torch.float64)) < TIGHT
    mean, std = rpst.calc_mean_std(dev(c))
    wm, wsd = R.plane_stats(c, dtype=torch.float64)
    assert R.rel_l2(mean, wm) < TIGHT and R.rel_l2(std, wsd) < TIGHT
    cg, sg = dev(c).requires_grad_(), dev(s).requires_grad_()
    gc, gs = torch.autograd.grad(rpst.adaptive_instance_normalization(cg, sg), (cg, sg), dev(w))
    c64, s64 = c.double().requires_grad_(), s.double().requires_grad_()
    rc, rs = torch.autograd.grad(_ref_adain_autograd(c64, s64), (c64, s64), w.double())
    assert R.rel_l2(gc, rc) < 1e-4 and R.rel_l2(gs, rs) < 1e-4


def test_offset_view_of_mid_size_plane(rpst):
    """a +1-element view of a 96x96 plane is 4-byte aligned only: scalar pipelined path, real workspace"""
    shape = (1, 2, 96, 96)
    c, s = R.synth_features(shape, cfg=12)
    n = c.numel()
    cb, sb = torch.zeros(n + 1).cuda(), torch.zeros(n + 1).cuda()
    cb[1:].copy_(c.reshape(-1)); sb[1:].copy_(s.reshape(-1))
    cv, sv = cb[1:].view(shape), sb[1:].view(shape)
    assert cv.data_ptr() % 16 != 0 and cv.is_contiguous()
    want = R.adain(c, s, dtype=torch.float64)
    assert R.rel_l2(rpst.adaptive_instance_normalization(cv, sv), want) < TIGHT
    cg, sg = cv.detach().requires_grad_(), sv.detach().requires_grad_()
    w = torch.randn(shape, generator=torch.Generator().manual_seed(6))
    gc, _ = torch.autograd.grad(rpst.adaptive_instance_normalization(cg, sg), (cg, sg), dev(w))
    c64, s64 = c.double().requires_grad_(), s.double().requires_grad_()
    rc, _ = torch.autograd.grad(_ref_adain_autograd(c64, s64), (c64, s64), w.double())
    assert R.rel_l2(gc, rc) < 1e-4


def test_only_prev_requires_grad(rpst):
    """frozen encoder / detached features: the decoder state alone carries grad through `prev + AdaIN(c, s)`"""
    shape = (2, 3, 40, 40)
    c, s = R.synth_features(shape, cfg=13)
    prev = dev(torch.randn(shape, generator=torch.Generator().manual_seed(8))).requires_grad_()
    out = rpst.adain_blend(prev, dev(c).detach(), dev(s).detach())
    w = dev(torch.randn(shape, generator=torch.Generator().manual_seed(9)))
    (gp,) = torch.autograd.grad(out, (prev,), w)
    assert torch.equal(gp, w)
    assert R.rel_l2(out, R.adain(c, s, dtype=torch.float64) + prev.detach().cpu().double()) < TIGHT

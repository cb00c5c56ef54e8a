"""WCT linear algebra stage by stage against fp64 references (SURVEY.md §8 a5-a7): covariances and means of every
covariance path, the fp64 products of the Newton-Schulz iteration, the Jacobi eigensolver (every instantiation, its
eigenvalues, sweep counts, spectrum cut and scale equivariance), the Newton-Schulz roots, the transform and the colouring.

Every comparison is per element (per matrix for the roots) and per batch member, against a bound derived in the test.
The covariance and product stages are reached through the white-box hooks of librpst_debug.so
(include/rpst_debug.h); everything else through the product library.  Tests that name a kernel path assert that the
path ran (`path_taken` of the covariance hook, the Newton-Schulz flag counter)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import restate as R

pytestmark = pytest.mark.gpu

PATH_AUTO, PATH_TMA, PATH_STAGED, PATH_PACK = 0, 1, 2, 3
U64 = 2.0 ** -53                       # unit roundoff of fp64
COV_BOUND = {3: 3e-5, 1: 8e-3}         # e_ij = |C^ - C|_ij / sqrt(C_ii C_jj), see test_covariance_channels


@pytest.fixture(scope="module")
def rpst():
    import rpst as m
    return m


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dbg_check(D, code):
    if code != 0:
        msg = D.rpst_last_error()
        raise RuntimeError(f"librpst_debug error {code}: {msg.decode() if msg else ''}")


def _ws(nbytes):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device="cuda")


def covariances(x, passes, diag_add, path):
    """rpst_debug_wct_covariances on x [n, c, hw] fp32: (cov [n,c,c] fp64, mean [n,c] fp32, path that ran)."""
    import rpst
    D = rpst._lib.debug_lib()
    x = x.contiguous()
    n, c, hw = x.shape
    ws = _ws(D.rpst_debug_wct_covariances_workspace_bytes(n, c, hw))
    cov = torch.empty(n, c, c, dtype=torch.float64, device="cuda")
    mean = torch.empty(n, c, dtype=torch.float32, device="cuda")
    taken = ctypes.c_int32(-1)
    _dbg_check(D, D.rpst_debug_wct_covariances(x.data_ptr(), n, c, hw, passes, diag_add, path, cov.data_ptr(), mean.data_ptr(),
                                               ctypes.addressof(taken), ws.data_ptr(), ws.numel(), _stream()))
    torch.cuda.synchronize()
    return cov, mean, taken.value


def reference_covariances(x):
    """fp64 centred covariance [n,c,c] (/ (hw - 1)) and means [n,c] of the fp32 tensor x [n,c,hw]."""
    xd = x.double()
    mu = xd.mean(dim=2, keepdim=True)
    xc = xd - mu
    return xc @ xc.transpose(1, 2) / (x.shape[2] - 1), mu[..., 0]


def cov_errors(x, cov, mean, diag_add):
    """Per sample: max_ij |C^ - C|_ij / sqrt(C_ii C_jj) and max_i |mu^ - mu|_i / (|mu_i| + sigma_i)."""
    C, mu = reference_covariances(x)
    c = x.shape[1]
    want = C + diag_add * torch.eye(c, dtype=torch.float64, device=C.device)
    d = C.diagonal(dim1=1, dim2=2)
    e = ((cov - want).abs() / (d[:, :, None] * d[:, None, :]).sqrt()).amax(dim=(1, 2))
    m = ((mean.double() - mu).abs() / (mu.abs() + d.sqrt())).amax(dim=1)
    return e.tolist(), m.tolist()


def features(n, c, hw, seed, offset=0.5):
    """relu'd normal features through a random channel mixing (correlated channels, covariance far from diagonal), with
    per-channel magnitudes spread over 2^-3 .. 2^3."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.relu(torch.randn(n, c, hw, generator=g, device="cuda") + offset)
    mix = torch.randn(c, c, generator=g, device="cuda") / c ** 0.5
    scale = 2.0 ** torch.randint(-3, 4, (c, 1), generator=g, device="cuda").float()
    return (scale * (mix @ x)).contiguous()


def sign_pattern(n, c, hw, seed):
    """Negative control: every channel is a scaled copy of one +-1 pattern, x_ip = v_i s_p with v_i = 1 + (2i + 1) 2^-12.
    v_i needs 12 mantissa bits, so a single bf16 (8 bits) rounds every element of a channel the same way: those errors do
    NOT average out over hw as they do on random data, and only a bf16x3 split (16 bits) stays within 2^-15."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    s = torch.randint(0, 2, (n, 1, hw), generator=g, device="cuda").float() * 2 - 1
    v = 1.0 + (2 * torch.arange(c, device="cuda", dtype=torch.float32) + 1) * 2.0 ** -12
    return (v.view(1, c, 1) * s).contiguous()


def ragged_hw(k_tiles):
    """hw with exactly k_tiles tiles of 64 positions, the last one partial (hw % 4 == 0, so the fused kernels apply)."""
    return 64 if k_tiles == 1 else 64 * (k_tiles - 1) + 36


# ============================================================================================= A. covariances and means
# Bounds.  passes = 3: each element of (x - shift) is split into bf16 hi + lo (16 significant bits, relative error
# <= 2^-17 per element), so every product x_ip x_jp carries <= 2 * 2^-17 + 2^-18 (the dropped lo*lo term) of |x_ip x_jp|;
# summed over p, Cauchy-Schwarz bounds sum_p |x_ip x_jp| by (hw - 1) sqrt(C_ii C_jj) for centred data, giving
# e_ij <= 2^-15.4 plus the fp32 accumulation of the tensor cores (<= 2^-24 per position of a CTA's slice, random on
# random data): 3e-5 ~ 2^-15.  passes = 1: one bf16 per element (2^-9 each), e_ij <= 2^-8 = 3.9e-3, so 8e-3.
# Means: exact shift + fp64 sum of the fp32 row sums of (x - shift), rounded to fp32: 2^-24 |mu| + sum errors << 1e-6.
def _assert_cov(x, passes, diag_add, path, want_path):
    cov, mean, taken = covariances(x, passes, diag_add, path)
    assert taken == want_path, (taken, want_path)
    e, m = cov_errors(x, cov, mean, diag_add)
    for b in range(x.shape[0]):
        assert e[b] <= COV_BOUND[passes], (b, passes, e[b])
        assert m[b] <= 1e-6, (b, m[b])
    return e


@pytest.mark.parametrize("passes", [3, 1])
@pytest.mark.parametrize("c", [1, 2, 63, 64, 65, 127, 128, 129, 200, 255, 256])
def test_covariance_channels(c, passes):
    """Production dispatch at 150 k-tiles (the one-launch TMA kernel on a 148-SM B200): channel counts around the 128-row
    boundary (padding to 128 / 256 rows from 129 on; the SYRK skips block (1,0) for rows >= 128), content-side diag_add."""
    x = features(2, c, ragged_hw(150), seed=100 + c)
    _assert_cov(x, passes, 1.0, PATH_AUTO, PATH_TMA)


@pytest.mark.parametrize("c", [257, 384, 512])
def test_covariance_pack_path_channels(c):
    """More than 256 channels: pack + split-K tcgen05 GEMM + fp64 reduce."""
    x = features(2, c, 2100, seed=200 + c)
    _assert_cov(x, 3, 1.0, PATH_AUTO, PATH_PACK)


@pytest.mark.parametrize("k_tiles", [64, 100, 144, 145, 147, 148, 149, 4096])
def test_covariance_grid_sizes(k_tiles):
    """Grid = min(SMs, k-tiles) CTAs of the one-launch kernel, whose in-kernel finalize deals the per-CTA partial Grams over
    18 slices: 144 .. 149 k-tiles reach the last slices (zs + 144 < 148).  4096 k-tiles is one config #3 plane (256 x 512^2)."""
    c = 256
    if k_tiles == 4096:
        x = features(1, c, 512 * 512, seed=3)
    else:
        x = features(2, c, ragged_hw(k_tiles), seed=300 + k_tiles)
    _assert_cov(x, 3, 1.0, PATH_AUTO, PATH_TMA)


@pytest.mark.parametrize("k_tiles", [1, 2, 17, 18, 19, 37, 63])
def test_covariance_forced_tma_small_grids(k_tiles):
    """The one-launch kernel below its 64-CTA production threshold: a finalize spread over few CTAs (one CTA walks every
    row at 1 CTA), partial slices that are mostly empty."""
    x = features(2, 200, ragged_hw(k_tiles), seed=400 + k_tiles)
    _assert_cov(x, 3, 0.0, PATH_TMA, PATH_TMA)


@pytest.mark.parametrize("c,hw,path", [(64, ragged_hw(11), PATH_AUTO), (256, 64 * 63, PATH_AUTO), (1, 64, PATH_AUTO),
                                       (129, ragged_hw(150), PATH_STAGED), (256, ragged_hw(300), PATH_STAGED)])
def test_covariance_register_staged(c, hw, path):
    """Register-staged kernel + separate rowsum / finalize launches: production for 64 <= hw with < 64 k-tiles, forced
    at large grids (two converter groups per CTA, every CTA with several k-tiles)."""
    x = features(2, c, hw, seed=500 + c)
    _assert_cov(x, 3, 1.0, path, PATH_STAGED)


@pytest.mark.parametrize("c,hw", [(64, 33 * 31), (128, 60), (3, 25), (200, 4097), (5, 6)])
def test_covariance_pack_path_small_or_unaligned(c, hw):
    """hw % 4 != 0 or hw < 64: pack + GEMM + reduce, with ragged k-tiles and channel tiles."""
    x = features(2, c, hw, seed=600 + c)
    _assert_cov(x, 3, 1.0, PATH_AUTO, PATH_PACK)


@pytest.mark.parametrize("path", [PATH_TMA, PATH_STAGED, PATH_PACK])
def test_covariance_mean_far_from_zero(path):
    """|mean| >> std (channel means 40 .. 230, std 0.05 .. 0.4): centring by a sub-sampled shift (fused kernels) or by the
    fp32 mean (pack path) must keep the rank-1 correction free of cancellation."""
    c, hw = 64, ragged_hw(150)
    g = torch.Generator(device="cuda").manual_seed(21)
    sd = 0.05 * 2.0 ** torch.randint(0, 4, (c, 1), generator=g, device="cuda").float()
    mix = torch.eye(c, device="cuda") + 0.3 * torch.randn(c, c, generator=g, device="cuda") / c ** 0.5
    x = mix @ (torch.randn(2, c, hw, generator=g, device="cuda") * sd)
    x = (x + 40.0 + 3.0 * torch.arange(c, device="cuda").view(1, c, 1)).contiguous()
    _assert_cov(x, 3, 1.0, path, path)


@pytest.mark.parametrize("path", [PATH_TMA, PATH_STAGED, PATH_PACK])
def test_covariance_negative_control_sign_pattern(path):
    """On random data bf16 rounding errors average out over hw and passes = 1 would meet the passes = 3 bound, which then
    proves nothing.  On the sign pattern they do not: passes = 1 must violate the 3e-5 bound, passes = 3 must meet it.
    hw = 64 x 148 keeps every CTA's fp32 accumulation to one k-tile (same-sign terms accumulate their rounding)."""
    x = sign_pattern(2, 128, 64 * 148, seed=7)
    e3 = _assert_cov(x, 3, 1.0, path, path)
    cov, mean, taken = covariances(x, 1, 1.0, path)
    assert taken == path
    e1, _ = cov_errors(x, cov, mean, 1.0)
    for b in range(2):
        assert e1[b] > COV_BOUND[3], (b, e1[b], e3[b])


# ============================================================================================= B. fp64 products
def dgemm(a, b, dmma=True):
    import rpst
    D = rpst._lib.debug_lib()
    batch, n = a.shape[:2]
    c = torch.empty_like(a)
    if not dmma:
        _dbg_check(D, D.rpst_set_tuning(b"ns_dmma", 0))
    try:
        _dbg_check(D, D.rpst_debug_dgemm_batched(a.data_ptr(), b.data_ptr(), c.data_ptr(), batch, n, _stream()))
        torch.cuda.synchronize()
    finally:
        if not dmma:
            D.rpst_set_tuning(b"ns_dmma", 1)
    return c


def _check_dgemm(n, batch, dmma):
    """|C^ - C|_ij <= 2 gamma_n (|A||B|)_ij: the kernel's fp64 product and the reference's (cuBLAS fp64) are each within
    gamma_n = n u / (1 - n u) (|A||B|)_ij of the exact one, whatever the summation order.  Rows of both operands are
    scaled by 2^-20 .. 2^20, so a product that mixed up rows, columns, k-tiles or batch members fails by orders of
    magnitude."""
    g = torch.Generator(device="cuda").manual_seed(1000 * n + batch)
    def operand():
        m = torch.randn(batch, n, n, generator=g, device="cuda", dtype=torch.float64)
        return m * 2.0 ** torch.randint(-20, 21, (batch, n, 1), generator=g, device="cuda").double()
    a, b = operand(), operand()
    got = dgemm(a, b, dmma)
    want = a @ b
    gam = n * U64 / (1 - n * U64)
    bound = 2 * gam * (a.abs() @ b.abs())
    ratio = ((got - want).abs() / bound).amax(dim=(1, 2))
    for k in range(batch):
        assert ratio[k] <= 1.0, (n, batch, k, float(ratio[k]))


@pytest.mark.parametrize("batch", [1, 16])
@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 127, 128, 129, 130, 200, 255, 256, 257, 511, 512])
def test_dgemm_batched(n, batch):
    """Odd n: DFMA register-staged kernel; even n: DMMA kernel, 64-row tiles for batch 1 and 128-row tiles for batch 16
    from n = 200 on (gemm_tile_rows: fewer than 2/3 of the SMs busy -> 64 rows)."""
    _check_dgemm(n, batch, True)


@pytest.mark.parametrize("n,batch", [(64, 1), (130, 16), (256, 1), (512, 2)])
def test_dgemm_batched_even_dfma(n, batch):
    """The DFMA kernel's cp.async path (even n) only runs with the ns_dmma knob off: no shape reaches it."""
    _check_dgemm(n, batch, False)


# ============================================================================================= C. eigensolver
def spectrum_matrices(spectra, seed):
    """A_b = Q_b diag(e_b) Q_b^T from an fp64 QR, with Q_b returned (CPU fp64)."""
    g = torch.Generator().manual_seed(seed)
    a, q = [], []
    for e in spectra:
        n = len(e)
        qb, _ = torch.linalg.qr(torch.randn(n, n, dtype=torch.float64, generator=g))
        ab = (qb * torch.as_tensor(e, dtype=torch.float64)) @ qb.t()
        a.append((ab + ab.t()) / 2)
        q.append(qb)
    return torch.stack(a), torch.stack(q)


def sym_eig(a, diag_add):
    """rpst_sym_eig_fn: sqrt, inv_sqrt, eigenvalues (column norms, i.e. |lambda + diag_add|, unsorted) and sweeps."""
    import rpst
    L = rpst._lib.lib()
    a = a.cuda().contiguous()
    b, n = a.shape[:2]
    ws = _ws(L.rpst_sym_eig_fn_workspace_bytes(b, n))
    rs, ri = torch.empty_like(a), torch.empty_like(a)
    ev = torch.empty(b, n, dtype=torch.float64, device="cuda")
    sw = torch.full((b,), -1, dtype=torch.int32, device="cuda")
    rpst._lib.check(L.rpst_sym_eig_fn(a.data_ptr(), b, n, diag_add, rs.data_ptr(), ri.data_ptr(), ev.data_ptr(), sw.data_ptr(),
                                      ws.data_ptr(), ws.numel(), _stream()))
    torch.cuda.synchronize()
    return rs.cpu(), ri.cpu(), ev.cpu(), sw.cpu()


def rel_fro(got, want):
    return float((got - want).norm() / want.norm())


def _check_eig(spectra, diag_add, seed):
    """Per member: sorted eigenvalues within 16 n u max|lambda| of |e + diag_add| (Weyl: one-sided Jacobi is backward stable
    with a backward error of a few n u ||A|| after its sweeps); sqrt within 1e-11 and inv_sqrt within 1e-11 kappa (the
    root's condition numbers sqrt(kappa) / 2 and kappa / 2 times that backward error); fewer than 20 sweeps (converged)."""
    a, q = spectrum_matrices(spectra, seed)
    rs, ri, ev, sw = sym_eig(a, diag_add)
    for b, e in enumerate(spectra):
        lam = np.abs(np.asarray(e, dtype=np.float64) + diag_add)
        n = len(e)
        got = np.sort(ev[b].numpy())
        tol = 16 * n * U64 * lam.max()
        assert np.abs(got - np.sort(lam)).max() <= tol, (b, n, np.abs(got - np.sort(lam)).max() / lam.max())
        assert 0 < int(sw[b]) < 20, (b, int(sw[b]))
        lt = torch.as_tensor(lam)
        want_r = (q[b] * lt.sqrt()) @ q[b].t()
        want_i = (q[b] / lt.sqrt()) @ q[b].t()
        kappa = float(lam.max() / lam.min())
        assert rel_fro(rs[b], want_r) <= 1e-11, (b, n, rel_fro(rs[b], want_r))
        assert rel_fro(ri[b], want_i) <= 1e-11 * kappa, (b, n, rel_fro(ri[b], want_i), kappa)


def _spectra(n, batch, seed):
    rng = np.random.default_rng(seed)
    return [10.0 ** rng.uniform(-3, 0, n) for _ in range(batch)]


@pytest.mark.parametrize("diag_add", [0.0, 1e-4])
@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 64, 65, 128, 129, 256, 257, 511, 512])
def test_eig_16_column_blocks(n, diag_add):
    """Every 16-column-block instantiation (padded orders 32 .. 512, cluster sizes 1 .. 16), padded and exact orders."""
    _check_eig(_spectra(n, 2, n), diag_add, seed=n)


@pytest.mark.parametrize("diag_add", [0.0, 1e-4])
@pytest.mark.parametrize("n,batch", [(64, 81), (128, 41), (256, 21)])
def test_eig_32_column_blocks(n, batch, diag_add):
    """32-column blocks run when batch * (padded order / 32) > 160 CTAs (eig_decompose): 81 x 64, 41 x 128, 21 x 256."""
    assert batch * (n // 32) > 160
    _check_eig(_spectra(n, batch, 7 * n), diag_add, seed=7 * n)


def test_eig_spectrum_cut():
    """network/wct_rp.py:14-17: eigenvalues below 1e-5 are dropped from both roots (3e-6 here), 3e-5 is kept."""
    rng = np.random.default_rng(11)
    e = np.concatenate([[3e-6, 3e-5], 10.0 ** rng.uniform(-4, 0, 62)])
    a, q = spectrum_matrices([e], seed=11)
    rs, ri, ev, sw = sym_eig(a, 0.0)
    assert np.abs(np.sort(ev[0].numpy()) - np.sort(e)).max() <= 16 * 64 * U64
    keep = torch.as_tensor(np.where(e >= 1e-5, 1.0, 0.0))
    et = torch.as_tensor(e)
    want_r = (q[0] * (et.sqrt() * keep)) @ q[0].t()
    want_i = (q[0] * (keep / et.sqrt())) @ q[0].t()
    assert rel_fro(rs[0], want_r) <= 1e-11, rel_fro(rs[0], want_r)
    assert rel_fro(ri[0], want_i) <= 1e-11 * 3e4, rel_fro(ri[0], want_i)
    assert 0 < int(sw[0]) < 20


def test_eig_indefinite_input_abs_semantics(rpst):
    """torch.svd in network/wct_rp.py:11 takes |lambda|: an indefinite input gives V diag(|lambda + 1e-4|^(1/2)) V^T."""
    rng = np.random.default_rng(12)
    e = 10.0 ** rng.uniform(-2, 0, 96) * np.where(rng.uniform(size=96) < 0.4, -1.0, 1.0)
    a, q = spectrum_matrices([e], seed=12)
    got = rpst.matrix_sqrt(a[0].cuda()).cpu()
    assert rel_fro(got, R.matrix_sqrt(a[0])) <= 1e-11, rel_fro(got, R.matrix_sqrt(a[0]))
    want = (q[0] * torch.as_tensor(np.abs(e + 1e-4)).sqrt()) @ q[0].t()
    assert rel_fro(got, want) <= 1e-11


def test_eig_scale_equivariance():
    """sqrt(4^j A) = 2^j sqrt(A) for j in [-30, 30], diag_add = 0: scaling by a power of four is exact in fp64 and the
    solver must not depend on the magnitude of its input.  The spectrum 2^56 x [1e-3, 1] keeps 4^-30 A above the 1e-5 cut
    (6e-5); at the other end the eigenvalues reach 8e34 (squared column norms 7e69).  Before the power-of-two rescaling of the
    rotation angle, lambda_i lambda_j > ~1.8e19 overflowed fp32, such pairs counted as converged and were never rotated
    (measured on a B200: relative error 2.5 from j = -10 on after one "converged" sweep, NaN from j = 5 on)."""
    n = 32
    e = 2.0 ** 56 * np.logspace(0, -3, n)
    a, q = spectrum_matrices([e], seed=13)
    js = list(range(-30, 31))
    batch = torch.cat([a * 4.0 ** j for j in js])
    rs, _, ev, sw = sym_eig(batch, 0.0)
    want = (q[0] * torch.as_tensor(e).sqrt()) @ q[0].t()
    j0 = js.index(0)
    equi = [rel_fro(rs[k] / 2.0 ** j, rs[j0]) for k, j in enumerate(js)]
    acc = [rel_fro(rs[k] / 2.0 ** j, want) for k, j in enumerate(js)]
    assert max(equi) <= 1e-12 and max(acc) <= 1e-11, (max(equi), max(acc), [int(s) for s in sw])
    assert int(sw.max()) < 20, [int(s) for s in sw]


def test_eig_mixed_scale_batch():
    """One batch, one 1e12-scaled member among ordinary ones: every member converges to its own roots."""
    spectra = _spectra(64, 3, 14)
    spectra[1] = spectra[1] * 1e12
    a, q = spectrum_matrices(spectra, seed=14)
    rs, ri, ev, sw = sym_eig(a, 0.0)
    for b, e in enumerate(spectra):
        et = torch.as_tensor(e)
        want_r = (q[b] * et.sqrt()) @ q[b].t()
        assert rel_fro(rs[b], want_r) <= 1e-11, (b, rel_fro(rs[b], want_r), int(sw[b]))
        assert np.abs(np.sort(ev[b].numpy()) - np.sort(e)).max() <= 16 * 64 * U64 * e.max()
        assert 0 < int(sw[b]) < 20


# ============================================================================================= D. Newton-Schulz roots
@pytest.mark.parametrize("n,batch", [(1, 1), (2, 1), (33, 2), (63, 4), (64, 1), (64, 16), (65, 3), (129, 2), (130, 1),
                                     (200, 2), (256, 1), (256, 16), (257, 1), (512, 1), (512, 3)])
def test_newton_schulz_roots(rpst, n, batch):
    """rpst_spd_roots on prescribed spectra in [0.1, 100] (kappa 1e3) with the exact lmin: the products run on the same
    kernel variants as test_dgemm_batched (odd n DFMA, even n DMMA with 64- / 128-row tiles).  Per matrix: sqrt within
    1e-11, inv_sqrt within 1e-14 kappa + 1e-11 (the accepted iteration leaves ||Z Y - I|| ~ 1e-14; rounding of its ~12
    steps of products).  No matrix may be flagged: a faulty product would otherwise hide behind the Jacobi fallback."""
    rng = np.random.default_rng(n)
    spectra = [10.0 ** rng.uniform(-1, 2, n) for _ in range(batch)]
    for s in spectra:
        s[0], s[-1] = 0.1, 100.0
    a, q = spectrum_matrices(spectra, seed=n + batch)
    before = rpst.get_tuning("wct_ns_flagged")
    root, iroot, flags = rpst.spd_roots(a.cuda(), lmin=0.1, diag_add=0.0)
    assert flags.tolist() == [0] * batch
    assert rpst.get_tuning("wct_ns_flagged") == before
    root, iroot = root.cpu(), iroot.cpu()
    for b, e in enumerate(spectra):
        et = torch.as_tensor(e)
        kappa = float(et.max() / et.min())
        er = rel_fro(root[b], (q[b] * et.sqrt()) @ q[b].t())
        ei = rel_fro(iroot[b], (q[b] / et.sqrt()) @ q[b].t())
        assert er <= 1e-11, (b, er)
        assert ei <= 1e-14 * kappa + 1e-11, (b, ei)


# ============================================================================================= E. transform
# (n, c, hw_c, hw_s, covariance path): c <= 64 takes the Jacobi solver only, c > 64 the Newton-Schulz roots
TRANSFORM_CASES = [(2, 32, 640, 704, PATH_STAGED), (2, 64, 64 * 80, 64 * 75, PATH_TMA), (2, 128, ragged_hw(150), 9600, PATH_TMA),
                   (1, 200, 1023, 1105, PATH_PACK), (1, 256, 64 * 40, 64 * 50, PATH_STAGED), (1, 512, 2100, 2200, PATH_PACK)]
# measured on a B200: at most 2.3e-6 over these cases; the bound is ~4x that
TRANSFORM_BOUND = 1e-5


@pytest.mark.parametrize("method", ["closed-form", "original"])
@pytest.mark.parametrize("n,c,hw_c,hw_s,path", TRANSFORM_CASES)
def test_transform_against_fp64_covariances(rpst, n, c, hw_c, hw_s, path, method):
    """T^ of wct_fuse against network/wct_rp.py:96-110 evaluated on the fp64 covariances of the same fp32 inputs:
    max|T^ - T| / max|T| per sample.  Well conditioned (hw >= 4c, mixed channels): the fp32-grade covariances (2^-15)
    pass through roots of condition ~1 (the +I of the content side, hw >= 4c on the style side), so errors stay at a
    few 1e-6."""
    ct = features(n, c, hw_c, seed=700 + c)
    st = features(n, c, hw_s, seed=800 + c, offset=1.0) * 2
    for x in (ct, st):
        assert covariances(x, 3, 0.0, PATH_AUTO)[2] == path
    before = rpst.get_tuning("wct_ns_flagged")
    _, tr = rpst.wct_fuse(ct.view(n, c, 1, hw_c), st.view(n, c, 1, hw_s), method, return_transform=True)
    assert rpst.get_tuning("wct_ns_flagged") == before          # c > 64: the Newton-Schulz roots were accepted
    tr = tr.cpu()
    for b in range(n):
        _, _, cov_c, _, cov_s = R.wct_covariances(ct[b].double().cpu(), st[b].double().cpu())
        want = R.wct_transform_matrix(cov_c, cov_s, method)
        err = float((tr[b] - want).abs().max() / want.abs().max())
        assert err <= TRANSFORM_BOUND, (b, method, err)


# ============================================================================================= F. colouring
def _check_colouring(ct, st, precision):
    """o = T^ (x - mu_c) + mu_s in fp64 with the kernel's own T^ and fp64 means; per element
    |o^ - o| <= 2^-15 (|T^| |x - mu_c|)_ip + 2^-22 |o_ip|: bf16x3 splits of (x - mu_c) and of fp32(T^) (2^-17 each, 2^-24 for
    the fp32 rounding of T^) and fp32 accumulation over c; the fp32 bias mu_s costs 2^-24 |mu_s| <= 2^-22 |o|.
    Returns the largest error / bound ratio of each sample."""
    import rpst
    n, c, hw = ct.shape
    out, tr = rpst.wct_fuse(ct.view(n, c, 1, hw), st.view(n, c, 1, st.shape[2]), precision=precision, return_transform=True)
    xd = ct.double()
    xc = xd - xd.mean(dim=2, keepdim=True)
    want = tr @ xc + st.double().mean(dim=2, keepdim=True)
    bound = 2.0 ** -15 * (tr.abs() @ xc.abs()) + 2.0 ** -22 * want.abs()
    return ((out.view(n, c, hw).double() - want).abs() / bound).amax(dim=(1, 2)).tolist()


@pytest.mark.parametrize("hw", [4097, 33 * 31])
@pytest.mark.parametrize("c", [3, 64, 65, 200, 256, 512])
def test_colouring_per_element(c, hw):
    """The fused colouring kernel (pwconv.cu) over a batch of 3 samples with scales 1, 8 and 1/4: a mix-up of sample indexing
    (transforms, means, planes) fails the per-element bound."""
    scales = torch.tensor([1.0, 8.0, 0.25], device="cuda").view(3, 1, 1)
    ct = (features(3, c, hw, seed=900 + c) * scales).contiguous()
    st = (features(3, c, hw + 8, seed=950 + c, offset=1.0) / scales).contiguous()
    r = _check_colouring(ct, st, "fp32")
    assert max(r) <= 1.0, r


def test_colouring_negative_control_sign_pattern():
    """On sign-pattern content the single-bf16 colouring (precision bf16) violates the fp32-grade bound, the bf16x3 one
    meets it."""
    ct = sign_pattern(2, 64, 4096, seed=17)
    st = features(2, 64, 4096, seed=18, offset=1.0)
    r3 = _check_colouring(ct, st, "fp32")
    r1 = _check_colouring(ct, st, "bf16")
    assert max(r3) <= 1.0, r3
    assert min(r1) > 1.0, r1

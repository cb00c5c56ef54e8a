"""Host-side mirror of the reference's transform FUNCTIONS (same names, arguments and error
behaviour), each a thin call into librpst through the C ABI.

Reference interfaces mirrored (paths relative to the reference root):
  calc_mean_std                        network/base.py:399-407
  adaptive_instance_normalization      network/base.py:410-418
  mean_variance_norm                   network/sanet.py:20-24
plus the fused forms the reference spells as two ops:
  adain_blend(prev, c, s)              network/adain_rp.py:300-301  (`stylized + AdaIN(c, s)`)
  adain_concat(prev, c, s)             network/adain_rp.py:793      (`cat([stylized, AdaIN(c, s)], 1)`)
  adain_mapped(c, s, cmap, smap, prev) network/adain_rp.py:230-249,304-311 (channel shuffle / sort folded into the loads)
"""
from __future__ import annotations

import functools
from typing import Optional, Tuple

import torch

from . import _lib

EPS = 1e-5


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _cuda_tensors(values):
    for v in values:
        if isinstance(v, torch.Tensor):
            if v.is_cuda:
                yield v
        elif isinstance(v, (list, tuple)):
            for w in v:
                if isinstance(w, torch.Tensor) and w.is_cuda:
                    yield w


def device_guard(fn):
    """Entry-point decorator: librpst launches on the CURRENT device and stream, so every tensor argument must
    live on one device and the call runs with that device current (the reference's torch ops follow their
    tensors' device; a model on cuda:1 must keep working while cuda:0 is current)."""

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        for t in _cuda_tensors(args):
            if dev is None:
                dev = t.device
            elif t.device != dev:
                raise RuntimeError(f"rpst.{fn.__name__}: tensor arguments live on different devices ({dev} and {t.device})")
        if kwargs:
            for t in _cuda_tensors(kwargs.values()):
                if dev is None:
                    dev = t.device
                elif t.device != dev:
                    raise RuntimeError(f"rpst.{fn.__name__}: tensor arguments live on different devices ({dev} and {t.device})")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)

    return wrapper


def _prep(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError(f"rpst: `{name}` must be a CUDA tensor (there is no CPU path)")
    if t.dtype != torch.float32:
        raise TypeError(f"rpst: `{name}` must be float32, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


_DIRECT_MAX_HW = 16384        # vectorised register-resident kernel: hw % 4 == 0, every pointer 16-byte aligned
_DIRECT_MAX_HW_SCALAR = 4096  # scalar register-resident kernel (odd plane sizes / 4-byte aligned views)
_tiny_ws = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _goes_direct(hw: int, tensors) -> bool:
    """Mirror of the dispatch in csrc/adain.cu (`run_adain`, `rpst_adain_bwd`): the workspace-free direct
    kernel serves planes <= 4096 elements always, and <= 16384 only on the 128-bit path."""
    if hw <= _DIRECT_MAX_HW_SCALAR:
        return True
    return hw <= _DIRECT_MAX_HW and hw % 4 == 0 and all(t is None or t.data_ptr() % 16 == 0 for t in tensors)


def _plane_workspace(query, args, hw: int, device, tensors=()) -> torch.Tensor:
    """Workspace for the plane kernels; planes that are certain to take the register-resident kernel never
    touch it, so a cached 256-byte buffer is passed and the size query is skipped (config #1 is
    launch-latency bound, every host us counts).  Everything else asks the library."""
    if _goes_direct(hw, tensors):
        key = (device.type, device.index)
        ws = _tiny_ws.get(key)
        if ws is None:
            ws = _tiny_ws[key] = torch.empty(256, dtype=torch.uint8, device=device)
        return ws
    return _workspace(query(*args), device)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


# ------------------------------------------------------------------------------------ raw calls
def _stats_raw(feat: torch.Tensor, eps: float) -> Tuple[torch.Tensor, torch.Tensor]:
    n, c = feat.shape[:2]
    hw = feat[0, 0].numel() if feat.numel() else 0
    mean = torch.empty(n * c, dtype=torch.float32, device=feat.device)
    std = torch.empty_like(mean)
    L = _lib.lib()
    ws = _plane_workspace(L.rpst_stats_workspace_bytes, (n * c, hw), hw, feat.device, (feat,))
    _lib.check(L.rpst_stats_nchw(feat.data_ptr(), n * c, hw, eps, mean.data_ptr(), std.data_ptr(),
                                 ws.data_ptr(), ws.numel(), _stream()))
    return mean, std


def _adain_raw(content, style, prev, out, out_batch_stride, eps, want_saved):
    n, c = content.shape[:2]
    hw = content[0, 0].numel() if content.numel() else 0
    saved = torch.empty(n * c, 4, dtype=torch.float32, device=content.device) if want_saved else None
    L = _lib.lib()
    ws = _plane_workspace(L.rpst_adain_workspace_bytes, (n, c, hw), hw, content.device, (content, style, prev, out))
    if out_batch_stride % 4:
        ws = _workspace(L.rpst_adain_workspace_bytes(n, c, hw), content.device)
    _lib.check(L.rpst_adain_fwd(content.data_ptr(), _ptr(style), _ptr(prev), out.data_ptr(), n, c, hw,
                                out_batch_stride, eps, _ptr(saved), ws.data_ptr(), ws.numel(), _stream()))
    return saved


def _adain_bwd_raw(grad_out, content, style, saved, need_style):
    n, c = content.shape[:2]
    hw = content[0, 0].numel() if content.numel() else 0
    dc = torch.empty_like(content)
    ds = torch.empty_like(content) if need_style else None
    L = _lib.lib()
    ws = _plane_workspace(L.rpst_adain_bwd_workspace_bytes, (n, c, hw), hw, content.device,
                          (grad_out, content, style if need_style else None, dc, ds))
    _lib.check(L.rpst_adain_bwd(grad_out.data_ptr(), content.data_ptr(), _ptr(style) if need_style else None,
                                saved.data_ptr(), dc.data_ptr(), _ptr(ds), n, c, hw,
                                ws.data_ptr(), ws.numel(), _stream()))
    return dc, ds


class _AdaINFn(torch.autograd.Function):
    """out = AdaIN(content, style) [+ prev]; style None => mean_variance_norm."""

    @staticmethod
    def forward(ctx, content, style, prev):
        out = torch.empty_like(content)
        n, c = content.shape[:2]
        hw = content[0, 0].numel() if content.numel() else 0
        need_grad = content.requires_grad or (style is not None and style.requires_grad)
        saved = _adain_raw(content, style, prev, out, c * hw, EPS, need_grad)
        if need_grad:
            ctx.save_for_backward(content, style if style is not None else content, saved)
        ctx.only_prev = not need_grad      # frozen encoder / detached features: only the decoder state carries grad
        ctx.has_style = style is not None
        ctx.has_prev = prev is not None
        return out

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.only_prev:
            return None, None, (grad_out if ctx.has_prev else None)
        content, style, saved = ctx.saved_tensors
        grad_out = grad_out.contiguous()
        need_style = ctx.has_style and ctx.needs_input_grad[1]
        dc, ds = _adain_bwd_raw(grad_out, content, style, saved, need_style)
        return (dc if ctx.needs_input_grad[0] else None, ds,
                grad_out if (ctx.has_prev and ctx.needs_input_grad[2]) else None)


# ------------------------------------------------------------------------------------ public API
@device_guard
def calc_mean_std(feat: torch.Tensor, eps: float = EPS) -> Tuple[torch.Tensor, torch.Tensor]:
    """Drop-in for network/base.py:399 — returns (mean, std), both [N,C,1,1]."""
    size = feat.size()
    assert (len(size) == 4)
    n, c = size[:2]
    if feat.requires_grad and torch.is_grad_enabled():
        # style-loss statistics need autograd; keep them differentiable through a tiny torch graph
        # built on the kernel's numbers: d(mean)/dx and d(std)/dx are cheap closed forms.
        return _StatsFn.apply(feat, eps)
    mean, std = _stats_raw(_prep(feat, "feat"), eps)
    return mean.view(n, c, 1, 1), std.view(n, c, 1, 1)


class _StatsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feat, eps):
        x = _prep(feat, "feat")
        n, c = x.shape[:2]
        mean, std = _stats_raw(x, eps)
        mean, std = mean.view(n, c, 1, 1), std.view(n, c, 1, 1)
        ctx.save_for_backward(x, mean, std)
        return mean, std

    @staticmethod
    def backward(ctx, g_mean, g_std):
        x, mean, std = ctx.saved_tensors
        hw = x[0, 0].numel()
        # d mean/dx = 1/HW ; d std/dx = (x-mean)/((HW-1) std): one fused plane-affine pass
        scale = (g_std / ((hw - 1) * std)).reshape(-1).contiguous()
        shift = (g_mean / hw - scale.view_as(mean) * mean).reshape(-1).contiguous()
        out = torch.empty_like(x)
        _lib.check(_lib.lib().rpst_plane_affine(x.data_ptr(), scale.data_ptr(), shift.data_ptr(), out.data_ptr(),
                                                x.shape[0] * x.shape[1], hw, _stream()))
        return out, None


def _needs_grad(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _adain_nograd(content, style, prev):
    out = torch.empty_like(content)
    c = content.shape[1]
    hw = content[0, 0].numel() if content.numel() else 0
    _adain_raw(content, style, prev, out, c * hw, EPS, False)
    return out


@device_guard
def adaptive_instance_normalization(content_feat: torch.Tensor, style_feat: torch.Tensor) -> torch.Tensor:
    """Drop-in for network/base.py:410."""
    assert (content_feat.size() == style_feat.size())
    assert content_feat.dim() == 4
    c, s = _prep(content_feat, "content_feat"), _prep(style_feat, "style_feat")
    if not _needs_grad(c, s):
        return _adain_nograd(c, s, None)
    return _AdaINFn.apply(c, s, None)


@device_guard
def adain_blend(prev: torch.Tensor, content_feat: torch.Tensor, style_feat: torch.Tensor) -> torch.Tensor:
    """`prev + AdaIN(content_feat, style_feat)` in one pass (network/adain_rp.py:300-301)."""
    assert (content_feat.size() == style_feat.size())
    assert (prev.size() == content_feat.size())
    c, s, p = _prep(content_feat, "content_feat"), _prep(style_feat, "style_feat"), _prep(prev, "prev")
    if not _needs_grad(c, s, p):
        return _adain_nograd(c, s, p)
    return _AdaINFn.apply(c, s, p)


@device_guard
def adain_concat(prev: torch.Tensor, content_feat: torch.Tensor, style_feat: torch.Tensor) -> torch.Tensor:
    """`torch.cat([prev, AdaIN(content_feat, style_feat)], dim=1)` with the AdaIN half written
    straight into the channel slice of the result (network/adain_rp.py:793).  Inference only."""
    assert (content_feat.size() == style_feat.size())
    assert prev.shape[0] == content_feat.shape[0] and prev.shape[2:] == content_feat.shape[2:]
    if torch.is_grad_enabled() and (prev.requires_grad or content_feat.requires_grad or style_feat.requires_grad):
        return torch.cat([prev, adaptive_instance_normalization(content_feat, style_feat)], dim=1)
    c = _prep(content_feat, "content_feat")
    s = _prep(style_feat, "style_feat")
    n, cp = prev.shape[:2]
    cc = c.shape[1]
    hw = c[0, 0].numel()
    out = torch.empty((n, cp + cc) + tuple(c.shape[2:]), dtype=c.dtype, device=c.device)
    out[:, :cp].copy_(prev)
    _adain_raw(c, s, None, out[:, cp:], (cp + cc) * hw, EPS, False)
    return out


def shuffle_map(n: int, c: int, groups: int = 4, device=None) -> torch.Tensor:
    """Plane map of `MultiScaleAdaINRPNet.shuffle` (network/adain_rp.py:304-311):
    `feats.view(N, g, C//g, H, W).permute(0, 2, 1, 3, 4)` => output channel j reads channel
    (j % g) * (C//g) + j // g.  Returns int32 [N*C] global plane indices."""
    j = torch.arange(c, device=device)
    src = (j % groups) * (c // groups) + j // groups
    return (src[None, :] + torch.arange(n, device=device)[:, None] * c).reshape(-1).to(torch.int32)


def sort_map(attention: torch.Tensor) -> torch.Tensor:
    """Plane map of `sort_by_weights` (network/adain_rp.py:230-249): per sample, channels in descending
    order of the SE attention weight [N,C,1,1].  Returns int32 [N*C] global plane indices."""
    n, c = attention.shape[:2]
    _, indexes = attention.sort(dim=1, descending=True)
    indexes = indexes.view(n, c)
    return (indexes + torch.arange(n, device=attention.device)[:, None] * c).reshape(-1).to(torch.int32)


def compose_maps(first: Optional[torch.Tensor], then: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """Map of `then(first(x))`: output plane p reads first[then[p]]."""
    if first is None:
        return then
    if then is None:
        return first
    return first[then.long()].contiguous()


def _check_map(m: Optional[torch.Tensor], name: str, planes: int) -> Optional[torch.Tensor]:
    """A plane map argument: None (identity) or a CUDA int32 tensor with one entry per output plane."""
    if m is None:
        return None
    if not m.is_cuda or m.dtype != torch.int32 or m.numel() != planes:
        raise TypeError(f"rpst: `{name}` must be a CUDA int32 tensor with N*C = {planes} entries")
    return m.contiguous()


@device_guard
def adain_mapped(content_feat: torch.Tensor, style_feat: torch.Tensor, content_map: Optional[torch.Tensor] = None,
                 style_map: Optional[torch.Tensor] = None, prev: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`[prev +] AdaIN(content_feat.flatten(0,1)[content_map], style_feat.flatten(0,1)[style_map])` without
    materialising the permuted tensors (SURVEY.md §8f rank 3).  Maps are int32 [N*C] plane indices."""
    assert (content_feat.size() == style_feat.size())
    assert content_feat.dim() == 4
    c, s = _prep(content_feat, "content_feat"), _prep(style_feat, "style_feat")
    p = None if prev is None else _prep(prev, "prev")
    n, ch = c.shape[:2]
    hw = c[0, 0].numel() if c.numel() else 0
    cm, sm = _check_map(content_map, "content_map", n * ch), _check_map(style_map, "style_map", n * ch)
    if _needs_grad(c, s, p):
        # training: gather through autograd, then the differentiable kernel path
        cg = c if cm is None else c.flatten(0, 1)[cm.long()].view_as(c)
        sg = s if sm is None else s.flatten(0, 1)[sm.long()].view_as(s)
        return _AdaINFn.apply(cg.contiguous(), sg.contiguous(), p)
    out = torch.empty_like(c)
    L = _lib.lib()
    ws = _plane_workspace(L.rpst_adain_workspace_bytes, (n, ch, hw), hw, c.device, (c, s, p, out))
    _lib.check(L.rpst_adain_fwd_mapped(c.data_ptr(), s.data_ptr(), _ptr(p), out.data_ptr(), n, ch, hw, ch * hw, EPS,
                                       _ptr(cm), _ptr(sm), ws.data_ptr(), ws.numel(), _stream()))
    return out


@device_guard
def mean_variance_norm(feat: torch.Tensor) -> torch.Tensor:
    """Drop-in for network/sanet.py:20."""
    assert feat.dim() == 4
    x = _prep(feat, "feat")
    if not _needs_grad(x):
        return _adain_nograd(x, None, None)
    return _AdaINFn.apply(x, None, None)


@device_guard
def plane_affine(x: torch.Tensor, scale: torch.Tensor, shift: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[n,c,:,:] = x[n,c,:,:] * scale[n,c] (+ shift[n,c])."""
    x = _prep(x, "x")
    n, c = x.shape[:2]
    scale = _prep(scale.reshape(-1), "scale")
    assert scale.numel() == n * c
    if shift is not None:
        shift = _prep(shift.reshape(-1), "shift")
    out = torch.empty_like(x)
    _lib.check(_lib.lib().rpst_plane_affine(x.data_ptr(), scale.data_ptr(), _ptr(shift), out.data_ptr(),
                                            n * c, x[0, 0].numel() if x.numel() else 0, _stream()))
    return out

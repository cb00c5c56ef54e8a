"""Segment (mask-label) AdaIN — host-side mirror of network/base.py:494-530 and of the batch loop
`do_mask_stylized` (network/adain_rp.py:313-319, network/base.py:595-601).

The reference takes *paths* to label PNGs and resizes them with PIL inside the transform
(network/base.py:450-451).  Here label maps enter as integer tensors at feature resolution; a path
(or anything `PIL.Image.open` accepts) is still accepted and loaded the way the reference does, so
`test.py`-style callers keep working."""
from __future__ import annotations

from typing import Optional, Sequence, Union

import numpy as np
import torch

from . import _lib
from .functional import EPS, _check_map, _prep, _ptr, _stream, _workspace, device_guard

LabelArg = Union[str, torch.Tensor, np.ndarray]


def load_label_map(src: LabelArg, width: int, height: int, device) -> torch.Tensor:
    """Label map -> uint8 CUDA tensor [height, width].  Paths follow network/base.py:450:
    `np.asarray(Image.open(path).resize((W, H)))` with PIL's default filter."""
    if isinstance(src, torch.Tensor):
        lab = src
    elif isinstance(src, np.ndarray):
        lab = torch.from_numpy(np.ascontiguousarray(src))
    else:
        from PIL import Image
        lab = torch.from_numpy(np.asarray(Image.open(src).resize((width, height))).copy())
    if lab.dim() == 3 and lab.shape[0] == 1:
        lab = lab[0]
    assert lab.dim() == 2 and tuple(lab.shape) == (height, width), \
        f"label map {tuple(lab.shape)} does not match the feature resolution {(height, width)}"
    if lab.dtype != torch.uint8:
        assert int(lab.min()) >= 0 and int(lab.max()) <= 255, "label values must fit uint8"
        lab = lab.to(torch.uint8)
    return lab.to(device).contiguous()


def stack_label_maps(masks: Union[torch.Tensor, Sequence[LabelArg]], width: int, height: int, device) -> torch.Tensor:
    """Per-sample label maps (paths/arrays/tensors, see `load_label_map`), or a ready [N,H,W] tensor ->
    uint8 CUDA tensor [N, height, width]."""
    if isinstance(masks, torch.Tensor) and masks.dim() == 3:
        return masks.to(device, torch.uint8).contiguous()
    return torch.stack([load_label_map(m, width, height, device) for m in masks], dim=0)


def _refuse_grad(*tensors) -> None:
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise NotImplementedError(
            "rpst: segment AdaIN has no backward pass (the reference only calls it from test() under "
            "torch.no_grad(), network/adain_rp.py:251-262); call it under torch.no_grad() or detach the inputs")


def _seg_adain_into(out, out_batch_stride, content_feat, style_feat, c_labels, s_labels, prev, content_map, style_map,
                    want_info):
    """Segment AdaIN of [N,C,Hc,Wc] features into `out`, whose plane (i, ch) starts at
    out.data_ptr() + (i*out_batch_stride + ch*Hc*Wc) floats; returns the label table or None."""
    c = _prep(content_feat, "content_feat")
    s = _prep(style_feat, "style_feat")
    n, ch, hc, wc = c.shape
    hs, ws_ = s.shape[2:]
    assert c_labels.dtype == torch.uint8 and s_labels.dtype == torch.uint8 and c_labels.is_cuda and s_labels.is_cuda
    assert tuple(c_labels.shape) == (n, hc, wc) and tuple(s_labels.shape) == (n, hs, ws_)
    cl, sl = c_labels.contiguous(), s_labels.contiguous()
    if prev is not None:
        assert prev.shape == c.shape
        prev = _prep(prev, "prev")
    cm, sm = _check_map(content_map, "content_map", n * ch), _check_map(style_map, "style_map", n * ch)
    info = torch.empty(n, 256, 3, dtype=torch.int32, device=c.device) if want_info else None
    L = _lib.lib()
    ws = _workspace(L.rpst_seg_adain_workspace_bytes(n, ch, hc * wc, hs * ws_), c.device)
    _lib.check(L.rpst_seg_adain_fwd_mapped(c.data_ptr(), s.data_ptr(), cl.data_ptr(), sl.data_ptr(), _ptr(prev),
                                           out.data_ptr(), n, ch, hc * wc, hs * ws_, out_batch_stride, EPS,
                                           _ptr(cm), _ptr(sm), _ptr(info), ws.data_ptr(), ws.numel(), _stream()))
    return info


@device_guard
def seg_adain_batch(content_feat: torch.Tensor, style_feat: torch.Tensor, c_labels: torch.Tensor,
                    s_labels: torch.Tensor, prev: Optional[torch.Tensor] = None, return_info: bool = False, *,
                    content_map: Optional[torch.Tensor] = None, style_map: Optional[torch.Tensor] = None):
    """Batched segment AdaIN.  content [N,C,Hc,Wc], style [N,C,Hs,Ws], labels uint8 [N,Hc,Wc] /
    [N,Hs,Ws].  `prev` (same shape as content) is added to the result in the same pass.
    With `return_info` also returns the [N,256,3] int32 table (cnt_c, cnt_s, usable).
    `content_map` / `style_map` (int32 [N*C] plane indices, as in `adain_mapped`) make output plane p read
    `content_feat.flatten(0,1)[content_map[p]]` / `style_feat.flatten(0,1)[style_map[p]]` without
    materialising the permuted tensors; labels, `prev` and the label table stay those of the output sample."""
    assert content_feat.dim() == 4 and style_feat.dim() == 4
    assert content_feat.shape[:2] == style_feat.shape[:2], "batch/channel mismatch"
    _refuse_grad(content_feat, style_feat, prev)
    out = torch.empty(content_feat.shape, dtype=torch.float32, device=content_feat.device)
    ch, hw = content_feat.shape[1], content_feat.shape[2] * content_feat.shape[3]
    info = _seg_adain_into(out, ch * hw, content_feat, style_feat, c_labels, s_labels, prev, content_map, style_map,
                           return_info)
    return (out, info) if return_info else out


@device_guard
def seg_adain_concat(prev: torch.Tensor, content_feat: torch.Tensor, style_feat: torch.Tensor, c_labels: torch.Tensor,
                     s_labels: torch.Tensor, *, content_map: Optional[torch.Tensor] = None,
                     style_map: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`torch.cat([prev, seg_adain_batch(content_feat, style_feat, c_labels, s_labels)], dim=1)` with the
    segment half written straight into the channel slice of the result (the masked branch of
    network/adain_rp.py:793, mirroring `adain_concat`).  Maps as in `seg_adain_batch`.  Segment AdaIN has no
    backward pass; a `prev` that requires grad keeps its gradient through an ordinary `torch.cat`."""
    assert content_feat.dim() == 4 and style_feat.dim() == 4
    assert content_feat.shape[:2] == style_feat.shape[:2], "batch/channel mismatch"
    assert prev.dim() == 4 and prev.shape[0] == content_feat.shape[0] and prev.shape[2:] == content_feat.shape[2:]
    _refuse_grad(content_feat, style_feat)
    if torch.is_grad_enabled() and prev.requires_grad:
        return torch.cat([prev, seg_adain_batch(content_feat, style_feat, c_labels, s_labels, content_map=content_map,
                                                style_map=style_map)], dim=1)
    n, cp = prev.shape[:2]
    cc, hw = content_feat.shape[1], content_feat.shape[2] * content_feat.shape[3]
    out = torch.empty((n, cp + cc) + tuple(content_feat.shape[2:]), dtype=torch.float32, device=content_feat.device)
    out[:, :cp].copy_(prev)
    _seg_adain_into(out[:, cp:], (cp + cc) * hw, content_feat, style_feat, c_labels, s_labels, None, content_map,
                    style_map, False)
    return out


@device_guard
def adaptive_instance_normalization_with_segment(content_feat: torch.Tensor, style_feat: torch.Tensor,
                                                 content_seg_path: LabelArg, style_seg_path: LabelArg) -> torch.Tensor:
    """Drop-in for network/base.py:494 — (1,c,hc,wc), (1,c,hs,ws), two label maps (paths, arrays or
    tensors) -> (1,c,hc,wc)."""
    assert content_feat.shape[0] == 1 and style_feat.shape[0] == 1
    hc, wc = content_feat.shape[2:]
    hs, ws = style_feat.shape[2:]
    cl = load_label_map(content_seg_path, wc, hc, content_feat.device)
    sl = load_label_map(style_seg_path, ws, hs, style_feat.device)
    return seg_adain_batch(content_feat, style_feat, cl[None], sl[None])


@device_guard
def do_mask_stylized(content_feat: torch.Tensor, style_feat: torch.Tensor, c_masks: Sequence[LabelArg],
                     s_masks: Sequence[LabelArg], prev: Optional[torch.Tensor] = None, *,
                     content_map: Optional[torch.Tensor] = None, style_map: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Replacement for the per-sample Python loop network/adain_rp.py:313-319: one launch for the
    whole batch.  `c_masks[i]` / `s_masks[i]` are per-sample label maps (paths/arrays/tensors), or a
    ready [N,H,W] uint8 tensor.  Plane maps as in `seg_adain_batch`."""
    hc, wc = content_feat.shape[2:]
    hs, ws = style_feat.shape[2:]
    dev = content_feat.device
    return seg_adain_batch(content_feat, style_feat, stack_label_maps(c_masks, wc, hc, dev),
                           stack_label_maps(s_masks, ws, hs, dev), prev, content_map=content_map, style_map=style_map)

"""Decode loops of the reference's multiscale networks with the blend fused into the transform.

The reference spells the multiscale blend as two ops, `stylized + AdaIN(c_l, s_l)`
(network/adain_rp.py:300-301); these replacements make it one kernel call (`adain_blend`).  They are
installed over `<Class>.decode` by `rpst.install()` and also usable directly (`multiscale_transform`)."""
from __future__ import annotations

from typing import List, Sequence

import torch

from . import functional as F
from . import segment as SEG


def multiscale_transform(content_feats: Sequence[torch.Tensor], style_feats: Sequence[torch.Tensor],
                         prevs: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    """The transform calls of `MultiScaleAdaINRPNet.decode` with the decoder convolutions factored
    out (features ordered shallow -> deep, `prevs[l]` = decoder state blended at level l); outputs
    ordered deep -> shallow.  This is the hot path bench.py times."""
    outs = [F.adaptive_instance_normalization(content_feats[-1], style_feats[-1])]
    for l in range(len(content_feats) - 2, -1, -1):
        outs.append(F.adain_blend(prevs[l], content_feats[l], style_feats[l]))
    return outs


def decode_multiscale(self, content_feats, style_feats, use_mask=False, c_mask_path=None, s_mask_path=None,
                      plane_maps=None):
    """MultiScaleAdaINRPNet.decode (network/adain_rp.py:286-302): top level plain (seg-)AdaIN, every
    shallower level `decoder(prev + (seg-)AdaIN(c_l, s_l))` with the add fused into the transform.
    `sort_by_weights` (:230-249, applied here when `self._sort`) and the channel `shuffle` of `test()`
    (:256-260, handed over as `plane_maps` by `test_multiscale`) become plane maps of the kernel call
    instead of permuted copies, in the masked (segment AdaIN) branch too.  Like the reference, content and
    style are sorted by the SAME attention weights (the ones the shared encoder stored last)."""
    levels = len(content_feats)
    maps = list(plane_maps) if plane_maps is not None else [None] * levels
    if self._sort:
        for idx, enc in enumerate(self.rp_shared_encoder):
            maps[idx] = F.compose_maps(maps[idx], F.sort_map(enc.attention_map))

    def level(l, prev):
        cf, sf = content_feats[l], style_feats[l]
        if use_mask:
            return SEG.do_mask_stylized(cf, sf, c_mask_path, s_mask_path, prev=prev, content_map=maps[l],
                                        style_map=maps[l])
        if maps[l] is not None:
            return F.adain_mapped(cf, sf, maps[l], maps[l], prev=prev)
        return F.adaptive_instance_normalization(cf, sf) if prev is None else F.adain_blend(prev, cf, sf)

    stylized = self.rp_decoder[0](level(levels - 1, None))
    for i, l in enumerate(range(levels - 2, -1, -1)):
        stylized = self.rp_decoder[i + 1](level(l, stylized))
    return stylized


def test_multiscale(self, content, style, iterations=0, bid=0, c_mask_path=None, s_mask_path=None):
    """MultiScaleAdaINRPNet.test (network/adain_rp.py:251-269) with `self.shuffle` (:304-311) turned
    into plane maps for the transform (levels above `_shuffle_layers` stay unshuffled)."""
    self.eval()
    with torch.no_grad():
        content_feats = self.encode_rp_intermediate(content)
        style_feats = self.encode_rp_intermediate(style)
        if getattr(type(self), "decode", decode_multiscale) is decode_multiscale:
            maps = None
            if self._shuffle:
                maps = [None if idx > self._shuffle_layers else
                        F.shuffle_map(c.shape[0], c.shape[1], 4, c.device) for idx, c in enumerate(content_feats)]
            stylized = decode_multiscale(self, content_feats, style_feats, use_mask=self.config['use_mask'],
                                         c_mask_path=c_mask_path, s_mask_path=s_mask_path, plane_maps=maps)
        else:
            # subclasses that inherit test() but bring their own decode loop (CCAM, MST, SELast, LDMS*): shuffle as
            # the reference does (:256-260) and hand over to THEIR decode
            if self._shuffle:
                content_feats = [self.shuffle(c, idx) for idx, c in enumerate(content_feats)]
                style_feats = [self.shuffle(s, idx) for idx, s in enumerate(style_feats)]
            stylized = self.decode(content_feats, style_feats, use_mask=self.config['use_mask'],
                                   c_mask_path=c_mask_path, s_mask_path=s_mask_path)
        self.train()
        return stylized


def _top(self, content_feats, style_feats, use_mask, c_mask_path, s_mask_path):
    if use_mask:
        return SEG.do_mask_stylized(content_feats[-1], style_feats[-1], c_mask_path, s_mask_path)
    return F.adaptive_instance_normalization(content_feats[-1], style_feats[-1])


def decode_ldms(self, content_feats, style_feats, use_mask=False, c_mask_path=None, s_mask_path=None):
    """LDMSAdaINRPNet.decode (network/adain_rp.py:538-553; inherited by LDMS 2/3): decoder blocks are
    attributes `rp_dec{i}`; lower levels use the running decoder state as content,
    `stylized + AdaIN(stylized, s_l)` (prev aliases content), only while `i < stylized_layers-1`."""
    stylized = self.rp_dec0(_top(self, content_feats, style_feats, use_mask, c_mask_path, s_mask_path))
    lower = list(zip(content_feats[:-1], style_feats[:-1]))[::-1]
    for i, (cf, sf) in enumerate(lower):
        if i < self.stylized_layers - 1:
            if use_mask:
                fused = SEG.do_mask_stylized(cf, sf, c_mask_path, s_mask_path, prev=stylized)
            else:
                fused = F.adain_blend(stylized, stylized, sf)
        else:
            fused = stylized + []   # the reference adds an empty list here (:543,552) and fails the same way
        stylized = getattr(self, f'rp_dec{i + 1}')(fused)
    return stylized


def decode_ld_concat(self, content_feats, style_feats, use_mask=False, c_mask_path=None, s_mask_path=None):
    """LDMSAdaINRPNet4.decode (network/adain_rp.py:780-799, inherited by LDMS 5):
    `cat([stylized, (seg-)AdaIN(c_l, s_l)], 1)` with the AdaIN half written straight into the result."""
    stylized = self.rp_dec0(_top(self, content_feats, style_feats, use_mask, c_mask_path, s_mask_path))
    lower = list(zip(content_feats[:-1], style_feats[:-1]))[::-1]
    for i, (cf, sf) in enumerate(lower):
        if use_mask:
            hc, wc = cf.shape[2:]
            hs, ws = sf.shape[2:]
            fused = SEG.seg_adain_concat(stylized, cf, sf, SEG.stack_label_maps(c_mask_path, wc, hc, cf.device),
                                         SEG.stack_label_maps(s_mask_path, ws, hs, sf.device))
        else:
            fused = F.adain_concat(stylized, cf, sf)
        stylized = getattr(self, f'rp_dec{i + 1}')(fused)
    return stylized


PATCHED_TESTS = {"MultiScaleAdaINRPNet": test_multiscale}

PATCHED_DECODES = {
    "MultiScaleAdaINRPNet": decode_multiscale,
    "LDMSAdaINRPNet": decode_ldms,
    "LDMSAdaINRPNet4": decode_ld_concat,
}

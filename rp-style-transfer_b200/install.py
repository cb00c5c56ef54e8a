"""Drop-in installation into an already-imported reference tree.

`install()` rebinds the reference's transform functions, modules and methods to the rpst
implementations inside every `network.*` module.  The reference binds aliases at import time
(`AdaIN`, `AdaINSeg` in network/adain_rp.py:3-4, network/wct_rp.py:2, network/seg_adain_rp.py:3) and
star-imports network.base everywhere, so each namespace is patched, not just `network.base`
(SURVEY.md §7).  `uninstall()` restores the originals."""
from __future__ import annotations

import functools
import sys
from typing import Dict, List, Tuple

from . import functional as F
from . import losses as LOSS
from . import modules as M
from . import mrf as MRF
from . import sanet as SA
from . import segment as SEG
from . import wct as WCT
from .decode import PATCHED_DECODES, PATCHED_TESTS, SEGMENT_GRAD_DECODES

# reference name -> replacement (applied wherever the name exists in a network.* namespace)
NAME_MAP = {
    "calc_mean_std": F.calc_mean_std,
    "adaptive_instance_normalization": F.adaptive_instance_normalization,
    "AdaIN": F.adaptive_instance_normalization,
    "adaptive_instance_normalization_with_segment": SEG.adaptive_instance_normalization_with_segment,
    "AdaINSeg": SEG.adaptive_instance_normalization_with_segment,
    "mean_variance_norm": F.mean_variance_norm,
    "cal_dist": MRF.cal_dist,
    "cal_affinity_map": MRF.cal_affinity_map,
    "cal_affinity_matrix": SA.cal_affinity_matrix,
    "matrix_sqrt": WCT.matrix_sqrt,
    "matrix_inv_sqrt": WCT.matrix_inv_sqrt,
    "MRFLoss": MRF.MRFLoss,
    "SELayer": M.SELayer,
    "SANet": SA.SANet,
    "AdaptiveSANet": SA.AdaptiveSANet,
    "Transform": SA.Transform,
    "AdaptiveTransform": SA.AdaptiveTransform,
    "AEAModule": SA.AEAModule,
    "AEALReluModule": SA.AEALReluModule,
}

_saved: List[Tuple[object, str, object]] = []


def _patch(obj, name, value):
    _saved.append((obj, name, getattr(obj, name)))
    setattr(obj, name, value)


def install(package: str = "network", segment_grad: bool = False) -> Dict[str, int]:
    """Patch every imported `<package>.*` module; returns {name: number of namespaces patched}.
    `segment_grad=True` makes segment AdaIN differentiable wherever it is patched in (`AdaINSeg`,
    `do_mask_stylized` and the masked branches of the decodes), so masked training loops run under autograd."""
    if _saved:
        return {}
    counts: Dict[str, int] = {}
    name_map = NAME_MAP
    decodes = PATCHED_DECODES
    if segment_grad:
        seg = functools.partial(SEG.adaptive_instance_normalization_with_segment, differentiable=True)
        name_map = dict(NAME_MAP, adaptive_instance_normalization_with_segment=seg, AdaINSeg=seg)
        decodes = SEGMENT_GRAD_DECODES
    mods = [m for n, m in list(sys.modules.items()) if m is not None and (n == package or n.startswith(package + "."))]
    if not mods:
        raise RuntimeError(f"rpst.install: package '{package}' is not imported")
    for mod in mods:
        for name, repl in name_map.items():
            if name in vars(mod) and vars(mod)[name] is not repl:
                _patch(mod, name, repl)
                counts[name] = counts.get(name, 0) + 1
    # bound methods: WCT fuse / whiten_and_color and the decode loops that spell the blend as two ops
    seen = set()
    for mod in mods:
        for cname, cls in list(vars(mod).items()):
            if not isinstance(cls, type) or id(cls) in seen:
                continue
            seen.add(id(cls))
            if cname == "WCTRPNet" or any(b.__name__ == "WCTRPNet" for b in cls.__mro__):
                if "fuse" in vars(cls):
                    _patch(cls, "fuse", WCT.fuse)
                    counts["WCTRPNet.fuse"] = counts.get("WCTRPNet.fuse", 0) + 1
                if "whiten_and_color" in vars(cls):
                    _patch(cls, "whiten_and_color", lambda self, cF, sF, method="closed-form": WCT.whiten_and_color(cF, sF, method))
                    counts["WCTRPNet.whiten_and_color"] = counts.get("WCTRPNet.whiten_and_color", 0) + 1
            if cname in decodes and "decode" in vars(cls):
                _patch(cls, "decode", decodes[cname])
                counts[cname + ".decode"] = 1
            if cname in PATCHED_TESTS and "test" in vars(cls):
                _patch(cls, "test", PATCHED_TESTS[cname])
                counts[cname + ".test"] = 1
            # loss statistics (SURVEY.md §8f rank 1): methods that only use self.mse_loss
            if "calc_style_loss" in vars(cls):
                _patch(cls, "calc_style_loss", lambda self, input, target: LOSS.calc_style_loss(input, target))
                counts["calc_style_loss"] = counts.get("calc_style_loss", 0) + 1
            if "calc_content_loss" in vars(cls):
                _patch(cls, "calc_content_loss",
                       lambda self, input, target, norm=False: LOSS.calc_content_loss(input, target, norm))
                counts["calc_content_loss"] = counts.get("calc_content_loss", 0) + 1
            if "do_mask_stylized" in vars(cls):
                _patch(cls, "do_mask_stylized",
                       lambda self, cf, sf, cm, sm: SEG.do_mask_stylized(cf, sf, cm, sm, differentiable=segment_grad))
                counts["do_mask_stylized"] = counts.get("do_mask_stylized", 0) + 1
    return counts


def uninstall() -> None:
    while _saved:
        obj, name, value = _saved.pop()
        setattr(obj, name, value)

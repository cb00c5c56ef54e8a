"""Drop-in installation into the real reference tree (no GPU, so only the rebinding is checked — the numerics
of every replacement are covered by the -m gpu tests).  All but the state-dict test need the reference tree
itself (RPST_REFERENCE_ROOT) and skip without it."""
import sys

import pytest

from oracle.reference_loader import load_reference, reference_available

needs_reference = pytest.mark.skipif(not reference_available(), reason="reference tree not found (RPST_REFERENCE_ROOT)")


@pytest.mark.reference
@needs_reference
def test_install_rebinds_every_namespace_and_restores():
    import rpst
    net = load_reference()
    base, adain_rp, wct_rp, sanet, mrf_rp = (sys.modules[f"network.{n}"] for n in ("base", "adain_rp", "wct_rp", "sanet", "mrf_rp"))
    orig_adain = base.adaptive_instance_normalization
    orig_decode = adain_rp.MultiScaleAdaINRPNet.decode
    counts = rpst.install()
    try:
        # import-time aliases in three modules (network/adain_rp.py:3-4, wct_rp.py:2, seg_adain_rp.py:3)
        assert adain_rp.AdaIN is rpst.adaptive_instance_normalization
        assert wct_rp.AdaIN is rpst.adaptive_instance_normalization
        assert sys.modules["network.seg_adain_rp"].AdaIN is rpst.adaptive_instance_normalization
        assert adain_rp.AdaINSeg is rpst.adaptive_instance_normalization_with_segment
        assert counts["calc_mean_std"] >= 6 and counts["AdaIN"] >= 3
        for mod in (base, adain_rp, wct_rp, sanet, mrf_rp):
            assert mod.calc_mean_std is rpst.calc_mean_std
        assert sanet.SANet is rpst.SANet and sanet.Transform is rpst.Transform
        assert sanet.mean_variance_norm is rpst.mean_variance_norm
        assert mrf_rp.MRFLoss is rpst.MRFLoss and base.cal_dist is rpst.cal_dist
        assert wct_rp.matrix_sqrt is rpst.matrix_sqrt
        assert wct_rp.WCTRPNet.fuse is not None and "WCTRPNet.fuse" in counts
        assert adain_rp.MultiScaleAdaINRPNet.decode is not orig_decode
        assert adain_rp.LDMSAdaINRPNet2.decode is adain_rp.LDMSAdaINRPNet.decode     # inherited patch
        assert net.SELayer is rpst.SELayer or sys.modules["network.attention"].SELayer is rpst.SELayer
        # loss-statistics methods (SURVEY.md §8f rank 1) on every class that defines them
        assert counts["calc_style_loss"] >= 3 and counts["calc_content_loss"] >= 3
        assert adain_rp.AdaINRPNet.calc_style_loss is not None
        import inspect
        assert "norm" in inspect.signature(sanet.SAModel.calc_content_loss).parameters
        assert rpst.install() == {}                                                # idempotent
    finally:
        rpst.uninstall()
    assert base.adaptive_instance_normalization is orig_adain
    assert adain_rp.MultiScaleAdaINRPNet.decode is orig_decode


def test_state_dict_names_match_reference(golden):
    """Key names, order and shapes of the reference's own modules as oracle/gen_golden.py recorded them
    (SANet / Transform / AdaptiveSANet / AdaptiveTransform at 16 planes, both clamp modules; SELayer(32)'s
    fc[0] / fc[2] weights): reference checkpoints load unchanged."""
    import torch
    import rpst
    g = golden("sanet")
    torch.manual_seed(0)
    cases = [(rpst.SANet(16), "sanet."), (rpst.Transform(16), "transform.")]
    for mode in ("aea", "relu"):
        cases += [(rpst.AdaptiveSANet(16, 64, ada_module=mode), f"ada_{mode}."),
                  (rpst.AdaptiveTransform(16, 64, 16, ada_module=mode), f"adatr_{mode}.")]
    se = golden("se")
    cases.append((rpst.SELayer(32, reduction=16), {"fc.0.weight": se["w1"], "fc.2.weight": se["w2"]}))
    for ours, theirs in cases:
        if isinstance(theirs, str):
            theirs = {k[len(theirs):]: v for k, v in g.items() if k.startswith(theirs)}
        a = ours.state_dict()
        assert list(a.keys()) == list(theirs.keys())
        assert all(a[k].shape == theirs[k].shape for k in a)
        ours.load_state_dict(theirs)   # reference checkpoints load unchanged


@pytest.mark.reference
@needs_reference
def test_patched_test_respects_subclass_decode():
    """CCAM / MST / SELast / LDMS* inherit MultiScaleAdaINRPNet.test() but define their own decode(): the patched
    test() must shuffle like the reference and call THEIR decode, not the fused multiscale one."""
    import torch
    import rpst
    load_reference()
    adain_rp = sys.modules["network.adain_rp"]
    rpst.install()
    try:
        calls = {}

        class Sub(adain_rp.SELastMultiScaleAdaINRPNet):
            def __init__(self):                       # bypass the heavy constructor
                torch.nn.Module.__init__(self)
                self._shuffle, self._shuffle_layers, self._sort = True, 0, False
                self.config = {"use_mask": False}

            def encode_rp_intermediate(self, x):
                return [x, x * 2]

            def decode(self, content_feats, style_feats, use_mask=False, c_mask_path=None, s_mask_path=None):
                calls["feats"] = content_feats
                return content_feats[0]

        assert adain_rp.SELastMultiScaleAdaINRPNet.test is adain_rp.MultiScaleAdaINRPNet.test   # inherited, patched
        x = torch.arange(2 * 8 * 2 * 2, dtype=torch.float32).view(2, 8, 2, 2)
        out = Sub().test(x, x)
        want0 = x.view(2, 4, 2, 2, 2).permute(0, 2, 1, 3, 4).contiguous().view(2, 8, 2, 2)    # level 0 shuffled (:304-311)
        assert torch.equal(calls["feats"][0], want0) and torch.equal(calls["feats"][1], x * 2)  # level 1 > _shuffle_layers
        assert torch.equal(out, want0)
    finally:
        rpst.uninstall()


@pytest.mark.reference
@needs_reference
def test_label_map_loader_matches_the_reference_png_path(tmp_path):
    """`test.py` hands PNG paths to the segment transform; the reference reads and resizes them with PIL
    (network/base.py:448-449).  The rpst loader must produce the same label maps, and the validity table the
    reference derives from them (`compute_label_info`, :421-439) must match the oracle's rule."""
    import numpy as np
    import torch
    from PIL import Image
    import rpst
    from oracle import restate as R
    load_reference()
    base = sys.modules["network.base"]
    rng = np.random.default_rng(0)
    big_c = np.kron(rng.integers(0, 5, (6, 8)), np.ones((16, 16))).astype(np.uint8)     # 96 x 128 blocky map
    big_s = np.kron(rng.integers(0, 5, (5, 7)), np.ones((16, 16))).astype(np.uint8)     # 80 x 112
    cp, sp = str(tmp_path / "c.png"), str(tmp_path / "s.png")
    Image.fromarray(big_c).save(cp)
    Image.fromarray(big_s).save(sp)
    (wc, hc), (ws, hs) = (32, 24), (28, 20)                                              # feature resolutions (W, H)
    c_seg, s_seg, label_set, label_indicator = base.get_segment_and_info(cp, sp, (wc, hc), (ws, hs))
    got_c = rpst.load_label_map(cp, wc, hc, "cpu")
    got_s = rpst.load_label_map(sp, ws, hs, "cpu")
    assert got_c.dtype == torch.uint8 and tuple(got_c.shape) == (hc, wc)
    assert np.array_equal(got_c.numpy(), c_seg) and np.array_equal(got_s.numpy(), s_seg)
    valid = R.segment_label_validity(got_c, got_s)
    for lab in label_set:
        assert bool(label_indicator[lab]) == valid[int(lab)], lab

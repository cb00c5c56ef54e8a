"""rpst — B200-native stylization transform for RP-Style-Transfer (hot path only, see DESIGN.md).

`import rpst` works through the alias package at the repo root; this directory is the product.
Everything here calls hand-written sm_100a kernels through the C ABI in include/rpst.h."""
from . import _lib
from ._lib import RpstError, get_tuning, set_tuning
from .functional import (adain_blend, adain_concat, adain_mapped, adaptive_instance_normalization, calc_mean_std,
                         compose_maps, mean_variance_norm, plane_affine, shuffle_map, sort_map)

from . import losses
from .losses import calc_content_loss, calc_style_loss
from .modules import CCAMDec, SELayer, ccam_attention
from .mrf import MRFLoss, cal_affinity_map, cal_dist, mrf_match, packed_gemm
from .wct import matrix_inv_sqrt, matrix_sqrt, spd_roots, wct_fuse, whiten_and_color
from .sanet import (AdaptiveSANet, AdaptiveTransform, AEALReluModule, AEAModule, SANet, Transform, attention_core,
                    cal_affinity_matrix)
from .segment import (adaptive_instance_normalization_with_segment, do_mask_stylized, load_label_map, seg_adain_batch,
                      seg_adain_concat)

from .conv import adain_from_stats, conv1x1
from .decode import multiscale_transform
from .install import install, uninstall

AdaIN = adaptive_instance_normalization
AdaINSeg = adaptive_instance_normalization_with_segment


def version() -> int:
    return int(_lib.lib().rpst_version())

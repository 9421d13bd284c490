"""ups_b200 — B200-native (sm_100a) implementation of the per-step part-disentanglement hot
path of CompVis/unsupervised-part-segmentation, behind the reference's helper signatures.

    from ups_b200 import nn, model, tps, pooling       # reference-named helpers
    from ups_b200.step import PartStep                 # the fused forward+backward step
"""
from . import _cabi, ops, nn, tps, model, pooling, configs  # noqa: F401
from .configs import PathConfig  # noqa: F401
from .nn import (softmax, spatial_softmax, hard_max, straight_through_estimator,  # noqa: F401
                 hard_max_straight_through, apply_partwise, mask2hotmask, unpool_features_gathered,
                 probs_to_mu_sigma, mumford_shah, mumford_shah_sums, edge_set, MeanFieldDistribution, mask2rgb)
from .model import (mask_parts, encode_parts, unpool_features, inject_features, make_tps,  # noqa: F401
                    categorical_kl, weak_cross_entropy, images_from_uint8, inject_conv2d, decode_conv2d,
                    parts_conv2d, encode_conv2d)
from .pooling import pool_features, pool_unpool_block, get_features, part_mean_pool  # noqa: F401
from .tps import tps_parameters, make_input_tps_param, ThinPlateSpline  # noqa: F401

__version__ = "0.1.0"

"""Shared helpers for the parity tests: build an engine + oracle pair from one config and one parameter set."""
import numpy as np
import torch

from oracle import ecnf_oracle as O
from ecnf_b200.engine import CnfConfig, Engine


def make_pair(n, dim, blocks, units, H, T=8, n_features=1, sigma_min=0.01, base_scale=1.0, seed=0,
              head_variance=1.0, bias_std=0.1, zero_time=False, normalization_constant=1.0):
    ocfg = O.CnfConfig(n_frames=n, dim=dim, sigma_min=sigma_min, base_scale=base_scale, n_blocks_egnn=blocks,
                       mlp_units=tuple(units), n_invariant_feat_hidden=H, time_embedding_dim=T,
                       n_features=n_features, normalization_constant=normalization_constant)
    flat = O.init_params(ocfg, seed=seed, head_variance=head_variance, bias_std=bias_std)
    flat["EGNN_0/final_scaling"] = np.asarray(1.25, np.float32)
    if zero_time:   # autonomous, smooth-in-t field: the adaptive step sequence is then not chaotic
        for b in range(blocks):
            flat[f"EGNN_0/Dense_{b}/kernel"][H:] = 0.0
    tree = O.flat_to_nested(flat)
    ecfg = CnfConfig(n, dim, sigma_min, base_scale, blocks, tuple(units), H, T, n_features, normalization_constant)
    return ocfg, flat, tree, ecfg


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


CASES = {
    # name: (n, dim, blocks, units, H, n_features)
    "small_64_32": (5, 3, 2, (64, 64), 32, 3),
    "dw4": (4, 2, 3, (128, 128, 128), 64, 1),
    "lj13": (13, 3, 3, (128, 128, 128), 64, 1),
    "one_block": (6, 3, 1, (64, 64), 32, 1),
    "qm9_like": (7, 3, 2, (256, 256), 32, 1),
}

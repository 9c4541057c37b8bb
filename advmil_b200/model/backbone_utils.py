"""Layer library: parameter containers whose names/shapes match the reference's state_dict
(model/backbone_utils.py) plus the host-side index helpers.  The containers do not run arithmetic layer by layer;
the fused CUDA path reads their parameters (see ABMIL / EmbedXLayer / Generator / PrjDiscriminator).
"""
from __future__ import annotations

import torch
import torch.nn as nn


class Attn_Net_Gated(nn.Module):
    """Gated attention scorer (reference model/backbone_utils.py:11-29): parameters attention_a.0, attention_b.0,
    attention_c.  forward() returns (scores [N, n_classes], x) through the fused gate kernel."""

    def __init__(self, L=1024, D=256, dropout=False, n_classes=1):
        super().__init__()
        a = [nn.Linear(L, D), nn.Tanh()]
        b = [nn.Linear(L, D), nn.Sigmoid()]
        if dropout:
            a.append(nn.Dropout(0.25))
            b.append(nn.Dropout(0.25))
        self.attention_a = nn.Sequential(*a)
        self.attention_b = nn.Sequential(*b)
        self.attention_c = nn.Linear(D, n_classes)
        self.has_dropout = bool(dropout)
        assert n_classes == 1, "the fused gate kernel scores one class (the reference always uses n_classes=1)"

    def forward(self, x):
        from .. import ops, get_precision
        from ..utils.func import next_dropout_seed
        train = self.training and self.has_dropout
        s, _ = ops.gated_score_forward(x, self.attention_a[0].weight, self.attention_a[0].bias, self.attention_b[0].weight,
                                       self.attention_b[0].bias, self.attention_c.weight.reshape(-1), self.attention_c.bias,
                                       p_drop=0.25 if train else 0.0, seed=next_dropout_seed() if train else 0,
                                       train=train, precision=ops.PRECISIONS[get_precision()], save=False)
        return s.unsqueeze(-1), x  # inference-only entry point; training goes through the fused backbones


class GAPool(nn.Module):
    """Global attention pooling container (reference model/backbone_utils.py:31-56): fc1.0, score.0, fc2."""

    def __init__(self, in_dim, hid_dim, dropout=0.25):
        super().__init__()
        self.fc1 = nn.Sequential(nn.Linear(in_dim, hid_dim), nn.Tanh(), nn.Dropout(dropout))
        self.score = nn.Sequential(nn.Linear(in_dim, hid_dim), nn.Sigmoid(), nn.Dropout(dropout))
        self.fc2 = nn.Linear(hid_dim, 1)
        self.p = dropout


def sequence2square_index(n_rows: int, s: int = 4) -> torch.Tensor:
    """Index form of sequence2square (reference model/backbone_utils.py:62-69): row n -> (region n // s^2,
    grid row (n % s^2) // s, grid col n % s).  Asserts N % s^2 == 0 like the reference (:65)."""
    assert n_rows % (s * s) == 0
    n = torch.arange(n_rows)
    return torch.stack([n // (s * s), (n % (s * s)) // s, n % s], dim=1)


class AVGPoolPatchEmbedding(nn.Module):
    """Patch embedding container (reference model/backbone_utils.py:129-168): conv, norm, ReLU, 4x4 average pool.  The
    fused kernels cover what the AdvMIL configs reach: scale 4, stride 1, no depth-wise conv, and ksize 1 (per-patch linear,
    config/cfg_nlst.yaml:41-42) or 3 (3x3 convolution over each region's 4x4 grid of patches, zero padded at its border;
    the reference class's default, disc_netx_ksize: 3)."""

    def __init__(self, in_dim, out_dim, scale: int = 4, dw_conv=False, ksize=3, stride=1):
        super().__init__()
        assert scale == 4, "It only supports for scale = 4"
        assert ksize == 1 or ksize == 3, "It only supports for ksize = 1 or 3"
        if stride != 1 or dw_conv:
            raise NotImplementedError("advmil_b200 fuses the stride-1, non-depth-wise patch embedding only")
        self.scale, self.stride = scale, stride
        self.conv = nn.Conv2d(in_dim, out_dim, ksize, stride, padding=(ksize - 1) // 2)
        self.pool = nn.AdaptiveAvgPool2d(1)
        self.norm = nn.LayerNorm(out_dim)
        self.act = nn.ReLU(inplace=True)

    def forward(self, x):
        """x [1,N,C] -> [1,N/16,C'] (inference-only entry point; training goes through PrjDiscriminator)."""
        from .. import ops, get_precision
        bags = ops.PackedBags.from_single(x)
        cfg = ops.DiscConfig(C=self.conv.in_channels, d=self.conv.out_channels, t1=1, t2=self.conv.out_channels,
                             ln_eps=self.norm.eps, ksize=self.conv.kernel_size[0])
        params = [self.conv.weight, self.conv.bias, self.norm.weight, self.norm.bias] + [None] * 20
        acts = ops.disc_embed_forward(cfg, params, bags, ops.PRECISIONS[get_precision()], save=False)
        return acts["emb"].unsqueeze(0)


def make_embedding_layer(backbone: str, args):
    if backbone == "avgpool":
        return AVGPoolPatchEmbedding(args.in_dim, args.out_dim, args.scale, args.dw_conv, args.ksize)
    if backbone == "gapool":
        raise NotImplementedError("gapool patch embedding is outside the AdvMIL hot path (disc_netx_backbone: avgpool)")
    raise NotImplementedError(f"{backbone} has not implemented.")


def make_transformer_layer(backbone: str, args):
    """[B, N, C] --Transformer--> [B, N, C] (reference model/backbone_utils.py:112-127).  The returned nn.TransformerEncoder
    is a parameter container (same state_dict names and default initialisation as the reference's); DualTrans_HS runs its
    arithmetic in the fused CUDA path."""
    if backbone == "Transformer":
        layer = nn.TransformerEncoderLayer(args.d_model, args.nhead, dim_feedforward=args.d_model, dropout=args.dropout,
                                           activation="relu", batch_first=True)
        return nn.TransformerEncoder(layer, num_layers=args.num_layers)
    if backbone == "Identity":
        return nn.Identity()
    raise NotImplementedError(f"{backbone} has not implemented.")

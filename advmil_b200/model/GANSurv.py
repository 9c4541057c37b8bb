"""Generator and projection discriminator with the reference's module surface (model/GANSurv.py), executed by the
fused sm_100a kernels behind the C ABI.  `forward` keeps the reference's single-bag signature; `forward_packed`
is the same computation over packed variable-length bags (one launch sequence for the whole step).
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
import torch.nn as nn

from .. import get_precision, ops
from ..utils.func import generate_noise, next_dropout_seed
from .model_utils import EmbedXLayer, make_embedding_y_layer, make_noise_mlp_layer

_OUT_SCALE = {"sigmoid": 1, "exp": 2}


class Generator(nn.Module):
    """G(X, noise) -> t_hat: MIL backbone + noise-concat MLP head (reference model/GANSurv.py:13-49)."""

    def __init__(self, dim_in, dim_out, backbone: nn.Module, args_noise, norm=False, dropout=0.25, out_scale: str = "sigmoid"):
        super().__init__()
        self.noise = args_noise.noise
        self.hops = args_noise.hops
        self.noise_dist = "uniform" if args_noise.noise_dist is None else args_noise.noise_dist
        assert len(self.noise) == self.hops + 1
        if self.hops != 1 or dim_out != 1 or norm:
            raise NotImplementedError("the fused generator head covers hops=1, dim_out=1, norm=False (config/cfg_nlst.yaml:29-33)")
        self.MLPs = make_noise_mlp_layer(dim_in, dim_out, self.noise, hops=self.hops, norm=norm, dropout=dropout)
        self.backbone = backbone
        self.out_scale = out_scale
        self.dim_in, self.p_head = dim_in, dropout

    # -- plumbing ---------------------------------------------------------------------------------
    def config(self) -> ops.GenConfig:
        return self.backbone.config(hid=self.MLPs[0][0].out_features, noise=(int(self.noise[0] == 1), int(self.noise[1] == 1)),
                                    out_scale=_OUT_SCALE.get(self.out_scale, 0), p_head=self.p_head)

    def gen_params(self):
        if self.backbone.kind == "patch":
            return [None] * 10 + self.head_params()
        return self.backbone.gen_params(self.MLPs)

    def head_params(self):
        return [self.MLPs[0][0].weight, self.MLPs[0][0].bias, self.MLPs[1][0].weight, self.MLPs[1][0].bias]

    def draw_noise(self, n_bags: int, device, zero_noise: bool, generator=None):
        """Noise tensors in the order Generator.forward draws them (reference :33-38): one per layer with flag 1,
        from the CPU generator (utils/func.py:154-164; `generator`: a private CPU generator instead of the default
        one, used per rank under data parallelism).  zero_noise -> None (the kernels read zeros)."""
        widths = [self.dim_in, self.MLPs[0][0].out_features]
        out = []
        for i in range(2):
            if self.noise[i] == 1 and not zero_noise:
                out.append(generate_noise(n_bags, widths[i], to_device=device, distribution=self.noise_dist, generator=generator))
            else:
                out.append(None)
        return out

    # -- reference surface ------------------------------------------------------------------------
    def forward(self, x, x_ext, zero_noise=False):
        """x [1,N,C]; x_ext ignored for ABMIL, cluster ids for DeepAttMISL, region coordinates (or None) for ESAT -> [1,1]."""
        if self.backbone.kind == "patch":
            return self.forward_packed(ops.PackedBags.from_single(x), zero_noise=zero_noise, coord=x_ext)
        if self.backbone.kind == "cluster":
            hc = self.backbone.cluster_rows(x, x_ext)
            # the attention stage sees num_clusters rows per bag: always the exact fp32 engine
            return self.forward_packed(ops.PackedBags(hc, [self.backbone.num_clusters]), zero_noise=zero_noise, x_grad=hc,
                                       precision=ops.FP32)
        return self.forward_packed(ops.PackedBags.from_single(x), zero_noise=zero_noise)

    def forward_packed(self, bags: ops.PackedBags, noise: Optional[Sequence[Optional[torch.Tensor]]] = None,
                       zero_noise: bool = False, x_grad: Optional[torch.Tensor] = None,
                       precision: Optional[int] = None, coord=None, reuse_embedding=None, acts_sink=None) -> torch.Tensor:
        """Packed bags -> [bags, 1].  reuse_embedding (ESAT): activations of an earlier forward over the same bags,
        coordinates and embedding parameters whose patch embedding is shared; acts_sink (ESAT): a list that receives this
        forward's activation dict (what a later call passes as reuse_embedding)."""
        precision = ops.PRECISIONS[get_precision()] if precision is None else precision
        n0, n1 = noise if noise is not None else self.draw_noise(bags.bags, bags.x.device, zero_noise)
        train = self.training
        if self.backbone.kind == "patch":
            bb = self.backbone
            masks = getattr(self, "_inject_masks", None) if train else None
            pe = None if reuse_embedding is not None else bb.positional(bags, coord)
            pred = ops.EsatFn.apply(bb.esat_config(), self.config(), bags, pe, n0, n1, train, next_dropout_seed() if train else 0,
                                    masks, precision, reuse_embedding, acts_sink, *bb.esat_params(), *self.head_params())
            return pred.unsqueeze(-1)
        from .. import library
        seed, masks = next_dropout_seed() if train else 0, getattr(self, "_inject_masks", None)
        if library.should_dispatch(bags.x):
            # registered operator advmil_b200::generator_fwd (torch.library: CUDA impl over the C ABI, fake impl, autograd)
            pred = library.generator(self.config(), bags, n0, n1, train, seed, masks, precision, self.gen_params(), x_grad=x_grad)
        else:
            pred = ops.GeneratorFn.apply(self.config(), bags, x_grad, n0, n1, train, seed, masks, precision, *self.gen_params())
        return pred.unsqueeze(-1)


class PrjDiscriminator(nn.Module):
    """D(X, t): region-level instance projection discriminator (reference model/GANSurv.py:71-105)."""

    def __init__(self, args_netx, args_nety, prj_path="x", inner_product="bag"):
        super().__init__()
        assert inner_product in ["bag", "instance"]
        self.inner_product = inner_product
        self.net_pair_one = EmbedXLayer(args_netx)
        self.net_pair_two = make_embedding_y_layer(args_nety)
        dim_x, dim_y = args_netx.out_dim, args_nety.hid_dims[-1]
        if len(args_nety.hid_dims) != 2 or args_nety.norm or args_nety.dropout or args_nety.in_dim != 1 or dim_x != dim_y:
            raise NotImplementedError("the fused RLIP head covers disc_nety: in_dim 1, two hidden dims, no norm/dropout, "
                                      "last dim == disc_netx_out_dim (config/cfg_nlst.yaml:44-47)")
        self.prj_path = prj_path
        if prj_path == "x":
            self.prj_layer = nn.Linear(dim_x, 1)
        elif prj_path == "y":
            self.prj_layer = nn.Linear(dim_y, 1)
        else:
            self.prj_layer = None
        self.dims = (args_netx.in_dim, dim_x, args_nety.hid_dims[0], dim_y)
        print("[info] Discriminator is with projection: {}".format(self.prj_path))

    def config(self) -> ops.DiscConfig:
        C, d, t1, t2 = self.dims
        return ops.DiscConfig(C=C, d=d, t1=t1, t2=t2, inner_instance=int(self.inner_product == "instance"),
                              prj_path={"x": 1, "y": 2}.get(self.prj_path, 0), p=self.net_pair_one.p,
                              ln_eps=self.net_pair_one.embedding.norm.eps, ksize=self.net_pair_one.embedding.conv.kernel_size[0])

    def disc_params(self):
        y = self.net_pair_two
        pr = self.prj_layer
        return self.net_pair_one.disc_params() + [y[0][0].weight, y[0][0].bias, y[1][0].weight, y[1][0].bias,
                                                  None if pr is None else pr.weight, None if pr is None else pr.bias]

    def forward(self, x, t):
        """x [1,N,C] (N % 16 == 0), t [1,1] -> [1,1]."""
        return self.forward_packed(ops.PackedBags.from_single(x), t)

    def forward_packed(self, bags: ops.PackedBags, t: torch.Tensor) -> torch.Tensor:
        train = self.training
        from .. import library
        seed, masks = next_dropout_seed() if train else 0, getattr(self, "_inject_masks", None)
        if library.should_dispatch(bags.x):
            # registered operator advmil_b200::discriminator_fwd (torch.library: CUDA impl over the C ABI, fake impl, autograd)
            out = library.discriminator(self.config(), bags, t.reshape(-1), train, seed, masks, ops.PRECISIONS[get_precision()], self.disc_params())
        else:
            out = ops.DiscriminatorFn.apply(self.config(), bags, t.reshape(-1), train, seed, masks, ops.PRECISIONS[get_precision()],
                                            *self.disc_params())
        return out.unsqueeze(-1)

    def embed_packed(self, bags: ops.PackedBags) -> torch.Tensor:
        """Region embedding [rows/16, d] of packed bags (net_pair_one.embedding) as its own autograd node: the embedding has
        no dropout, so the real and the fake pairs of a D step share it (`head_packed`)."""
        return ops.DiscEmbedFn.apply(self.config(), bags, ops.PRECISIONS[get_precision()], *self.disc_params())

    def head_packed(self, bags: ops.PackedBags, emb: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        """D(x, t) from a precomputed region embedding -> [bags, 1]."""
        train = self.training
        out = ops.DiscHeadFn.apply(self.config(), bags, emb, t.reshape(-1), train, next_dropout_seed() if train else 0,
                                   getattr(self, "_inject_masks", None), ops.PRECISIONS[get_precision()], *self.disc_params())
        return out.unsqueeze(-1)


class Discriminator(PrjDiscriminator):
    """Concat discriminator (reference model/GANSurv.py:52-68): out = fc(cat[EmbedX(x), time_embed(t)]).  Same fused RLIP
    embedding / head kernels as PrjDiscriminator; only the per-bag tail differs (C ABI prj_path 3)."""

    def __init__(self, args_netx, args_nety, **kws):
        nn.Module.__init__(self)
        self.inner_product = "bag"
        self.net_pair_one = EmbedXLayer(args_netx)
        self.net_pair_two = make_embedding_y_layer(args_nety)
        dim_x, dim_y = args_netx.out_dim, args_nety.hid_dims[-1]
        if len(args_nety.hid_dims) != 2 or args_nety.norm or args_nety.dropout or args_nety.in_dim != 1 or dim_x != dim_y:
            raise NotImplementedError("the fused RLIP head covers disc_nety: in_dim 1, two hidden dims, no norm/dropout, "
                                      "last dim == disc_netx_out_dim (config/cfg_nlst.yaml:44-47)")
        self.prj_path = "cat"
        self.fc = nn.Linear(dim_x + dim_y, 1)
        self.dims = (args_netx.in_dim, dim_x, args_nety.hid_dims[0], dim_y)
        print("[info] Typical discriminator without projection")

    def config(self) -> ops.DiscConfig:
        C, d, t1, t2 = self.dims
        return ops.DiscConfig(C=C, d=d, t1=t1, t2=t2, inner_instance=0, prj_path=3, p=self.net_pair_one.p,
                              ln_eps=self.net_pair_one.embedding.norm.eps, ksize=self.net_pair_one.embedding.conv.kernel_size[0])

    def disc_params(self):
        y = self.net_pair_two
        return self.net_pair_one.disc_params() + [y[0][0].weight, y[0][0].bias, y[1][0].weight, y[1][0].bias,
                                                  self.fc.weight, self.fc.bias]

"""MIL encoders with the reference's constructor/forward surface and state_dict layout (model/backbone.py),
executed by the fused CUDA path: ABMIL, DeepAttMISL (`cluster`) and the ESAT transformer DualTrans_HS (`patch`).
PatchGCN (`graph`, needs torch_geometric) is out of scope (SURVEY.md §2.1) and raises NotImplementedError.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import List, Optional

import torch
import torch.nn as nn

from .. import get_precision, ops
from ..utils.func import next_dropout_seed
from .backbone_utils import Attn_Net_Gated, GAPool, make_embedding_layer, make_transformer_layer


def load_backbone_param(mode, dims):
    """Default parameters per mode (reference model/backbone.py:29-45)."""
    if mode == "patch":
        param_emb = SimpleNamespace(in_dim=dims[0], out_dim=dims[1], scale=4, dw_conv=False, ksize=1)
        param_tra = SimpleNamespace(d_model=dims[1], nhead=8, dropout=0.25, num_layers=1)
        return [dims[:3], "avgpool", param_emb, "Transformer", param_tra], {"dropout": 0.25}
    if mode == "cluster":
        return [dims[:3]], {"num_clusters": 8, "dropout": 0.25}
    if mode == "graph":
        raise NotImplementedError("backbone mode 'graph' (PatchGCN) is outside the B200 hot path (abmil / cluster / patch are built)")
    return [dims[:3]], {"dropout": 0.25}


def Model_Zoo(mode):
    if mode == "patch":
        return DualTrans_HS
    if mode == "cluster":
        return DeepAttMISL
    if mode == "graph":
        raise NotImplementedError("backbone mode 'graph' (PatchGCN) is outside the B200 hot path (abmil / cluster / patch are built)")
    return ABMIL


def load_backbone(mode, dims):
    """Same contract as the reference's load_backbone (model/backbone.py:47-51)."""
    net = Model_Zoo(mode)
    args, kws = load_backbone_param(mode, dims)
    return net(*args, **kws)


class _GatedMILBase(nn.Module):
    """Shared plumbing: collects the 14 generator tensors (GEN_TENSORS order) and runs the fused path."""

    kind = "abmil"

    def gen_params(self, head: Optional[nn.ModuleList] = None):
        an = self.attention_net
        gate = an[3]
        rho = getattr(self, "rho", None)
        p = [an[0].weight, an[0].bias, gate.attention_a[0].weight, gate.attention_a[0].bias, gate.attention_b[0].weight,
             gate.attention_b[0].bias, gate.attention_c.weight, gate.attention_c.bias,
             None if rho is None else rho[0].weight, None if rho is None else rho[0].bias]
        if head is None:
            p += [None, None, None, None]
        else:
            p += [head[0][0].weight, head[0][0].bias, head[1][0].weight, head[1][0].bias]
        return p


class ABMIL(_GatedMILBase):
    """Attention MIL encoder (reference model/backbone.py:54-86): attention_net = [Linear, ReLU, Dropout,
    Attn_Net_Gated], rho = [Linear, ReLU, Dropout]."""

    def __init__(self, dims: List, dropout: float = 0.25):
        super().__init__()
        assert len(dims) == 3
        dim_in, dim_hid, dim_out = dims
        self.dims = (dim_in, dim_hid, dim_out)
        self.p = dropout
        self.attention_net = nn.Sequential(nn.Linear(dim_in, dim_hid), nn.ReLU(), nn.Dropout(dropout),
                                           Attn_Net_Gated(L=dim_hid, D=dim_hid, dropout=dropout, n_classes=1))
        self.rho = nn.Sequential(nn.Linear(dim_hid, dim_out), nn.ReLU(), nn.Dropout(dropout))

    def config(self, hid=0, noise=(0, 0), out_scale=0, p_head=0.0) -> ops.GenConfig:
        C, h, o = self.dims
        return ops.GenConfig(C=C, h=h, o=o, hid=hid, noise0=noise[0], noise1=noise[1], out_scale=out_scale,
                             p_backbone=self.p, p_head=p_head)

    def forward(self, x_path, *args):
        """x_path [1,N,C] -> H [1,dim_out] (backbone-only mode of the fused generator kernels)."""
        bags = ops.PackedBags.from_single(x_path)
        H = ops.GeneratorFn.apply(self.config(), bags, None, None, None, self.training,
                                  next_dropout_seed() if self.training else 0, getattr(self, "_inject_masks", None),
                                  ops.PRECISIONS[get_precision()], *self.gen_params())
        return H


class DeepAttMISL(_GatedMILBase):
    """Cluster-based encoder (reference model/backbone.py:89-123): phis (1x1 conv == linear) + ReLU per instance,
    mean per cluster id (zeros for an empty cluster), then Linear+ReLU+Dropout, gated attention over the clusters."""

    kind = "cluster"

    def __init__(self, dims: List, num_clusters=8, dropout=0.25):
        super().__init__()
        assert len(dims) == 3
        dim_in, dim_hid, dim_out = dims
        assert dim_hid == dim_out
        self.dims = (dim_in, dim_hid, dim_out)
        self.dim_hid = dim_hid
        self.num_clusters = num_clusters
        self.p = dropout
        self.phis = nn.Sequential(nn.Conv2d(dim_in, dim_hid, 1), nn.ReLU())
        self.pool1d = nn.AdaptiveAvgPool1d(1)
        self.attention_net = nn.Sequential(nn.Linear(dim_hid, dim_hid), nn.ReLU(), nn.Dropout(dropout),
                                           Attn_Net_Gated(L=dim_hid, D=dim_hid, dropout=dropout, n_classes=1))

    def config(self, hid=0, noise=(0, 0), out_scale=0, p_head=0.0) -> ops.GenConfig:
        _, h, _ = self.dims
        # the attention stage sees "bags" of num_clusters rows of width h; no rho layer (H = w @ g)
        return ops.GenConfig(C=h, h=h, o=h, hid=hid, noise0=noise[0], noise1=noise[1], out_scale=out_scale,
                             p_backbone=self.p, p_head=p_head, has_rho=False)

    def phi_params(self):
        """The parameters of phis.0: the 1x1 conv weight [h, C, 1, 1] (contiguous: the memory of the [h, C] projection
        weight) and its bias [h]."""
        return self.phis[0].weight, self.phis[0].bias

    def cluster_rows(self, x_path: torch.Tensor, cluster_id: torch.Tensor, lengths=None, offsets=None) -> torch.Tensor:
        """[rows,C] (+ ids) -> per-(bag, cluster) mean of relu(phis(x)) [bags*num_clusters, h], differentiable.
        offsets: the packed bags' int32 device offsets when the caller already has them (building them here costs a
        synchronous pageable H2D copy, i.e. a host-device sync per call)."""
        x = x_path[0] if x_path.dim() == 3 else x_path
        cid = cluster_id.reshape(-1)  # accepts the handler's [1,N] as well as [N] (reference quirk A.4#7)
        assert cid.shape[0] == x.shape[0], "one cluster id per instance (dataset/PatchWSI.py:93)"
        lengths = [x.shape[0]] if lengths is None else lengths
        W = self.phis[0].weight
        return ClusterPoolFn.apply(x, cid if cid.dtype == torch.int32 else cid.to(torch.int32), lengths, self.num_clusters,
                                   ops.PRECISIONS[get_precision()], W.reshape(W.shape[0], -1), self.phis[0].bias, offsets)

    def cluster_bags(self, hc: torch.Tensor, n_bags: int) -> "ops.PackedBags":
        """Packed view of the per-(bag, cluster) rows: num_clusters rows per bag; the device offsets are cached per shape."""
        key = (n_bags, str(hc.device))
        cache = self.__dict__.setdefault("_cluster_offsets", {})
        if key not in cache:
            cache[key] = torch.arange(0, (n_bags + 1) * self.num_clusters, self.num_clusters, dtype=torch.int32, device=hc.device)
        return ops.PackedBags(hc, [self.num_clusters] * n_bags, offsets=cache[key])

    def forward(self, x_path, cluster_id, *args):
        hc = self.cluster_rows(x_path, cluster_id)
        bags = ops.PackedBags(hc, [self.num_clusters])
        H = ops.GeneratorFn.apply(self.config(), bags, hc, None, None, self.training,
                                  next_dropout_seed() if self.training else 0, getattr(self, "_inject_masks", None),
                                  ops.FP32, *self.gen_params())   # num_clusters rows: always the exact fp32 engine
        return H


class DualTrans_HS(nn.Module):
    """ESAT encoder (reference model/backbone.py:171-196): AVGPoolPatchEmbedding -> (+ sincos PE of the region
    coordinates) -> one post-norm nn.TransformerEncoderLayer over the regions of the bag -> GAPool.  The sub-modules are
    parameter containers with the reference's state_dict names; the arithmetic runs in advmil_esat_fwd/bwd."""

    kind = "patch"

    def __init__(self, dims: List, emb_backbone: str, args_emb_backbone, tra_backbone: str, args_tra_backbone,
                 dropout: float = 0.25):
        super().__init__()
        assert len(dims) == 3  # dim_in, dim_hid, dim_out = [1024, 384, 384]
        dim_in, dim_hid, dim_out = dims
        assert dim_hid == dim_out
        assert emb_backbone in ["avgpool", "gapool"]
        assert tra_backbone in ["Transformer", "Identity"]
        if tra_backbone != "Transformer" or args_tra_backbone.num_layers != 1:
            raise NotImplementedError("the fused ESAT path covers one Transformer encoder layer (model/backbone.py:33)")
        self.dims = (dim_in, dim_hid, dim_out)
        self.patch_embedding_layer = make_embedding_layer(emb_backbone, args_emb_backbone)
        if self.patch_embedding_layer.conv.kernel_size != (1, 1):
            # advmil_esat_fwd / _bwd take the patch embedding as a per-patch linear [d, C]; load_backbone fixes ksize 1 (:21)
            raise NotImplementedError("the fused ESAT path covers the ksize-1 patch embedding only")
        self.dim_hid = dim_hid
        self.patch_encoder_layer = make_transformer_layer(tra_backbone, args_tra_backbone)
        self.pool = GAPool(dim_out, dim_out)
        self.nhead, self.p = args_tra_backbone.nhead, args_tra_backbone.dropout
        assert self.pool.p == self.p, "encoder-layer and GAPool dropout share one probability in the fused path"

    def esat_config(self) -> ops.EsatConfig:
        layer = self.patch_encoder_layer.layers[0]
        return ops.EsatConfig(C=self.dims[0], d=self.dim_hid, ff=layer.linear1.out_features, nhead=self.nhead, p=self.p,
                              ln_eps=layer.norm1.eps)

    def config(self, hid=0, noise=(0, 0), out_scale=0, p_head=0.0) -> ops.GenConfig:
        """The Generator's noise head on top of H (no rho layer)."""
        d = self.dim_hid
        return ops.GenConfig(C=d, h=d, o=d, hid=hid, noise0=noise[0], noise1=noise[1], out_scale=out_scale, p_backbone=0.0,
                             p_head=p_head, has_rho=False)

    def esat_params(self):
        e, layer, pool = self.patch_embedding_layer, self.patch_encoder_layer.layers[0], self.pool
        sa = layer.self_attn
        return [e.conv.weight, e.conv.bias, e.norm.weight, e.norm.bias, sa.in_proj_weight, sa.in_proj_bias,
                sa.out_proj.weight, sa.out_proj.bias, layer.linear1.weight, layer.linear1.bias, layer.linear2.weight,
                layer.linear2.bias, layer.norm1.weight, layer.norm1.bias, layer.norm2.weight, layer.norm2.bias,
                pool.fc1[0].weight, pool.fc1[0].bias, pool.score[0].weight, pool.score[0].bias, pool.fc2.weight, pool.fc2.bias]

    def positional(self, bags: ops.PackedBags, coord) -> Optional[torch.Tensor]:
        """coord: None (no PE, model/backbone.py:192) or the regions' discretised coordinates [1,R,2] / [R,2]."""
        if coord is None:
            return None
        if coord.dim() == 3:
            assert coord.shape[0] == 1   # backbone_utils.py:91
            coord = coord.squeeze(0)
        if coord.dim() != 2 or coord.shape[-1] != 2:   # the handler's placeholder Tensor([0]) (dataset/PatchWSI.py:83) fails in the reference too
            raise IndexError("Dimension out of range: coord must be [B, N, 2] region coordinates or None "
                             "(model/backbone_utils.py:90-99)")
        return ops.sincos_pe(coord, bags, self.dim_hid)

    def forward_packed(self, bags: ops.PackedBags, coord=None, head=None, head_params=(None,) * 4, noise=(None, None),
                       precision: Optional[int] = None) -> torch.Tensor:
        precision = ops.PRECISIONS[get_precision()] if precision is None else precision
        train = self.training
        return ops.EsatFn.apply(self.esat_config(), head, bags, self.positional(bags, coord), noise[0], noise[1], train,
                                next_dropout_seed() if train else 0, getattr(self, "_inject_masks", None) if train else None,
                                precision, None, None, *self.esat_params(), *head_params)

    def forward(self, x, coord, *args):
        """x: [B, N, d], coord: the coordinates after discretization if not None -> H [1, dim_out]."""
        return self.forward_packed(ops.PackedBags.from_single(x), coord)


class ClusterPoolFn(torch.autograd.Function):
    """K9: hx = relu(x Wphi^T + b) on every row (projection GEMM), then segment-mean by cluster id."""

    @staticmethod
    def forward(ctx, x, cid, lengths, ncl, precision, W, b, offsets=None):
        import ctypes as C
        from .. import _lib
        lib = _lib.load()
        bags = ops.PackedBags(x.detach(), lengths, offsets=offsets).for_precision(precision)
        hx = ops.linear_forward(bags.x, W.detach(), b.detach(), act=1, precision=precision)
        elem = ops.ELEM_BF16 if hx.dtype == torch.bfloat16 else ops.ELEM_F32
        h = W.shape[0]
        out = torch.empty(bags.bags * ncl, h, dtype=torch.float32, device=x.device)
        counts = torch.empty(bags.bags * ncl, dtype=torch.int32, device=x.device)
        cid = cid.contiguous()
        wsb = lib.advmil_segment_mean_workspace_bytes(bags.rows, bags.bags, h, ncl)
        ws = torch.empty(max(wsb, 256), dtype=torch.uint8, device=x.device)
        _lib.check(lib.advmil_segment_mean_by_id_fwd(hx.data_ptr(), elem, cid.data_ptr(), bags.offsets.data_ptr(), bags.offsets_host,
                                                     bags.rows, bags.bags, h, ncl, out.data_ptr(), counts.data_ptr(),
                                                     ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream),
                   "advmil_segment_mean_by_id_fwd")
        ctx.saved = (bags, hx, cid, counts, W, ncl, precision)
        return out

    @staticmethod
    def backward(ctx, d_out):
        from .. import _lib
        lib = _lib.load()
        bags, hx, cid, counts, W, ncl, precision = ctx.saved
        h = W.shape[0]
        d_hx = torch.empty_like(hx)
        d_out = d_out.contiguous().float()
        elem = ops.ELEM_BF16 if hx.dtype == torch.bfloat16 else ops.ELEM_F32
        _lib.check(lib.advmil_segment_mean_by_id_bwd(d_out.data_ptr(), hx.data_ptr(), elem, cid.data_ptr(), bags.offsets.data_ptr(),
                                                     counts.data_ptr(), bags.rows, bags.bags, h, ncl, 1, d_hx.data_ptr(),
                                                     torch.cuda.current_stream().cuda_stream), "advmil_segment_mean_by_id_bwd")
        _, dW, db = ops.linear_backward(d_hx, bags.x, W.detach(), need_dx=False, precision=precision)
        return None, None, None, None, None, dW.reshape(W.shape), db, None

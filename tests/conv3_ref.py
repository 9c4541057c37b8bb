"""Reference for the 3x3 patch embedding (disc_netx_ksize: 3) used by the ksize-3 tests.

AVGPoolPatchEmbedding.forward (reference model/backbone_utils.py:158-168) with ksize 3: the rows of every region form a
4x4 image (row 16r + 4i + j = region r, grid row i, grid column j), Conv2d(C -> d, 3, stride 1, padding 1) runs on each
image on its own, then LayerNorm, ReLU and the 16-row mean as for ksize 1.  `region_embed` follows the oracle's
`region_embed` (same storage points `_q` / `_qg`, so `O.bf16_storage()` emulates the bf16 path) and hands 1x1 weights to
it; `oracle_conv3()` routes the oracle's discriminator, trainer and step functions through it."""
import contextlib
from types import SimpleNamespace

import torch
import torch.nn.functional as F

from oracle import advmil_oracle as O

_REGION_EMBED_1X1 = O.region_embed


def region_embed(sd, x, prefix="net_pair_one.embedding", eps=1e-5):
    W = sd[f"{prefix}.conv.weight"]
    if W.shape[-1] == 1:
        return _REGION_EMBED_1X1(sd, x, prefix, eps)
    N, C = x.shape
    assert N % 16 == 0
    img = O._q(x).reshape(N // 16, 4, 4, C).permute(0, 3, 1, 2)
    y = F.conv2d(img, O._q(W), sd[f"{prefix}.conv.bias"], padding=1)            # [R, d, 4, 4]
    y = O._q(O._qg(y.permute(0, 2, 3, 1).reshape(N, -1)))
    e = torch.relu(F.layer_norm(y, (y.shape[-1],), sd[f"{prefix}.norm.weight"], sd[f"{prefix}.norm.bias"], eps))
    return {"y": y, "e": e, "emb": e.reshape(N // 16, 16, -1).mean(dim=1)}


@contextlib.contextmanager
def oracle_conv3():
    prev, O.region_embed = O.region_embed, region_embed
    try:
        yield
    finally:
        O.region_embed = prev


def d_shapes(C=1024, d=128, ty=(64, 128), ksize=3):
    sh = dict(O.D_SHAPES(C, d, ty))
    sh["net_pair_one.embedding.conv.weight"] = (d, C, ksize, ksize)
    return sh


def dcat_shapes(C=1024, d=128, ty=(64, 128), ksize=3):
    sh = dict(O.DCAT_SHAPES(C, d, ty))
    sh["net_pair_one.embedding.conv.weight"] = (d, C, ksize, ksize)
    return sh


def build_D3(C=1024, d=128, iprd="instance", prj="x", cat=False, device="cuda"):
    from advmil_b200.model.GANSurv import Discriminator, PrjDiscriminator
    ax = SimpleNamespace(in_dim=C, out_dim=d, ksize=3, backbone="avgpool", dropout=0.25)
    ay = SimpleNamespace(in_dim=1, hid_dims=[64, 128] if d == 128 else [d // 2, d], norm=False, dropout=0.0)
    D = Discriminator(ax, ay) if cat else PrjDiscriminator(ax, ay, prj_path=prj, inner_product=iprd)
    return D.to(device)

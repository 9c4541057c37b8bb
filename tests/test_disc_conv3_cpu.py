"""CPU: the 3x3 patch embedding of the RLIP discriminator (disc_netx_ksize: 3) -- the reference used by the GPU tests
against a composition of the torch modules AVGPoolPatchEmbedding is built from, the module surface (state dict, argument
checks) and the registered operators on the meta device.  No kernel runs."""
import pytest
import torch
import torch.nn as nn
from torch.func import functional_call

from advmil_b200 import library, ops
from oracle import advmil_oracle as O
from tests.conv3_ref import build_D3, d_shapes, dcat_shapes, region_embed
from tests.test_library_meta import _bags, _meta


def _module_region_embed(sd, x, prefix="net_pair_one.embedding", eps=1e-5):
    """AVGPoolPatchEmbedding.forward (reference model/backbone_utils.py:158-168) composed from nn modules: sequence2square,
    Conv2d(C, d, 3, 1, padding=1), square2sequence, LayerNorm, ReLU, back to the square, AdaptiveAvgPool2d(1)."""
    W, b = sd[f"{prefix}.conv.weight"], sd[f"{prefix}.conv.bias"]
    d, C = W.shape[:2]
    N = x.shape[0]
    R = N // 16
    conv = nn.Conv2d(C, d, 3, 1, padding=1).to(x.dtype)
    norm = nn.LayerNorm(d, eps=eps).to(x.dtype)
    sq = x.reshape(R, 4, 4, C).permute(0, 3, 1, 2)                                   # sequence2square
    y = functional_call(conv, {"weight": W, "bias": b}, (sq,))
    seq = y.permute(0, 2, 3, 1).reshape(R, 16, d)                                     # square2sequence
    e = nn.ReLU()(functional_call(norm, {"weight": sd[f"{prefix}.norm.weight"], "bias": sd[f"{prefix}.norm.bias"]}, (seq,)))
    emb = nn.AdaptiveAvgPool2d(1)(e.reshape(R, 4, 4, d).permute(0, 3, 1, 2)).reshape(R, d)
    return {"y": seq.reshape(N, d), "e": e.reshape(N, d), "emb": emb}


def _rel(a, b):
    a, b = a.detach(), b.detach()
    return float((a - b).abs().max() / (b.abs().max() + 1e-300))


def test_reference_region_embed_matches_torch_modules_float64():
    C, d, N = 64, 32, 16 * 13
    sd = {k: v.double().requires_grad_(True) for k, v in O.synth_state_dict(d_shapes(C, d, (16, 32)), 1).items()
          if k.startswith("net_pair_one.embedding.")}
    sd2 = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    x = O.synth_bag(N, 2, C).double().requires_grad_(True)
    x2 = x.detach().clone().requires_grad_(True)
    g = torch.randn(N // 16, d, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    a, m = region_embed(sd, x), _module_region_embed(sd2, x2)
    assert _rel(a["emb"], m["emb"]) < 1e-12 and _rel(a["y"], m["y"]) < 1e-12
    (a["emb"] * g).sum().backward()
    (m["emb"] * g).sum().backward()
    assert _rel(x.grad, x2.grad) < 1e-12
    for k in sd:
        assert _rel(sd[k].grad, sd2[k].grad) < 1e-12, k


def test_reference_region_embed_keeps_regions_apart():
    """A change in one row moves only the embedding of its own region (bags are whole regions)."""
    C, d, N = 64, 32, 16 * 5
    sd = {k: v.double() for k, v in O.synth_state_dict(d_shapes(C, d, (16, 32)), 4).items()}
    x = O.synth_bag(N, 5, C).double()
    e0 = region_embed(sd, x)["emb"]
    x[16 * 2 + 15] += 1.0
    moved = (region_embed(sd, x)["emb"] - e0).abs().amax(dim=1) > 0
    assert moved.tolist() == [False, False, True, False, False]


def _both(fn):
    """fn() under the 3x3 reference and under the torch-module composition"""
    res = []
    for impl in (region_embed, _module_region_embed):
        prev, O.region_embed = O.region_embed, impl
        try:
            res.append(fn())
        finally:
            O.region_embed = prev
    return res


def test_trainer_step_with_conv3_matches_torch_modules_float64():
    """One D step + G step of the oracle trainer with the 3x3 embedding, against the same trainer whose embedding is the
    torch-module composition: losses, predictions and every gradient in float64."""
    C, d, h, o = 64, 32, 32, 32
    Ns = [48, 160, 32]
    B = len(Ns)
    sdG = O.synth_state_dict(O.G_SHAPES(C, h, o), 6, dtype=torch.float64)
    sdD = O.synth_state_dict(d_shapes(C, d, (16, 32)), 7, dtype=torch.float64)
    xs = [O.synth_bag(n, 8 + i, C).double() for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 9)
    ts, es = ts.double(), es.double()
    es[0] = 1.0
    vis = [True, False, True]
    nd = [torch.rand(o // 2, dtype=torch.float64, generator=torch.Generator().manual_seed(10 + i)) for i in range(B)]
    ng = [torch.rand(o // 2, dtype=torch.float64, generator=torch.Generator().manual_seed(20 + i)) for i in range(B)]
    a, b = _both(lambda: O.CpuTrainer(sdG, sdD).step(xs, ts, es, vis, nd, ng))
    for k in ("dis_loss", "gen_loss", "t_reg", "total"):
        assert abs(a[k] - b[k]) <= 1e-12 * max(1.0, abs(b[k])), k
    for k in ("pred_d", "pred_g", "fake_d", "fake_g"):
        assert _rel(a[k], b[k]) < 1e-12, k
    for key in ("d_grads", "g_grads"):
        for k in b[key]:
            assert _rel(a[key][k], b[key][k]) < 1e-10, (key, k)


@pytest.mark.parametrize("kind", ["instance", "bag", "cat"])
def test_discriminator_forward_with_conv3_matches_torch_modules_float64(kind):
    C, d, N = 64, 32, 16 * 9
    shapes = (dcat_shapes if kind == "cat" else d_shapes)(C, d, (16, 32))
    sd = O.synth_state_dict(shapes, 11, dtype=torch.float64)
    x = O.synth_bag(N, 12, C).double()
    t = torch.tensor([[0.3]], dtype=torch.float64)

    def run():
        r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        out = O.catdisc_forward(r, x, t) if kind == "cat" else O.prjdisc_forward(r, x, t, inner_product=kind)
        out["out"].sum().backward()
        return out["out"].detach(), {k: v.grad for k, v in r.items()}

    (oa, ga), (ob, gb) = _both(run)
    assert _rel(oa, ob) < 1e-12
    for k in gb:
        if gb[k] is not None:
            assert _rel(ga[k], gb[k]) < 1e-10, k


def test_ksize3_discriminators_have_the_reference_state_dict():
    D = build_D3(64, 32, device="cpu")
    assert {k: tuple(v.shape) for k, v in D.state_dict().items()} == d_shapes(64, 32, (16, 32))
    assert D.config().ksize == 3 and library.disc_cfg_lists(D.config())[0][-1] == 3
    Dc = build_D3(64, 32, cat=True, device="cpu")
    assert {k: tuple(v.shape) for k, v in Dc.state_dict().items()} == dcat_shapes(64, 32, (16, 32))
    assert Dc.config().ksize == 3
    n = sum(v.numel() for v in build_D3(device="cpu").state_dict().values())
    assert n == 1254914
    cfg = library._disc_cfg(*library.disc_cfg_lists(D.config()))
    assert cfg == D.config()


def test_unsupported_patch_embeddings_still_raise():
    from advmil_b200.model.backbone_utils import AVGPoolPatchEmbedding
    with pytest.raises(AssertionError):
        AVGPoolPatchEmbedding(64, 32, 4, False, 2)
    with pytest.raises(NotImplementedError):
        AVGPoolPatchEmbedding(64, 32, 4, False, 3, stride=2)
    with pytest.raises(NotImplementedError):
        AVGPoolPatchEmbedding(64, 32, 4, True, 3)
    assert AVGPoolPatchEmbedding(64, 32, 4, False, 3).conv.weight.shape == (32, 64, 3, 3)


def test_esat_generator_still_rejects_a_3x3_patch_embedding():
    """The ESAT generator's C path takes its patch embedding as a per-patch linear [d, C]; its constructor refuses ksize 3
    (load_backbone fixes ksize 1, model/backbone.py:21) instead of running a 3x3 weight as if it were 1x1."""
    from advmil_b200.model.backbone import DualTrans_HS, load_backbone_param
    args, kws = load_backbone_param("patch", [64, 32, 32])
    args[2].ksize = 3
    with pytest.raises(NotImplementedError):
        DualTrans_HS(*args, **kws)
    args[2].ksize = 1
    assert DualTrans_HS(*args, **kws).patch_embedding_layer.conv.weight.shape == (32, 64, 1, 1)


def test_ksize3_abi_field():
    cfg = ops.DiscConfig(C=64, d=32, t1=16, t2=32, ksize=3)
    assert cfg.c([None] * 24).ksize == 3
    assert ops.DiscConfig(C=64, d=32, t1=16, t2=32).c([None] * 24).ksize == 1


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "bf16"])
def test_ksize3_discriminator_op_differentiates_on_meta(precision):
    D = build_D3(device="cpu")
    D.train()
    dp = _meta(D.disc_params())
    bags = _bags([320, 640], dtype=torch.bfloat16 if precision == "bf16" else torch.float32)
    t = torch.empty(2, device="meta", requires_grad=True)
    f = library.discriminator(D.config(), bags, t, True, 12, None, ops.PRECISIONS[precision], dp)
    assert tuple(f.shape) == (2,)
    f.sum().backward()
    assert t.grad is not None
    for p in dp:
        if p is not None:
            assert p.grad is not None and p.grad.shape == p.shape
    assert dp[0].shape == (128, 1024, 3, 3)

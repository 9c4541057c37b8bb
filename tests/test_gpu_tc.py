"""GPU: the tcgen05/TMA/TMEM engine (precision mode 'tf32') — stage level against fp32 matmul, module level against the
oracle.  Tolerance: north_star's reduced-precision bound 2e-2 (norm-wise per tensor); the stage tests use the much
tighter 3e-3 that single-pass TF32 (10-bit mantissa) must meet, so descriptor/layout bugs cannot hide."""
import numpy as np
import pytest
import torch

import advmil_b200
from advmil_b200 import ops
from oracle import advmil_oracle as O
from tests.util import assert_close, build_D, build_G, d_masks, g_masks, to_dev_masks

pytestmark = pytest.mark.gpu
TF32 = ops.TF32


def _rel(a, b):
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


@pytest.mark.parametrize("rows,K,N", [(1000, 1024, 384), (4096, 384, 768), (256, 1024, 128), (130, 64, 256), (8192, 768, 384)])
def test_tc_linear_fwd(rows, K, N):
    g = torch.Generator(device="cuda").manual_seed(rows + N)
    x = torch.randn(rows, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    y = ops.linear_forward(x, W, b, act=1, precision=TF32)
    ref = torch.relu(x.double() @ W.double().t() + b.double()).float()
    assert _rel(y, ref) < 3e-3, _rel(y, ref)
    y0 = ops.linear_forward(x, W, None, act=0, precision=TF32)
    ref0 = (x.double() @ W.double().t()).float()
    assert _rel(y0, ref0) < 3e-3, _rel(y0, ref0)


@pytest.mark.parametrize("rows,K,N", [(8192, 1024, 384), (5000, 384, 768), (4096, 1024, 128), (16384, 256, 256)])
def test_tc_linear_bwd(rows, K, N):
    g = torch.Generator(device="cuda").manual_seed(rows + K)
    x = torch.randn(rows, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    dY = torch.randn(rows, N, device="cuda", generator=g)
    dX, dW, db = ops.linear_backward(dY, x, W, precision=TF32)
    assert _rel(dW, (dY.double().t() @ x.double()).float()) < 3e-3
    assert _rel(dX, (dY.double() @ W.double()).float()) < 3e-3
    assert _rel(db, dY.double().sum(0).float()) < 1e-5


def test_tc_gated_score_and_embed():
    g = torch.Generator(device="cuda").manual_seed(7)
    rows, L, D = 1000, 384, 384
    v = torch.randn(rows, L, device="cuda", generator=g)
    Wa, Wb = [torch.randn(D, L, device="cuda", generator=g) / L ** 0.5 for _ in range(2)]
    ba, bb, wc = [torch.randn(D, device="cuda", generator=g) * 0.1 for _ in range(3)]
    bc = torch.randn(1, device="cuda", generator=g)
    s, ab = ops.gated_score_forward(v, Wa, ba, Wb, bb, wc, bc, precision=TF32)
    a = torch.tanh(v.double() @ Wa.double().t() + ba.double())
    b = torch.sigmoid(v.double() @ Wb.double().t() + bb.double())
    ref = ((a * b) @ wc.double() + bc.double()).float()
    assert _rel(s, ref) < 5e-3, _rel(s, ref)
    j = torch.arange(D, device="cuda")
    ca = 128 * (j // 64) + j % 64
    assert _rel(ab[:, ca], a.float()) < 5e-3 and _rel(ab[:, ca + 64], b.float()) < 5e-3
    # K5+K6 through the embedding container
    from advmil_b200.model.backbone_utils import AVGPoolPatchEmbedding
    advmil_b200.set_precision("tf32")
    try:
        emb_mod = AVGPoolPatchEmbedding(1024, 128, 4, False, 1).cuda()
        sd = {k.replace("net_pair_one.embedding.", ""): t for k, t in O.synth_state_dict(O.D_SHAPES(), 3).items()
              if k.startswith("net_pair_one.embedding.")}
        emb_mod.load_state_dict(sd)
        x = O.synth_bag(1600, 5)
        out = emb_mod(x.cuda().unsqueeze(0))[0]
        full = {"net_pair_one.embedding." + k: t for k, t in sd.items()}
        ref = O.region_embed(full, x)["emb"]
        assert_close(out.cpu(), ref, 2e-2, "emb tf32")
        assert _rel(out.cpu(), ref) < 5e-3
    finally:
        advmil_b200.set_precision("fp32")


@pytest.mark.parametrize("N,train", [(4096, False), (2000, True)])
def test_tf32_mode_generator_and_discriminator_vs_oracle(N, train):
    advmil_b200.set_precision("tf32")
    try:
        dims = (1024, 384, 384)
        sdG, sdD = O.synth_state_dict(O.G_SHAPES(*dims), 1), O.synth_state_dict(O.D_SHAPES(), 2)
        G, D = build_G(dims), build_D()
        G.load_state_dict(sdG)
        D.load_state_dict(sdD)
        N16 = N // 16 * 16
        x = O.synth_bag(N16, 3)
        noise = torch.tensor(np.random.default_rng(4).uniform(size=(1, 192)), dtype=torch.float32)
        gm = g_masks(N16, 384, 384, 50) if train else None
        dm = d_masks(N16 // 16, 128, 60) if train else None
        G.train(train)
        D.train(train)
        if train:
            G._inject_masks, D._inject_masks = to_dev_masks(gm), to_dev_masks(dm)
        bags = ops.PackedBags.from_single(x.cuda())
        pred = G.forward_packed(bags, noise=[None, noise.cuda()])
        f = D.forward_packed(bags, pred)
        (f.sum() + pred.sum()).backward()
        rG = {k: v.clone().requires_grad_(True) for k, v in sdG.items()}
        rD = {k: v.clone().requires_grad_(True) for k, v in sdD.items()}
        og = O.generator_forward(rG, x, [None, noise], (0, 1), gm)
        of = O.prjdisc_forward(rD, x, og["pred"], dm)["out"]
        (of.sum() + og["pred"].sum()).backward()
        assert_close(pred.detach().cpu(), og["pred"].detach(), 2e-2, "pred")
        assert_close(f.detach().cpu(), of.detach(), 2e-2, "f", atol_scale=0.1)
        gmax = max(float(v.grad.abs().max()) for v in list(rG.values()) + list(rD.values()) if v.grad is not None)
        for mod, ref in ((G, rG), (D, rD)):
            for k, p in mod.named_parameters():
                if ref[k].grad is None or float(ref[k].grad.abs().max()) < 1e-7:
                    continue
                assert_close(p.grad.cpu(), ref[k].grad, 2e-2, "grad " + k, atol=2e-5 * gmax)
    finally:
        advmil_b200.set_precision("fp32")

"""GPU: the bf16 storage mode (precision 'bf16': x and the [rows, *] activations in bfloat16, tcgen05 kind::f16 with fp32
accumulation; statistics, region/bag-level tensors, parameters, gradients and Adam state fp32).

Tolerance: north_star's bf16 bound, 2e-2 norm-wise per tensor, against the fp32 oracle on the SAME fp32 inputs (the
bf16 rounding of x is part of the mode).  Stage-level tests compare against float64 matmuls of the bf16-rounded operands
with 6e-3 (one bf16 output rounding = 2^-9 plus accumulation noise), so descriptor / layout bugs cannot hide."""
import numpy as np
import pytest
import torch

import advmil_b200
from advmil_b200 import ops
from oracle import advmil_oracle as O
from tests.util import assert_close, build_D, build_G, d_masks, g_masks, golden, to_dev_masks

pytestmark = pytest.mark.gpu
BF16 = ops.BF16
TOL = 2e-2


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))


def _r(t):   # bf16 rounding of an fp32 tensor, kept in float64
    return t.to(torch.bfloat16).double()


def test_cast_kernel_matches_round_to_nearest_even():
    g = torch.Generator(device="cuda").manual_seed(1)
    for n in (8, 1000, 4099, 1 << 20):
        x = torch.randn(n, device="cuda", generator=g) * 3
        y = ops.cast_bf16(x)
        assert y.dtype == torch.bfloat16 and torch.equal(y, x.to(torch.bfloat16))


@pytest.mark.parametrize("rows,K,N", [(1000, 1024, 384), (4096, 384, 768), (256, 1024, 128), (48, 64, 256), (8192, 768, 384), (1, 1024, 384)])
def test_bf16_linear_fwd(rows, K, N):
    g = torch.Generator(device="cuda").manual_seed(rows + N)
    x = torch.randn(rows, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g)
    y = ops.linear_forward(x, W, b, act=1, precision=BF16)
    assert y.dtype == torch.bfloat16
    ref = torch.relu(_r(x) @ _r(W).t() + b.double())
    assert _rel(y, ref) < 6e-3, _rel(y, ref)
    y0 = ops.linear_forward(x, W, None, act=0, precision=BF16)
    assert _rel(y0, _r(x) @ _r(W).t()) < 6e-3


@pytest.mark.parametrize("rows,K,N", [(8192, 1024, 384), (5000, 384, 768), (4096, 1024, 128), (16384, 256, 256), (100, 1024, 128)])
def test_bf16_linear_bwd(rows, K, N):
    g = torch.Generator(device="cuda").manual_seed(rows + K)
    x = torch.randn(rows, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    dY = torch.randn(rows, N, device="cuda", generator=g)
    dX, dW, db = ops.linear_backward(dY, x, W, precision=BF16)
    assert dW.dtype == torch.float32 and dX.dtype == torch.bfloat16
    assert _rel(dW, _r(dY).t() @ _r(x)) < 2e-3          # fp32 output: only accumulation noise
    assert _rel(dX, _r(dY) @ _r(W)) < 6e-3
    assert _rel(db, _r(dY).sum(0)) < 1e-4


def test_bf16_gated_score_pool_and_embed():
    g = torch.Generator(device="cuda").manual_seed(7)
    rows, L, D = 1000, 384, 384
    v = torch.randn(rows, L, device="cuda", generator=g)
    Wa, Wb = [torch.randn(D, L, device="cuda", generator=g) / L ** 0.5 for _ in range(2)]
    ba, bb, wc = [torch.randn(D, device="cuda", generator=g) * 0.1 for _ in range(3)]
    bc = torch.randn(1, device="cuda", generator=g)
    s, ab = ops.gated_score_forward(v, Wa, ba, Wb, bb, wc, bc, precision=BF16)
    a = torch.tanh(_r(v) @ _r(Wa).t() + ba.double())
    b = torch.sigmoid(_r(v) @ _r(Wb).t() + bb.double())
    ref = (a * b) @ wc.double() + bc.double()
    assert _rel(s, ref) < 6e-3, _rel(s, ref)
    j = torch.arange(D, device="cuda")
    ca = 128 * (j // 64) + j % 64
    assert ab.dtype == torch.bfloat16
    assert _rel(ab[:, ca], a) < 8e-3 and _rel(ab[:, ca + 64], b) < 8e-3
    # segmented softmax + pooling on bf16 rows == the fp32 kernel on the same (bf16-representable) values
    bags = ops.PackedBags(v, [400, 16, 584])
    vb = ops.cast_bf16(v)
    w1, z1, m1 = ops.seg_softmax_pool(s, vb, bags, want_mean=True)
    w0, z0, m0 = ops.seg_softmax_pool(s, vb.float(), bags, want_mean=True)
    assert _rel(w1, w0) < 1e-6 and _rel(z1, z0) < 1e-5 and _rel(m1, m0) < 1e-5
    # K5+K6 through the embedding container
    from advmil_b200.model.backbone_utils import AVGPoolPatchEmbedding
    advmil_b200.set_precision("bf16")
    try:
        emb_mod = AVGPoolPatchEmbedding(1024, 128, 4, False, 1).cuda()
        sd = {k.replace("net_pair_one.embedding.", ""): t for k, t in O.synth_state_dict(O.D_SHAPES(), 3).items()
              if k.startswith("net_pair_one.embedding.")}
        emb_mod.load_state_dict(sd)
        x = O.synth_bag(1600, 5)
        out = emb_mod(x.cuda().unsqueeze(0))[0]
        full = {"net_pair_one.embedding." + k: t for k, t in sd.items()}
        ref = O.region_embed(full, x)["emb"]
        assert_close(out.cpu(), ref, TOL, "emb bf16")
    finally:
        advmil_b200.set_precision("fp32")


@pytest.mark.parametrize("N,train", [(4096, False), (2000, True), (48, True)])
def test_bf16_mode_generator_and_discriminator_vs_oracle(N, train):
    advmil_b200.set_precision("bf16")
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
        # (1) against the fp32 oracle (the reference's arithmetic): 2e-2.  The two first-layer weight gradients are the
        #     exception: x W^T evaluated on bf16 operands flips the ReLU mask of the ~0.3% of pre-activations within one
        #     bf16 rounding of zero, each flip adds/removes one full term of a sum of random-sign terms -- ANY bf16
        #     evaluation shows this (the emulating oracle below reproduces the same 3-9e-2) -- so they get 1e-1 here and
        #     the tight check in (2).
        # (2) against the oracle emulating the bf16 storage points (oracle.bf16_storage): 1e-2, every tensor (the region-level
        #     contractions run on tf32 tensor cores in this mode, which the emulation does not model).
        FLIP = ("backbone.attention_net.0.weight", "net_pair_one.embedding.conv.weight", "backbone.attention_net.0.bias",
                "net_pair_one.embedding.conv.bias", "net_pair_one.embedding.norm.weight", "net_pair_one.embedding.norm.bias")
        for emulate, tol in ((False, TOL), (True, 1e-2)):
            rG = {k: v.clone().requires_grad_(True) for k, v in sdG.items()}
            rD = {k: v.clone().requires_grad_(True) for k, v in sdD.items()}
            if emulate:
                with O.bf16_storage():
                    og = O.generator_forward(rG, x, [None, noise], (0, 1), gm)
                    of = O.prjdisc_forward(rD, x, og["pred"], dm)["out"]
                    (of.sum() + og["pred"].sum()).backward()
            else:
                og = O.generator_forward(rG, x, [None, noise], (0, 1), gm)
                of = O.prjdisc_forward(rD, x, og["pred"], dm)["out"]
                (of.sum() + og["pred"].sum()).backward()
            tag = " (bf16-storage oracle)" if emulate else " (fp32 oracle)"
            assert_close(pred.detach().cpu(), og["pred"].detach(), tol, "pred" + tag)
            assert_close(f.detach().cpu(), of.detach(), tol, "f" + tag, atol_scale=0.1)
            gmax = max(float(v.grad.abs().max()) for v in list(rG.values()) + list(rD.values()) if v.grad is not None)
            for mod, ref in ((G, rG), (D, rD)):
                for k, p in mod.named_parameters():
                    if ref[k].grad is None or float(ref[k].grad.abs().max()) < 1e-7 or k.endswith(("attention_c.bias", "pool.fc2.bias")):
                        continue   # mathematically-zero gradients (softmax shift invariance)
                    t = 1e-1 if (not emulate and k in FLIP) else tol
                    assert_close(p.grad.cpu(), ref[k].grad, t, "grad " + k + tag, atol=(1e-4 if not emulate else 2e-5) * gmax)
    finally:
        advmil_b200.set_precision("fp32")


def test_bf16_fused_step_vs_reference_golden():
    """One D step + G step + Adam in the bf16 mode against the fp32 fixture of the live reference: per-bag outputs and
    losses within 2e-2; bf16 features handed in directly (the packed loader's bf16 format) give the same result as fp32
    features cast by the library."""
    from advmil_b200.step import AdvStep
    g = golden("step_full")
    C, h, o, d, seed, n_steps = [int(v) for v in g["cfg"][:6]]
    Ns = [int(v) for v in g["cfg"][6:]]
    B = len(Ns)
    sdG = O.synth_state_dict(O.G_SHAPES(C, h, o), seed)
    sdD = O.synth_state_dict(O.D_SHAPES(C, d, (64, 128) if d == 128 else (d // 2, d)), seed + 50)
    xs = [O.synth_bag(n, seed + i, C).cuda() for i, n in enumerate(Ns)]
    t, e = torch.tensor(g["t"]).cuda(), torch.tensor(g["e"]).cuda()
    vis = torch.tensor(g["visible"].astype(np.uint8)).cuda()

    def cat(per_bag, keys):
        return {k: torch.cat([m[k] for m in per_bag], dim=0).to(torch.uint8).contiguous().cuda() for k in keys}

    outs = []
    for native in (False, True):
        G, D = build_G((C, h, o)), build_D(C, d)
        G.load_state_dict(sdG)
        D.load_state_dict(sdD)
        eng = AdvStep(G, D, precision="bf16")
        bags = ops.PackedBags.from_list([x.to(torch.bfloat16) for x in xs] if native else xs)
        rng = np.random.default_rng(seed)
        nzD = torch.tensor(np.concatenate([rng.uniform(size=(1, o // 2)) for _ in range(B)]), dtype=torch.float32).cuda()
        nzG = torch.tensor(np.concatenate([rng.uniform(size=(1, o // 2)) for _ in range(B)]), dtype=torch.float32).cuda()
        mr = cat([d_masks(Ns[i] // 16, d, seed + 10 * i) for i in range(B)], ["fc1", "ga", "gs", "fc2"])
        mf = cat([d_masks(Ns[i] // 16, d, seed + 10 * i + 5) for i in range(B)], ["fc1", "ga", "gs", "fc2"])
        mg = cat([g_masks(Ns[i], h, o, seed + 10 * i) for i in range(B)], ["h", "a", "b", "rho", "mlp0"])
        out = eng.step(bags, t, e, vis, noise_d=nzD, noise_g=nzG, masks_d_real=mr, masks_d_fake=mf, masks_g=mg)
        L = eng.loss_dict(out)
        outs.append((out, L, [p.detach().clone() for p in G.parameters()]))
        assert_close(out["pred_d"].cpu(), g["pred_d0"], TOL, "pred_d")
        assert_close(out["pred_g"].cpu(), g["pred_g0"], TOL, "pred_g")
        assert_close(out["f_fake_d"].cpu(), g["fake_d0"], TOL, "fake_d", atol_scale=1e-1)
        assert_close(out["f_fake_g"].cpu(), g["fake_g0"], TOL, "fake_g", atol_scale=1e-1)
        assert abs(L["dis_loss"] - float(g["dis_loss0"])) < TOL
        assert abs(L["gen_loss"] - float(g["gen_loss0"])) < TOL
        assert abs(L["t_reg_loss"] - float(g["t_reg0"])) < TOL
    (o0, L0, p0), (o1, L1, p1) = outs
    assert torch.equal(o0["pred_g"], o1["pred_g"]) and torch.equal(o0["f_fake_g"], o1["f_fake_g"])
    for a, b in zip(p0, p1):
        assert torch.equal(a, b)


def test_precision_and_element_type_must_agree():
    from advmil_b200 import _lib
    x = torch.randn(64, 1024, device="cuda").to(torch.bfloat16)
    bags = ops.PackedBags(x, [64])
    G = build_G().eval()
    with pytest.raises(_lib.AdvmilError):
        G.forward_packed(bags, precision=ops.TF32)


@pytest.mark.parametrize("mode", ["tf32", "bf16"])
def test_cluster_generator_reduced_precision_vs_golden(mode):
    """DeepAttMISL (cfg4): the N-row phi projection and the per-cluster segment mean run on the tensor-core engine in the
    reduced-precision modes (bf16: x and relu(phi(x)) stored in bf16); the 8-row attention stage always runs in fp32."""
    g = golden("g_cluster_full")
    C, h, N, seed, empty = [int(v) for v in g["cfg"]]
    sd = O.synth_state_dict(O.G_CLUSTER_SHAPES(C, h), seed + 20)
    G = build_G((C, h, h), mode="cluster").eval()
    G.load_state_dict({k: v.clone() for k, v in sd.items()})
    x = O.synth_bag(N, seed, C)
    cid = torch.tensor(g["cid"], dtype=torch.float32)
    noise = torch.tensor(np.random.default_rng(seed + 7).uniform(size=(1, h // 2)), dtype=torch.float32)
    G.draw_noise = lambda nb, dev, zero: [None, noise.to(dev)]
    advmil_b200.set_precision(mode)
    try:
        pred = G(x.cuda().unsqueeze(0), cid.cuda())
        pred.sum().backward()
    finally:
        advmil_b200.set_precision("fp32")
    assert_close(pred.detach().cpu(), g["pred"], TOL, "pred")
    from tests.util import sub
    gmax = max(float(np.abs(g["grad." + k]).max()) for k, _ in G.named_parameters())
    for k, p in G.named_parameters():
        ref = g["grad." + k]
        if float(np.abs(ref).max()) < 1e-7:
            continue
        flip = k.startswith("backbone.phis.0")     # first-layer ReLU-mask flips (see the ABMIL test above)
        assert_close(sub(p.grad), ref, 1e-1 if (flip and mode == "bf16") else TOL, "grad " + k, atol=1e-4 * gmax)

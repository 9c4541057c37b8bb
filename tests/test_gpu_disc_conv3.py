"""GPU: the 3x3 patch embedding of the RLIP discriminator (disc_netx_ksize: 3) in every precision mode.

  * halo / leakage: integer-valued inputs make every product and sum exact in bf16, tf32 and fp32, so y_pre must equal the
    exact convolution bit for bit: nothing crosses a region or a bag, the zero padding sits at each region border, and the
    tail tile past the last region is clean;
  * stage level: embedding forward and backward against the oracle (fp32 / tf32x3 at 1e-5, tf32 and bf16 at the 1x1
    stage-level bounds), at sizes where the tcgen05 engines run in the fp32-element modes too;
  * modules, registered operators, and the fused steps (AdvStep, EsatAdvStep) against O.CpuTrainer."""
import numpy as np
import pytest
import torch

from advmil_b200 import library, ops
from oracle import advmil_oracle as O
from tests.conv3_ref import build_D3, d_shapes, dcat_shapes, oracle_conv3, region_embed
from tests.util import assert_close, build_G, d_masks, g_masks, grad_floor

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ZERO_GRAD = ("pool.fc2.bias", "attention_c.bias")
MODES = {"fp32": ops.FP32, "tf32": ops.TF32, "tf32x3": ops.TF32X3, "bf16": ops.BF16}
EMB_KEYS = ("conv.weight", "conv.bias", "norm.weight", "norm.bias")


def _emb_params(C, d, seed):
    sd = O.synth_state_dict(d_shapes(C, d), seed)
    return {k: sd["net_pair_one.embedding." + k] for k in EMB_KEYS}


def _cfg(C, d, eps=1e-5):
    return ops.DiscConfig(C=C, d=d, t1=1, t2=d, ksize=3, ln_eps=eps)


def _embed(p, x, lengths, mode, d_emb=None, eps=1e-5):
    """ops.disc_embed_forward (+ backward when d_emb is given) on the device; returns (emb, y_pre, grads)"""
    C, d = p["conv.weight"].shape[1], p["conv.weight"].shape[0]
    params = [p[k].cuda() for k in EMB_KEYS] + [None] * 20
    bags = ops.PackedBags(x.cuda(), lengths)
    acts = ops.disc_embed_forward(_cfg(C, d, eps), params, bags, MODES[mode], save=True)
    grads = None
    if d_emb is not None:
        grads = [torch.empty_like(t) for t in params[:4]] + [None] * 20
        ops.disc_embed_backward(_cfg(C, d, eps), params, bags, acts, d_emb.cuda(), grads)
        grads = [g.cpu() for g in grads[:4]]
    return acts["emb"].cpu(), acts["y_pre"].float().cpu(), grads


def _exact_conv(x, W, b):
    R, C = x.shape[0] // 16, x.shape[1]
    img = x.double().reshape(R, 4, 4, C).permute(0, 3, 1, 2)
    y = torch.nn.functional.conv2d(img, W.double(), b.double(), padding=1)
    return y.permute(0, 2, 3, 1).reshape(x.shape[0], -1)


@pytest.mark.parametrize("mode", list(MODES))
def test_conv3_halo_and_no_leakage_bit_exact(mode):
    """One impulse row per region, at each of the 16 grid positions, in the first and last region of bags of 3, 37 and 19
    regions (59 in all: the last 128-row tile is partly past the end).  Small integers times multiples of 1/8 keep every
    product and sum exact in bf16 / tf32, so y_pre is compared bit for bit with the exact convolution."""
    C, d = 1024, 128
    lengths = [48, 592, 304]
    N = sum(lengths)
    g = torch.Generator().manual_seed(11)
    W = torch.randint(-2, 3, (d, C, 3, 3), generator=g).float() / 8
    b = torch.randint(-8, 9, (d,), generator=g).float() / 8
    x = torch.zeros(N, C)
    starts = np.cumsum([0] + lengths[:-1])
    regions = []
    for s, n in zip(starts, lengths):
        regions += [s // 16, (s + n) // 16 - 1]
    regions += [r for r in range(N // 16) if r not in regions][:16 - len(regions) % 16]
    for k, r in enumerate(regions):
        row = 16 * r + k % 16
        ch = torch.randperm(C, generator=g)[:6]
        x[row, ch] = torch.randint(1, 3, (6,), generator=g).float() * torch.where(torch.rand(6, generator=g) < 0.5, -1.0, 1.0)
    p = {"conv.weight": W, "conv.bias": b, "norm.weight": torch.ones(d), "norm.bias": torch.zeros(d)}
    _, y_pre, _ = _embed(p, x, lengths, mode)
    ref = _exact_conv(x, W, b)
    assert torch.equal(y_pre.double(), ref), f"{mode}: {(y_pre.double() - ref).abs().max():.3e}"
    # rows outside every impulse's 3x3 neighbourhood in its own region are exactly the bias
    hit = torch.zeros(N, dtype=torch.bool)
    for k, r in enumerate(regions):
        i0, j0 = divmod(k % 16, 4)
        for i in range(max(0, i0 - 1), min(4, i0 + 2)):
            for j in range(max(0, j0 - 1), min(4, j0 + 2)):
                hit[16 * r + 4 * i + j] = True
    assert torch.equal(y_pre[~hit], b.expand(int((~hit).sum()), d))


@pytest.mark.parametrize("mode", list(MODES))
def test_conv3_weight_gradient_bit_exact(mode):
    """dWc bit for bit.  Every output channel gets the same filter, so each row of y_pre is constant across its columns:
    LayerNorm's centred values are exactly 0, rstd = 1 with ln_eps = 1, and with beta = 1 every ReLU is open, so
    d_y = d_emb / 16 exactly for region gradients whose entries sum to 0.  Impulse rows of small integers and d_emb in
    multiples of 16 make every product and sum exact, so dWc[o, c, kh, kw] = sum_n d_y[n, o] x[neighbour(n, kh, kw), c]
    must come out bit for bit.  Impulses sit in two of every three regions at all 16 grid positions, d_emb selects the
    first and last region of every bag and every fourth one (some with an impulse in their own 4x4 grid, some without, all
    next to regions that have one), so a tap that reads across a region or bag border changes the result.  5040 rows: the
    tcgen05 engine runs in the fp32-element modes too, and the last 128-row tile is partly past the end."""
    C, d = 1024, 128
    lengths = [48, 4096 + 592, 304]
    N = sum(lengths)
    R = N // 16
    g = torch.Generator().manual_seed(23)
    W = (torch.randint(-2, 3, (1, C, 3, 3), generator=g).float() / 8).expand(d, C, 3, 3).contiguous()
    p = {"conv.weight": W, "conv.bias": torch.full((d,), 0.25), "norm.weight": torch.ones(d), "norm.bias": torch.ones(d)}
    x = torch.zeros(N, C)
    for r in range(R):
        if r % 3 != 1:
            ch = torch.randperm(C, generator=g)[:6]
            x[16 * r + r % 16, ch] = torch.randint(1, 3, (6,), generator=g).float() * torch.where(torch.rand(6, generator=g) < 0.5, -1.0, 1.0)
    starts = np.cumsum([0] + lengths)
    sel = sorted({r for r in range(R) if r % 4 == 0} | {int(s) // 16 for s in starts[:-1]} | {int(s) // 16 - 1 for s in starts[1:]})
    d_emb = torch.zeros(R, d)
    for r in sel:
        v = torch.randint(1, 3, (d // 2,), generator=g).float() * 16 * torch.where(torch.rand(d // 2, generator=g) < 0.5, -1.0, 1.0)
        d_emb[r] = torch.cat([v, -v])[torch.randperm(d, generator=g)]
    _, y_pre, grads = _embed(p, x, lengths, mode, d_emb, eps=1.0)
    assert torch.equal(y_pre, y_pre[:, :1].expand_as(y_pre))          # the construction: constant rows
    Wd = W.double().requires_grad_(True)
    d_y = (d_emb / 16).repeat_interleave(16, dim=0).double()
    _exact_conv(x.double(), Wd, torch.zeros(d, dtype=torch.float64)).mul(d_y).sum().backward()
    assert bool(Wd.grad.abs().max() > 0)
    assert torch.equal(grads[0].double(), Wd.grad), f"{mode}: {(grads[0].double() - Wd.grad).abs().max():.3e}"


def test_conv3_bf16_rejects_channels_the_weight_gradient_cannot_tile():
    """bf16 runs only on tcgen05, whose 3x3 weight gradient tiles 9 C columns by 128 or 256 without straddling a tap: the
    forward already refuses C % 128 != 0 in bf16 instead of failing later in the backward; fp32 runs it on the FFMA path."""
    C, d = 192, 128
    p = {k: v[:, :C].contiguous() if k == "conv.weight" else v for k, v in _emb_params(1024, d, 24).items()}
    x = O.synth_bag(320, 25, C)
    with pytest.raises(ops._lib.AdvmilError, match="C % 128"):
        _embed(p, x, [320], "bf16")
    emb, _, _ = _embed(p, x, [320], "fp32")
    assert_close(emb, region_embed({"net_pair_one.embedding." + k: v for k, v in p.items()}, x)["emb"], RTOL, "emb C=192")


@pytest.mark.parametrize("mode,lengths", [
    ("fp32", [16, 320, 1600, 48]), ("fp32", [4096, 784]),
    ("tf32x3", [16, 320, 1600, 48]), ("tf32x3", [4096, 2048, 16]),
    ("tf32", [4096, 2048, 16]), ("bf16", [16, 320, 1600, 48, 2048]),
])
def test_conv3_embedding_fwd_bwd_vs_oracle(mode, lengths):
    """Forward against the oracle; backward against the float64 chain (LayerNorm / ReLU / mean backward, then the exact
    convolution's weight gradient) evaluated at the kernel's own saved y_pre.  The backward is compared at the forward's
    saved activations because the ReLU derivative jumps: a few of the 10^6 LayerNorm outputs lie within the forward's
    rounding of zero, and where the device and the oracle's CPU convolution land on different sides of it, a whole
    9 C-long row of dWc moves by d_y x (measured: up to 1.7e-2 of the tensor's largest entry in tf32x3, with the
    embedding itself within 1e-5).  bf16 is compared with the oracle that rounds at the same storage points."""
    C, d = 1024, 128
    N = sum(lengths)
    p = _emb_params(C, d, 31)
    x = O.synth_bag(N, 32)
    d_emb = torch.randn(N // 16, d, generator=torch.Generator().manual_seed(33))
    emb, y_pre, grads = _embed(p, x, lengths, mode, d_emb)
    sd = {"net_pair_one.embedding." + k: v.clone().requires_grad_(True) for k, v in p.items()}
    if mode == "bf16":
        with O.bf16_storage():
            ref = region_embed(sd, x)
            (ref["emb"] * d_emb).sum().backward()
        assert_close(emb, ref["emb"].detach(), 2e-2, "emb")
        for k, a in zip(EMB_KEYS, grads):
            assert_close(a, sd["net_pair_one.embedding." + k].grad, 2e-2, "grad " + k)
        return
    ref = region_embed(sd, x)
    assert_close(emb, ref["emb"].detach(), RTOL if mode != "tf32" else 2e-2, "emb")
    g64 = {k: v.double().requires_grad_(True) for k, v in p.items()}
    y = y_pre.double().requires_grad_(True)
    e = torch.relu(torch.nn.functional.layer_norm(y, (d,), g64["norm.weight"], g64["norm.bias"], 1e-5))
    (e.reshape(N // 16, 16, d).mean(1) * d_emb.double()).sum().backward()
    _exact_conv(x.double(), g64["conv.weight"], g64["conv.bias"]).mul(y.grad).sum().backward()
    rg = [g64[k].grad for k in EMB_KEYS]
    tol, floor = (5e-3, 0.0) if mode == "tf32" else (2e-5, 8 * grad_floor(rg))
    for k, a, e in zip(EMB_KEYS, grads, rg):
        assert_close(a, e, tol, "grad " + k, atol=floor)


@pytest.mark.parametrize("kind", ["instance-x", "bag-x", "cat"])
def test_conv3_discriminator_modules_vs_oracle(kind):
    C, d, N = 1024, 128, 4096 + 320
    iprd, cat = kind.split("-")[0], kind == "cat"
    shapes = dcat_shapes(C, d) if cat else d_shapes(C, d)
    sd = O.synth_state_dict(shapes, 41)
    D = build_D3(C, d, iprd="bag" if cat else iprd, cat=cat)
    assert {k: tuple(v.shape) for k, v in D.state_dict().items()} == shapes
    D.load_state_dict(sd)
    D.train(True)
    dm = d_masks(N // 16, d, 42)
    from tests.util import to_dev_masks
    D._inject_masks = to_dev_masks(dm)
    x = O.synth_bag(N, 43)
    t = torch.tensor([[0.4]], requires_grad=True)
    tc = t.detach().cuda().requires_grad_(True)
    out = D(x.cuda().unsqueeze(0), tc)
    out.sum().backward()
    r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    with oracle_conv3():
        ro = O.catdisc_forward(r, x, t, dm) if cat else O.prjdisc_forward(r, x, t, dm, inner_product=iprd)
    ro["out"].sum().backward()
    assert_close(out.detach().cpu().reshape(-1), ro["out"].detach().reshape(-1), RTOL, "out", atol_scale=0.1)
    assert_close(tc.grad.cpu().reshape(-1), t.grad.reshape(-1), 2e-5, "d_t", atol_scale=0.1)
    floor = grad_floor([v.grad for v in r.values()])
    for k, prm in D.named_parameters():
        if r[k].grad is None or k.endswith(ZERO_GRAD):
            continue
        assert_close(prm.grad.cpu(), r[k].grad, 2e-5, "grad " + k, atol=8 * floor)


def test_conv3_registered_ops_equal_glue_and_opcheck():
    C, d = 1024, 128
    D = build_D3(C, d)
    D.load_state_dict(O.synth_state_dict(d_shapes(C, d), 51))
    D.eval()
    x = O.synth_bag(640, 52).cuda()
    bags = ops.PackedBags.from_list([x[:320], x[320:]])
    outs, grads = [], []
    for mode in (False, True):
        library.use_registered_ops(mode)
        try:
            D.zero_grad()
            t = torch.tensor([0.3, 0.7], device="cuda", requires_grad=True)
            o = D.forward_packed(bags, t)
            o.sum().backward()
            outs.append(o.detach())
            grads.append([p.grad.clone() for p in D.parameters()] + [t.grad.clone()])
        finally:
            library.use_registered_ops("auto")
    assert torch.equal(outs[0], outs[1])
    for a, b in zip(*grads):
        assert torch.equal(a, b)
    dcfg, dfcfg = library.disc_cfg_lists(D.config())
    assert dcfg[-1] == 3
    t = torch.rand(2, device="cuda", requires_grad=True)
    dargs = (bags.x, bags.offsets, list(bags.lengths), dcfg, dfcfg, t, False, 0, ops.FP32, True,
             library._dense([None] * 4, bags.x), library._dense(D.disc_params(), bags.x))
    torch.library.opcheck(torch.ops.advmil_b200.discriminator_fwd.default, dargs, test_utils=("test_schema", "test_faketensor"))
    saved = [v.detach() for v in torch.ops.advmil_b200.discriminator_fwd(*dargs)[1:]]
    bargs = (bags.x, bags.offsets, list(bags.lengths), dcfg, dfcfg, t.detach(), False, 0, ops.FP32,
             library._dense([None] * 4, bags.x), [v.detach() for v in library._dense(D.disc_params(), bags.x)], saved,
             torch.rand(2, device="cuda"), True, True)
    torch.library.opcheck(torch.ops.advmil_b200.discriminator_bwd.default, bargs, test_utils=("test_schema", "test_faketensor"))


def _cat_masks(per_bag, keys):
    return {k: torch.cat([m[k] for m in per_bag], dim=0).to(torch.uint8).contiguous().cuda() for k in keys}


@pytest.mark.parametrize("precision", ["fp32", "tf32x3"])
def test_conv3_adv_step_vs_oracle_trainer(precision):
    """AdvStep with a ksize-3 D: two optimiser steps against the oracle trainer, mixed labelled / unlabelled bags; the tf32x3
    case has a 4096-row bag so that the tcgen05 forward and weight-gradient engines run."""
    from advmil_b200.step import AdvStep
    from tests.test_gpu_bf16_step import _named_grads
    Ns = [160, 320, 96, 640, 48] if precision == "fp32" else [160, 4096, 96, 640]
    B = len(Ns)
    sdG, sdD = O.synth_state_dict(O.G_SHAPES(), 61), O.synth_state_dict(d_shapes(), 62)
    tr = O.CpuTrainer(sdG, sdD)
    G, D = build_G(), build_D3()
    G.load_state_dict(sdG)
    D.load_state_dict(sdD)
    eng = AdvStep(G, D, precision=precision)
    xs = [O.synth_bag(n, 70 + i) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 63)
    es[1] = 1.0
    vis = [True, True, False, True, False][:B]
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    for step in range(2):
        rng = np.random.default_rng(64 + step)
        nd = torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32)
        ng = torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32)
        mr = [d_masks(n // 16, 128, 300 + 10 * i + step) for i, n in enumerate(Ns)]
        mf = [d_masks(n // 16, 128, 400 + 10 * i + step) for i, n in enumerate(Ns)]
        mg = [g_masks(n, 384, 384, 500 + 10 * i + step) for i, n in enumerate(Ns)]
        with oracle_conv3():
            ref = tr.step(xs, ts, es, vis, list(nd), list(ng), mr, mf, mg)
        out = eng.step(bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(), noise_d=nd.cuda(), noise_g=ng.cuda(),
                       masks_d_real=_cat_masks(mr, ["fc1", "ga", "gs", "fc2"]), masks_d_fake=_cat_masks(mf, ["fc1", "ga", "gs", "fc2"]),
                       masks_g=_cat_masks(mg, ["h", "a", "b", "rho", "mlp0"]))
        L = eng.loss_dict(out)
        assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, f"pred_d {step}")
        assert_close(out["pred_g"].cpu(), ref["pred_g"].reshape(-1), RTOL, f"pred_g {step}")
        assert_close(out["f_fake_d"].cpu(), ref["fake_d"].reshape(-1), RTOL, f"fake_d {step}", atol_scale=1e-1)
        assert_close(out["f_fake_g"].cpu(), ref["fake_g"].reshape(-1), RTOL, f"fake_g {step}", atol_scale=1e-1)
        assert abs(L["dis_loss"] - ref["dis_loss"]) < 2e-5 and abs(L["gen_loss"] - ref["gen_loss"]) < 2e-5
        assert abs(L["t_reg_loss"] - ref["t_reg"]) < 2e-5 and abs(L["gen_total_loss"] - ref["total"]) < 2e-5
        if step == 0:
            gD = _named_grads(D, eng.D)
            floor = max(grad_floor(list(ref["d_grads"].values())), 2.0 ** -23 / B)
            for k, g in gD.items():
                if not k.endswith(ZERO_GRAD):
                    assert_close(g.cpu(), ref["d_grads"][k], RTOL, "D grad " + k, atol=8 * floor)
            small = {k: v.abs() < 1e-3 * v.abs().max() for k, v in ref["d_grads"].items()}
    # post-Adam parameters: an entry whose gradient is a rounding-level remainder of cancelling terms moves by +-lr
    # whichever its sign (Adam's update is ~lr * sign(g) on the first step); the 3x3 weight has 1.2 M entries, so some
    # have |g| under 1e-3 of the tensor's largest.  Those are bounded by the two-step Adam move, the rest at 1e-5.
    for k, p in D.named_parameters():
        if not k.endswith(ZERO_GRAD):
            a, e = p.detach().cpu(), tr.sdD[k].detach()
            m = small[k]
            assert_close(a[~m], e[~m], RTOL, "D param " + k, atol=8e-5 * 2 * 2e-2)
            if bool(m.any()):
                assert float((a[m] - e[m]).abs().max()) <= 2 * 2 * 8e-5, k
    for k, p in G.named_parameters():
        if not k.endswith(ZERO_GRAD):
            assert_close(p.detach().cpu(), tr.sdG[k].detach(), RTOL, "G param " + k, atol=8e-5 * 2 * 2e-2)


def test_conv3_adv_step_bf16_vs_fp32_and_bf16_storage_oracles():
    """bf16 AdvStep with a ksize-3 D, one step, with the yardsticks of test_gpu_bf16_step.py: 2e-2 of each tensor's largest
    entry against the fp32 oracle outside that file's SENSITIVE list (6e-1 inside it), and 5e-3 for every tensor against the
    oracle that rounds at the bf16 path's storage points.  The conv weight is on the SENSITIVE list for the reason given
    there (ReLU units within one bf16 rounding of zero flip); the storage oracle bounds it at the tight tolerance."""
    from advmil_b200.step import AdvStep
    from tests.test_gpu_bf16_step import EMU_TOL, SENSITIVE, SENSITIVE_TOL, TOL, _named_grads
    Ns = [320, 1600, 48, 16, 2048, 640]
    B = len(Ns)
    sdG, sdD = O.synth_state_dict(O.G_SHAPES(), 81), O.synth_state_dict(d_shapes(), 82)
    xs = [O.synth_bag(n, 90 + i) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 83)
    es[0], es[1] = 1.0, 0.0
    vis = [True] * B
    vis[2] = False
    G, D = build_G(), build_D3()
    G.load_state_dict(sdG)
    D.load_state_dict(sdD)
    eng = AdvStep(G, D, precision="bf16")
    tr32, tremu = O.CpuTrainer(sdG, sdD), O.CpuTrainer(sdG, sdD)
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    rng = np.random.default_rng(84)
    nd = torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32)
    ng = torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32)
    mr = [d_masks(n // 16, 128, 400 + 10 * i) for i, n in enumerate(Ns)]
    mf = [d_masks(n // 16, 128, 500 + 10 * i) for i, n in enumerate(Ns)]
    mg = [g_masks(n, 384, 384, 600 + 10 * i) for i, n in enumerate(Ns)]
    pG0 = {k: v.detach().clone() for k, v in G.named_parameters()}
    with oracle_conv3():
        ref = tr32.step(xs, ts, es, vis, list(nd), list(ng), mr, mf, mg)
        with O.bf16_storage():
            emu = tremu.step(xs, ts, es, vis, list(nd), list(ng), mr, mf, mg)
    out = eng.step(bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(), noise_d=nd.cuda(), noise_g=ng.cuda(),
                   masks_d_real=_cat_masks(mr, ["fc1", "ga", "gs", "fc2"]), masks_d_fake=_cat_masks(mf, ["fc1", "ga", "gs", "fc2"]),
                   masks_g=_cat_masks(mg, ["h", "a", "b", "rho", "mlp0"]))
    L = eng.loss_dict(out)
    assert abs(L["dis_loss"] - ref["dis_loss"]) < TOL and abs(L["gen_total_loss"] - ref["total"]) < TOL
    problems = []
    got = {"D": _named_grads(D, eng.D), "G": _named_grads(G, eng.G)}
    for net, key in (("D", "d_grads"), ("G", "g_grads")):
        gmax32 = max(float(v.abs().max()) for v in ref[key].values())
        gmaxe = max(float(v.abs().max()) for v in emu[key].values())
        for k, gcu in got[net].items():
            if k.endswith(ZERO_GRAD):
                continue
            g = gcu.detach().cpu().double()
            if net == "G":
                g = g + 1e-5 * torch.sign(pG0[k].cpu()).double()
            e32 = float((g - ref[key][k].double()).abs().max()); s32 = float(ref[key][k].abs().max())
            ee = float((g - emu[key][k].double()).abs().max()); se = float(emu[key][k].abs().max())
            tol = SENSITIVE_TOL if k.endswith(SENSITIVE) else TOL
            if not e32 <= tol * s32 + 1e-4 * gmax32:
                problems.append(f"{net} grad {k} vs fp32 oracle: {e32:.3e} of {s32:.3e}")
            if not ee <= EMU_TOL * se + 2e-5 * gmaxe:
                problems.append(f"{net} grad {k} vs bf16-storage oracle: {ee:.3e} of {se:.3e}")
    assert not problems, "\n".join(problems)


def test_conv3_esat_adv_step_vs_oracle_trainer_and_module_step():
    """EsatAdvStep (C-fused ESAT step) with a ksize-3 RLIP discriminator in fp32: two steps against the oracle trainer and
    against ModuleAdvStep; the ESAT generator's own patch embedding stays 1x1."""
    from advmil_b200.step import EsatAdvStep, ModuleAdvStep
    C, d = 1024, 384
    Ns = [160, 320, 96, 640]
    B = len(Ns)

    def nets():
        sdG, sdD = O.synth_state_dict(O.G_ESAT_SHAPES(C, d), 171), O.synth_state_dict(d_shapes(), 172)
        G, D = build_G((C, d, d), mode="patch"), build_D3()
        G.load_state_dict(sdG)
        D.load_state_dict(sdD)
        G.backbone.p = G.backbone.pool.p = 0.0
        G.p_head = 0.0
        D.net_pair_one.p = 0.0
        return sdG, sdD, G, D

    sdG, sdD, G, D = nets()
    _, _, G2, D2 = nets()
    tr = O.CpuTrainer(sdG, sdD, backbone="patch")
    eng, mod = EsatAdvStep(G, D), ModuleAdvStep(G2, D2)
    xs = [O.synth_bag(n, 180 + i, C) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 173)
    es[0] = 1.0
    vis = [True, True, False, True]
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    for step in range(2):
        rng = np.random.default_rng(174 + step)
        nd = torch.tensor(rng.uniform(size=(B, d // 2)), dtype=torch.float32)
        ng = torch.tensor(rng.uniform(size=(B, d // 2)), dtype=torch.float32)
        with oracle_conv3():
            ref = tr.step(xs, ts, es, vis, list(nd), list(ng))
        args = (bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda())
        out = eng.step(*args, noise_d=nd.cuda(), noise_g=ng.cuda())
        om = mod.step(*args, noise_d=nd.cuda(), noise_g=ng.cuda())
        L = eng.loss_dict(out)
        assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, f"pred_d {step}")
        assert_close(out["pred_g"].cpu(), ref["pred_g"].reshape(-1), RTOL, f"pred_g {step}")
        assert_close(out["f_fake_d"].cpu(), ref["fake_d"].reshape(-1), RTOL, f"fake_d {step}", atol_scale=1e-1)
        assert_close(out["f_fake_g"].cpu(), ref["fake_g"].reshape(-1), RTOL, f"fake_g {step}", atol_scale=1e-1)
        assert abs(L["dis_loss"] - ref["dis_loss"]) < 2e-5 and abs(L["gen_loss"] - ref["gen_loss"]) < 2e-5
        assert_close(out["pred_g"].cpu(), om["pred_g"].cpu(), RTOL, f"pred_g vs module step {step}")
    for (k, p), p2 in zip(D.named_parameters(), D2.parameters()):
        if not k.endswith(ZERO_GRAD):
            assert_close(p.detach().cpu(), tr.sdD[k].detach(), RTOL, "D param " + k, atol=8e-5 * 2 * 2e-2)
            assert_close(p.detach().cpu(), p2.detach().cpu(), RTOL, "D param vs module step " + k, atol=8e-5 * 2 * 2e-2)


def test_conv3_sample_inference_runs():
    from advmil_b200.step import sample_inference
    G, D = build_G(), build_D3()
    G.load_state_dict(O.synth_state_dict(O.G_SHAPES(), 91))
    D.load_state_dict(O.synth_state_dict(d_shapes(), 92))
    bags = ops.PackedBags.from_list([O.synth_bag(n, 93 + i).cuda() for i, n in enumerate((160, 320))])
    for precision in ("fp32", "bf16"):
        res = sample_inference(G, D, bags, times_test_sample=4, precision=precision)
        vals = res.values() if isinstance(res, dict) else (res if isinstance(res, (tuple, list)) else [res])
        assert all(bool(torch.isfinite(torch.as_tensor(v)).all()) for v in vals if torch.is_tensor(v))


def test_conv3_full_size_bf16_step_is_deterministic():
    """16 x 16384 rows, bf16, one AdvStep twice from the same state: bitwise equal outputs and parameters."""
    from advmil_b200.step import AdvStep
    Ns = [16384] * 16
    B = len(Ns)
    xs = torch.cat([O.synth_bag(n, 200 + i) for i, n in enumerate(Ns[:2])] * (B // 2)).cuda()
    ts, es = O.synth_labels(B, 201)
    vis = torch.ones(B, dtype=torch.uint8).cuda()
    import itertools
    from advmil_b200.utils import func
    results = []
    for _ in range(2):
        func._seed_counter = itertools.count(12345)     # the same in-kernel dropout seeds for both runs
        G, D = build_G(), build_D3()
        G.load_state_dict(O.synth_state_dict(O.G_SHAPES(), 202))
        D.load_state_dict(O.synth_state_dict(d_shapes(), 203))
        eng = AdvStep(G, D, precision="bf16")
        bags = ops.PackedBags(xs, Ns)
        nz = torch.full((B, 192), 0.5, device="cuda")
        out = eng.step(bags, ts.cuda(), es.cuda(), vis, noise_d=nz, noise_g=nz)
        torch.cuda.synchronize()
        results.append([out["f_fake_d"].clone(), out["pred_g"].clone()] + [p.detach().clone() for p in D.parameters()])
    for a, b in zip(*results):
        assert torch.equal(a, b)

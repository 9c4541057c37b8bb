"""GPU: the RLIP discriminator at disc_netx_out_dim 64 and 256 (d; disc_nety_hid_dims = [d / 2, d]) in every precision mode.

  * modules against the oracle: d in {64, 256} x ksize {1, 3} x {instance / x, bag / y, concat} x four precision modes, on
    ragged bags that straddle the 128-row tiles, with injected dropout masks: forward, every discriminator gradient, dL/dt;
  * stage level against float64: the tcgen05 region embedding (1x1 and 3x3) and the region chain at 64 and 256 columns;
    every case first shows that its bound catches a lost K block and a one-row shift of an output tile;
  * one full D + G + Adam step of AdvStep (d = 64 and 256), ModuleAdvStep, EsatAdvStep and ClusterAdvStep (d = 256)
    against the oracle trainer, in fp32, and of AdvStep in bf16;
  * refusals: the bf16 mode still refuses widths its kernels do not run (d = 96); fp32 runs them."""
import numpy as np
import pytest
import torch

import advmil_b200
from advmil_b200 import ops
from oracle import advmil_oracle as O
from tests.conv3_ref import build_D3, d_shapes, dcat_shapes, oracle_conv3
from tests.test_gpu_bf16_step import SENSITIVE, SENSITIVE_TOL
from tests.util import assert_close, build_D, build_G, condition_esat_case, d_masks, g_masks, grad_floor, to_dev_masks

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ZERO_GRAD = ("pool.fc2.bias", "attention_c.bias")
MODES = {"fp32": ops.FP32, "tf32": ops.TF32, "tf32x3": ops.TF32X3, "bf16": ops.BF16}
EMB_KEYS = ("conv.weight", "conv.bias", "norm.weight", "norm.bias")
KBLK = {"tf32": 32, "tf32x3": 32, "bf16": 64}


def _shapes(C, d, ksize, cat):
    ty = (d // 2, d)
    if ksize == 3:
        return dcat_shapes(C, d, ty) if cat else d_shapes(C, d, ty)
    return dict(O.DCAT_SHAPES(C, d, ty)) if cat else dict(O.D_SHAPES(C, d, ty))


def _build(C, d, ksize, iprd, prj, cat):
    if ksize == 3 or cat:
        return build_D3(C, d, iprd=iprd, prj=prj, cat=cat) if ksize == 3 else _build_cat1(C, d)
    return build_D(C, d, iprd=iprd, prj=prj)


def _build_cat1(C, d):
    from types import SimpleNamespace
    from advmil_b200.model.GANSurv import Discriminator
    ax = SimpleNamespace(in_dim=C, out_dim=d, ksize=1, backbone="avgpool", dropout=0.25)
    ay = SimpleNamespace(in_dim=1, hid_dims=[d // 2, d], norm=False, dropout=0.0)
    return Discriminator(ax, ay).cuda()


def _oracle(ksize):
    import contextlib
    return oracle_conv3() if ksize == 3 else contextlib.nullcontext()


KINDS = ["instance-x", "bag-y", "cat"]
LR = 8e-5
# Tensors upstream of a region-level ReLU (the patch embedding's, the region MLP's): a ReLU argument within the forward's
# rounding of zero takes different branches on the device and in the oracle, and moves whole rows of their gradients.
#  * fp32 / tf32x3: the cases are moved off those boundaries first (_condition_disc), then EVERY tensor is held at 2e-5;
#  * tf32: the tf32 rounding of y (~1e-3) puts thousands of arguments within reach of zero, which no conditioning removes;
#    these six tensors are checked at the stage level against float64 evaluated at the kernel's own saved activations
#    (test_tc_region_embedding_vs_float64) and skipped in the module comparison; every other tensor is held at 2e-2;
#  * bf16: the yardsticks of tests/test_gpu_bf16.py -- 2e-2 against the fp32 oracle (its FLIP tensors, here these six,
#    at the bf16 step tests' SENSITIVE bound), and 1e-2 against the bf16-storage oracle for every tensor.
UPSTREAM = ("embedding.conv.weight", "embedding.conv.bias", "embedding.norm.weight", "embedding.norm.bias",
            "net_pair_one.fc1.0.weight", "net_pair_one.fc1.0.bias")


def _ln_arg(s, x, ksize):
    """float64 LayerNorm output (the ReLU's argument) of the patch embedding for x [16 R, C]"""
    P = "net_pair_one.embedding."
    W = s[P + "conv.weight"]
    d, C = W.shape[0], x.shape[1]
    if ksize == 3:
        img = x.reshape(-1, 4, 4, C).permute(0, 3, 1, 2)
        y = torch.nn.functional.conv2d(img, W, s[P + "conv.bias"], padding=1).permute(0, 2, 3, 1).reshape(-1, d)
    else:
        y = x @ W.reshape(d, C).T + s[P + "conv.bias"]
    return torch.nn.functional.layer_norm(y, (d,), s[P + "norm.weight"], s[P + "norm.bias"], 1e-5)


def _condition_disc(sd, xs, ksize, mask_sets, p=0.25, margin=1e-4, region_margin=None, bag_margin=None, iters=60):
    """Moves a discriminator case off the ReLU boundaries of its fp32-grade evaluation (cf. tests/util.py:
    condition_esat_case): rows of x whose embedding has a LayerNorm output within `margin` of zero get a small deterministic
    perturbation; region-MLP (fc1.0) and bag-MLP (fc2.0, under every mask set of the bag) columns with a pre-activation
    within `margin` of zero get a bias nudge, until the float64 evaluation has none left.  region_margin / bag_margin
    (default: margin) widen the MLP margins where the mode perturbs those pre-activations more (bf16)."""
    region_margin = margin if region_margin is None else region_margin
    bag_margin = margin if bag_margin is None else bag_margin
    P = "net_pair_one."
    sd = {k: v.clone() for k, v in sd.items()}
    xs = [x.clone() for x in xs]
    g = torch.Generator().manual_seed(4321)
    for _ in range(iters):
        s = {k: v.double() for k, v in sd.items()}
        clean, embs = True, []
        for i, x in enumerate(xs):
            a = _ln_arg(s, x.double(), ksize)
            bad = torch.nonzero((a.abs() < margin).any(dim=1)).reshape(-1)
            if bad.numel():
                xs[i][bad] += 1e-2 * torch.randn(bad.numel(), x.shape[1], generator=g)
                clean = False
            embs.append(torch.relu(a).reshape(-1, 16, a.shape[1]).mean(1))
        if not clean:
            continue
        pre = torch.cat(embs) @ s[P + "fc1.0.weight"].T + s[P + "fc1.0.bias"]
        cols = torch.nonzero((pre.abs() < region_margin).any(dim=0)).reshape(-1)
        if cols.numel():
            sd[P + "fc1.0.bias"][cols] += max(1e-3, 2 * region_margin)
            continue
        for e, masks in zip(embs, mask_sets):
            for m in masks:
                m = m or {}
                fi = O._eff_mlp(e, s, P + "fc1", m.get("fc1"), p)
                bag = O.gapool(s, fi, P + "pool", m, p)["out"]
                pre2 = bag @ s[P + "fc2.0.weight"].T + s[P + "fc2.0.bias"]
                cols = torch.nonzero((pre2.abs() < bag_margin).any(dim=0)).reshape(-1)
                if cols.numel():
                    sd[P + "fc2.0.bias"][cols] += max(1e-3, 2 * bag_margin)
                    clean = False
        if clean:
            return sd, xs
    raise AssertionError("could not condition the discriminator case")


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("ksize", [1, 3])
@pytest.mark.parametrize("d", [64, 256])
def test_disc_width_modules_vs_oracle(d, ksize, kind, mode):
    C = 1024
    lengths = [4096 + 320, 48, 1600]          # tiles straddle bag borders; the last 128-row tile is partly past the end
    N = sum(lengths)
    cat = kind == "cat"
    iprd, prj = ("bag", "x") if cat else kind.split("-")
    shapes = _shapes(C, d, ksize, cat)
    sd = O.synth_state_dict(shapes, 41 + d + ksize)
    D = _build(C, d, ksize, iprd, prj, cat)
    assert {k: tuple(v.shape) for k, v in D.state_dict().items()} == {k: tuple(v) for k, v in shapes.items()}
    xs = [O.synth_bag(n, 43 + i) for i, n in enumerate(lengths)]
    dms = [d_masks(n // 16, d, 42 + 7 * i) for i, n in enumerate(lengths)]
    if mode in ("fp32", "tf32x3"):
        sd, xs = _condition_disc(sd, xs, ksize, [[m] for m in dms])
    elif mode == "bf16":       # the MLPs' ReLUs (the embedding's: see UPSTREAM)
        sd, xs = _condition_disc(sd, xs, ksize, [[m] for m in dms], margin=0.0, region_margin=5e-4, bag_margin=2e-2)
    D.load_state_dict(sd)
    D.train(True)
    D._inject_masks = to_dev_masks({k: torch.cat([m[k] for m in dms], dim=0) for k in dms[0]})
    ts = torch.tensor([[0.4], [0.7], [0.2]])
    tc = ts.reshape(-1).cuda().requires_grad_(True)
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    advmil_b200.set_precision(mode)
    try:
        out = D.forward_packed(bags, tc)
        out.sum().backward()
    finally:
        advmil_b200.set_precision("fp32")

    def ref_run(storage):
        r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        outs, t_grads = [], []
        for x, t, m in zip(xs, ts, dms):
            tt = t.reshape(1, 1).clone().requires_grad_(True)
            with _oracle(ksize):
                o = O.catdisc_forward(r, x, tt, m) if cat else O.prjdisc_forward(r, x, tt, m, inner_product=iprd, prj_path=prj)
            o["out"].sum().backward()
            outs.append(o["out"].detach().reshape(-1))
            t_grads.append(tt.grad.reshape(-1))
        return torch.cat(outs), torch.cat(t_grads), {k: v.grad for k, v in r.items()}

    ro, rt, rg = ref_run(False)
    got = {k: p.grad.cpu() for k, p in D.named_parameters()}
    if mode == "bf16":
        with O.bf16_storage():
            eo, et, eg = ref_run(True)
        for ref_o, ref_t, ref_g, tol, atol_f, tag in ((ro, rt, rg, 2e-2, 1e-4, "fp32 oracle"), (eo, et, eg, 1e-2, 2e-5, "bf16-storage oracle")):
            assert_close(out.detach().cpu(), ref_o, tol, "out vs " + tag, atol_scale=0.1)
            assert_close(tc.grad.cpu(), ref_t, tol, "d_t vs " + tag, atol_scale=0.1)
            gmax = max(float(v.abs().max()) for v in ref_g.values() if v is not None)
            for k, g in got.items():
                if ref_g[k] is None or k.endswith(ZERO_GRAD):
                    continue
                t = SENSITIVE_TOL if (tag == "fp32 oracle" and k.endswith(UPSTREAM)) else tol
                assert_close(g, ref_g[k], t, f"grad {k} vs {tag}", atol=atol_f * gmax)
        return
    tol = 2e-2 if mode == "tf32" else RTOL
    assert_close(out.detach().cpu(), ro, tol, "out", atol_scale=0.1)
    assert_close(tc.grad.cpu(), rt, 2 * tol, "d_t", atol_scale=0.1)
    floor = grad_floor(list(rg.values()))
    for k, g in got.items():
        if rg[k] is None or k.endswith(ZERO_GRAD) or (mode == "tf32" and k.endswith(UPSTREAM)):
            continue
        assert_close(g, rg[k], 2 * tol, "grad " + k, atol=8 * floor)


# ---------------------------------------------------------------------------------------------------------------------
# stage level against float64
# ---------------------------------------------------------------------------------------------------------------------
def _emb_case(C, d, ksize, seed):
    sd = O.synth_state_dict(_shapes(C, d, ksize, False), seed)
    return {k: sd["net_pair_one.embedding." + k] for k in EMB_KEYS}


def _emb64(p, x, ksize, drop_k=None):
    """float64 region embedding; drop_k = (k0, k1) removes that block of input channels from the contraction"""
    W = p["conv.weight"].double()
    if drop_k is not None:
        W = W.clone()
        W[:, drop_k[0]:drop_k[1]] = 0
    xd = x.double()
    R, C, d = x.shape[0] // 16, x.shape[1], W.shape[0]
    if ksize == 3:
        img = xd.reshape(R, 4, 4, C).permute(0, 3, 1, 2)
        y = torch.nn.functional.conv2d(img, W, p["conv.bias"].double(), padding=1).permute(0, 2, 3, 1).reshape(-1, d)
    else:
        y = xd @ W.reshape(d, C).T + p["conv.bias"].double()
    e = torch.relu(torch.nn.functional.layer_norm(y, (d,), p["norm.weight"].double(), p["norm.bias"].double(), 1e-5))
    return e.reshape(R, 16, d).mean(1), y


STAGE_TOL = {"tf32": 2e-2, "tf32x3": 1e-5, "bf16": 2e-2}


@pytest.mark.parametrize("mode", ["tf32", "tf32x3", "bf16"])
@pytest.mark.parametrize("ksize", [1, 3])
@pytest.mark.parametrize("d", [64, 256])
def test_tc_region_embedding_vs_float64(d, ksize, mode):
    """The tcgen05 LN-pool epilogue at 64 / 256 columns (rows >= 128: the tensor-core engine runs in every mode).  The bound
    is checked to catch a lost K block of the contraction and a one-row shift of an output tile before it is applied."""
    C = 1024
    lengths = [4096 + 320, 1600]
    N = sum(lengths)
    p = _emb_case(C, d, ksize, 61 + d)
    x = O.synth_bag(N, 62)
    params = [p[k].cuda() for k in EMB_KEYS] + [None] * 20
    cfg = ops.DiscConfig(C=C, d=d, t1=1, t2=d, ksize=ksize)
    bags = ops.PackedBags(x.cuda(), lengths)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        acts = ops.disc_embed_forward(cfg, params, bags, MODES[mode], save=True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert any("tc_rows_kernel" in n for n in names), "the embedding did not run on the tcgen05 engine"
    assert not any("gemm_simt_kernel" in n for n in names), "the embedding fell back to the FFMA engine"
    emb = acts["emb"].double().cpu()
    d_emb = torch.randn(N // 16, d, generator=torch.Generator().manual_seed(63))
    grads = [torch.empty_like(t) for t in params[:4]] + [None] * 20
    ops.disc_embed_backward(cfg, params, bags, acts, d_emb.cuda(), grads)
    ref, _ = _emb64(p, x.float() if mode != "bf16" else x.bfloat16().float(), ksize)
    tol = STAGE_TOL[mode]
    bound = tol * ref.abs() + tol * float(ref.abs().max())

    def caught(cand):
        return bool(((cand - ref).abs() > bound).any())
    lost, _ = _emb64(p, x.float(), ksize, drop_k=(0, KBLK[mode]))
    assert caught(lost), "the bound would not catch a lost K block"
    shifted = ref.clone()
    shifted[:8] = ref[1:9]                                  # one 128-row tile (8 regions) shifted by a region row
    assert caught(shifted), "the bound would not catch a one-row shift"
    assert not caught(emb), f"{mode} d={d} ksize={ksize}: {float((emb - ref).abs().max()):.3e}"
    # backward (LN-pool backward + weight gradient) against the float64 chain at the kernel's own saved y_pre (the ReLU
    # branches are the forward's), with the operands as the mode stores them
    xs = x.bfloat16().double() if mode == "bf16" else x.double()
    g64 = {k: p[k].double().requires_grad_(True) for k in EMB_KEYS}
    y = acts["y_pre"].double().cpu().requires_grad_(True)
    e = torch.relu(torch.nn.functional.layer_norm(y, (d,), g64["norm.weight"], g64["norm.bias"], 1e-5))
    (e.reshape(N // 16, 16, d).mean(1) * d_emb.double()).sum().backward()
    dy = y.grad.bfloat16().double() if mode == "bf16" else y.grad
    Wv = g64["conv.weight"]
    if ksize == 3:
        img = xs.reshape(N // 16, 4, 4, C).permute(0, 3, 1, 2)
        yy = torch.nn.functional.conv2d(img, Wv, g64["conv.bias"], padding=1).permute(0, 2, 3, 1).reshape(-1, d)
    else:
        yy = xs @ Wv.reshape(d, C).T + g64["conv.bias"]
    (yy * dy).sum().backward()
    rg = [g64[k].grad for k in EMB_KEYS]
    gtol = {"tf32": 5e-3, "tf32x3": 2e-5, "bf16": 2e-2}[mode]
    floor = 8 * grad_floor(rg) if mode == "tf32x3" else 0.0
    for k, a, r in zip(EMB_KEYS, grads, rg):
        assert_close(a.cpu(), r, gtol, f"grad {k}", atol=floor)


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("d", [64, 256])
def test_region_chain_vs_float64(d, mode):
    """f1, fi and the gate logits of the region chain (split-tf32 mma.sync) at d = 64 / 256: fp32-grade in every mode (the
    chain's inputs are fp32 in every mode), within 1e-5 of float64, ragged region counts across the 32 / 64-region CTAs."""
    C = 1024
    lengths = [4096 + 320, 48, 1600]
    N, R = sum(lengths), sum(lengths) // 16
    sd = O.synth_state_dict(_shapes(C, d, 1, False), 71 + d)
    D = build_D(C, d)
    D.load_state_dict(sd)
    D.eval()
    bags = ops.PackedBags.from_list([O.synth_bag(n, 72 + i).cuda() for i, n in enumerate(lengths)])
    cfg = D.config()
    params = D.disc_params()
    emb = ops.disc_embed_forward(cfg, params, bags, MODES[mode], save=False)["emb"]
    head = ops.disc_head_forward(cfg, params, bags, emb, torch.rand(3, device="cuda"), train=False, precision=MODES[mode])
    P = "net_pair_one."
    s = {k: v.double() for k, v in sd.items()}
    e = emb.double().cpu()
    f1 = torch.relu(e @ s[P + "fc1.0.weight"].T + s[P + "fc1.0.bias"])
    fi = f1 @ s[P + "fc1.3.weight"].T + s[P + "fc1.3.bias"]
    a = torch.tanh(fi @ s[P + "pool.fc1.0.weight"].T + s[P + "pool.fc1.0.bias"])
    b = torch.sigmoid(fi @ s[P + "pool.score.0.weight"].T + s[P + "pool.score.0.bias"])
    rep = ((a * b) @ s[P + "pool.fc2.weight"].T + s[P + "pool.fc2.bias"]).reshape(-1)
    # the same chain with one 16-wide K block of each contraction lost (the smallest weight stage, KC = 16)
    k0 = torch.ones(d, dtype=torch.float64)
    k0[:16] = 0
    kh = torch.ones(d // 2, dtype=torch.float64)
    kh[:16] = 0
    f1_l = torch.relu((e * k0) @ s[P + "fc1.0.weight"].T + s[P + "fc1.0.bias"])
    fi_l = (f1 * kh) @ s[P + "fc1.3.weight"].T + s[P + "fc1.3.bias"]
    a_l = torch.tanh((fi * k0) @ s[P + "pool.fc1.0.weight"].T + s[P + "pool.fc1.0.bias"])
    rep_l = ((a_l * b) @ s[P + "pool.fc2.weight"].T + s[P + "pool.fc2.bias"]).reshape(-1)
    for name, got, ref, lost in (("f1", head["f1"], f1, f1_l), ("fi", head["fi"], fi, fi_l), ("rep", head["rep"], rep, rep_l)):
        got = got.double().cpu()
        bound = 1e-5 * ref.abs() + 1e-5 * float(ref.abs().max())
        assert bool(((lost - ref).abs() > bound).any()), f"{name}: the bound would not catch a lost K block"
        shifted = ref.clone()
        shifted[:32] = ref[1:33]
        assert bool(((shifted - ref).abs() > bound).any()), f"{name}: the bound would not catch a one-row shift"
        assert not bool(((got - ref).abs() > bound).any()), f"{name} d={d} {mode}: {float((got - ref).abs().max()):.3e}"
    assert head["f1"].shape == (R, d // 2) and head["fi"].shape == (R, d)


# ---------------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------------
def test_bf16_refuses_unsupported_width_and_fp32_runs_it():
    C, d = 1024, 96
    sd = O.synth_state_dict(_shapes(C, d, 1, False), 81)
    D = build_D(C, d)
    D.load_state_dict(sd)
    D.eval()
    x = O.synth_bag(320, 82)
    bags = ops.PackedBags.from_single(x.cuda())
    t = torch.tensor([0.5], device="cuda")
    advmil_b200.set_precision("bf16")
    try:
        with pytest.raises(ops._lib.AdvmilError, match="bf16"):
            D.forward_packed(bags, t)
    finally:
        advmil_b200.set_precision("fp32")
    out = D.forward_packed(bags, t)
    ref = O.prjdisc_forward(sd, x, t.cpu().reshape(1, 1), None)["out"]
    assert_close(out.detach().cpu().reshape(-1), ref.detach().reshape(-1), RTOL, "out d=96", atol_scale=0.1)


# ---------------------------------------------------------------------------------------------------------------------
# one full D + G + Adam step against the oracle trainer
# ---------------------------------------------------------------------------------------------------------------------
def _cat_masks(per_bag, keys):
    return {k: torch.cat([m[k] for m in per_bag], dim=0).to(torch.uint8).contiguous().cuda() for k in keys}


def _step_vs_oracle(engine, d, precision):
    """One D + G + Adam step against the oracle trainer.  fp32: the case is moved off the discriminator's ReLU boundaries
    (_condition_disc, under the real / fake mask sets of the D phase and the mask-free G phase), then every D gradient is
    held at 1e-5 with the grad floor, and the D and G parameters after Adam at 1e-5.  bf16: the yardsticks of
    tests/test_gpu_bf16_step.py -- D gradients within 2e-2 of the fp32 oracle (its SENSITIVE tensors at SENSITIVE_TOL)
    and, for the ABMIL generator the storage oracle models, within EMU_TOL of the bf16-storage oracle for every tensor;
    after Adam, entries whose gradient is at least half of the tensor's largest agree with the fp32 trainer to 3e-3 lr (the
    first Adam step moves an entry by lr * sign(g): a wrong sign shows as 2 lr)."""
    from advmil_b200.step import AdvStep, ClusterAdvStep, EsatAdvStep, ModuleAdvStep
    from tests.test_gpu_bf16_step import EMU_TOL, _named_grads
    C, h = 1024, 384
    if engine in ("adv", "module"):
        mode, shapesG, Ns = "abmil", O.G_SHAPES(), [4096 + 160, 320, 96, 640]
    elif engine == "cluster":
        mode, shapesG, Ns = "cluster", O.G_CLUSTER_SHAPES(C, h), [160, 4096 + 320, 96, 640]
    else:
        mode, shapesG, Ns = "patch", O.G_ESAT_SHAPES(C, h), [160, 320, 96, 640]
    backbone = {"abmil": "abmil", "cluster": "cluster", "patch": "patch"}[mode]
    B = len(Ns)
    sdG, sdD = O.synth_state_dict(shapesG, 111 + d), O.synth_state_dict(O.D_SHAPES(C, d, (d // 2, d)), 112 + d)
    xs = [O.synth_bag(n, 120 + i, C) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 113)
    es[0] = 1.0
    vis = [True, True, False, True]
    rng = np.random.default_rng(114)
    nd = torch.tensor(rng.uniform(size=(B, h // 2)), dtype=torch.float32)
    ng = torch.tensor(rng.uniform(size=(B, h // 2)), dtype=torch.float32)
    kw, rkw = dict(noise_d=nd.cuda(), noise_g=ng.cuda()), {}
    mr = mf = mg = None
    if engine != "esat":
        mr = [d_masks(n // 16, d, 300 + 10 * i) for i, n in enumerate(Ns)]
        mf = [d_masks(n // 16, d, 400 + 10 * i) for i, n in enumerate(Ns)]
        if engine == "cluster":
            mg = [{"h": O.synth_masks((8, h), 0.75, 500 + 10 * i), "a": O.synth_masks((8, h), 0.75, 501 + 10 * i),
                   "b": O.synth_masks((8, h), 0.75, 502 + 10 * i), "mlp0": O.synth_masks((1, h // 2), 0.4, 503 + 10 * i)}
                  for i in range(B)]
            gkeys = ["h", "a", "b", "mlp0"]
            cids = [torch.tensor(rng.integers(0, 8, size=n), dtype=torch.float32) for n in Ns]
            kw["ext"] = torch.cat(cids).cuda()
            rkw["exts"] = cids
        else:
            mg = [g_masks(n, h, h, 500 + 10 * i) for i, n in enumerate(Ns)]
            gkeys = ["h", "a", "b", "rho", "mlp0"]
        kw.update(masks_d_real=_cat_masks(mr, ["fc1", "ga", "gs", "fc2"]), masks_d_fake=_cat_masks(mf, ["fc1", "ga", "gs", "fc2"]),
                  masks_g=_cat_masks(mg, gkeys))
    p_d = 0.0 if engine == "esat" else 0.25
    mask_sets = [[None] if mr is None else [mr[i], mf[i], None] for i in range(B)]
    if precision == "fp32":
        for _ in range(2):         # the ESAT generator's own ReLU boundaries as well (tests/util.py:condition_esat_case)
            if engine == "esat":
                sdG, xs = condition_esat_case(sdG, xs, None, [[None]] * B)
            sdD, xs = _condition_disc(sdD, xs, 1, mask_sets, p=p_d)
    else:                      # bf16: the MLPs' ReLUs (the embedding's tensors are SENSITIVE against the fp32 oracle)
        sdD, xs = _condition_disc(sdD, xs, 1, mask_sets, p=p_d, margin=0.0, region_margin=5e-4, bag_margin=2e-2)
    G, D = build_G((C, h, h), mode=mode), build_D(C, d)
    G.load_state_dict(sdG)
    D.load_state_dict(sdD)
    if engine == "esat":
        G.backbone.p = G.backbone.pool.p = 0.0
        G.p_head = 0.0
        D.net_pair_one.p = 0.0
    cls = {"adv": AdvStep, "module": ModuleAdvStep, "cluster": ClusterAdvStep, "esat": EsatAdvStep}[engine]
    eng = cls(G, D, precision=precision)
    pD0 = {k: v.detach().clone() for k, v in D.named_parameters()}
    pG0 = {k: v.detach().clone() for k, v in G.named_parameters()}
    tr = O.CpuTrainer(sdG, sdD, backbone=backbone)
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    rargs = (xs, ts, es, vis, list(nd), list(ng)) + (() if mr is None else (mr, mf, mg))
    ref = tr.step(*rargs, **rkw)
    out = eng.step(bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(), **kw)
    L = eng.loss_dict(out) if hasattr(eng, "loss_dict") else {k: float(out[k]) for k in ("dis_loss", "gen_loss", "gen_total_loss") if k in out}
    gD = _named_grads(D, eng.D)
    if precision == "bf16":
        for k, r in (("dis_loss", "dis_loss"), ("gen_total_loss", "total")):
            if k in L:
                assert abs(L[k] - ref[r]) <= 2e-2 * abs(ref[r]) + 1e-4, (k, L[k], ref[r])
        refs = [(ref, SENSITIVE_TOL, 2e-2, 1e-4, "fp32 oracle")]
        if mode == "abmil":
            tremu = O.CpuTrainer(sdG, sdD, backbone=backbone)
            with O.bf16_storage():
                refs.append((tremu.step(*rargs, **rkw), EMU_TOL, EMU_TOL, 2e-5, "bf16-storage oracle"))
        problems = []
        for rr, tol_s, tol, atol_f, tag in refs:
            gmax = max(float(v.abs().max()) for v in rr["d_grads"].values())
            for k, g in gD.items():
                if k.endswith(ZERO_GRAD):
                    continue
                g = g.detach().double().cpu()
                e = rr["d_grads"][k].double()
                t = tol_s if k.endswith(SENSITIVE) else tol
                err, scale = float((g - e).abs().max()), float(e.abs().max())
                if not err <= t * scale + atol_f * gmax:
                    problems.append(f"D grad {k} vs {tag}: {err:.3e} of {scale:.3e} (tol {t})")
        for net, mod, p0, sd_ref, key in (("D", D, pD0, tr.sdD, "d_grads"), ("G", G, pG0, tr.sdG, "g_grads")):
            for k, prm in mod.named_parameters():
                if k.endswith(ZERO_GRAD):
                    continue
                dp = (prm.detach() - p0[k]).cpu().double()
                dr = (sd_ref[k].detach() - (sdD if net == "D" else sdG)[k]).double()
                assert float(dp.abs().max()) <= (1.0 + 1e-3) * LR * 3.2, (net, k)
                gr = ref[key][k].double().abs()
                if float(gr.max()) == 0:
                    continue
                big = gr >= 0.5 * gr.max()
                dd = float((dp - dr)[big].abs().max())
                if not dd <= 3e-3 * LR:
                    problems.append(f"{net} param {k} after Adam: {dd / LR:.3e} lr")
        assert not problems, "\n".join(problems)
        return
    assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, "pred_d")
    assert_close(out["pred_g"].cpu(), ref["pred_g"].reshape(-1), RTOL, "pred_g")
    assert_close(out["f_fake_d"].cpu(), ref["fake_d"].reshape(-1), RTOL, "fake_d", atol_scale=1e-1)
    assert_close(out["f_fake_g"].cpu(), ref["fake_g"].reshape(-1), RTOL, "fake_g", atol_scale=1e-1)
    for k, r in (("dis_loss", "dis_loss"), ("gen_loss", "gen_loss"), ("gen_total_loss", "total")):
        if k in L:
            assert abs(L[k] - ref[r]) < 2e-5, (k, L[k], ref[r])
    floor = max(grad_floor(list(ref["d_grads"].values())), 2.0 ** -23 / B)
    small = {}
    for k, g in gD.items():
        if not k.endswith(ZERO_GRAD):
            assert_close(g.detach().cpu(), ref["d_grads"][k], RTOL, "D grad " + k, atol=8 * floor)
            small[k] = ref["d_grads"][k].abs() < 1e-3 * ref["d_grads"][k].abs().max()
    # post-Adam (as tests/test_gpu_disc_conv3.py): an entry whose gradient is a rounding-level remainder of cancelling terms
    # moves by about +-lr whatever its sign; those are bounded by the Adam move, the rest at 1e-5
    for k, prm in D.named_parameters():
        if not k.endswith(ZERO_GRAD):
            a, e, m = prm.detach().cpu(), tr.sdD[k].detach(), small[k]
            assert_close(a[~m], e[~m], RTOL, "D param " + k, atol=8e-5 * 2e-2)
            if bool(m.any()):
                assert float((a[m] - e[m]).abs().max()) <= 2 * 8e-5, k
    for k, prm in G.named_parameters():
        if not k.endswith(ZERO_GRAD):
            a, e = prm.detach().cpu(), tr.sdG[k].detach()
            gr = ref["g_grads"][k].abs()
            m = gr < 1e-3 * gr.max()
            assert_close(a[~m], e[~m], RTOL, "G param " + k, atol=8e-5 * 2e-2)
            if bool(m.any()):
                assert float((a[m] - e[m]).abs().max()) <= 2 * 8e-5, k


@pytest.mark.parametrize("engine,d,precision", [
    ("adv", 64, "fp32"), ("adv", 256, "fp32"), ("adv", 64, "bf16"), ("adv", 256, "bf16"),
    ("module", 256, "fp32"), ("esat", 256, "fp32"), ("cluster", 256, "fp32"),
    ("module", 256, "bf16"), ("esat", 256, "bf16"), ("cluster", 256, "bf16"),
])
def test_disc_width_step_vs_oracle_trainer(engine, d, precision):
    _step_vs_oracle(engine, d, precision)

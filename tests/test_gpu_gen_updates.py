"""GPU: `gen_updates` G updates per D update (model/model_handler.py:328-335) in every adversarial step engine -- AdvStep,
ClusterAdvStep, EsatAdvStep (advmil_adv_step*_gen, then advmil_adv_step*_gen_next per further update) and ModuleAdvStep --
against the oracle's restatement of `_update_disc` followed by gen_updates x `_update_gen`, with the tolerances of the
existing step tests (tests/test_gpu_step.py, tests/test_gpu_cluster_step.py, tests/test_gpu_bf16_step.py)."""
import itertools

import numpy as np
import pytest
import torch

from oracle import advmil_oracle as O
from tests.util import assert_close, build_D, build_G, d_masks, esat_masks, g_masks

pytestmark = pytest.mark.gpu
RTOL = 1e-5
ZERO_GRAD = ("pool.fc2.bias", "attention_c.bias")
DKEYS = ["fc1", "ga", "gs", "fc2"]


class GenUpdatesTrainer(O.CpuTrainer):
    """CpuTrainer with `gen_updates` G updates after the D update: one `_update_gen` per update, each with its own noise and
    generator masks, D in eval mode with its post-update parameters.  Per update: t_reg, gen_loss, total (recon + coef_gan
    x gen + coef_l1 x sum|W_G|), sum|W_G| before that update's Adam step, pred_g and D(x, pred_g); the G gradients of the
    later updates with loss_reg_l1's sub-gradient coef_l1 x sign(W_G) taken out (the CUDA engines apply it in the Adam kernel)."""

    def l1(self):
        return float(sum(float(v.detach().abs().sum()) for v in self.sdG.values()))

    def step_k(self, bags, ts, es, visible, noise_d, noise_gs, d_masks_real=None, d_masks_fake=None, g_masks=None, exts=None):
        g_masks = g_masks or [None] * len(noise_gs)
        l1 = self.l1()                     # G does not change in the D phase
        ref = self.step(bags, ts, es, visible, noise_d, noise_gs[0], d_masks_real, d_masks_fake, g_masks[0], exts)
        gens = [dict(ref, l1=l1)]
        for ng, mg in zip(noise_gs[1:], g_masks[1:]):
            l1 = self.l1()
            sign = {k: torch.sign(v.detach()) for k, v in self.sdG.items()}
            nzg = [[None, n.reshape(1, -1)] for n in ng]
            g = O.gen_step_loss(self.sdG, self.sdD, bags, ts, es, visible, nzg, mg, self.coef_gan, self.coef_l1, exts=exts,
                                backbone=self.backbone)
            self.optG.zero_grad()
            for v in self.sdD.values():
                v.grad = None
            g["loss"].backward()
            g_grads = {k: v.grad.clone() - self.coef_l1 * sign[k] for k, v in self.sdG.items()}
            self.optG.step()
            gens.append({"gen_loss": float(g["gen_loss"]), "t_reg": float(g["t_reg"]), "total": float(g["loss"]), "l1": l1,
                         "pred_g": g["pred"].detach(), "fake_g": g["fake"].detach(), "g_grads": g_grads})
        return ref, gens


def _cat(per_bag, keys):
    return {k: torch.cat([m[k] for m in per_bag], dim=0).to(torch.uint8).contiguous().cuda() for k in keys}


def _check_gen_losses(gl, gens, coef_l1, tol, where):
    """gen_losses rows (t_reg, gen, t_reg + coef_gan * gen, sum|W_G|) against the oracle's per-update values."""
    gl = gl.detach().double().cpu().numpy()
    assert gl.shape == (len(gens), 4), gl.shape
    for u, r in enumerate(gens):
        assert abs(gl[u, 0] - r["t_reg"]) < tol, (where, u, "t_reg", gl[u, 0], r["t_reg"])
        assert abs(gl[u, 1] - r["gen_loss"]) < tol, (where, u, "gen", gl[u, 1], r["gen_loss"])
        assert abs(gl[u, 2] + coef_l1 * gl[u, 3] - r["total"]) < tol, (where, u, "total", gl[u, 2], r["total"])
        assert abs(gl[u, 3] - r["l1"]) <= 1e-5 * r["l1"], (where, u, "l1", gl[u, 3], r["l1"])


def _check_params(G, D, tr, adam_steps):
    """Post-Adam parameters.  Adam moves an entry whose gradient is at the rounding level of its tensor by up to lr per step,
    in a direction that rounding decides; over `adam_steps` G steps a few such entries of the first layers (and, through
    pred_g, of D) drift apart by a few hundredths of lr per step: the floor is 5e-2 lr per G Adam step (the two-step tests
    of tests/test_gpu_step.py use 2e-2 lr per step)."""
    atol = 8e-5 * adam_steps * 5e-2
    for k, p in D.named_parameters():
        if not k.endswith(ZERO_GRAD):
            assert_close(p.detach().cpu(), tr.sdD[k].detach(), RTOL, "D param " + k, atol=atol)
    for k, p in G.named_parameters():
        if not k.endswith(ZERO_GRAD):
            assert_close(p.detach().cpu(), tr.sdG[k].detach(), RTOL, "G param " + k, atol=atol)


def _nets(kind, sdG, sdD, C=1024, h=384):
    G, D = build_G((C, h, h), mode=kind), build_D()
    G.load_state_dict(sdG)
    D.load_state_dict(sdD)
    return G, D


# ---------------------------------------------------------------------------------------------------------------------
# the C-fused ABMIL and DeepAttMISL steps: fp32 and tf32x3, injected masks per update, ragged bags, an unlabelled bag
# (and an empty cluster), two optimiser steps
# ---------------------------------------------------------------------------------------------------------------------
def _case(kind):
    h = 384
    if kind == "abmil":
        Ns = [160, 320, 96, 640, 48]
        sdG, sdD = O.synth_state_dict(O.G_SHAPES(), 41), O.synth_state_dict(O.D_SHAPES(), 42)
        vis = [True, True, False, True, True]
        exts = None
    else:
        Ns = [160, 320, 96]
        sdG, sdD = O.synth_state_dict(O.G_CLUSTER_SHAPES(1024, h), 43), O.synth_state_dict(O.D_SHAPES(), 44)
        vis = [True, False, True]
        rng = np.random.default_rng(45)
        exts = [torch.tensor(rng.integers(0, 8, size=n), dtype=torch.float32) for n in Ns]
        exts[1][exts[1] == 5] = 4.0        # cluster 5 of bag 1 is empty (model/backbone.py:114-115)
    xs = [O.synth_bag(n, 46 + i) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(len(Ns), 47)
    es[0] = 1.0
    return Ns, sdG, sdD, xs, ts, es, vis, exts


def _gmask(kind, Ns, seed, h=384):
    if kind == "abmil":
        return [g_masks(n, h, h, seed + 10 * i) for i, n in enumerate(Ns)]
    return [{"h": O.synth_masks((8, h), 0.75, seed + 10 * i), "a": O.synth_masks((8, h), 0.75, seed + 10 * i + 1),
             "b": O.synth_masks((8, h), 0.75, seed + 10 * i + 2), "mlp0": O.synth_masks((1, h // 2), 0.4, seed + 10 * i + 3)}
            for i in range(len(Ns))]


GKEYS = {"abmil": ["h", "a", "b", "rho", "mlp0"], "cluster": ["h", "a", "b", "mlp0"]}


@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("prec", ["fp32", "tf32x3"])
@pytest.mark.parametrize("kind", ["abmil", "cluster"])
def test_fused_step_gen_updates_vs_oracle_trainer(kind, prec, k):
    from advmil_b200 import ops
    from advmil_b200.step import AdvStep, ClusterAdvStep
    Ns, sdG, sdD, xs, ts, es, vis, exts = _case(kind)
    B = len(Ns)
    tr = GenUpdatesTrainer(sdG, sdD, backbone=kind)
    G, D = _nets(kind, sdG, sdD)
    eng = (AdvStep if kind == "abmil" else ClusterAdvStep)(G, D, precision=prec, gen_updates=k)
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    kw = {} if exts is None else {"ext": torch.cat(exts).cuda()}
    for step in range(2):
        rng = np.random.default_rng(60 + step)
        nd = torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32)
        ngs = [torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32) for _ in range(k)]
        mr = [d_masks(n // 16, 128, 300 + 10 * i + step) for i, n in enumerate(Ns)]
        mf = [d_masks(n // 16, 128, 400 + 10 * i + step) for i, n in enumerate(Ns)]
        mgs = [_gmask(kind, Ns, 500 + 100 * u + step) for u in range(k)]
        ref, gens = tr.step_k(xs, ts, es, vis, list(nd), [list(n) for n in ngs], mr, mf, mgs, exts=exts)
        out = eng.step(bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(), noise_d=nd.cuda(),
                       noise_g=[n.cuda() for n in ngs], masks_d_real=_cat(mr, DKEYS), masks_d_fake=_cat(mf, DKEYS),
                       masks_g=[_cat(m, GKEYS[kind]) for m in mgs], **kw)
        L = eng.loss_dict(out)
        assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, f"pred_d {step}")
        assert_close(out["pred_g"].cpu(), gens[-1]["pred_g"].reshape(-1), RTOL, f"pred_g {step}")
        assert_close(out["f_fake_g"].cpu(), gens[-1]["fake_g"].reshape(-1), RTOL, f"fake_g {step}", atol_scale=1e-1)
        assert abs(L["dis_loss"] - ref["dis_loss"]) < 2e-5
        assert abs(L["gen_loss"] - gens[-1]["gen_loss"]) < 2e-5 and abs(L["t_reg_loss"] - gens[-1]["t_reg"]) < 2e-5
        assert abs(L["gen_total_loss"] - gens[-1]["total"]) < 2e-5
        _check_gen_losses(out["gen_losses"], gens, eng.coef_l1, 2e-5, f"{kind} {prec} step {step}")
    assert eng.G.step_count == 2 * k and eng.D.step_count == 2
    _check_params(G, D, tr, 2 * k)


def _esat_nets_without_dropout(C, d, seed_g, seed_d):
    sdG, sdD = O.synth_state_dict(O.G_ESAT_SHAPES(C, d), seed_g), O.synth_state_dict(O.D_SHAPES(), seed_d)
    G, D = _nets("patch", sdG, sdD, C, d)
    G.backbone.p = G.backbone.pool.p = 0.0          # the C step draws its own dropout bits: compare the deterministic arithmetic
    G.p_head = 0.0
    D.net_pair_one.p = 0.0
    return sdG, sdD, G, D


@pytest.mark.parametrize("k", [2, 3])
def test_c_fused_esat_step_gen_updates_vs_oracle_trainer(k):
    """EsatAdvStep in fp32 with the dropout probabilities zeroed (as test_c_fused_esat_step_vs_oracle_trainer_and_module_step):
    every later G update recomputes the patch embedding from the updated parameters."""
    from advmil_b200 import ops
    from advmil_b200.step import EsatAdvStep
    C, d = 1024, 384
    Ns = [160, 320, 96, 640]
    B = len(Ns)
    sdG, sdD, G, D = _esat_nets_without_dropout(C, d, 171, 172)
    tr = GenUpdatesTrainer(sdG, sdD, backbone="patch")
    eng = EsatAdvStep(G, D, gen_updates=k)
    xs = [O.synth_bag(n, 180 + i, C) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 173)
    es[0] = 1.0
    vis = [True, True, False, True]
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    for step in range(2):
        rng = np.random.default_rng(174 + step)
        nd = torch.tensor(rng.uniform(size=(B, d // 2)), dtype=torch.float32)
        ngs = [torch.tensor(rng.uniform(size=(B, d // 2)), dtype=torch.float32) for _ in range(k)]
        ref, gens = tr.step_k(xs, ts, es, vis, list(nd), [list(n) for n in ngs])
        out = eng.step(bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(), noise_d=nd.cuda(),
                       noise_g=[n.cuda() for n in ngs])
        L = eng.loss_dict(out)
        assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, f"pred_d {step}")
        assert_close(out["pred_g"].cpu(), gens[-1]["pred_g"].reshape(-1), RTOL, f"pred_g {step}")
        assert_close(out["f_fake_g"].cpu(), gens[-1]["fake_g"].reshape(-1), RTOL, f"fake_g {step}", atol_scale=1e-1)
        assert abs(L["dis_loss"] - ref["dis_loss"]) < 2e-5 and abs(L["gen_total_loss"] - gens[-1]["total"]) < 2e-5
        _check_gen_losses(out["gen_losses"], gens, eng.coef_l1, 2e-5, f"esat step {step}")
    _check_params(G, D, tr, 2 * k)


@pytest.mark.parametrize("kind", ["abmil", "cluster", "patch"])
def test_module_step_gen_updates_vs_oracle_trainer(kind):
    """ModuleAdvStep with each generator backbone, gen_updates = 2, injected masks at every dropout site of every update."""
    from advmil_b200 import ops
    from advmil_b200.step import ModuleAdvStep
    k, h = 2, 384
    if kind == "patch":
        Ns, vis = [160, 320, 96, 640], [True, True, False, True]
        sdG, sdD = O.synth_state_dict(O.G_ESAT_SHAPES(1024, h), 131), O.synth_state_dict(O.D_SHAPES(), 132)
        xs = [O.synth_bag(n, 140 + i) for i, n in enumerate(Ns)]
        ts, es = O.synth_labels(len(Ns), 133)
        es[0] = 1.0
        exts = None
    else:
        Ns, sdG, sdD, xs, ts, es, vis, exts = _case(kind)
    B = len(Ns)
    tr = GenUpdatesTrainer(sdG, sdD, backbone=kind)
    G, D = _nets(kind, sdG, sdD)
    eng = ModuleAdvStep(G, D, gen_updates=k)
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    for step in range(2):
        rng = np.random.default_rng(70 + step)
        nd = torch.tensor(rng.uniform(size=(B, h // 2)), dtype=torch.float32)
        ngs = [torch.tensor(rng.uniform(size=(B, h // 2)), dtype=torch.float32) for _ in range(k)]
        mr = [d_masks(n // 16, 128, 600 + 10 * i + step) for i, n in enumerate(Ns)]
        mf = [d_masks(n // 16, 128, 700 + 10 * i + step) for i, n in enumerate(Ns)]
        if kind == "patch":
            mgs = [[esat_masks(n // 16, h, 800 + 100 * u + 10 * i + step) for i, n in enumerate(Ns)] for u in range(k)]
            mgd = []
            for m in mgs:
                dm = _cat(m, ["sa", "ff1", "ff2", "ga", "gs", "mlp0"])
                dm["attn"] = [mi["attn"].to(torch.uint8).cuda() for mi in m]
                mgd.append(dm)
        else:
            mgs = [_gmask(kind, Ns, 800 + 100 * u + step) for u in range(k)]
            mgd = [_cat(m, GKEYS[kind]) for m in mgs]
        ref, gens = tr.step_k(xs, ts, es, vis, list(nd), [list(n) for n in ngs], mr, mf, mgs, exts=exts)
        kw = {} if exts is None else {"ext": torch.cat(exts).cuda()}
        out = eng.step(bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(), noise_d=nd.cuda(),
                       noise_g=[n.cuda() for n in ngs], masks_d_real=_cat(mr, DKEYS), masks_d_fake=_cat(mf, DKEYS), masks_g=mgd, **kw)
        assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, f"pred_d {step}")
        assert_close(out["pred_g"].cpu(), gens[-1]["pred_g"].reshape(-1), RTOL, f"pred_g {step}")
        assert_close(out["f_fake_g"].cpu(), gens[-1]["fake_g"].reshape(-1), RTOL, f"fake_g {step}", atol_scale=1e-1)
        assert abs(float(out["dis_loss"]) - ref["dis_loss"]) < 2e-5
        assert abs(float(out["gen_total_loss"]) - gens[-1]["total"]) < 2e-5
        _check_gen_losses(out["gen_losses"], gens, eng.coef_l1, 2e-5, f"module {kind} step {step}")
    assert eng.G.step_count == 2 * k and eng.D.step_count == 2
    _check_params(G, D, tr, 2 * k)


def test_bf16_fused_step_gen_updates_vs_bf16_storage_oracle():
    """bf16 AdvStep at gen_updates = 2, one optimiser step, at the bounds of tests/test_gpu_bf16_step.py: losses of both G
    updates within 2e-2 of the fp32 oracle, D gradients (before any G update) against the fp32 and the bf16-storage
    oracle, the last G update's gradients against the bf16-storage oracle (which holds the same post-Adam parameters up to
    Adam's lr-sized steps of near-zero gradients), and every Adam move bounded by lr x ~3.16 per update."""
    from advmil_b200 import ops
    from advmil_b200.step import AdvStep
    from tests.test_gpu_bf16_step import EMU_TOL, LR, SENSITIVE, SENSITIVE_TOL, TOL, _named_grads
    k = 2
    Ns = [320, 1600, 48, 16, 2048, 640]
    B = len(Ns)
    sdG, sdD = O.synth_state_dict(O.G_SHAPES(), 311), O.synth_state_dict(O.D_SHAPES(), 312)
    xs = [O.synth_bag(n, 320 + i) for i, n in enumerate(Ns)]
    ts, es = O.synth_labels(B, 313)
    es[0], es[1] = 1.0, 0.0
    vis = [True] * B
    vis[2] = False
    G, D = _nets("abmil", sdG, sdD)
    eng = AdvStep(G, D, precision="bf16", gen_updates=k)
    tr32, tremu = GenUpdatesTrainer(sdG, sdD), GenUpdatesTrainer(sdG, sdD)
    rng = np.random.default_rng(314)
    nd = torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32)
    ngs = [torch.tensor(rng.uniform(size=(B, 192)), dtype=torch.float32) for _ in range(k)]
    mr = [d_masks(n // 16, 128, 400 + 10 * i) for i, n in enumerate(Ns)]
    mf = [d_masks(n // 16, 128, 500 + 10 * i) for i, n in enumerate(Ns)]
    mgs = [[g_masks(n, 384, 384, 600 + 100 * u + 10 * i) for i, n in enumerate(Ns)] for u in range(k)]
    pG0 = {kk: v.detach().clone() for kk, v in G.named_parameters()}
    ref, gens = tr32.step_k(xs, ts, es, vis, list(nd), [list(n) for n in ngs], mr, mf, mgs)
    with O.bf16_storage():
        emu, emu_gens = tremu.step_k(xs, ts, es, vis, list(nd), [list(n) for n in ngs], mr, mf, mgs)
    out = eng.step(ops.PackedBags.from_list([x.cuda() for x in xs]), ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda(),
                   noise_d=nd.cuda(), noise_g=[n.cuda() for n in ngs], masks_d_real=_cat(mr, DKEYS), masks_d_fake=_cat(mf, DKEYS),
                   masks_g=[_cat(m, GKEYS["abmil"]) for m in mgs])
    L = eng.loss_dict(out)
    assert abs(L["dis_loss"] - ref["dis_loss"]) < TOL
    gl = out["gen_losses"].double().cpu().numpy()
    for u in range(k):
        assert abs(gl[u, 2] + eng.coef_l1 * gl[u, 3] - gens[u]["total"]) < TOL, (u, gl[u], gens[u]["total"])
        assert abs(gl[u, 0] - gens[u]["t_reg"]) < TOL, (u, gl[u], gens[u]["t_reg"])
    problems = []
    gd = _named_grads(D, eng.D)
    gmax32 = max(float(v.abs().max()) for v in ref["d_grads"].values())
    gmaxe = max(float(v.abs().max()) for v in emu["d_grads"].values())
    for kk, gcu in gd.items():
        if kk.endswith(ZERO_GRAD):
            continue
        g = gcu.detach().double().cpu()
        e32, s32 = float((g - ref["d_grads"][kk].double()).abs().max()), float(ref["d_grads"][kk].abs().max())
        ee, se = float((g - emu["d_grads"][kk].double()).abs().max()), float(emu["d_grads"][kk].abs().max())
        tol = SENSITIVE_TOL if kk.endswith(SENSITIVE) else TOL
        if not e32 <= tol * s32 + 1e-4 * gmax32:
            problems.append(f"D grad {kk} vs fp32 oracle: {e32:.3e} of {s32:.3e}")
        if not ee <= EMU_TOL * se + 2e-5 * gmaxe:
            problems.append(f"D grad {kk} vs bf16-storage oracle: {ee:.3e} of {se:.3e}")
    gg = _named_grads(G, eng.G)
    eg = emu_gens[-1]["g_grads"]
    gmaxe = max(float(v.abs().max()) for v in eg.values())
    for kk, gcu in gg.items():
        if kk.endswith(ZERO_GRAD):
            continue
        g = gcu.detach().double().cpu()          # the oracle's later-update gradients are given without loss_reg_l1's term
        tol = SENSITIVE_TOL if kk.endswith(SENSITIVE) else TOL
        ee, se = float((g - eg[kk].double()).abs().max()), float(eg[kk].abs().max())
        if not ee <= tol * se + 1e-4 * gmaxe:
            problems.append(f"last G update grad {kk} vs bf16-storage oracle: {ee:.3e} of {se:.3e}")
    for kk, p in G.named_parameters():
        assert float((p.detach() - pG0[kk]).abs().max()) <= (1.0 + 1e-3) * LR * k * 3.2, kk
    assert not problems, "\n".join(problems)


# ---------------------------------------------------------------------------------------------------------------------
# determinism, noise order, reuse of D's embedding, argument checks
# ---------------------------------------------------------------------------------------------------------------------
def _bf16_engine(kind, k):
    """A small bf16 engine of each kind with in-kernel dropout, its step inputs and step kwargs."""
    from advmil_b200 import ops
    from advmil_b200.step import AdvStep, ClusterAdvStep, EsatAdvStep
    h = 384
    Ns = [1040, 4112, 48, 16]
    shapes = {"abmil": O.G_SHAPES(), "cluster": O.G_CLUSTER_SHAPES(1024, h), "patch": O.G_ESAT_SHAPES(1024, h)}[kind]
    G, D = _nets(kind, O.synth_state_dict(shapes, 81), O.synth_state_dict(O.D_SHAPES(), 82))
    cls = {"abmil": AdvStep, "cluster": ClusterAdvStep, "patch": EsatAdvStep}[kind]
    eng = cls(G, D, precision="bf16", gen_updates=k)
    seeds = itertools.count(777)
    eng._seed = lambda: next(seeds)
    bags = ops.PackedBags.from_list([O.synth_bag(n, 90 + i).cuda() for i, n in enumerate(Ns)])
    ts, es = O.synth_labels(len(Ns), 83)
    kw = {}
    if kind == "cluster":
        kw["ext"] = torch.randint(0, 8, (sum(Ns),), generator=torch.Generator().manual_seed(3), dtype=torch.int32).cuda()
    return eng, (bags, ts.cuda(), es.cuda(), torch.ones(len(Ns), dtype=torch.uint8).cuda()), kw


@pytest.mark.parametrize("kind", ["abmil", "cluster", "patch"])
def test_seeded_gen_updates_steps_repeat_bit_for_bit(kind):
    k = 3
    runs = []
    for _ in range(2):
        eng, args, kw = _bf16_engine(kind, k)
        rng = np.random.default_rng(5)
        outs = []
        for s in range(2):
            nz = [torch.tensor(rng.uniform(size=(4, 192)), dtype=torch.float32).cuda() for _ in range(k + 1)]
            outs.append(eng.step(*args, noise_d=nz[0], noise_g=nz[1:], **kw))
        torch.cuda.synchronize()
        runs.append((outs, eng.G.flat.clone(), eng.D.flat.clone()))
    (o1, g1, d1), (o2, g2, d2) = runs
    for a, b in zip(o1, o2):
        for key in ("losses", "gen_losses", "pred_d", "pred_g", "f_d", "f_fake_g"):
            assert torch.equal(a[key], b[key]), key
    assert torch.equal(g1, g2) and torch.equal(d1, d2)
    # the later updates did run: their losses differ from the first update's
    assert not torch.equal(o1[0]["gen_losses"][0], o1[0]["gen_losses"][1])


@pytest.mark.parametrize("kind", ["abmil", "cluster", "patch"])
def test_engine_noise_equals_explicit_draws_in_order(kind):
    """With no noise given the engine draws the D phase's [bags, hid] noise, then one per G update, from the CPU generator."""
    k = 3
    eng, args, kw = _bf16_engine(kind, k)
    torch.manual_seed(2024)
    o1 = eng.step(*args, **kw)
    torch.cuda.synchronize()
    res1 = (o1["gen_losses"].clone(), o1["pred_d"].clone(), o1["pred_g"].clone(), eng.G.flat.clone())
    eng2, args2, kw2 = _bf16_engine(kind, k)
    torch.manual_seed(2024)
    nb = args2[0].bags
    draws = [eng2.netG.draw_noise(nb, "cuda", False)[1] for _ in range(k + 1)]
    o2 = eng2.step(*args2, noise_d=draws[0], noise_g=draws[1:], **kw2)
    torch.cuda.synchronize()
    res2 = (o2["gen_losses"], o2["pred_d"], o2["pred_g"], eng2.G.flat)
    for a, b in zip(res1, res2):
        assert torch.equal(a, b)


def test_d_embedding_runs_once_per_step_for_any_gen_updates():
    """The stage profiler's embed_fwd launches per step do not grow with gen_updates for the ABMIL and DeepAttMISL steps (D's
    region embedding of the G phase is reused by the later updates); the ESAT step adds exactly its own patch embedding
    (recomputed from the updated G) per further update."""
    from advmil_b200 import _lib
    lib = _lib.load()
    import ctypes as C
    n = len(_lib.PROF_TAGS)
    emb = _lib.PROF_TAGS.index("embed_fwd")

    def embed_launches(kind, k):
        eng, args, kw = _bf16_engine(kind, k)
        eng.step(*args, **kw)                         # warm-up (workspace, side stream)
        torch.cuda.synchronize()
        ms, cnt = (C.c_double * n)(), (C.c_int64 * n)()
        lib.advmil_profile_read(ms, cnt, n)
        lib.advmil_profile_enable(1)
        try:
            eng.step(*args, **kw)
            torch.cuda.synchronize()
        finally:
            lib.advmil_profile_enable(0)
        lib.advmil_profile_read(ms, cnt, n)
        return int(cnt[emb])

    for kind in ("abmil", "cluster", "patch"):
        c = [embed_launches(kind, k) for k in (1, 2, 3)]
        assert c[0] >= 1, (kind, c)
        if kind == "patch":
            assert c == [c[0], c[0] + 1, c[0] + 2], (kind, c)
        else:
            assert c == [c[0]] * 3, (kind, c)


@pytest.mark.parametrize("kind", ["abmil", "cluster", "patch"])
def test_one_update_step_returns_the_outputs_of_a_one_update_step(kind):
    """gen_updates = 1 (the default) returns the same output entries as a step without the setting: gen_losses only appears
    with several G updates (bench.py --dump-outputs writes every tensor of the step's result)."""
    eng, args, kw = _bf16_engine(kind, 1)
    out = eng.step(*args, **kw)
    assert set(out) == {"losses", "pred_d", "pred_g", "f_d", "f_fake_g", "real_mask", "f_fake_d", "f_real", "_keep"}, sorted(out)
    assert out["losses"].shape == (8,)
    eng2, args2, kw2 = _bf16_engine(kind, 2)
    assert eng2.step(*args2, **kw2)["gen_losses"].shape == (2, 4)


def test_gen_updates_argument_checks():
    from advmil_b200.step import AdvStep, ClusterAdvStep, EsatAdvStep, ModuleAdvStep
    h = 384
    for cls, kind, shapes in ((AdvStep, "abmil", O.G_SHAPES()), (ClusterAdvStep, "cluster", O.G_CLUSTER_SHAPES(1024, h)),
                              (EsatAdvStep, "patch", O.G_ESAT_SHAPES(1024, h)), (ModuleAdvStep, "abmil", O.G_SHAPES())):
        for bad in (0, -1, 1.5, 2.0, "2", True, None):
            G, D = _nets(kind, O.synth_state_dict(shapes, 1), O.synth_state_dict(O.D_SHAPES(), 2))
            with pytest.raises(ValueError, match="gen_updates"):
                cls(G, D, gen_updates=bad)
    nz = torch.rand(4, 192, device="cuda")
    for kind in ("abmil", "cluster"):
        eng, args, kw = _bf16_engine(kind, 2)
        with pytest.raises(ValueError, match="noise_g"):
            eng.step(*args, noise_g=nz, **kw)                        # one tensor for two updates
        with pytest.raises(ValueError, match="noise_g"):
            eng.step(*args, noise_g=[nz, nz, nz], **kw)
        with pytest.raises(ValueError, match="masks_g"):
            eng.step(*args, noise_g=[nz, nz], masks_g={}, **kw)      # one mask set for two updates
        with pytest.raises(ValueError, match="masks_g"):
            eng.step(*args, noise_g=[nz, nz], masks_g=[{}], **kw)
    eng, args, kw = _bf16_engine("patch", 1)
    with pytest.raises(ValueError, match="noise_g"):
        eng.step(*args, noise_g=[nz, nz])
    G, D = _nets("abmil", O.synth_state_dict(O.G_SHAPES(), 1), O.synth_state_dict(O.D_SHAPES(), 2))
    mod = ModuleAdvStep(G, D, gen_updates=3)
    with pytest.raises(ValueError, match="noise_g"):
        mod.step(*args, noise_g=[nz, nz])


# ---------------------------------------------------------------------------------------------------------------------
# data parallel
# ---------------------------------------------------------------------------------------------------------------------
def _run_dp(rank, world, port, q):
    from advmil_b200 import ops
    from advmil_b200.dataset.packed import shard_bags_balanced
    from advmil_b200.step import AdvStep
    from tests.test_gpu_dp import NS, _build, _inputs
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        torch.distributed.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                                             device_id=dev)
    G, D = _build(dev)
    eng = AdvStep(G, D, gen_updates=2)
    xs, t, e, vis, nd, ng = _inputs()
    ng2 = torch.tensor(np.random.default_rng(7).uniform(size=ng.shape), dtype=torch.float32)
    mine = shard_bags_balanced(NS, world)[rank]
    bags = ops.PackedBags.from_list([xs[i].to(dev) for i in mine])
    out = eng.step(bags, t[mine].to(dev), e[mine].to(dev), vis[mine].to(dev), noise_d=nd[mine].to(dev),
                   noise_g=[ng[mine].to(dev), ng2[mine].to(dev)])
    torch.cuda.synchronize()
    gl = out["gen_losses"].clone()
    if world > 1:
        part = gl[:, :3].contiguous()                    # loss kernels write rank-local contributions; sum|W_G| is global
        torch.distributed.all_reduce(part)
        gl[:, :3] = part
    if rank == 0:
        q.put((eng.G.grad.cpu().numpy(), eng.D.grad.cpu().numpy(), gl.cpu().numpy(), eng.G.flat.cpu().numpy()))
    if world > 1:
        torch.distributed.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_gen_updates_step_equals_single_rank():
    from tests.test_gpu_dp import _launch
    res = {world: _launch(_run_dp, world) for world in (1, 2)}
    g1, d1, l1, p1 = res[1]
    g2, d2, l2, p2 = res[2]
    assert float(np.abs(g1 - g2).max()) <= 1e-5 * float(np.abs(g1).max())
    assert float(np.abs(d1 - d2).max()) <= 1e-5 * float(np.abs(d1).max())
    assert float(np.abs(l1 - l2).max()) <= 1e-5 * max(1.0, float(np.abs(l1).max()))
    assert float(np.abs(p1 - p2).max()) <= 4 * 8e-5

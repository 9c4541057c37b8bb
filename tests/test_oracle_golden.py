"""CPU: the oracle restatement against the golden fixtures written by the live reference (oracle/make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import advmil_oracle as O
from tests.util import d_masks, esat_masks, g_masks, golden, sub


def _grads_match(sdr, g, prefix="grad.", skip=()):
    for k, v in sdr.items():
        if k.endswith(skip) and skip:
            continue
        ref = g[prefix + k]
        scale = max(float(np.abs(ref).max()), 1e-6)
        assert float(np.abs(sub(v.grad) - ref).max()) <= 2e-5 * scale + 2e-9, k


@pytest.mark.parametrize("name", ["g_abmil_eval_full", "g_abmil_train_full", "g_abmil_eval_small", "g_abmil_train_small"])
def test_generator_oracle_vs_reference(name):
    g = golden(name)
    C, h, o, N, train, seed, nonneg = [int(v) for v in g["cfg"]]
    sd = {k: v.requires_grad_(True) for k, v in O.synth_state_dict(O.G_SHAPES(C, h, o), seed).items()}
    x = O.synth_bag(N, seed, C, bool(nonneg))
    noise = torch.tensor(np.random.default_rng(seed + 7).uniform(size=(1, o // 2)), dtype=torch.float32)
    masks = g_masks(N, h, o, seed * 10) if train else None
    out = O.generator_forward(sd, x, [None, noise], (0, 1), masks)
    out["pred"].sum().backward()
    assert float(np.abs(out["pred"].detach().numpy() - g["pred"]).max()) < 1e-6
    assert float(np.abs(out["z"].detach().numpy() - g["z"]).max()) < 1e-5
    assert float(np.abs(out["H"].detach().numpy() - g["H"]).max()) < 1e-5
    assert float(np.abs(sub(out["s"]) - g["s"]).max()) < 1e-5
    _grads_match(sd, g)


@pytest.mark.parametrize("name", ["d_rlip_eval_full", "d_rlip_train_full", "d_rlip_eval_small", "d_bag_train_small"])
def test_discriminator_oracle_vs_reference(name):
    g = golden(name)
    C, d, N, train, seed, inst, prjx = [int(v) for v in g["cfg"]]
    ty = (64, 128) if d == 128 else (d // 2, d)
    sd = {k: v.requires_grad_(True) for k, v in O.synth_state_dict(O.D_SHAPES(C, d, ty), seed + 50).items()}
    x = O.synth_bag(N, seed, C)
    t = torch.tensor([[0.37]], requires_grad=True)
    masks = d_masks(N // 16, d, seed * 10 + 5) if train else None
    out = O.prjdisc_forward(sd, x, t, masks, "instance" if inst else "bag", "x" if prjx else "y")
    out["out"].sum().backward()
    assert float(np.abs(out["out"].detach().numpy() - g["out"]).max()) < 1e-6
    assert float(np.abs(sub(out["emb"], 2048) - g["emb"]).max()) < 1e-5
    assert float(np.abs(sub(out["fi"], 2048) - g["fi"]).max()) < 1e-5
    assert float(np.abs(out["hx"].detach().numpy() - g["hx"]).max()) < 1e-5
    assert float(np.abs(t.grad.numpy() - g["dt"]).max()) < 1e-6
    _grads_match(sd, g)


@pytest.mark.parametrize("name", ["d_cat_train_full", "d_cat_eval_small"])
def test_concat_discriminator_oracle_vs_reference(name):
    """Discriminator (disc_type 'cat', model/GANSurv.py:52-68); gradients pinned by the reference run in float64.
    The embedding gradients of this variant are ill-conditioned in fp32: there the oracle's value depends on the summation
    order of the CPU's kernels (measured: under 1e-5 of the tensor maximum at 4 or 8 threads, 7e-3 at 1 or 16 and more),
    so the parameter gradients are compared from a float64 run of the oracle, like the fixture's."""
    g = golden(name)
    C, d, N, train, seed = [int(v) for v in g["cfg"]]
    ty = (64, 128) if d == 128 else (d // 2, d)
    sd = {k: v.requires_grad_(True) for k, v in O.synth_state_dict(O.DCAT_SHAPES(C, d, ty), seed + 50).items()}
    x = O.synth_bag(N, seed, C)
    t = torch.tensor([[0.61]], requires_grad=True)
    masks = d_masks(N // 16, d, seed * 10 + 5) if train else None
    out = O.catdisc_forward(sd, x, t, masks)
    out["out"].sum().backward()
    assert float(np.abs(out["out"].detach().numpy() - g["out"]).max()) < 1e-6
    assert float(np.abs(t.grad.numpy() - g["dt"]).max()) < 1e-6
    sd = {k: v.detach().double().requires_grad_(True) for k, v in sd.items()}
    O.catdisc_forward(sd, x.double(), torch.tensor([[0.61]], dtype=torch.float64), masks)["out"].sum().backward()
    for k, v in sd.items():
        ref = g["grad." + k]
        if float(np.abs(ref).max()) < 1e-8:
            continue
        assert float(np.abs(sub(v.grad) - ref).max()) <= 1e-4 * float(np.abs(ref).max()), k


@pytest.mark.parametrize("name", ["g_cluster_full", "g_cluster_empty_small"])
def test_cluster_oracle_vs_reference(name):
    g = golden(name)
    C, h, N, seed, empty = [int(v) for v in g["cfg"]]
    sd = {k: v.requires_grad_(True) for k, v in O.synth_state_dict(O.G_CLUSTER_SHAPES(C, h), seed + 20).items()}
    x = O.synth_bag(N, seed, C)
    noise = torch.tensor(np.random.default_rng(seed + 7).uniform(size=(1, h // 2)), dtype=torch.float32)
    out = O.generator_forward(sd, x, [None, noise], (0, 1), None, "cluster", torch.tensor(g["cid"], dtype=torch.float32))
    out["pred"].sum().backward()
    assert float(np.abs(out["pred"].detach().numpy() - g["pred"]).max()) < 1e-6
    if empty:
        assert int((g["cid"] == 5).sum()) == 0 and float(out["hc"][5].abs().max()) == 0.0   # zeros for the empty cluster
    _grads_match(sd, g)


@pytest.mark.parametrize("name", ["step_small", "step_full"])
def test_step_oracle_vs_reference(name):
    """D step + G step + both Adam updates: oracle CpuTrainer vs the reference's modules/losses/optimisers."""
    g = golden(name)
    C, h, o, d, seed, n_steps = [int(v) for v in g["cfg"][:6]]
    Ns = [int(v) for v in g["cfg"][6:]]
    B = len(Ns)
    tr = O.CpuTrainer(O.synth_state_dict(O.G_SHAPES(C, h, o), seed),
                      O.synth_state_dict(O.D_SHAPES(C, d, (64, 128) if d == 128 else (d // 2, d)), seed + 50))
    bags = [O.synth_bag(n, seed + i, C) for i, n in enumerate(Ns)]
    ts, es, vis = torch.tensor(g["t"]), torch.tensor(g["e"]), list(g["visible"])
    for step in range(n_steps):
        rng = np.random.default_rng(seed + 100 * step)
        nzD = [torch.tensor(rng.uniform(size=(1, o // 2)), dtype=torch.float32) for _ in range(B)]
        nzG = [torch.tensor(rng.uniform(size=(1, o // 2)), dtype=torch.float32) for _ in range(B)]
        mr = [d_masks(Ns[i] // 16, d, seed + 1000 * step + 10 * i) for i in range(B)]
        mf = [d_masks(Ns[i] // 16, d, seed + 1000 * step + 10 * i + 5) for i in range(B)]
        mg = [g_masks(Ns[i], h, o, seed + 2000 * step + 10 * i) for i in range(B)]
        r = tr.step(bags, ts, es, vis, nzD, nzG, mr, mf, mg)
        assert abs(r["dis_loss"] - float(g[f"dis_loss{step}"])) < 1e-6
        assert abs(r["gen_loss"] - float(g[f"gen_loss{step}"])) < 1e-6
        assert abs(r["t_reg"] - float(g[f"t_reg{step}"])) < 1e-6
        assert abs(r["total"] - float(g[f"total{step}"])) < 1e-6
        assert float((r["pred_g"] - torch.tensor(g[f"pred_g{step}"])).abs().max()) < 1e-6
        assert float((r["fake_d"] - torch.tensor(g[f"fake_d{step}"])).abs().max()) < 1e-6
    for k, v in tr.sdG.items():
        assert float(np.abs(sub(v) - g["gparam." + k]).max()) < 1e-6, k
    for k, v in tr.sdD.items():
        if k.endswith("pool.fc2.bias"):      # mathematically-zero gradient: Adam turns rounding noise into +-lr steps
            continue
        assert float(np.abs(sub(v) - g["dparam." + k]).max()) < 2e-6, k


def test_misc_fixtures():
    g = golden("misc")
    # region <-> patch index map (tools/big_to_small_patching.py): bit-exact, float64 output
    l1 = O.region_index_map(g["l2_coords"], 256, 4)
    assert l1.dtype == np.float64 and np.array_equal(l1, g["l1_coords"])
    # sequence2square: row n -> region n//16, grid (n%16)//4, n%4
    sq = g["seq2sq"]                      # [4 regions, C=3, 4, 4] built from arange(64*3).reshape(1,64,3)
    n = np.arange(64)
    expect = np.arange(64 * 3, dtype=np.float32).reshape(64, 3)
    got = sq.transpose(0, 2, 3, 1)[O.region_of_row(n), (n % 16) // 4, n % 4]
    assert np.array_equal(got, expect)
    assert np.array_equal(g["sq2seq"].reshape(64, 3), expect)
    # C-index with ties, lower median, noise stream, losses
    ci = O.concordance_index(g["ci_t"], g["ci_e"], g["ci_pred"])
    assert abs(ci - float(g["ci"])) < 1e-12
    med = O.lower_median(torch.tensor(g["med_in"]), dim=0)
    assert np.array_equal(med.numpy(), g["med_out"])
    assert bool(g["noise_eq"].all())
    fr, ff = torch.tensor([0.3, -1.2, 2.0]), torch.tensor([-0.5, 0.1, 0.7, -2.0])
    for w in ("bce", "hinge", "wasserstein"):
        assert abs(float(O.real_fake_loss(fr, ff, w)) - float(g["rf_" + w])) < 1e-6
        assert abs(float(O.real_fake_loss(None, ff, w)) - float(g["rf_noreal_" + w])) < 1e-6
    p_, t_, e_ = torch.tensor([0.2, 0.9, 0.5, 0.4]), torch.tensor([0.5, 0.3, 0.5, 0.8]), torch.tensor([1., 0., 0., 1.])
    assert abs(float(O.recon_loss(p_, t_, e_, 0.0, 0.0, "l1")) - float(g["recon_l1"])) < 1e-7
    assert abs(float(O.recon_loss(p_, t_, e_, 0.3, 0.1, "l2")) - float(g["recon_l2"])) < 1e-7
    kept = g["mask_bag_rows_kept"].reshape(10, 16)
    assert np.all(kept.all(axis=1) | (~kept).all(axis=1)) and kept.any()   # whole 16-row regions kept or zeroed


@pytest.mark.parametrize("name", ["g_esat_eval_full", "g_esat_train_full", "g_esat_train_small", "g_esat_eval_small"])
def test_esat_generator_oracle_vs_reference(name):
    """Generator over DualTrans_HS / ESAT (bcb_mode 'patch', model/backbone.py:171-196): region embedding, sincos PE,
    one post-norm TransformerEncoderLayer (attention-probability dropout included), GAPool, noise head."""
    g = golden(name)
    C, d, N, train, seed, with_coord = [int(v) for v in g["cfg"]]
    sd = {k: v.requires_grad_(True) for k, v in O.synth_state_dict(O.G_ESAT_SHAPES(C, d), seed).items()}
    x = O.synth_bag(N, seed, C)
    noise = torch.tensor(np.random.default_rng(seed + 7).uniform(size=(1, d // 2)), dtype=torch.float32)
    coord = torch.tensor(g["coord"]) if with_coord else None
    masks = esat_masks(N // 16, d, seed * 10) if train else None
    out = O.generator_forward(sd, x, [None, noise], (0, 1), masks, backbone="patch", coord=coord)
    out["pred"].sum().backward()
    assert float(np.abs(out["pred"].detach().numpy() - g["pred"]).max()) < 1e-6
    assert float(np.abs(out["H"].detach().numpy() - g["H"]).max()) < 1e-5
    assert float(np.abs(sub(out["emb"]) - g["emb"]).max()) < 1e-5
    assert float(np.abs(sub(out["x2"]) - g["x2"]).max()) < 1e-5
    _grads_match(sd, g, skip=("pool.fc2.bias",))      # mathematically zero (softmax shift invariance): rounding noise

"""GPU: the C-fused step of the DeepAttMISL generator (`ClusterAdvStep`, bcb_mode cluster) and its K9 kernel -- the
projection + ReLU + per-(bag, cluster) mean in one tcgen05 pass (`advmil_cluster_pool_fwd`) and its backward
(`advmil_cluster_pool_bwd`) -- against float64 references, the oracle trainer and `ModuleAdvStep`."""
import itertools

import numpy as np
import pytest
import torch

from oracle import advmil_oracle as O
from tests.util import assert_close, build_D, build_G, d_masks

pytestmark = pytest.mark.gpu
RTOL = 1e-5
BF16_TOL = 2e-2          # the bf16-class norm-wise bound of the step tests (tests/test_gpu_bf16_step.py)
ZERO_GRAD = ("pool.fc2.bias", "attention_c.bias")
LENGTHS = [16, 16, 48, 160, 1040, 4112]      # several bags per 128-row tile, boundaries inside tiles
POOL_TOL = {"tf32": 4e-3, "tf32x3": 1e-5, "bf16": 1e-4}       # bf16: the reference sees the same bf16-rounded operands


def _lib():
    from advmil_b200 import _lib
    return _lib.load()


def _cat_masks(per_bag, keys):
    return {k: torch.cat([m[k] for m in per_bag], dim=0).to(torch.uint8).contiguous().cuda() for k in keys}


def _pool_case(ncl, seed=7, C=1024, h=384):
    g = torch.Generator().manual_seed(seed)
    rows = sum(LENGTHS)
    x = torch.randn(rows, C, generator=g)
    W = torch.randn(h, C, generator=g) * 0.03
    b = torch.randn(h, generator=g) * 0.1
    cid = torch.randint(0, ncl, (rows,), generator=g, dtype=torch.int32)
    beg3 = sum(LENGTHS[:3])
    seg3 = cid[beg3:beg3 + LENGTHS[3]]
    seg3[seg3 == 2] = 3                      # bag 3 has an empty cluster
    cid[5] = -1                              # ids outside [0, ncl) count nowhere
    cid[100] = ncl
    cid[rows - 1] = ncl + 3
    return x, W, b, cid


def _operands(x, W, prec):
    """What the kernel multiplies, in float64: bf16-rounded x and W in the bf16 mode, the fp32 values otherwise."""
    if prec == "bf16":
        return x.to(torch.bfloat16).double(), W.to(torch.bfloat16).double()
    return x.double(), W.double()


def _ref_mean(pre, cid, ncl):
    """Per-(bag, cluster) mean of relu(pre) and the counts (model/backbone.py:105-117), float64."""
    v = torch.relu(pre)
    hcs, cnts = [], []
    off = 0
    for n in LENGTHS:
        for k in range(ncl):
            sel = cid[off:off + n] == k
            cnts.append(int(sel.sum()))
            hcs.append(v[off:off + n][sel].mean(0) if sel.any() else torch.zeros(v.shape[1], dtype=v.dtype))
        off += n
    return torch.stack(hcs), torch.tensor(cnts, dtype=torch.int32)


def _pool_fwd(bags, W, b, cid, ncl, prec):
    from advmil_b200 import ops
    lib = _lib()
    h = W.shape[0]
    hc = torch.empty(bags.bags * ncl, h, dtype=torch.float32, device="cuda")
    counts = torch.empty(bags.bags * ncl, dtype=torch.int32, device="cuda")
    keep = torch.empty(bags.rows, h // 32, dtype=torch.int32, device="cuda")
    ws = torch.empty(lib.advmil_cluster_pool_workspace_bytes(bags.rows, bags.bags, h, ncl), dtype=torch.uint8, device="cuda")
    rc = lib.advmil_cluster_pool_fwd(bags.x.data_ptr(), W.data_ptr(), b.data_ptr(), cid.data_ptr(), bags.offsets.data_ptr(),
                                     bags.offsets_host, bags.rows, bags.bags, bags.C, h, ncl, ops.PRECISIONS[prec], hc.data_ptr(),
                                     counts.data_ptr(), keep.data_ptr(), ws.data_ptr(), ws.numel(),
                                     torch.cuda.current_stream().cuda_stream)
    return rc, hc, counts, keep


def _unpack(keep):
    bits = (keep.unsqueeze(-1) >> torch.arange(32, device=keep.device, dtype=torch.int32)) & 1
    return bits.reshape(keep.shape[0], -1).bool()


@pytest.mark.parametrize("ncl", [8, 16])
@pytest.mark.parametrize("prec", ["tf32", "tf32x3", "bf16"])
def test_fused_pool_forward_vs_float64(prec, ncl):
    from advmil_b200 import ops
    x, W, b, cid = _pool_case(ncl)
    bags = ops.PackedBags(x.cuda(), LENGTHS).for_precision(ops.PRECISIONS[prec])
    Wd, bd, cidd = W.cuda(), b.cuda(), cid.cuda()
    rc, hc, counts, keep = _pool_fwd(bags, Wd, bd, cidd, ncl, prec)
    assert rc == 0, _lib().advmil_last_error()
    xr, Wr = _operands(x, W, prec)
    ref, ref_cnt = _ref_mean(xr @ Wr.T + b.double(), cid, ncl)
    assert torch.equal(counts.cpu(), ref_cnt)
    assert_close(hc.cpu(), ref, POOL_TOL[prec], f"hc {prec} ncl={ncl}")
    # the keep bits are the ReLU mask of the same mode's linear_fwd (same mainloop, same K order)
    hx = ops.linear_forward(bags.x, Wd, bd, act=1, precision=ops.PRECISIONS[prec])
    assert torch.equal(_unpack(keep), hx > 0)
    # deterministic: a second call is bitwise identical
    rc2, hc2, counts2, keep2 = _pool_fwd(bags, Wd, bd, cidd, ncl, prec)
    assert rc2 == 0 and torch.equal(hc, hc2) and torch.equal(counts, counts2) and torch.equal(keep, keep2)


@pytest.mark.parametrize("prec", ["tf32", "tf32x3", "bf16"])
def test_fused_pool_backward_and_weight_grads_vs_float64(prec):
    from advmil_b200 import ops
    ncl = 8
    lib = _lib()
    x, W, b, cid = _pool_case(ncl, seed=11)
    bags = ops.PackedBags(x.cuda(), LENGTHS).for_precision(ops.PRECISIONS[prec])
    Wd, bd, cidd = W.cuda(), b.cuda(), cid.cuda()
    rc, hc, counts, keep = _pool_fwd(bags, Wd, bd, cidd, ncl, prec)
    assert rc == 0
    d_hc = torch.randn(hc.shape, generator=torch.Generator().manual_seed(12)).cuda()
    d_hx = torch.empty(bags.rows, W.shape[0], dtype=bags.x.dtype, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    assert lib.advmil_cluster_pool_bwd(d_hc.data_ptr(), keep.data_ptr(), cidd.data_ptr(), bags.offsets.data_ptr(), counts.data_ptr(),
                                       bags.rows, bags.bags, W.shape[0], ncl, ops.PRECISIONS[prec], d_hx.data_ptr(), st) == 0
    # the same d_hx as the module path's segment-mean backward on the kept activation
    hx = ops.linear_forward(bags.x, Wd, bd, act=1, precision=ops.PRECISIONS[prec])
    d_mod = torch.empty_like(hx)
    elem = ops.ELEM_BF16 if hx.dtype == torch.bfloat16 else ops.ELEM_F32
    assert lib.advmil_segment_mean_by_id_bwd(d_hc.data_ptr(), hx.data_ptr(), elem, cidd.data_ptr(), bags.offsets.data_ptr(),
                                             counts.data_ptr(), bags.rows, bags.bags, W.shape[0], ncl, 1, d_mod.data_ptr(), st) == 0
    assert torch.equal(d_hx, d_mod)
    _, dW, db = ops.linear_backward(d_hx, bags.x, Wd, need_dx=False, precision=ops.PRECISIONS[prec])
    xr, Wr = _operands(x, W, prec)
    Wr.requires_grad_(True)
    br = b.double().requires_grad_(True)
    ref, _ = _ref_mean(xr @ Wr.T + br, cid, ncl)
    (ref * d_hc.cpu().double()).sum().backward()
    # tf32: the weight-gradient GEMM truncates both operands to 10 mantissa bits (and so does its accumulation chain)
    tol = {"tf32": 2e-2, "tf32x3": 1e-5, "bf16": 1e-2}[prec]
    assert_close(dW.cpu(), Wr.grad, tol, f"dW {prec}")
    assert_close(db.cpu(), br.grad, tol, f"db {prec}")


def _step_case(seed=151):
    Cdim, h = 1024, 384
    sdG, sdD = O.synth_state_dict(O.G_CLUSTER_SHAPES(Cdim, h), seed), O.synth_state_dict(O.D_SHAPES(), seed + 1)
    return Cdim, h, sdG, sdD


def _engines(kind, sdG, sdD, prec, Cdim=1024, h=384):
    from advmil_b200.step import ClusterAdvStep, ModuleAdvStep
    G, D = build_G((Cdim, h, h), mode="cluster"), build_D()
    G.load_state_dict(sdG)
    D.load_state_dict(sdD)
    cls = ClusterAdvStep if kind == "fused" else ModuleAdvStep
    return G, D, cls(G, D, precision=prec)


def _run_vs_oracle(prec, Ns, es_fix=None, vis=None, steps=2):
    """Two steps of ClusterAdvStep (and, outside the exact modes, ModuleAdvStep in the same mode) against the oracle trainer
    with injected masks: the checks of test_module_step_with_cluster_generator_vs_oracle_trainer."""
    from advmil_b200 import ops
    Cdim, h, sdG, sdD = _step_case()
    B = len(Ns)
    tr = O.CpuTrainer(sdG, sdD, backbone="cluster")
    G, D, eng = _engines("fused", sdG, sdD, prec)
    mod = None if prec in ("fp32", "tf32x3") else _engines("module", sdG, sdD, prec)
    xs = [O.synth_bag(n, 160 + i, Cdim) for i, n in enumerate(Ns)]
    rng = np.random.default_rng(153)
    cids = [torch.tensor(rng.integers(0, 8, size=n), dtype=torch.float32) for n in Ns]
    cids[1][cids[1] == 5] = 4.0            # cluster 5 of bag 1 is empty (model/backbone.py:114-115)
    ts, es = O.synth_labels(B, 154)
    es[0] = 1.0
    if es_fix is not None:
        es[:] = es_fix
    vis = vis or [True] * B
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    ext = torch.cat(cids).cuda()
    for step in range(steps):
        nd = torch.tensor(rng.uniform(size=(B, h // 2)), dtype=torch.float32)
        ng = torch.tensor(rng.uniform(size=(B, h // 2)), dtype=torch.float32)
        mr = [d_masks(n // 16, 128, 900 + 10 * i + step) for i, n in enumerate(Ns)]
        mf = [d_masks(n // 16, 128, 950 + 10 * i + step) for i, n in enumerate(Ns)]
        mg = [{"h": O.synth_masks((8, h), 0.75, 1000 + 10 * i + step), "a": O.synth_masks((8, h), 0.75, 1001 + 10 * i + step),
               "b": O.synth_masks((8, h), 0.75, 1002 + 10 * i + step), "mlp0": O.synth_masks((1, h // 2), 0.4, 1003 + 10 * i + step)}
              for i in range(B)]
        ref = tr.step(xs, ts, es, vis, list(nd), list(ng), mr, mf, mg, exts=cids)
        kw = dict(noise_d=nd.cuda(), noise_g=ng.cuda(), masks_d_real=_cat_masks(mr, ["fc1", "ga", "gs", "fc2"]),
                  masks_d_fake=_cat_masks(mf, ["fc1", "ga", "gs", "fc2"]), masks_g=_cat_masks(mg, ["h", "a", "b", "mlp0"]), ext=ext)
        args = (bags, ts.cuda(), es.cuda(), torch.tensor(vis, dtype=torch.uint8).cuda())
        out = eng.step(*args, **kw)
        L = eng.loss_dict(out)
        if prec in ("fp32", "tf32x3"):
            assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), RTOL, f"pred_d {step}")
            assert_close(out["pred_g"].cpu(), ref["pred_g"].reshape(-1), RTOL, f"pred_g {step}")
            assert_close(out["f_fake_g"].cpu(), ref["fake_g"].reshape(-1), RTOL, f"fake_g {step}", atol_scale=1e-1)
            assert abs(L["dis_loss"] - ref["dis_loss"]) < 2e-5 and abs(L["gen_total_loss"] - ref["total"]) < 2e-5
            assert abs(L["t_reg_loss"] - ref["t_reg"]) < 2e-5 and abs(L["gen_loss"] - ref["gen_loss"]) < 2e-5
        else:
            assert_close(out["pred_d"].cpu(), ref["pred_d"].reshape(-1), BF16_TOL, f"pred_d {step}")
            assert_close(out["pred_g"].cpu(), ref["pred_g"].reshape(-1), BF16_TOL, f"pred_g {step}")
            assert_close(out["f_fake_g"].cpu(), ref["fake_g"].reshape(-1), BF16_TOL, f"fake_g {step}")
            for k, r in (("dis_loss", "dis_loss"), ("gen_total_loss", "total"), ("t_reg_loss", "t_reg")):
                assert abs(L[k] - ref[r]) <= BF16_TOL * abs(ref[r]) + 1e-4, (k, L[k], ref[r])
            mG, mD, meng = mod
            mo = meng.step(*args, **kw)
            assert_close(out["pred_d"].cpu(), mo["pred_d"].cpu(), BF16_TOL, f"pred_d vs module {step}")
            assert_close(out["pred_g"].cpu(), mo["pred_g"].cpu(), BF16_TOL, f"pred_g vs module {step}")
            assert abs(L["dis_loss"] - float(mo["dis_loss"])) <= BF16_TOL * abs(float(mo["dis_loss"])) + 1e-4
            # both engines flatten netG.parameters() in the same order
            for (name, _), gv, mv in zip(G.named_parameters(), eng.G.grad_views, meng.G.grad_views):
                if not name.endswith(ZERO_GRAD):
                    assert_close(gv.cpu(), mv.cpu(), BF16_TOL, f"G grad {name} vs module, step {step}", atol=1e-7)
    if prec in ("fp32", "tf32x3"):
        for k, p in D.named_parameters():
            if not k.endswith(ZERO_GRAD):
                assert_close(p.detach().cpu(), tr.sdD[k].detach(), RTOL, "D param " + k, atol=8e-5 * 2 * 2e-2)
        for k, p in G.named_parameters():
            if not k.endswith(ZERO_GRAD):
                assert_close(p.detach().cpu(), tr.sdG[k].detach(), RTOL, "G param " + k, atol=8e-5 * 2 * 2e-2)


@pytest.mark.parametrize("prec", ["fp32", "tf32x3", "tf32", "bf16"])
def test_cluster_step_vs_oracle_trainer(prec):
    _run_vs_oracle(prec, [160, 320, 96])


def test_cluster_step_without_real_pairs():
    _run_vs_oracle("fp32", [160, 320, 96], es_fix=0.0)


def test_cluster_step_semi_supervised():
    _run_vs_oracle("tf32x3", [160, 320, 96], vis=[True, False, True])


def test_cluster_step_seeded_is_deterministic():
    from advmil_b200 import ops
    Cdim, h, sdG, sdD = _step_case(171)
    Ns = [1040, 4112, 48, 16]
    xs = [O.synth_bag(n, 180 + i, Cdim) for i, n in enumerate(Ns)]
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    ext = torch.randint(0, 8, (sum(Ns),), generator=torch.Generator().manual_seed(3), dtype=torch.int32).cuda()
    ts, es = O.synth_labels(len(Ns), 172)
    vis = torch.ones(len(Ns), dtype=torch.uint8).cuda()
    rng = np.random.default_rng(5)
    noise = [torch.tensor(rng.uniform(size=(len(Ns), h // 2)), dtype=torch.float32).cuda() for _ in range(4)]
    runs = []
    for _ in range(2):
        G, D, eng = _engines("fused", sdG, sdD, "bf16")
        seeds = itertools.count(12345)
        eng._seed = lambda: next(seeds)
        outs = [eng.step(bags, ts.cuda(), es.cuda(), vis, noise_d=noise[2 * s], noise_g=noise[2 * s + 1], ext=ext) for s in range(2)]
        torch.cuda.synchronize()
        runs.append((outs, eng.G.flat.clone(), eng.D.flat.clone()))
    (o1, g1, d1), (o2, g2, d2) = runs
    for a, b in zip(o1, o2):
        for k in ("losses", "pred_d", "pred_g", "f_d", "f_fake_g"):
            assert torch.equal(a[k], b[k]), k
    assert torch.equal(g1, g2) and torch.equal(d1, d2)


def test_cluster_step_rejections():
    from advmil_b200 import _lib as L, ops
    from advmil_b200.step import ClusterAdvStep
    Cdim, h, sdG, sdD = _step_case()
    G, D, eng = _engines("fused", sdG, sdD, "bf16")
    t, e, vis = torch.rand(2).cuda(), torch.ones(2).cuda(), torch.ones(2, dtype=torch.uint8).cuda()
    odd = ops.PackedBags.from_list([torch.randn(40, Cdim).cuda(), torch.randn(32, Cdim).cuda()])
    with pytest.raises(AssertionError, match="multiple of 16"):
        eng.step(odd, t, e, vis, ext=torch.zeros(72, dtype=torch.int32).cuda())
    ok = ops.PackedBags.from_list([torch.randn(48, Cdim).cuda(), torch.randn(32, Cdim).cuda()])
    with pytest.raises(ValueError, match="ext"):
        eng.step(ok, t, e, vis)
    G17 = build_G((Cdim, h, h), mode="cluster")
    G17.backbone.num_clusters = 17
    with pytest.raises(NotImplementedError, match="ModuleAdvStep"):
        ClusterAdvStep(G17, build_D())
    for mode in ("abmil", "patch"):
        with pytest.raises(NotImplementedError, match="ClusterAdvStep is the C-fused step"):
            ClusterAdvStep(build_G((Cdim, h, h), mode=mode), build_D())
    # the C entry rejects 17 clusters too
    eng2 = _engines("fused", sdG, sdD, "bf16")[2]
    eng2.netG.backbone.num_clusters = 17
    with pytest.raises(L.AdvmilError, match="num_clusters"):
        eng2.step(ok, t, e, vis, ext=torch.zeros(80, dtype=torch.int32).cuda())
    x, W, b, cid = _pool_case(8)
    bags = ops.PackedBags(x.cuda(), LENGTHS).for_precision(ops.BF16)
    rc = _pool_fwd(bags, W.cuda(), b.cuda(), cid.cuda(), 17, "bf16")[0]
    assert rc == 1 and b"num_clusters" in _lib().advmil_last_error()


def test_abmil_step_points_to_the_cluster_step():
    from advmil_b200.step import AdvStep
    with pytest.raises(NotImplementedError, match="ClusterAdvStep"):
        AdvStep(build_G((1024, 384, 384), mode="cluster"), build_D())

"""Throughput of the adversarial step with the DeepAttMISL generator (bcb_mode cluster) on one GPU.

  1. `ModuleAdvStep` (the route bench.py's cluster leg times) and the C-fused `ClusterAdvStep`, alternated in one process on
     the inputs of bench.py:leg_cluster: 16 bags x 16384 rows of bf16 features (512 MiB; fp32, 1 GiB, in the tf32 run: larger
     than the 126 MB L2, so every pass reads x from HBM), 8 clusters, bag 0 with an empty cluster.  bags/s and ms per step over blocks of steps timed
     with CUDA events after a warm-up, the cyclic GC kept out of the timed region (as bench.timed does).  bf16, and one run
     in tf32.
  2. Per-stage times of one fused step from the library's profiler tags (a separate run: tracing slows the host): K9 (the
     projection + ReLU + per-(bag, cluster) mean pass, TFLOP/s on 2 C h FLOP per row, 206 GFLOP per step), the expansion
     of d_hc into d_hx, dWphi and dbphi.
Writes profiles/cluster_step_bench.json with the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import gc
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from advmil_b200 import _lib, ops  # noqa: E402
from oracle import advmil_oracle as O  # noqa: E402

NTAGS = len(_lib.PROF_TAGS)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, plim, clk = [v.strip() for v in q[0].split(",")]
    return {"gpu": name, "power_limit": plim, "max_sm_clock": clk, "torch_name": torch.cuda.get_device_name(0)}


def build_nets():
    """the configs' DeepAttMISL G (1024-384-384, 8 clusters, noise head 0-1) and RLIP D (1024 -> 128) on cuda"""
    from types import SimpleNamespace
    from advmil_b200.model.backbone import load_backbone
    from advmil_b200.model.GANSurv import Generator, PrjDiscriminator
    G = Generator(384, 1, load_backbone("cluster", [1024, 384, 384]), SimpleNamespace(noise=[0, 1], hops=1, noise_dist="uniform"),
                  False, 0.6, "sigmoid").cuda()
    D = PrjDiscriminator(SimpleNamespace(in_dim=1024, out_dim=128, ksize=1, backbone="avgpool", dropout=0.25),
                         SimpleNamespace(in_dim=1, hid_dims=[64, 128], norm=False, dropout=0.0), prj_path="x",
                         inner_product="instance").cuda()
    G.load_state_dict(O.synth_state_dict(O.G_CLUSTER_SHAPES(1024, 384), 402))
    D.load_state_dict(O.synth_state_dict(O.D_SHAPES(), 403))
    return G, D


def inputs(B, N, precision):
    x = torch.cat([O.synth_bag(N, 400 + i) for i in range(B)])
    x = (x.to(torch.bfloat16) if precision == "bf16" else x).cuda()          # the tf32 mode reads fp32 features
    bags = ops.PackedBags(x, [N] * B)
    g = torch.Generator(device="cuda").manual_seed(7)
    cid = torch.randint(0, 8, (bags.rows,), device="cuda", generator=g).float()
    cid[:N][cid[:N] == 5] = 4.0                       # bag 0 has an empty cluster (model/backbone.py:114-115)
    ts, es = O.synth_labels(B, 401)
    ts, es, vis = ts.cuda(), es.cuda(), torch.ones(B, dtype=torch.uint8, device="cuda")
    counts = (float(((es == 1) & (vis != 0)).sum()), float(B), float(vis.sum()))
    nz = torch.rand(B, 192, device="cuda")
    return bags, cid, ts, es, vis, counts, nz


def step_bench(precision, B, N, steps, warmup, reps):
    from advmil_b200.step import ClusterAdvStep, ModuleAdvStep
    bags, cid, ts, es, vis, counts, nz = inputs(B, N, precision)
    engines = {}
    for name, cls in (("ModuleAdvStep", ModuleAdvStep), ("ClusterAdvStep", ClusterAdvStep)):
        G, D = build_nets()
        engines[name] = cls(G, D, precision=precision)

    def one(name):
        return engines[name].step(bags, ts, es, vis, noise_d=nz, noise_g=nz, global_counts=counts, ext=cid)
    for _ in range(warmup):
        for name in engines:
            one(name)
    torch.cuda.synchronize()
    ms = {name: [] for name in engines}
    for _ in range(reps):                          # alternate the engines block by block
        for name in engines:
            gc.collect()
            gc.disable()
            try:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(steps):
                    one(name)
                b.record()
                torch.cuda.synchronize()
            finally:
                gc.enable()
            ms[name].append(a.elapsed_time(b) / steps)
    out = {}
    for name, v in ms.items():
        v = np.array(v)
        out[name] = {"ms_per_step_median": float(np.median(v)), "ms_per_step_min": float(v.min()), "ms_per_step_max": float(v.max()),
                     "bags_per_s": B / (float(np.median(v)) / 1e3), "blocks": reps, "steps_per_block": steps}
        print(precision, name, json.dumps(out[name]), flush=True)
    out["speedup_median"] = out["ModuleAdvStep"]["ms_per_step_median"] / out["ClusterAdvStep"]["ms_per_step_median"]
    return out, engines["ClusterAdvStep"], (bags, cid, ts, es, vis, counts, nz)


def stage_bench(eng, data, iters, C_=1024, h=384):
    lib = _lib.load()
    bags, cid, ts, es, vis, counts, nz = data
    ms = (C.c_double * NTAGS)()
    cnt = (C.c_int64 * NTAGS)()
    torch.cuda.synchronize()
    lib.advmil_profile_read(ms, cnt, NTAGS)
    lib.advmil_profile_enable(1)
    for _ in range(iters):
        eng.step(bags, ts, es, vis, noise_d=nz, noise_g=nz, global_counts=counts, ext=cid)
    torch.cuda.synchronize()
    lib.advmil_profile_enable(0)
    lib.advmil_profile_read(ms, cnt, NTAGS)
    tag = {n: i for i, n in enumerate(_lib.PROF_TAGS)}
    per = lambda n: ms[tag[n]] / iters                    # noqa: E731  ms per step under the tag
    flop = 2.0 * C_ * h * bags.rows
    # K9 is one launch per step.  bwd_data / bwd_w_proj / colsum per step also hold the attention stage's small launches
    # (num_clusters rows per bag), so they bound the N-row pieces (d_hx expansion, dWphi, dbphi) from above
    out = {"k9_proj_segmean_ms": per("proj_segmean_fwd"), "k9_tflops": flop / per("proj_segmean_fwd") / 1e9,
           "k9_gflop": flop / 1e9, "bwd_data_ms_incl_d_hx_expand": per("bwd_data"), "bwd_w_proj_ms_incl_dWphi": per("bwd_w_proj"),
           "dWphi_tflops_lower_bound": flop / per("bwd_w_proj") / 1e9, "colsum_ms_incl_dbphi": per("colsum"), "steps": iters,
           "all_tags_ms_per_step": {n: ms[i] / iters for i, n in enumerate(_lib.PROF_TAGS) if cnt[i]}}
    print("stages", json.dumps(out), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bags", type=int, default=16)
    ap.add_argument("--rows", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cluster_step_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    res = {"device": gpu_info(), "bags": args.bags, "rows_per_bag": args.rows, "C": 1024, "h": 384, "clusters": 8}
    res["bf16"], eng, data = step_bench("bf16", args.bags, args.rows, args.steps, args.warmup, args.reps)
    res["stages_bf16"] = stage_bench(eng, data, args.steps)
    del eng, data
    torch.cuda.empty_cache()
    res["tf32"], eng, data = step_bench("tf32", args.bags, args.rows, args.steps, args.warmup, max(1, args.reps - 1))
    res["stages_tf32"] = stage_bench(eng, data, args.steps)
    res["device_after"] = gpu_info()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

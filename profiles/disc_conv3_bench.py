"""Throughput of the 3x3 patch embedding of the RLIP discriminator (disc_netx_ksize: 3) on one GPU.

  1. the conv-embed forward (tap-major weight repack + implicit-GEMM conv with the LayerNorm / ReLU / region-mean epilogue)
     and the dWc launch (weight-gradient GEMM over 9 taps + split-K reduce into [d, C, 3, 3]) at 16 x 16384 rows in bf16,
     tf32 and tf32x3: CUDA events of the library's own stage profiler around each launch, summed over many launches;
     TFLOP/s on 2 * 9 * C * d FLOP per row (618.5 GFLOP per launch) and the share of the tensor peak bench.py's roofline
     uses (bench.load_peaks: bf16 figure; half of it for tf32 operands);
  2. the reference's route on the same GPU: F.conv2d in bf16, channels-last, on [R, 1024, 4, 4] alone, and with the
     sequence2square / square2sequence copies, LayerNorm, ReLU and the 4x4 average pool;
  3. the bf16 AdvStep (one D update + one G update) with a ksize-1 and a ksize-3 discriminator, alternated in one process.

x (16 x 16384 x 1024 bf16 = 512 MiB, fp32 1 GiB) does not fit the 126 MB L2, so every launch reads it from HBM.
Writes profiles/<out>.json with the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from advmil_b200 import _lib, ops  # noqa: E402
from oracle import advmil_oracle as O  # noqa: E402

PROF_EMBED, PROF_BWD_W_EMBED = _lib.PROF_TAGS.index("embed_fwd"), _lib.PROF_TAGS.index("bwd_w_embed")
NTAGS = len(_lib.PROF_TAGS)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, plim, clk = [v.strip() for v in q[0].split(",")]
    return {"gpu": name, "power_limit": plim, "max_sm_clock": clk, "torch_name": torch.cuda.get_device_name(0)}


def profile_read(lib):
    ms = (C.c_double * NTAGS)()
    cnt = (C.c_int64 * NTAGS)()
    lib.advmil_profile_read(ms, cnt, NTAGS)
    return list(ms), list(cnt)


def events_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def stage_bench(rows, C_, d, iters, peaks):
    lib = _lib.load()
    flop = 2.0 * 9 * C_ * d * rows
    sd = O.synth_state_dict({"w": (d, C_, 3, 3), "b": (d,), "g": (d,), "be": (d,)}, 1)
    params = [sd["w"].cuda(), sd["b"].cuda(), (sd["g"] + 1).cuda(), sd["be"].cuda()] + [None] * 20
    cfg = ops.DiscConfig(C=C_, d=d, t1=1, t2=d, ksize=3)
    x32 = torch.randn(rows, C_, device="cuda")
    bags = ops.PackedBags(x32, [rows // 16] * 16)
    d_emb = torch.randn(rows // 16, d, device="cuda")
    out = {}
    for mode in ("bf16", "tf32", "tf32x3"):
        prec = ops.PRECISIONS[mode]
        b = bags.for_precision(prec)
        grads = [torch.empty_like(t) for t in params[:4]] + [None] * 20
        acts = ops.disc_embed_forward(cfg, params, b, prec, save=True)
        for _ in range(3):                                           # warm-up: module load, tensor maps, scratch growth
            acts = ops.disc_embed_forward(cfg, params, b, prec, save=True)
            ops.disc_embed_backward(cfg, params, b, acts, d_emb, grads)
        torch.cuda.synchronize()
        profile_read(lib)
        lib.advmil_profile_enable(1)
        for _ in range(iters):
            acts = ops.disc_embed_forward(cfg, params, b, prec, save=True)
            ops.disc_embed_backward(cfg, params, b, acts, d_emb, grads)
        torch.cuda.synchronize()
        lib.advmil_profile_enable(0)
        ms, cnt = profile_read(lib)
        fwd, wg = ms[PROF_EMBED] / cnt[PROF_EMBED], ms[PROF_BWD_W_EMBED] / cnt[PROF_BWD_W_EMBED]
        peak = peaks["tflops"] * (1.0 if mode == "bf16" else 0.5)
        out[mode] = {"fwd_ms": fwd, "fwd_tflops": flop / fwd / 1e9, "fwd_frac_peak": flop / fwd / 1e9 / peak,
                     "dwc_ms": wg, "dwc_tflops": flop / wg / 1e9, "dwc_frac_peak": flop / wg / 1e9 / peak,
                     "launches": cnt[PROF_EMBED], "peak_tflops": peak}
        print(mode, json.dumps(out[mode]), flush=True)
    return out


def cudnn_bench(rows, C_, d, iters):
    R = rows // 16
    flop = 2.0 * 9 * C_ * d * rows
    conv = torch.nn.Conv2d(C_, d, 3, 1, padding=1).cuda().to(torch.bfloat16).to(memory_format=torch.channels_last)
    norm = torch.nn.LayerNorm(d).cuda().to(torch.bfloat16)
    x = torch.randn(rows, C_, device="cuda", dtype=torch.bfloat16)
    img = x.view(R, 4, 4, C_).permute(0, 3, 1, 2)                    # channels-last view: no copy
    torch.backends.cudnn.benchmark = True

    @torch.no_grad()
    def conv_only():
        return conv(img)

    @torch.no_grad()
    def full():
        sq = x.view(R, 4, 4, C_).permute(0, 3, 1, 2).contiguous()       # sequence2square as the reference writes it
        y = conv(sq)
        seq = y.permute(0, 2, 3, 1).reshape(R, 16, d).contiguous()      # square2sequence
        e = torch.relu(norm(seq))
        return F.adaptive_avg_pool2d(e.view(R, 4, 4, d).permute(0, 3, 1, 2), 1)

    res = {}
    for name, fn in (("conv2d_channels_last", conv_only), ("conv2d_with_copies_ln_relu_pool", full)):
        for _ in range(5):
            fn()
        ms = events_ms(fn, iters)
        res[name] = {"ms": ms, "tflops_conv_flop": flop / ms / 1e9}
        print(name, json.dumps(res[name]), flush=True)
    return res


def build_nets(ksize):
    """the configs' G (ABMIL 1024-384-384, noise head 0-1) and RLIP D (1024 -> 128, time embedding 64-128) on cuda, with the
    discriminator's patch embedding at `ksize`"""
    from types import SimpleNamespace
    from advmil_b200.model.backbone import load_backbone
    from advmil_b200.model.GANSurv import Generator, PrjDiscriminator
    G = Generator(384, 1, load_backbone("abmil", [1024, 384, 384]), SimpleNamespace(noise=[0, 1], hops=1, noise_dist="uniform"),
                  False, 0.6, "sigmoid").cuda()
    D = PrjDiscriminator(SimpleNamespace(in_dim=1024, out_dim=128, ksize=ksize, backbone="avgpool", dropout=0.25),
                         SimpleNamespace(in_dim=1, hid_dims=[64, 128], norm=False, dropout=0.0), prj_path="x",
                         inner_product="instance").cuda()
    shapes = dict(O.D_SHAPES())
    shapes["net_pair_one.embedding.conv.weight"] = (128, 1024, ksize, ksize)
    G.load_state_dict(O.synth_state_dict(O.G_SHAPES(), 302))
    D.load_state_dict(O.synth_state_dict(shapes, 303))
    return G, D


def step_bench(steps, warmup):
    from advmil_b200.step import AdvStep
    Ns = [16384] * 16
    B = len(Ns)
    x = torch.cat([O.synth_bag(16384, 300 + i) for i in range(B)]).to(torch.bfloat16).cuda()
    bags = ops.PackedBags(x, Ns)
    ts, es = O.synth_labels(B, 301)
    ts, es, vis = ts.cuda(), es.cuda(), torch.ones(B, dtype=torch.uint8, device="cuda")
    engines = {}
    for k in (1, 3):
        G, D = build_nets(k)
        engines[k] = AdvStep(G, D, precision="bf16")
    times = {1: [], 3: []}
    for rep in range(warmup + steps):
        for k in (1, 3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            engines[k].step(bags, ts, es, vis)
            torch.cuda.synchronize()
            if rep >= warmup:
                times[k].append(time.perf_counter() - t0)
    out = {}
    for k in (1, 3):
        t = np.array(times[k])
        flop_row = 5511168 if k == 1 else 11802624
        out[f"ksize{k}"] = {"step_ms_median": 1e3 * float(np.median(t)), "step_ms_min": 1e3 * float(t.min()),
                            "step_ms_max": 1e3 * float(t.max()), "bags_per_s": B / float(np.median(t)),
                            "algorithmic_tflops": flop_row * sum(Ns) / float(np.median(t)) / 1e12, "steps": len(t)}
        print(f"step ksize{k}", json.dumps(out[f"ksize{k}"]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=16 * 16384)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "disc_conv3_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    import bench
    info = gpu_info()
    peaks = bench.load_peaks(10.0)                 # the stage loops below run for seconds: the sustained figure
    res = {"device": info, "rows": args.rows, "C": 1024, "d": 128, "gflop_per_launch": 2 * 9 * 1024 * 128 * args.rows / 1e9,
           "peak": {"bf16_tflops": peaks["tflops"], "source": peaks["src"], "kind": peaks["kind"], "tf32_rule": "half the bf16 figure"}}
    res["stage"] = stage_bench(args.rows, 1024, 128, args.iters, peaks)
    res["cudnn_reference_route"] = cudnn_bench(args.rows, 1024, 128, args.iters)
    res["adv_step_bf16_16x16384"] = step_bench(args.steps, args.warmup)
    res["device_after"] = gpu_info()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

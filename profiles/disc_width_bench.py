"""The bf16 AdvStep (one D update + one G update, 16 x 16384 x 1024) with the RLIP discriminator at disc_netx_out_dim
d = 64, 128 and 256, each with a 1x1 and a 3x3 patch embedding, alternated in one process on one GPU.

For every configuration: host-clock step times around a device synchronise (profiler off), then the library's CUDA-event
stage profiler over separate steps for the embedding forward, its weight gradient (bwd_w_embed), head_fwd and head_bwd.
The embedding's share of the bf16 tensor peak (bench.load_peaks, as DESIGN.md §5) is 2 K d FLOP per row (K = C for 1x1,
9 C for 3x3) over the profiled embed_fwd time.  x (512 MiB in bf16) does not fit the 126 MB L2.  Writes the JSON record
with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from advmil_b200 import _lib, ops  # noqa: E402
from oracle import advmil_oracle as O  # noqa: E402
from profiles.disc_conv3_bench import gpu_info, profile_read  # noqa: E402

TAGS = ("embed_fwd", "bwd_w_embed", "head_fwd", "head_bwd")
WIDTHS, KSIZES = (64, 128, 256), (1, 3)


def build_nets(d, ksize):
    from types import SimpleNamespace
    from advmil_b200.model.backbone import load_backbone
    from advmil_b200.model.GANSurv import Generator, PrjDiscriminator
    G = Generator(384, 1, load_backbone("abmil", [1024, 384, 384]), SimpleNamespace(noise=[0, 1], hops=1, noise_dist="uniform"),
                  False, 0.6, "sigmoid").cuda()
    D = PrjDiscriminator(SimpleNamespace(in_dim=1024, out_dim=d, ksize=ksize, backbone="avgpool", dropout=0.25),
                         SimpleNamespace(in_dim=1, hid_dims=[d // 2, d], norm=False, dropout=0.0), prj_path="x",
                         inner_product="instance").cuda()
    shapes = dict(O.D_SHAPES(1024, d, (d // 2, d)))
    shapes["net_pair_one.embedding.conv.weight"] = (d, 1024, ksize, ksize)
    G.load_state_dict(O.synth_state_dict(O.G_SHAPES(), 302))
    D.load_state_dict(O.synth_state_dict(shapes, 303))
    return G, D


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--prof-steps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "disc_width_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    import bench
    from advmil_b200.step import AdvStep
    info = gpu_info()
    lib = _lib.load()
    Ns = [16384] * 16
    B, rows = len(Ns), sum(Ns)
    x = torch.cat([O.synth_bag(16384, 300 + i) for i in range(B)]).to(torch.bfloat16).cuda()
    bags = ops.PackedBags(x, Ns)
    ts, es = O.synth_labels(B, 301)
    ts, es, vis = ts.cuda(), es.cuda(), torch.ones(B, dtype=torch.uint8, device="cuda")
    confs = [(d, k) for d in WIDTHS for k in KSIZES]
    engines = {c: AdvStep(*build_nets(*c), precision="bf16") for c in confs}
    times = {c: [] for c in confs}
    for rep in range(args.warmup + args.steps):
        for c in confs:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            engines[c].step(bags, ts, es, vis)
            torch.cuda.synchronize()
            if rep >= args.warmup:
                times[c].append(time.perf_counter() - t0)
    stages = {c: {t: 0.0 for t in TAGS} for c in confs}
    counts = {c: {t: 0 for t in TAGS} for c in confs}
    for rep in range(args.prof_steps):
        for c in confs:
            torch.cuda.synchronize()
            profile_read(lib)
            lib.advmil_profile_enable(1)
            engines[c].step(bags, ts, es, vis)
            torch.cuda.synchronize()
            lib.advmil_profile_enable(0)
            ms, cnt = profile_read(lib)
            for t in TAGS:
                i = _lib.PROF_TAGS.index(t)
                stages[c][t] += ms[i]
                counts[c][t] += cnt[i]
    peaks = bench.load_peaks(0.1)              # one embedding launch lasts well under a second: the burst figure
    res = {"device": info, "bags": B, "rows_per_bag": 16384, "C": 1024, "precision": "bf16",
           "peak": {"bf16_tflops": peaks["tflops"], "source": peaks["src"], "kind": peaks["kind"]}, "configs": {}}
    for d, k in confs:
        t = np.array(times[(d, k)])
        st = {tag: {"ms_per_step": stages[(d, k)][tag] / args.prof_steps, "launches_per_step": counts[(d, k)][tag] / args.prof_steps}
              for tag in TAGS}
        # the D phase embeds the bags once per step (the G phase once more, without saving y_pre): per-launch time
        # (at d = 128, ksize 1 the D phase's embedding runs fused with the generator's projection, under proj_embed_fwd)
        n_emb = counts[(d, k)]["embed_fwd"]
        emb_ms = stages[(d, k)]["embed_fwd"] / n_emb if n_emb else None
        flop = 2.0 * 1024 * k * k * d * rows
        row = {"step_ms_median": 1e3 * float(np.median(t)), "step_ms_min": 1e3 * float(t.min()), "step_ms_max": 1e3 * float(t.max()),
               "steps": len(t), "stages": st, "embed_fwd_ms_per_launch": emb_ms, "embed_gflop_per_launch": flop / 1e9,
               "embed_tflops": flop / emb_ms / 1e9 if emb_ms else None,
               "embed_frac_bf16_peak": flop / emb_ms / 1e9 / peaks["tflops"] if emb_ms else None}
        res["configs"][f"d{d}_ksize{k}"] = row
        print(f"d{d} ksize{k}", json.dumps(row), flush=True)
    res["device_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

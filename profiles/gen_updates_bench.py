"""Step time of the C-fused adversarial steps with gen_updates = 1, 2 and 3 G updates per D update (model_handler.py:328-335):
bf16 AdvStep, ClusterAdvStep and EsatAdvStep at 16 x 16384 x 1024, the nine (engine, gen_updates) configurations alternated in
one process on one GPU.

For every configuration: host-clock step times around a device synchronise (profiler off; median, min, max), then the
library's CUDA-event stage profiler over separate steps for the per-step launch count and time of embed_fwd (the RLIP
embedding of x, and the ESAT generator's patch embedding).  x (512 MiB in bf16) does not fit the 126 MB L2.  Writes the
JSON record with the GPU's name and power limit read in the same run."""
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
from tests.util import build_D, build_G  # noqa: E402

ENGINES = ("AdvStep", "ClusterAdvStep", "EsatAdvStep")
KS = (1, 2, 3)


def build_engine(name, k):
    from advmil_b200 import step
    kind = {"AdvStep": "abmil", "ClusterAdvStep": "cluster", "EsatAdvStep": "patch"}[name]
    shapes = {"abmil": O.G_SHAPES(), "cluster": O.G_CLUSTER_SHAPES(1024, 384), "patch": O.G_ESAT_SHAPES(1024, 384)}[kind]
    G, D = build_G((1024, 384, 384), mode=kind), build_D()
    G.load_state_dict(O.synth_state_dict(shapes, 402))
    D.load_state_dict(O.synth_state_dict(O.D_SHAPES(), 403))
    return getattr(step, name)(G, D, precision="bf16", gen_updates=k)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--prof-steps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gen_updates_bench.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    info = gpu_info()
    lib = _lib.load()
    Ns = [16384] * 16
    B = len(Ns)
    x = torch.cat([O.synth_bag(16384, 400 + i) for i in range(B)]).to(torch.bfloat16).cuda()
    bags = ops.PackedBags(x, Ns)
    ts, es = O.synth_labels(B, 401)
    ts, es, vis = ts.cuda(), es.cuda(), torch.ones(B, dtype=torch.uint8, device="cuda")
    ext = torch.randint(0, 8, (sum(Ns),), generator=torch.Generator().manual_seed(404), dtype=torch.int32).cuda()
    confs = [(n, k) for n in ENGINES for k in KS]
    engines = {c: build_engine(*c) for c in confs}

    def one(c):
        kw = {"ext": ext} if c[0] == "ClusterAdvStep" else {}
        engines[c].step(bags, ts, es, vis, **kw)

    times = {c: [] for c in confs}
    for rep in range(args.warmup + args.steps):
        for c in confs:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            one(c)
            torch.cuda.synchronize()
            if rep >= args.warmup:
                times[c].append(time.perf_counter() - t0)
    emb = _lib.PROF_TAGS.index("embed_fwd")
    prof = {c: [0.0, 0] for c in confs}
    for rep in range(args.prof_steps):
        for c in confs:
            torch.cuda.synchronize()
            profile_read(lib)
            lib.advmil_profile_enable(1)
            one(c)
            torch.cuda.synchronize()
            lib.advmil_profile_enable(0)
            ms, cnt = profile_read(lib)
            prof[c][0] += ms[emb]
            prof[c][1] += cnt[emb]
    res = {"device": info, "bags": B, "rows_per_bag": 16384, "C": 1024, "precision": "bf16", "steps": args.steps,
           "warmup": args.warmup, "prof_steps": args.prof_steps, "configs": {}}
    for name, k in confs:
        t = 1e3 * np.array(times[(name, k)])
        row = {"step_ms_median": float(np.median(t)), "step_ms_min": float(t.min()), "step_ms_max": float(t.max()),
               "embed_fwd_launches_per_step": prof[(name, k)][1] / args.prof_steps,
               "embed_fwd_ms_per_step": prof[(name, k)][0] / args.prof_steps}
        res["configs"][f"{name}_gen_updates{k}"] = row
        print(f"{name} gen_updates={k}", json.dumps(row), flush=True)
    res["device_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()

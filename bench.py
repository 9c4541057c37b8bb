#!/usr/bin/env python
"""bags/sec of one full adversarial G+D train step (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision bf16|tf32x3|tf32|fp32] [--impl reference]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): AdvMIL-ABMIL, synthetic bags of 16,384 x 1024 features, 16 bags per optimiser
step and per GPU (bp_every_batch, config/cfg_nlst.yaml:71) = 512 MiB (bf16) / 1 GiB (fp32) of features per step per GPU
(>> 126 MB L2, two alternating steps: no L2 flush needed).  A "step" = _update_disc + _update_gen
(model/model_handler.py:349-498): both forward/backward passes and both Adam updates.  Weak scaling: every rank owns 16
bags; gradients all-reduced (NCCL).

Printed JSON line
  value / ms_per_step   device-timed bags/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e                   the same through the public API (DeviceFeeder + AdvStep) with the pinned-host -> device copy of
                        every step's bags and a device -> host read of the losses inside the timed region
  roofline              dominant kernel class from live CUDA events; peak = burst figure for a timed region under 1 s,
                        sustained otherwise (MEASURED_PEAKS.json)
  modes                 the other precision modes of configs[1] (fp32 = exact FFMA, tf32x3 = split-tf32 tensor cores,
                        tf32), short legs under the same timing rules
  configs               configs[2] ragged packed bags (sharded with shard_bags_balanced under --gpus N), configs[3]
                        DeepAttMISL cluster generator, configs[4] semi-supervised (60 % labelled)
  sustained             the default step held for >= 3 s with NVML clocks / power
  dropin_handler        the reference's UNMODIFIED MyHandler._update_disc/_update_gen around the advmil_b200 modules
  gpu_eager_baseline    the same unmodified handler around the reference's own modules `.cuda()` on the same B200
  cpu_baseline          ... and on this box's host cores (kind "reference" when oracle/_ref is staged, else the oracle port)
`--impl reference` times only that CPU path (the reference arm of the driver).
`--dump-outputs DIR` writes what the last timed step produced as DIR/<name>.npy (see dump_outputs); the inputs, weights,
noise and dropout seeds depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import contextlib
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace as NS

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "bags/sec per G+D train step (16k x 1024 bags)"
N_ROWS, C_IN, BAGS_PER_STEP = 16384, 1024, 16
FLOP_PER_ROW = {  # algorithmic FLOPs per instance row per launch (SURVEY.md §8d)
    "proj_fwd": 2 * 1024 * 384, "gate_fwd": 2 * 384 * 768 + 768, "embed_fwd": 2 * 1024 * 128,
    "proj_embed_fwd": 2 * 1024 * (384 + 128),      # K1 + K5 in one pass over x (stacked weights)
    "bwd_data": 2 * 768 * 384, "bwd_w_gate": 2 * 768 * 384, "bwd_w_proj": 2 * 384 * 1024, "bwd_w_embed": 2 * 128 * 1024,
}
PRECISION_DTYPE = {"fp32": "f32", "tf32": "tf32", "tf32x3": "tf32x3 (split tf32, fp32-grade)", "bf16": "bf16"}


def bytes_per_row(es):
    """Algorithmic HBM bytes per instance row per launch for the streaming kernels; es = bytes per activation element
    (4 in the fp32/tf32 modes, 2 in the bf16 mode).  pool: read h + s, write w; pool_gate_bwd: read h, ab, write dAB;
    ln_bwd: read y_pre, write dy (+ d_emb/16); colsum: read dh; dropout: read h_eval, write h."""
    return {"pool_fwd": 384 * es + 8, "pool_gate_bwd": 384 * es + 2 * 768 * es + 8, "ln_bwd": 2 * 128 * es + 32,
            "colsum": 384 * es, "dropout": 2 * 384 * es}


def load_peaks(timed_region_s):
    """Roofline denominators.  MEASURED_PEAKS.json holds a burst bf16 figure (best of 10 back-to-back matmuls at full clocks)
    and a sustained one (4 s loop, clocks pulled down by the power cap): a timed region under one second runs in the
    burst regime, a longer one in the sustained regime."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    burst = timed_region_s < 1.0
    if os.path.exists(path):
        d = json.load(open(path))
        tf = d["bf16_tflops"] if burst else d.get("bf16_tflops_sustained", d["bf16_tflops"])
        return {"hbm_gbs": d["hbm_gbs"], "tflops": tf, "src": "measured", "kind": "burst" if burst else "sustained"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "src": "fallback (B200_PROFILING.md)", "kind": "fallback"}


class NvmlSampler(threading.Thread):
    """Samples SM clocks / power / throttle reasons through NVML every 10 ms while a timed region runs (the recipe's clocks
    line, B200_PROFILING.md; nvidia-smi's own start-up is longer than a short timed region)."""

    def __init__(self, gpu_index=0, period=0.01):
        super().__init__(daemon=True)
        self.gpu, self.period, self.rows, self._stop_evt, self.ok = gpu_index, period, [], threading.Event(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                ids = [v for v in vis.split(",") if v.strip() != ""]
                if gpu_index < len(ids) and ids[gpu_index].strip().isdigit():
                    idx = int(ids[gpu_index])
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    reasons = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    watts = float("nan")
                self.rows.append((mhz, reasons, time.perf_counter(), watts))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self, t0=None, t1=None):
        """t0, t1: perf_counter bounds of the timed region; only samples taken inside it are reported."""
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        if t0 is not None:
            inside = [r for r in self.rows if t0 <= r[2] <= t1]
            self.rows = inside if inside else self.rows[-3:]
        if not self.ok or not self.rows:
            return None
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                "hw_power_brake_slowdown": 0x80}
        seen = set()
        for r in self.rows:
            for name, b in bits.items():
                if r[1] & b:
                    seen.add(name)
        watts = [r[3] for r in self.rows if r[3] == r[3]]
        return {"sm_mhz": float(np.median([r[0] for r in self.rows])), "sm_max_mhz": self.max_mhz, "reasons": sorted(seen),
                "samples": len(self.rows), "power_w_median": float(np.median(watts)) if watts else None,
                "power_w_max": float(np.max(watts)) if watts else None, "source": "nvml"}


class ClockSampler(threading.Thread):
    """Fallback: samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    ok = True

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self, t0=None, t1=None):
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_sampler(local_rank):
    s = NvmlSampler(local_rank)
    return s if s.ok else ClockSampler(local_rank)


# ------------------------------------------------------------------------------------------------------
# Reference legs: the reference's own modules / losses / optimiser factory under its UNMODIFIED handler methods
# (oracle/ref_harness.py; staged copy oracle/_ref on the GPU box).  Fallback: the oracle port.
# ------------------------------------------------------------------------------------------------------
def _reference_available():
    try:
        from oracle import ref_import
        return ref_import.available()
    except Exception:
        return False


def _synthetic_labels(n, seed=42):
    rng = np.random.default_rng(seed)
    t = [float(rng.uniform(0.02, 0.98)) for _ in range(n)]
    e = [float(rng.uniform() < 0.347) for _ in range(n)]
    e[0] = 1.0
    return t, e


def handler_leg(impl, device, feats, steps, warmup, precision=None, cfg_over=None):
    """bags/s of `_update_disc` + `_update_gen` (model_handler.py:328-335) of the unmodified MyHandler over `feats`
    (list of fp32 [N, 1024] tensors already on `device`), 16 bags per optimiser step like the reference's loop.
    impl 'reference' = the reference's modules, 'advmil_b200' = the drop-in modules (four-import swap)."""
    import tempfile

    from oracle import ref_harness as H
    tmp = tempfile.mkdtemp(prefix="advmil_bench_")
    cfg = H.load_cfg(path_patch=tmp, path_label=os.path.join(tmp, "none.csv"), data_split_path=os.path.join(tmp, "s{}.npz"),
                     save_path=os.path.join(tmp, "run"), bcb_mode="abmil", **(cfg_over or {}))
    if precision is not None:
        import advmil_b200
        saved = advmil_b200.get_precision()
        advmil_b200.set_precision(precision)
    try:
        h = H.make_handler(cfg, impl, device)
        nb = len(feats)
        t, e = _synthetic_labels(nb)
        dev = feats[0].device
        xs = [[f.unsqueeze(0), torch.Tensor([0]).unsqueeze(0).to(dev)] for f in feats]
        ys = [torch.tensor([[t[i], e[i]]], device=dev) for i in range(nb)]
        times = []
        launches = None
        with H.device_context(device):
            for it in range(warmup + steps):
                if dev.type == "cuda":
                    torch.cuda.synchronize()
                t0 = time.perf_counter()
                H.handler_step(h, 16 * (it + 1), xs, ys)
                if dev.type == "cuda":
                    torch.cuda.synchronize()
                if it >= warmup:
                    times.append(time.perf_counter() - t0)
            if dev.type == "cuda":
                try:
                    from torch.profiler import ProfilerActivity, profile
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        H.handler_step(h, 16, xs, ys)
                        torch.cuda.synchronize()
                    launches = sum(1 for ev in prof.events() if str(ev.device_type).endswith("CUDA") and "memcpy" not in ev.name.lower()
                                   and "memset" not in ev.name.lower())
                except Exception:
                    launches = None
        mean_s = float(np.mean(times))
        return {"value": nb / mean_s, "unit": "bags/s", "ms_per_step": mean_s * 1e3, "bags_per_step": nb, "steps": steps,
                "warmup": warmup, "gpu_launches_per_step": launches}
    finally:
        if precision is not None:
            advmil_b200.set_precision(saved)


def cpu_reference_leg(n_rows, bags, steps, warmup, threads=None):
    """The reference's CPU path on this box's host cores: its own modules, losses and optimiser factory under the unmodified
    `_update_disc` / `_update_gen` (kind 'reference'); the oracle port when the staged tree is missing (kind 'port')."""
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    gen = torch.Generator().manual_seed(42)
    if _reference_available():
        feats = [torch.randn(n_rows, C_IN, generator=gen) for _ in range(bags)]
        r = handler_leg("reference", "cpu", feats, steps, warmup)
        return {"value": r["value"], "unit": "bags/s", "cores": threads, "kind": "reference", "ms_per_step": r["ms_per_step"],
                "same_config": bags == BAGS_PER_STEP and n_rows == N_ROWS,
                "sample": f"{steps} steps x {bags} bags of {n_rows}x1024 fp32 after {warmup} warm-up: the reference's own "
                          "G/D modules, losses and Adam under the unmodified MyHandler._update_disc/_update_gen "
                          "(oracle/_ref, `.cuda()` shimmed to identity), torch CPU fp32"}
    from oracle import advmil_oracle as O
    tr = O.CpuTrainer(O.synth_state_dict(O.G_SHAPES(), 42), O.synth_state_dict(O.D_SHAPES(), 43))
    xs = [torch.randn(n_rows, C_IN, generator=gen) for _ in range(bags)]
    ts, es = O.synth_labels(bags, 42)
    es[0] = 1.0
    times = []
    for it in range(warmup + steps):
        nzd = [torch.rand(1, 192) for _ in xs]
        nzg = [torch.rand(1, 192) for _ in xs]
        gm = [O.random_g_masks(n_rows, 384, 384, gen) for _ in xs]
        dmr = [O.random_d_masks(n_rows // 16, 128, gen) for _ in xs]
        dmf = [O.random_d_masks(n_rows // 16, 128, gen) for _ in xs]
        t0 = time.perf_counter()
        tr.step(xs, ts, es, [True] * bags, nzd, nzg, dmr, dmf, gm)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    mean_s = float(np.mean(times))
    return {"value": bags / mean_s, "unit": "bags/s", "cores": threads, "kind": "port", "ms_per_step": mean_s * 1e3,
            "same_config": False,
            "sample": f"{steps} steps x {bags} bags of {n_rows}x1024 after {warmup} warm-up, oracle port (reference tree not staged)"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    cb = cpu_reference_leg(args.rows, args.bags, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "bags/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"AdvMIL-ABMIL G+D step, {args.bags} synthetic bags of {args.rows}x1024 fp32 per step (configs[1]); "
                               "D step + G step + both Adam updates",
                   "sample": cb["sample"]},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config")},
        "e2e": {"value": cb["value"], "unit": "bags/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# product-side helpers
# ------------------------------------------------------------------------------------------------------
def build_networks(dev, backbone="abmil"):
    """G and D exactly as MyHandler.__init__ builds them from config/cfg_nlst.yaml (model_handler.py:74-91), from the
    advmil_b200 modules; init_weights on G only (:81)."""
    from advmil_b200.model.backbone import load_backbone
    from advmil_b200.model.GANSurv import Generator, PrjDiscriminator
    from advmil_b200.model.model_utils import init_weights
    with contextlib.redirect_stdout(sys.stderr):              # the modules print the reference's [info] lines
        G = Generator(384, 1, load_backbone(backbone, [C_IN, 384, 384]), NS(noise=[0, 1], hops=1, noise_dist="uniform"), False, 0.6,
                      "sigmoid")
        G.apply(init_weights)
        D = PrjDiscriminator(NS(in_dim=C_IN, out_dim=128, ksize=1, backbone="avgpool", dropout=0.25),
                             NS(in_dim=1, hid_dims=[64, 128], norm=False, dropout=0.0), prj_path="x", inner_product="instance")
    return G.to(dev), D.to(dev)


class Ctx:
    def __init__(self, args, rank, world, local_rank):
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.dev = torch.device("cuda", local_rank)

    def barrier(self):
        if self.world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = torch.tensor([float(v)], device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        t = torch.tensor([float(v)], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM)
        return float(t.item())


def timed(ctx, fn, steps, warmup):
    """W untimed + K timed calls of fn(i) between barrier + synchronize; CUDA events on the launching stream, max over ranks.
    Returns (ms for the K steps, host issue ms per step)."""
    import gc
    for i in range(warmup):
        fn(i)
    # the cyclic garbage collector stays out of the timed region (as timeit does): a generation-2 pass over the interpreter's
    # objects costs tens of ms, which doubled the 10-step host-bound legs (ModuleAdvStep) in two runs out of three
    gc.collect()
    gc_was_enabled = gc.isenabled()
    gc.disable()
    try:
        ctx.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        th0 = time.perf_counter()
        for i in range(steps):
            fn(warmup + i)
        host_ms = (time.perf_counter() - th0) * 1e3 / steps
        ev1.record()
        ctx.barrier()
    finally:
        if gc_was_enabled:
            gc.enable()
    return ctx.max_over_ranks(ev0.elapsed_time(ev1)), host_ms


def resident_steps(ctx, steps):
    from advmil_b200 import ops
    out = []
    for st in steps:
        out.append((ops.PackedBags(st.x.to(ctx.dev), st.lengths), st.t.to(ctx.dev), st.e.to(ctx.dev), st.visible.to(ctx.dev)))
    return out


def local_counts(st):
    return (float(((st.e == 1) & (st.visible != 0)).sum()), float(len(st.lengths)), float(st.visible.sum()))


def dump_outputs(out_dir, out, engine):
    """`--dump-outputs`: the tensors the engine's step returned (losses, per-bag predictions and discriminator outputs, the
    real-pair mask) and the flat G / D parameters that step left behind after both Adam updates, as out_dir/<name>.npy in
    float32 (about 5 MB for the ABMIL networks).  Call it after the timed region and before anything else steps the engine."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v for k, v in out.items() if isinstance(v, torch.Tensor)}
    arrays.update(params_G=engine.G.flat, params_D=engine.D.flat)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def leg_mode(ctx, precision, res_bf16, counts, steps, warmup):
    """configs[1] in another precision mode: the same bags (the bf16 values widened to fp32 on the device -- exactly
    representable), a fresh pair of networks and engine."""
    from advmil_b200 import ops
    from advmil_b200.step import AdvStep
    G, D = build_networks(ctx.dev)
    eng = AdvStep(G, D, precision=precision)
    res = [(ops.PackedBags(b.x.float(), b.lengths), t, e, v) for (b, t, e, v) in res_bf16[:2]]
    nz = torch.rand(len(res[0][0].lengths), 192, device=ctx.dev)

    def one(i):
        b, t, e, v = res[i % len(res)]
        return eng.step(b, t, e, v, noise_d=nz, noise_g=nz, global_counts=counts[i % len(res)])
    ms, _ = timed(ctx, one, steps, warmup)
    nb = len(res[0][0].lengths)
    out = {"value": nb * ctx.world * steps / (ms / 1e3), "unit": "bags/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "dtype": PRECISION_DTYPE[precision]}
    del eng, res
    torch.cuda.empty_cache()
    return out


def leg_ragged(ctx, precision, steps, warmup):
    """configs[2]: 16 x world packed bags per step with lengths log-uniform in [1024, 100000] (multiples of 16), sharded
    over the ranks by greedy row balancing (dataset/packed.shard_bags_balanced); NCCL all-reduce of the flat gradients."""
    from advmil_b200 import ops
    from advmil_b200.dataset.packed import loguniform_rows, shard_bags_balanced
    from advmil_b200.step import AdvStep
    args = ctx.args
    G, D = build_networks(ctx.dev)
    eng = AdvStep(G, D, precision=precision)
    feat_dtype = torch.bfloat16 if precision == "bf16" else torch.float32
    draw = loguniform_rows()
    res, counts, rows_local, rows_global = [], [], [], []
    for k in range(2):
        rng = np.random.default_rng(4242 + k)                       # every rank draws the same global step ...
        lens = [draw(rng) for _ in range(args.bags * ctx.world)]
        t, e = _synthetic_labels(len(lens), 77 + k)
        mine = shard_bags_balanced(lens, ctx.world)[ctx.rank]        # ... and keeps its balanced shard
        g = torch.Generator(device=ctx.dev).manual_seed(1000 + 10 * k + ctx.rank)
        x = torch.randn(sum(lens[i] for i in mine), C_IN, device=ctx.dev, generator=g).to(feat_dtype)
        res.append((ops.PackedBags(x, [lens[i] for i in mine]), torch.tensor([t[i] for i in mine], device=ctx.dev),
                    torch.tensor([e[i] for i in mine], device=ctx.dev), torch.ones(len(mine), dtype=torch.uint8, device=ctx.dev)))
        counts.append((float(sum(e)), float(len(lens)), float(len(lens))))
        rows_local.append(sum(lens[i] for i in mine))
        rows_global.append(sum(lens))
    nzs = [torch.rand(len(r[0].lengths), 192, device=ctx.dev) for r in res]

    def one(i):
        b, t, e, v = res[i % 2]
        return eng.step(b, t, e, v, noise_d=nzs[i % 2], noise_g=nzs[i % 2], global_counts=counts[i % 2])
    ms, _ = timed(ctx, one, steps, warmup)
    out = {"value": args.bags * ctx.world * steps / (ms / 1e3), "unit": "bags/s", "ms_per_step": ms / steps, "steps": steps,
           "warmup": warmup, "rows_per_step_global": int(np.mean(rows_global)),
           "rows_per_step_this_rank": int(np.mean(rows_local)), "rows_per_s": float(np.mean(rows_global)) * steps / (ms / 1e3),
           "bags_per_step_global": args.bags * ctx.world, "sharding": "shard_bags_balanced (greedy by rows)",
           "data": "synthetic, generated on the device (this leg has no end-to-end number)"}
    del eng, res
    torch.cuda.empty_cache()
    return out


def leg_cluster(ctx, precision, res_main, counts, steps, warmup):
    """configs[3]: DeepAttMISL generator (8 clusters, ids per row) + RLIP discriminator through step.ModuleAdvStep."""
    from advmil_b200.step import ModuleAdvStep
    G, D = build_networks(ctx.dev, "cluster")
    eng = ModuleAdvStep(G, D, precision=precision)
    b0 = res_main[0][0]
    g = torch.Generator(device=ctx.dev).manual_seed(7)
    cid = torch.randint(0, 8, (b0.rows,), device=ctx.dev, generator=g).float()
    cid[:b0.lengths[0]][cid[:b0.lengths[0]] == 5] = 4.0                 # bag 0 has an empty cluster (model/backbone.py:114-115)
    nz = torch.rand(len(b0.lengths), 192, device=ctx.dev)

    def one(i):
        b, t, e, v = res_main[i % len(res_main)]
        return eng.step(b, t, e, v, noise_d=nz, noise_g=nz, global_counts=counts[i % len(res_main)], ext=cid)
    ms, _ = timed(ctx, one, steps, warmup)
    out = {"value": len(b0.lengths) * ctx.world * steps / (ms / 1e3), "unit": "bags/s", "ms_per_step": ms / steps, "steps": steps,
           "warmup": warmup, "engine": "ModuleAdvStep", "clusters": 8, "empty_cluster_in_bag0": True}
    del eng
    torch.cuda.empty_cache()
    return out


def leg_ssl(ctx, precision, res_main, steps, warmup):
    """configs[4]: semi-supervised step -- 60 % of the bags labelled (ssl_num_labeled, cfg:88): unlabelled bags feed only
    fake pairs to D and no reconstruction loss to G (model_handler.py:361-377,473-481); RLIP at 16 patches per region."""
    from advmil_b200.step import AdvStep
    G, D = build_networks(ctx.dev)
    eng = AdvStep(G, D, precision=precision)
    nb = len(res_main[0][0].lengths)
    rng = np.random.default_rng(5)
    vis_h = (rng.uniform(size=nb) < 0.6).astype(np.uint8)
    vis_h[0] = 1
    vis = torch.tensor(vis_h, device=ctx.dev)
    cnts = []
    for (b, t, e, v) in res_main:
        eh = e.cpu().numpy()
        cnts.append((float(((eh == 1) & (vis_h != 0)).sum()) * ctx.world, float(nb * ctx.world), float(vis_h.sum()) * ctx.world))
    nz = torch.rand(nb, 192, device=ctx.dev)

    def one(i):
        b, t, e, v = res_main[i % len(res_main)]
        return eng.step(b, t, e, vis, noise_d=nz, noise_g=nz, global_counts=cnts[i % len(res_main)])
    ms, _ = timed(ctx, one, steps, warmup)
    out = {"value": nb * ctx.world * steps / (ms / 1e3), "unit": "bags/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "labelled_bags": int(vis_h.sum()), "bags": nb}
    del eng
    torch.cuda.empty_cache()
    return out


def leg_sustained(ctx, one_step, bags, seconds, ms_per_step_hint):
    """The default step held for `seconds`: what the step does once the power cap pulls the clocks down."""
    n = max(50, int(seconds * 1e3 / max(ms_per_step_hint, 0.05)))
    sampler = make_sampler(ctx.local_rank)
    for i in range(3):
        one_step(i)
    ctx.barrier()
    if ctx.rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    th0 = time.perf_counter()
    ev0.record()
    for i in range(n):
        one_step(i)
    ev1.record()
    ctx.barrier()
    clocks = sampler.stop(th0, time.perf_counter()) if ctx.rank == 0 else None
    ms = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    return {"value": bags * ctx.world * n / (ms / 1e3), "unit": "bags/s", "ms_per_step": ms / n, "steps": n, "seconds": ms / 1e3,
            "clocks": clocks}


# ------------------------------------------------------------------------------------------------------
def run_esat(args, rank, world, local_rank):
    """`--backbone patch`: the same metric for the ESAT generator (DualTrans_HS, bcb_mode patch; the reference's default
    backbone) with the RLIP discriminator, through step.ModuleAdvStep.  Same shape, timing rules and JSON keys as the ABMIL
    line; the roofline object is the self-attention forward kernel against the tf32 tensor peak (half the measured bf16
    figure: MEASURED_PEAKS.json holds no tf32 number)."""
    from advmil_b200 import _lib, ops
    from advmil_b200.dataset.packed import DeviceFeeder, synthetic_steps
    from advmil_b200.step import EsatAdvStep, ModuleAdvStep

    ctx = Ctx(args, rank, world, local_rank)
    dev = ctx.dev
    lib = _lib.load()
    torch.manual_seed(42)
    G, D = build_networks(dev, "patch")
    # the C-fused ESAT step (advmil_adv_step_esat_disc / _gen); ADVMIL_ESAT_ENGINE=module times the Python-composed ModuleAdvStep
    use_c = os.environ.get("ADVMIL_ESAT_ENGINE", "c") != "module"
    eng = (EsatAdvStep if use_c else ModuleAdvStep)(G, D, precision=args.precision)
    feat_dtype = torch.bfloat16 if args.precision == "bf16" else torch.float32
    steps = synthetic_steps(args.warmup + args.steps, args.bags, args.rows, C_IN, seed=42 + rank, distinct=2, dtype=feat_dtype)
    resident = resident_steps(ctx, steps[:2])
    nz = torch.rand(args.bags, 192, device=dev)
    counts = [tuple(c * world for c in local_counts(s)) for s in steps[:2]]

    def one_step(i):
        b, t, e, v = resident[i % 2]
        return eng.step(b, t, e, v, noise_d=nz, noise_g=nz, global_counts=counts[i % 2])

    sampler = make_sampler(local_rank)
    if rank == 0:
        sampler.start()
    for i in range(args.warmup):
        one_step(i)
    ctx.barrier()
    lib.advmil_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    th0 = time.perf_counter()
    for i in range(args.steps):
        out = one_step(args.warmup + i)
    ev1.record()
    ctx.barrier()
    clocks = sampler.stop(th0, time.perf_counter()) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, eng)
    launches = int(lib.advmil_launch_count(0))
    ms_dev = ctx.max_over_ranks(ev0.elapsed_time(ev1))
    value = args.bags * world * args.steps / (ms_dev / 1e3)
    ntags = len(_lib.PROF_TAGS)
    pms, pcnt = (C.c_double * ntags)(), (C.c_int64 * ntags)()
    prof_steps = min(args.steps, 10)
    lib.advmil_profile_enable(1)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for i in range(prof_steps):
        one_step(i)
    pe1.record()
    torch.cuda.synchronize()
    lib.advmil_profile_enable(0)
    lib.advmil_profile_read(pms, pcnt, ntags)
    prof_ms = pe0.elapsed_time(pe1)
    R = args.rows // 16
    pair_flop = 2.0 * 48 * 8 * args.bags * R * R                    # one [R, R] x 48 contraction over 8 heads and all bags
    flop = {"attn_fwd": 2 * pair_flop, "attn_bwd": 5 * pair_flop}   # algorithmic: S, PV / S, dP, dV, dK, dQ
    kern = {}
    for i, tag in enumerate(_lib.PROF_TAGS):
        if pcnt[i]:
            avg = pms[i] / pcnt[i]
            kern[tag] = {"ms_per_launch": avg, "launches_per_step": pcnt[i] / prof_steps, "share_of_step": pms[i] / prof_ms}
            if tag in flop:
                kern[tag]["tflops"] = flop[tag] / (avg * 1e-3) / 1e12
    peaks = load_peaks(ms_dev / 1e3)
    roof = None
    if "attn_fwd" in kern and args.precision != "fp32":
        roof = {"kernel": "attn_fwd", "bound": "tensor", "achieved": kern["attn_fwd"]["tflops"], "peak": peaks["tflops"] / 2, "unit": "TFLOP/s",
                "frac": kern["attn_fwd"]["tflops"] / (peaks["tflops"] / 2), "traffic": None,
                "peak_source": f"{peaks['src']} bf16 {peaks['kind']} / 2 (tf32 operands; tcgen05 forward kernel, eval and train launches averaged)"}
    p12 = args.precision == "bf16" and args.transport in ("p12", "vl")
    if p12:
        for st in steps[:2]:
            st.packvl() if args.transport == "vl" else st.pack12()
    it = iter(DeviceFeeder(steps, device=dev, depth=2))
    h2d = steps[0].nbytes
    for i in range(args.warmup):
        s = next(it)
        o = eng.step(s.bags, s.t, s.e, s.visible, global_counts=s.counts if world == 1 else None)
        float(o["losses"][0] if use_c else o["dis_loss"])
    ctx.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        s = next(it)
        o = eng.step(s.bags, s.t, s.e, s.visible, global_counts=s.counts if world == 1 else None)
        if use_c:
            ld = eng.loss_dict(o)                                                                   # device -> host read of the result
            host = [ld[k] for k in ("dis_loss", "gen_loss", "t_reg_loss", "gen_total_loss")]
        else:
            host = [float(o[k]) for k in ("dis_loss", "gen_loss", "t_reg_loss", "gen_total_loss")]     # device -> host read of the result
    e1.record()
    ctx.barrier()
    wall = time.perf_counter() - t0
    ems = ctx.max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3))
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "bags/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": PRECISION_DTYPE[args.precision], "data": "synthetic",
                "config": {"workload": f"AdvMIL-ESAT (bcb_mode patch: DualTrans_HS generator, RLIP discriminator) G+D step, {args.bags} "
                                       f"synthetic bags of {args.rows}x1024 per step per GPU; D step + G step + both Adam updates",
                           "rows_per_step_per_gpu": args.bags * args.rows, "precision_mode": args.precision,
                           "engine": "EsatAdvStep (C-fused: advmil_adv_step_esat_disc/gen)" if use_c else "ModuleAdvStep (Python-composed)",
                           "l2": "inputs (two alternating steps of 512 MiB or more) larger than the 126 MB L2; no flush",
                           "parallelism": f"dp{world} (bags sharded, NCCL all-reduce of flat G/D grads)"},
                "e2e": {"value": args.bags * world * args.steps / (ems / 1e3), "unit": "bags/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": 16, "transport": args.transport if p12 else "raw"},
                "gpu_launches": launches, "roofline": roof, "kernels": kern, "cpu_baseline": None, "clocks": clocks,
                "losses_last_step": dict(zip(("dis_loss", "gen_loss", "t_reg_loss", "gen_total_loss"), host))}
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
def run_main(args, rank, world, local_rank):
    import advmil_b200
    from advmil_b200 import _lib, ops
    from advmil_b200.dataset.packed import DeviceFeeder, loguniform_rows, synthetic_steps
    from advmil_b200.step import AdvStep

    ctx = Ctx(args, rank, world, local_rank)
    dev = ctx.dev
    lib = _lib.load()
    # NUMA: pin this rank to its GPU's cores before the pinned staging memory is allocated (first touch)
    from advmil_b200.dataset.packed import bind_host_to_gpu
    numa = bind_host_to_gpu(local_rank, ranks_on_node=world, local_rank=local_rank) if world > 1 else {"bound": False}
    if numa.get("bound"):
        torch.set_num_threads(max(1, min(numa["cpus"], 8)))
    advmil_b200.set_precision(args.precision)
    torch.manual_seed(42)
    G, D = build_networks(dev)
    engine = AdvStep(G, D, precision=args.precision)

    # ---- synthetic bags in pinned host memory: 2 distinct steps cycled ----
    n_total = args.warmup + args.steps
    feat_dtype = torch.bfloat16 if args.precision == "bf16" else torch.float32     # the packed loader's storage format
    steps = synthetic_steps(n_total, args.bags, loguniform_rows() if args.ragged else args.rows, C_IN, seed=42 + rank,
                            distinct=2, dtype=feat_dtype)

    # ================= (A) device-resident timing: `value` =================
    resident = resident_steps(ctx, steps[:2])
    nz = [torch.rand(args.bags, 192, device=dev) for _ in range(2)]
    hostcounts = [tuple(c * world for c in local_counts(s)) for s in steps[:2]]

    def one_step(i):
        b, t, e, v = resident[i % 2]
        return engine.step(b, t, e, v, noise_d=nz[0], noise_g=nz[1], global_counts=hostcounts[i % 2])

    sampler = make_sampler(local_rank)
    if rank == 0:
        sampler.start()             # started before the warm-up: nothing but the timed loop sits between the barriers
    for i in range(args.warmup):
        one_step(i)
    ctx.barrier()
    lib.advmil_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    th0 = time.perf_counter()
    for i in range(args.steps):
        out = one_step(args.warmup + i)
    host_ms = (time.perf_counter() - th0) * 1e3 / args.steps      # CPU time to ISSUE one step (no sync inside the loop)
    ev1.record()
    ctx.barrier()
    clocks = sampler.stop(th0, time.perf_counter()) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, engine)
    ms = ev0.elapsed_time(ev1)
    launches = int(lib.advmil_launch_count(0))
    # per-kernel-class CUDA-event timing in a SEPARATE pass (the event records perturb the step, so they stay out of the
    # timed region above); shares are relative to this pass's own step time
    ntags = len(_lib.PROF_TAGS)
    pms, pcnt = (C.c_double * ntags)(), (C.c_int64 * ntags)()
    prof_steps = min(args.steps, 10)
    lib.advmil_profile_enable(1)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for i in range(prof_steps):
        one_step(args.warmup + args.steps + i)
    pe1.record()
    torch.cuda.synchronize()
    lib.advmil_profile_enable(0)
    lib.advmil_profile_read(pms, pcnt, ntags)
    prof_ms = pe0.elapsed_time(pe1)
    ms_dev = ctx.max_over_ranks(ms)
    value = args.bags * world * args.steps / (ms_dev / 1e3)
    losses = engine.loss_dict(out)

    # ================= (B) end-to-end through the public API: pinned host -> device every step =================
    p12 = args.precision == "bf16" and args.transport in ("p12", "vl")
    if p12:
        for st in steps[:2]:      # done once, at packing time (the list cycles the same two steps)
            st.packvl() if args.transport == "vl" else st.pack12()
    feeder = DeviceFeeder(steps, device=dev, depth=2)
    it = iter(feeder)
    h2d = steps[0].nbytes
    for i in range(args.warmup):
        s = next(it)
        o = engine.step(s.bags, s.t, s.e, s.visible, global_counts=s.counts if world == 1 else None)
        engine.loss_dict(o)
    ctx.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    d2h = 0
    for i in range(args.steps):
        s = next(it)
        o = engine.step(s.bags, s.t, s.e, s.visible, global_counts=s.counts if world == 1 else None)
        host = o["losses"].tolist()      # device -> host read of the step's result
        d2h = len(host) * 4
    e1.record()
    ctx.barrier()
    wall = time.perf_counter() - t0
    ems = ctx.max_over_ranks(max(e0.elapsed_time(e1), wall * 1e3))
    e2e_value = args.bags * world * args.steps / (ems / 1e3)
    del it, feeder

    # ================= roofline of the dominant kernel class =================
    peaks = load_peaks(ms_dev / 1e3)
    rows_per_launch = int(np.mean([sum(st.lengths) for st in steps[:2]]))
    BYTES_PER_ROW = bytes_per_row(2 if args.precision == "bf16" else 4)
    kern = {}
    for i, tag in enumerate(_lib.PROF_TAGS):
        if pcnt[i] == 0:
            continue
        avg_ms = pms[i] / pcnt[i]
        ent = {"ms_per_launch": avg_ms, "launches_per_step": pcnt[i] / prof_steps, "share_of_step": pms[i] / prof_ms}
        if tag in FLOP_PER_ROW:
            ent["tflops"] = FLOP_PER_ROW[tag] * rows_per_launch / (avg_ms * 1e-3) / 1e12
        if tag in BYTES_PER_ROW:
            ent["gbs"] = BYTES_PER_ROW[tag] * rows_per_launch / (avg_ms * 1e-3) / 1e9
        kern[tag] = ent
    rated = [k for k in kern if k in FLOP_PER_ROW or k in BYTES_PER_ROW]      # composites (latency-bound) have no roofline
    top = max(rated, key=lambda k: kern[k]["share_of_step"]) if rated else None
    roof = None
    traffic = None
    for tname in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if top is not None and traffic is None and os.path.exists(tpath):
            tj = json.load(open(tpath))
            tm = tj.get(args.precision, {})
            if tj.get("rows_per_launch") == rows_per_launch and top in tm:
                traffic = tm[top]["read"] + tm[top]["write"]   # bytes per launch from the committed ncu --set full capture
    if top is not None:
        # in the tf32 modes the tensor peak is half the bf16 figure (MEASURED_PEAKS.json holds no tf32 number)
        tpeak = peaks["tflops"] * (1.0 if args.precision == "bf16" else 0.5)
        if top in FLOP_PER_ROW:
            roof = {"kernel": top, "bound": "tensor", "achieved": kern[top]["tflops"], "peak": tpeak,
                    "unit": "TFLOP/s", "frac": kern[top]["tflops"] / tpeak, "traffic": traffic,
                    "peak_source": f"{peaks['src']} bf16 {peaks['kind']}" + ("" if args.precision == "bf16" else " / 2 (tf32 operands)"),
                    "peak_rule": "timed region %.3f s: %s" % (ms_dev / 1e3, "burst (< 1 s, full clocks)" if peaks["kind"] == "burst" else peaks["kind"])}
        else:
            roof = {"kernel": top, "bound": "hbm", "achieved": kern[top]["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": kern[top]["gbs"] / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peaks["src"]}

    extras = {}
    if not args.no_extra_legs and not args.ragged:
        es, ew = min(args.steps, 10), 3
        # ---- configs[2]: ragged packed bags, sharded over the ranks (every N) ----
        extras.setdefault("configs", {})["ragged"] = leg_ragged(ctx, args.precision, es, ew)
        if world == 1:
            # ---- the other precision modes of configs[1] ----
            modes = {}
            for mode in ("tf32", "tf32x3", "fp32"):
                if mode == args.precision:
                    continue
                try:
                    modes[mode] = leg_mode(ctx, mode, resident, hostcounts, 3 if mode == "fp32" else es, ew)
                except Exception as ex:       # a mode that cannot run must show up as such, not vanish
                    modes[mode] = {"error": str(ex)[:300]}
            extras["modes"] = modes
            extras["configs"]["cluster"] = leg_cluster(ctx, args.precision, resident, hostcounts, es, ew)
            extras["configs"]["ssl"] = leg_ssl(ctx, args.precision, resident, es, ew)
        # ---- sustained: the default step for >= 3 s ----
        extras["sustained"] = leg_sustained(ctx, one_step, args.bags, args.sustained_seconds, ms_dev / args.steps)

    # ================= handler legs and CPU baseline (rank 0, N=1 only; bounded samples) =================
    cpu = dropin = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.ragged:
        have_ref = _reference_available()
        if have_ref and not args.no_extra_legs:
            feats32 = [resident[0][0].x[o:o + n].float() for o, n in zip(resident[0][0].offsets_list[:-1], resident[0][0].lengths)]
            try:
                eager = handler_leg("reference", "cuda", feats32, 5, 3)
                eager.update(note="the reference's own modules `.cuda()` fp32 under the unmodified MyHandler._update_disc/_update_gen on "
                                  "this B200 (stock settings: cuDNN conv may use TF32, matmul fp32); 16 device-resident bags per step",
                             same_config=True)
            except Exception as ex:
                eager = {"error": str(ex)[:300]}
            try:
                dropin = {}
                for mode in dict.fromkeys([args.precision, "fp32"]):
                    dropin[mode] = handler_leg("advmil_b200", "cuda", feats32, 5, 3, precision=mode)
                dropin["note"] = ("the same unmodified handler methods around the advmil_b200 modules (four-import swap, per-bag "
                                  "calls, torch autograd between the modules, torch.optim.Adam): what a user gets without touching "
                                  "the training loop; the fused AdvStep (`value`) replaces that loop")
            except Exception as ex:
                dropin = {"error": str(ex)[:300]}
            del feats32
            torch.cuda.empty_cache()
        cb = cpu_reference_leg(args.rows, args.bags if have_ref else 1, 3, 1)
        cpu = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "same_config", "ms_per_step")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "bags/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": PRECISION_DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": (f"AdvMIL-ABMIL G+D step, {args.bags} synthetic bags of {args.rows}x1024 per step per GPU "
                                    "(configs[1]); D step + G step + both Adam updates") if not args.ragged else
                                   (f"AdvMIL-ABMIL G+D step, {args.bags} packed bags per step per GPU with lengths log-uniform in "
                                    f"[1024, 100000] (configs[2]; mean {rows_per_launch} rows per step)"),
                       "rows_per_step_per_gpu": rows_per_launch,
                       "precision_mode": args.precision,
                       "feature_format": ("bf16 (packed loader's bf16 storage: features rounded once at packing time, fp32 "
                                          "accumulation/statistics/parameters)" if args.precision == "bf16" else "fp32"),
                       "l2": f"inputs ({steps[0].x.numel() * steps[0].x.element_size() >> 20} MiB/step, two alternating "
                             "steps) larger than the 126 MB L2; no flush",
                       "parallelism": f"dp{world} (bags sharded, NCCL all-reduce of flat G/D grads)",
                       "tolerances": "fp32 / tf32x3 modes: 1e-5 norm-wise per tensor (|a-e| <= 1e-5 |e| + 1e-5 max|e|), full-size "
                                     "gradients within 4x the reference's own fp32-vs-fp64 error; bf16 mode: 2e-2 norm-wise "
                                     "(per-tensor measured errors in DESIGN.md §2)"},
            "e2e": {"value": e2e_value, "unit": "bags/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "h2d_gbs_per_gpu": h2d * args.steps / (ems / 1e3) / 1e9, "host_numa_binding": numa,
                    "transport": (("vl: the packed loader's lossless entropy-coded form of the bf16 features (8 bits sign+mantissa, "
                                   "canonical-Huffman exponent codes in 32 sub-streams per 4096 elements, sparse escapes; %.2f bits "
                                   "per element; encoded once at packing time like the bf16 rounding itself, held in pinned host "
                                   "memory), copied and decoded on the device inside the timed region" % (8.0 * steps[0].vl.nbytes / steps[0].vl.lo.numel()))
                                  if (p12 and args.transport == "vl") else
                                  "p12: the packed loader's lossless 12-bit form of the bf16 features (8 bits sign+mantissa, 4-bit "
                                  "exponent code, sparse escapes; encoded once at packing time like the bf16 rounding itself, held "
                                  "in pinned host memory), copied and decoded on the device inside the timed region"
                                  if p12 else "raw"),
                    "note": "pinned host -> device copy of every step's features overlapped with the previous step's compute "
                            "(DeviceFeeder); bound by the PCIe link when h2d_gbs_per_gpu is ~55 GB/s"},
            "gpu_launches": launches, "host_issue_ms_per_step": host_ms, "profiled_pass_ms_per_step": prof_ms / prof_steps,
            "roofline": roof, "kernels": kern, "cpu_baseline": cpu, "gpu_eager_baseline": eager, "dropin_handler": dropin,
            "clocks": clocks, "losses_last_step": losses,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="advmil_b200")
    ap.add_argument("--precision", default=os.environ.get("ADVMIL_PRECISION", "bf16"), choices=["bf16", "tf32", "tf32x3", "fp32"])
    ap.add_argument("--rows", type=int, default=N_ROWS)
    ap.add_argument("--bags", type=int, default=BAGS_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline and the two handler legs")
    ap.add_argument("--no-extra-legs", action="store_true", help="only the main line (value / e2e / roofline)")
    ap.add_argument("--sustained-seconds", type=float, default=3.0)
    ap.add_argument("--transport", default=os.environ.get("ADVMIL_TRANSPORT", "vl"), choices=["vl", "p12", "raw"],
                    help="end-to-end leg, bf16 mode: copy the features in the packed loader's lossless entropy-coded transport "
                         "format (vl, ~10.9 bits per element), its fixed 12-bit form (p12) -- both decoded on the device -- or as raw bf16")
    ap.add_argument("--backbone", default="abmil", choices=["abmil", "patch"],
                    help="generator backbone: abmil (the benchmark's workload, C-fused AdvStep) or patch (ESAT, C-fused EsatAdvStep)")
    ap.add_argument("--ragged", action="store_true",
                    help="main line on configs[2] instead of configs[1]: bag lengths log-uniform in [1024, 100000]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step and the parameters it left as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the timed GPU step; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    assert args.warmup >= 3, "timing rule: at least 3 warm-up steps"
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.backbone == "patch":
            run_esat(args, rank, world, local_rank)
        else:
            run_main(args, rank, world, local_rank)
    finally:
        if world > 1:
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()

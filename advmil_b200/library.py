"""torch.library registration of the hot-path operators (namespace `advmil_b200`).

The reference's "FFI" for this path is the nn.Module surface; north_star asks for the kernels to sit behind thin
torch.library / C-ABI custom ops.  The C ABI is `libadvmil_b200.so` (ctypes, `_lib.py`); this module registers the two
operators the drop-in modules call -- the packed generator and the packed discriminator, forward and backward -- as
`torch.library.custom_op`s with

  * a CUDA implementation that calls the C ABI (through the same `ops.generator_forward` / `ops.disc_*` glue),
  * a fake (meta) implementation that only computes output shapes, so FakeTensor tracing / `torch.compile` /
    `torch.export` of code that calls the modules sees ordinary operators with known shapes,
  * `register_autograd`: the backward is itself a registered operator (`*_bwd`), gradients flow to the parameters, the
    noise-conditioned prediction t (discriminator) and, in the fp32/tf32 modes, the bag rows (generator, optional).

Schema conventions: packed bags are (x [rows, C], offsets int32 [bags+1] on the device, lengths int[]); configuration
is an int[] + float[] pair (see `_gen_cfg` / `_disc_cfg`); parameters travel as `Tensor?[]` in the C ABI's tensor order
(`_lib.GEN_TENSORS` / `_lib.DISC_TENSORS`); injected dropout masks (parity tests) as `Tensor?[]`.

`ops.GeneratorFn` / `ops.DiscriminatorFn` (autograd.Function) remain for the ESAT and DeepAttMISL paths and as the
implementation the operators are checked against (tests/test_gpu_library.py)."""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch
from torch import Tensor

from . import _lib, ops

_GEN_MASKS = ("h", "a", "b", "rho", "mlp0")
_DISC_MASKS = ("fc1", "ga", "gs", "fc2")
_GEN_SAVED = ("h", "ab", "s", "w", "z", "H", "H1", "pre", "pred")
_HEAD_SAVED = ("f1", "fi", "ab", "rep", "attn", "bagv", "fbar", "g1", "hx", "u1", "ht", "out")


def _gen_cfg(icfg: Sequence[int], fcfg: Sequence[float]) -> ops.GenConfig:
    C, h, o, hid, n0, n1, scale, has_rho = [int(v) for v in icfg]
    return ops.GenConfig(C=C, h=h, o=o, hid=hid, noise0=n0, noise1=n1, out_scale=scale, p_backbone=float(fcfg[0]),
                         p_head=float(fcfg[1]), has_rho=bool(has_rho))


def gen_cfg_lists(cfg: ops.GenConfig):
    return ([cfg.C, cfg.h, cfg.o, cfg.hid, cfg.noise0, cfg.noise1, cfg.out_scale, int(cfg.has_rho)], [cfg.p_backbone, cfg.p_head])


def _disc_cfg(icfg: Sequence[int], fcfg: Sequence[float]) -> ops.DiscConfig:
    C, d, t1, t2, inner, prj, ksize = [int(v) for v in icfg]
    return ops.DiscConfig(C=C, d=d, t1=t1, t2=t2, inner_instance=inner, prj_path=prj, p=float(fcfg[0]), ln_eps=float(fcfg[1]),
                          ksize=ksize)


def disc_cfg_lists(cfg: ops.DiscConfig):
    return ([cfg.C, cfg.d, cfg.t1, cfg.t2, cfg.inner_instance, cfg.prj_path, cfg.ksize], [cfg.p, cfg.ln_eps])


_MODE = None


def use_registered_ops(mode=None) -> str:
    """How the drop-in modules reach the kernels: "auto" (default; env ADVMIL_REGISTERED_OPS) = through the registered
    operators whenever the call is being traced (torch.compile / torch.export / FakeTensor / meta tensors) and through the
    autograd.Function glue in plain eager mode, "1" = always through the registered operators, "0" = never.  Both paths run the
    same C entry points (tests/test_gpu_library.py checks them bit for bit); the dispatcher round trip of an operator with
    ~45 tensor arguments costs ~0.3 ms per call, which is a third of the reference handler's per-bag step on a B200."""
    global _MODE
    if mode is not None:
        _MODE = {True: "1", False: "0"}.get(mode, str(mode))
    if _MODE is None:
        import os
        _MODE = os.environ.get("ADVMIL_REGISTERED_OPS", "auto")
    return _MODE


def should_dispatch(x: Tensor) -> bool:
    mode = use_registered_ops()
    if mode == "1":
        return True
    if mode == "0":
        return False
    if x.device.type == "meta" or torch.compiler.is_compiling():
        return True
    from torch._subclasses.fake_tensor import FakeTensor
    return isinstance(x, FakeTensor)


def _masks(names, masks: Sequence[Optional[Tensor]]):
    return {k: m for k, m in zip(names, masks) if m is not None and m.numel()}


def _opt(ts: Sequence[Optional[Tensor]]):
    """Placeholders (0 elements) back to None."""
    return [None if (t is None or t.numel() == 0) else t for t in ts]


def _dense(ts: Sequence[Optional[Tensor]], like: Tensor):
    """Absent tensors -> 0-element placeholders.  torch.library's autograd glue treats a list argument that holds a None
    as an opaque leaf (no gradients flow into ANY of its tensors, and the backward must return a bare None for it); a list
    of tensors only is flattened and differentiated element-wise.  So the parameter and mask lists always travel dense."""
    return [like.new_empty(0, dtype=torch.float32) if t is None else t for t in ts]


def _act(precision: int):
    return ops.act_dtype(precision)


# =====================================================================================================
# generator
# =====================================================================================================
@torch.library.custom_op("advmil_b200::generator_fwd", mutates_args=(), device_types="cuda")
def generator_fwd(x: Tensor, offsets: Tensor, lengths: List[int], icfg: List[int], fcfg: List[float], noise0: Optional[Tensor],
                  noise1: Optional[Tensor], train: bool, seed: int, precision: int, save: bool, masks: List[Tensor],
                  params: List[Tensor]) -> List[Tensor]:
    """-> [out [bags] (pred, or H [bags, o] without a head), h, ab, s, w, z, H, H1, pre, pred] (ab empty unless `save`)."""
    cfg = _gen_cfg(icfg, fcfg)
    params = _opt(params)
    bags = ops.PackedBags(x, lengths, offsets=offsets)
    acts = ops.generator_forward(cfg, params, bags, noise0, noise1, train, seed, _masks(_GEN_MASKS, masks), precision, save=save)
    head = params[_lib.GEN_TENSORS.index("W0")] is not None
    out = (acts["pred"] if head else acts["H"]).clone()
    saved = [acts[k] if acts[k] is not None else x.new_empty(0) for k in _GEN_SAVED]
    return [out] + saved


@generator_fwd.register_fake
def _(x, offsets, lengths, icfg, fcfg, noise0, noise1, train, seed, precision, save, masks, params):
    cfg = _gen_cfg(icfg, fcfg)
    params = _opt(params)
    rows, nb = x.shape[0], len(lengths)
    f32 = dict(dtype=torch.float32, device=x.device)
    act = dict(dtype=_act(precision), device=x.device)
    abw = 128 * ((cfg.h + 63) // 64)
    head = params[_lib.GEN_TENSORS.index("W0")] is not None
    out = torch.empty(nb, **f32) if head else torch.empty(nb, cfg.o, **f32)
    return [out, torch.empty(rows, cfg.h, **act), torch.empty((rows, abw) if save else (0,), **act), torch.empty(rows, **f32),
            torch.empty(rows, **f32), torch.empty(nb, cfg.h, **f32), torch.empty(nb, cfg.o, **f32),
            torch.empty(nb, max(cfg.hid, 1), **f32), torch.empty(nb, **f32), torch.empty(nb, **f32)]


@torch.library.custom_op("advmil_b200::generator_bwd", mutates_args=(), device_types="cuda")
def generator_bwd(x: Tensor, offsets: Tensor, lengths: List[int], icfg: List[int], fcfg: List[float], noise0: Optional[Tensor],
                  noise1: Optional[Tensor], train: bool, seed: int, precision: int, masks: List[Tensor],
                  params: List[Tensor], saved: List[Tensor], d_out: Tensor, need_dx: bool) -> List[Tensor]:
    """-> gradients of the 14 generator tensors (empty for absent ones) + dx (empty unless need_dx)."""
    cfg = _gen_cfg(icfg, fcfg)
    params = _opt(params)
    bags = ops.PackedBags(x, lengths, offsets=offsets)
    acts = {k: (v if v.numel() else None) for k, v in zip(_GEN_SAVED, saved)}
    acts.update(noise0=None if noise0 is None else ops._f32c(noise0), noise1=None if noise1 is None else ops._f32c(noise1),
                h_eval=None, masks=_masks(_GEN_MASKS, masks), seed=int(seed), train=bool(train), precision=int(precision))
    grads, dx = ops.generator_backward(cfg, [None if p is None else p.detach() for p in params], bags, acts, d_out.contiguous(),
                                       need_dx=need_dx)
    return [g if g is not None else x.new_empty(0, dtype=torch.float32) for g in grads] + [dx if dx is not None else x.new_empty(0)]


@generator_bwd.register_fake
def _(x, offsets, lengths, icfg, fcfg, noise0, noise1, train, seed, precision, masks, params, saved, d_out, need_dx):
    return [torch.empty_like(p, dtype=torch.float32) for p in params] + \
           [torch.empty_like(x) if need_dx else x.new_empty(0)]


def _stash(ctx, output, tensors, lists):
    """Everything the backward needs goes through save_for_backward (outputs stored as plain attributes of the node would form
    a reference cycle output -> grad_fn -> ctx -> output that only the cyclic collector frees: activations of every bag
    of a step would pile up in HBM); the activation outputs are marked non-differentiable (no grad_fn, no zero-filled
    gradients materialised for them)."""
    flat, layout = [], []
    for t in tensors:
        layout.append(None if t is None else len(flat))
        if t is not None:
            flat.append(t)
    spans = []
    for ts in lists:
        spans.append((len(flat), len(ts)))
        flat.extend(ts)
    ctx.save_for_backward(*flat)
    ctx.layout, ctx.spans = layout, spans
    ctx.mark_non_differentiable(*output[1:])
    ctx.set_materialize_grads(False)


def _unstash(ctx):
    flat = ctx.saved_tensors
    return [None if i is None else flat[i] for i in ctx.layout], [list(flat[a:a + n]) for a, n in ctx.spans]


def _gen_setup(ctx, inputs, output):
    (x, offsets, lengths, icfg, fcfg, noise0, noise1, train, seed, precision, save, masks, params) = inputs
    ctx.args = (lengths, icfg, fcfg, train, seed, precision)
    _stash(ctx, output, [x, offsets, noise0, noise1], [masks, params, list(output[1:])])
    ctx.n_masks = len(masks)
    ctx.need_dx = bool(x.requires_grad)


def _gen_backward(ctx, grads):
    lengths, icfg, fcfg, train, seed, precision = ctx.args
    (x, offsets, noise0, noise1), (masks, params, saved) = _unstash(ctx)
    d_out = grads[0]
    none = (None,) * 11 + ([None] * ctx.n_masks,)
    if d_out is None:
        return none + ([None] * len(params),)
    res = generator_bwd(x, offsets, lengths, icfg, fcfg, noise0, noise1, train, seed, precision, masks, params, saved,
                        d_out.contiguous(), ctx.need_dx)
    n = len(params)
    pg = [res[i].reshape(p.shape) if p.numel() else None for i, p in enumerate(params)]
    dx = res[n] if ctx.need_dx else None
    return (dx,) + none[1:] + (pg,)


generator_fwd.register_autograd(_gen_backward, setup_context=_gen_setup)


def generator(cfg: ops.GenConfig, bags: ops.PackedBags, noise0, noise1, train: bool, seed: int, masks, precision: int,
              params: Sequence[Optional[Tensor]], x_grad: Optional[Tensor] = None) -> Tensor:
    """pred [bags] (or H [bags, o] in backbone-only mode) through the registered operator."""
    icfg, fcfg = gen_cfg_lists(cfg)
    need = any(p is not None and p.requires_grad for p in params) or (x_grad is not None and x_grad.requires_grad)
    m = masks or {}
    x = x_grad if (x_grad is not None and x_grad.requires_grad) else bags.x
    return torch.ops.advmil_b200.generator_fwd(x, bags.offsets, list(bags.lengths), icfg, fcfg, noise0, noise1, bool(train), int(seed),
                                               int(precision), bool(need), _dense([m.get(k) for k in _GEN_MASKS], x),
                                               _dense(params, x))[0]


# =====================================================================================================
# discriminator (region embedding + RLIP head)
# =====================================================================================================
@torch.library.custom_op("advmil_b200::discriminator_fwd", mutates_args=(), device_types="cuda")
def discriminator_fwd(x: Tensor, offsets: Tensor, lengths: List[int], icfg: List[int], fcfg: List[float], t: Tensor, train: bool,
                      seed: int, precision: int, save: bool, masks: List[Tensor],
                      params: List[Tensor]) -> List[Tensor]:
    """-> [out [bags], emb [R, d], y_pre [rows, d] (empty unless `save`), f1, fi, ab, rep, attn, bagv, fbar, g1, hx, u1, ht, out]."""
    cfg = _disc_cfg(icfg, fcfg)
    params = _opt(params)
    bags = ops.PackedBags(x, lengths, offsets=offsets)
    emb = ops.disc_embed_forward(cfg, params, bags, precision, save=save)
    head = ops.disc_head_forward(cfg, params, bags, emb["emb"], t.detach(), train, seed, _masks(_DISC_MASKS, masks), precision)
    y_pre = emb["y_pre"] if emb["y_pre"] is not None else x.new_empty(0)
    return [head["out"].clone(), emb["emb"], y_pre] + [head[k] for k in _HEAD_SAVED]


@discriminator_fwd.register_fake
def _(x, offsets, lengths, icfg, fcfg, t, train, seed, precision, save, masks, params):
    cfg = _disc_cfg(icfg, fcfg)
    rows, nb, R, d, dh = x.shape[0], len(lengths), x.shape[0] // 16, cfg.d, cfg.d // 2
    f = dict(dtype=torch.float32, device=x.device)
    abw = 128 * ((d + 63) // 64)
    e = torch.empty
    return [e(nb, **f), e(R, d, **f), e((rows, d) if save else (0,), dtype=_act(precision), device=x.device), e(R, dh, **f), e(R, d, **f),
            e(R, abw, **f), e(R, **f), e(R, **f), e(nb, d, **f), e(nb, d, **f), e(nb, dh, **f), e(nb, d, **f), e(nb, cfg.t1, **f),
            e(nb, cfg.t2, **f), e(nb, **f)]


@torch.library.custom_op("advmil_b200::discriminator_bwd", mutates_args=(), device_types="cuda")
def discriminator_bwd(x: Tensor, offsets: Tensor, lengths: List[int], icfg: List[int], fcfg: List[float], t: Tensor, train: bool,
                      seed: int, precision: int, masks: List[Tensor], params: List[Tensor], saved: List[Tensor],
                      d_out: Tensor, need_param_grads: bool, need_dt: bool) -> List[Tensor]:
    """-> gradients of the 24 discriminator tensors (empty when not requested / absent) + d_t [bags] (empty unless need_dt)."""
    cfg = _disc_cfg(icfg, fcfg)
    params = _opt(params)
    bags = ops.PackedBags(x, lengths, offsets=offsets)
    det = [None if p is None else p.detach() for p in params]
    emb, y_pre = saved[0], saved[1]
    head = dict(zip(_HEAD_SAVED, saved[2:]))
    head.update(emb=emb, t=ops._f32c(t.reshape(-1)), masks=_masks(_DISC_MASKS, masks), seed=int(seed), train=bool(train),
                precision=int(precision))
    dev = x.device
    d_t = torch.empty(bags.bags, dtype=torch.float32, device=dev) if need_dt else None
    grads, d_emb = None, None
    if need_param_grads:
        grads = [None if p is None else torch.empty_like(p, dtype=torch.float32) for p in det]
        d_emb = torch.empty_like(emb)
    ops.disc_head_backward(cfg, det, bags, head, d_out.contiguous(), d_emb, d_t, grads, accumulate=False)
    if need_param_grads:
        ops.disc_embed_backward(cfg, det, bags, {"emb": emb, "y_pre": y_pre if y_pre.numel() else None, "precision": int(precision)},
                                d_emb, grads, accumulate=False)
    def empty():                                          # one storage per output: operator outputs must not alias each other
        return x.new_empty(0, dtype=torch.float32)
    out = [empty() if (grads is None or g is None) else g for g in (grads if grads is not None else [None] * len(params))]
    return out + [d_t if d_t is not None else empty()]


@discriminator_bwd.register_fake
def _(x, offsets, lengths, icfg, fcfg, t, train, seed, precision, masks, params, saved, d_out, need_param_grads, need_dt):
    out = [torch.empty_like(p, dtype=torch.float32) if need_param_grads else x.new_empty(0, dtype=torch.float32) for p in params]
    return out + [torch.empty(len(lengths), dtype=torch.float32, device=x.device) if need_dt else x.new_empty(0, dtype=torch.float32)]


def _disc_setup(ctx, inputs, output):
    (x, offsets, lengths, icfg, fcfg, t, train, seed, precision, save, masks, params) = inputs
    ctx.args = (lengths, icfg, fcfg, train, seed, precision)
    _stash(ctx, output, [x, offsets, t], [masks, params, list(output[1:])])
    ctx.n_masks = len(masks)
    ctx.need_param_grads = bool(save)
    ctx.need_dt = bool(t.requires_grad)


def _disc_backward(ctx, grads):
    lengths, icfg, fcfg, train, seed, precision = ctx.args
    (x, offsets, t), (masks, params, saved) = _unstash(ctx)
    d_out = grads[0]
    none = (None,) * 10 + ([None] * ctx.n_masks,)
    if d_out is None:
        return none + ([None] * len(params),)
    res = discriminator_bwd(x, offsets, lengths, icfg, fcfg, t, train, seed, precision, masks, params, saved,
                            d_out.contiguous(), ctx.need_param_grads, ctx.need_dt)
    n = len(params)
    pg = [res[i].reshape(p.shape) if (p.numel() and ctx.need_param_grads) else None for i, p in enumerate(params)]
    d_t = res[n].reshape(t.shape) if ctx.need_dt else None
    return none[:5] + (d_t,) + none[6:] + (pg,)


discriminator_fwd.register_autograd(_disc_backward, setup_context=_disc_setup)


def discriminator(cfg: ops.DiscConfig, bags: ops.PackedBags, t: Tensor, train: bool, seed: int, masks, precision: int,
                  params: Sequence[Optional[Tensor]]) -> Tensor:
    """out [bags] = D(packed bags, t [bags]) through the registered operator."""
    icfg, fcfg = disc_cfg_lists(cfg)
    need = any(p is not None and p.requires_grad for p in params)
    m = masks or {}
    return torch.ops.advmil_b200.discriminator_fwd(bags.x, bags.offsets, list(bags.lengths), icfg, fcfg, t.reshape(-1), bool(train),
                                                   int(seed), int(precision), bool(need),
                                                   _dense([m.get(k) for k in _DISC_MASKS], bags.x), _dense(params, bags.x))[0]

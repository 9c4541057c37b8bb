"""Torch-side glue over the C ABI: packed bags, buffer allocation, autograd Functions.

PyTorch is plumbing here (device memory, streams, autograd graph edges); all arithmetic of the hot path
runs in libadvmil_b200.so.  Every function raises if the library is missing or a tensor is not on a CUDA
device: there is deliberately no CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib
from ._lib import (Bags, DiscGrads, DiscParams, EmbedActs, EsatActs, EsatGrads, EsatParams, GenActs, GenGrads, GenParams, HeadActs,
                   DISC_TENSORS, ESAT_TENSORS, GEN_TENSORS, check)

FP32, TF32, TF32X3, BF16 = 0, 1, 2, 3
PRECISIONS = {"fp32": FP32, "tf32": TF32, "tf32x3": TF32X3, "bf16": BF16}
ELEM_F32, ELEM_BF16 = 0, 1


def act_dtype(precision: int) -> torch.dtype:
    """Element type of the [rows, *] activation tensors (and of x) in a precision mode."""
    return torch.bfloat16 if int(precision) == BF16 else torch.float32


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(t: torch.Tensor, what: str):
    if not (t.is_cuda or t.device.type == "meta"):      # meta: shape-only tracing through the registered operators (library.py)
        raise _lib.AdvmilError(f"{what} must be a CUDA tensor: advmil_b200 has no CPU path")


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 copy of a CUDA tensor with the library's own kernel (advmil_cast_f32_to_bf16)."""
    lib = _lib.load()
    _need_cuda(x, "x")
    x = _f32c(x)
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    check(lib.advmil_cast_f32_to_bf16(x.data_ptr(), x.numel(), out.data_ptr(), _stream()), "advmil_cast_f32_to_bf16")
    return out


_CAST_CACHE: list = []   # [(data_ptr, version, shape, bf16 copy)], newest last


def _cached_cast(x: torch.Tensor) -> torch.Tensor:
    """The drop-in modules are called several times per bag with the same feature tensor (G and D, D step and G step,
    model/model_handler.py:383-461): keep the last two bf16 copies keyed on (pointer, version, shape)."""
    key = (x.data_ptr(), x._version, tuple(x.shape))
    for k in _CAST_CACHE:
        if k[:3] == key:
            return k[3]
    y = cast_bf16(x)
    _CAST_CACHE.append(key + (y, x))   # holding x keeps its address from being recycled while the entry lives
    if len(_CAST_CACHE) > 2:
        _CAST_CACHE.pop(0)
    return y


_OFFS_RING: dict = {}      # device -> [pinned int32 ring, next slot]
_OFFS_SLOT, _OFFS_SLOTS = 1024, 64


def _device_offsets(offs, device) -> torch.Tensor:
    """int32 offsets [bags + 1] on the device WITHOUT a host-device synchronisation: `torch.tensor(list, device=cuda)` is a
    pageable copy that blocks the host until the device has drained, once per module call in the reference's per-bag loop.
    One bag (the handler's batch_size 1): generated on the device (arange).  Several bags: staged through a ring of pinned
    slots and copied asynchronously (a slot is reused after 64 later calls; longer offset lists fall back to the blocking copy)."""
    if device.type != "cuda":
        return torch.tensor(offs, dtype=torch.int32, device=device)
    if len(offs) == 2 and offs[1] > 0:
        return torch.arange(0, offs[1] + 1, offs[1], dtype=torch.int32, device=device)
    if len(offs) > _OFFS_SLOT:
        return torch.tensor(offs, dtype=torch.int32, device=device)
    ring = _OFFS_RING.get(device)
    if ring is None:
        try:
            ring = [torch.empty(_OFFS_SLOTS, _OFFS_SLOT, dtype=torch.int32).pin_memory(), 0]
        except RuntimeError:
            return torch.tensor(offs, dtype=torch.int32, device=device)
        _OFFS_RING[device] = ring
    slot = ring[0][ring[1] % _OFFS_SLOTS, :len(offs)]
    ring[1] += 1
    slot.copy_(torch.tensor(offs, dtype=torch.int32))
    return slot.to(device, non_blocking=True)


class PackedBags:
    """Packed variable-length bags: x [rows, C] fp32 (or bf16 for the bf16 mode) + int32 offsets [bags+1] (AdvmilBags)."""

    def __init__(self, x: torch.Tensor, lengths: Sequence[int], offsets: Optional[torch.Tensor] = None):
        """offsets: optional int32 device tensor [bags+1] already holding the prefix sums of `lengths` (the asynchronous
        feeder copies it from pinned memory; building it here costs a synchronous pageable H2D copy)."""
        _need_cuda(x, "bag features")
        assert x.dim() == 2, "packed features must be [rows, C]"
        self.x = (x if x.is_contiguous() else x.contiguous()) if x.dtype == torch.bfloat16 else _f32c(x)
        self._alt = None
        self.lengths = [int(n) for n in lengths]
        assert sum(self.lengths) == self.x.shape[0], "bag lengths do not sum to the number of rows"
        offs = [0]
        for n in self.lengths:
            offs.append(offs[-1] + n)
        self.offsets_list = offs
        self.offsets_host = (C.c_int32 * len(offs))(*offs)
        self.offsets = _device_offsets(offs, x.device) if offsets is None else offsets
        self.rows, self.C = self.x.shape
        self.bags = len(self.lengths)

    @staticmethod
    def from_single(x: torch.Tensor) -> "PackedBags":
        """Accepts the reference's [1, N, C] (default_collate, batch_size 1) or [N, C]."""
        if x.dim() == 3:
            assert x.shape[0] == 1, "the reference path is batch_size == 1 (config/cfg_nlst.yaml:70)"
            x = x[0]
        return PackedBags(x, [x.shape[0]])

    @staticmethod
    def from_list(xs: Sequence[torch.Tensor]) -> "PackedBags":
        xs = [x[0] if x.dim() == 3 else x for x in xs]
        return PackedBags(torch.cat(xs, dim=0) if len(xs) > 1 else xs[0], [x.shape[0] for x in xs])

    @property
    def elem(self) -> int:
        return ELEM_BF16 if self.x.dtype == torch.bfloat16 else ELEM_F32

    def for_precision(self, precision: int) -> "PackedBags":
        """The same bags with x in the element type the precision mode computes on.  fp32 -> bf16 runs the library's cast
        kernel once and is cached; bf16 features cannot be widened back (load fp32 features for the fp32/tf32 modes)."""
        want = act_dtype(precision)
        if self.x.dtype == want:
            return self
        if want != torch.bfloat16:
            raise _lib.AdvmilError("bf16 bag features can only be used with the bf16 precision mode")
        if self._alt is None:
            alt = PackedBags.__new__(PackedBags)
            alt.__dict__.update(self.__dict__)
            alt.x = _cached_cast(self.x)
            alt._alt = None
            self._alt = alt
        return self._alt

    def c(self) -> Bags:
        return Bags(self.x.data_ptr(), self.offsets.data_ptr(), self.offsets_host, self.rows, self.bags, self.C,
                    max(self.lengths), self.elem)


# -------------------------------------------------------------------------------------------------
# generator
# -------------------------------------------------------------------------------------------------
@dataclass
class GenConfig:
    C: int
    h: int
    o: int
    hid: int
    noise0: int = 0
    noise1: int = 1
    out_scale: int = 1          # 0 none, 1 sigmoid, 2 exp
    p_backbone: float = 0.25
    p_head: float = 0.6
    has_rho: bool = True

    def c(self, params: Sequence[Optional[torch.Tensor]]) -> GenParams:
        s = GenParams()
        for name, t in zip(GEN_TENSORS, params):
            setattr(s, name, _ptr(t))
        s.C, s.h, s.o, s.hid = self.C, self.h, self.o, self.hid
        s.noise0, s.noise1, s.out_scale = self.noise0, self.noise1, self.out_scale
        s.p_backbone, s.p_head = self.p_backbone, self.p_head
        return s


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def generator_forward(cfg: GenConfig, params: Sequence[Optional[torch.Tensor]], bags: PackedBags,
                      noise0: Optional[torch.Tensor], noise1: Optional[torch.Tensor], train: bool = False,
                      seed: int = 0, masks: Optional[Dict[str, torch.Tensor]] = None, precision: int = FP32,
                      save: bool = True, h_eval: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """K1+K2+K3+K4 over packed bags.  Returns the activation dict (also what backward needs)."""
    lib = _lib.load()
    bags = bags.for_precision(precision)
    dev = bags.x.device
    rows, nb = bags.rows, bags.bags
    abw = lib.advmil_gate_packed_width(cfg.h)
    f = dict(dtype=torch.float32, device=dev)
    fa = dict(dtype=act_dtype(precision), device=dev)
    if h_eval is not None:
        assert h_eval.dtype == fa["dtype"], "h_eval must come from a forward in the same precision mode"
    acts = {
        "h": torch.empty(rows, cfg.h, **fa), "s": torch.empty(rows, **f), "w": torch.empty(rows, **f),
        "z": torch.empty(nb, cfg.h, **f), "H": torch.empty(nb, cfg.o, **f), "H1": torch.empty(nb, max(cfg.hid, 1), **f),
        "pre": torch.empty(nb, **f), "pred": torch.empty(nb, **f),
        "ab": torch.empty(rows, abw, **fa) if save else None,
        "noise0": None if noise0 is None else _f32c(noise0), "noise1": None if noise1 is None else _f32c(noise1),
        "h_eval": h_eval, "masks": masks or {}, "seed": int(seed), "train": bool(train), "precision": int(precision),
    }
    p = cfg.c(params)
    ws = _ws(lib.advmil_generator_workspace_bytes(C.byref(p), rows, nb, 0), dev)
    a = _gen_acts_struct(acts, ws)
    b = bags.c()
    check(lib.advmil_generator_fwd(C.byref(p), C.byref(b), C.byref(a), _stream()), "advmil_generator_fwd")
    return acts


def _gen_acts_struct(acts, ws) -> GenActs:
    a = GenActs()
    for k in ("h", "ab", "s", "w", "z", "H", "H1", "pre", "pred", "noise0", "noise1", "h_eval"):
        setattr(a, k, _ptr(acts.get(k)))
    m = acts["masks"]
    for k in ("h", "a", "b", "rho", "mlp0"):
        setattr(a, "mask_" + k, _ptr(m.get(k)))
    a.seed, a.train, a.precision = acts["seed"], int(acts["train"]), acts["precision"]
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    return a


def generator_backward(cfg: GenConfig, params, bags: PackedBags, acts, d_pred: torch.Tensor, need_dx: bool = False):
    """Returns (list of 14 parameter gradients, dx or None).  d_pred: [bags] (or dL/dH [bags,o] in backbone-only mode)."""
    lib = _lib.load()
    bags = bags.for_precision(acts["precision"])
    dev = bags.x.device
    p = cfg.c(params)
    grads = [None if t is None else torch.empty_like(t, dtype=torch.float32) for t in params]
    if need_dx and acts["precision"] == BF16:
        raise _lib.AdvmilError("gradients w.r.t. the bag features are not available in the bf16 mode")
    dx = torch.empty_like(bags.x) if need_dx else None
    g = GenGrads()
    for name, t in zip(GEN_TENSORS, grads):
        setattr(g, name, _ptr(t))
    g.dx = _ptr(dx)
    ws = _ws(lib.advmil_generator_workspace_bytes(C.byref(p), bags.rows, bags.bags, 1), dev)
    a = _gen_acts_struct(acts, ws)
    b = bags.c()
    d_pred = _f32c(d_pred.reshape(-1))
    check(lib.advmil_generator_bwd(C.byref(p), C.byref(b), C.byref(a), d_pred.data_ptr(), C.byref(g), _stream()),
          "advmil_generator_bwd")
    return grads, dx


def generator_sample(cfg: GenConfig, params, H: torch.Tensor, noise1: Optional[torch.Tensor], samples: int,
                     noise0: Optional[torch.Tensor] = None) -> torch.Tensor:
    """S head evaluations per bag from one backbone pass. H [bags,o]; noise1 [S,bags,hid] -> [S,bags]."""
    lib = _lib.load()
    p = cfg.c(params)
    nb = H.shape[0]
    out = torch.empty(samples, nb, dtype=torch.float32, device=H.device)
    check(lib.advmil_generator_sample(C.byref(p), _f32c(H).data_ptr(), _ptr(noise0), _ptr(noise1), nb, samples,
                                      out.data_ptr(), _stream()), "advmil_generator_sample")
    return out


class GeneratorFn(torch.autograd.Function):
    """pred[bags] = G(packed bags) (or H[bags,o] in backbone-only mode, W0 is None); gradients for the 14 generator
    tensors (K10) and, when `x_grad` (the tensor behind bags.x) requires grad, for the bag rows."""

    @staticmethod
    def forward(ctx, cfg, bags, x_grad, noise0, noise1, train, seed, masks, precision, *params):
        need = any(p is not None and p.requires_grad for p in params) or (x_grad is not None and x_grad.requires_grad)
        acts = generator_forward(cfg, params, bags, noise0, noise1, train, seed, masks, precision, save=need)
        ctx.cfg, ctx.bags, ctx.acts, ctx.params = cfg, bags, acts, params
        ctx.need_dx = x_grad is not None and x_grad.requires_grad
        ctx.x_shape = None if x_grad is None else x_grad.shape
        head = params[GEN_TENSORS.index("W0")] is not None
        return (acts["pred"] if head else acts["H"]).clone()

    @staticmethod
    def backward(ctx, d_out):
        grads, dx = generator_backward(ctx.cfg, [None if p is None else p.detach() for p in ctx.params], ctx.bags,
                                       ctx.acts, d_out.contiguous(), need_dx=ctx.need_dx)
        if dx is not None:
            dx = dx.reshape(ctx.x_shape)
        return (None, None, dx) + (None,) * 6 + tuple(grads)


# -------------------------------------------------------------------------------------------------
# ESAT backbone (DualTrans_HS, reference model/backbone.py:171-196) + noise head
# -------------------------------------------------------------------------------------------------
@dataclass
class EsatConfig:
    C: int
    d: int
    ff: int
    nhead: int = 8
    p: float = 0.25
    ln_eps: float = 1e-5

    def c(self, params: Sequence[Optional[torch.Tensor]]) -> EsatParams:
        s = EsatParams()
        for name, t in zip(ESAT_TENSORS, params):
            setattr(s, name, _ptr(t))
        s.C, s.d, s.ff, s.nhead, s.p, s.ln_eps = self.C, self.d, self.ff, self.nhead, self.p, self.ln_eps
        return s


def sincos_pe(coord: torch.Tensor, bags: PackedBags, d: int) -> torch.Tensor:
    """compute_pe (reference model/backbone_utils.py:79-99) for packed bags: coord [R,2] integer region coordinates ->
    PE [R,d].  omega is evaluated exactly as the reference evaluates it (d/4 values); the kernel does the rest."""
    lib = _lib.load()
    _need_cuda(coord, "coord")
    assert coord.dim() == 2 and coord.shape[1] == 2 and coord.shape[0] == bags.rows // 16, "one (x, y) per 16-row region"
    assert d % 4 == 0, "feature dimension must be multiple of 4 for sincos emb"
    omega = torch.arange(d // 4) / (d // 4 - 1)
    omega = (1.0 / (10000 ** omega)).to(torch.float32).to(coord.device)
    c = coord.to(torch.int64).contiguous()
    pe = torch.empty(c.shape[0], d, dtype=torch.float32, device=coord.device)
    ws = _ws(4096, coord.device)
    check(lib.advmil_sincos_pe(c.data_ptr(), bags.offsets.data_ptr(), bags.bags, d, omega.data_ptr(), pe.data_ptr(), ws.data_ptr(),
                               ws.numel(), _stream()), "advmil_sincos_pe")
    return pe


def _esat_structs(cfg: EsatConfig, head: Optional[GenConfig], params, head_params, acts, ws):
    p = cfg.c(params)
    hp = None
    if head is not None:
        hp = head.c([None] * 10 + list(head_params))
    a = EsatActs()
    for n in _lib.ESAT_ACTS:
        setattr(a, n, _ptr(acts.get(n)))
    a.pe, a.noise0, a.noise1 = _ptr(acts.get("pe")), _ptr(acts.get("noise0")), _ptr(acts.get("noise1"))
    m = acts["masks"]
    a.mask_attn, a.mask_attn_off = _ptr(m.get("attn")), _ptr(m.get("attn_off"))
    for k in ("sa", "ff1", "ff2", "ga", "gs", "mlp0"):
        setattr(a, "mask_" + k, _ptr(m.get(k)))
    a.seed, a.train, a.precision = acts["seed"], int(acts["train"]), acts["precision"]
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    a.emb_ready = int(bool(acts.get("emb_ready")))
    return p, hp, a


def esat_prepare_masks(masks, bags: PackedBags, nhead: int):
    """Injected keep masks (tests): 'attn' may be a list of per-bag [nhead, R_b, R_b] tensors; it is flattened and its
    per-bag element offsets are added as 'attn_off'."""
    if not masks:
        return {}
    m = {k: v for k, v in masks.items() if k != "attn"}
    if masks.get("attn") is not None:
        per_bag = masks["attn"] if isinstance(masks["attn"], (list, tuple)) else [masks["attn"]]
        assert len(per_bag) == bags.bags
        offs, tot = [], 0
        for t, n in zip(per_bag, bags.lengths):
            assert tuple(t.shape) == (nhead, n // 16, n // 16), "attention mask of a bag is [nhead, R_b, R_b]"
            offs.append(tot)
            tot += t.numel()
        m["attn"] = torch.cat([t.reshape(-1) for t in per_bag]).to(torch.uint8).contiguous()
        m["attn_off"] = torch.tensor(offs, dtype=torch.int64, device=bags.x.device)
    return {k: (v if k == "attn_off" else v.to(torch.uint8).contiguous()) for k, v in m.items()}


def esat_forward(cfg: EsatConfig, head: Optional[GenConfig], params, head_params, bags: PackedBags, pe=None, noise0=None,
                 noise1=None, train=False, seed=0, masks=None, precision: int = FP32, reuse=None) -> Dict[str, torch.Tensor]:
    """reuse: the activation dict of an earlier forward over the SAME bags, positional embedding and conv / norm
    parameters (e.g. the eval pass of the D step): its patch embedding (y_pre, emb) is shared instead of recomputed."""
    lib = _lib.load()
    bags = bags.for_precision(precision)
    dev = bags.x.device
    rows, nb, R, d = bags.rows, bags.bags, bags.rows // 16, cfg.d
    abw = lib.advmil_gate_packed_width(d)
    f = dict(dtype=torch.float32, device=dev)
    acts = {"y_pre": torch.empty(rows, d, dtype=act_dtype(precision), device=dev), "emb": torch.empty(R, d, **f),
            "qkv": torch.empty(R, 3 * d, **f), "lse": torch.empty(cfg.nhead, R, **f), "ctx": torch.empty(R, d, **f),
            "s1": torch.empty(R, d, **f), "x1": torch.empty(R, d, **f), "f": torch.empty(R, cfg.ff, **f),
            "s2": torch.empty(R, d, **f), "x2": torch.empty(R, d, **f), "ab": torch.empty(R, abw, **f),
            "rep": torch.empty(R, **f), "attn": torch.empty(R, **f), "H": torch.empty(nb, d, **f),
            "pe": None if pe is None else _f32c(pe), "noise0": None if noise0 is None else _f32c(noise0),
            "noise1": None if noise1 is None else _f32c(noise1), "masks": esat_prepare_masks(masks, bags, cfg.nhead),
            "seed": int(seed), "train": bool(train), "precision": int(precision)}
    if head is not None:
        acts.update(H1=torch.empty(nb, head.hid, **f), pre=torch.empty(nb, **f), pred=torch.empty(nb, **f))
    if reuse is not None:
        assert reuse["precision"] == int(precision) and reuse["y_pre"].shape == acts["y_pre"].shape
        acts.update(y_pre=reuse["y_pre"], emb=reuse["emb"], emb_ready=True)
    p0, hp0 = cfg.c(params), (None if head is None else head.c([None] * 10 + list(head_params)))
    ws = _ws(lib.advmil_esat_workspace_bytes(C.byref(p0), None if hp0 is None else C.byref(hp0), rows, nb, 0), dev)
    p, hp, a = _esat_structs(cfg, head, params, head_params, acts, ws)
    b = bags.c()
    check(lib.advmil_esat_fwd(C.byref(p), None if hp is None else C.byref(hp), C.byref(b), C.byref(a), _stream()), "advmil_esat_fwd")
    return acts


def esat_backward(cfg: EsatConfig, head: Optional[GenConfig], params, head_params, bags: PackedBags, acts, d_out: torch.Tensor):
    lib = _lib.load()
    bags = bags.for_precision(acts["precision"])
    dev = bags.x.device
    grads = [None if t is None else torch.empty_like(t, dtype=torch.float32) for t in params]
    hgrads = [None if t is None else torch.empty_like(t, dtype=torch.float32) for t in head_params]
    g = EsatGrads()
    for n, t in zip(ESAT_TENSORS, grads):
        setattr(g, n, _ptr(t))
    hg = GenGrads()
    for n, t in zip(GEN_TENSORS[10:], hgrads):
        setattr(hg, n, _ptr(t))
    p0, hp0 = cfg.c(params), (None if head is None else head.c([None] * 10 + list(head_params)))
    ws = _ws(lib.advmil_esat_workspace_bytes(C.byref(p0), None if hp0 is None else C.byref(hp0), bags.rows, bags.bags, 1), dev)
    p, hp, a = _esat_structs(cfg, head, params, head_params, acts, ws)
    b = bags.c()
    d_out = _f32c(d_out)
    check(lib.advmil_esat_bwd(C.byref(p), None if hp is None else C.byref(hp), C.byref(b), C.byref(a), d_out.data_ptr(), C.byref(g),
                              None if head is None else C.byref(hg), _stream()), "advmil_esat_bwd")
    return grads, hgrads


class EsatFn(torch.autograd.Function):
    """pred[bags] (with a head) or H[bags,d] of the ESAT generator over packed bags; gradients for the 22 backbone tensors
    and the 4 head tensors.  The bag features get no gradient (they are pre-extracted inputs)."""

    @staticmethod
    def forward(ctx, cfg, head, bags, pe, noise0, noise1, train, seed, masks, precision, reuse, sink, *tensors):
        """sink: optional list that receives this forward's activation dict (the caller that wants to share the patch
        embedding with a later pass over the same bags -- step.ModuleAdvStep -- owns it; nothing is kept globally)."""
        params, head_params = tensors[:len(ESAT_TENSORS)], tensors[len(ESAT_TENSORS):]
        acts = esat_forward(cfg, head, params, head_params, bags, pe, noise0, noise1, train, seed, masks, precision, reuse=reuse)
        if sink is not None:
            sink.append(acts)
        ctx.cfg, ctx.head, ctx.bags, ctx.acts, ctx.tensors = cfg, head, bags, acts, tensors
        return (acts["pred"] if head is not None else acts["H"]).clone()

    @staticmethod
    def backward(ctx, d_out):
        n = len(ESAT_TENSORS)
        det = [None if t is None else t.detach() for t in ctx.tensors]
        grads, hgrads = esat_backward(ctx.cfg, ctx.head, det[:n], det[n:], ctx.bags, ctx.acts, d_out.contiguous())
        return (None,) * 12 + tuple(grads) + tuple(hgrads)


# -------------------------------------------------------------------------------------------------
# discriminator
# -------------------------------------------------------------------------------------------------
@dataclass
class DiscConfig:
    C: int
    d: int
    t1: int
    t2: int
    inner_instance: int = 1
    prj_path: int = 1
    p: float = 0.25
    ln_eps: float = 1e-5
    ksize: int = 1          # patch-embedding conv kernel: 1 (per-patch linear) or 3 (3x3 inside each 4x4 region)

    def c(self, params) -> DiscParams:
        s = DiscParams()
        for name, t in zip(DISC_TENSORS, params):
            setattr(s, name, _ptr(t))
        s.C, s.d, s.t1, s.t2 = self.C, self.d, self.t1, self.t2
        s.inner_instance, s.prj_path, s.p, s.ln_eps, s.ksize = self.inner_instance, self.prj_path, self.p, self.ln_eps, self.ksize
        return s


def disc_embed_forward(cfg: DiscConfig, params, bags: PackedBags, precision: int = FP32, save: bool = True):
    lib = _lib.load()
    bags = bags.for_precision(precision)
    dev = bags.x.device
    assert bags.rows % 16 == 0 and all(n % 16 == 0 for n in bags.lengths), \
        "every bag must hold a multiple of 16 instances (model/backbone_utils.py:65)"
    acts = {"emb": torch.empty(bags.rows // 16, cfg.d, dtype=torch.float32, device=dev),
            "y_pre": torch.empty(bags.rows, cfg.d, dtype=act_dtype(precision), device=dev) if save else None,
            "precision": int(precision)}
    p = cfg.c(params)
    # the exact-fp32 FFMA embedding at d = 256 (fp32 mode; tf32 / tf32x3 below one 128-row tile or at C % 32 != 0) runs its
    # LayerNorm as a second pass over y: scratch for y when y_pre is not kept
    ffma = int(precision) == FP32 or (int(precision) != BF16 and (bags.rows < 128 or cfg.C % 32 != 0))
    ws = torch.empty(bags.rows * cfg.d * 4, dtype=torch.uint8, device=dev) if not save and cfg.d > 128 and ffma else None
    a = EmbedActs(acts["emb"].data_ptr(), _ptr(acts["y_pre"]), int(precision), _ptr(ws), 0 if ws is None else ws.numel())
    b = bags.c()
    check(lib.advmil_disc_embed_fwd(C.byref(p), C.byref(b), C.byref(a), _stream()), "advmil_disc_embed_fwd")
    return acts


def disc_embed_backward(cfg: DiscConfig, params, bags: PackedBags, acts, d_emb: torch.Tensor, grads, accumulate=False):
    lib = _lib.load()
    bags = bags.for_precision(acts["precision"])
    p = cfg.c(params)
    ws = _ws(lib.advmil_disc_workspace_bytes(C.byref(p), bags.rows, bags.bags, 1), bags.x.device)
    a = EmbedActs(acts["emb"].data_ptr(), _ptr(acts["y_pre"]), acts["precision"], ws.data_ptr(), ws.numel())
    g = _disc_grads_struct(grads)
    b = bags.c()
    check(lib.advmil_disc_embed_bwd(C.byref(p), C.byref(b), C.byref(a), _f32c(d_emb).data_ptr(), C.byref(g),
                                    int(accumulate), _stream()), "advmil_disc_embed_bwd")


def _disc_grads_struct(grads) -> DiscGrads:
    g = DiscGrads()
    for name, t in zip(DISC_TENSORS, grads):
        setattr(g, name, _ptr(t))
    return g


def _head_struct(acts, ws) -> HeadActs:
    a = HeadActs()
    for k in ("emb", "t", "f1", "fi", "ab", "rep", "attn", "bagv", "fbar", "g1", "hx", "u1", "ht", "out"):
        setattr(a, k, _ptr(acts[k]))
    m = acts["masks"]
    for k in ("fc1", "ga", "gs", "fc2"):
        setattr(a, "mask_" + k, _ptr(m.get(k)))
    a.seed, a.train, a.precision = acts["seed"], int(acts["train"]), int(acts.get("precision", FP32))
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    return a


def disc_head_forward(cfg: DiscConfig, params, bags: PackedBags, emb: torch.Tensor, t: torch.Tensor,
                      train: bool = False, seed: int = 0, masks=None, precision: int = FP32):
    lib = _lib.load()
    dev = bags.x.device
    R, nb, d, dh = bags.rows // 16, bags.bags, cfg.d, cfg.d // 2
    abw = lib.advmil_gate_packed_width(d)
    f = dict(dtype=torch.float32, device=dev)
    acts = {"emb": emb, "t": _f32c(t.reshape(-1)), "f1": torch.empty(R, dh, **f), "fi": torch.empty(R, d, **f),
            "ab": torch.empty(R, abw, **f), "rep": torch.empty(R, **f), "attn": torch.empty(R, **f),
            "bagv": torch.empty(nb, d, **f), "fbar": torch.empty(nb, d, **f), "g1": torch.empty(nb, dh, **f),
            "hx": torch.empty(nb, d, **f), "u1": torch.empty(nb, cfg.t1, **f), "ht": torch.empty(nb, cfg.t2, **f),
            "out": torch.empty(nb, **f), "masks": masks or {}, "seed": int(seed), "train": bool(train),
            "precision": int(precision)}
    p = cfg.c(params)
    ws = _ws(lib.advmil_disc_workspace_bytes(C.byref(p), bags.rows, nb, 0), dev)
    a = _head_struct(acts, ws)
    b = bags.c()
    check(lib.advmil_disc_head_fwd(C.byref(p), C.byref(b), C.byref(a), _stream()), "advmil_disc_head_fwd")
    return acts


def disc_head_backward(cfg: DiscConfig, params, bags: PackedBags, acts, d_out: torch.Tensor,
                       d_emb: Optional[torch.Tensor], d_t: Optional[torch.Tensor], grads, accumulate=False):
    """grads: list of 24 tensors (or None to skip parameter gradients)."""
    lib = _lib.load()
    p = cfg.c(params)
    ws = _ws(lib.advmil_disc_workspace_bytes(C.byref(p), bags.rows, bags.bags, 1), bags.x.device)
    a = _head_struct(acts, ws)
    b = bags.c()
    g = _disc_grads_struct(grads) if grads is not None else None
    check(lib.advmil_disc_head_bwd(C.byref(p), C.byref(b), C.byref(a), _f32c(d_out.reshape(-1)).data_ptr(), _ptr(d_emb),
                                   _ptr(d_t), C.byref(g) if g is not None else None, int(accumulate), _stream()),
          "advmil_disc_head_bwd")


class DiscriminatorFn(torch.autograd.Function):
    """out[bags] = D(packed bags, t[bags]); gradients for t and the 24 discriminator tensors."""

    @staticmethod
    def forward(ctx, cfg, bags, t, train, seed, masks, precision, *params):
        need_param_grads = any(p is not None and p.requires_grad for p in params)
        emb = disc_embed_forward(cfg, params, bags, precision, save=need_param_grads)
        head = disc_head_forward(cfg, params, bags, emb["emb"], t.detach(), train, seed, masks, precision)
        ctx.cfg, ctx.bags, ctx.emb, ctx.head, ctx.params = cfg, bags, emb, head, params
        ctx.need_param_grads = need_param_grads
        ctx.t_shape = t.shape
        return head["out"].clone()

    @staticmethod
    def backward(ctx, d_out):
        cfg, bags, params = ctx.cfg, ctx.bags, [None if p is None else p.detach() for p in ctx.params]
        d_t = torch.empty(bags.bags, dtype=torch.float32, device=bags.x.device) if ctx.needs_input_grad[2] else None
        grads = None
        d_emb = None
        if ctx.need_param_grads:
            grads = [None if t is None else torch.empty_like(t, dtype=torch.float32) for t in params]
            d_emb = torch.empty_like(ctx.emb["emb"])
        disc_head_backward(cfg, params, bags, ctx.head, d_out.contiguous(), d_emb, d_t, grads, accumulate=False)
        if ctx.need_param_grads:
            disc_embed_backward(cfg, params, bags, ctx.emb, d_emb, grads, accumulate=False)
        out_grads = tuple(grads) if grads is not None else (None,) * len(params)
        return (None, None, None if d_t is None else d_t.reshape(ctx.t_shape), None, None, None, None) + out_grads


class DiscEmbedFn(torch.autograd.Function):
    """emb[R, d] = AVGPoolPatchEmbedding(packed bags) (K5+K6) as its own autograd node: several head passes over the same
    bags (the real and the fake pairs of a D step) share one embedding, and autograd sums their d_emb before the single
    LayerNorm/region-mean backward and weight-gradient GEMM."""

    @staticmethod
    def forward(ctx, cfg, bags, precision, *params):
        need = any(p is not None and p.requires_grad for p in params[:4])
        acts = disc_embed_forward(cfg, params, bags, precision, save=need)
        ctx.cfg, ctx.bags, ctx.acts, ctx.params = cfg, bags, acts, params
        return acts["emb"]

    @staticmethod
    def backward(ctx, d_emb):
        params = [None if p is None else p.detach() for p in ctx.params]
        grads = [None if (t is None or i >= 4) else torch.empty_like(t, dtype=torch.float32) for i, t in enumerate(params)]
        disc_embed_backward(ctx.cfg, params, ctx.bags, ctx.acts, d_emb.contiguous(), grads, accumulate=False)
        return (None, None, None) + tuple(grads)


class DiscHeadFn(torch.autograd.Function):
    """out[bags] = RLIP head(emb, t): region MLP, GAPool, bag MLP, time embedding, inner product / projection; gradients
    for emb, t and the head tensors (the embedding's own four tensors get none here)."""

    @staticmethod
    def forward(ctx, cfg, bags, emb, t, train, seed, masks, precision, *params):
        head = disc_head_forward(cfg, params, bags, emb.detach(), t.detach(), train, seed, masks, precision)
        ctx.cfg, ctx.bags, ctx.head, ctx.params, ctx.t_shape = cfg, bags, head, params, t.shape
        ctx.need_param_grads = any(p is not None and p.requires_grad for p in params)
        return head["out"].clone()

    @staticmethod
    def backward(ctx, d_out):
        cfg, bags, params = ctx.cfg, ctx.bags, [None if p is None else p.detach() for p in ctx.params]
        dev = bags.x.device
        d_t = torch.empty(bags.bags, dtype=torch.float32, device=dev) if ctx.needs_input_grad[3] else None
        d_emb = torch.empty(bags.rows // 16, cfg.d, dtype=torch.float32, device=dev) if ctx.needs_input_grad[2] else None
        grads = None
        if ctx.need_param_grads:
            grads = [None if (t is None or i < 4) else torch.empty_like(t, dtype=torch.float32) for i, t in enumerate(params)]
        disc_head_backward(cfg, params, bags, ctx.head, d_out.contiguous(), d_emb, d_t, grads, accumulate=False)
        out_grads = tuple(grads) if grads is not None else (None,) * len(params)
        return (None, None, d_emb, None if d_t is None else d_t.reshape(ctx.t_shape), None, None, None, None) + out_grads


# -------------------------------------------------------------------------------------------------
# small stage-level wrappers (used by the DeepAttMISL path, the loader tools and the kernel tests)
# -------------------------------------------------------------------------------------------------
def _act_in(t: torch.Tensor, precision: int) -> torch.Tensor:
    """Activation operand in the element type of the precision mode (fp32 inputs are cast for the bf16 mode)."""
    want = act_dtype(precision)
    if t.dtype != want:
        t = cast_bf16(t) if want == torch.bfloat16 else t.float()
    return t if t.is_contiguous() else t.contiguous()


def linear_forward(x, W, b, act=0, p_drop=0.0, mask=None, seed=0, site=0, train=False, precision=FP32):
    lib = _lib.load()
    _need_cuda(x, "x")
    x, W = _act_in(x, precision), _f32c(W)
    rows, K = x.shape
    N = W.shape[0]
    y = torch.empty(rows, N, dtype=act_dtype(precision), device=x.device)
    check(lib.advmil_linear_fwd(x.data_ptr(), W.data_ptr(), _ptr(b), rows, K, N, act, p_drop, _ptr(mask), seed, site,
                                int(train), precision, y.data_ptr(), _stream()), "advmil_linear_fwd")
    return y


def linear_backward(dY, X, W, need_dx=True, need_dw=True, need_db=True, precision=FP32):
    lib = _lib.load()
    dY = _act_in(dY, precision)
    X = None if X is None else _act_in(X, precision)
    rows, N = dY.shape
    K = W.shape[1]
    dev = dY.device
    dX = torch.empty(rows, K, dtype=act_dtype(precision), device=dev) if need_dx else None
    dW = torch.empty(N, K, dtype=torch.float32, device=dev) if need_dw else None
    db = torch.empty(N, dtype=torch.float32, device=dev) if need_db else None
    ws = _ws(lib.advmil_linear_bwd_workspace_bytes(rows, K, N), dev)
    check(lib.advmil_linear_bwd(dY.data_ptr(), _ptr(X), _ptr(W), rows, K, N, _ptr(dX), _ptr(dW), _ptr(db), 0, precision,
                                ws.data_ptr(), ws.numel(), _stream()), "advmil_linear_bwd")
    return dX, dW, db


def gated_score_forward(v, Wa, ba, Wb, bb, wc, bc, p_drop=0.0, mask_a=None, mask_b=None, seed=0, train=False,
                        precision=FP32, save=True):
    lib = _lib.load()
    v = _act_in(v, precision)
    rows, L = v.shape
    D = Wa.shape[0]
    abw = lib.advmil_gate_packed_width(D)
    ab = torch.empty(rows, abw, dtype=act_dtype(precision), device=v.device) if save else None
    s = torch.empty(rows, dtype=torch.float32, device=v.device)
    ws = _ws((abw * L + abw + (abw // 128) * rows + 1024) * 4 + 4096, v.device)
    check(lib.advmil_gated_score_fwd(v.data_ptr(), Wa.data_ptr(), ba.data_ptr(), Wb.data_ptr(), bb.data_ptr(),
                                     wc.data_ptr(), bc.data_ptr(), rows, L, D, p_drop, _ptr(mask_a), _ptr(mask_b), seed,
                                     0, int(train), precision, _ptr(ab), s.data_ptr(), ws.data_ptr(), ws.numel(),
                                     _stream()), "advmil_gated_score_fwd")
    return s, ab


def seg_softmax_pool(s, v, bags_like: PackedBags, offsets=None, offsets_host=None, lengths=None, want_mean=False):
    """w = per-bag softmax(s), z[b] = sum_n w_n v_n (and the plain per-bag mean when want_mean).  v: fp32 or bf16."""
    lib = _lib.load()
    v = v.contiguous() if v.dtype == torch.bfloat16 else _f32c(v)
    rows, width = v.shape
    if offsets is None:
        offsets, offsets_host, nb = bags_like.offsets, bags_like.offsets_host, bags_like.bags
    else:
        nb = len(lengths)
    w = torch.empty(rows, dtype=torch.float32, device=v.device)
    z = torch.empty(nb, width, dtype=torch.float32, device=v.device)
    mean = torch.empty(nb, width, dtype=torch.float32, device=v.device) if want_mean else None
    ws = _ws(lib.advmil_seg_pool_workspace_bytes(rows, nb, width), v.device)
    check(lib.advmil_seg_softmax_pool_fwd(_f32c(s).data_ptr(), v.data_ptr(), ELEM_BF16 if v.dtype == torch.bfloat16 else ELEM_F32,
                                          offsets.data_ptr(), offsets_host, rows, nb, width, w.data_ptr(), z.data_ptr(),
                                          _ptr(mean), ws.data_ptr(), ws.numel(), _stream()), "advmil_seg_softmax_pool_fwd")
    return w, z, mean


def region_index_map(coords_l2: torch.Tensor, patch_size: int = 256, scale: int = 4) -> torch.Tensor:
    """tools/big_to_small_patching.py:59-76 on the device: [m,2] int64 -> [16m,2] float64."""
    lib = _lib.load()
    _need_cuda(coords_l2, "coords")
    c2 = coords_l2.to(torch.int64).contiguous()
    m = c2.shape[0]
    out = torch.empty(m * scale * scale, 2, dtype=torch.float64, device=c2.device)
    check(lib.advmil_region_index_map(c2.data_ptr(), m, patch_size, scale, out.data_ptr(), _stream()), "advmil_region_index_map")
    return out


def region_of_rows(rows: int, scale: int = 4, device="cuda") -> torch.Tensor:
    lib = _lib.load()
    out = torch.empty(rows, 3, dtype=torch.int32, device=device)
    check(lib.advmil_region_of_rows(rows, scale, out.data_ptr(), _stream()), "advmil_region_of_rows")
    return out


DROP_SITES = {"h": 1, "a": 2, "b": 3, "rho": 4, "mlp0": 5, "fc1": 11, "ga": 12, "gs": 13, "fc2": 14,
              "attn": 21, "sa": 22, "ff1": 23, "ff2": 24}     # attn: row = region * nhead + head, col = key region


def dropout_mask(seed: int, site: str, p: float, rows: int, width: int, device="cuda") -> torch.Tensor:
    """The uint8 keep mask the kernels generate on the fly for `site` under `seed` (test / debugging aid)."""
    lib = _lib.load()
    out = torch.empty(rows, width, dtype=torch.uint8, device=device)
    check(lib.advmil_dropout_mask(int(seed), DROP_SITES[site], float(p), rows, width, out.data_ptr(), _stream()),
          "advmil_dropout_mask")
    return out


def launch_count(reset: bool = False) -> int:
    return int(_lib.load().advmil_launch_count(int(reset)))

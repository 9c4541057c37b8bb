"""Fused adversarial step over packed bags: one D update + `gen_updates` G updates, the semantics of
MyHandler._update_disc + gen_updates x _update_gen (reference model/model_handler.py:328-335,349-498), without the
handler's redundant work:

  * the D-step generator forward (eval) and the G-step generator forward (train) share the x.W1^T projection
    (G's parameters do not change in between; dropout is applied to the cached eval activations);
  * real and fake pairs of the D step share one region-embedding pass (the embedding has no dropout);
  * no boolean-mask copies of x (model_handler.py:376,400,461), no per-bag .cpu()/.item() syncs, no empty_cache;
  * the G step asks D only for dL/dt (SURVEY.md A.2) and never accumulates D-parameter gradients;
  * parameters and gradients live in flat fp32 buffers: one NCCL all-reduce and one fused Adam launch per network.

Data parallel: every rank holds a shard of the step's bags; losses are normalised by GLOBAL pair counts so that the
sum of per-rank gradients is the single-process gradient; L1 / weight decay are applied once, inside the Adam kernel,
after the all-reduce.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence

import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import check
from .utils.func import next_dropout_seed


class FlatParams:
    """Re-homes a module's parameters as views of one flat fp32 buffer (and a matching flat gradient buffer)."""

    def __init__(self, module: nn.Module, tensors: Sequence[Optional[torch.Tensor]], weight_decay_rule: bool):
        named = {id(p): n for n, p in module.named_parameters()}
        self.order = [t for t in tensors if t is not None]
        dev = self.order[0].device
        total = sum((t.numel() + 3) // 4 * 4 for t in self.order)  # keep every tensor 16-byte aligned
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(total, dtype=torch.float32, device=dev)
        self.wd_mask = torch.zeros(total, dtype=torch.uint8, device=dev)
        self.views, self.grad_views = [], []
        off = 0
        for t in self.order:
            n = t.numel()
            v = self.flat[off:off + n].view_as(t)
            v.copy_(t.data)
            t.data = v
            self.views.append(v)
            self.grad_views.append(self.grad[off:off + n].view_as(t))
            name = named.get(id(t), "")
            # add_weight_decay rule (reference optim/optim_factory.py:25-37): 1-D tensors and *.bias get no decay
            if weight_decay_rule and not (t.dim() == 1 or name.endswith(".bias")):
                self.wd_mask[off:off + n] = 1
            off += (n + 3) // 4 * 4
        self.total = total
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.step_count = 0

    def broadcast(self, group=None, src: int = 0):
        """Data parallel: every replica starts from rank `src`'s parameters and optimiser state (a checkpoint loaded on one
        rank only, or a different seed per rank, would otherwise make the replicas diverge silently)."""
        for t in (self.flat, self.m, self.v):
            torch.distributed.broadcast(t, src, group=group)
        cnt = torch.tensor([self.step_count], dtype=torch.int64, device=self.flat.device)
        torch.distributed.broadcast(cnt, src, group=group)
        self.step_count = int(cnt.item())

    def grads_for(self, tensors: Sequence[Optional[torch.Tensor]]):
        idx = {id(t): i for i, t in enumerate(self.order)}
        return [None if t is None else self.grad_views[idx[id(t)]] for t in tensors]

    def adam(self, lr, weight_decay=0.0, l1_coef=0.0, betas=(0.9, 0.999), eps=1e-8):
        lib = _lib.load()
        self.step_count += 1
        check(lib.advmil_adam_step(self.flat.data_ptr(), self.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(),
                                   self.wd_mask.data_ptr() if weight_decay else None, self.total, lr, betas[0], betas[1],
                                   eps, weight_decay, l1_coef, self.step_count, 1.0,
                                   torch.cuda.current_stream().cuda_stream), "advmil_adam_step")


class _DataParallelMixin:
    """One process per GPU; the only exchange is the all-reduce of the flat gradient buckets.  Replicas are synchronised at
    construction (broadcast of parameters and Adam state from rank 0); every rank mixes its rank into the dropout seeds and
    draws its generator noise from its own CPU generator, so shards do not repeat each other's masks and noise (a single
    process keeps the default generator: the reference's stream, utils/func.py:154-164)."""

    def _init_gen_updates(self, gen_updates):
        """G updates per D update (config key `gen_updates`, model/model_handler.py:328-335)."""
        if isinstance(gen_updates, bool) or not isinstance(gen_updates, int) or gen_updates < 1:
            raise ValueError(f"gen_updates must be an integer >= 1, got {gen_updates!r}")
        self.gen_updates = gen_updates

    def _per_update(self, v, what):
        """One value per G update: `v` itself when gen_updates == 1, else a sequence of gen_updates values (None: [None] * k)."""
        k = self.gen_updates
        if v is None:
            return [None] * k
        if isinstance(v, (list, tuple)):
            if len(v) != k:
                raise ValueError(f"{what}: {len(v)} values for gen_updates={k}")
            return list(v)
        if k != 1:
            raise ValueError(f"{what}: gen_updates={k} needs a sequence of {k} values, one per G update")
        return [v]

    def _init_dp(self, process_group):
        self.pg = process_group
        self.world, self.rank = 1, 0
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
            self.rank = torch.distributed.get_rank(process_group)
        self._noise_gen = None
        if self.world > 1:
            self.G.broadcast(process_group)
            self.D.broadcast(process_group)
            self._noise_gen = torch.Generator().manual_seed((torch.initial_seed() + 7919 * (self.rank + 1)) % (2 ** 63))

    def _allreduce(self, t: torch.Tensor):
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM, group=self.pg)

    def _seed(self) -> int:
        return next_dropout_seed() ^ (self.rank * 0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF)

    def _draw(self, nb, dev):
        """Noise for the second head layer, drawn like Generator.forward does (model/GANSurv.py:33-38)."""
        return self.netG.draw_noise(nb, dev, False, generator=self._noise_gen)[1]

    def global_losses(self, losses: torch.Tensor) -> torch.Tensor:
        """The step's loss scalars are rank-local partial sums over GLOBAL pair counts: their sum over the ranks is the value
        the reference prints (one small all-reduce; call it only when the values are logged)."""
        if self.world > 1:
            losses = losses.clone()
            self._allreduce(losses)
        return losses


class AdvStep(_DataParallelMixin):
    def __init__(self, netG, netD, lr_g=8e-5, lr_d=8e-5, weight_decay_g=5e-4, coef_gan=0.004, coef_l1=1e-5,
                 loss_d="bce", recon_norm="l1", recon_alpha=0.0, recon_gamma=0.0, precision="fp32",
                 process_group=None, gen_updates=1):
        if netG.backbone.kind != "abmil":
            other = {"cluster": "ClusterAdvStep", "patch": "EsatAdvStep"}.get(netG.backbone.kind, "ModuleAdvStep")
            raise NotImplementedError(f"AdvStep is the C-fused step of the ABMIL generator; use {other} for bcb_mode "
                                      f"'{netG.backbone.kind}'")
        if list(netG.noise) != [0, 1]:
            raise NotImplementedError(f"AdvStep covers gen_noi_noise '0-1' (config/cfg_nlst.yaml:30), got {list(netG.noise)}: noise "
                                      "on the first head layer runs through the module path (Generator.forward / ModuleAdvStep)")
        self.netG, self.netD = netG, netD
        self.gcfg, self.dcfg = netG.config(), netD.config()
        self.gparams, self.dparams = netG.gen_params(), netD.disc_params()
        self.G = FlatParams(netG, self.gparams, weight_decay_rule=True)
        self.D = FlatParams(netD, self.dparams, weight_decay_rule=False)
        self.ggrads, self.dgrads = self.G.grads_for(self.gparams), self.D.grads_for(self.dparams)
        self._init_hparams(lr_g, lr_d, weight_decay_g, coef_gan, coef_l1, loss_d, recon_norm, recon_alpha, recon_gamma, precision,
                           process_group, gen_updates)

    def _init_hparams(self, lr_g, lr_d, weight_decay_g, coef_gan, coef_l1, loss_d, recon_norm, recon_alpha, recon_gamma, precision,
                      process_group, gen_updates):
        """Optimiser, loss, precision and schedule settings of the C-fused steps; runs after self.G / self.D exist."""
        self._init_gen_updates(gen_updates)
        self.lr_g, self.lr_d, self.wd_g = lr_g, lr_d, weight_decay_g
        self.coef_gan, self.coef_l1 = coef_gan, coef_l1
        self.loss_d = {"bce": 0, "hinge": 1, "wasserstein": 2}[loss_d]
        self.recon = ({"l1": 0, "l2": 1}[recon_norm], recon_alpha, recon_gamma)
        self.precision = ops.PRECISIONS[precision]
        self._inflight = None
        self._init_dp(process_group)

    # ---------------------------------------------------------------------------------------------
    def _structs(self):
        """C views of the parameter / gradient tensors (their storage is the flat buffers and never moves)."""
        if getattr(self, "_c", None) is None:
            gp, dp = self.gcfg.c(self.gparams), self.dcfg.c(self.dparams)
            gg, dg = _lib.GenGrads(), _lib.DiscGrads()
            for name, tns in zip(_lib.GEN_TENSORS, self.ggrads):
                setattr(gg, name, None if tns is None else tns.data_ptr())
            gg.dx = None
            for name, tns in zip(_lib.DISC_TENSORS, self.dgrads):
                setattr(dg, name, None if tns is None else tns.data_ptr())
            self._c = (gp, dp, gg, dg)
        return self._c

    def _inputs(self, bags, t, e, visible, global_counts):
        """The bags in this engine's precision, t / e / visible as flat device vectors, and the GLOBAL pair counts
        (n_real, n_fake, n_visible): an all-reduce and one host sync unless the caller passes them."""
        bags = bags.for_precision(self.precision)   # bf16 mode: bf16 features as packed by the loader, or one cast here
        dev, nb = bags.x.device, bags.bags
        t = t.reshape(-1).contiguous().float()
        e = e.reshape(-1).contiguous().float()
        visible = visible.reshape(-1).to(torch.uint8).contiguous()
        if global_counts is None:
            real_mask = ((e == 1) & (visible != 0))                      # model_handler.py:373-375
            cnt = torch.stack([real_mask.sum(), torch.tensor(nb, device=dev), visible.sum()]).float()
            self._allreduce(cnt)
            counts = [float(v) for v in cnt.tolist()]
        else:
            counts = [float(v) for v in global_counts]
        return bags, t, e, visible, counts

    def _noise(self, nb, dev, noise_d, noise_g):
        """Noise of the D phase's generator pass and of every G update's pass (a list), drawn in that order where not given."""
        noise_g = self._per_update(noise_g, "noise_g")
        noise_d = (noise_d if noise_d is not None else self._draw(nb, dev)).contiguous().float()
        noise_g = [(n if n is not None else self._draw(nb, dev)).contiguous().float() for n in noise_g]
        return noise_d, noise_g

    def _workspace(self, need, dev) -> torch.Tensor:
        """The step's workspace of at least `need` bytes: grow-only, so steady-state steps allocate nothing."""
        ws = getattr(self, "_ws", None)
        if ws is None or ws.numel() < need or ws.device != dev:
            self._ws = ws = torch.empty(int(need * 1.05) + 4096, dtype=torch.uint8, device=dev)
        return ws

    def _outputs(self, nb, dev):
        """The step's output tensors, and lbuf [gen_updates, 8]: row u holds the loss slots of G update u.  `losses` (the
        layout of the C ABI: D loss, then the G terms) is the last row, which the D phase writes too.  With gen_updates > 1,
        gen_losses [gen_updates, 4]: t_reg, gen, t_reg + coef_gan * gen and sum|W_G| of every G update (with one update
        those are losses[1:5], and the outputs are those of a one-update step as before)."""
        f32 = dict(dtype=torch.float32, device=dev)
        lbuf = torch.zeros(self.gen_updates, 8, **f32)
        out = {"losses": lbuf[-1], "pred_d": torch.empty(nb, **f32), "pred_g": torch.empty(nb, **f32),
               "f_d": torch.empty(2 * nb, **f32), "f_fake_g": torch.empty(nb, **f32),
               "real_mask": torch.empty(nb, dtype=torch.uint8, device=dev)}
        if self.gen_updates > 1:
            out["gen_losses"] = lbuf[:, 1:5]
        return out, lbuf

    def _fill_args(self, a, bags, t, e, visible, noise_d, noise_g, counts, out, ws):
        """The fields that StepArgs and EsatStepArgs share by name (the dropout seeds are drawn here: D's, then the first G
        update's; noise_g: the first G update's noise)."""
        a.bags = C.pointer(bags.c())
        a.t, a.e, a.visible = t.data_ptr(), e.data_ptr(), visible.data_ptr()
        a.noise_d, a.noise_g = noise_d.data_ptr(), noise_g.data_ptr()
        a.seed_d, a.seed_g = self._seed(), self._seed()
        a.n_real, a.n_fake, a.n_visible = counts
        a.loss_d = self.loss_d
        a.recon_norm, a.recon_alpha, a.recon_gamma = self.recon
        a.coef_gan, a.precision = self.coef_gan, self.precision
        a.losses, a.pred_d, a.f_fake_d, a.real_mask = (out["losses"].data_ptr(), out["pred_d"].data_ptr(),
                                                       out["f_d"].data_ptr(), out["real_mask"].data_ptr())
        a.pred_g, a.f_fake_g = out["pred_g"].data_ptr(), out["f_fake_g"].data_ptr()
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()

    def _update(self, lib, disc_fn: str, gen_fn: str, args, a, gen_fields, out, lbuf, nb, n_real, keep) -> Dict:
        """The library's D call, D all-reduce and Adam, then per G update its G call (`gen_fn`, then `gen_fn`_next), L1 value,
        G all-reduce and Adam.  a: the AdvmilStepArgs-like fields of `args`; gen_fields: per G update, the fields of `a` that
        update sets (its noise and injected masks).  keep: the step's input tensors, alive until the stream is done with them."""
        st = torch.cuda.current_stream().cuda_stream
        # ---------------- D step: D.train / G.eval (model_handler.py:355-356) ----------------
        check(getattr(lib, disc_fn)(C.byref(args), st), disc_fn)
        self._allreduce(self.D.grad)
        self.D.adam(self.lr_d)
        # ---------------- G steps: D.eval / G.train (model_handler.py:432-433), gen_updates times ----------------
        for u, fields in enumerate(gen_fields):
            fn = gen_fn if u == 0 else gen_fn + "_next"
            if u > 0:
                for name, v in fields.items():
                    setattr(a, name, v)
                a.seed_g = self._seed()
            a.losses = lbuf[u].data_ptr()
            check(getattr(lib, fn)(C.byref(args), st), fn)
            if self.coef_l1 > 1e-8:
                check(lib.advmil_abs_sum(self.G.flat.data_ptr(), self.G.total, lbuf[u][4:].data_ptr(), st), "advmil_abs_sum")
            self._allreduce(self.G.grad)
            self.G.adam(self.lr_g, weight_decay=self.wd_g, l1_coef=self.coef_l1 if self.coef_l1 > 1e-8 else 0.0)
        out["f_fake_d"] = out["f_d"][:nb]
        out["f_real"] = out["f_d"][nb:] if n_real > 0 else None
        out["_keep"] = keep
        # pred_g / noise_g / the masks are also touched by the library's side stream (the forked train forward): the engine
        # keeps the step's tensors until the NEXT step has been issued, by which time the main stream has joined the side
        # stream -- a caller that drops `out` early cannot hand their memory back to the allocator under the side stream
        self._inflight = out
        return out

    @staticmethod
    def _gen_fields(noise_g, masks_g, keys):
        """Per G update: the AdvmilStepArgs fields of its noise and of its injected masks (over `keys`)."""
        return [dict({"noise_g": n.data_ptr()}, **{"g_mask_" + k: ops._ptr((m or {}).get(k)) for k in keys})
                for n, m in zip(noise_g, masks_g)]

    @staticmethod
    def _cat_masks(fake, real, keys):
        """Injected discriminator masks of the batched head pass: FAKE pairs first, then REAL pairs."""
        if not fake and not real:
            return {}
        assert fake and real, "inject masks for both the real and the fake pairs (or for neither)"
        return {k: torch.cat([fake[k], real[k]], dim=0).contiguous() for k in keys}

    def step(self, bags: ops.PackedBags, t: torch.Tensor, e: torch.Tensor, visible: torch.Tensor,
             noise_d: Optional[torch.Tensor] = None, noise_g: Optional[torch.Tensor] = None,
             masks_d_real=None, masks_d_fake=None, masks_g=None, global_counts=None) -> Dict:
        """t, e: [bags] float32 device; visible: [bags] uint8 device (label_visible_mask).  noise_*: [bags, hid] device
        (drawn like utils/func.generate_noise when None: noise_d, then one draw per G update).  noise_g and masks_g: one
        value, or a sequence of gen_updates values (one per G update).  Returns device tensors only (no host sync when
        global_counts is given); losses / pred_g / f_fake_g are those of the last G update; with gen_updates > 1,
        gen_losses [gen_updates, 4] holds every update's.  One C call per phase (advmil_adv_step_disc / _gen / _gen_next) issues the launch sequence."""
        lib = _lib.load()
        bags, t, e, visible, counts = self._inputs(bags, t, e, visible, global_counts)
        dev, nb = bags.x.device, bags.bags
        mgs = [m or {} for m in self._per_update(masks_g, "masks_g")]
        noise_d, noise_g = self._noise(nb, dev, noise_d, noise_g)
        gp, dp, gg, dg = self._structs()
        ws = self._workspace(lib.advmil_adv_step_workspace_bytes(C.byref(gp), C.byref(dp), bags.rows, nb, self.precision), dev)
        out, lbuf = self._outputs(nb, dev)
        md = self._cat_masks(masks_d_fake, masks_d_real, ("fc1", "ga", "gs", "fc2"))
        a = _lib.StepArgs()
        a.gen, a.disc, a.gen_grads, a.disc_grads = C.pointer(gp), C.pointer(dp), C.pointer(gg), C.pointer(dg)
        fields = self._gen_fields(noise_g, mgs, ("h", "a", "b", "rho", "mlp0"))
        for name, v in fields[0].items():
            setattr(a, name, v)
        for k in ("fc1", "ga", "gs", "fc2"):
            setattr(a, "d_mask_" + k, ops._ptr(md.get(k)))
        self._fill_args(a, bags, t, e, visible, noise_d, noise_g[0], counts, out, ws)
        return self._update(lib, "advmil_adv_step_disc", "advmil_adv_step_gen", a, a, fields, out, lbuf, nb, counts[0],
                            (t, e, visible, noise_d, noise_g, md, mgs, bags))

    def loss_dict(self, out) -> Dict[str, float]:
        """Host copy of the step's scalars (one sync): the values the handler prints (model_handler.py:413,486-494); under
        data parallelism the sum over the ranks (the per-rank values are partial sums over global counts)."""
        v = self.global_losses(out["losses"]).tolist()
        l1 = self.coef_l1 * v[4] if self.coef_l1 > 1e-8 else 0.0
        return {"dis_loss": v[0], "t_reg_loss": v[1], "gen_loss": v[2], "gen_total_loss": v[3] + l1}


class EsatAdvStep(AdvStep):
    """The C-fused adversarial step for the ESAT generator (`bcb_mode: patch`, DualTrans_HS + noise head) with the RLIP
    discriminator: `advmil_adv_step_esat_disc / _gen` issue the launch sequence of `ModuleAdvStep` from two host calls (no
    Python between the kernels, one grow-only workspace, the D phase's eval pass hands its patch embedding to the G phase's
    train pass).  Same step semantics, outputs and `loss_dict` as `AdvStep` (model/model_handler.py:349-498).  In-kernel dropout
    only: injected masks (parity tests) go through `ModuleAdvStep`.  coord: region coordinates for the sincos positional
    embedding, or None (what the handler passes, model_handler.py:613)."""

    def __init__(self, netG, netD, lr_g=8e-5, lr_d=8e-5, weight_decay_g=5e-4, coef_gan=0.004, coef_l1=1e-5,
                 loss_d="bce", recon_norm="l1", recon_alpha=0.0, recon_gamma=0.0, precision="fp32", process_group=None,
                 gen_updates=1):
        if netG.backbone.kind != "patch":
            raise NotImplementedError(f"EsatAdvStep is the C-fused step of the ESAT generator, got bcb_mode '{netG.backbone.kind}'")
        if list(netG.noise) != [0, 1]:
            raise NotImplementedError(f"EsatAdvStep covers gen_noi_noise '0-1', got {list(netG.noise)}")
        self.netG, self.netD = netG, netD
        bb = netG.backbone
        self.ecfg, self.hcfg, self.dcfg = bb.esat_config(), netG.config(), netD.config()
        self.eparams, self.hparams, self.dparams = bb.esat_params(), netG.head_params(), netD.disc_params()
        self.G = FlatParams(netG, list(netG.parameters()), weight_decay_rule=True)
        self.D = FlatParams(netD, self.dparams, weight_decay_rule=False)
        self.egrads, self.hgrads, self.dgrads = self.G.grads_for(self.eparams), self.G.grads_for(self.hparams), self.D.grads_for(self.dparams)
        assert self.G.total == sum((t.numel() + 3) // 4 * 4 for t in self.eparams + self.hparams), "generator parameters outside the ESAT step"
        self._init_hparams(lr_g, lr_d, weight_decay_g, coef_gan, coef_l1, loss_d, recon_norm, recon_alpha, recon_gamma, precision,
                           process_group, gen_updates)

    def _structs(self):
        if getattr(self, "_c", None) is None:
            ep, hp, dp = self.ecfg.c(self.eparams), self.hcfg.c([None] * 10 + list(self.hparams)), self.dcfg.c(self.dparams)
            eg, hg, dg = _lib.EsatGrads(), _lib.GenGrads(), _lib.DiscGrads()
            for name, tns in zip(_lib.ESAT_TENSORS, self.egrads):
                setattr(eg, name, tns.data_ptr())
            for name, tns in zip(_lib.GEN_TENSORS, [None] * 10 + list(self.hgrads)):
                setattr(hg, name, None if tns is None else tns.data_ptr())
            hg.dx = None
            for name, tns in zip(_lib.DISC_TENSORS, self.dgrads):
                setattr(dg, name, None if tns is None else tns.data_ptr())
            self._c = (ep, hp, dp, eg, hg, dg)
        return self._c

    def step(self, bags: ops.PackedBags, t: torch.Tensor, e: torch.Tensor, visible: torch.Tensor,
             noise_d: Optional[torch.Tensor] = None, noise_g: Optional[torch.Tensor] = None, coord=None, global_counts=None) -> Dict:
        lib = _lib.load()
        bags, t, e, visible, counts = self._inputs(bags, t, e, visible, global_counts)
        dev, nb = bags.x.device, bags.bags
        noise_d, noise_g = self._noise(nb, dev, noise_d, noise_g)
        pe = self.netG.backbone.positional(bags, coord)
        ep, hp, dp, eg, hg, dg = self._structs()
        ws = self._workspace(lib.advmil_adv_step_esat_workspace_bytes(C.byref(ep), C.byref(hp), C.byref(dp), bags.rows, nb,
                                                                      self.precision), dev)
        out, lbuf = self._outputs(nb, dev)
        a = _lib.EsatStepArgs()
        a.esat, a.head, a.disc = C.pointer(ep), C.pointer(hp), C.pointer(dp)
        a.esat_grads, a.head_grads, a.disc_grads = C.pointer(eg), C.pointer(hg), C.pointer(dg)
        a.pe = ops._ptr(pe)
        self._fill_args(a, bags, t, e, visible, noise_d, noise_g[0], counts, out, ws)
        return self._update(lib, "advmil_adv_step_esat_disc", "advmil_adv_step_esat_gen", a, a,
                            self._gen_fields(noise_g, [None] * len(noise_g), ()), out, lbuf, nb, counts[0],
                            (t, e, visible, noise_d, noise_g, pe, bags))


class ClusterAdvStep(AdvStep):
    """The C-fused adversarial step for the DeepAttMISL generator (`bcb_mode: cluster`) with the RLIP discriminator:
    `advmil_adv_step_cluster_disc / _gen` issue the launch sequence of `ModuleAdvStep` from two host calls.  The projection
    of phis runs once per step: one tcgen05 pass computes relu(x Wphi^T + b), its per-(bag, cluster) means and the ReLU keep
    bits without writing the activation (the fp32 mode composes the FFMA projection and the segment mean), and the D
    phase's eval pass and the G phase's train pass of the attention stage both start from those means.  Same step
    semantics, outputs and `loss_dict` as `AdvStep` (model/model_handler.py:349-498).  `step(..., ext=cluster ids)`;
    injected generator masks are over the attention stage's [bags * num_clusters, h] rows, as in `ModuleAdvStep`."""

    def __init__(self, netG, netD, lr_g=8e-5, lr_d=8e-5, weight_decay_g=5e-4, coef_gan=0.004, coef_l1=1e-5,
                 loss_d="bce", recon_norm="l1", recon_alpha=0.0, recon_gamma=0.0, precision="fp32", process_group=None,
                 gen_updates=1):
        bb = netG.backbone
        if bb.kind != "cluster":
            raise NotImplementedError(f"ClusterAdvStep is the C-fused step of the DeepAttMISL generator, got bcb_mode '{bb.kind}': "
                                      "use AdvStep (abmil), EsatAdvStep (patch) or ModuleAdvStep")
        if list(netG.noise) != [0, 1]:
            raise NotImplementedError(f"ClusterAdvStep covers gen_noi_noise '0-1', got {list(netG.noise)}: use ModuleAdvStep")
        if not 1 <= bb.num_clusters <= 16:
            raise NotImplementedError(f"ClusterAdvStep covers 1..16 clusters, got {bb.num_clusters}: use ModuleAdvStep")
        if netD.config().ksize not in (0, 1):
            raise NotImplementedError("ClusterAdvStep covers the ksize-1 discriminator: use ModuleAdvStep")
        self.netG, self.netD = netG, netD
        self.gcfg, self.dcfg = netG.config(), netD.config()
        self.gparams, self.dparams = netG.gen_params(), netD.disc_params()
        self.G = FlatParams(netG, list(netG.parameters()), weight_decay_rule=True)
        self.Wphi, self.bphi = bb.phi_params()            # after FlatParams: views of the flat buffer
        self.D = FlatParams(netD, self.dparams, weight_decay_rule=False)
        self.ggrads, self.dgrads = self.G.grads_for(self.gparams), self.D.grads_for(self.dparams)
        self.dWphi, self.dbphi = self.G.grads_for([self.Wphi, self.bphi])
        covered = [t for t in self.gparams if t is not None] + [self.Wphi, self.bphi]
        assert self.G.total == sum((t.numel() + 3) // 4 * 4 for t in covered), "generator parameters outside the cluster step"
        self._init_hparams(lr_g, lr_d, weight_decay_g, coef_gan, coef_l1, loss_d, recon_norm, recon_alpha, recon_gamma, precision,
                           process_group, gen_updates)

    def step(self, bags: ops.PackedBags, t: torch.Tensor, e: torch.Tensor, visible: torch.Tensor,
             noise_d: Optional[torch.Tensor] = None, noise_g: Optional[torch.Tensor] = None, ext=None,
             masks_d_real=None, masks_d_fake=None, masks_g=None, global_counts=None) -> Dict:
        """ext: the cluster id of every row, [rows] or [1, rows], float (what the handler passes) or int32 (used as is)."""
        if ext is None:
            raise ValueError("ClusterAdvStep.step needs the cluster id of every row (ext)")
        lib = _lib.load()
        bags, t, e, visible, counts = self._inputs(bags, t, e, visible, global_counts)
        dev, nb = bags.x.device, bags.bags
        cid = ext.reshape(-1)
        cid = (cid if cid.dtype == torch.int32 else cid.to(torch.int32)).contiguous()
        assert cid.numel() == bags.rows and cid.device == dev, "one cluster id per row, on the bags' device"
        mgs = [{k: v.contiguous() for k, v in (m or {}).items()} for m in self._per_update(masks_g, "masks_g")]
        noise_d, noise_g = self._noise(nb, dev, noise_d, noise_g)
        gp, dp, gg, dg = self._structs()
        ncl = self.netG.backbone.num_clusters
        ws = self._workspace(lib.advmil_adv_step_cluster_workspace_bytes(C.byref(gp), C.byref(dp), bags.rows, nb, ncl,
                                                                         self.precision), dev)
        out, lbuf = self._outputs(nb, dev)
        md = self._cat_masks(masks_d_fake, masks_d_real, ("fc1", "ga", "gs", "fc2"))
        ca = _lib.ClusterStepArgs()
        a = ca.base
        a.gen, a.disc, a.gen_grads, a.disc_grads = C.pointer(gp), C.pointer(dp), C.pointer(gg), C.pointer(dg)
        fields = self._gen_fields(noise_g, mgs, ("h", "a", "b", "mlp0"))
        for name, v in fields[0].items():
            setattr(a, name, v)
        for k in ("fc1", "ga", "gs", "fc2"):
            setattr(a, "d_mask_" + k, ops._ptr(md.get(k)))
        self._fill_args(a, bags, t, e, visible, noise_d, noise_g[0], counts, out, ws)
        ca.Wphi, ca.bphi, ca.dWphi, ca.dbphi = self.Wphi.data_ptr(), self.bphi.data_ptr(), self.dWphi.data_ptr(), self.dbphi.data_ptr()
        ca.cid, ca.num_clusters = cid.data_ptr(), ncl
        return self._update(lib, "advmil_adv_step_cluster_disc", "advmil_adv_step_cluster_gen", ca, a, fields, out, lbuf, nb, counts[0],
                            (t, e, visible, noise_d, noise_g, md, mgs, cid, bags))


class ModuleAdvStep(_DataParallelMixin):
    """One D update + `gen_updates` G updates over packed bags for any built generator backbone (ABMIL, DeepAttMISL, ESAT), composed from
    the modules' packed forwards and their autograd Functions: the same step semantics as `AdvStep`
    (model/model_handler.py:349-498; global-count loss normalisation, flat parameter buffers, one all-reduce and one fused
    Adam launch per network, L1 and weight decay inside the Adam kernel) without the ABMIL-specific cross-phase sharing
    of `advmil_adv_step_disc/gen`.  Used for `bcb_mode: patch`; `AdvStep` remains the path for the ABMIL benchmark."""

    def __init__(self, netG, netD, lr_g=8e-5, lr_d=8e-5, weight_decay_g=5e-4, coef_gan=0.004, coef_l1=1e-5, loss_d="bce",
                 recon_norm="l1", recon_alpha=0.0, recon_gamma=0.0, precision="fp32", process_group=None, gen_updates=1):
        assert recon_norm in ("l1", "l2"), recon_norm          # loss/utils.py:21-41
        self._init_gen_updates(gen_updates)
        self.recon_norm = recon_norm
        self.netG, self.netD = netG, netD
        self.gparams = [p for p in netG.parameters()]
        self.dparams = [p for p in netD.parameters()]
        self.G = FlatParams(netG, self.gparams, weight_decay_rule=True)
        self.D = FlatParams(netD, self.dparams, weight_decay_rule=False)
        for p, g in zip(self.gparams, self.G.grad_views):
            p.grad = g                      # autograd accumulates in place into the flat gradient buffers (do not call
                                            # zero_grad(set_to_none=True) on these modules: step() zeroes the buffers itself)
        for p, g in zip(self.dparams, self.D.grad_views):
            p.grad = g
        self.lr_g, self.lr_d, self.wd_g = lr_g, lr_d, weight_decay_g
        self.coef_gan, self.coef_l1, self.loss_d = coef_gan, coef_l1, loss_d
        self.recon_alpha, self.recon_gamma = recon_alpha, recon_gamma
        self.precision, self.precision_name = ops.PRECISIONS[precision], precision
        self._gmods, self._dmods = list(netG.modules()), list(netD.modules())
        self._init_dp(process_group)

    @staticmethod
    def _set_training(mods, flag: bool):
        """nn.Module.train(flag) without the recursion and the __setattr__ hooks: ~150 sub-modules are toggled four times per
        step, which cost 1.5 ms of host time per step through the module API."""
        for m in mods:
            m.__dict__["training"] = flag

    def step(self, *args, **kwargs) -> Dict:
        """See `_step`; runs it under this engine's precision mode (the modules read the package-wide setting)."""
        from . import get_precision, set_precision
        saved = get_precision()
        set_precision(self.precision_name)
        try:
            return self._step(*args, **kwargs)
        finally:
            set_precision(saved)

    def _disc_loss(self, f_real, f_fake, real_mask, n_real, n_fake):
        """real_fake_loss (loss/utils.py:182-203) over packed bags: every bag has a fake pair, bags under `real_mask` a real
        pair; means are over the GLOBAL pair counts."""
        m = real_mask.float()
        if self.loss_d == "bce":
            loss = -(1.0 - torch.log(torch.sigmoid(f_fake) + 1e-8)).sum() / n_fake
            if n_real > 0:
                loss = loss - (m * torch.log(torch.sigmoid(f_real) + 1e-8)).sum() / n_real
        elif self.loss_d == "hinge":
            loss = torch.relu(1.0 + f_fake).sum() / n_fake
            if n_real > 0:
                loss = loss + (m * torch.relu(1.0 - f_real)).sum() / n_real
        elif self.loss_d == "wasserstein":
            loss = f_fake.sum() / n_fake
            if n_real > 0:
                loss = loss - (m * f_real).sum() / n_real
        else:
            raise ValueError(self.loss_d)
        return loss

    def _generate(self, bags: ops.PackedBags, noise, ext, coord, reuse=None, sink=None):
        """G over packed bags: ext = cluster ids [rows] (DeepAttMISL), coord = region coordinates [R,2] or None (ESAT).
        reuse (ESAT): activations of the D step's eval pass -- G's parameters do not change between the two passes and the
        patch embedding has no dropout, so the G step's train pass shares its x.Wc^T projection and LayerNorm stream."""
        G = self.netG
        kind = G.backbone.kind
        if kind == "cluster":
            bb = G.backbone
            hc = bb.cluster_rows(bags.x, ext, bags.lengths, offsets=bags.offsets)          # [bags * clusters, h], differentiable
            # the attention stage sees num_clusters rows per bag: always the exact fp32 engine (like Generator.forward)
            return G.forward_packed(bb.cluster_bags(hc, bags.bags), noise=noise, x_grad=hc, precision=ops.FP32)
        kw = {"coord": coord, "reuse_embedding": reuse, "acts_sink": sink} if kind == "patch" else {}
        return G.forward_packed(bags, noise=noise, precision=self.precision, **kw)

    def _step(self, bags: ops.PackedBags, t, e, visible, noise_d=None, noise_g=None, coord=None, global_counts=None,
              masks_d_real=None, masks_d_fake=None, masks_g=None, ext=None) -> Dict:
        G, D = self.netG, self.netD
        bags = bags.for_precision(self.precision)
        dev, nb = bags.x.device, bags.bags
        t, e = t.reshape(-1).float(), e.reshape(-1).float()
        vis = visible.reshape(-1) != 0
        real_mask = (e == 1) & vis
        if global_counts is None:
            cnt = torch.stack([real_mask.sum(), torch.tensor(nb, device=dev), vis.sum()]).float()
            self._allreduce(cnt)
            n_real, n_fake, n_vis = [float(v) for v in cnt.tolist()]
        else:
            n_real, n_fake, n_vis = [float(v) for v in global_counts]
        noise_g, masks_g = self._per_update(noise_g, "noise_g"), self._per_update(masks_g, "masks_g")
        nz_d = [None, noise_d if noise_d is not None else self._draw(nb, dev)]
        nz_g = [[None, n if n is not None else self._draw(nb, dev)] for n in noise_g]
        # ---------------- D step: D.train / G.eval (model_handler.py:355-356) ----------------
        self._set_training(self._dmods, True)
        self._set_training(self._gmods, False)
        self.D.grad.zero_()
        with torch.no_grad():
            sink = [] if G.backbone.kind == "patch" else None      # this step's own hand-off of the patch embedding
            pred_d = self._generate(bags, nz_d, ext, coord, sink=sink)
        shared = sink[0] if sink else None
        emb = D.embed_packed(bags)          # shared by the fake and the real pairs (no dropout in the embedding)
        D._inject_masks = masks_d_fake
        f_fake = D.head_packed(bags, emb, pred_d.detach()).reshape(-1)
        f_real = None
        if n_real > 0:
            D._inject_masks = masks_d_real
            f_real = D.head_packed(bags, emb, t.reshape(-1, 1)).reshape(-1)
        dis_loss = self._disc_loss(f_real, f_fake, real_mask, n_real, n_fake)
        dis_loss.backward()
        self._allreduce(self.D.grad)
        self.D.adam(self.lr_d)
        # ---------------- G steps: D.eval / G.train (model_handler.py:432-433), gen_updates times ----------------
        self._set_training(self._dmods, False)
        self._set_training(self._gmods, True)
        for p in self.dparams:
            p.requires_grad_(False)         # D only hands dL/dt back to G
        gen_losses = []
        try:
            for u in range(self.gen_updates):
                self.G.grad.zero_()
                G._inject_masks = masks_g[u]
                pred_g = self._generate(bags, nz_g[u], ext, coord, reuse=shared if u == 0 else None)
                shared = sink = None        # the patch embedding of the D step's pass serves the first update only
                f_g = D.forward_packed(bags, pred_g).reshape(-1)
                gen_loss = -f_g.sum() / n_fake                                    # fake_generator_loss (loss/utils.py:205-208)
                pg = pred_g.reshape(-1)
                lo = e * torch.abs(pg - t)                                        # recon_loss (loss/utils.py:21-41)
                lc = (1.0 - e) * torch.relu(self.recon_gamma - (pg - t))
                if self.recon_norm == "l2":
                    lo, lc = lo * lo, lc * lc
                t_reg = (vis.float() * ((1.0 - self.recon_alpha) * (lo + lc) + self.recon_alpha * lo)).sum() / max(n_vis, 1.0)
                total = t_reg + self.coef_gan * gen_loss
                total.backward()
                self._allreduce(self.G.grad)
                l1 = self.G.flat.abs().sum() if self.coef_l1 > 1e-8 else None    # value only; its gradient is in the Adam kernel
                self.G.adam(self.lr_g, weight_decay=self.wd_g, l1_coef=self.coef_l1 if self.coef_l1 > 1e-8 else 0.0)
                gen_losses.append((t_reg.detach(), gen_loss.detach(), total.detach(), l1))
        finally:
            for p in self.dparams:
                p.requires_grad_(True)
        t_reg, gen_loss, total, l1 = gen_losses[-1]
        out = {"dis_loss": dis_loss.detach(), "gen_loss": gen_loss, "t_reg_loss": t_reg,
               "gen_total_loss": total + (self.coef_l1 * l1 if l1 is not None else 0.0),
               "pred_d": pred_d.reshape(-1), "pred_g": pred_g.detach().reshape(-1), "f_fake_d": f_fake.detach(),
               "f_real": None if f_real is None else f_real.detach(), "f_fake_g": f_g.detach()}
        if self.gen_updates > 1:      # as in AdvStep: [gen_updates, 4] t_reg, gen, t_reg + coef_gan * gen, sum|W_G|
            out["gen_losses"] = torch.stack([torch.stack([a, b, c, torch.zeros_like(c) if d is None else d])
                                             for a, b, c, d in gen_losses])
        return out


@torch.no_grad()
def sample_inference(netG, netD, bags: ops.PackedBags, times_test_sample: int = 30, zero_noise: bool = False,
                     precision: str = "fp32", coord=None, ext=None):
    """MyHandler.test_model for a batch of bags (reference model/model_handler.py:598-643) from ONE backbone pass, for any
    built generator backbone: y_hat [bags,1] with its own noise draw, f_fake = D(x, y_hat) [bags,1], dist_y_hat [bags,S,1]
    from S more draws, avg_y_hat = lower median over the S draws (torch.median semantics).  coord: region coordinates of the
    ESAT generator (None = no positional embedding, what the handler passes, :613); ext: cluster ids per row (DeepAttMISL).
    Runs under `precision` (the modules read the package-wide mode, which is restored afterwards)."""
    from . import get_precision, set_precision
    saved = get_precision()
    set_precision(precision)
    try:
        return _sample_inference(netG, netD, bags, times_test_sample, zero_noise, precision, coord, ext)
    finally:
        set_precision(saved)


def _sample_inference(netG, netD, bags, times_test_sample, zero_noise, precision, coord, ext):
    cfg, params = netG.config(), netG.gen_params()
    prec = ops.PRECISIONS[precision]
    bags = bags.for_precision(prec)
    nb, dev = bags.bags, bags.x.device
    kind = netG.backbone.kind
    was_training = netG.training
    netG.eval()
    try:
        n0, n1 = netG.draw_noise(nb, dev, zero_noise)
        if kind == "abmil":
            acts = ops.generator_forward(cfg, params, bags, n0, n1, train=False, precision=prec, save=False)
            y_hat, H = acts["pred"].reshape(nb, 1), acts["H"]
        elif kind == "patch":          # ESAT: the bag embedding H is handed out by the forward's activation sink
            sink = []
            y_hat = netG.forward_packed(bags, noise=[n0, n1], precision=prec, coord=coord, acts_sink=sink).reshape(nb, 1)
            H = sink[0]["H"]
        elif kind == "cluster":        # DeepAttMISL: per-(bag, cluster) means, then the 8-row attention stage in fp32
            assert ext is not None, "the cluster generator needs the cluster id of every row (ext)"
            bb = netG.backbone
            hc = bb.cluster_rows(bags.x, ext, bags.lengths, offsets=bags.offsets)
            acts = ops.generator_forward(cfg, params, ops.PackedBags(hc, [bb.num_clusters] * nb), n0, n1, train=False,
                                         precision=ops.FP32, save=False)
            y_hat, H = acts["pred"].reshape(nb, 1), acts["H"]
        else:
            raise NotImplementedError(f"sample_inference: generator backbone '{kind}'")
    finally:
        netG.train(was_training)
    f_fake = netD.forward_packed(bags, y_hat)
    res = {"y_hat": y_hat, "f_fake": f_fake}
    if times_test_sample > 1:
        S = times_test_sample
        draws0, draws1 = [], []
        for _ in range(S):      # same CPU-RNG call order as the reference's loop (:626-635)
            a, b = netG.draw_noise(nb, dev, zero_noise)
            draws0.append(a)
            draws1.append(b)
        N0 = None if draws0[0] is None else torch.stack(draws0)
        N1 = None if draws1[0] is None else torch.stack(draws1)
        ys = ops.generator_sample(cfg, params, H, N1, S, noise0=N0)      # [S, bags]
        res["dist_y_hat"] = ys.transpose(0, 1).unsqueeze(-1).contiguous()        # [bags, S, 1]
        res["avg_y_hat"] = torch.median(ys, dim=0)[0].reshape(nb, 1)
    return res

"""TEST / BASELINE INFRASTRUCTURE -- drives the reference's UNMODIFIED `MyHandler` (model/model_handler.py).

Only bench.py's baseline legs use this file; the product path never imports it.

What it offers
  * `load_cfg(**over)`        the reference's own config/cfg_nlst.yaml with overrides (bcb_mode, paths, ...);
  * `write_synthetic_dataset` per-slide `.pt` feature files + label table + split `.npz` in the layout README.md:72-89 /
                              dataset/PatchWSI.py:65-94 / utils/io.py:10-76,140-150 expect;
  * `make_handler(cfg, impl, device)`
        impl "reference"    -> `model.model_handler.MyHandler` exactly as the reference imports it;
        impl "advmil_b200"  -> the SAME file executed a second time as `model.model_handler_b200` while
                               `sys.modules["model.GANSurv" | "model.backbone" | "model.model_utils"]` point at the
                               advmil_b200 modules: the four relative imports of model_handler.py:13-16 resolve to the
                               B200 implementation, every other line of the handler is the reference's (this is the
                               "four-import swap" of INTEGRATION.md §1, done without editing the file);
        device "cpu"        -> `.cuda()` calls of the handler become identities (CPU baseline); "cuda" leaves them alone;
  * `InMemoryBags`            a Dataset with WSIPatch's item format fed from tensors (for timing without disk IO);
  * `handler_step(handler, xs, ys, ...)`  = `_update_disc` + `_update_gen` (model_handler.py:328-335).

Environment shims (the handler file itself is never edited): `WANDB_MODE=disabled`; torch 2.11 removed the `verbose`
keyword of `ReduceLROnPlateau` that model_handler.py:109 passes, so the scheduler class is wrapped to drop it.
"""
from __future__ import annotations

import contextlib
import importlib
import importlib.util
import io
import os
import sys
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import ref_import

SWAPPED = ("model.GANSurv", "model.backbone", "model.model_utils")


def _shim_environment():
    os.environ.setdefault("WANDB_MODE", "disabled")
    os.environ.setdefault("WANDB_SILENT", "true")
    from torch.optim import lr_scheduler
    cls = lr_scheduler.ReduceLROnPlateau
    if not getattr(cls, "_advmil_verbose_shim", False):
        import inspect
        if "verbose" not in inspect.signature(cls.__init__).parameters:
            class ReduceLROnPlateau(cls):                      # accepts and ignores the removed keyword
                _advmil_verbose_shim = True

                def __init__(self, *a, verbose=None, **k):
                    super().__init__(*a, **k)
            lr_scheduler.ReduceLROnPlateau = ReduceLROnPlateau


def handler_module(impl: str = "reference"):
    """The reference's model_handler module; impl 'advmil_b200' = a second execution of the same file with the four model
    imports resolved to the advmil_b200 modules."""
    _shim_environment()
    ref_import.import_reference()
    base = importlib.import_module("model.model_handler")
    if impl == "reference":
        return base
    assert impl == "advmil_b200", impl
    name = "model.model_handler_b200"
    if name in sys.modules:
        return sys.modules[name]
    import advmil_b200.model.backbone as bb
    import advmil_b200.model.GANSurv as gs
    import advmil_b200.model.model_utils as mu
    saved = {k: sys.modules.get(k) for k in SWAPPED}
    sys.modules.update({"model.GANSurv": gs, "model.backbone": bb, "model.model_utils": mu})
    try:
        spec = importlib.util.spec_from_file_location(name, base.__file__)
        mod = importlib.util.module_from_spec(spec)
        mod.__package__ = "model"
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    assert mod.Generator is gs.Generator and mod.load_backbone is bb.load_backbone and mod.init_weights is mu.init_weights
    return mod


def load_cfg(**over) -> Dict:
    import yaml
    path = os.path.join(ref_import.REF_ROOT, "config", "cfg_nlst.yaml")
    cfg = yaml.safe_load(open(path))
    cfg.update(cuda_id=0, data_split_seed=0, num_workers=0, save_prediction=False, wandb_dir="/tmp", bcb_mode="abmil")
    cfg.update(over)
    return cfg


def write_synthetic_dataset(root: str, n_patients: int, rows, seed: int = 42, C: int = 1024, n_val: int = 0,
                            event_rate: float = 0.347, nonneg: bool = False) -> Dict[str, str]:
    """One slide per patient: `<root>/pt_files/<sid>.pt` = fp32 [rows_i, C]; `<root>/labels.csv` with the columns
    utils/io.py:27 asserts; `<root>/split-fold0.npz` with train/val(/test) patient ids (utils/io.py:140-150).
    `rows`: int or a per-patient list (multiples of 16 for the RLIP discriminator)."""
    import pandas as pd
    os.makedirs(os.path.join(root, "pt_files"), exist_ok=True)
    rows = [int(rows)] * n_patients if np.isscalar(rows) else [int(r) for r in rows]
    rng = np.random.default_rng(seed)
    recs, pids = [], []
    for i in range(n_patients):
        g = torch.Generator().manual_seed(seed + i)
        x = torch.randn(rows[i], C, generator=g)
        if nonneg:
            x = torch.relu(x) * 0.5
        pid, sid = f"P{i:05d}", f"S{i:05d}"
        torch.save(x, os.path.join(root, "pt_files", sid + ".pt"))
        recs.append({"pathology_id": sid, "patient_id": pid, "e": int(rng.uniform() < event_rate), "t": float(rng.integers(30, 2500))})
        pids.append(pid)
    if not any(r["e"] for r in recs):
        recs[0]["e"] = 1
    pd.DataFrame(recs).to_csv(os.path.join(root, "labels.csv"), index=False)
    n_train = n_patients - n_val
    np.savez(os.path.join(root, "split-fold0.npz"), train_patients=np.array(pids[:n_train]),
             val_patients=np.array(pids[n_train:] if n_val else pids[:1]))
    return {"path_patch": os.path.join(root, "pt_files"), "path_label": os.path.join(root, "labels.csv"),
            "data_split_path": os.path.join(root, "split-fold{}.npz"), "save_path": os.path.join(root, "results", "run")}


@contextlib.contextmanager
def _cuda_as_identity():
    """CPU baseline: the handler's hard-coded `.cuda()` / `torch.cuda.set_device` (model_handler.py:40,90-91,315-316)
    become no-ops for the duration of the block."""
    saved = (torch.cuda.set_device, nn.Module.cuda, torch.Tensor.cuda)
    torch.cuda.set_device = lambda *a, **k: None
    nn.Module.cuda = lambda self, *a, **k: self
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        yield
    finally:
        torch.cuda.set_device, nn.Module.cuda, torch.Tensor.cuda = saved


def device_context(device: str):
    return _cuda_as_identity() if device == "cpu" else contextlib.nullcontext()


def make_handler(cfg: Dict, impl: str = "reference", device: str = "cuda", quiet: bool = True):
    """`MyHandler(cfg)` (model_handler.py:36-137), unmodified."""
    mod = handler_module(impl)
    sink = io.StringIO()
    with device_context(device), (contextlib.redirect_stdout(sink) if quiet else contextlib.nullcontext()):
        h = mod.MyHandler(dict(cfg))
    return h


def set_dropout(module: nn.Module, p: float):
    """Sets every dropout probability of a reference OR advmil_b200 module tree (test aid: p = 0 makes a training epoch
    independent of the dropout generator, which differs by design -- Philox vs counter hash)."""
    for m in module.modules():
        if isinstance(m, nn.Dropout):
            m.p = p
        for attr in ("p", "p_head"):
            if isinstance(getattr(m, attr, None), float) and not isinstance(m, nn.Dropout):
                setattr(m, attr, p)


class InMemoryBags(torch.utils.data.Dataset):
    """WSIPatch's item format (dataset/PatchWSI.py:65-83: `index, (feats, Tensor([0])), label`) from tensors in memory."""

    def __init__(self, feats: Sequence[torch.Tensor], t: Sequence[float], e: Sequence[float], cycle: int = 1):
        self.feats, self.t, self.e, self.cycle = list(feats), list(t), list(e), cycle
        self.pids = [f"P{i:05d}" for i in range(len(self))]

    def __len__(self):
        return len(self.t) * self.cycle if len(self.feats) == len(self.t) else len(self.t)

    def __getitem__(self, index):
        j = index % len(self.feats)
        k = index % len(self.t)
        return (torch.Tensor([index]).to(torch.int), (self.feats[j], torch.Tensor([0])),
                torch.Tensor((self.t[k], self.e[k])).to(torch.float))


def collate_to_handler(items, device: str):
    """What `_train_each_epoch` (model_handler.py:311-319) builds per bag from the DataLoader: x = [feats[1,N,C], ext[1,1]],
    y = [1,2]."""
    xs, ys = [], []
    for _idx, (feats, ext), label in items:
        xs.append([feats.unsqueeze(0).to(device), ext.unsqueeze(0).to(device)])
        ys.append(label.unsqueeze(0).to(device))
    return xs, ys


def handler_step(handler, i_batch: int, xs, ys, mode: str = "wlabel", label_visible_mask: Optional[List[bool]] = None,
                 quiet: bool = True):
    """One optimiser step of the reference: `_update_disc` then `gen_updates` x `_update_gen` (model_handler.py:328-335)."""
    sink = io.StringIO()
    with (contextlib.redirect_stdout(sink) if quiet else contextlib.nullcontext()):
        preds, fakes = handler._update_disc(i_batch, xs, ys, mode, label_visible_mask)
        for _ in range(handler.cfg["gen_updates"]):
            handler._update_gen(i_batch, xs, ys, mode, label_visible_mask)
    return preds, fakes, sink.getvalue()


def parse_losses(log: str) -> Dict[str, List[float]]:
    """dis_loss / gen_loss / t_reg_loss / gen_totol_loss series from the handler's own prints (model_handler.py:413,487-489)."""
    import re
    out = {"dis_loss": [], "gen_loss": [], "t_reg_loss": [], "gen_totol_loss": []}
    for k in out:
        out[k] = [float(v) for v in re.findall(k + r": (-?[0-9.]+(?:e-?[0-9]+)?)", log)]
    return out

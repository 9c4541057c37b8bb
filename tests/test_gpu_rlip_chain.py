"""Region-level chain of the RLIP head (csrc/rlip_chain.cu; reference model/model_utils.py:202-210 and
model/backbone_utils.py:47-56).  rlip_chain_fwd runs one of two tilings chosen by the region count of the launch: 64-region
CTAs while the launch fits two of them per SM, 32-region CTAs beyond.  Both are checked against the CPU oracle (eval and
train with injected masks; outputs, dt and every D gradient): the 64-region tiling on region counts that leave ragged tiles
(1, 37, 100 and 165 regions), the 32-region tiling on a count above the threshold.  The two tilings are also compared with
each other on the same bag, once alone and once packed with a bag that pushes the launch over the threshold."""
import numpy as np
import pytest
import torch

from advmil_b200 import ops
from oracle import advmil_oracle as O
from tests.util import build_D, d_masks, to_dev_masks

pytestmark = pytest.mark.gpu


def _close(a, e, rtol, name, atol=0.0):
    scale = float(np.abs(e).max())
    err = np.abs(a.astype(np.float64) - e.astype(np.float64))
    tol = rtol * np.abs(e) + rtol * scale + atol + 1e-12
    assert not (err > tol).any(), f"{name}: max err {err.max():.3e} (scale {scale:.3e})"


def _vs_oracle(N, train, seed, C=1024):
    sd = O.synth_state_dict(O.D_SHAPES(C, 128, (64, 128)), seed + 50)
    D = build_D(C, 128, "instance", "x")
    D.load_state_dict({k: v.clone() for k, v in sd.items()})
    x = O.synth_bag(N, seed, C)
    masks = d_masks(N // 16, 128, seed * 10 + 5) if train else None
    D.train(train)
    if train:
        D._inject_masks = to_dev_masks(masks)
    t = torch.tensor([[0.41]], device="cuda", requires_grad=True)
    o = D(x.cuda().unsqueeze(0), t)
    o.sum().backward()
    got = {"out": o.detach().cpu().numpy(), "dt": t.grad.cpu().numpy()}
    got.update({"g." + k: p.grad.detach().cpu().numpy() for k, p in D.named_parameters()})

    sdr = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    t2 = torch.tensor([[0.41]], requires_grad=True)
    od = O.prjdisc_forward(sdr, x, t2, masks, "instance", "x")
    od["out"].sum().backward()
    ref = {"out": od["out"].detach().numpy(), "dt": t2.grad.numpy()}
    ref.update({"g." + k: v.grad.numpy() for k, v in sdr.items() if v.grad is not None})

    # fp32 mode: 1e-5, norm-wise per tensor; gradients that cancel to ~0 are skipped as in
    # test_gpu_parity_modules._cmp_grads; the same rule: |a - e| <= 1e-5 (|e| + max|e|) + one fp32 ulp of the network's
    # largest gradient entry (tests/util.py)
    floor = max(2.0 ** -23 * float(np.abs(v).max()) for k, v in ref.items() if k.startswith("g."))
    for k, e in ref.items():
        if float(np.abs(e).max()) < 1e-7:
            continue
        _close(got[k], e, 1e-5, f"N={N} train={train}: {k}", atol=floor if k.startswith("g.") else 0.0)


def test_chain_variants_agree_with_the_oracle_and_with_each_other():
    for N, train, seed in ((16, True, 3), (592, False, 4), (1600, True, 5), (2640, True, 6)):
        _vs_oracle(N, train, seed)
    # above the threshold (cdiv(R, 64) > 2 * SMs): the 32-region tiling; 64 input features keep the oracle cheap
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    R_big = 2 * sms * 64 + 37
    _vs_oracle(16 * R_big, True, 7, C=64)

    # the same 165-region bag through both tilings: alone (64-region CTAs), then first in a launch that also holds R_big
    # regions (32-region CTAs); forward outputs to fp32 rounding (same absolute floor as test_discriminator_vs_oracle)
    C = 64
    D = build_D(C, 128, "instance", "x").eval()
    D.load_state_dict(O.synth_state_dict(O.D_SHAPES(C, 128, (64, 128)), 58))
    x = O.synth_bag(2640, 8, C).cuda()
    filler = O.synth_bag(16 * R_big, 9, C).cuda()
    with torch.no_grad():
        alone = D.forward_packed(ops.PackedBags.from_single(x), torch.tensor([[0.41]], device="cuda")).reshape(-1)
        packed = D.forward_packed(ops.PackedBags.from_list([x, filler]), torch.tensor([[0.41], [0.7]], device="cuda")).reshape(-1)
    _close(packed[:1].cpu().numpy(), alone.cpu().numpy(), 1e-5, "64-region vs 32-region tiling", atol=1e-5 * 1e-2)

"""GPU: the ESAT self-attention kernels at stage level (`advmil_mha_fwd/_bwd`): the tcgen05 forward (head widths 16/32/48/64)
against a float64 torch reference and against the FFMA kernels, on ragged bags whose region counts straddle the 128-key tiles
(1, 37, 128, 129, 300 regions), eval and with in-kernel dropout (the tensor-core forward must drop the same probabilities as
the FFMA forward: same generator, same indices), and the backward pass of the tensor-core mode against autograd.  Head
width 8 has no tcgen05 kernel: in the tf32 mode it runs the FFMA kernels, checked by the same cases."""
import ctypes as C

import numpy as np
import pytest
import torch

from advmil_b200 import _lib, ops

pytestmark = pytest.mark.gpu
RB = [1, 37, 128, 129, 300]


def _offsets(rb):
    offs = [0]
    for n in rb:
        offs.append(offs[-1] + n)
    return torch.tensor(offs, dtype=torch.int32, device="cuda"), (C.c_int32 * len(offs))(*offs)


def _fwd(qkv, rb, d, heads, precision, p=0.0, seed=0, train=0):
    lib = _lib.load()
    R = qkv.shape[0]
    od, oh = _offsets(rb)
    ctx = torch.full((R, d), float("nan"), device="cuda")
    lse = torch.full((heads, R), float("nan"), device="cuda")
    _lib.check(lib.advmil_mha_fwd(qkv.data_ptr(), od.data_ptr(), oh, len(rb), d, heads, p, seed, train, None, None, precision,
                                  ctx.data_ptr(), lse.data_ptr(), torch.cuda.current_stream().cuda_stream), "advmil_mha_fwd")
    return ctx, lse


def _ref(qkv, rb, d, heads):
    hd = d // heads
    q, k, v = qkv.double().split(d, dim=1)
    outs, lses, r0 = [], [], 0
    for n in rb:
        qs, ks, vs = (t[r0:r0 + n].reshape(n, heads, hd).transpose(0, 1) for t in (q, k, v))
        s = qs @ ks.transpose(1, 2) / np.sqrt(hd)
        lses.append(torch.logsumexp(s, dim=-1))
        outs.append((torch.softmax(s, dim=-1) @ vs).transpose(0, 1).reshape(n, d))
        r0 += n
    return torch.cat(outs), torch.cat(lses, dim=1)


@pytest.mark.parametrize("hd", [8, 16, 32, 48, 64])
def test_tcgen05_attention_forward_vs_float64_and_ffma(hd):
    heads = 4
    d = hd * heads
    torch.manual_seed(hd)
    qkv = torch.randn(sum(RB), 3 * d, device="cuda")
    ref, ref_lse = _ref(qkv, RB, d, heads)
    exact, exact_lse = _fwd(qkv, RB, d, heads, ops.FP32)
    assert float((exact.double() - ref).abs().max()) < 2e-5 and float((exact_lse.double() - ref_lse).abs().max()) < 2e-5
    tc, tc_lse = _fwd(qkv, RB, d, heads, ops.PRECISIONS["tf32"])
    assert not bool(torch.isnan(tc).any()) and not bool(torch.isnan(tc_lse).any())
    scale = float(ref.abs().max())
    assert float((tc.double() - ref).abs().max()) < 6e-3 * scale           # tf32 operands (10-bit mantissa) on both contractions
    assert float((tc_lse.double() - ref_lse).abs().max()) < 2e-2


def test_tcgen05_attention_dropout_uses_the_generator_of_the_other_kernels():
    """In-kernel dropout: the tensor-core forward and the FFMA forward draw the same keep bits (counter generator keyed by
    (region, head) row and key column), so their outputs agree to tf32 accuracy, and a third of the output mass is gone
    compared with eval (p = 0.25 with the 1 / (1 - p) rescale keeps the expectation, not the value)."""
    heads, hd = 8, 48
    d = heads * hd
    torch.manual_seed(7)
    qkv = torch.randn(sum(RB), 3 * d, device="cuda")
    a, _ = _fwd(qkv, RB, d, heads, ops.FP32, p=0.25, seed=1234, train=1)
    b, _ = _fwd(qkv, RB, d, heads, ops.PRECISIONS["tf32"], p=0.25, seed=1234, train=1)
    e, _ = _fwd(qkv, RB, d, heads, ops.FP32)
    scale = float(a.abs().max())
    assert float((a - b).abs().max()) < 6e-3 * scale
    assert float((a - e).abs().max()) > 1e-2 * scale                       # dropout really happened
    c, _ = _fwd(qkv, RB, d, heads, ops.PRECISIONS["tf32"], p=0.25, seed=1235, train=1)
    assert float((b - c).abs().max()) > 1e-2 * scale                       # and depends on the seed


@pytest.mark.parametrize("hd", [8, 16, 32, 48, 64])
def test_tensor_core_attention_backward_vs_autograd(hd):
    heads = 4
    d = hd * heads
    torch.manual_seed(100 + hd)
    R = sum(RB)
    qkv = torch.randn(R, 3 * d, device="cuda")
    g = torch.randn(R, d, device="cuda")
    x = qkv.double().requires_grad_(True)
    ref, _ = _ref(x, RB, d, heads)
    (ref * g.double()).sum().backward()
    lib = _lib.load()
    prec = ops.PRECISIONS["tf32"]
    ctx, lse = _fwd(qkv, RB, d, heads, prec)
    od, oh = _offsets(RB)
    d_qkv = torch.full_like(qkv, float("nan"))
    scratch = torch.empty(heads * R, device="cuda")
    _lib.check(lib.advmil_mha_bwd(qkv.data_ptr(), ctx.data_ptr(), g.data_ptr(), lse.data_ptr(), od.data_ptr(), oh, len(RB), d, heads, 0.0,
                                  0, 0, None, None, prec, d_qkv.data_ptr(), scratch.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "advmil_mha_bwd")
    scale = float(x.grad.abs().max())
    assert not bool(torch.isnan(d_qkv).any())
    assert float((d_qkv.double() - x.grad).abs().max()) < 1e-2 * scale


def _bwd(qkv, g, rb, d, heads, precision, p=0.0, seed=0, train=0):
    lib = _lib.load()
    R = qkv.shape[0]
    ctx, lse = _fwd(qkv, rb, d, heads, precision, p=p, seed=seed, train=train)
    od, oh = _offsets(rb)
    d_qkv = torch.full_like(qkv, float("nan"))
    scratch = torch.empty(heads * R, device="cuda")
    _lib.check(lib.advmil_mha_bwd(qkv.data_ptr(), ctx.data_ptr(), g.data_ptr(), lse.data_ptr(), od.data_ptr(), oh, len(rb), d, heads, p,
                                  seed, train, None, None, precision, d_qkv.data_ptr(), scratch.data_ptr(),
                                  torch.cuda.current_stream().cuda_stream), "advmil_mha_bwd")
    return d_qkv


@pytest.mark.parametrize("hd", [32, 48])
def test_tcgen05_attention_backward_with_dropout_equals_the_ffma_backward(hd):
    """Same seed, dropout on: the tcgen05 dQ and dK/dV passes (the latter shares each 32-bit draw between the two lanes of a key
    pair) drop exactly the probabilities the FFMA kernels drop -- the gradients agree to tf32 accuracy -- and they are
    deterministic from run to run."""
    heads = 4
    d = hd * heads
    torch.manual_seed(200 + hd)
    R = sum(RB)
    qkv = torch.randn(R, 3 * d, device="cuda")
    g = torch.randn(R, d, device="cuda")
    exact = _bwd(qkv, g, RB, d, heads, ops.FP32, p=0.25, seed=77, train=1)
    tc = _bwd(qkv, g, RB, d, heads, ops.PRECISIONS["tf32"], p=0.25, seed=77, train=1)
    tc2 = _bwd(qkv, g, RB, d, heads, ops.PRECISIONS["tf32"], p=0.25, seed=77, train=1)
    other = _bwd(qkv, g, RB, d, heads, ops.PRECISIONS["tf32"], p=0.25, seed=78, train=1)
    scale = float(exact.abs().max())
    assert not bool(torch.isnan(tc).any())
    assert float((tc - exact).abs().max()) < 1e-2 * scale
    assert torch.equal(tc, tc2)
    assert float((tc - other).abs().max()) > 5e-2 * scale

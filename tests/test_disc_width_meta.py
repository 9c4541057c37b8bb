"""CPU: the registered discriminator operators trace on the meta device at disc_netx_out_dim 64 and 256 (d), with the
shapes of every output and a backward that reaches every parameter.  No kernel runs."""
import pytest
import torch

from advmil_b200 import library, ops
from tests.test_library_meta import _bags, _meta
from tests.util import build_D


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("d", [64, 256])
def test_discriminator_op_traces_on_meta_at_width(d, precision):
    D = build_D(d=d, device="cpu")
    D.train()
    dp = _meta(D.disc_params())
    bags = _bags([320, 640])
    t = torch.empty(2, device="meta", requires_grad=True)
    u8 = dict(dtype=torch.uint8, device="meta")
    dm = {"fc1": torch.empty(60, d // 2, **u8), "ga": torch.empty(60, d, **u8), "gs": torch.empty(60, d, **u8),
          "fc2": torch.empty(2, d // 2, **u8)}
    f = library.discriminator(D.config(), bags, t, True, 12, dm, ops.PRECISIONS[precision], dp)
    assert tuple(f.shape) == (2,) and f.dtype == torch.float32
    f.sum().backward()
    assert t.grad is not None and tuple(t.grad.shape) == (2,)
    for p in dp:
        if p is not None:
            assert p.grad is not None and p.grad.shape == p.shape
    assert D.config().d == d

"""GPU: the per-bag kernels against float64, over bag counts, bag lengths and widths on both sides of their thresholds.

Kernels: segmented softmax pooling (seg_kernels.cu), the per-(bag, cluster) mean, the generator noise head, the RLIP tail,
the losses, Adam, the L1 sum (tail_kernels.cu) and the fp32 -> bf16 cast.  They are called through the C ABI.

References are float64, built from exactly the values the kernel consumes (bf16 inputs as bf16, fp32 otherwise).  Every
output is prefilled with NaN, so an element the kernel does not write fails; the `+=` outputs (loss_out, losses, the
abs_sum result) are prefilled with a known value and checked as prefill + result.

Bounds come from the arithmetic, not from a run (u = 2^-24, the fp32 unit roundoff):
  * a sum whose additions form chains of at most D steps (per-thread loops, shared-memory folds, warp / block trees)
    errs by at most D u sum |terms|; each case computes D from the kernel's launch geometry;
  * expf errs by at most 2 ulp, and its argument (a difference of two floats) by u |argument|, so exp(s - M) carries
    (2 + |s - M|) u of relative error;
  * products, quotients and the bf16 rounding of an output add one rounding each (2^-9 relative for bf16).
Before a bound is relied on, the case shows that it catches a planted fault at that shape (`_check`): the float64
reference rebuilt with one row dropped at a chunk boundary, with one bag's output taken from another bag, with a slice
of a mat-vec lost, and the like.  Shapes the library refuses are asserted by status code and `advmil_last_error` text.
Gradients that pass through a whole network (the generator's, the RLIP head's) are held at the fp32 parity bound of the
module tests (`_parity_tol`: 2e-5 of each entry and of the tensor's largest entry, plus 8 gradient floors of
tests/util.py; 1e-5 for the tail's own outputs), after the case is moved off its ReLU boundaries; these bounds too must
first see their planted faults (a cluster rank's slice of a gradient lost, a bag left out of a sum over bags, d_bagv's
columns or d_fbar lost)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from advmil_b200 import _lib, ops
from oracle import advmil_oracle as O
from tests.util import assert_close, grad_floor

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
BF16_HALF_ULP = 2.0 ** -8          # relative rounding error of round-to-nearest-even to bf16 (8 significant bits)
SUBNORMAL = 2.0 ** -149
ERR_INVALID = 1
F64 = torch.float64


def _lib_():
    return _lib.load()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _last_error():
    return _lib_().advmil_last_error().decode()


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), dtype=dtype, device="cuda")


def _ptr(t):
    return None if t is None else t.data_ptr()


def _bad(got, ref, tol):
    """number of elements outside the bound (a NaN is outside)"""
    err = (got.double() - ref.double()).abs()
    return int((~(err <= tol)).sum())


def _check(name, got, ref, tol, faults):
    """each planted fault must violate the bound at this shape; then the kernel's output must meet it"""
    assert faults, name
    for fname, fref in faults.items():
        assert _bad(fref, ref, tol) > 0, f"{name}: the bound cannot see the planted fault '{fname}'"
    n = _bad(got, ref, tol)
    if n:
        err = (got.double() - ref.double()).abs()
        ratio = float(torch.nan_to_num(err / tol, nan=float("inf")).max())
        raise AssertionError(f"{name}: {n}/{ref.numel()} elements outside the bound (worst error / bound {ratio:.3g})")


def _swap_bags(t):
    """bag 0's output exchanged with the bag whose output differs most from it"""
    j = int((t - t[:1]).abs().reshape(t.shape[0], -1).sum(1).argmax())
    f = t.clone()
    f[0], f[j] = t[j], t[0]
    return f


def _refuse(status, pattern):
    assert status == ERR_INVALID, status
    assert pattern in _last_error(), _last_error()


def _offsets(lengths):
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int32)
    return torch.tensor(offs, device="cuda"), (C.c_int32 * len(offs))(*offs.tolist()), offs


def _bag_ids(lengths):
    return torch.repeat_interleave(torch.arange(len(lengths), device="cuda"), torch.tensor(lengths, device="cuda"))


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


# =====================================================================================================================
# 1. segmented softmax pool: advmil_seg_softmax_pool_fwd
# =====================================================================================================================
POOL_CH = 256                                      # rows per chunk (seg_kernels.cu)
POOL_WIDTHS = [("f32", 4), ("f32", 64), ("f32", 384), ("f32", 1000), ("f32", 1024), ("bf16", 8), ("bf16", 384), ("bf16", 1024)]
POOL_LENGTHS = {
    "edges": [1, 255, 256, 257, 512, 513],         # chunk boundaries on both sides
    "long": [16384],                               # 64 chunks: the benchmark's bag size
    "many": None,                                  # 300 bags of 1-40 rows: the z CTAs outnumber the w CTAs
}
LOGITS = ("random", "apart", "equal", "dominant")


def _pool_threads(width, vec):
    """seg_softmax_pool_fwd_t's block size and row groups (RG)"""
    wv = width // vec
    threads = 256
    if (8 * wv) % 32 == 0 and 8 * wv <= 512:
        threads = 8 * wv
    elif (4 * wv) % 32 == 0 and 4 * wv <= 512:
        threads = 4 * wv
    return threads, min(threads // wv, POOL_CH)


def _pool_lengths(name):
    if POOL_LENGTHS[name] is not None:
        return list(POOL_LENGTHS[name])
    return torch.randint(1, 41, (300,), generator=torch.Generator().manual_seed(7)).tolist()


def _drop_row(lengths):
    """(bag, packed row) of the fault row: the first row of the second chunk of the longest bag (its last row if shorter)"""
    b = int(np.argmax(lengths))
    return b, int(np.sum(lengths[:b])) + min(POOL_CH, lengths[b] - 1)


def _logits(kind, lengths, g):
    rows = sum(lengths)
    bag = _bag_ids(lengths)
    offs = torch.tensor(np.concatenate([[0], np.cumsum(lengths)[:-1]]), device="cuda")
    pos = torch.arange(rows, device="cuda") - offs[bag]
    if kind == "equal":
        return torch.full((rows,), 0.7, device="cuda")
    s = torch.randn(rows, device="cuda", generator=g) * 2
    if kind == "apart":                 # chunk maxima 150 apart: the low chunks' rescale exp(m_c - M) is exactly 0
        s = s * 0.5 - 150.0 * ((pos // POOL_CH) % 2 == 0).float()
    elif kind == "dominant":            # one row dominates its bag (the fault row, when there is one)
        s[_drop_row(lengths)[1]] += 30.0
    else:                               # the fault row carries one of its bag's largest weights
        s[_drop_row(lengths)[1]] = float(s.max())
    return s


def _pool_ref(s, v64, lengths, drop=None):
    """float64 softmax pool; drop: a packed row left out (the planted fault)"""
    bag = _bag_ids(lengths)
    nb, width = len(lengths), v64.shape[1]
    s64 = s.double()
    keep = torch.ones_like(s64)
    if drop is not None:
        keep[drop] = 0
    M = torch.full((nb,), -math.inf, dtype=F64, device="cuda").scatter_reduce(0, bag, s64, "amax")
    e = torch.exp(s64 - M[bag]) * keep
    L = torch.zeros(nb, dtype=F64, device="cuda").index_add(0, bag, e)
    w = torch.where(L[bag] > 0, e / L[bag], torch.zeros_like(e))
    z = torch.zeros(nb, width, dtype=F64, device="cuda").index_add(0, bag, w[:, None] * v64)
    cnt = torch.zeros(nb, dtype=F64, device="cuda").index_add(0, bag, keep)
    mean = torch.zeros(nb, width, dtype=F64, device="cuda").index_add(0, bag, v64 * keep[:, None]) / cnt.clamp(min=1)[:, None]
    return w, z, mean, M


def _pool_call(s, v, lengths, want_mean, rows=None):
    lib = _lib_()
    rows, width = v.shape[0] if rows is None else rows, v.shape[1]
    nb = len(lengths)
    offs, offs_h, _ = _offsets(lengths)
    w, z = _nan(max(rows, 1)), _nan(nb, width)
    mean = _nan(nb, width) if want_mean else None
    ws = torch.empty(lib.advmil_seg_pool_workspace_bytes(rows, nb, width), dtype=torch.uint8, device="cuda")
    elem = ops.ELEM_BF16 if v.dtype == torch.bfloat16 else ops.ELEM_F32
    st = lib.advmil_seg_softmax_pool_fwd(s.data_ptr(), v.data_ptr(), elem, offs.data_ptr(), offs_h, rows, nb, width, w.data_ptr(),
                                         z.data_ptr(), _ptr(mean), ws.data_ptr(), ws.numel(), _stream())
    return st, w, z, mean


def _pool_cases():
    out = []
    for elem, width in POOL_WIDTHS:
        for lname in POOL_LENGTHS:
            for i, kind in enumerate(LOGITS):
                out.append(pytest.param(elem, width, lname, kind, i % 2 == 0, id=f"{elem}-w{width}-{lname}-{kind}"))
    return out


@pytest.mark.parametrize("elem,width,lname,kind,want_mean", _pool_cases())
def test_seg_softmax_pool_vs_float64(elem, width, lname, kind, want_mean):
    """w, z (and the plain mean) against float64, Σw = 1 per bag.  Thread choice 8·WV / 4·WV / 256 and the row groups
    follow _pool_threads; width 1000 leaves a partial row group, fp32 1024 runs one row group (RG = 1)."""
    vec = 8 if elem == "bf16" else 4
    threads, RG = _pool_threads(width, vec)
    lengths = _pool_lengths(lname)
    g = _gen(width * 7 + len(lengths))
    rows = sum(lengths)
    v = torch.randn(rows, width, device="cuda", generator=g)
    fb, fr = _drop_row(lengths)
    v[fr] = (2 + v[fr].abs()) * torch.sign(torch.randn(width, device="cuda", generator=g))   # a fault row that matters
    if elem == "bf16":
        v = v.to(torch.bfloat16)
    s = _logits(kind, lengths, g)
    st, w, z, mean = _pool_call(s, v, lengths, want_mean)
    assert st == 0, _last_error()

    v64 = v.double()
    w_ref, z_ref, m_ref, M = _pool_ref(s, v64, lengths)
    bag = _bag_ids(lengths)
    nb = len(lengths)
    dev = (s.double() - M[bag]).abs()                        # |s - M|: the exp argument's size
    nch = -(-max(lengths) // POOL_CH)
    d_rows = -(-POOL_CH // RG) + 4 + RG                      # per-thread chain over the chunk's rows + the RG fold
    d_z = d_rows + -(-nch // 8) + 8 + 2                      # + 8 chunk groups + their fold + the 1/L product
    d_L = 2 * (-(-POOL_CH // threads) + 10) + -(-nch // 256) + 10
    sum_wdev = torch.zeros(nb, dtype=F64, device="cuda").index_add(0, bag, w_ref * dev)
    k_L = 8 + d_L + 2 * sum_wdev                             # relative error of L = Σ_c l_c exp(m_c - M), in ulps
    # SUBNORMAL: the spacing of fp32 subnormals; weights far below their bag's maximum are subnormal or 0
    tol_w = U * w_ref * (6 + 2 * dev + k_L[bag]) + 4 * SUBNORMAL
    awv = w_ref[:, None] * v64.abs()
    a_z = torch.zeros(nb, width, dtype=F64, device="cuda").index_add(0, bag, awv * (d_z + 6 + 2 * dev[:, None]))
    tol_z = U * (a_z + k_L[:, None] * z_ref.abs()) + 4 * SUBNORMAL

    fw, fz, fm, _ = _pool_ref(s, v64, lengths, drop=fr)
    _check("w", w, w_ref, tol_w, {"row dropped at a chunk boundary": fw})
    zf = {"row dropped at a chunk boundary": fz}
    if nb > 1:
        zf["bag from its neighbour"] = _swap_bags(z_ref)
    _check("z", z, z_ref, tol_z, zf)
    sw = torch.zeros(nb, dtype=F64, device="cuda").index_add(0, bag, w.double())
    tol_sw = torch.zeros(nb, dtype=F64, device="cuda").index_add(0, bag, tol_w) + 2 * U
    assert bool(((sw - 1).abs() <= tol_sw).all()), f"Σw - 1: {float((sw - 1).abs().max()):.3e}"
    if want_mean:
        cnt = torch.tensor(lengths, dtype=F64, device="cuda")
        a_m = torch.zeros(nb, width, dtype=F64, device="cuda").index_add(0, bag, v64.abs()) / cnt[:, None]
        tol_m = U * ((d_z + 4) * a_m + m_ref.abs())
        mf = {"row dropped at a chunk boundary": fm}
        if nb > 1:
            mf["bag from its neighbour"] = _swap_bags(m_ref)
        _check("mean", mean, m_ref, tol_m, mf)


@pytest.mark.parametrize("elem,width,lengths,pattern", [
    ("f32", 64, [3, 0, 5], "bag 1 is empty"),
    ("bf16", 64, [0], "bag 0 is empty"),
    ("f32", 6, [5, 7], "width 6 must be a multiple of 4 and <= 1024"),
    ("bf16", 12, [5, 7], "width 12 must be a multiple of 8 and <= 1024"),
    ("f32", 1028, [5, 7], "width 1028 must be a multiple of 4 and <= 1024"),
    ("bf16", 1032, [5, 7], "width 1032 must be a multiple of 8 and <= 1024"),
], ids=["f32-empty-bag", "bf16-empty-bag", "f32-width6", "bf16-width12", "f32-width1028", "bf16-width1032"])
def test_seg_softmax_pool_refuses(elem, width, lengths, pattern):
    rows = sum(lengths)
    v = torch.randn(max(rows, 1), width, device="cuda")
    if elem == "bf16":
        v = v.to(torch.bfloat16)
    s = torch.randn(max(rows, 1), device="cuda")
    st, *_ = _pool_call(s, v, lengths, True, rows=rows)
    _refuse(st, pattern)


# =====================================================================================================================
# 2. per-(bag, cluster) mean: advmil_segment_mean_by_id_fwd / _bwd (the module path of bcb_mode: cluster)
# =====================================================================================================================
CL_CH = 128                                         # rows per chunk (tail_kernels.cu)
SEG_LENGTHS = {"edges": [127, 128, 129, 1000], "many": None}
# (ncl, width): ncl * width * 4 bytes below, at and above the 48 KB opt-in threshold, and at the 96 KB limit
SEG_SHAPES = [(1, 384), (10, 1228), (10, 1232), (64, 192), (64, 196), (64, 384)]


def _seg_lengths(name):
    if SEG_LENGTHS[name] is not None:
        return list(SEG_LENGTHS[name])
    return torch.randint(1, 41, (300,), generator=torch.Generator().manual_seed(11)).tolist()


def _seg_ref(v64, cid, lengths, ncl, drop=None):
    bag = _bag_ids(lengths)
    ok = (cid >= 0) & (cid < ncl)
    if drop is not None:
        ok = ok.clone()
        ok[drop] = False
    key = torch.where(ok, bag * ncl + cid.long(), torch.zeros_like(bag))
    w = ok.double()
    nb = len(lengths)
    sums = torch.zeros(nb * ncl, v64.shape[1], dtype=F64, device="cuda").index_add(0, key, v64 * w[:, None])
    asum = torch.zeros(nb * ncl, v64.shape[1], dtype=F64, device="cuda").index_add(0, key, v64.abs() * w[:, None])
    cnt = torch.zeros(nb * ncl, dtype=F64, device="cuda").index_add(0, key, w)
    out = torch.where(cnt[:, None] > 0, sums / cnt.clamp(min=1)[:, None], torch.zeros_like(sums))
    return out, cnt, asum


def _seg_fwd(v, cid, lengths, ncl):
    lib = _lib_()
    rows, width = v.shape
    nb = len(lengths)
    offs, offs_h, _ = _offsets(lengths)
    out, counts = _nan(max(nb * ncl, 1), width), torch.full((max(nb * ncl, 1),), -7, dtype=torch.int32, device="cuda")
    ws = torch.empty(max(lib.advmil_segment_mean_workspace_bytes(rows, nb, width, ncl), 256), dtype=torch.uint8, device="cuda")
    elem = ops.ELEM_BF16 if v.dtype == torch.bfloat16 else ops.ELEM_F32
    st = lib.advmil_segment_mean_by_id_fwd(v.data_ptr(), elem, cid.data_ptr(), offs.data_ptr(), offs_h, rows, nb, width, ncl,
                                           out.data_ptr(), counts.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
    return st, out, counts


def _seg_cases():
    out = []
    for elem in ("f32", "bf16"):
        for ncl, width in SEG_SHAPES:
            for lname in SEG_LENGTHS:
                if lname == "many" and width > 400:
                    continue
                out.append(pytest.param(elem, ncl, width, lname, id=f"{elem}-ncl{ncl}-w{width}-{lname}"))
    return out


@pytest.mark.parametrize("elem,ncl,width,lname", _seg_cases())
def test_segment_mean_by_id_vs_float64(elem, ncl, width, lname):
    """Forward: means against float64, counts exact, empty clusters zero with count 0, ids -1 and >= ncl counted nowhere.
    Backward (relu_mask 0 and 1) against float64 autograd of the same mean."""
    lengths = _seg_lengths(lname)
    rows, nb = sum(lengths), len(lengths)
    g = _gen(ncl * 1000 + width + nb)
    v = torch.randn(rows, width, device="cuda", generator=g)
    cid = torch.randint(-1, ncl + 2, (rows,), device="cuda", generator=g, dtype=torch.int32)   # -1, ncl, ncl+1 mixed in
    if ncl > 1:
        cid[cid == ncl - 1] = ncl + 1                   # cluster ncl-1 is empty in every bag
    bag0 = int(np.argmax(lengths))
    fr = int(np.sum(lengths[:bag0])) + min(CL_CH, lengths[bag0] - 1)   # fault row: the first row of a second chunk
    cid[fr] = 0
    cid[fr - 1] = 1 if ncl > 1 else -1                  # the fault row's neighbour feeds another mean (or none)
    v[fr] = (2 + v[fr].abs()) * torch.sign(torch.randn(width, device="cuda", generator=g))
    if elem == "bf16":
        v = v.to(torch.bfloat16)
    st, out, counts = _seg_fwd(v, cid, lengths, ncl)
    assert st == 0, _last_error()
    v64 = v.double()
    ref, cnt, asum = _seg_ref(v64, cid, lengths, ncl)
    assert torch.equal(counts.long().cpu(), cnt.long().cpu()), "counts"
    if ncl > 1:
        assert bool((counts.view(nb, ncl)[:, ncl - 1] == 0).all()) and bool((out.view(nb, ncl, width)[:, ncl - 1] == 0).all())
    nch = -(-max(lengths) // CL_CH)
    D = CL_CH + nch + 2                                  # per-thread chain over a chunk's rows, then over the chunks
    tol = U * (D * asum / cnt.clamp(min=1)[:, None] + ref.abs())
    fref, _, _ = _seg_ref(v64, cid, lengths, ncl, drop=fr)
    faults = {"row dropped at a chunk boundary": fref}
    if nb > 1:
        faults["bag from its neighbour"] = torch.cat([ref[ncl:2 * ncl], ref[:ncl], ref[2 * ncl:]])
    _check("out", out, ref, tol, faults)

    d_out = torch.randn(nb * ncl, width, device="cuda", generator=g)
    offs, _, _ = _offsets(lengths)
    lib = _lib_()
    for relu_mask in (0, 1):
        d_v = torch.full((rows, width), float("nan"), dtype=v.dtype, device="cuda")
        st = lib.advmil_segment_mean_by_id_bwd(d_out.data_ptr(), v.data_ptr(), ops.ELEM_BF16 if elem == "bf16" else ops.ELEM_F32,
                                               cid.data_ptr(), offs.data_ptr(), counts.data_ptr(), rows, nb, width, ncl, relu_mask,
                                               d_v.data_ptr(), _stream())
        assert st == 0, _last_error()
        x = v64.clone().requires_grad_(True)
        m, _, _ = _seg_ref(torch.relu(x) if relu_mask else x, cid, lengths, ncl)
        (m * d_out.double()).sum().backward()
        gref = x.grad
        rel = (BF16_HALF_ULP + 3 * U) if elem == "bf16" else 3 * U     # 1 / count, the product (, the bf16 store)
        shifted = gref.clone()
        shifted[fr] = gref[fr - 1]
        _check(f"d_v relu_mask={relu_mask}", d_v, gref, rel * gref.abs(), {"row from its neighbour": shifted})


@pytest.mark.parametrize("ncl,width,pattern", [
    (64, 388, "clusters*width too large"), (1, 24577, "clusters*width too large"), (65, 8, "bad arguments"), (0, 8, "bad arguments"),
])
def test_segment_mean_by_id_refuses(ncl, width, pattern):
    v = torch.randn(12, width, device="cuda")
    cid = torch.zeros(12, dtype=torch.int32, device="cuda")
    st, _, _ = _seg_fwd(v, cid, [5, 7], ncl)
    _refuse(st, pattern)


# =====================================================================================================================
# 3. generator noise head: advmil_generator_sample, and its gradients through advmil_generator_bwd
# =====================================================================================================================
HEAD_CS = 8                                          # CTAs per cluster (tail_kernels.cu)
# (o, hid): the default; a small one where most cluster ranks own no slice; o and hid not multiples of 4 (scalar paths)
HEAD_WIDTHS = [(384, 192), (8, 4), (10, 5)]


def _head_slices(n):
    per = (-(-n // HEAD_CS) + 3) & ~3
    return [(min(n, r * per), min(n, min(n, r * per) + per)) for r in range(HEAD_CS)]


def _dot_chain(n):
    """deepest addition chain of the head / tail mat-vecs over n inputs (col_dot: n / 4 per accumulator)"""
    return n // 4 + 16


def _lin_err(W, x, ex, b, chain):
    """y = W x + b in float64 for a batch of rows x, with the bound of its fp32 evaluation: the propagated input error
    |W| ex plus chain u (|W| |x| + |b|)"""
    y = x @ W.t() + b
    ey = ex @ W.abs().t() + U * (chain * (x.abs() @ W.abs().t()) + b.abs() + y.abs())
    return y, ey


def _head_ref(W0, b0, Wl, bl, H, n0, n1, out_scale, drop_units=None):
    """[S, bags] outputs and bounds.  drop_units: hidden units left out (a rank's lost slice)."""
    S = n1.shape[0] if n1 is not None else n0.shape[0] if n0 is not None else 1
    nb = H.shape[0]
    x = H.double()[None].expand(S, nb, -1)
    if n0 is not None:
        x = torch.cat([x, n0.double()], dim=2)
    h1, e1 = _lin_err(W0.double(), x, torch.zeros_like(x), b0.double(), _dot_chain(x.shape[2]))
    h1 = torch.relu(h1)
    if drop_units is not None:
        h1[..., drop_units] = 0
    xx, ex = h1, e1
    if n1 is not None:
        xx = torch.cat([h1, n1.double()], dim=2)
        ex = torch.cat([e1, torch.zeros_like(n1, dtype=F64)], dim=2)
    pre, ep = _lin_err(Wl.double(), xx, ex, bl.double(), _dot_chain(xx.shape[2]) + 10)
    pre, ep = pre[..., 0], ep[..., 0]
    if out_scale == 1:
        y = torch.sigmoid(pre)
        return y, y * (1 - y) * ep + 6 * U * y
    if out_scale == 2:
        y = torch.exp(pre)
        return y, y * (ep * 1.01 + (4 + pre.abs()) * U)
    return pre, ep


def _head_params(o, hid, noise0, noise1, g):
    W0 = torch.randn(hid, o * (1 + noise0), device="cuda", generator=g) * (o * (1 + noise0)) ** -0.5
    b0 = 2 + 0.3 * torch.rand(hid, device="cuda", generator=g)        # hidden units active: a lost slice shows
    Wl = torch.randn(1, hid * (1 + noise1), device="cuda", generator=g)
    Wl = (0.5 + Wl.abs()) * torch.sign(Wl) * hid ** -0.5              # every hidden unit reaches the output
    bl = torch.randn(1, device="cuda", generator=g) * 0.1
    return W0, b0, Wl, bl


def _sample_cases():
    out = []
    i = 0
    for o, hid in HEAD_WIDTHS:
        for nb in (1, 16, 300):
            for S in (1, 30):
                noise0, noise1, scale = i % 2, (i // 2) % 2, i % 3
                i += 1
                out.append(pytest.param(o, hid, nb, S, noise0, noise1, scale,
                                        id=f"o{o}-hid{hid}-bags{nb}-S{S}-n0{noise0}-n1{noise1}-scale{scale}"))
    return out


@pytest.mark.parametrize("o,hid,nb,S,noise0,noise1,out_scale", _sample_cases())
def test_generator_sample_vs_float64(o, hid, nb, S, noise0, noise1, out_scale):
    """S draws per bag from H [bags, o]: out[s, b] = scale(Wl [relu(W0 [H | noise0] + b0) | noise1] + bl)."""
    g = _gen(o * 31 + nb * 7 + S)
    W0, b0, Wl, bl = _head_params(o, hid, noise0, noise1, g)
    H = torch.relu(torch.randn(nb, o, device="cuda", generator=g))
    n0 = torch.rand(S, nb, o, device="cuda", generator=g) if noise0 else None
    n1 = torch.rand(S, nb, hid, device="cuda", generator=g) if noise1 else None
    p = _lib.GenParams()
    p.W0, p.b0, p.Wl, p.bl = W0.data_ptr(), b0.data_ptr(), Wl.data_ptr(), bl.data_ptr()
    p.C, p.h, p.o, p.hid = o, o, o, hid
    p.noise0, p.noise1, p.out_scale = noise0, noise1, out_scale
    out = _nan(S, nb)
    st = _lib_().advmil_generator_sample(C.byref(p), H.data_ptr(), _ptr(n0), _ptr(n1), nb, S, out.data_ptr(), _stream())
    assert st == 0, _last_error()
    n1r = n1 if noise1 else None
    ref, tol = _head_ref(W0, b0, Wl, bl, H, n0, n1r, out_scale)
    ref, tol = ref.expand(S, nb), tol.expand(S, nb)
    # a rank's slice of the hidden layer lost: the last rank that owns a non-empty slice
    beg, end = [sl for sl in _head_slices(hid) if sl[1] > sl[0]][-1]
    faults = {f"hidden slice [{beg}, {end}) lost": _head_ref(W0, b0, Wl, bl, H, n0, n1r, out_scale, list(range(beg, end)))[0]
              .expand(S, nb)}
    if nb > 1:
        faults["bag from its neighbour"] = _swap_bags(ref.t()).t()
    _check("out", out, ref, tol, faults)


def _gen_sd(C_, h, o, hid, seed):
    shapes = dict(O.G_SHAPES(C_, h, o))
    shapes["MLPs.0.0.weight"], shapes["MLPs.0.0.bias"] = (hid, o), (hid,)
    shapes["MLPs.1.0.weight"] = (1, 2 * hid)
    return O.synth_state_dict(shapes, seed)


def _condition_gen(sd, xs, noise, margin=1e-4, iters=30):
    """Moves the case off the generator's ReLU boundaries (cf. tests/util.py: condition_esat_case): rows of x with a
    first-layer pre-activation within `margin` of zero get a small perturbation, rho and MLPs.0 columns a bias nudge, until
    the float64 oracle sees none left.  A ReLU argument within rounding of zero may take either branch in fp32, and one
    flipped branch moves a whole gradient row."""
    sd = {k: v.clone() for k, v in sd.items()}
    xs = [x.clone() for x in xs]
    g = torch.Generator().manual_seed(93)
    W1, b1 = "backbone.attention_net.0.weight", "backbone.attention_net.0.bias"
    for _ in range(iters):
        s = {k: v.double() for k, v in sd.items()}
        clean = True
        for x in xs:
            bad = torch.nonzero(((x.double() @ s[W1].T + s[b1]).abs() < margin).any(dim=1)).reshape(-1)
            if bad.numel():
                x[bad] += 1e-2 * torch.randn(bad.numel(), x.shape[1], generator=g)
                clean = False
        if not clean:
            continue
        for i, x in enumerate(xs):
            z = O.abmil_forward(s, x.double())["z"]
            pre_rho = z @ s["backbone.rho.0.weight"].T + s["backbone.rho.0.bias"]
            pre_mlp = torch.relu(pre_rho) @ s["MLPs.0.0.weight"].T + s["MLPs.0.0.bias"]
            for key, pre in (("backbone.rho.0.bias", pre_rho), ("MLPs.0.0.bias", pre_mlp)):
                cols = torch.nonzero((pre.abs() < margin).any(dim=0)).reshape(-1)
                if cols.numel():
                    sd[key][cols] += 2 * margin
                    clean = False
        if clean:
            return sd, xs
    raise AssertionError("could not condition the generator case")


GEN_KEYS = ["backbone.attention_net.0.weight", "backbone.attention_net.0.bias",
            "backbone.attention_net.3.attention_a.0.weight", "backbone.attention_net.3.attention_a.0.bias",
            "backbone.attention_net.3.attention_b.0.weight", "backbone.attention_net.3.attention_b.0.bias",
            "backbone.attention_net.3.attention_c.weight", "backbone.attention_net.3.attention_c.bias",
            "backbone.rho.0.weight", "backbone.rho.0.bias", "MLPs.0.0.weight", "MLPs.0.0.bias", "MLPs.1.0.weight", "MLPs.1.0.bias"]


def _parity_tol(ref, rtol, atol):
    """the bound of tests/util.py:assert_close: rtol |e| + rtol max|e| + atol"""
    return rtol * ref.abs() + rtol * float(ref.abs().max()) + atol


def _last_slice(n):
    """[beg, end) of the last cluster rank that owns a non-empty slice of n outputs (head_slice)"""
    return [sl for sl in _head_slices(n) if sl[1] > sl[0]][-1]


def _gen_oracle(sd, xs, noise, d_pred, fault=None):
    """float64 autograd of the oracle generator over the bags: pred and the 14 gradients.  fault: ("z" | "H", beg, end)
    drops that column slice of dL/dz or dL/dH (one cluster rank's share of gen_head_bwd lost), ("bag", j) leaves bag j
    out of the sums over bags."""
    r = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    preds = []
    for i, x in enumerate(xs):
        bb = O.generator_forward(r, x.double(), [None, noise[i:i + 1].double()], (0, 1))
        if fault is not None and fault[0] in ("z", "H"):
            _, beg, end = fault
            bb[fault[0]].register_hook(lambda g, beg=beg, end=end: torch.cat([g[:, :beg], 0 * g[:, beg:end], g[:, end:]], 1))
        preds.append(bb["pred"].reshape(-1))
    pred = torch.cat(preds)
    w = d_pred.cpu().double().clone()
    if fault is not None and fault[0] == "bag":
        w[fault[1]] = 0
    (pred * w).sum().backward()
    return pred.detach(), {k: r[k].grad for k in GEN_KEYS}


@pytest.mark.parametrize("C_,h,o,hid", [(1024, 384, 384, 192), (64, 8, 8, 4), (64, 64, 10, 5)],
                         ids=["default", "small-empty-ranks", "o10-hid5-scalar"])
def test_generator_head_gradients_vs_oracle(C_, h, o, hid):
    """All 14 generator gradients of advmil_generator_bwd in fp32 (eval mode, noise1 on) against float64 autograd of the
    oracle; the head's block_colmat / col_dot paths and the cluster's column slices at these widths.  The bound is the fp32
    parity bound of the module tests (2e-5 of each entry and of the tensor's largest entry, plus 8 gradient floors); it
    must see, per tensor, the faults that reach it: one cluster rank's column slice of dL/dH or of dL/dz lost (at the small
    widths most ranks own none, and at o = 10 the last slice is partial), and one bag left out of the sums over bags."""
    sd = _gen_sd(C_, h, o, hid, 90 + o)
    lengths = [37, 200, 5]
    xs = [O.synth_bag(n, 91 + i, C_) for i, n in enumerate(lengths)]
    noise = torch.rand(len(lengths), hid, generator=torch.Generator().manual_seed(92))
    sd, xs = _condition_gen(sd, xs, noise)
    cfg = ops.GenConfig(C=C_, h=h, o=o, hid=hid, noise0=0, noise1=1, out_scale=1)
    params = [sd[k].cuda() for k in GEN_KEYS]
    bags = ops.PackedBags.from_list([x.cuda() for x in xs])
    acts = ops.generator_forward(cfg, params, bags, None, noise.cuda(), train=False)
    d_pred = torch.linspace(0.5, 1.5, len(lengths), device="cuda")
    grads, _ = ops.generator_backward(cfg, params, bags, acts, d_pred)
    pred, ref = _gen_oracle(sd, xs, noise, d_pred)
    assert_close(acts["pred"].cpu(), pred, 1e-5, "pred")
    sh, sz = _last_slice(o), _last_slice(h)
    fault_sets = {f"dH slice [{sh[0]}, {sh[1]}) lost": _gen_oracle(sd, xs, noise, d_pred, ("H",) + sh)[1],
                  f"dz slice [{sz[0]}, {sz[1]}) lost": _gen_oracle(sd, xs, noise, d_pred, ("z",) + sz)[1],
                  "bag 1 left out of the sums": _gen_oracle(sd, xs, noise, d_pred, ("bag", 1))[1]}
    reaches = {"MLPs.": ("bag 1",), "backbone.rho.": ("bag 1", "dH"), "backbone.attention_net.": ("dH", "dz")}
    floor = 8 * grad_floor(list(ref.values()))
    n = 0
    for k, got in zip(GEN_KEYS, grads):
        if k.endswith("attention_c.bias"):          # mathematically zero (softmax shift)
            continue
        kinds = next(v for p, v in reaches.items() if k.startswith(p))
        faults = {name: f[k] for name, f in fault_sets.items() if name.startswith(kinds)}
        _check("grad " + k, got.cpu(), ref[k], _parity_tol(ref[k], 2e-5, floor), faults)
        n += 1
    assert n == 13


# =====================================================================================================================
# 4. RLIP tail: rlip_tail_fwd / rlip_tail_bwd through advmil_disc_head_fwd / _bwd (fp32)
# =====================================================================================================================
TAIL = ["F2a_w", "F2a_b", "F2b_w", "F2b_b", "T1_w", "T1_b", "T2_w", "T2_b", "Pr_w", "Pr_b"]


def _disc_params(d, t1, prj, g, C_=16):
    dh = d // 2
    sh = {"Wc": (d, C_), "bc": (d,), "ln_g": (d,), "ln_b": (d,), "F1a_w": (dh, d), "F1a_b": (dh,), "F1b_w": (d, dh), "F1b_b": (d,),
          "Pg_w": (d, d), "Pg_b": (d,), "Ps_w": (d, d), "Ps_b": (d,), "Pc_w": (1, d), "Pc_b": (1,), "F2a_w": (dh, d), "F2a_b": (dh,),
          "F2b_w": (d, dh), "F2b_b": (d,), "T1_w": (t1, 1), "T1_b": (t1,), "T2_w": (d, t1), "T2_b": (d,)}
    if prj:
        sh["Pr_w"], sh["Pr_b"] = (1, 2 * d if prj == 3 else d), (1,)
    p = {k: torch.randn(*s, device="cuda", generator=g) * (s[-1] ** -0.5 if len(s) == 2 else 0.3) for k, s in sh.items()}
    return p


def _tail_ref(p, bagv, fbar, t, cfg, drop_last_ht=False):
    """float64 of the tail from the kernel's own bagv / fbar: fc2 MLP, time embedding, inner product, projection.
    `terms` [bags, K] are the products the output sums (its bias aside)."""
    d = cfg.d
    P = {k: v.double() for k, v in p.items() if v is not None}
    g1 = torch.relu(bagv @ P["F2a_w"].t() + P["F2a_b"])
    hx = g1 @ P["F2b_w"].t() + P["F2b_b"]
    u1 = torch.relu(t[:, None] * P["T1_w"].t() + P["T1_b"])
    ht = torch.relu(u1 @ P["T2_w"].t() + P["T2_b"])
    if drop_last_ht:
        ht = ht.clone()
        ht[:, -4:] = 0
    if cfg.prj_path == 3:
        terms = torch.cat([hx * P["Pr_w"][0, :d], ht * P["Pr_w"][0, d:]], dim=1)
    else:
        terms = [(fbar if cfg.inner_instance else hx) * ht]
        if cfg.prj_path in (1, 2):
            terms.append((hx if cfg.prj_path == 1 else ht) * P["Pr_w"][0])
        terms = torch.cat(terms, dim=1)
    out = terms.sum(1) + (P["Pr_b"] if cfg.prj_path else 0.0)
    return {"g1": g1, "hx": hx, "u1": u1, "ht": ht, "out": out, "terms": terms}


def _tail_abs(p, bagv, fbar, t, cfg):
    """the same chain on absolute values: a bound on sum |terms| of every output (ReLU and its argument's magnitude)"""
    d = cfg.d
    P = {k: v.double().abs() for k, v in p.items() if v is not None}
    g1 = bagv.abs() @ P["F2a_w"].t() + P["F2a_b"]
    hx = g1 @ P["F2b_w"].t() + P["F2b_b"]
    u1 = t.abs()[:, None] * P["T1_w"].t() + P["T1_b"]
    ht = u1 @ P["T2_w"].t() + P["T2_b"]
    if cfg.prj_path == 3:
        out = hx @ P["Pr_w"][0, :d] + ht @ P["Pr_w"][0, d:] + P["Pr_b"]
    else:
        out = ((fbar.abs() if cfg.inner_instance else hx) * ht).sum(1)
        if cfg.prj_path in (1, 2):
            out = out + (hx if cfg.prj_path == 1 else ht) @ P["Pr_w"][0] + P["Pr_b"]
    return {"g1": g1, "hx": hx, "u1": u1, "ht": ht, "out": out}


def _head_fwd(cfg, plist, bags, emb, t):
    """advmil_disc_head_fwd with every activation prefilled with NaN; returns (status, activations)"""
    lib = _lib_()
    R, nb, d, dh = bags.rows // 16, bags.bags, cfg.d, cfg.d // 2
    abw = lib.advmil_gate_packed_width(d)
    acts = {"emb": emb, "t": t, "f1": _nan(R, dh), "fi": _nan(R, d), "ab": _nan(R, abw), "rep": _nan(R), "attn": _nan(R),
            "bagv": _nan(nb, d), "fbar": _nan(nb, d), "g1": _nan(nb, dh), "hx": _nan(nb, d), "u1": _nan(nb, cfg.t1),
            "ht": _nan(nb, cfg.t2), "out": _nan(nb), "masks": {}, "seed": 0, "train": False, "precision": ops.FP32}
    pc = cfg.c(plist)
    ws = torch.empty(lib.advmil_disc_workspace_bytes(C.byref(pc), bags.rows, nb, 0), dtype=torch.uint8, device="cuda")
    a = ops._head_struct(acts, ws)
    b = bags.c()
    return lib.advmil_disc_head_fwd(C.byref(pc), C.byref(b), C.byref(a), _stream()), acts


def _tail_case(d, t1, prj, inner, nb, seed):
    cfg = ops.DiscConfig(C=16, d=d, t1=t1, t2=d, inner_instance=inner, prj_path=prj, p=0.25)
    g = _gen(seed)
    p = _disc_params(d, t1, prj, g)
    for key, sl in (("F2a_b", slice(0, 4)), ("T1_b", slice(0, 4)), ("T2_b", slice(-4, None))):
        p[key][sl] = 1.0                                 # the planted-fault rows are active ReLUs
    lengths = [16 * (1 + (i + 2) % 3) for i in range(nb)]      # 3, 1, 2, 3, ... regions: one bag alone still has 3
    bags = ops.PackedBags(torch.zeros(sum(lengths), 16, device="cuda"), lengths)
    emb = torch.relu(torch.randn(sum(lengths) // 16, d, device="cuda", generator=g))
    t = torch.rand(nb, device="cuda", generator=g) * 2
    return cfg, p, lengths, bags, emb, t, g


# (d, t1): vec_ok needs d % 8, t1 % 4 and t2 % 4 == 0; t1 = 50 (disc_nety_hid_dims [50, 128]) takes the scalar warp_dot /
# col_dot side.  d = 100 with hid_dims [50, 100] does not reach the tail: its region MLP (d / 2 = 50 columns) is refused.
TAIL_DIMS = [(128, 64), (128, 50)]


def _tail_cases():
    out = []
    for d, t1 in TAIL_DIMS:
        for kind in ("none-instance", "none-bag", "x-instance", "x-bag", "y-instance", "y-bag", "cat"):
            for nb in (1, 300):
                out.append(pytest.param(d, t1, kind, nb, id=f"d{d}-t1{t1}-{'vec' if t1 % 4 == 0 else 'scalar'}-{kind}-bags{nb}"))
    return out


@pytest.mark.parametrize("d,t1,kind,nb", _tail_cases())
def test_rlip_tail_vs_float64(d, t1, kind, nb):
    """g1, hx, u1, ht and out of rlip_tail_fwd, and d_t and the tail's parameter gradients of rlip_tail_bwd (+ the outer
    sums), against float64 of the oracle's tail (time_embed, the fc2 MLP, the inner product and projection of
    model/GANSurv.py) evaluated at the kernel's own pooled bagv / fbar, in fp32; then d_emb of the whole head backward
    against float64 autograd of the head from emb, which is where rlip_tail_bwd's d_bagv and d_fbar arrive.  Bags whose
    ReLU arguments (region MLP, bag MLP, time MLP) lie within `margin` of zero get a new t and embedding first (as
    test_gpu_disc_width.py moves its cases off the boundaries)."""
    prj = {"none": 0, "x": 1, "y": 2, "cat": 3}[kind.split("-")[0]]
    inner = int(kind.endswith("instance"))
    cfg, p, lengths, bags, emb, t, g = _tail_case(d, t1, prj, inner, nb, d * 13 + t1 + prj * 3 + inner + nb)
    plist = [p.get(k) for k in _lib.DISC_TENSORS]
    P = {k: v.double() for k, v in p.items()}
    bag = _bag_ids(lengths)
    region_bag = bag[::16]
    margin = 1e-4
    for _ in range(30):
        st, acts = _head_fwd(cfg, plist, bags, emb, t)
        assert st == 0, _last_error()
        bagv, fbar = acts["bagv"].double(), acts["fbar"].double()
        pre_g = bagv @ P["F2a_w"].t() + P["F2a_b"]
        pre_u = t.double()[:, None] * P["T1_w"].t() + P["T1_b"]
        pre_h = torch.relu(pre_u) @ P["T2_w"].t() + P["T2_b"]
        pre_f = emb.double() @ P["F1a_w"].t() + P["F1a_b"]
        bad_region = pre_f.abs().lt(margin).any(dim=1)
        bad = torch.cat([pre_g, pre_u, pre_h], dim=1).abs().lt(margin).any(dim=1)
        bad[region_bag[bad_region]] = True
        if not bool(bad.any()):
            break
        t[bad] = torch.rand(int(bad.sum()), device="cuda", generator=g) * 2
        rb = bad[region_bag]
        emb[rb] = torch.relu(torch.randn(int(rb.sum()), d, device="cuda", generator=g))
    assert not bool(bad.any()), "could not condition the tail"
    ref = _tail_ref(p, bagv, fbar, t.double(), cfg)
    mag = _tail_abs(p, bagv, fbar, t.double(), cfg)
    # each layer errs by at most chain u of its |terms| (mat-vec chains, the inner product's block_sum); out is three
    # layers deep, and every layer's |terms| are bounded by the absolute-value chain
    chain = _dot_chain(max(d, t1)) + 24
    lost_ht = _tail_ref(p, bagv, fbar, t.double(), cfg, drop_last_ht=True)["ht"]
    terms = ref["terms"]
    lost_term = ref["out"] - terms.gather(1, terms.abs().argmax(1, keepdim=True))[:, 0]
    for name in ("g1", "hx", "u1", "ht", "out"):
        tol = 3 * chain * U * mag[name] + 2 * U * ref[name].abs()
        if name == "out":
            faults = {"largest term of the sum lost": lost_term}
        elif name == "ht":
            faults = {"last 4-row group lost": lost_ht}
        else:
            f = ref[name].clone()
            f[:, :4] = 0
            faults = {"first 4-row group lost": f}
        if nb > 1:
            faults["bag from its neighbour"] = _swap_bags(ref[name])
        _check(name, acts[name], ref[name], tol, faults)

    # backward, tail level: d_t and the tail's parameter gradients against float64 autograd at the kernel's bagv / fbar
    d_out = torch.randn(nb, device="cuda", generator=g)
    grads = [None if v is None else torch.full_like(v, float("nan")) for v in plist]
    d_t, d_emb = _nan(nb), _nan(*emb.shape)
    ops.disc_head_backward(cfg, plist, bags, acts, d_out, d_emb, d_t, grads)
    j = int(d_out.abs().argmax())

    def tail_grads(weights):
        Pg = {k: v.double().requires_grad_(True) for k, v in p.items()}
        tt = t.double().requires_grad_(True)
        (_tail_ref(Pg, bagv, fbar, tt, cfg)["out"] * weights).sum().backward()
        out = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in Pg.items()}   # unused: zero
        out["d_t"] = tt.grad
        return out
    w = d_out.double()
    want = tail_grads(w)
    w_lost = w.clone()
    w_lost[j] = 0
    lost = tail_grads(w_lost)                           # bag j left out of the sums over bags
    floor = 8 * grad_floor([want[k].cpu() for k in TAIL if k in want] + [want["d_t"].cpu()])
    faults = {f"bag {j} left out": lost["d_t"]}
    if nb > 1:
        faults["d_t from another bag"] = _swap_bags(want["d_t"])
    _check("d_t", d_t, want["d_t"], _parity_tol(want["d_t"], 1e-5, floor), faults)
    n = 0
    for k, got in zip(_lib.DISC_TENSORS, grads):
        if k in TAIL and k in want:
            if not bool(want[k].any()):                 # a tensor the output does not use: its gradient is exactly 0
                assert bool((got == 0).all()), f"grad {k}: expected zeros"
            else:
                _check("grad " + k, got, want[k], _parity_tol(want[k], 1e-5, floor), {f"bag {j} left out": lost[k]})
            n += 1
    assert n == (10 if prj else 8)

    # backward through the head: d_emb against float64 autograd of the whole head from emb.  It is where the tail's
    # d_bagv (F2a_w^T dg1: col_dot when t1 % 4 != 0, block_colmat otherwise) and d_fbar arrive; the bound must see four
    # columns of d_bagv lost, d_fbar lost (when the output uses it) and one region's gradient from another region.
    def head_d_emb(block=None):
        e = emb.double().requires_grad_(True)
        (_head64(P, e, t.double(), cfg, lengths, block) * w).sum().backward()
        return e.grad
    ref_e = head_d_emb()
    faults = {"region from another region": _swap_bags(ref_e)}
    if not (inner and prj in (0, 2)):                   # the output uses hx, so bagv
        faults[f"d_bagv columns [{d - 4}, {d}) lost"] = head_d_emb(("bagv", slice(d - 4, d)))
    if inner and prj != 3:                              # the output uses fbar
        faults["d_fbar lost"] = head_d_emb(("fbar", slice(0, d)))
    _check("d_emb", d_emb, ref_e, _parity_tol(ref_e, 2e-5, 8 * grad_floor([ref_e.cpu()])), faults)


def _block_grad(x, cols):
    """x with its gradient stopped in columns `cols` (the value unchanged)"""
    m = torch.zeros_like(x)
    m[:, cols] = 1
    return x - x * m + (x * m).detach()


def _head64(P, emb, t, cfg, lengths, block=None):
    """float64 RLIP head from the region embedding (model/model_utils.py EmbedXLayer after the embedding, eval mode):
    region MLP, gated attention pooling per bag (bagv) and the plain region mean (fbar), then the tail.  block:
    ("bagv" | "fbar", columns) stops the gradient through those columns (a planted fault)."""
    rb = _bag_ids(lengths)[::16]
    nb = len(lengths)
    f1 = torch.relu(emb @ P["F1a_w"].t() + P["F1a_b"])
    fi = f1 @ P["F1b_w"].t() + P["F1b_b"]
    a = torch.tanh(fi @ P["Pg_w"].t() + P["Pg_b"])
    b = torch.sigmoid(fi @ P["Ps_w"].t() + P["Ps_b"])
    rep = (a * b) @ P["Pc_w"][0] + P["Pc_b"]
    with torch.no_grad():
        M = torch.full((nb,), -math.inf, dtype=F64, device="cuda").scatter_reduce(0, rb, rep, "amax")
    ex = torch.exp(rep - M[rb])
    attn = ex / torch.zeros(nb, dtype=F64, device="cuda").index_add(0, rb, ex)[rb]
    bagv = torch.zeros(nb, fi.shape[1], dtype=F64, device="cuda").index_add(0, rb, attn[:, None] * fi)
    cnt = torch.tensor([n // 16 for n in lengths], dtype=F64, device="cuda")
    fbar = torch.zeros(nb, fi.shape[1], dtype=F64, device="cuda").index_add(0, rb, fi) / cnt[:, None]
    if block is not None:
        if block[0] == "bagv":
            bagv = _block_grad(bagv, block[1])
        else:
            fbar = _block_grad(fbar, block[1])
    return _tail_ref(P, bagv, fbar, t, cfg)["out"]


def test_rlip_head_refuses_d100():
    """d = 100 (disc_nety_hid_dims [50, 100]): the region MLP's 50 columns are refused by the fp32 linear engine"""
    cfg, p, lengths, bags, emb, t, g = _tail_case(100, 50, 1, 1, 3, 5)
    st, _ = _head_fwd(cfg, [p.get(k) for k in _lib.DISC_TENSORS], bags, emb, t)
    _refuse(st, "linear_fwd: K=100 N=50 must be multiples of 4")


# =====================================================================================================================
# 5. losses: advmil_disc_loss (which 0 / 1 / 2) and advmil_gen_loss
# =====================================================================================================================
LOSS_BAGS = (1, 255, 256, 257, 4096)
WHICH = {0: "bce", 1: "hinge", 2: "wasserstein"}


def _mask(kind, nb, g):
    if kind == "off":
        return torch.zeros(nb, dtype=torch.uint8, device="cuda")
    if kind == "on":
        return torch.ones(nb, dtype=torch.uint8, device="cuda")
    m = (torch.rand(nb, device="cuda", generator=g) < 0.4).to(torch.uint8)
    m[0] = 1
    return m


@pytest.mark.parametrize("which", [0, 1, 2], ids=list(WHICH.values()))
@pytest.mark.parametrize("nb", LOSS_BAGS)
@pytest.mark.parametrize("mkind", ["off", "mixed", "on"])
def test_disc_loss_vs_oracle(which, nb, mkind):
    """loss_out[0] += loss, d_real, d_fake against float64 autograd of oracle.real_fake_loss.  Hinge arguments exactly 0
    (f_fake = -1, f_real = 1) take torch's subgradient 0."""
    g = _gen(nb * 3 + which)
    f_real = torch.randn(nb, device="cuda", generator=g) * 2
    f_fake = torch.randn(nb, device="cuda", generator=g) * 2
    f_fake[1::7] = -1.0
    f_real[2::5] = 1.0
    f_fake[0], f_real[0] = 0.5, -0.5                    # bag 0 has nonzero terms and gradients of every kind
    mask = _mask(mkind, nb, g)
    n_real, n_fake = float(mask.sum()), float(nb)
    loss, d_real, d_fake = torch.full((1,), 0.625, device="cuda"), _nan(nb), _nan(nb)
    st = _lib_().advmil_disc_loss(f_real.data_ptr(), f_fake.data_ptr(), mask.data_ptr(), nb, which, n_real, n_fake, loss.data_ptr(),
                                  d_real.data_ptr(), d_fake.data_ptr(), _stream())
    assert st == 0, _last_error()
    fr, ff = f_real.double().requires_grad_(True), f_fake.double().requires_grad_(True)
    sel = mask.bool()
    L = O.real_fake_loss(fr[sel] if n_real > 0 else None, ff, WHICH[which])
    L.backward()
    gr = fr.grad if fr.grad is not None else torch.zeros_like(fr)
    # per-term magnitudes: 1 + |log σ| (bce), |1 ± f| (hinge), |f| (wasserstein); chain: bags / 256 per thread + block_sum
    with torch.no_grad():
        if which == 0:
            lf = -(1 - torch.log(torch.sigmoid(ff) + 1e-8))
            tf, tr = lf.abs(), torch.log(torch.sigmoid(fr) + 1e-8).abs()
        elif which == 1:
            lf = torch.relu(1 + ff)
            tf, tr = 1 + ff.abs(), 1 + fr.abs()
        else:
            lf = ff
            tf, tr = ff.abs(), fr.abs()
        chain = -(-nb // 256) + 16                       # bags per thread, then block_sum
        s = tf.sum() / n_fake + (tr[sel].sum() / n_real if n_real > 0 else 0.0)
        tol_l = chain * U * (float(s) + 0.625) + 8 * U * float(s)
        want = 0.625 + float(L)
        fault_l = want - float(lf[lf.abs().argmax()]) / n_fake
        assert abs(fault_l - want) > tol_l, "the loss bound cannot see a bag dropped from the sum"
        assert abs(float(loss) - want) <= tol_l, (float(loss), want, tol_l)
        extra = (4 / n_fake) if which == 0 else 0.0       # bce: σ and its complement carry absolute errors of a few u
        tol_f = 8 * U * (ff.grad.abs() + extra)
        tol_r = 8 * U * (gr.abs() + extra * sel.double() * (n_fake / max(n_real, 1)))
        _check("d_fake", d_fake, ff.grad, tol_f, {"mean over one bag more": ff.grad * nb / (nb + 1)})
        rf = {"mask ignored": torch.where(sel, gr, gr + 1.0 / max(n_real, 1))} if not bool(sel.all()) else \
            {"mean over one bag more": gr * n_real / (n_real + 1)}
        _check("d_real", d_real, gr, tol_r, rf)
    if which == 1:                                      # the kinks: subgradient 0, exactly
        assert bool((d_fake[1::7] == 0).all())
        assert bool((d_real[2::5] == 0).all())


def _grid(g, n, lo, hi):
    """values on a 2^-12 grid: differences of two of them are exact in fp32, so the kinks are decided identically"""
    return torch.randint(int(lo * 4096), int(hi * 4096), (n,), device="cuda", generator=g).float() / 4096


@pytest.mark.parametrize("nb", LOSS_BAGS)
@pytest.mark.parametrize("vkind", ["off", "mixed", "on"])
@pytest.mark.parametrize("norm,alpha,gamma,coef_gan", [(0, 0.0, 0.0, 0.004), (1, 0.3, 0.125, 0.004), (0, 0.5, 0.25, 0.0),
                                                       (1, 0.0, 0.0, 0.0)], ids=["l1", "l2-alpha-gamma", "l1-alpha-gamma-nogan",
                                                                                  "l2-nogan"])
def test_gen_loss_vs_oracle(nb, vkind, norm, alpha, gamma, coef_gan):
    """losses[0..2] += recon, gen, total; d_pred (recon part) and d_fake against float64 autograd of oracle.recon_loss and
    fake_generator_loss.  Recon differences and margins exactly 0 take torch's subgradient 0."""
    g = _gen(nb * 5 + norm + int(gamma * 8))
    pred, t = _grid(g, nb, 0, 4), _grid(g, nb, 0, 4)
    e = (torch.rand(nb, device="cuda", generator=g) < 0.4).float()
    pred[2::6] = t[2::6]                                # difference 0
    pred[3::6] = t[3::6] + gamma                        # margin 0
    e[2::6] = 1.0
    e[3::6] = 0.0
    pred[0], e[0] = t[0] + 0.5, 1.0                     # bag 0 has a nonzero gradient
    f_fake = torch.randn(nb, device="cuda", generator=g)
    vis = _mask(vkind, nb, g)
    n_vis, n_fake = float(vis.sum()), float(nb)
    pre = torch.tensor([0.5, -0.25, 0.75], device="cuda")
    losses, d_pred, d_fake = pre.clone(), _nan(nb), _nan(nb)
    st = _lib_().advmil_gen_loss(pred.data_ptr(), t.data_ptr(), e.data_ptr(), vis.data_ptr(), f_fake.data_ptr(), nb, n_vis, n_fake,
                                 coef_gan, alpha, gamma, norm, losses.data_ptr(), d_pred.data_ptr(), d_fake.data_ptr(), _stream())
    assert st == 0, _last_error()
    p64, ff = pred.double().requires_grad_(True), f_fake.double().requires_grad_(True)
    sel = vis.bool()
    if n_vis > 0:
        rec = O.recon_loss(p64[sel], t.double()[sel], e.double()[sel], alpha, gamma, "l2" if norm else "l1")
    else:
        rec = (p64 * 0).sum()
    gen = O.fake_generator_loss(ff)
    total = rec if coef_gan == 0.0 else rec + coef_gan * gen
    (rec + coef_gan * gen).backward()
    with torch.no_grad():
        m = (p64.abs() + t.double().abs() + abs(gamma) + 1) ** (1 + norm) * 2
        chain = -(-nb // 256) + 16
        s_rec = float((m * sel.double()).sum() / max(n_vis, 1))
        s_gen = float(ff.abs().sum() / n_fake)
        want = pre.double() + torch.tensor([float(rec), float(gen), float(total)], dtype=F64, device="cuda")
        tol = chain * U * (torch.tensor([s_rec, s_gen, s_rec + coef_gan * s_gen], dtype=F64, device="cuda") + pre.double().abs())
        tol = tol + 8 * U * torch.tensor([s_rec, s_gen, s_rec + coef_gan * s_gen], dtype=F64, device="cuda")
        drop = want.clone()
        drop[1] -= float(-f_fake[f_fake.abs().argmax()]) / n_fake    # a bag dropped from the gen sum
        faults = {"bag dropped from the gen sum": drop}
        if n_vis > 0:
            swapped = want.clone()
            swapped[0], swapped[1] = want[1], want[0]
            if float((swapped - want).abs()[:2].max()) > float(tol[:2].max()):
                faults["recon and gen swapped"] = swapped
        _check("losses", losses, want, tol, faults)
        base = p64.abs() + t.double().abs() + abs(gamma) + 1
        tol_p = 16 * U * base ** norm * sel.double() / max(n_vis, 1) + 8 * U * p64.grad.abs()
        pf = {"visible ignored": torch.where(sel, p64.grad, p64.grad + 1.0)} if not bool(sel.all()) else {
            "mean over one bag more": p64.grad * n_vis / (n_vis + 1)}
        _check("d_pred", d_pred, p64.grad, tol_p, pf)
        _check("d_fake", d_fake, ff.grad, 2 * U * ff.grad.abs(), {"coef_gan ignored": ff.grad - 1.0 / n_fake})
    kink = torch.zeros(nb, dtype=torch.bool, device="cuda")
    kink[2::6] = kink[3::6] = True
    assert bool((d_pred[kink & sel] == 0).all()), "recon kinks must take the subgradient 0"


# =====================================================================================================================
# 6. Adam: advmil_adam_step
# =====================================================================================================================
ADAM_N = (0, 1, 255, 256, 257, 1_000_003)


def _adam_ref(p, gr, m, v, wd_mask, lr, b1, b2, eps, wd, l1, step, gs, wd_shift=False, l1_at_zero=None):
    """float64 restatement of oracle.adam_step with the L1 subgradient and the gradient scale, with the error bound of its
    fp32 evaluation.  wd_shift / l1_at_zero plant faults (the decay mask of a neighbour; a nonzero sign at p == 0)."""
    p, gr, m, v = p.double(), gr.double(), m.double(), v.double()
    mask = wd_mask.double()
    if wd_shift:
        mask = torch.roll(mask, 1)
    sgn = torch.sign(p)
    if l1_at_zero is not None:
        sgn = torch.where(p == 0, torch.full_like(p, l1_at_zero), sgn)
    g = gr * gs + l1 * sgn + wd * mask * p
    ga = (gr * gs).abs() + abs(l1) + wd * mask * p.abs()               # Σ|terms| of the gradient
    eg = 3 * U * ga
    m1 = b1 * m + (1 - b1) * g
    v1 = b2 * v + (1 - b2) * g * g
    em = (1 - b1) * eg + 4 * U * (b1 * m.abs() + (1 - b1) * ga)
    ev = (1 - b2) * 2 * ga * eg + 4 * U * (b2 * v + (1 - b2) * ga * ga)
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    c = 1 / math.sqrt(bc2)
    denom = v1.sqrt() * c + eps
    step_size = lr / bc1
    upd = step_size * m1 / denom
    sq = v1.sqrt().clamp(min=1e-300)
    e_den = c * ev / (2 * sq) + 4 * U * denom
    e_upd = step_size * (em / denom + m1.abs() * e_den / denom ** 2) + 4 * U * upd.abs()
    p1 = p - upd
    return p1, m1, v1, e_upd + U * (p.abs() + p1.abs()), em, ev


@pytest.mark.parametrize("n", ADAM_N)
@pytest.mark.parametrize("step", [1, 10_000])
def test_adam_step_vs_float64(n, step):
    """p, m and v after one step: mixed wd_mask, l1_coef with some parameters exactly 0 (sign 0), grad_scale 0.5."""
    # the hyper-parameters as the kernel receives them (fp32)
    lr, b1, b2, eps, wd, l1, gs = (float(np.float32(a)) for a in (8e-5, 0.9, 0.999, 1e-8, 0.05, 1e-3, 0.5))
    g = _gen(n % 9973 + step)
    p = torch.randn(n, device="cuda", generator=g)
    p[::5] = 0.0
    gr = torch.randn(n, device="cuda", generator=g) * 1e-2
    gr[::5] *= 0.01                                      # at p == 0 the L1 sign decides the gradient's sign
    if step == 1:
        m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    else:
        m = torch.randn(n, device="cuda", generator=g) * 1e-2
        v = torch.rand(n, device="cuda", generator=g) * 1e-4
    wd_mask = (torch.rand(n, device="cuda", generator=g) < 0.5).to(torch.uint8)
    P, M, V = p.clone(), m.clone(), v.clone()
    st = _lib_().advmil_adam_step(P.data_ptr(), gr.data_ptr(), M.data_ptr(), V.data_ptr(), wd_mask.data_ptr(), n, lr, b1, b2, eps, wd,
                                  l1, step, gs, _stream())
    assert st == 0, _last_error()
    if n == 0:
        return
    pr, mr, vr, ep, em, ev = _adam_ref(p, gr, m, v, wd_mask, lr, b1, b2, eps, wd, l1, step, gs)
    faults = {}
    if n > 1:
        faults["decay mask of the neighbour"] = _adam_ref(p, gr, m, v, wd_mask, lr, b1, b2, eps, wd, l1, step, gs, wd_shift=True)
    faults["sign 1 at p == 0"] = _adam_ref(p, gr, m, v, wd_mask, lr, b1, b2, eps, wd, l1, step, gs, l1_at_zero=1.0)
    for i, (name, got, ref, tol) in enumerate((("p", P, pr, ep), ("m", M, mr, em), ("v", V, vr, ev))):
        _check(name, got, ref, tol, {k: f[i] for k, f in faults.items()})


# =====================================================================================================================
# 7. L1 sum: advmil_abs_sum
# =====================================================================================================================
ABS_THREADS = 8 * 1024                               # 8 CTAs of 1024 threads (one cluster)
ABS_UNROLL = 4 * ABS_THREADS * 4                     # floats covered by one unrolled iteration of every thread


@pytest.mark.parametrize("n", [1, 3, 4, 5, ABS_UNROLL - 4, ABS_UNROLL - 1, ABS_UNROLL, ABS_UNROLL + 1, ABS_UNROLL + 4,
                               3_000_001])
@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "offset1"])
def test_abs_sum_vs_float64(n, offset):
    """out[0] += Σ|p| on the float4 path (four vectors in flight, then the scalar tail) and, one float off 16 bytes, on the
    scalar path.  The last element (in the tail) and one vector at the unroll boundary are the planted faults."""
    g = _gen(n + offset)
    buf = (torch.rand(n + 4, device="cuda", generator=g) + 0.5) * torch.sign(torch.randn(n + 4, device="cuda", generator=g))
    p = buf[offset:offset + n]
    assert (p.data_ptr() % 16 == 0) == (offset == 0)
    out = torch.full((1,), 1.5, device="cuda")
    st = _lib_().advmil_abs_sum(p.data_ptr(), n, out.data_ptr(), _stream())
    assert st == 0, _last_error()
    a = p.double().abs()
    want = 1.5 + a.sum()
    per_thread = -(-n // (4 * ABS_THREADS))          # float4 loads per thread
    chain = per_thread + 4 + 10 + HEAD_CS + 2        # a thread's accumulator, the 4-term bracket, block_sum, the 8 ranks
    tol = chain * U * want
    if n <= 1 << 20:
        faults = {"last element lost": want - a[-1]}
        if n >= ABS_UNROLL:
            faults["vector at the unroll boundary lost"] = want - a[ABS_UNROLL - 4:ABS_UNROLL].sum()
    else:                                            # fp32 cannot resolve one element of millions: one unrolled pass
        faults = {"one unrolled pass of every thread lost": want - a[:ABS_UNROLL].sum()}
    _check("sum", out.double()[0], want, tol, faults)


# =====================================================================================================================
# 8. fp32 -> bf16 cast: advmil_cast_f32_to_bf16
# =====================================================================================================================
SPECIAL_BITS = [0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001, 0x7F800001,  # ±0, ±inf, NaNs
                0x00000001, 0x80000001, 0x00008000, 0x00018000, 0x007FFFFF, 0x807F8000, 0x00800000,  # subnormals, min normal
                0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000,              # half-ulp ties: to even down, to even up
                0x3F808001, 0x3F807FFF,                                      # just above / below a tie
                0x7F7F7FFF, 0x7F7F8000, 0x7F7FFFFF, 0xFF7F8000, 0xFF7FFFFF]  # largest finite that stays / rounds to inf


def _rne_bits(bits):
    """float32 bit patterns -> bf16 bit patterns, round to nearest even (torch's c10::BFloat16 rule); NaN -> -1"""
    u = bits.astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF
    nan = ((u & 0x7F800000) == 0x7F800000) & ((u & 0x7FFFFF) != 0)
    return np.where(nan, -1, r.astype(np.int64))


# one pass of the grid covers 148 * 16 CTAs * 256 threads * 8 = 4,849,664 elements: 10,000,037 takes the grid-stride loop
# three times, the last pass ending in a scalar tail
@pytest.mark.parametrize("n", [1, 7, 8, 9, 10_000_037])
def test_cast_f32_to_bf16_bit_exact(n):
    """bit-exact against round-to-nearest-even for every non-NaN input; NaN stays NaN (payload may differ)."""
    rng = np.random.default_rng(n)
    bits = rng.integers(0, 2 ** 32, size=n, dtype=np.uint64).astype(np.uint32)
    k = min(n, len(SPECIAL_BITS))
    # the short cases take the specials from the front (odd n: the back) of the list: the vector path and the scalar tail
    bits[:k] = np.array(SPECIAL_BITS[-k:] if n % 2 and n < len(SPECIAL_BITS) else SPECIAL_BITS[:k], dtype=np.uint32)
    x = torch.from_numpy(bits.view(np.float32).copy()).cuda()
    out = torch.full((n,), -1, dtype=torch.int16, device="cuda")          # 0xFFFF: a NaN, so an unwritten element fails
    st = _lib_().advmil_cast_f32_to_bf16(x.data_ptr(), n, out.data_ptr(), _stream())
    assert st == 0, _last_error()
    ref = _rne_bits(bits)
    nonnan = ref >= 0
    # the reference rule agrees with torch's conversion on the host (normal and infinite inputs: some host conversion
    # paths treat subnormal inputs as zero)
    th = torch.from_numpy(bits.view(np.float32).copy()).to(torch.bfloat16).view(torch.int16).numpy().astype(np.int64) & 0xFFFF
    normal = nonnan & (((bits >> 23) & 0xFF) != 0)
    assert np.array_equal(th[normal], ref[normal])
    trunc = (bits.astype(np.int64) >> 16) & 0xFFFF
    if n >= len(SPECIAL_BITS):
        assert not np.array_equal(trunc[nonnan], ref[nonnan]), "the data cannot tell rounding from truncation"
    got = out.cpu().numpy().astype(np.int64) & 0xFFFF
    bad = np.nonzero(got[nonnan] != ref[nonnan])[0]
    assert bad.size == 0, f"{bad.size} mismatches, first input 0x{int(bits[nonnan][bad[0]]):08x}: " \
                          f"0x{int(got[nonnan][bad[0]]):04x} != 0x{int(ref[nonnan][bad[0]]):04x}"
    gv = out.view(torch.bfloat16).float().cpu().numpy()
    assert np.isnan(gv[~nonnan]).all()


@pytest.mark.parametrize("which", ["in", "out"])
def test_cast_f32_to_bf16_refuses_misaligned(which):
    x = torch.randn(64, device="cuda")
    out = torch.empty(64, dtype=torch.bfloat16, device="cuda")
    pin = x.data_ptr() + (4 if which == "in" else 0)
    pout = out.data_ptr() + (2 if which == "out" else 0)
    st = _lib_().advmil_cast_f32_to_bf16(pin, 32, pout, _stream())
    _refuse(st, "cast_f32_to_bf16: pointers must be 16-byte aligned")

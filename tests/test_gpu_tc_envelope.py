"""GPU: the tcgen05 GEMM engine (csrc/gemm_tc.cu) over the whole envelope its dispatchers accept, in tf32, tf32x3 and bf16.

`tc_rows_kernel` (linear forward, gate, region embedding, backward data) is launched at every BLOCK_N that `pick_block_n`
selects (64 / 128 / 192 / 256), `tc_wgrad_kernel` at every BLOCK_N of `wgrad_block_n` (64 / 128 / 256; it has no
192-wide tile) and on the transposed (`wgrad_swap`) path.  Every row-count threshold of the dispatchers is run on both
sides: tf32 rows 127 / 128 (FFMA / tcgen05), weight-gradient rows 4095 / 4096 (tf32 and tf32x3), the split-tf32
weight gradient's 2048-row split cap (16384 / 16385 rows at N1 = N2 = 768, 18 tiles: 8 splits by SM count, 9 by the cap on
a 148-SM B200), and backward data's Ny * Nx <= 2^20.

References are float64 on the device, from the operands as the mode consumes them (bf16: x and W rounded to nearest even,
as `to_bf16_kernel` does; tf32 / tf32x3: the fp32 values as stored).  Bounds, per tensor and element by element relative to
the tensor's largest entry (`_rel`), are those of the existing stage tests: tf32 3e-3 (test_gpu_tc.py; 5e-3 for the gate
and the embedding, whose epilogues use tanh.approx / the tf32 LayerNorm input), tf32x3 4e-6 (test_gpu_tf32x3.py; gate
score 5e-6), bf16 6e-3 for bf16 outputs and 2e-3 for fp32 outputs (test_gpu_bf16.py; the packed gate activations 8e-3),
and 1e-5 wherever the FFMA engine runs.

The tf32x3 bound is 4e-6 per 1024 chained K steps (`_tol`).  The tensor core accumulates with truncation, so the
split-tf32 error grows linearly with the number of MMAs chained into one TMEM accumulator: measured on a B200, about
2.6e-6 per 1024 of K (5e-6 at K = 2048, 1e-5 at backward data's Ny = 4096, and 4.4-5e-6 for weight-gradient splits of
2048 rows), so 4e-6, which the existing tests meet at K <= 1024, does not hold across the envelope.  The weight gradient's
chain is its rows per split (`_x3_wgrad_chain`, the dispatcher's rule).  The self-check shows that the scaled bound still
sees a lost K block and a shifted row at every such shape.

Every case first shows on the host that its bound is able to fail: the float64 reference is rebuilt once without the last
K block's contribution and once with one 128-row output tile shifted down by one row, and both faulty references must
violate the bound at that shape (`_sensitive`)."""
import numpy as np
import pytest
import torch

import advmil_b200
from advmil_b200 import _lib, ops
from oracle import advmil_oracle as O
from tests.util import assert_close, build_G, g_masks, grad_floor, to_dev_masks

pytestmark = pytest.mark.gpu

MODES = ("tf32", "tf32x3", "bf16")
PREC = {"tf32": ops.TF32, "tf32x3": ops.TF32X3, "bf16": ops.BF16}
KBLK = {"tf32": 32, "tf32x3": 32, "bf16": 64}          # TcElem<T>::KBLK: the K block of a ring stage
TOL_ACT = {"tf32": 3e-3, "tf32x3": 4e-6, "bf16": 6e-3}  # outputs in the mode's element type (y, dX, y_pre)
TOL_F32 = {"tf32": 3e-3, "tf32x3": 4e-6, "bf16": 2e-3}  # fp32 outputs (dW, the region embedding)
TOL_GATE_S = {"tf32": 5e-3, "tf32x3": 5e-6, "bf16": 6e-3}
TOL_GATE_AB = {"tf32": 5e-3, "tf32x3": 4e-6, "bf16": 8e-3}
TOL_FFMA = 1e-5
TILE_M = 128
SITE_USER = 100                                          # linear_fwd keys its dropout sites at SITE_USER + site

# pick_block_n (gemm_tc.cu): 192 when N % 192 == 0 and N % 256 != 0, else 256 when N % 256 == 0, else 128 when
# N % 128 == 0, else 64 for N == 64
BLOCK_N = {64: 64,      # N == 64
           128: 128,    # 128 % 192 != 0, 128 % 256 != 0, 128 % 128 == 0
           192: 192,    # 192 % 192 == 0, 192 % 256 != 0
           256: 256,    # 256 % 192 != 0, 256 % 256 == 0
           384: 192,    # 384 % 192 == 0, 384 % 256 != 0
           512: 256,    # 512 % 192 != 0, 512 % 256 == 0
           640: 128,    # 640 % 192 != 0, 640 % 256 != 0, 640 % 128 == 0
           768: 256}    # 768 % 192 == 0 but 768 % 256 == 0


def _block_n(N):
    if N % 192 == 0 and N % 256 != 0:
        return 192
    if N % 256 == 0:
        return 256
    if N % 128 == 0:
        return 128
    return 64 if N == 64 else 0


def _wgrad_block_n(N2):
    if N2 % 256 == 0:
        return 256
    if N2 % 128 == 0:
        return 128
    return 64 if N2 == 64 else 0


def _wgrad_swap(N1, N2):
    return _wgrad_block_n(N2) == 128 and N1 % 256 == 0 and N2 % 128 == 0


def _tc_rows(mode, rows):
    """rows_ok: the bf16 mode runs any row count on tcgen05, the fp32-element modes from one 128-row tile up"""
    return rows >= 1 if mode == "bf16" else rows >= TILE_M


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _op(t, mode):
    """What the mode multiplies, in float64: bf16 (round to nearest even) in the bf16 mode, the fp32 values otherwise."""
    return t.to(torch.bfloat16).double() if mode == "bf16" else t.double()


def _rel(a, b):
    """largest element-wise error relative to the reference tensor's largest entry"""
    return float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))


def _shift_tile(t):
    """the last 128-row tile of t shifted down by one row (its first row zero): a wrong row in the epilogue's store"""
    t = t.clone()
    r0 = (t.shape[0] - 1) // TILE_M * TILE_M
    t[r0 + 1:] = t[r0:-1].clone()
    t[r0] = 0
    return t


def _sensitive(name, tol, ref, lost_k, shifted):
    """the bound must see a lost K block and a one-row shift of a tile at this shape"""
    assert _rel(lost_k, ref) > tol, f"{name}: bound {tol:.1e} cannot see a lost K block ({_rel(lost_k, ref):.2e})"
    assert _rel(shifted, ref) > tol, f"{name}: bound {tol:.1e} cannot see a shifted row ({_rel(shifted, ref):.2e})"


def _check(name, out, ref, tol, lost_k, shifted):
    _sensitive(name, tol, ref, lost_k, shifted)
    err = _rel(out, ref)
    assert err < tol, f"{name}: {err:.3e} >= {tol:.1e}"


def _tol(mode, table, kchain):
    """the mode's bound for an output whose accumulator chains kchain K steps (see the module docstring)"""
    return table[mode] * (max(1.0, kchain / 1024) if mode == "tf32x3" else 1.0)


def _cdiv(a, b):
    return (a + b - 1) // b


def _x3_wgrad_chain(rows, N1, N2):
    """rows per split of the split-tf32 weight gradient: wgrad_splits (gemm_tc.cu) with the 2048-row cap"""
    if _wgrad_swap(N1, N2):
        N1, N2 = N2, N1
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = _cdiv(N1, TILE_M) * (N2 // _wgrad_block_n(N2))
    s = max(min(max(1, sms // tiles), max(1, rows // 1024)), _cdiv(rows, 2048))
    return _cdiv(_cdiv(rows, s), KBLK["tf32x3"]) * KBLK["tf32x3"]


def _last_block(K, kb):
    """start of the last K block (the partial one when K is not a multiple of kb)"""
    return (K - 1) // kb * kb


def _randn(g, *shape, scale=1.0):
    return torch.randn(*shape, device="cuda", generator=g) * scale


# =====================================================================================================================
# linear forward: advmil_linear_fwd
# =====================================================================================================================
NS = (64, 128, 192, 256, 384, 512, 640, 768)
ROWS_FWD = {"bf16": (1, 17, 127, 128, 129, 1000), "tf32": (127, 128, 129, 1000), "tf32x3": (127, 128, 129, 1000)}


def _k_list(mode):
    kb = KBLK[mode]
    # 1 block, 3 blocks (fewer than the ring's stages), many blocks: 1024 and 2048 (multiples of every stage count that
    # divides a power of two) and 37 blocks, a prime count, so the ring's phase is not back at zero when K ends
    return (kb, 3 * kb, 1024, 37 * kb, 2048)


def _fwd_cases():
    out = []
    for mode in MODES:
        ks, rs = _k_list(mode), ROWS_FWD[mode]
        i = 0
        for ni, N in enumerate(NS):
            assert _block_n(N) == BLOCK_N[N]
            for j in range(3):
                K, rows = ks[(ni + 2 * j) % len(ks)], rs[i % len(rs)]
                act, bias = i % 2, (i // 2) % 2 == 0      # three consecutive cases per N cover both values of each
                i += 1
                eng = f"bn{BLOCK_N[N]}" if _tc_rows(mode, rows) else "ffma"
                out.append(pytest.param(mode, rows, K, N, act, bias,
                                        id=f"{mode}-{eng}-rows{rows}-K{K}-N{N}-act{act}-{'bias' if bias else 'nobias'}"))
    return out


def _linear_ref(x, W, b, act, mode, kmax=None):
    xo, Wo = _op(x, mode), _op(W, mode)
    if kmax is not None:
        xo, Wo = xo[:, :kmax], Wo[:, :kmax]
    y = xo @ Wo.t()
    if b is not None:
        y = y + b.double()
    return torch.relu(y) if act else y


def _fwd_operands(rows, K, N, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = _randn(g, rows, K)
    W = _randn(g, N, K, scale=K ** -0.5)
    b = _randn(g, N, scale=0.5)
    return x, W, b


@pytest.mark.parametrize("mode,rows,K,N,act,bias", _fwd_cases())
def test_linear_fwd(mode, rows, K, N, act, bias):
    x, W, b = _fwd_operands(rows, K, N, rows * 7 + K + N)
    b = b if bias else None
    y = ops.linear_forward(x, W, b, act=act, precision=PREC[mode])
    assert y.dtype == (torch.bfloat16 if mode == "bf16" else torch.float32)
    ref = _linear_ref(x, W, b, act, mode)
    tol = _tol(mode, TOL_ACT, K) if _tc_rows(mode, rows) else TOL_FFMA
    _check("y", y, ref, tol, _linear_ref(x, W, b, act, mode, _last_block(K, KBLK[mode])), _shift_tile(ref))


@pytest.mark.parametrize("mode", MODES)
def test_linear_fwd_tiles_wrap_in_persistent_ctas(mode):
    """N = 64 and one K block: 3 * SMs * 128 + 37 rows give every persistent CTA at least three tiles, so the smem ring
    and the two TMEM accumulators wrap between tiles while each tile is a single stage; the last tile is partial."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    rows, K, N = 3 * sms * TILE_M + 37, KBLK[mode], 64
    x, W, b = _fwd_operands(rows, K, N, 99)
    y = ops.linear_forward(x, W, b, act=1, precision=PREC[mode])
    ref = _linear_ref(x, W, b, 1, mode)
    _check("y", y, ref, TOL_ACT[mode], _linear_ref(x, W, b, 1, mode, 0), _shift_tile(ref))


def _user_mask(seed, site, p, rows, N):
    lib = _lib.load()
    m = torch.empty(rows, N, dtype=torch.uint8, device="cuda")
    _lib.check(lib.advmil_dropout_mask(seed, SITE_USER + site, p, rows, N, m.data_ptr(), _stream()), "advmil_dropout_mask")
    return m


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("rows,K,N,site", [(129, 96, 64, 3), (1001, 1024, 384, 7), (257, 192, 640, 0)])
def test_linear_fwd_dropout_seeded_injected_and_eval(mode, rows, K, N, site):
    """train = 1, p = 0.25: the seeded run equals the reference built with advmil_dropout_mask's bits for site
    SITE_USER + site (each draw serves two columns: odd rows and the 64-wide block included); injecting that mask
    reproduces the seeded run bit for bit; train = 0 applies no dropout."""
    K = K if K % KBLK[mode] == 0 else KBLK[mode] * 3
    p, seed = 0.25, 1234 + rows
    x, W, b = _fwd_operands(rows, K, N, rows + site)
    P = PREC[mode]
    y = ops.linear_forward(x, W, b, act=1, p_drop=p, seed=seed, site=site, train=True, precision=P)
    mask = _user_mask(seed, site, p, rows, N)
    frac = float(mask.float().mean())
    assert 0.7 < frac < 0.8, frac
    keep = mask.double() / (1 - p)
    ref = _linear_ref(x, W, b, 1, mode) * keep
    lost = _linear_ref(x, W, b, 1, mode, _last_block(K, KBLK[mode])) * keep
    _check("y train", y, ref, _tol(mode, TOL_ACT, K), lost, _shift_tile(ref))
    y_inj = ops.linear_forward(x, W, b, act=1, p_drop=p, mask=mask, seed=seed, site=site, train=True, precision=P)
    assert torch.equal(y_inj, y)
    y_eval = ops.linear_forward(x, W, b, act=1, p_drop=p, seed=seed, site=site, train=False, precision=P)
    ref0 = _linear_ref(x, W, b, 1, mode)
    _check("y eval", y_eval, ref0, _tol(mode, TOL_ACT, K), _linear_ref(x, W, b, 1, mode, _last_block(K, KBLK[mode])), _shift_tile(ref0))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("K,N", [(1024, 320), (100, 384)])
def test_linear_fwd_shapes_the_engine_refuses(mode, K, N):
    """N = 320 (no tile width divides it) and K = 100 (no K block divides it): bf16 has no other engine and must refuse;
    the fp32-element modes fall back to the FFMA engine."""
    rows = 300
    x, W, b = _fwd_operands(rows, K, N, K + N)
    if mode == "bf16":
        with pytest.raises(_lib.AdvmilError, match="bf16 mode runs only on the tcgen05 engine"):
            ops.linear_forward(x, W, b, act=1, precision=PREC[mode])
        return
    y = ops.linear_forward(x, W, b, act=1, precision=PREC[mode])
    ref = _linear_ref(x, W, b, 1, mode)
    _check("y", y, ref, TOL_FFMA, _linear_ref(x, W, b, 1, mode, _last_block(K, KBLK[mode])), _shift_tile(ref))


# =====================================================================================================================
# gated attention score: advmil_gated_score_fwd
# =====================================================================================================================
def _gate_cases():
    out = []
    for mode in MODES:
        rows_list = (1, 129, 1000) if mode == "bf16" else (129, 1000)
        i = 0
        for D in (128, 256, 384, 512):
            for L in (KBLK[mode], 384):
                rows, train = rows_list[i % len(rows_list)], i % 2 == 1
                i += 1
                out.append(pytest.param(mode, rows, L, D, train, id=f"{mode}-rows{rows}-L{L}-D{D}-{'train' if train else 'eval'}"))
    return out


def _gate_ref(v, Wa, ba, Wb, bb, wc, bc, mode, ma=None, mb=None, p=0.25, lmax=None):
    vo, Wao, Wbo = _op(v, mode), _op(Wa, mode), _op(Wb, mode)
    if lmax is not None:
        vo, Wao, Wbo = vo[:, :lmax], Wao[:, :lmax], Wbo[:, :lmax]
    a = torch.tanh(vo @ Wao.t() + ba.double())
    b = torch.sigmoid(vo @ Wbo.t() + bb.double())
    if ma is None:
        s = (a * b) @ wc.double() + bc.double()
        return s, a, b
    ka, kb = ma.double(), mb.double()
    s = ((a * ka / (1 - p)) * (b * kb / (1 - p))) @ wc.double() + bc.double()
    # the stored sigmoid carries the pair's joint keep bit in its sign; both stored values are the undropped activations
    return s, a, torch.where((ka * kb) > 0, b, -b)


@pytest.mark.parametrize("mode,rows,L,D,train", _gate_cases())
def test_gated_score(mode, rows, L, D, train):
    """s and both halves of the packed `ab` (tanh_j at 128 (j / 64) + j % 64, sigmoid_j 64 columns further).

    Train mode with injected mask_a / mask_b: the pair (tanh_j, sigmoid_j) contributes to s iff BOTH masks keep it,
    scaled by 1 / keep^2, exactly as the reference's two independent dropouts act through the product a_j b_j.  The
    in-kernel generator instead draws that joint keep bit directly (Bernoulli((1-p)^2) from 8 bits per pair, Drop::pair_gate)
    and advmil_dropout_mask materialises it as the tanh site's mask with an all-ones sigmoid mask -- so injecting the
    pair (joint, ones) reproduces a seeded run, and injecting two independent masks is the reference's semantics.  In
    both cases `ab` stores the undropped tanh and sigmoid, the sigmoid's sign set to the joint keep bit (header,
    AdvmilGenActs.ab); the dropout itself acts through s and, in the backward, through that sign."""
    g = torch.Generator(device="cuda").manual_seed(rows + L + D)
    v = _randn(g, rows, L)
    Wa, Wb = _randn(g, D, L, scale=L ** -0.5), _randn(g, D, L, scale=L ** -0.5)
    ba, bb, wc = _randn(g, D, scale=0.1), _randn(g, D, scale=0.1), _randn(g, D, scale=D ** -0.5)
    bc = _randn(g, 1, scale=0.1)
    p = 0.25
    ma = mb = None
    if train:
        ma = (torch.rand(rows, D, device="cuda", generator=g) < 0.75).to(torch.uint8)
        mb = (torch.rand(rows, D, device="cuda", generator=g) < 0.75).to(torch.uint8)
    s, ab = ops.gated_score_forward(v, Wa, ba, Wb, bb, wc, bc, p_drop=p if train else 0.0, mask_a=ma, mask_b=mb,
                                    seed=5, train=train, precision=PREC[mode])
    ref_s, ref_a, ref_b = _gate_ref(v, Wa, ba, Wb, bb, wc, bc, mode, ma, mb, p)
    lost_s, lost_a, lost_b = _gate_ref(v, Wa, ba, Wb, bb, wc, bc, mode, ma, mb, p, _last_block(L, KBLK[mode]))
    j = torch.arange(D, device="cuda")
    ca = 128 * (j // 64) + j % 64
    assert ab.shape[1] == _lib.load().advmil_gate_packed_width(D)
    tc = _tc_rows(mode, rows)
    ts, tab = (TOL_GATE_S[mode], TOL_GATE_AB[mode]) if tc else (TOL_FFMA, TOL_FFMA)
    _check("s", s, ref_s, ts, lost_s, _shift_tile(ref_s))
    _check("ab tanh", ab[:, ca], ref_a, tab, lost_a, _shift_tile(ref_a))
    _check("ab sigmoid", ab[:, ca + 64], ref_b, tab, lost_b, _shift_tile(ref_b))
    if train:
        assert torch.equal(ab[:, ca + 64] > 0, (ma & mb) > 0)


@pytest.mark.parametrize("D", [64, 192])
def test_gated_score_bf16_refuses_widths_without_a_whole_gate_block(D):
    rows, L = 256, 128
    g = torch.Generator(device="cuda").manual_seed(D)
    v = _randn(g, rows, L)
    Wa, Wb = _randn(g, D, L, scale=L ** -0.5), _randn(g, D, L, scale=L ** -0.5)
    ba, bb, wc, bc = _randn(g, D), _randn(g, D), _randn(g, D), _randn(g, 1)
    with pytest.raises(_lib.AdvmilError, match="gated_score_fwd: .*bf16 mode runs only on the tcgen05 engine"):
        ops.gated_score_forward(v, Wa, ba, Wb, bb, wc, bc, precision=ops.BF16)


# =====================================================================================================================
# backward: advmil_linear_bwd through the library handle (accumulate settable)
# =====================================================================================================================
def _ptr(t):
    return None if t is None else t.data_ptr()


def _linear_bwd(dY, X, W, mode, dX=None, dW=None, db=None, accumulate=0):
    lib = _lib.load()
    rows, N = dY.shape
    K = W.shape[1]
    dY = ops.cast_bf16(dY) if mode == "bf16" else dY
    X = None if X is None else (ops.cast_bf16(X) if mode == "bf16" else X)
    ws = torch.empty(lib.advmil_linear_bwd_workspace_bytes(rows, K, N), dtype=torch.uint8, device=dY.device)
    _lib.check(lib.advmil_linear_bwd(dY.data_ptr(), _ptr(X), W.data_ptr(), rows, K, N, _ptr(dX), _ptr(dW), _ptr(db),
                                     accumulate, PREC[mode], ws.data_ptr(), ws.numel(), _stream()), "advmil_linear_bwd")


def _dx_cases():
    out = []
    for mode in MODES:
        kb = KBLK[mode]
        i = 0
        for Nx in (64, 128, 384, 256, 640, 512):           # BLOCK_N 64, 128, 192, 256, 128, 256
            for Ny in (kb, 384, 1024):
                rows = (1000, 129, 4099)[i % 3] if mode != "bf16" else (1, 129, 1000)[i % 3]
                i += 1
                out.append(pytest.param(mode, rows, Ny, Nx, id=f"{mode}-bn{BLOCK_N[Nx]}-rows{rows}-Ny{Ny}-Nx{Nx}"))
        # Ny * Nx == 2^20: still tcgen05; one K block more: FFMA in the fp32-element modes, a refusal in bf16
        out.append(pytest.param(mode, 300, 4096, 256, id=f"{mode}-bn256-rows300-Ny4096-Nx256-at-2^20"))
        out.append(pytest.param(mode, 300, 4096 + kb, 256, id=f"{mode}-{'refused' if mode == 'bf16' else 'ffma'}-rows300-Ny{4096 + kb}-Nx256-above-2^20"))
    return out


@pytest.mark.parametrize("mode,rows,Ny,Nx", _dx_cases())
def test_linear_bwd_data(mode, rows, Ny, Nx):
    """dX [rows, Nx] = dY [rows, Ny] W [Ny, Nx]: the backward-data pass runs tc_rows_kernel over W^T (Ny is its K)."""
    g = torch.Generator(device="cuda").manual_seed(rows + Ny + Nx)
    dY = _randn(g, rows, Ny)
    W = _randn(g, Ny, Nx, scale=Ny ** -0.5)
    dX = torch.empty(rows, Nx, dtype=torch.bfloat16 if mode == "bf16" else torch.float32, device="cuda")
    tc = _tc_rows(mode, rows) and Ny * Nx <= 1 << 20
    if mode == "bf16" and not tc:
        with pytest.raises(_lib.AdvmilError, match="bwd_data: .*bf16 mode runs only on the tcgen05 engine"):
            _linear_bwd(dY, None, W, mode, dX=dX)
        return
    _linear_bwd(dY, None, W, mode, dX=dX)
    ref = _op(dY, mode) @ _op(W, mode)
    k0 = _last_block(Ny, KBLK[mode])
    _check("dX", dX, ref, _tol(mode, TOL_ACT, Ny) if tc else TOL_FFMA, _op(dY, mode)[:, :k0] @ _op(W, mode)[:k0], _shift_tile(ref))


ROWS_DW = {"tf32": (4095, 4096, 4097), "bf16": (1, 63, 64, 65, 1000), "tf32x3": (4095, 4096, 4097)}


def _dw_engine(mode, rows, N1, N2):
    if mode != "bf16" and rows < 4096:
        return "ffma"
    if _wgrad_swap(N1, N2):
        return "swap-bn256"
    return f"bn{_wgrad_block_n(N2)}"


def _dw_cases():
    out = []
    for mode in MODES:
        rs = ROWS_DW[mode]
        i = 0
        for N2 in (64, 128, 256, 384, 768):                 # wgrad BLOCK_N 64, 128, 256, 128, 256
            for N1 in (64, 192, 768):                       # one partial 128-row M tile, a full and a partial one, six full
                if (N1, N2) == (768, 384):
                    continue                                # the transposed path: below, on both sides of the threshold
                rows = rs[i % len(rs)]
                i += 1
                out.append(pytest.param(mode, rows, N1, N2, id=f"{mode}-{_dw_engine(mode, rows, N1, N2)}-rows{rows}-N1{N1}-N2{N2}"))
        for rows in ((1000, 65) if mode == "bf16" else (4095, 4096)):
            out.append(pytest.param(mode, rows, 768, 384, id=f"{mode}-{_dw_engine(mode, rows, 768, 384)}-rows{rows}-N1768-N2384"))
    # split-tf32: 16384 rows in 8 splits of 2048 (SM count and cap agree), 16385 rows in 9 (the 2048-row cap decides)
    for rows in (16384, 16385):
        out.append(pytest.param("tf32x3", rows, 768, 768, id=f"tf32x3-bn256-rows{rows}-N1768-N2768-split-cap"))
    return out


def _dw_ref(dY, X, mode, rmax=None):
    d, x = _op(dY, mode), _op(X, mode)
    if rmax is not None:
        d, x = d[:rmax], x[:rmax]
    return d.t() @ x


@pytest.mark.parametrize("mode,rows,N1,N2", _dw_cases())
def test_linear_bwd_weight_and_bias(mode, rows, N1, N2):
    """dW [N1, N2] = dY^T X (tc_wgrad_kernel + split-K reduce: the row count is its K), db = colsum(dY)."""
    g = torch.Generator(device="cuda").manual_seed(rows + N1 * 3 + N2)
    dY = _randn(g, rows, N1)
    X = _randn(g, rows, N2)
    W = torch.empty(N1, N2, device="cuda")
    dW = torch.empty(N1, N2, device="cuda")
    db = torch.empty(N1, device="cuda")
    _linear_bwd(dY, X, W, mode, dW=dW, db=db)
    ref = _dw_ref(dY, X, mode)
    tc = mode == "bf16" or rows >= 4096
    tol = _tol(mode, TOL_F32, _x3_wgrad_chain(rows, N1, N2)) if tc else TOL_FFMA
    _check("dW", dW, ref, tol, _dw_ref(dY, X, mode, _last_block(rows, KBLK[mode])), _shift_tile(ref))
    assert _rel(db, _op(dY, mode).sum(0)) < (1e-4 if mode == "bf16" else 1e-5)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("N1,N2", [(192, 256), (768, 384)], ids=["normal", "swapped"])
def test_linear_bwd_accumulates_into_dw_and_db(mode, N1, N2):
    """accumulate = 1: dW and db come back as prefill + gradient, on the normal and on the transposed wgrad path."""
    assert _wgrad_swap(N1, N2) == (N1 == 768)
    rows = 1000 if mode == "bf16" else 4096
    g = torch.Generator(device="cuda").manual_seed(N1 + N2)
    dY, X = _randn(g, rows, N1), _randn(g, rows, N2)
    W = torch.empty(N1, N2, device="cuda")
    pre_w, pre_b = _randn(g, N1, N2, scale=8.0), _randn(g, N1, scale=8.0)
    dW, db = pre_w.clone(), pre_b.clone()
    _linear_bwd(dY, X, W, mode, dW=dW, db=db, accumulate=1)
    ref = pre_w.double() + _dw_ref(dY, X, mode)
    lost = pre_w.double() + _dw_ref(dY, X, mode, _last_block(rows, KBLK[mode]))
    tol = _tol(mode, TOL_F32, _x3_wgrad_chain(rows, N1, N2))
    _check("dW (accumulate)", dW, ref, tol, lost, _shift_tile(ref))
    assert _rel(db, pre_b.double() + _op(dY, mode).sum(0)) < (1e-4 if mode == "bf16" else 1e-5)
    assert _rel(_dw_ref(dY, X, mode), ref) > tol              # the bound sees a prefill that was overwritten


# =====================================================================================================================
# region embedding (ksize 1, d = 128): ops.disc_embed_forward / disc_embed_backward
# =====================================================================================================================
EMB_KEYS = ("conv.weight", "conv.bias", "norm.weight", "norm.bias")
EMB_LENGTHS = {
    "16": [16],                         # one region, bf16 only (the fp32-element modes start at one tile)
    "128": [16, 112],                   # one full tile, two bags
    "144": [144],                       # 128 + 16: one region in a second, partial tile
    "ragged144": [48, 96],              # the tile boundary at row 128 falls inside the second bag's region group
    "1600": [400, 16, 1184],            # 13 tiles, the last one partial, bag boundaries inside tiles
}


def _emb_cases():
    out = []
    for mode in MODES:
        for name, lengths in EMB_LENGTHS.items():
            if name == "16" and mode != "bf16":
                continue
            acc = name in ("144", "1600")
            out.append(pytest.param(mode, lengths, acc, id=f"{mode}-rows{name}-{'accumulate' if acc else 'overwrite'}"))
    return out


def _emb_chain(y, p64, R, d, d_emb=None):
    e = torch.relu(torch.nn.functional.layer_norm(y, (d,), p64["norm.weight"], p64["norm.bias"], 1e-5))
    return e.reshape(R, 16, d).mean(1)


@pytest.mark.parametrize("mode,lengths,accumulate", _emb_cases())
def test_region_embedding_fwd_bwd(mode, lengths, accumulate):
    """emb and y_pre against float64 LayerNorm -> ReLU -> 16-row mean; dWc, dbc, dgamma, dbeta against float64 autograd
    of the same chain, taken at the kernel's own saved y_pre (the ReLU derivative jumps; see test_gpu_disc_conv3.py).
    In bf16 the activation gradient d_y is stored in bf16 before the weight gradient, as the mode does."""
    C, d = 1024, 128
    rows, R = sum(lengths), sum(lengths) // 16
    sd = O.synth_state_dict(O.D_SHAPES(C, d), 41)
    p = {k: sd["net_pair_one.embedding." + k] for k in EMB_KEYS}
    x = O.synth_bag(rows, 42, C)
    d_emb = torch.randn(R, d, generator=torch.Generator().manual_seed(43)).cuda()
    cfg = ops.DiscConfig(C=C, d=d, t1=1, t2=d, ksize=1)
    params = [p[k].cuda() for k in EMB_KEYS] + [None] * 20
    bags = ops.PackedBags(x.cuda(), lengths)
    acts = ops.disc_embed_forward(cfg, params, bags, PREC[mode], save=True)
    pre = [torch.randn(t.shape, generator=torch.Generator().manual_seed(44 + i)).cuda() for i, t in enumerate(params[:4])]
    grads = [t.clone() if accumulate else torch.empty_like(t) for t in pre] + [None] * 20
    ops.disc_embed_backward(cfg, params, bags, acts, d_emb, grads, accumulate=accumulate)

    xg = x.cuda()
    p64 = {k: v.cuda().double() for k, v in p.items()}
    Wc = p64["conv.weight"].reshape(d, C)
    xo, Wo = _op(xg, mode), _op(Wc, mode)
    y_ref = xo @ Wo.t() + p64["conv.bias"]
    k0 = _last_block(C, KBLK[mode])
    y_lost = xo[:, :k0] @ Wo[:, :k0].t() + p64["conv.bias"]
    y_shift = _shift_tile(y_ref)
    tc = _tc_rows(mode, rows)
    _check("y_pre", acts["y_pre"], y_ref, TOL_ACT[mode] if tc else TOL_FFMA, y_lost, y_shift)
    emb_ref = _emb_chain(y_ref, p64, R, d)
    # tf32: test_gpu_tc.py's 5e-3; tf32x3: test_gpu_tf32x3.py's rtol 1e-5 on |e| plus 1e-5 of the largest entry
    t_emb = {"tf32": 5e-3, "tf32x3": 2e-5, "bf16": 2e-3}[mode] if tc else TOL_FFMA
    _check("emb", acts["emb"], emb_ref, t_emb, _emb_chain(y_lost, p64, R, d), _emb_chain(y_shift, p64, R, d))

    y = acts["y_pre"].double().requires_grad_(True)
    g64 = {k: v.clone().requires_grad_(True) for k, v in p64.items() if k.startswith("norm")}
    (_emb_chain(y, {**p64, **g64}, R, d) * d_emb.double()).sum().backward()
    dy = y.grad.to(torch.bfloat16).double() if mode == "bf16" else y.grad
    base = [t.double() if accumulate else torch.zeros_like(t, dtype=torch.float64) for t in pre]
    dWc_ref = base[0] + (dy.t() @ xo).reshape(base[0].shape)
    dWc_lost = base[0] + (dy[:_last_block(rows, KBLK[mode])].t() @ xo[:_last_block(rows, KBLK[mode])]).reshape(base[0].shape)
    tc_w = mode == "bf16" or rows >= 4096
    _check("dWc", grads[0], dWc_ref, TOL_F32[mode] if tc_w else TOL_FFMA, dWc_lost,
           _shift_tile(dWc_ref.reshape(d, C)).reshape(base[0].shape))
    floor = grad_floor([t.cpu() for t in (y.grad.sum(0), g64["norm.weight"].grad, g64["norm.bias"].grad)])
    for name, got, want in (("dbc", grads[1], base[1] + y.grad.sum(0)),
                            ("dgamma", grads[2], base[2] + g64["norm.weight"].grad),
                            ("dbeta", grads[3], base[3] + g64["norm.bias"].grad)):
        assert_close(got.cpu(), want.cpu(), 1e-5, name, atol=8 * floor)


# =====================================================================================================================
# generator parity at non-default widths (the module tests run only C, h, o = 1024, 384, 384 in these modes)
# =====================================================================================================================
GEN_DIMS = [(512, 256, 256), (768, 512, 512), (1024, 128, 128), (1024, 64, 64), (1024, 192, 192)]
ZERO_GRAD = ("pool.fc2.bias", "attention_c.bias")


def _gen_cases():
    out = []
    for mode in MODES:
        for dims in GEN_DIMS:
            for train in (False, True):
                refused = mode == "bf16" and dims[1] % 128 != 0
                if refused and train:
                    continue
                out.append(pytest.param(mode, dims, train, id=f"{mode}-C{dims[0]}-h{dims[1]}-o{dims[2]}-"
                                        + ("refused" if refused else "train" if train else "eval")))
    return out


@pytest.mark.parametrize("mode,dims,train", _gen_cases())
def test_generator_parity_at_other_widths(mode, dims, train):
    """Forward and all 14 gradients against the oracle.  Covers the backward-data extras (pooling term w dz, mean term,
    ReLU / dropout mask with 1 / keep folded into W^T, column sums) at BLOCK_N 64, 128, 256, K1 at every block width,
    dW1 with a 64-row M tile, and the gate on its FFMA fallback (h = 64, 192) beside tcgen05 neighbours.  tf32x3: the
    fp32 tolerance of test_x3_mode_generator_and_discriminator_vs_oracle; tf32: 2e-2; bf16: the bf16-storage oracle at
    the bound of test_bf16_mode_generator_and_discriminator_vs_oracle, and widths without a whole gate block refused.

    The first layer's gradients (attention_net.0) are compared with the float64 chain taken at the kernel's own ReLU
    branch, as test_gpu_disc_conv3.py does for the embedding: of the 10^5-10^6 pre-activations a few lie within the mode's
    rounding of zero (measured: one in tf32x3 at 768 x 512, several in tf32), and where the device and the CPU oracle take
    different sides, a whole row of dW1 moves by dh x (up to 5e-2 of the tensor's largest entry).  The oracle's dL/dh is
    routed through the ReLU mask of the same K1 evaluated by advmil_linear_fwd in the mode."""
    C, h, o = dims
    N = 1000
    sd = O.synth_state_dict(O.G_SHAPES(C, h, o), 60 + h)
    G = build_G(dims)
    G.load_state_dict({k: v.clone() for k, v in sd.items()})
    x = O.synth_bag(N, 61, C)
    noise = torch.tensor(np.random.default_rng(62).uniform(size=(1, o // 2)), dtype=torch.float32)
    gm = g_masks(N, h, o, 63) if train else None
    G.train(train)
    if train:
        G._inject_masks = to_dev_masks(gm)
    advmil_b200.set_precision(mode)
    try:
        bags = ops.PackedBags.from_single(x.cuda())
        if mode == "bf16" and h % 128 != 0:
            with pytest.raises(_lib.AdvmilError, match="gated_score_fwd: .*bf16 mode runs only on the tcgen05 engine"):
                G.forward_packed(bags, noise=[None, noise.cuda()])
            return
        pred = G.forward_packed(bags, noise=[None, noise.cuda()])
        pred.sum().backward()
    finally:
        advmil_b200.set_precision("fp32")
    rG = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    if mode == "bf16":
        with O.bf16_storage():
            og = O.generator_forward(rG, x, [None, noise], (0, 1), gm)
            og["pred"].sum().backward()
    else:
        og = O.generator_forward(rG, x, [None, noise], (0, 1), gm)
        og["h"].retain_grad()
        og["pred"].sum().backward()
        W1, b1 = "backbone.attention_net.0.weight", "backbone.attention_net.0.bias"
        pre = ops.linear_forward(x.cuda(), sd[W1].cuda(), sd[b1].cuda(), act=0, precision=PREC[mode]).cpu().double()
        dh = og["h"].grad.double() * (gm["h"].double() / 0.75 if train else 1.0)
        d_pre = dh * (pre > 0)
        first = {W1: d_pre.t() @ x.double(), b1: d_pre.sum(0)}
        assert 0 < float((pre > 0).double().mean()) < 1
    rtol = {"tf32x3": 1e-5, "tf32": 2e-2, "bf16": 1e-2}[mode]
    assert_close(pred.detach().cpu(), og["pred"].detach(), rtol, "pred")
    gmax = max(float(v.grad.abs().max()) for v in rG.values() if v.grad is not None)
    floor = 8 * grad_floor([v.grad for v in rG.values()]) if mode == "tf32x3" else 2e-5 * gmax
    gtol = 2e-5 if mode == "tf32x3" else rtol
    n = 0
    for k, p in G.named_parameters():
        if rG[k].grad is None or k.endswith(ZERO_GRAD):
            continue
        want = first[k] if mode != "bf16" and k in first else rG[k].grad
        assert_close(p.grad.cpu(), want, gtol, "grad " + k, atol=floor)
        n += 1
    assert n == 13            # the 14 parameter tensors minus attention_c.bias (mathematically zero: softmax shift)


# =====================================================================================================================
# a second device in the same process
# =====================================================================================================================
@pytest.mark.parametrize("mode", ["tf32", "bf16"])
def test_engine_on_a_second_device_in_one_process(mode):
    """linear_forward and linear_backward (dW at 4096 rows: tcgen05 in tf32 too) on cuda:0, then cuda:1, then cuda:0:
    the kernels' large dynamic shared-memory opt-in has to hold on every device the process uses."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rows, K, N = 4096, 384, 256
    for dev in (0, 1, 0):
        with torch.cuda.device(dev):
            g = torch.Generator(device=f"cuda:{dev}").manual_seed(dev + 1)
            x = torch.randn(rows, K, device=f"cuda:{dev}", generator=g)
            W = torch.randn(N, K, device=f"cuda:{dev}", generator=g) * K ** -0.5
            b = torch.randn(N, device=f"cuda:{dev}", generator=g)
            dY = torch.randn(rows, N, device=f"cuda:{dev}", generator=g)
            y = ops.linear_forward(x, W, b, act=1, precision=PREC[mode])
            assert _rel(y, torch.relu(_op(x, mode) @ _op(W, mode).t() + b.double())) < TOL_ACT[mode], dev
            dX, dW, db = ops.linear_backward(dY, x, W, precision=PREC[mode])
            assert _rel(dX, _op(dY, mode) @ _op(W, mode)) < TOL_ACT[mode], dev
            assert _rel(dW, _op(dY, mode).t() @ _op(x, mode)) < TOL_F32[mode], dev
            assert _rel(db, _op(dY, mode).sum(0)) < 1e-4, dev
            torch.cuda.synchronize()

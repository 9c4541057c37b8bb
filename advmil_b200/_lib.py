"""ctypes binding of libadvmil_b200.so (include/advmil_b200.h).  Fails loudly when the library is missing:
there is no CPU or PyTorch fallback for the hot path."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libadvmil_b200.so")

c_fp = C.c_void_p   # device float*
c_u8p = C.c_void_p  # device uint8*
c_ip = C.c_void_p   # int32*


class Bags(C.Structure):
    _fields_ = [("x", c_fp), ("offsets", c_ip), ("offsets_host", C.POINTER(C.c_int32)),
                ("rows", C.c_int32), ("bags", C.c_int32), ("C", C.c_int32), ("max_bag_rows", C.c_int32),
                ("elem", C.c_int32)]


GEN_TENSORS = ["W1", "b1", "Wa", "ba", "Wb", "bb", "wc", "bc", "Wrho", "brho", "W0", "b0", "Wl", "bl"]


class GenParams(C.Structure):
    _fields_ = [(n, c_fp) for n in GEN_TENSORS] + [
        ("C", C.c_int32), ("h", C.c_int32), ("o", C.c_int32), ("hid", C.c_int32),
        ("noise0", C.c_int32), ("noise1", C.c_int32), ("out_scale", C.c_int32),
        ("p_backbone", C.c_float), ("p_head", C.c_float)]


class GenGrads(C.Structure):
    _fields_ = [(n, c_fp) for n in GEN_TENSORS] + [("dx", c_fp)]


class GenActs(C.Structure):
    _fields_ = [("h", c_fp), ("ab", c_fp), ("s", c_fp), ("w", c_fp), ("z", c_fp), ("H", c_fp), ("H1", c_fp),
                ("pre", c_fp), ("pred", c_fp), ("noise0", c_fp), ("noise1", c_fp), ("h_eval", c_fp),
                ("mask_h", c_u8p), ("mask_a", c_u8p), ("mask_b", c_u8p), ("mask_rho", c_u8p), ("mask_mlp0", c_u8p),
                ("seed", C.c_uint64), ("train", C.c_int32), ("precision", C.c_int32),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("h_drop_out", c_fp), ("seed_drop", C.c_uint64), ("mask_h_drop", c_u8p), ("h_ready", C.c_int32)]


DISC_TENSORS = ["Wc", "bc", "ln_g", "ln_b", "F1a_w", "F1a_b", "F1b_w", "F1b_b", "Pg_w", "Pg_b", "Ps_w", "Ps_b",
                "Pc_w", "Pc_b", "F2a_w", "F2a_b", "F2b_w", "F2b_b", "T1_w", "T1_b", "T2_w", "T2_b", "Pr_w", "Pr_b"]


class DiscParams(C.Structure):
    _fields_ = [(n, c_fp) for n in DISC_TENSORS] + [
        ("C", C.c_int32), ("d", C.c_int32), ("t1", C.c_int32), ("t2", C.c_int32),
        ("inner_instance", C.c_int32), ("prj_path", C.c_int32), ("p", C.c_float), ("ln_eps", C.c_float), ("ksize", C.c_int32)]


class DiscGrads(C.Structure):
    _fields_ = [(n, c_fp) for n in DISC_TENSORS]


class EmbedActs(C.Structure):
    _fields_ = [("emb", c_fp), ("y_pre", c_fp), ("precision", C.c_int32),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class HeadActs(C.Structure):
    _fields_ = [("emb", c_fp), ("t", c_fp), ("f1", c_fp), ("fi", c_fp), ("ab", c_fp), ("rep", c_fp), ("attn", c_fp),
                ("bagv", c_fp), ("fbar", c_fp), ("g1", c_fp), ("hx", c_fp), ("u1", c_fp), ("ht", c_fp), ("out", c_fp),
                ("mask_fc1", c_u8p), ("mask_ga", c_u8p), ("mask_gs", c_u8p), ("mask_fc2", c_u8p),
                ("seed", C.c_uint64), ("train", C.c_int32), ("precision", C.c_int32),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class StepArgs(C.Structure):
    _fields_ = [("gen", C.POINTER(GenParams)), ("disc", C.POINTER(DiscParams)), ("gen_grads", C.POINTER(GenGrads)),
                ("disc_grads", C.POINTER(DiscGrads)), ("bags", C.POINTER(Bags)),
                ("t", c_fp), ("e", c_fp), ("visible", c_u8p), ("noise_d", c_fp), ("noise_g", c_fp),
                ("g_mask_h", c_u8p), ("g_mask_a", c_u8p), ("g_mask_b", c_u8p), ("g_mask_rho", c_u8p), ("g_mask_mlp0", c_u8p),
                ("d_mask_fc1", c_u8p), ("d_mask_ga", c_u8p), ("d_mask_gs", c_u8p), ("d_mask_fc2", c_u8p),
                ("seed_d", C.c_uint64), ("seed_g", C.c_uint64),
                ("n_real", C.c_float), ("n_fake", C.c_float), ("n_visible", C.c_float), ("loss_d", C.c_int32),
                ("coef_gan", C.c_float), ("recon_alpha", C.c_float), ("recon_gamma", C.c_float), ("recon_norm", C.c_int32),
                ("precision", C.c_int32),
                ("losses", c_fp), ("pred_d", c_fp), ("f_fake_d", c_fp), ("real_mask", c_u8p), ("pred_g", c_fp), ("f_fake_g", c_fp),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


ESAT_TENSORS = ["Wc", "bc", "ln_g", "ln_b", "Win", "bin", "Wout", "bout", "W1", "b1", "W2", "b2", "n1_g", "n1_b", "n2_g", "n2_b",
                "Pa_w", "Pa_b", "Ps_w", "Ps_b", "Pc_w", "Pc_b"]


class EsatParams(C.Structure):
    _fields_ = [(n, c_fp) for n in ESAT_TENSORS] + [
        ("C", C.c_int32), ("d", C.c_int32), ("ff", C.c_int32), ("nhead", C.c_int32), ("p", C.c_float), ("ln_eps", C.c_float)]


class EsatGrads(C.Structure):
    _fields_ = [(n, c_fp) for n in ESAT_TENSORS]


ESAT_ACTS = ["y_pre", "emb", "qkv", "lse", "ctx", "s1", "x1", "f", "s2", "x2", "ab", "rep", "attn", "H", "H1", "pre", "pred"]


class EsatActs(C.Structure):
    _fields_ = [(n, c_fp) for n in ESAT_ACTS] + [
        ("pe", c_fp), ("noise0", c_fp), ("noise1", c_fp), ("mask_attn", c_u8p), ("mask_attn_off", C.c_void_p),
        ("mask_sa", c_u8p), ("mask_ff1", c_u8p), ("mask_ff2", c_u8p), ("mask_ga", c_u8p), ("mask_gs", c_u8p), ("mask_mlp0", c_u8p),
        ("seed", C.c_uint64), ("train", C.c_int32), ("precision", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("emb_ready", C.c_int32)]


class EsatStepArgs(C.Structure):
    _fields_ = [("esat", C.POINTER(EsatParams)), ("head", C.POINTER(GenParams)), ("disc", C.POINTER(DiscParams)),
                ("esat_grads", C.POINTER(EsatGrads)), ("head_grads", C.POINTER(GenGrads)), ("disc_grads", C.POINTER(DiscGrads)),
                ("bags", C.POINTER(Bags)),
                ("t", c_fp), ("e", c_fp), ("visible", c_u8p), ("noise_d", c_fp), ("noise_g", c_fp), ("pe", c_fp),
                ("seed_d", C.c_uint64), ("seed_g", C.c_uint64),
                ("n_real", C.c_float), ("n_fake", C.c_float), ("n_visible", C.c_float), ("loss_d", C.c_int32),
                ("coef_gan", C.c_float), ("recon_alpha", C.c_float), ("recon_gamma", C.c_float), ("recon_norm", C.c_int32),
                ("precision", C.c_int32),
                ("losses", c_fp), ("pred_d", c_fp), ("f_fake_d", c_fp), ("real_mask", c_u8p), ("pred_g", c_fp), ("f_fake_g", c_fp),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class ClusterStepArgs(C.Structure):
    _fields_ = [("base", StepArgs), ("Wphi", c_fp), ("bphi", c_fp), ("dWphi", c_fp), ("dbphi", c_fp), ("cid", c_ip),
                ("num_clusters", C.c_int32)]


ABI_STRUCTS = [Bags, GenParams, GenGrads, GenActs, DiscParams, DiscGrads, EmbedActs, HeadActs, StepArgs, EsatParams, EsatGrads,
               EsatActs, EsatStepArgs, ClusterStepArgs]

# every symbol include/advmil_b200.h declares: name -> (restype, argtypes)
_i32, _i64, _f, _vp, _sz, _u64 = C.c_int32, C.c_int64, C.c_float, C.c_void_p, C.c_size_t, C.c_uint64
_P = C.POINTER
SYMBOLS = {
    "advmil_abi_version": (C.c_int, []),
    "advmil_last_error": (C.c_char_p, []),
    "advmil_abi_sizeof": (_sz, [C.c_int]),
    "advmil_launch_count": (_i64, [C.c_int]),
    "advmil_gate_packed_width": (_i32, [_i32]),
    "advmil_profile_enable": (C.c_int, [C.c_int]),
    "advmil_profile_read": (C.c_int, [_P(C.c_double), _P(C.c_int64), _i32]),
    "advmil_generator_workspace_bytes": (_sz, [_P(GenParams), _i32, _i32, _i32]),
    "advmil_generator_fwd": (C.c_int, [_P(GenParams), _P(Bags), _P(GenActs), _vp]),
    "advmil_generator_bwd": (C.c_int, [_P(GenParams), _P(Bags), _P(GenActs), _vp, _P(GenGrads), _vp]),
    "advmil_generator_sample": (C.c_int, [_P(GenParams), _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "advmil_disc_workspace_bytes": (_sz, [_P(DiscParams), _i32, _i32, _i32]),
    "advmil_disc_embed_fwd": (C.c_int, [_P(DiscParams), _P(Bags), _P(EmbedActs), _vp]),
    "advmil_disc_embed_bwd": (C.c_int, [_P(DiscParams), _P(Bags), _P(EmbedActs), _vp, _P(DiscGrads), _i32, _vp]),
    "advmil_disc_head_fwd": (C.c_int, [_P(DiscParams), _P(Bags), _P(HeadActs), _vp]),
    "advmil_disc_head_bwd": (C.c_int, [_P(DiscParams), _P(Bags), _P(HeadActs), _vp, _vp, _vp, _P(DiscGrads), _i32, _vp]),
    "advmil_segment_mean_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "advmil_segment_mean_by_id_fwd": (C.c_int, [_vp, _i32, _vp, _vp, _P(C.c_int32), _i32, _i32, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "advmil_segment_mean_by_id_bwd": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "advmil_linear_fwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _f, _vp, _u64, _i32, _i32, _i32, _vp, _vp]),
    "advmil_linear_bwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _vp, _sz, _vp]),
    "advmil_linear_bwd_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "advmil_gated_score_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f, _vp, _vp, _u64, _i32,
                                         _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "advmil_seg_softmax_pool_fwd": (C.c_int, [_vp, _vp, _i32, _vp, _P(C.c_int32), _i32, _i32, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "advmil_cast_f32_to_bf16": (C.c_int, [_vp, _i64, _vp, _vp]),
    "advmil_dropout_mask": (C.c_int, [_u64, _i32, _f, _i32, _i32, _vp, _vp]),
    "advmil_cindex_counts": (C.c_int, [_vp, _vp, _vp, _i32, _f, _vp, _vp]),
    "advmil_cindex_counts_f64": (C.c_int, [_vp, _vp, _vp, _i32, C.c_double, _vp, _vp]),
    "advmil_adv_step_workspace_bytes": (_sz, [_P(GenParams), _P(DiscParams), _i32, _i32, _i32]),
    "advmil_adv_step_disc": (C.c_int, [_P(StepArgs), _vp]),
    "advmil_adv_step_gen": (C.c_int, [_P(StepArgs), _vp]),
    "advmil_adv_step_gen_next": (C.c_int, [_P(StepArgs), _vp]),
    "advmil_seg_pool_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "advmil_region_index_map": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "advmil_region_of_rows": (C.c_int, [_i32, _i32, _vp, _vp]),
    "advmil_disc_loss": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _f, _f, _vp, _vp, _vp, _vp]),
    "advmil_gen_loss": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _f, _f, _f, _f, _f, _i32, _vp, _vp, _vp, _vp]),
    "advmil_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _f, _i32, _f, _vp]),
    "advmil_abs_sum": (C.c_int, [_vp, _i64, _vp, _vp]),
    "advmil_esat_workspace_bytes": (_sz, [_P(EsatParams), _P(GenParams), _i32, _i32, _i32]),
    "advmil_esat_fwd": (C.c_int, [_P(EsatParams), _P(GenParams), _P(Bags), _P(EsatActs), _vp]),
    "advmil_esat_bwd": (C.c_int, [_P(EsatParams), _P(GenParams), _P(Bags), _P(EsatActs), _vp, _P(EsatGrads), _P(GenGrads), _vp]),
    "advmil_sincos_pe": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _sz, _vp]),
    "advmil_adv_step_esat_workspace_bytes": (_sz, [_P(EsatParams), _P(GenParams), _P(DiscParams), _i32, _i32, _i32]),
    "advmil_adv_step_esat_disc": (C.c_int, [_P(EsatStepArgs), _vp]),
    "advmil_adv_step_esat_gen": (C.c_int, [_P(EsatStepArgs), _vp]),
    "advmil_adv_step_esat_gen_next": (C.c_int, [_P(EsatStepArgs), _vp]),
    "advmil_adv_step_cluster_workspace_bytes": (_sz, [_P(GenParams), _P(DiscParams), _i32, _i32, _i32, _i32]),
    "advmil_adv_step_cluster_disc": (C.c_int, [_P(ClusterStepArgs), _vp]),
    "advmil_adv_step_cluster_gen": (C.c_int, [_P(ClusterStepArgs), _vp]),
    "advmil_adv_step_cluster_gen_next": (C.c_int, [_P(ClusterStepArgs), _vp]),
    "advmil_cluster_pool_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "advmil_cluster_pool_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _P(C.c_int32), _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp,
                                          _vp, _sz, _vp]),
    "advmil_cluster_pool_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "advmil_mha_fwd": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _f, _u64, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "advmil_mha_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f, _u64, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "advmil_bf16p12_decode": (C.c_int, [_vp, _vp, C.c_char_p, _vp, _vp, _i64, _i32, _vp, _vp]),
    "advmil_bf16vl_encode": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _P(_i64), _P(_i64)]),
    "advmil_bf16vl_tables": (C.c_int, [_vp, _vp, _vp, _vp]),
    "advmil_bf16vl_encode_with_tables": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _P(_i64), _P(_i64)]),
    "advmil_bf16vl_decode_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    "advmil_bf16vl_decode": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp]),
}

PROF_TAGS = ["proj_fwd", "gate_fwd", "pool_fwd", "embed_fwd", "pool_gate_bwd", "bwd_data", "bwd_w_gate", "bwd_w_proj",
             "ln_bwd", "bwd_w_embed", "colsum", "dropout", "head_fwd", "head_bwd", "gen_tail", "loss_opt", "proj_embed_fwd",
             "attn_fwd", "attn_bwd", "proj_segmean_fwd"]

_lib = None


class AdvmilError(RuntimeError):
    pass


def load():
    """Loads the shared library (once).  Raises if it has not been built — never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AdvmilError(f"{LIB_PATH} not found: build it with `python -m advmil_b200.build` "
                          "(the advmil_b200 hot path has no CPU/PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.advmil_abi_version() != 3:
        raise AdvmilError("libadvmil_b200.so ABI version mismatch")
    for i, st in enumerate(ABI_STRUCTS):
        if lib.advmil_abi_sizeof(i) != C.sizeof(st):
            raise AdvmilError(f"ABI struct {st.__name__}: C sizeof {lib.advmil_abi_sizeof(i)} != ctypes {C.sizeof(st)}")
    _lib = lib
    return lib


def check(status: int, what: str = ""):
    if status != 0:
        msg = load().advmil_last_error().decode(errors="replace")
        kinds = {1: "invalid argument", 2: "CUDA error", 3: "workspace too small", 4: "no device"}
        if status == 1 and "multiple of 16" in msg:
            raise AssertionError(msg)  # the reference raises AssertionError here (model/backbone_utils.py:65)
        raise AdvmilError(f"{what}: {kinds.get(status, status)}: {msg}")

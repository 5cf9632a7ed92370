"""ctypes binding of the C-ABI in include/hero_b200.h.

The product path has no CPU fallback: if `libhero_b200.so` is missing, `lib()` raises with the
build command instead of silently routing around the CUDA kernels.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# HERO_B200_LIB: load another build of the same C-ABI (tools/ablate.sh uses it for its timing
# variant); the default is the in-tree library
LIB_PATH = os.environ.get("HERO_B200_LIB") or os.path.join(_PKG, "libhero_b200.so")

_lib = None


class HeroError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    """Mirror of `hero_gemm_args` (include/hero_b200.h)."""
    _fields_ = [
        ("a", C.c_void_p), ("b", C.c_void_p),
        ("lda", C.c_int64), ("ldb", C.c_int64),
        ("a_mn_major", C.c_int32), ("b_mn_major", C.c_int32),
        ("m", C.c_int32), ("n", C.c_int32), ("k", C.c_int32),
        ("bias", C.c_void_p),
        ("resid", C.c_void_p), ("ld_resid", C.c_int64),
        ("aux_in", C.c_void_p), ("ld_aux_in", C.c_int64),
        ("aux_out", C.c_void_p), ("ld_aux_out", C.c_int64),
        ("out", C.c_void_p), ("ld_out", C.c_int64),
        ("act", C.c_int32), ("out_f32_accumulate", C.c_int32),
        ("drop_threshold", C.c_uint32), ("drop_key", C.c_uint32),
        ("drop_scale", C.c_float),
        ("block_n", C.c_int32), ("k_splits", C.c_int32), ("cta_pair", C.c_int32),
        ("resid_f32", C.c_int32), ("out_f32_store", C.c_int32),
        ("a_lo", C.c_void_p), ("b_lo", C.c_void_p),
        ("resid_ln_mean", C.c_void_p), ("resid_ln_rstd", C.c_void_p),
        ("resid_ln_gamma", C.c_void_p), ("resid_ln_beta", C.c_void_p),
        ("ce_label", C.c_void_p), ("ce_partial", C.c_void_p), ("ce_label_logit", C.c_void_p),
        ("ce_lse", C.c_void_p), ("ce_grad", C.c_void_p), ("ce_ld_partial", C.c_int64),
        ("ce_n_valid", C.c_int32),
        ("out_colsum", C.c_void_p),
    ]


class LnArgs(C.Structure):
    """Mirror of `hero_ln_args` (include/hero_b200.h)."""
    _fields_ = [
        ("x", C.c_void_p), ("x_is_f32", C.c_int32),
        ("x_rows", C.c_void_p), ("add_tab", C.c_void_p), ("add_idx", C.c_void_p),
        ("add_vec", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
        ("eps", C.c_float), ("n_rows", C.c_int32), ("h", C.c_int32),
        ("y", C.c_void_p), ("y_lo", C.c_void_p), ("y_rows", C.c_void_p), ("y_f32", C.c_void_p),
        ("mean", C.c_void_p), ("rstd", C.c_void_p),
        ("drop_threshold", C.c_uint32), ("drop_key", C.c_uint32), ("drop_scale", C.c_float),
        ("dy", C.c_void_p), ("dx", C.c_void_p), ("dx_drop", C.c_void_p),
        ("drop2_threshold", C.c_uint32), ("drop2_key", C.c_uint32), ("drop2_scale", C.c_float),
        ("d_x_tab", C.c_void_p), ("x_pad_idx", C.c_int32),
        ("d_add_tab", C.c_void_p), ("add_pad_idx", C.c_int32),
        ("dgamma", C.c_void_p), ("dbeta", C.c_void_p), ("dbias", C.c_void_p),
    ]


class LayerWeights(C.Structure):
    """Mirror of `hero_layer_weights`."""
    _fields_ = [(n, C.c_void_p) for n in ("wqkv", "bqkv", "wo", "bo", "ln1_g", "ln1_b", "w1",
                                            "b1", "w2", "b2", "ln2_g", "ln2_b")]


class LayerActs(C.Structure):
    """Mirror of `hero_layer_acts`."""
    _fields_ = [(n, C.c_void_p) for n in ("qkv", "cx", "lse", "s1", "mean1", "rstd1", "a", "a_f32",
                                            "pre", "f", "s2", "mean2", "rstd2", "out", "out_f32")]


class LayerGrads(C.Structure):
    """Mirror of `hero_layer_grads`."""
    _fields_ = [(n, C.c_void_p) for n in ("dwqkv", "dbqkv", "dwo", "dbo", "dln1_g", "dln1_b",
                                            "dw1", "db1", "dw2", "db2", "dln2_g", "dln2_b")]


class StackArgs(C.Structure):
    """Mirror of `hero_stack_args`."""
    _fields_ = [
        ("n_layers", C.c_int32), ("n_tok", C.c_int32), ("hidden", C.c_int32),
        ("inter", C.c_int32), ("heads", C.c_int32), ("n_tiles", C.c_int32),
        ("n_long", C.c_int32), ("max_long", C.c_int32),
        ("eps", C.c_float),
        ("weights", C.POINTER(LayerWeights)), ("acts", C.POINTER(LayerActs)),
        ("grads", C.POINTER(LayerGrads)),
        ("x", C.c_void_p), ("x_f32", C.c_void_p),
        ("tile_tok0", C.c_void_p), ("tile_ntok", C.c_void_p), ("seq_lo", C.c_void_p),
        ("seq_hi", C.c_void_p),
        ("hidden_drop_threshold", C.c_uint32), ("attn_drop_threshold", C.c_uint32),
        ("drop_key", C.c_uint32),
        ("hidden_drop_scale", C.c_float), ("attn_drop_scale", C.c_float),
        ("dout", C.c_void_p), ("dx", C.c_void_p), ("scratch", C.c_void_p),
    ]


def _declare(lib):
    vp, i32, i64, f32, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_uint32
    lib.hero_last_error.restype = C.c_char_p
    lib.hero_last_error.argtypes = []
    lib.hero_version.restype = C.c_int
    lib.hero_sm_count.restype = C.c_int
    lib.hero_gemm_bf16.restype = C.c_int
    lib.hero_gemm_bf16.argtypes = [C.POINTER(GemmArgs), vp]

    def sig(name, *argtypes):
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = list(argtypes)

    sig("hero_ln_fwd", C.POINTER(LnArgs), vp)
    sig("hero_ln_bwd", C.POINTER(LnArgs), vp)
    sig("hero_attn_fwd", vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, f32, u32, u32,
        f32, vp)
    sig("hero_attn_bwd", vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, f32,
        u32, u32, f32, vp)
    sig("hero_gemm_profile_begin")
    sig("hero_gemm_profile_end", C.POINTER(C.c_double), C.POINTER(C.c_double),
        C.POINTER(C.c_int64))
    sig("hero_bert_stack_fwd", C.POINTER(StackArgs), vp)
    sig("hero_bert_stack_bwd", C.POINTER(StackArgs), vp)
    lib.hero_bert_stack_bwd_scratch_bytes.restype = C.c_int64
    lib.hero_bert_stack_bwd_scratch_bytes.argtypes = [i32, i32, i32]
    sig("hero_cast_f32_to_bf16", vp, vp, i64, vp)
    sig("hero_gather_rows_bf16", vp, vp, vp, i32, i32, vp)
    sig("hero_gather_rows_f32", vp, vp, vp, i32, i32, vp)
    sig("hero_gather_sum_rows_bf16", vp, vp, vp, vp, i32, i32, vp)
    sig("hero_gather_sum_rows_f32", vp, vp, vp, vp, i32, i32, vp)
    sig("hero_colsum_bf16", vp, i64, i32, i32, vp, vp)
    sig("hero_relu_bwd_bf16", vp, vp, vp, i64, vp)
    sig("hero_adamw_step", vp, vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, f32, vp, f32, vp)
    sig("hero_sumsq_f32", vp, i64, vp, vp)
    sig("hero_ce_finish", vp, i64, i32, vp, i32, vp, vp, vp)
    sig("hero_l2norm_split_f32", vp, i64, i32, f32, vp, vp, vp, vp)
    sig("hero_vsm_masked_max", vp, i64, vp, i32, i32, i32, vp, vp, vp)
    sig("hero_vsm_scores_bwd", vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp)
    sig("hero_vsm_span_fwd", vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp)
    sig("hero_vsm_span_bwd", vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp)
    sig("hero_videoqa_pool_fwd", vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp)
    sig("hero_videoqa_pool_bwd", vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp,
        vp, vp)


def lib():
    """Load (once) and return the shared library; raise if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HeroError(
                f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). "
                "Build it with `python -m hero_b200.build` (needs nvcc).")
        l = C.CDLL(LIB_PATH)
        _declare(l)
        _lib = l
    return _lib


def check(status):
    if status != 0:
        msg = lib().hero_last_error()
        raise HeroError(f"hero_b200 call failed (status {status}): "
                        f"{msg.decode() if msg else 'unknown error'}")

"""ctypes binding of libhba.so (the C-ABI declared in include/hba.h).

The product path has NO CPU fallback: importing this module without the compiled library raises,
and every op raises ``RuntimeError`` carrying ``hba_last_error()`` when the C-ABI reports an error.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhba.so")

HBA_ACT_NONE, HBA_ACT_QUICKGELU, HBA_ACT_GELU_ERF, HBA_ACT_QUICKGELU_GRAD, HBA_ACT_GELU_ERF_GRAD = range(5)
HBA_DT_F32, HBA_DT_BF16 = 0, 1

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class GemmParams(C.Structure):
    """Mirror of ``hba_gemm_params`` (include/hba.h)."""
    _fields_ = [
        ("A", vp), ("B", vp),
        ("M", i32), ("N", i32), ("K", i32),
        ("lda", i32), ("ldb", i32),
        ("nsplit", i32), ("a_lo_off", i32), ("b_lo_off", i32),
        ("alpha", f32),
        ("bias", vp), ("residual", vp), ("ldr", i32),
        ("act", i32),
        ("aux", vp), ("ld_aux", i32), ("aux_dtype", i32),
        ("pre_out", vp), ("ld_pre", i32), ("pre_dtype", i32),
        ("out_f32", vp), ("ld_f32", i32),
        ("out_bf16", vp), ("ld_bf16", i32), ("out_lo_off", i32),
        ("transpose_out", i32), ("max_ctas", i32),
        ("a_mn_major", i32), ("b_mn_major", i32),
        ("k_slices", i32), ("k_workspace", vp),
        ("colsum_partial", vp),
    ]


# name -> (restype, argtypes); must list every function declared in include/hba.h
SIGNATURES = {
    "hba_last_error": (C.c_char_p, []),
    "hba_abi_version": (i32, []),
    "hba_device_check": (i32, []),
    "hba_gemm_bf16": (i32, [C.POINTER(GemmParams), vp]),
    "hba_split_bf16": (i32, [vp, i64, i64, i64, vp, i64, i64, i32, vp]),
    "hba_layernorm_fwd": (i32, [vp, i64, i32, i64, i64, vp, vp, f32, vp, i64, vp, i64, i64, vp]),
    "hba_layernorm_bwd": (i32, [vp, i64, vp, i64, i32, i64, i64, vp, f32, vp, i64, i32, vp]),
    "hba_im2col_patches": (i32, [vp, i32, i32, i32, i32, vp, i64, i64, vp]),
    "hba_assemble_tokens_ln": (i32, [vp, i32, i32, i32, vp, vp, vp, vp, f32, vp, vp]),
    "hba_embed_tokens": (i32, [vp, i32, i32, i32, vp, vp, vp, vp]),
    "hba_gather_rows": (i32, [vp, i64, vp, i32, i32, vp, i64, vp]),
    "hba_attention_fwd": (i32, [vp, i32, i64, i32, i32, i32, i32, i32, vp, i64, i64, vp, i64, vp]),
    "hba_attention_bwd_row0": (i32, [vp, i32, i64, i32, i32, i32, vp, i64, vp, i64, vp]),
    "hba_dora_merge_fwd": (i32, [vp, vp, vp, vp, i32, i32, i32, f32, f32, vp, vp, i64, i64, vp, i64,
                                 i64, vp, vp]),
    "hba_dora_merge_bwd": (i32, [vp, i64, vp, vp, vp, vp, i32, i32, i32, f32, f32, vp, vp, vp, vp, vp]),
    "hba_cos_head_fwd": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, vp]),
    "hba_cos_head_bwd": (i32, [vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "hba_cos_mse_fwd": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]),
    "hba_cos_mse_bwd": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp, i64, vp, vp, vp, vp]),
    "hba_adamw_multi": (i32, [vp, vp, i32, i64, f32, f32, f32, f32, f32, i64, vp, vp, vp]),
    "hba_sgd_multi": (i32, [vp, vp, i32, i64, f32, f32, f32, i32, vp, vp]),
    "hba_sgd_staged": (i32, [vp, vp, i32, i64, f32, f32, f32, i32, vp, vp]),
    "hba_rdm_f64": (i32, [vp, i32, i32, vp, vp, vp]),
    "hba_rank_workspace_bytes": (i64, [i64]),
    "hba_rank_avg_f64": (i32, [vp, i64, vp, vp, i64, vp]),
    "hba_pearson_f64": (i32, [vp, vp, i64, vp, vp, vp]),
    "hba_rdm_spearman": (i32, [vp, i32, i32, vp, vp, vp, vp, vp, i64, vp]),
    "hba_rank_order_f64": (i32, [vp, i64, vp, vp, vp, i64, vp]),
    "hba_rsa_perm_workspace_bytes": (i64, [i32, i32]),
    "hba_rsa_perm_null": (i32, [vp, vp, i32, vp, i32, vp, vp, i64, vp]),
    "hba_rsa_boot_workspace_bytes": (i64, [i32, i32]),
    "hba_rsa_bootstrap": (i32, [vp, vp, vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, i64, vp]),
    "hba_kendall_workspace_bytes": (i64, [i64]),
    "hba_kendall_tau_f64": (i32, [vp, vp, vp, i64, vp, vp, vp, i64, vp]),
    "hba_softmax_ce_fwd_bwd": (i32, [vp, i64, vp, i32, i32, vp, vp, i64, vp, vp, vp]),
    "hba_colsum": (i32, [vp, i32, i64, i32, i64, vp, i32, vp, vp]),
    "hba_layernorm_param_grad": (i32, [vp, i64, vp, i64, i32, i64, i64, f32, vp, i32, vp, vp]),
    "hba_attention_bwd": (i32, [vp, i32, i64, i32, i32, i32, i32, vp, i32, i64, vp, i32, i64, vp]),
    "hba_layernorm_bwd_fused": (i32, [vp, i64, vp, i64, i32, i64, vp, f32, vp, i64, i32, vp, i64, i64, vp, i32, vp,
                                      vp, vp]),
    "hba_attention_fwd_lse": (i32, [vp, i64, i32, i32, i32, i32, vp, i64, vp, vp]),
    "hba_attention_bwd_lse": (i32, [vp, i64, i32, i32, i32, i32, vp, i64, vp, i64, vp, vp, i64, vp]),
    "hba_add_rows": (i32, [vp, i64, i64, vp, i64, i64, i32, vp]),
    "hba_nonfinite_flag": (i32, [vp, i64, vp, vp]),
}

_lib = None


def load():
    """Loads libhba.so (once). Raises ImportError with the build hint when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C vit-project_b200/csrc`). "
            "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export the symbol
        fn.restype = res
        fn.argtypes = args
    if lib.hba_abi_version() != 1:
        raise ImportError(f"{LIB_PATH}: ABI version {lib.hba_abi_version()} != 1, rebuild the extension")
    _lib = lib
    return lib


def last_error() -> str:
    return load().hba_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "libhba"):
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")

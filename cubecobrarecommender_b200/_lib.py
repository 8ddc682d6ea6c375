"""ctypes binding of libcubecobra_b200.so (the C ABI declared in include/cubecobra_b200.h).

There is no fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p, c_char_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcubecobra_b200.so")

P = c_void_p
I = c_int
I32 = c_int32
I64 = c_int64
U64 = c_uint64
F = c_float
D = c_double

# name -> (restype, argtypes); mirrors include/cubecobra_b200.h one to one
SIGNATURES = {
    "cc_last_error": (c_char_p, []),
    "cc_version": (I, []),
    "cc_device_check": (I, []),
    # (1) graph
    "cc_bits_words": (I64, [I64]),
    "cc_bits_cpad": (I64, [I32]),
    "cc_bitpack_cubes": (I, [P, P, I64, I32, P, P, P]),
    "cc_cooc_count": (I, [P, I64, I32, P, I64, I, P]),
    "cc_cooc_tc_chunk_cubes": (I64, [I64]),
    "cc_cooc_tc_workspace_bytes": (I64, [I64, I32]),
    "cc_cooc_count_tc": (I, [P, P, I64, I32, P, I64, P, I64, I, P, P]),
    "cc_row_normalise": (I, [P, I64, I32, P, I64, P, I64, P, I, D, P]),
    "cc_col_mass_workspace_bytes": (I64, [I32]),
    "cc_col_mass": (I, [P, I64, I32, P, P, P, P]),
    "cc_row_normalise_rows": (I, [P, I64, I32, I32, I32, P, I64, P, I64, P, I, D, P]),
    "cc_col_mass_rows": (I, [P, I64, I32, I32, I32, P, P, P, P]),
    "cc_col_mass_scale": (I, [P, I32, P]),
    "cc_create_adjacency_matrix_host": (I, [P, P, I64, I32, I, D, P, P]),
    # (2) scoring / top-N
    "cc_pairwise_leaf_count": (I64, [I64]),
    "cc_pairwise_plan_host": (I, [P, I32, P, P]),
    "cc_score_gather_f64": (I, [P, I64, I32, P, P, I32, P, P, I32, I, P, P, I64, P]),
    "cc_topn_workspace_bytes": (I64, [I32, I32, I32, I]),
    "cc_topn_masked_f32": (I, [P, I64, I32, I32, P, P, I, I, I32, P, I64, P, P, P, P]),
    "cc_topn_masked_sigmoid_f32": (I, [P, I64, I32, I32, P, P, I, I, I32, P, P, P, P]),
    "cc_topn_set_force_radix": (I, [I]),
    "cc_topn_set_algo": (I, [I]),
    "cc_topn_rowselect_profile_grid": (I64, [I32, I]),
    "cc_topn_rowselect_profile": (I, [P, I64, I32, I32, P, P, I32, I, P, P, P, P, P]),
    "cc_cuts_gather_f32": (I, [P, I64, I32, I32, P, P, I, P, P]),
    "cc_rank_targets_f32": (I, [P, I64, I32, I32, P, P, P, P, I, P, P]),
    "cc_rank_targets_f64": (I, [P, I64, I32, I32, P, P, P, P, P, P]),
    "cc_cosine_neg_f32": (I, [P, I64, I32, I32, I32, P, P]),
    "cc_topn_masked_f64": (I, [P, I64, I32, I32, P, P, I, I, I32, P, I64, P, P, P, P]),
    # (3) noise
    "cc_alias_build_host": (I, [P, I32, P, P]),
    "cc_noise_smem_bytes": (I64, [I32, I32]),
    "cc_noise": (I, [P, P, P, I32, I32, P, P, F, F, U64, P, I32, I32, P, P, P, I64, P, P, P, I64, P]),
    "cc_noise_ex": (I, [P, P, P, I32, I32, P, P, F, F, U64, P, I32, I32, P, P, P, I64, P, P, P, I64, I, P]),
    "cc_sample_reg_rows": (I, [P, P, I32, I32, U64, P, P, P]),
    "cc_cubes_to_bits": (I, [P, P, P, I32, I32, P, I64, P]),
    "cc_step_increment": (I, [P, P]),
    # (4) bag
    "cc_bag_fwd": (I, [P, I64, I32, P, P, P, I32, P, P, I64, I, I, P]),
    "cc_bag_bwd": (I, [P, I64, I32, P, P, P, I32, P, I64, P]),
    # (5) dense
    "cc_gemm_f32_simt": (I, [I, I, I, I, I, P, I64, P, I64, P, I64, P, I, P, I64, I, P]),
    "cc_gemm_tc": (I, [I, I, I, I, I, I, P, I64, P, I64, P, I64, P, I, P, I64, I, I, I, I, P]),
    "cc_gemm_bce_tc": (I, [I, I, I, I, P, I64, P, I64, P, P, I64, D, P, I64, P, P, I, I, P]),
    "cc_gemm_bce_tc_ex": (I, [I, I, I, I, P, I64, P, I64, P, P, I64, D, P, I64, P, P, I, I, P, P]),
    "cc_gemm_bce_partial_count": (I64, [I, I]),
    "cc_gemm_tc_set_pair_mode": (I, [I]),
    "cc_gemm_tc_plan": (I, [I, I, I, I, I, I, P]),
    "cc_gemm_tc_plan_ex": (I, [I, I, I, I, I, I, P]),
    "cc_gemm_tc_set_stream_k": (I, [I]),
    "cc_gemm_tc_set_dynamic_tiles": (I, [I]),
    "cc_gemm_tc_set_pdl": (I, [I]),
    "cc_gemm_tc_mn3_count": (I64, []),
    "cc_gemm_tc_register_readable": (I, [P, I64]),
    "cc_chain_tc": (I, [I, I, P, P, I64, P, P, P, P, P, P, P, P, I, P, P, I, P]),
    "cc_colsum_workspace_bytes": (I64, [I, I]),
    "cc_colsum_f32": (I, [P, I64, I, I, P, P, I, P]),
    "cc_relu_mask_f32": (I, [P, I64, P, I64, I, I, P]),
    # (6) losses / optimiser
    "cc_bce_logits_fwd_bwd": (I, [P, I64, P, I64, I32, I32, I32, D, P, I64, P, P]),
    "cc_softmax_kl_fuses_dbias": (I, [I32, I32, I64, I64, I64]),
    "cc_softmax_kl_fwd_bwd": (I, [P, I64, P, I64, P, I32, I32, I32, D, P, I64, P, I, P, P]),
    "cc_softmax_kl_fwd_bwd_ex": (I, [P, I64, P, I64, P, I32, I32, I32, D, P, I64, P, I, P, P, I64, P, P]),
    "cc_kl_target_table": (I, [P, I64, I32, I32, P, P]),
    "cc_softmax_kl_set_variant": (I, [I]),
    "cc_softmax_kl_fwd_bwd_metrics": (I, [P, I64, P, I64, P, I32, I32, I32, D, P, I64, P, I, P, P, I64, P, P, P, P]),
    "cc_kl_target_argmax": (I, [P, I64, I32, I32, P, P]),
    "cc_softmax_kl_loss": (I, [P, I64, P, I64, P, I32, I32, I32, P, P, P, P, I, P]),
    "cc_binary_accuracy_rows": (I, [P, I64, P, I64, I32, I32, P, P]),
    "cc_convert_f32_bf16": (I, [P, I64, P, I64, I32, I32, P]),
    "cc_loss_finalize": (I, [P, I32, D, P, I32, D, D, P, P]),
    "cc_adam_step_p2p": (I, [P, P, I, I, P, P, I64, I64, P, F, F, F, F, P, P, P]),
    "cc_adam_step": (I, [P, P, P, P, I64, P, F, F, F, F, P, P]),
    "cc_round_tf32": (I, [P, P, I64, P]),
    "cc_sigmoid_f32": (I, [P, P, I64, P]),
}


class CubeCobraError(RuntimeError):
    pass


_lib = None


def load(path: str | None = None):
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = path or os.environ.get("CUBECOBRA_B200_LIB", LIB_PATH)
    if not os.path.exists(path):
        raise CubeCobraError(
            f"{path} not found: build it with `python -m cubecobrarecommender_b200.build` "
            "(there is no CPU fallback)")
    import torch  # noqa: F401  (loads the CUDA runtime the library shares with torch)
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the ABI and the header disagree
        fn.restype = res
        fn.argtypes = args
    if lib.cc_version() != 100:
        raise CubeCobraError(f"libcubecobra_b200.so version {lib.cc_version()} != 100")
    _lib = lib
    return lib


def last_error() -> str:
    return (load().cc_last_error() or b"").decode("utf-8", "replace")


def check(rc: int, what: str = ""):
    if rc != 0:
        raise CubeCobraError(f"{what or 'libcubecobra_b200'} failed ({rc}): {last_error()}")


def call(name: str, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    fn = getattr(load(), name)
    check(fn(*args), name)


def ptr(t):
    """Device/host pointer of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return c_void_p(t.data_ptr())
    return c_void_p(t.ctypes.data)


def stream_ptr(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return c_void_p(s.cuda_stream)

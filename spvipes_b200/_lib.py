"""ctypes binding of libspvipes_b200.so (the C ABI declared in include/spvipes_b200.h).

There is no CPU fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPV_LIB") or os.path.join(_HERE, "libspvipes_b200.so")  # SPV_LIB: an A/B build of the same ABI

SRC_F32, SRC_U16_LOG1P, SRC_F32_LOG1P = 0, 1, 2
POE_LABEL, POE_PAIRED, POE_CLUSTER = 0, 1, 2
PARTNER_PAD, PARTNER_ABSENT = -1, -2
POE_MODES = {"label": POE_LABEL, "paired": POE_PAIRED, "cluster": POE_CLUSTER}
GENEC_ROWS = 21  # decoder_common.cuh GC_N
GC_THETA = 8  # row of theta = exp(px_r) in the per-gene constant table (decoder_common.cuh)
# widest latent input (P + S, plus one copy of the batch covariates per branch) of the decoder kernels: the fused tensor-core
# decoder (decoder_common.cuh ZK_MAX_LATENT) and every decoder path (DEC_MAX_LATENT: spv_dec_fold, spv_dec_gene_bwd)
ZK_MAX_LATENT = 58
DEC_MAX_LATENT = 96

p, i, ll, f, u64, u32 = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_ulonglong, C.c_uint

# name -> argtypes (must mirror include/spvipes_b200.h)
_SIGS = {
    "spv_abi_version": [],
    "spv_launch_count": [],
    "spv_arch_check": [i],
    "spv_copy2d_h2d": [p, ll, p, ll, ll, ll, p],
    "spv_gemm": [i, i, i, i, p, ll, p, p, ll, p, p, ll, i, i, i, i, ll, ll, ll, p, ll, i, i, i, p, p],
    "spv_gemm_fused": [i, i, i, i, p, ll, p, p, ll, p, p, ll, i, i, i, i, ll, ll, ll, p, ll, i, i, i, p, p, ll, p, ll, f, f, p, u64, u32, p, ll, p, p, ll, p],
    "spv_tc_gemm": [i, i, p, ll, p, ll, p, ll, i, i, i, p, i, i, i, p, p],
    "spv_tc_gemm_ex": [i, f, i, i, p, ll, p, ll, p, ll, i, i, i, p, i, i, i, p, p],
    "spv_tc_gemm_split": [i, i, p, p, ll, p, p, ll, p, ll, i, i, i, p, i, i, i, p, p],
    "spv_to_bf16": [p, ll, p, ll, i, i, p],
    "spv_to_f16": [p, ll, p, ll, i, i, p],
    "spv_to_bf16_split": [p, ll, p, p, ll, i, i, p],
    "spv_counts_to_bf16": [i, p, ll, p, p, p, ll, i, i, p, p, i, p],
    "spv_csr_max_genes": [i],
    "spv_csr_gather": [i, p, p, p, p, i, i, p, ll, p, p, ll, p, p, i, p],
    "spv_one_hot": [p, p, ll, i, i, p],
    "spv_cov_expand": [p, ll, p, p, ll, p, ll, i, i, i, i, p],
    "spv_cov_compact": [p, ll, p, ll, i, i, i, i, p, ll, p],
    "spv_library_size": [i, p, ll, p, i, i, p, p],
    "spv_dropout": [p, ll, i, i, p, ll, f, u64, u32, p, p],
    "spv_relu_bwd": [p, ll, p, ll, i, i, p, ll, f, p],
    "spv_bn_fwd": [p, ll, p, ll, i, i, p, p, f, f, p, p, p, p, i, i, p],
    "spv_bn_bwd": [p, ll, p, ll, p, ll, p, ll, i, i, p, p, p, p, p, p],
    "spv_colsum": [p, ll, i, i, p, p],
    "spv_pair_label": [p, p, p, p, i, i, p, p, p],
    "spv_plan_gather": [p, ll, p, p, i, i, p, p],
    "spv_plan_gather_bf16": [p, ll, p, p, i, i, p, p],
    "spv_plan_argmax": [p, i, i, p, p, p],
    "spv_plan_cluster_norm": [p, i, i, p, p, p, p, p],
    "spv_poe_fwd": [i, i, i, i, i, p, p, p, p, u64, p, p],
    "spv_poe_bwd": [i, i, i, i, i, p, p, p, p, u64, p, p, f, p],
    "spv_loss": [p, p, p, p, p, p, i, p, p, p],
    "spv_elbo_accumulate": [p, p, p, p, p, p, i, i, p, p, p],
    "spv_dec_fold": [p, ll, i, i, i, i, i, f, f, p, ll, i, i, p, p, p],
    "spv_dec_nb_fwd": [i, p, ll, ll, i, i, i, i, i, i, p, ll, i, p],
    "spv_dec_nb_bwd": [i, p, ll, ll, i, i, i, i, i, f, p, p, ll, p, ll, i, p],
    "spv_dec_nb_fwd_tc": [i, p, ll, p, ll, p, ll, i, p, p, i, i, i, i, i, i, i, p],
    "spv_dec_nb_elems_tc": [i, p, ll, p, ll, p, ll, i, p, p, i, i, i, i, i, i, p, ll, p],
    "spv_dec_nb_elems": [i, p, ll, ll, i, i, i, i, i, i, p, ll, i, p, ll, p],
    "spv_dec_nb_sample_tc": [p, p, ll, p, ll, i, p, p, i, i, i, i, i, i, u64, i, u32, i, p, ll, ll, p],
    "spv_nb_mixture_sample": [p, p, p, ll, p, i, i, i, p, ll, ll, u64, i, u32, p],
    "spv_dec_nb_rowreduce": [p, i, i, i, p, p, p],
    "spv_dec_gene_bwd": [p, ll, i, i, i, i, i, p],
    "spv_dec_gene_bwd_parts": [i],
    "spv_dec_nb_part_floats": [i, i],
    "spv_dec_stats_tc": [p, p, i, p, p, p, p, i, i, i, i, p],
    "spv_dec_theta_tables": [p, i, p, p, p],
    "spv_dec_nb_train_tc": [i, p, ll, p, ll, p, ll, i, p, p, p, ll, p, ll, i, i, i, i, i, i, p],
    "spv_dec_nb_train_colsum": [p, i, i, f, p, p],
    "spv_dec_zq4": [p, ll, p, p, ll, i, i, i, p],
    "spv_dec_dz4_combine": [p, ll, p, p, ll, i, i, i, p],
    "spv_dec_dzz_combine": [p, ll, p, p, p, i, p, ll, p, p, i, i, i, p, p],
    "spv_adam_tick": [p, p],
    "spv_adam": [p, p, p, p, ll, f, f, f, f, f, f, p, p, i, p, p, p, p, p, p, p, i, p],
    "spv_xgpu_allreduce": [p, p, p, ll, ll, i, i, i, p, i, p],
    "spv_xgpu_flag_ints": [],
}

_lib = None


class SpvError(RuntimeError):
    pass


def load():
    """Load the CUDA library; raises if it has not been built (python -m spvipes_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SpvError(f"{LIB_PATH} not found: build it with `python -m spvipes_b200.build` (no CPU fallback exists)")
    lib = C.CDLL(LIB_PATH)
    for name, args in _SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_longlong if name in ("spv_launch_count", "spv_dec_nb_part_floats") else C.c_int
    _lib = lib
    return lib


def exported_symbols():
    return list(_SIGS)


def check(rc: int, what: str):
    if rc != 0:
        raise SpvError(f"{what} failed with code {rc}")


def ptr(t):
    """device pointer of a torch tensor (or None -> NULL)"""
    return None if t is None else t.data_ptr()


def ptr_array(items):
    """host array of pointers from a list of tensors / ints / None"""
    arr = (C.c_void_p * len(items))()
    for k, it in enumerate(items):
        if it is None:
            arr[k] = None
        elif isinstance(it, int):
            arr[k] = it
        else:
            arr[k] = it.data_ptr()
    return arr


def int_array(items):
    arr = (C.c_int * len(items))()
    for k, it in enumerate(items):
        arr[k] = int(it)
    return arr


def ll_array(items):
    arr = (C.c_longlong * len(items))()
    for k, it in enumerate(items):
        arr[k] = int(it)
    return arr

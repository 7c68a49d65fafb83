"""ctypes binding of liblocator_b200.so (the C ABI in include/locator_b200.h).

There is no CPU fallback: importing this module fails loudly when the CUDA
library has not been built (``python -c 'import __graft_entry__ as g; g.build()'``
or ``make -C locator_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LOC_LIB_PATH") or os.path.join(_HERE, "lib", "liblocator_b200.so")  # override: A/B of builds


class LocatorCudaError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build the CUDA library first (make -C locator_b200/csrc). "
        "locator_b200 has no CPU fallback."
    )

lib = C.CDLL(LIB_PATH)


class LocState(C.Structure):
    _fields_ = [
        ("t", C.c_int32), ("epoch", C.c_int32), ("stopped", C.c_int32), ("improved", C.c_int32),
        ("best_epoch", C.c_int32), ("es_wait", C.c_int32), ("rlr_wait", C.c_int32), ("nonfinite", C.c_int32),
        ("lr", C.c_float), ("ckpt_best", C.c_float), ("last_loss", C.c_float), ("last_val_loss", C.c_float),
    ]


P = C.c_void_p
I64 = C.c_int64
I32 = C.c_int32

# name -> (restype, argtypes); every symbol include/locator_b200.h declares
SIGNATURES = {
    "loc_abi_version": (C.c_int, []),
    "loc_last_error": (C.c_char_p, []),
    "loc_l1_impl": (C.c_char_p, []),
    "loc_launch_count": (I64, []),
    "loc_site_stats": (C.c_int, [P, I64, I64, I32, P, P, P, P, P]),
    "loc_pack_sites": (C.c_int, [P, I64, I64, P, I64, P, I64, P]),
    "loc_compact_sites": (C.c_int, [P, I64, P, P, P]),
    "loc_missing_calls": (C.c_int, [P, I64, I64, P, I64, P, P, P, P, P]),
    "loc_bed_site_stats": (C.c_int, [P, I64, I64, I32, P, P, P, P, P]),
    "loc_bed_pack_sites": (C.c_int, [P, I64, I64, P, I64, P, I64, P]),
    "loc_bed_missing_calls": (C.c_int, [P, I64, I64, P, I64, P, P, P, P, P]),
    "loc_pack_sites_mapped": (C.c_int, [P, I64, I64, P, P, I64, P, I64, P]),
    "loc_bed_pack_sites_mapped": (C.c_int, [P, I64, I64, P, P, I64, P, I64, P]),
    "loc_site_sums": (C.c_int, [P, I64, I64, I64, P, P]),
    "loc_patch_calls": (C.c_int, [P, I64, P, P, P, I64, P]),
    "loc_pack_counts": (C.c_int, [P, I64, I64, P, I64, P]),
    "loc_unpack_counts": (C.c_int, [P, I64, I64, I64, P, P]),
    "loc_upload_pack_counts": (C.c_int, [P, I64, I64, P, I64, P]),
    "loc_gather_rows": (C.c_int, [P, I64, P, I64, P, P]),
    "loc_gather_cols": (C.c_int, [P, I64, I64, P, I64, P, I64, P]),
    "loc_replace_cols": (C.c_int, [P, I64, I64, P, I64, P, P]),
    "loc_blosc_decompress": (I64, [P, I64, P, I64]),
    "loc_zstd_decompress": (I64, [P, I64, P, I64]),
    "loc_np_legacy_binomial": (C.c_int, [P, C.POINTER(I32), I64, P, I64, I64, P]),
    "loc_np_legacy_permutation": (C.c_int, [P, C.POINTER(I32), I64, P]),
    "loc_vcf_count": (I64, [P, I64]),
    "loc_vcf_parse_gt": (C.c_int, [P, I64, I64, I64, P, P, I32]),
    "loc_model_create": (C.c_int, [C.POINTER(P), I64, I32, I32, I32, C.c_float, I32]),
    "loc_model_destroy": (C.c_int, [P]),
    "loc_model_pool_clear": (C.c_int, []),
    "loc_debug_timeline": (I64, [P, I64]),
    "loc_model_impl": (C.c_char_p, [P]),
    "loc_model_hidden_impl": (C.c_char_p, [P]),
    "loc_hidden_max_nlayers": (I32, [I32]),
    "loc_model_init": (C.c_int, [P, C.c_uint64, P]),
    "loc_model_num_weights": (C.c_int, [P]),
    "loc_model_weight_size": (I64, [P, I32]),
    "loc_model_set_weight": (C.c_int, [P, I32, P, I64, P]),
    "loc_model_get_weight": (C.c_int, [P, I32, P, I64, P]),
    "loc_model_get_adam": (C.c_int, [P, I32, P, P, I64, P]),
    "loc_model_set_shard": (C.c_int, [P, I64, I64]),
    "loc_model_set_exchange": (C.c_int, [P, P, P, P]),
    "loc_tp_create": (C.c_int, [C.POINTER(P), I32, I32, I32]),
    "loc_tp_handle": (C.c_int, [P, P]),
    "loc_tp_connect": (C.c_int, [P, P]),
    "loc_tp_error": (C.c_int, [P]),
    "loc_tp_destroy": (C.c_int, [P]),
    "loc_model_set_tp": (C.c_int, [P, P]),
    "loc_model_set_l1_ctas": (C.c_int, [P, I32]),
    "loc_model_set_schedule": (C.c_int, [P, C.c_float, I32]),
    "loc_model_bind_train": (C.c_int, [P, P, I64, I64, P]),
    "loc_model_bind_val": (C.c_int, [P, P, I64, I64, P]),
    "loc_model_set_dropout_masks": (C.c_int, [P, P, I64]),
    "loc_train_step": (C.c_int, [P, P, I32, P]),
    "loc_debug_stage": (C.c_int, [P, I32, P, I32, P]),
    "loc_debug_read": (I64, [P, I32, P, I64, P]),
    "loc_train_epochs": (C.c_int, [P, P, I32, P]),
    "loc_train_steps": (C.c_int, [P, P, I32, I32, P]),
    "loc_group_train_epochs": (C.c_int, [C.POINTER(P), I32, C.POINTER(P), I32, P]),
    "loc_eval": (C.c_int, [P, P, I64, I64, P, C.POINTER(C.c_float), P]),
    "loc_predict": (C.c_int, [P, P, I64, I64, P, P]),
    "loc_restore_best": (C.c_int, [P, P]),
    "loc_snapshot": (C.c_int, [P, P]),
    "loc_model_state": (C.c_int, [P, C.POINTER(LocState), P]),
    "loc_model_history": (C.c_int, [P, P, I32, P]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args


# loc_exchange_fn: int (*)(void* ctx, float* d_tile, int64_t n, void* stream)
EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)


def check(rc, what=""):
    if rc != 0:
        msg = lib.loc_last_error()
        raise LocatorCudaError(f"{what}: {msg.decode() if msg else 'unknown error'}")


def launch_count() -> int:
    return int(lib.loc_launch_count())

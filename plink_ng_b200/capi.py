"""ctypes binding of include/plink2_b200.h.  Fails loudly if the CUDA library is missing."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpl2gpu.so")


class Pl2Error(RuntimeError):
    pass


if not os.path.exists(_LIB_PATH):
    raise ImportError(
        f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc, sm_100a).  There is no CPU fallback."
    )

lib = C.CDLL(_LIB_PATH)

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
i32p = C.POINTER(C.c_int32)
f64p = C.POINTER(C.c_double)
vp = C.c_void_p

# name -> (restype, argtypes); must list every symbol include/plink2_b200.h declares
SIGNATURES = {
    "pl2gpu_device_count": (C.c_int, []),
    "pl2gpu_last_error": (C.c_char_p, []),
    "pl2gpu_abi_version": (C.c_int, []),
    "pl2gpu_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "pl2gpu_ctx_destroy": (C.c_int, [vp]),
    "pl2gpu_ctx_synchronize": (C.c_int, [vp]),
    "pl2gpu_ctx_stream": (vp, [vp]),
    "pl2gpu_ctx_launch_count": (C.c_uint64, [vp]),
    "pl2gpu_ctx_mem_info": (C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "pl2gpu_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(vp)]),
    "pl2gpu_host_free": (C.c_int, [vp]),
    "pl2gpu_ctx_event_record": (C.c_int, [vp, C.c_int]),
    "pl2gpu_ctx_event_elapsed_ms": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "pl2gpu_comm_unique_id": (C.c_int, [vp]),
    "pl2gpu_comm_init": (C.c_int, [vp, C.c_int, C.c_int, vp]),
    "pl2gpu_comm_destroy": (C.c_int, [vp]),
    "pl2gpu_comm_allreduce_sum_f64": (C.c_int, [vp, vp, C.c_uint64]),
    "pl2gpu_king_begin": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(vp)]),
    "pl2gpu_king_begin_ex": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.POINTER(vp)]),
    "pl2gpu_king_add_variants_sharded": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int]),
    "pl2gpu_king_mem_required": (C.c_uint64, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "pl2gpu_king_add_variants": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int]),
    "pl2gpu_king_get_counts": (C.c_int, [vp, C.c_uint32, C.c_uint32, vp, C.c_int]),
    "pl2gpu_king_get_kinship": (C.c_int, [vp, C.c_uint32, C.c_uint32, vp, C.c_int]),
    "pl2gpu_king_get_filtered": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_double, C.c_uint64, vp, vp, vp, C.POINTER(C.c_uint64)]),
    "pl2gpu_king_variants_added": (C.c_uint64, [vp]),
    "pl2gpu_king_last_kernel_ms": (C.c_int, [vp, C.POINTER(C.c_float)]),
    "pl2gpu_king_end": (C.c_int, [vp]),
    "pl2gpu_king_pairs_begin": (C.c_int, [vp, C.c_uint32, vp, C.c_uint64, C.POINTER(vp)]),
    "pl2gpu_king_pairs_add_variants": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int]),
    "pl2gpu_king_pairs_get_counts": (C.c_int, [vp, C.c_uint64, C.c_uint64, vp, C.c_int]),
    "pl2gpu_king_pairs_end": (C.c_int, [vp]),
    "pl2gpu_grm_begin": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(vp)]),
    "pl2gpu_grm_add_variants": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int, vp]),
    "pl2gpu_grm_add_variants_sharded": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, vp]),
    "pl2gpu_grm_get_rows": (C.c_int, [vp, C.c_uint32, C.c_uint32, vp, vp, C.c_uint64, C.c_int]),
    "pl2gpu_grm_variants_added": (C.c_uint64, [vp]),
    "pl2gpu_grm_eigen_topk": (C.c_int, [vp, C.c_uint32, vp, vp]),
    "pl2gpu_grm_end": (C.c_int, [vp]),
    "pl2gpu_pca_begin": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(vp)]),
    "pl2gpu_pca_add_variants": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int, vp]),
    "pl2gpu_pca_run": (C.c_int, [vp, vp, vp, vp]),
    "pl2gpu_pca_vscore": (C.c_int, [vp, vp, C.c_uint32, vp]),
    "pl2gpu_pca_begin_shard": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, vp]),
    "pl2gpu_pca_run_sharded": (C.c_int, [vp, vp, C.c_uint64, vp, vp]),
    "pl2gpu_pca_end": (C.c_int, [vp]),
    "pl2gpu_geno_counts": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, vp]),
    "pl2gpu_ld_band_flags": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_double, vp]),
    "pl2_indep_pairwise": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_uint32, vp, vp, C.c_uint32, C.c_uint32, C.c_double, C.c_int, vp, vp, C.c_int, vp]),
    "pl2_indep_pairwise_ex": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_uint32, vp, vp, C.c_uint32, C.c_uint32, C.c_double, C.c_int, vp, vp, C.c_int, vp, C.c_uint32, vp]),
    "pl2gpu_score_begin": (C.c_int, [vp, C.c_uint32, vp]),
    "pl2gpu_score_add_variants": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int, vp, vp]),
    "pl2gpu_score_get": (C.c_int, [vp, vp, vp, vp]),
    "pl2gpu_score_end": (C.c_int, [vp]),
    "pl2_ld_prune_walk": (C.c_int, [C.c_uint32, vp, vp, C.c_uint32, C.c_uint32, C.c_int, vp, vp, vp, C.c_uint32, C.c_uint32, vp]),
    "pl2gpu_int8_peak": (C.c_int, [vp, C.c_uint32, C.c_int, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pl2gpu_mxf4_peak": (C.c_int, [vp, C.c_uint32, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pl2gpu_selftest_umma": (C.c_int, [vp, C.c_int]),
    "pl2gpu_debug_umma": (
        C.c_int,
        [vp, vp, C.c_uint32, vp, C.c_uint32] + [C.c_uint32] * 9 + [vp],
    ),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return lib.pl2gpu_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise Pl2Error(f"{what} failed: {last_error()}")

"""ctypes binding of the C ABI in include/symmer_b200.h (symmer_b200/_lib/libsymmer_b200.so).

There is no CPU fallback: if the library is missing this module raises, and every operator in
`symmer_b200.ops` raises when no CUDA device is present.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libsymmer_b200.so")

c_i32, c_i64, c_f64, c_sz, c_p, c_u64 = (ctypes.c_int32, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t,
                                         ctypes.c_void_p, ctypes.c_uint64)

# name -> (restype, argtypes); mirrors include/symmer_b200.h one to one
SIGNATURES = {
    "sym_abi_version": (ctypes.c_int, []),
    "sym_last_error": (ctypes.c_char_p, []),
    "sym_check_device": (ctypes.c_int, [c_p, c_p, c_p]),
    "sym_pack": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p]),
    "sym_unpack": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p]),
    "sym_ycount": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p]),
    "sym_sketch_rows": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p]),
    "sym_cross_mul": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_p, c_p, c_p]),
    "sym_mul_cleanup_ws_bytes": (c_sz, [c_i64, c_i64, c_i32]),
    "sym_mul_cleanup": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_f64, c_p, c_p, c_i64, c_p, c_p,
                                       c_p, c_sz, c_p]),
    "sym_mul_cleanup_count": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_f64, c_p, c_p, c_p, c_sz, c_p]),
    "sym_mul_cleanup_emit": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_i64, c_p, c_p, c_p, c_sz, c_p]),
    "sym_mul_blocks_ws_bytes": (c_sz, [c_i64, c_i64, c_i32, c_p, c_i32]),
    "sym_mul_blocks_count": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_p, c_i32, c_f64, c_p, c_p, c_p,
                                            c_sz, c_p]),
    "sym_mul_blocks_count_tables": (ctypes.c_int, [c_p, c_p, c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_p, c_i32, c_f64,
                                                   c_p, c_p, c_p, c_p, c_sz, c_p]),
    "sym_mul_blocks_emit": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_p, c_i32, c_i64, c_p, c_p, c_p,
                                           c_sz, c_p]),
    "sym_mul_blocks_emit_spec": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_p, c_i32, c_f64, c_p, c_p, c_p,
                                                c_p, c_sz, c_p]),
    "sym_cleanup_ws_bytes": (c_sz, [c_i64, c_i32]),
    "sym_cleanup_count": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_f64, c_p, c_p, c_p, c_sz, c_p]),
    "sym_cleanup_emit": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_i64, c_p, c_p, c_p, c_sz, c_p]),
    "sym_cleanup": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_f64, c_p, c_p, c_i64, c_p, c_p, c_p, c_sz, c_p]),
    "sym_commute": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_i32, c_p, c_p]),
    "sym_commute_mma_ws_bytes": (c_sz, [c_i64, c_i64, c_i32]),
    "sym_commute_mma": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_i32, c_p, c_p, c_sz, c_p]),
    "sym_commute_mma_pitched": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_i32, c_p, c_i64, c_p, c_sz, c_p]),
    "sym_mirror_upper": (ctypes.c_int, [c_p, c_i64, c_i64, c_i64, c_p]),
    "sym_gather_column": (ctypes.c_int, [c_p, c_i64, c_i64, c_i64, c_p, c_p, c_p]),
    "sym_gather_rows": (ctypes.c_int, [c_p, c_p, c_p, c_i64, c_i32, c_p, c_p, c_p]),
    "sym_join_rows": (ctypes.c_int, [c_p, c_p, c_i64, c_p, c_p, c_p, c_i64, c_i32, c_p, c_p]),
    "sym_commute_bits": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_i32, c_p, c_p]),
    "sym_commute_qwc": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_i32, c_p, c_p]),
    "sym_gather_qubits": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_i32, c_p, c_p]),
    "sym_rotate_ws_bytes": (c_sz, [c_i64]),
    "sym_rotate": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_p, c_f64, c_f64, c_i32, c_f64, c_p, c_p, c_p, c_p, c_sz,
                                  c_p]),
    "sym_rotate_split_ws_bytes": (c_sz, [c_i64]),
    "sym_rotate_split": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "sym_term_masks": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_p, c_p, c_p, c_p]),
    "sym_apply": (ctypes.c_int, [c_p, c_p, c_p, c_i64, c_i32, c_p, c_p, c_i64, c_i64, c_i32, c_p]),
    "sym_expval": (ctypes.c_int, [c_p, c_p, c_p, c_i64, c_i32, c_p, c_p, c_i64, c_i64, c_i32, c_p]),
    "sym_expval_prepare_sym": (ctypes.c_int, [c_p, c_p, c_p, c_i64, c_p, c_p, c_p]),
    "sym_to_csr": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_p, c_i64, c_p, c_p, c_p, c_p, c_p]),
    "sym_pauli_decompose_dense": (ctypes.c_int, [c_p, c_i32, c_p, c_p]),
    "sym_pauli_decompose_diagonals": (ctypes.c_int, [c_p, c_i64, c_i32, c_p]),
    "sym_rows_from_masks": (ctypes.c_int, [c_p, c_p, c_p, c_i64, c_i32, c_p, c_p, c_p]),
    "sym_rref_ws_bytes": (c_sz, [c_i64]),
    "sym_rref": (ctypes.c_int, [c_p, c_i64, c_i64, c_i64, c_p, c_p, c_sz, c_p]),
    "sym_bit_transpose": (ctypes.c_int, [c_p, c_i64, c_i64, c_p, c_i64, c_p]),
    "sym_or_rows": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_p, c_p]),
    "sym_pack_matrix": (ctypes.c_int, [c_p, c_i64, c_i64, c_p, c_i64, c_p]),
    "sym_unpack_matrix": (ctypes.c_int, [c_p, c_i64, c_i64, c_i64, c_p, c_p]),
    "sym_project_ws_bytes": (c_sz, [c_i64, c_i32]),
    "sym_project": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_i32, c_p, c_p, c_i32, c_p, c_i32, c_p, c_p, c_p, c_p, c_p,
                                   c_sz, c_p]),
    "sym_nc_signs": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_i32, c_p, c_i32, c_p, c_i32, c_p, c_p, c_p]),
    "sym_nc_min_ws_bytes": (c_sz, [c_i64, c_i32]),
    "sym_nc_min": (ctypes.c_int, [c_p, c_p, c_p, c_i64, c_i32, c_i32, c_p, c_p, c_p, c_sz, c_p]),
    "sym_pair_records_ws_bytes": (c_sz, [c_i64, c_i64, c_i32]),
    "sym_pair_records": (ctypes.c_int, [c_p, c_i64, c_i64, c_i64, c_p, c_i64, c_i32, c_p, c_p, c_sz, c_p]),
    "sym_pair_records_blocks": (ctypes.c_int, [c_p, c_i64, c_p, c_i64, c_i32, c_p, c_i32, c_p, c_p, c_sz, c_p]),
    "sym_owner_classes": (ctypes.c_int, [c_p, c_i64, c_i32, c_i32, c_p, c_p, c_sz, c_p]),
    "sym_class_partition_ws_bytes": (c_sz, [c_i64]),
    "sym_class_partition": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_i32, c_p, c_p, c_p, c_p, c_p, c_sz, c_p]),
    "sym_partition_ws_bytes": (c_sz, [c_i64]),
    "sym_partition_records": (ctypes.c_int, [c_p, c_i64, c_i32, c_p, c_p, c_p, c_sz, c_p]),
    "sym_dedup_records_ws_bytes": (c_sz, [c_i64, c_i32]),
    "sym_dedup_records": (ctypes.c_int, [c_p, c_i64, c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_f64, c_p, c_p,
                                         c_i64, c_p, c_p, c_p, c_sz, c_p]),
    "sym_dedup_records_count": (ctypes.c_int, [c_p, c_i64, c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_f64, c_p,
                                               c_p, c_p, c_sz, c_p]),
    "sym_dedup_records_emit": (ctypes.c_int, [c_p, c_i64, c_p, c_p, c_i64, c_p, c_p, c_i64, c_i32, c_i64, c_p, c_p,
                                              c_p, c_sz, c_p]),
    "sym_set_tuning": (ctypes.c_int, [c_i32, c_i64]),
    "sym_set_emit_events": (ctypes.c_int, [c_p, c_p]),
    "sym_sort_pairs_ws_bytes": (c_sz, [c_i64]),
    "sym_sort_pairs": (ctypes.c_int, [c_p, c_p, c_i64, c_i32, c_p, c_sz, c_p]),
    "sym_debug_set_key_mask": (ctypes.c_int, [c_u64]),
    "sym_launch_count": (c_i64, []),
}

ERROR_NAMES = {-1: "SYM_E_INVALID", -2: "SYM_E_CUDA", -3: "SYM_E_WORKSPACE", -4: "SYM_E_CAPACITY",
               -5: "SYM_E_UNSUPPORTED"}


class SymmerB200Error(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


_lib = None


def load():
    """Load the shared library (building it first if the sources are newer and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    if not os.path.exists(LIB_PATH):
        _build.build()                 # builds in-tree with nvcc; raises if nvcc is missing
    elif _build.needs_build():
        # a .cu / .cuh / header newer than the library: a stale .so would silently run old kernels
        if os.path.exists(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")):
            _build.build()
        else:
            import warnings
            warnings.warn("symmer_b200: sources are newer than libsymmer_b200.so and nvcc is not available to rebuild it")
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"symmer_b200: CUDA library not found at {LIB_PATH}; run `python -m symmer_b200.build`")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.sym_abi_version() != 1:
        raise ImportError("symmer_b200: ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().sym_last_error()
        raise SymmerB200Error(rc, msg.decode() if msg else "")

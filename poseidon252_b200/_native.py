"""ctypes binding of include/poseidon252_b200.h.  The library MUST be present: there is no Python
or CPU fallback for any batch entry point (loading fails loudly with instructions)."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libposeidon252_b200.so")
_LIB = None

c_void_p, c_size_t, c_int, c_uint64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_uint64

# name -> (restype, argtypes): every symbol include/poseidon252_b200.h declares
SIGNATURES = {
    "p252_version": (ctypes.c_char_p, []),
    "p252_strerror": (ctypes.c_char_p, [c_int]),
    "p252_device_count": (c_int, [ctypes.POINTER(c_int)]),
    "p252_create": (c_int, [c_int, ctypes.POINTER(c_void_p)]),
    "p252_create_on_stream": (c_int, [c_int, c_void_p, ctypes.POINTER(c_void_p)]),
    "p252_destroy": (None, [c_void_p]),
    "p252_sync": (c_int, [c_void_p]),
    "p252_last_error": (ctypes.c_char_p, [c_void_p]),
    "p252_launch_count": (c_uint64, [c_void_p]),
    "p252_host_alloc": (c_int, [c_size_t, ctypes.POINTER(c_void_p)]),
    "p252_host_free": (c_int, [c_void_p]),
    "p252_domain_separator": (c_int, [c_int, ctypes.POINTER(c_uint64)]),
    "p252_tag_input": (c_int, [c_void_p, c_size_t, c_uint64, c_void_p, ctypes.POINTER(c_size_t)]),
    "p252_hash_to_scalar": (c_int, [c_void_p, c_size_t, c_void_p]),
    "p252_tag": (c_int, [c_void_p, c_size_t, c_uint64, c_void_p]),
    "p252_hash_tag": (c_int, [c_int, c_size_t, c_size_t, c_void_p]),
    "p252_encryption_tag": (c_int, [c_size_t, c_void_p]),
    "p252_permute_batch": (c_int, [c_void_p, c_void_p, c_size_t, c_int]),
    "p252_permute_batch_dense": (c_int, [c_void_p, c_void_p, c_size_t, c_int]),
    "p252_digest_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_size_t, c_void_p, c_size_t, c_int]),
    "p252_hash_batch": (c_int, [c_void_p, c_int, c_void_p, c_size_t, c_size_t, c_void_p, c_size_t, c_int]),
    "p252_hash_batch_truncated": (c_int, [c_void_p, c_int, c_void_p, c_size_t, c_size_t, c_void_p, c_size_t, c_int]),
    "p252_scalars_from_bytes": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_int]),
    "p252_scalars_to_bytes": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int]),
    "p252_encrypt_batch": (c_int, [c_void_p, c_void_p, c_size_t, c_size_t, c_void_p, c_void_p, c_void_p, c_int]),
    "p252_decrypt_batch": (c_int, [c_void_p, c_void_p, c_size_t, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p,
                                   ctypes.POINTER(c_size_t), c_int]),
    "p252_merkle4_level": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int]),
    "p252_merkle4_tree_nodes": (c_int, [c_size_t, ctypes.POINTER(c_size_t), ctypes.POINTER(c_int)]),
    "p252_merkle4_build": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int]),
    "p252_merkle_tree_nodes": (c_int, [c_int, c_size_t, ctypes.POINTER(c_size_t), ctypes.POINTER(c_int)]),
    "p252_merkle_build": (c_int, [c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_int]),
    "p252_get_kernel_info": (c_int, [c_void_p]),
    "p252_set_small_batch_max": (c_int, [c_void_p, c_size_t]),
    "p252_debug_fail_chunk": (c_int, [c_void_p, ctypes.c_longlong]),
    "p252_debug_staging_nonzero": (c_int, [c_void_p, ctypes.POINTER(c_size_t)]),
    "p252_merkle_open_batch": (c_int, [c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, c_void_p, c_int]),
    "p252_merkle_verify_batch": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p,
                                         ctypes.POINTER(c_size_t), c_int]),
    "p252_merkle_update_batch": (c_int, [c_void_p, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_size_t,
                                         ctypes.POINTER(c_size_t), c_int]),
    "p252_tree_level_timings": (c_int, [c_void_p, c_void_p, c_int, ctypes.POINTER(c_int), ctypes.POINTER(ctypes.c_float)]),
    "p252_dist_unique_id": (c_int, [c_void_p]),
    "p252_dist_init": (c_int, [c_void_p, c_void_p, c_int, c_int]),
    "p252_dist_finalize": (c_int, [c_void_p]),
    "p252_merkle4_shard_plan": (c_int, [c_size_t, c_int, c_int, c_void_p, c_int, ctypes.POINTER(c_int)]),
    "p252_merkle4_build_dist": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p, c_int]),
}

MEM_HOST, MEM_DEVICE, ASYNC, TIMING, NO_GATHER = 0, 1, 2, 4, 8


class KernelInfo(ctypes.Structure):
    """p252_kernel_info"""
    _fields_ = [("struct_size", ctypes.c_uint32), ("wide_mul_per_permutation", ctypes.c_uint32),
                ("dfma_per_permutation", ctypes.c_uint32), ("montmul_per_permutation", ctypes.c_uint32),
                ("threads_per_block", ctypes.c_uint32), ("min_blocks_per_sm", ctypes.c_uint32)]


class LevelTiming(ctypes.Structure):
    """p252_level_timing"""
    _fields_ = [("nodes", ctypes.c_uint64), ("my_nodes", ctypes.c_uint64), ("gather_bytes", ctypes.c_uint64),
                ("kernel_ms", ctypes.c_float), ("gather_ms", ctypes.c_float)]


class LevelPlan(ctypes.Structure):
    """p252_level_plan"""
    _fields_ = [("level_offset", ctypes.c_uint64), ("level_size", ctypes.c_uint64), ("my_offset", ctypes.c_uint64),
                ("my_count", ctypes.c_uint64), ("sharded", ctypes.c_int32), ("reserved", ctypes.c_int32)]

NCCL_UNIQUE_ID_BYTES = 128


def lib():
    """Load libposeidon252_b200.so (built in-tree by `python -m poseidon252_b200.build`)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "poseidon252_b200: %s is missing. Build the sm_100a library first "
                "(`python -m poseidon252_b200.build` or __graft_entry__.build()). "
                "There is no CPU fallback for the batch path." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)       # AttributeError = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        _LIB = handle
    return _LIB

"""ctypes binding of include/circkit_b200.h.  There is NO fallback: if the CUDA library is missing or
cannot be loaded this module raises, and every product entry point fails with it."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CIRCKIT_B200_LIB") or os.path.join(HERE, "libcirckit_b200.so")   # env: A/B builds

CK_OK = 0
CK_ERR_CUDA, CK_ERR_ARG, CK_ERR_STATE, CK_ERR_TOO_LONG, CK_ERR_TABLE_FULL = -1, -2, -3, -4, -5
CK_F_NORMALIZE, CK_F_NO_BYTES, CK_F_ALIGNED_OUT, CK_F_PACKED_IN, CK_F_SURVIVORS, CK_F_SINGLE_COPY = 1, 2, 4, 8, 16, 32
CK_PEER_HANDLE_BYTES = 64
CK_MONO_SENSITIVE, CK_MONO_FIRST_ONLY, CK_MONO_KEEP_ALL, CK_MONO_NONE = 1, 2, 4, 0xFFFFFFFF
CK_CMD_CANONICALIZE, CK_CMD_UNIQ, CK_CMD_MONOMERIZE = 1, 2, 3
CK_F_CANONICAL_BODY = 64
CK_DEFLATE_MAX_BYTES, CK_DEFLATE_DICT_BYTES = 64 << 20, 32768
CK_CLASS_2BIT_LE_512, CK_CLASS_2BIT_LE_2048, CK_CLASS_2BIT_LE_65536, CK_CLASS_2BIT_LE_425984 = 1, 2, 4, 8
CK_CLASS_2BIT_LE_4096, CK_CLASS_2BIT_LE_8192 = 1 << 10, 1 << 11


class CkConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("max_batch_bytes", C.c_uint64),
                ("max_batch_records", C.c_uint32), ("table_capacity", C.c_uint64)]


class CkPackedBatch(C.Structure):
    _fields_ = [("packed2", C.c_void_p), ("offsets", C.c_void_p), ("lens", C.c_void_p), ("lane", C.c_void_p),
                ("lane_bytes", C.c_void_p), ("lane_offsets", C.c_void_p), ("lane_bytes_total", C.c_uint64),
                ("n_records", C.c_uint32)]


class CkMonoOptions(C.Structure):
    _fields_ = [("seed_len", C.c_uint32), ("flags", C.c_uint32), ("overlap_dist", C.c_uint64),
                ("overlap_min_identity", C.c_double), ("min_length", C.c_uint64), ("max_length", C.c_uint64),
                ("min_overlap", C.c_uint64), ("min_overlap_percent", C.c_double)]


class NativeLibraryMissing(RuntimeError):
    pass


_vp, _u64, _u32, _i, _sz = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/circkit_b200.h declares
SIGNATURES = {
    "ck_init": (_i, [C.POINTER(CkConfig), C.POINTER(_vp)]),
    "ck_destroy": (None, [_vp]),
    "ck_last_error": (C.c_char_p, [_vp]),
    "ck_alloc_pinned": (_vp, [_vp, _sz]),
    "ck_free_pinned": (None, [_vp, _vp]),
    "ck_canon_submit": (_i, [_vp, _i, _vp, _vp, _u32, _u32]),
    "ck_canon_wait": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "ck_uniq_submit": (_i, [_vp, _i, _vp, _vp, _u32, _u32, _u64]),
    "ck_uniq_wait": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "ck_uniq_wait_survivors": (_i, [_vp, _i, C.POINTER(_u32), _vp, _vp, _vp, _vp, _vp, _vp]),
    "ck_uniq_reset": (_i, [_vp]),
    "ck_uniq_grow": (_i, [_vp, _u64]),
    "ck_uniq_table_info": (_i, [_vp, C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64)]),
    "ck_peer_export": (_i, [_vp, _u32, _u32, _u32, _vp]),
    "ck_peer_attach": (_i, [_vp, _vp]),
    "ck_dev_peer_first_index": (_i, [_vp, _vp, _vp, _u32, _u64, _vp, _u64, _vp]),
    "ck_pack2_words": (_u64, [_u64, _u32]),
    "ck_pack2_host": (_i, [_vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _u64, _vp, C.POINTER(_u64)]),
    "ck_canon_submit_packed": (_i, [_vp, _i, C.POINTER(CkPackedBatch), _u32]),
    "ck_uniq_submit_packed": (_i, [_vp, _i, C.POINTER(CkPackedBatch), _u32, _u64]),
    "ck_lmsr_index": (_i, [_vp, _vp, _sz, C.POINTER(_sz)]),
    "ck_lmsr": (_i, [_vp, _vp, _sz, _vp]),
    "ck_canonicalize": (_i, [_vp, _vp, _sz, _vp]),
    "ck_lmsr_index_batch": (_i, [_vp, _vp, _vp, _u32, _vp]),
    "ck_dev_workspace_bytes": (_u64, [_u32, _u64]),
    "ck_out_arena_bytes": (_u64, [_u64, _u32]),
    "ck_dev_canon_packed2": (_i, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _u64]),
    "ck_dev_canon_bytes": (_i, [_vp, _vp, _vp, _vp, _u32, _u64, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _u64]),
    "ck_dev_check": (_i, [_vp, _vp, _vp]),
    "ck_dev_table_bytes": (_u64, [_u64]),
    "ck_dev_table_clear": (_i, [_vp, _vp, _vp, _u64]),
    "ck_dev_table_insert": (_i, [_vp, _vp, _vp, _u64, _vp, _vp, _u64, _u32, _vp]),
    "ck_dev_table_first": (_i, [_vp, _vp, _vp, _u64, _vp, _u32, _vp]),
    "ck_dev_owner_partition": (_i, [_vp, _vp, _vp, _u32, _u64, _u32, _vp, _vp, _vp, _vp]),
    "ck_dev_table_insert_pairs": (_i, [_vp, _vp, _vp, _u64, _vp, _u32, _vp]),
    "ck_dev_owner_partition_padded": (_i, [_vp, _vp, _vp, _u32, _u64, _u32, _u32, _vp, _vp, _vp]),
    "ck_dev_owner_scatter_peers": (_i, [_vp, _vp, _vp, _u32, _u64, _u32, _u32, _u32, _vp, _vp, _vp]),
    "ck_dev_table_first_peers": (_i, [_vp, _vp, _vp, _u64, _vp, _u32, _u32, _u32, _vp]),
    "ck_dev_gather_first": (_i, [_vp, _vp, _vp, _vp, _u32, _vp]),
    "ck_dev_monomerize": (_i, [_vp, _vp, _vp, _vp, _vp, _u32, _u32, _u64, C.c_double, _u32, _vp]),
    "ck_dev_normalize": (_i, [_vp, _vp, _vp, _vp, _u32, _vp, _vp]),
    "ck_mono_submit": (_i, [_vp, _i, _vp, _vp, _u32, _u32, C.POINTER(CkMonoOptions)]),
    "ck_mono_wait": (_i, [_vp, _i, C.POINTER(_u32), _vp, _vp, _vp, _vp, _vp, _vp]),
    "ck_fasta_out_bytes": (_u64, [_u64, _u32]),
    "ck_fasta_submit": (_i, [_vp, _i, _vp, _u64, _u32, _u32, _u64, C.POINTER(CkMonoOptions), C.POINTER(_u32)]),
    "ck_fasta_wait": (_i, [_vp, _i, _vp, C.POINTER(_u64), C.POINTER(_u32), _vp, _vp, _vp, _vp, _vp]),
    "ck_deflate_bound": (_u64, [_u64]),
    "ck_deflate_submit": (_i, [_vp, _i, _vp, _u64, _vp, _u32, _u32]),
    "ck_deflate_wait": (_i, [_vp, _i, _vp, C.POINTER(_u64), C.POINTER(_u32)]),
    "ck_launch_count": (_u64, [_vp]),
    "ck_kernel_timing": (_i, [_vp, _i]),
    "ck_kernel_times": (_i, [_vp, _vp, _vp, _u32]),
    "ck_synth_offsets": (_i, [_vp, _vp, _u64, _u64, _u32, _u32, _u32, _u32, _u32, _vp, C.POINTER(_u64)]),
    "ck_synth_packed2": (_i, [_vp, _vp, _u64, _u64, _u32, _vp, _u32, _u32, _vp, _u32]),
    "ck_dev_unpack2": (_i, [_vp, _vp, _vp, _vp, _u32, _vp, _u32]),
    "ck_packed2_words": (_u64, [_u64, _u32, _u32]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} not found: build it with `python -m circkit_b200.build` "
                "(nvcc, sm_100a).  circkit_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)            # AttributeError if the library lacks a declared symbol
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib

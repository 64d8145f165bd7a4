"""ctypes binding of libpynqs_b200.so (C ABI: include/pynqs_b200.h).  No fallback: if the CUDA
library is missing or cannot be loaded, importing an op raises."""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libpynqs_b200.so")

# every symbol include/pynqs_b200.h declares (tests check the header against this list)
SYMBOLS = [
    "pynqs_abi_version", "pynqs_last_error", "pynqs_check_sorb", "pynqs_num_sd",
    "pynqs_tensor_to_onv", "pynqs_onv_to_tensor", "pynqs_comb", "pynqs_prepared_bytes", "pynqs_prepare_integrals",
    "pynqs_comb_hij_fused", "pynqs_hij",
    "pynqs_lut", "pynqs_hash_bytes", "pynqs_hash_build", "pynqs_lut_hashed",
    "pynqs_group_bytes", "pynqs_group_build", "pynqs_group_layout", "pynqs_eloc_scratch_bytes", "pynqs_eloc_sample_space",
    "pynqs_hamiltonian_scratch_bytes", "pynqs_hamiltonian_count", "pynqs_hamiltonian_emit", "pynqs_csr_spmm",
    "pynqs_reduce_scratch_bytes", "pynqs_reduce_count", "pynqs_reduce_emit", "pynqs_reduce_eloc",
    "pynqs_reduce_sample_scratch_bytes", "pynqs_reduce_sample_count", "pynqs_reduce_sample_emit",
    "pynqs_compact_scratch_bytes", "pynqs_lookup_count", "pynqs_lookup_emit", "pynqs_unique_count", "pynqs_unique_emit",
    "pynqs_merge_rank_sample", "pynqs_sort_bytes", "pynqs_sort_table", "pynqs_moments_scratch_bytes", "pynqs_weighted_moments",
    "pynqs_peer_gather", "pynqs_peer_gather_rows", "pynqs_set_tuning", "pynqs_l2_persist", "pynqs_launch_count",
]

OK, EVALUE, EOVERFLOW, ECUDA, EWORKSPACE = 0, 1, 2, 3, 4
F32, F64 = 0, 1

_lib = None


class PynqsLibraryMissing(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PynqsLibraryMissing(
            f"{LIB_PATH} not found: build it with `python -m pynqs_b200.build` (nvcc, sm_100a). "
            "pynqs_b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for s in SYMBOLS:
        getattr(lib, s)  # raises AttributeError if the build is stale
    lib.pynqs_last_error.restype = ctypes.c_char_p
    lib.pynqs_launch_count.restype = ctypes.c_int64
    lib.pynqs_reduce_scratch_bytes.restype = ctypes.c_int64
    lib.pynqs_reduce_sample_scratch_bytes.restype = ctypes.c_int64
    lib.pynqs_compact_scratch_bytes.restype = ctypes.c_int64
    lib.pynqs_sort_bytes.restype = ctypes.c_int64
    lib.pynqs_moments_scratch_bytes.restype = ctypes.c_int64
    if lib.pynqs_abi_version() != 1:
        raise RuntimeError("libpynqs_b200.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    return load().pynqs_last_error().decode()


def check(rc: int) -> None:
    """Map status codes to the exception types of the reference binding (bind.cpp:282-301)."""
    if rc == OK:
        return
    msg = last_error()
    if rc == EVALUE:
        raise ValueError(msg)
    if rc == EOVERFLOW:
        raise OverflowError(msg)
    raise RuntimeError(msg)


def set_tuning(name=None, value: int = 0) -> None:
    """Test / experiment knobs of the one-pass local energy (include/pynqs_b200.h); set_tuning() restores the defaults."""
    check(load().pynqs_set_tuning(name.encode() if name is not None else None, ctypes.c_int64(int(value))))


def launch_count() -> int:
    return int(load().pynqs_launch_count())


def vp(x) -> ctypes.c_void_p:
    return ctypes.c_void_p(x)


def i64(x) -> ctypes.c_int64:
    return ctypes.c_int64(int(x))

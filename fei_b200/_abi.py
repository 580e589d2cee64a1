"""ctypes binding of libfeiscan.so (include/feiscan.h).

This is the whole device boundary of the package: plain pointers and sizes, no torch.
Loading fails loudly when the library is missing; compute calls fail loudly (FeiCudaError)
when there is no CUDA device — there is no CPU implementation to fall back to.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfeiscan.so")

FEI_OK, FEI_E_CUDA, FEI_E_NCCL, FEI_E_CAPACITY, FEI_E_UNSUPPORTED, FEI_E_BADARG, FEI_E_STATE = 0, -1, -2, -3, -4, -5, -6
NCCL_ID_BYTES = 128
CHAIN_NCOLS = 10
J_NULL, J_STR, J_INT, J_FLOAT, J_TRUE, J_FALSE, J_BIGINT = range(7)


class FeiError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libfeiscan error {code}: {msg}")
        self.code = code


class FeiCudaError(FeiError):
    """No usable CUDA device / CUDA failure.  Never caught to run a CPU path."""


class FeiCapacityError(FeiError):
    pass


class CorpusHost(C.Structure):
    _fields_ = [
        ("n", C.c_uint64), ("global_base", C.c_uint64),
        ("hdr", C.c_void_p), ("hdr_off", C.c_void_p),
        ("body", C.c_void_p), ("body_off", C.c_void_p),
        ("name", C.c_void_p), ("name_off", C.c_void_p), ("name_spans", C.c_void_p),
        ("ts", C.c_void_p), ("wall", C.c_void_p), ("flags8", C.c_void_p), ("fsb", C.c_void_p),
    ]


class CorpusStats(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in
                ("n", "global_base", "hdr_bytes", "body_bytes", "tile_bytes", "name_bytes", "n_groups", "device_bytes")]


class ScanTiming(C.Structure):
    _fields_ = [("head_ms", C.c_float), ("body_ms", C.c_float), ("compact_ms", C.c_float), ("h2d_ms", C.c_float),
                ("d2h_ms", C.c_float), ("total_ms", C.c_float), ("kernel_launches", C.c_uint32),
                ("body_bytes_touched", C.c_uint64), ("body_bytes_read", C.c_uint64)]


class DirlistView(C.Structure):
    _fields_ = [("n", C.c_uint64), ("names", C.c_void_p), ("name_off", C.c_void_p), ("ts", C.c_void_p), ("wall", C.c_void_p), ("mtime_ns", C.c_void_p),
                ("ino", C.c_void_p), ("size", C.c_void_p), ("flags8", C.c_void_p), ("spans", C.c_void_p), ("status", C.c_void_p), ("flags_len", C.c_void_p)]


class JsonCol(C.Structure):
    _fields_ = [("tag", C.c_void_p), ("uniform_tag", C.c_int32), ("num", C.c_void_p), ("str", C.c_void_p), ("str_off", C.c_void_p)]


SORT_NONE, SORT_SLOT, SORT_NAME, SORT_NAME_UID, SORT_NAME_HOST, SORT_FLAGS, SORT_BODY, SORT_TS, SORT_WALL, SORT_KEYS = range(10)


class SortSpec(C.Structure):
    _fields_ = [("source", C.c_uint32), ("fallback", C.c_uint32), ("prog", C.c_void_p), ("prog_len", C.c_uint64), ("keys", C.c_void_p)]


class SortInfo(C.Structure):
    _fields_ = [("rounds", C.c_uint32), ("radix_passes", C.c_uint32), ("refined_rows", C.c_uint64), ("ms", C.c_float)]


_lib: Optional[C.CDLL] = None
_lock = threading.Lock()

_P = C.c_void_p
_U64 = C.c_uint64
_SIGS = {
    "fei_abi_version": (C.c_int, []),
    "fei_last_error": (C.c_char_p, []),
    "fei_init": (C.c_int, [C.c_int]),
    "fei_shutdown": (C.c_int, []),
    "fei_device_info": (C.c_int, [_P, _P, _P, _P]),
    "fei_host_register": (C.c_int, [_P, _U64]),
    "fei_host_unregister": (C.c_int, [_P]),
    "fei_microbench_alu": (C.c_int, [C.c_int, _P, _P]),
    "fei_host_copy_bench": (C.c_int, [_P, _U64, C.c_int, _P, _P]),
    "fei_dir_list": (C.c_int, [C.c_char_p, _P]),
    "fei_dirlist_view_get": (C.c_int, [_P, _P]),
    "fei_dirlist_free": (None, [_P]),
    "fei_read_files": (C.c_int, [C.c_char_p, _P, _P, _U64, _P, _P, C.c_int, _P, _P]),
    "fei_write_files": (C.c_int, [C.c_char_p, _P, _P, _P, _P, _U64, C.c_int]),
    "fei_corpus_create": (C.c_int, [_P]),
    "fei_corpus_destroy": (C.c_int, [_P]),
    "fei_corpus_load": (C.c_int, [_P, _P]),
    "fei_corpus_load_raw": (C.c_int, [_P, _P, _P, _P, _P]),
    "fei_corpus_last_load_timing": (C.c_int, [_P, _P]),
    "fei_corpus_stage_text": (C.c_int, [_P, _U64, _P, _U64, _U64]),
    "fei_corpus_load_raw_spans": (C.c_int, [_P, _P, _P, _U64, _P, _P, _P]),
    "fei_dir_list_names": (C.c_int, [C.c_char_p, _P]),
    "fei_host_arena_alloc": (C.c_int, [_U64, C.c_int, _P]),
    "fei_host_arena_free": (C.c_int, [_P, _U64]),
    "fei_read_dir_packed": (C.c_int, [C.c_char_p, _P, _P, _U64, _P, _U64, _P, _U64, C.c_int, _P, _P, _P, _P, _P]),
    "fei_corpus_synth": (C.c_int, [_P, _U64, _U64, _U64]),
    "fei_corpus_stats_get": (C.c_int, [_P, _P]),
    "fei_corpus_fetch": (C.c_int, [_P, _U64, _U64, _P, _U64, _P, _P, _U64, _P, _P, _P, _P, _P]),
    "fei_corpus_fetch_records": (C.c_int, [_P, _P, _U64, _P, _U64, _P, _P, _U64, _P]),
    "fei_corpus_save": (C.c_int, [_P, C.c_char_p]),
    "fei_corpus_load_snapshot": (C.c_int, [_P, C.c_char_p, _P]),
    "fei_scan_masks": (C.c_int, [_P, _P, _U64, _P]),
    "fei_scan_hits": (C.c_int, [_P, _P, _U64, _P, _P, _P]),
    "fei_scan_count": (C.c_int, [_P, _P, _U64, _P]),
    "fei_scan_last_timing": (C.c_int, [_P, _P]),
    "fei_corpus_token_histogram": (C.c_int, [_P, _P, _U64, C.c_uint8, _P, _U64, _P, _P, _P, _U64, _P]),
    "fei_corpus_slot_values": (C.c_int, [_P, _P, _U64, _P, _P, _P, _U64]),
    "fei_corpus_set_aux": (C.c_int, [_P, C.c_uint32, _P, _U64]),
    "fei_chain_validate_msgs": (C.c_int, [_P, _P, _P, _P, _P, _P, _U64, _U64, _P, _P, _P]),
    "fei_chain_validate_cols": (C.c_int, [_P, _P, _P, _U64, _U64, _P, _P, _P, _P, _U64, _P]),
    "fei_chain_create": (C.c_int, [_P]),
    "fei_chain_destroy": (C.c_int, [_P]),
    "fei_chain_load_msgs": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _U64, _U64]),
    "fei_chain_load_cols": (C.c_int, [_P, _P, _P, _P, _U64, _U64]),
    "fei_chain_synth": (C.c_int, [_P, _U64, _U64, _U64, C.c_int64]),
    "fei_chain_validate": (C.c_int, [_P, _P, _P, _P, _P]),
    "fei_chain_fetch": (C.c_int, [_P, _U64, _U64, _P, _U64, _P, _P, _P]),
    "fei_chain_serialize_cols": (C.c_int, [_P, _U64, _P, _U64, _P]),
    "fei_chain_mine": (C.c_int, [_P, C.c_uint32, _P, C.c_uint32, _U64, C.c_uint32, _U64, _P, _P, _P]),
    "fei_synth_record_host": (C.c_int, [_U64, _U64, _P, C.c_uint32, _P, _P, C.c_uint32, _P, _P, _P, _P, _P, _P, _P]),
    "fei_synth_block_host": (C.c_int, [_U64, _U64, _P, _P, _P, _P, _P]),
    "fei_synth_write_tree": (C.c_int, [C.c_char_p, C.c_char_p, _U64, _U64, _U64, C.c_int]),
    "fei_comm_unique_id": (C.c_int, [_P]),
    "fei_comm_init": (C.c_int, [_P, C.c_int, C.c_int]),
    "fei_comm_destroy": (C.c_int, []),
    "fei_comm_allgather_hits": (C.c_int, [_P, C.c_uint32, _P, _P, _P, _P]),
    "fei_comm_allreduce_first_bad": (C.c_int, [_P, _P]),
    "fei_comm_bind_corpus": (C.c_int, [_P]),
    "fei_comm_last_exchange_in_kernel": (C.c_int, []),
    "fei_comm_is_p2p": (C.c_int, []),
    "fei_comm_scan_gather": (C.c_int, [_P, _P, _U64, _P]),
    "fei_comm_gathered_checksum": (C.c_int, [C.c_uint32, _P, _P, _P]),
    "fei_comm_global_lists": (C.c_int, [C.c_uint32, _P, _P]),
    "fei_scan_list_checksum": (C.c_int, [_P, C.c_uint32, _P, _P]),
    "fei_scan_fetch_hits": (C.c_int, [_P, C.c_uint32, _P, _P]),
    "fei_sort_rows": (C.c_int, [_P, C.c_uint32, _P, _P, _U64, _P, C.c_int, _U64, _U64, _P, _P]),
}
EXPORTS = tuple(_SIGS)


def lib() -> C.CDLL:
    """Load libfeiscan.so (built in-tree by `make` / __graft_entry__.build())."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise ImportError(
                        f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
                        "fei_b200 has no CPU implementation of its scan / hash kernels.")
                l = C.CDLL(LIB_PATH)
                for name, (res, args) in _SIGS.items():
                    fn = getattr(l, name)       # AttributeError if the library does not export it
                    fn.restype, fn.argtypes = res, args
                _lib = l
    return _lib


def check(rc: int) -> None:
    if rc == FEI_OK:
        return
    msg = (lib().fei_last_error() or b"").decode("utf-8", "replace")
    if rc == FEI_E_CUDA:
        raise FeiCudaError(rc, msg)
    if rc == FEI_E_CAPACITY:
        raise FeiCapacityError(rc, msg)
    if rc == FEI_E_UNSUPPORTED:
        raise NotImplementedError(f"libfeiscan: {msg}")
    raise FeiError(rc, msg)


_init_device: Optional[int] = None


def init(device: Optional[int] = None) -> int:
    """Bind this process to one GPU (default: LOCAL_RANK or 0)."""
    global _init_device
    if device is None:
        device = int(os.environ.get("FEI_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    if _init_device != device:
        check(lib().fei_init(int(device)))
        _init_device = device
    return device


def ptr(a: Optional[np.ndarray]) -> Optional[int]:
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def device_info() -> dict:
    sm, hbm, maj, mnr = C.c_int(), C.c_uint64(), C.c_int(), C.c_int()
    check(lib().fei_device_info(C.byref(sm), C.byref(hbm), C.byref(maj), C.byref(mnr)))
    return {"sm_count": sm.value, "hbm_bytes": hbm.value, "cc": (maj.value, mnr.value)}


def sort_rows(corpora, row_corpus: np.ndarray, row_rec: np.ndarray, source: int, descending: bool = False, first: int = 0,
              count: Optional[int] = None, fallback: int = SORT_NONE, prog: Optional[bytes] = None, keys: Optional[np.ndarray] = None):
    """fei_sort_rows: (row indices at sorted positions [first, first + count), SortInfo).  `corpora`: Corpus handles;
    row i is record row_rec[i] of corpora[row_corpus[i]]."""
    rc = np.ascontiguousarray(row_corpus, dtype=np.uint32)
    rr = np.ascontiguousarray(row_rec, dtype=np.uint64)
    m = rr.size
    first = min(max(int(first), 0), m)
    n_out = m - first if count is None else max(0, min(int(count), m - first))
    out = np.zeros(max(1, n_out), dtype=np.uint64)
    hs = (C.c_void_p * max(1, len(corpora)))(*[c.handle for c in corpora])
    keys_a = np.ascontiguousarray(keys, dtype=np.uint64) if keys is not None else None
    spec = SortSpec(source, fallback, C.cast(C.c_char_p(prog), C.c_void_p) if prog is not None else None, len(prog) if prog is not None else 0,
                    ptr(keys_a))
    info = SortInfo()
    check(lib().fei_sort_rows(hs, len(corpora), ptr(rc), ptr(rr), m, C.byref(spec), 1 if descending else 0, first, n_out, ptr(out), C.byref(info)))
    return out[:n_out].astype(np.int64), info

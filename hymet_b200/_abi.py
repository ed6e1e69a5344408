"""ctypes binding of libhymet_screen.so (include/hymet_screen.h).

This is the whole Python<->CUDA seam: plain pointers and sizes, no torch types.
The library is built in-tree by hymet_b200.build (nvcc, sm_100a).  There is no
fallback of any kind: a missing library raises, a missing B200 makes hs_init fail.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)
f64p = C.POINTER(C.c_double)

HS_OK = 0
ERRORS = {-1: "HS_EINVAL", -2: "HS_ENODEV", -3: "HS_ECUDA", -4: "HS_EIO", -5: "HS_EFORMAT",
          -6: "HS_ENOMEM", -7: "HS_EUNSUPPORTED", -8: "HS_ENOSEQ", -9: "HS_ESTATE"}


class HsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code
        self.msg = msg


class DbInfo(C.Structure):
    _fields_ = [("k", C.c_uint32), ("s", C.c_uint32), ("seed", C.c_uint32), ("use64", C.c_uint32),
                ("n_refs", C.c_uint64), ("n_entries", C.c_uint64), ("n_distinct", C.c_uint64),
                ("n_buckets", C.c_uint64), ("max_key", C.c_uint64), ("device_bytes", C.c_uint64),
                ("bloom_bytes", C.c_uint64),
                ("t_parse_s", C.c_double), ("t_build_s", C.c_double),
                ("dense_max", C.c_uint64), ("bloom_keys", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("n_bases", C.c_uint64), ("n_records", C.c_uint64), ("n_positions", C.c_uint64),
                ("n_valid_kmers", C.c_uint64), ("n_probes", C.c_uint64), ("n_bucket_reads", C.c_uint64),
                ("n_hits", C.c_uint64), ("n_mix_inserts", C.c_uint64), ("set_size", C.c_uint64),
                ("n_mixture", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("n_launches", C.c_uint32), ("n_mix_passes", C.c_uint32),
                ("ms_stream", C.c_float), ("ms_reduce", C.c_float), ("ms_reset", C.c_float),
                ("reduce_path", C.c_uint32), ("n_touched", C.c_uint32), ("n_hit_refs", C.c_uint32),
                ("n_pairs", C.c_uint32), ("exchange_overflow", C.c_uint32), ("exchange_max_pairs", C.c_uint32),
                ("mix_unsettled", C.c_uint32)]

    def asdict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


# name -> (restype, argtypes).  Must list every symbol include/hymet_screen.h declares
# (tests/test_abi.py checks the header against this table and against the .so).
SIGNATURES = {
    "hs_version": (C.c_char_p, []),
    "hs_last_error": (C.c_char_p, []),
    "hs_init": (C.c_int, [C.c_int]),
    "hs_sm_count": (C.c_int, []),
    "hs_host_placement": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hs_msh_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "hs_msh_info": (C.c_int, [C.c_void_p, C.POINTER(DbInfo)]),
    "hs_msh_ref": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), u64p, u64p,
                             C.POINTER(u64p)]),
    "hs_msh_free": (None, [C.c_void_p]),
    "hs_db_from_msh": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "hs_db_load_msh": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "hs_db_from_msh_multi": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, C.POINTER(C.c_void_p)]),
    "hs_db_segments": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32), u64p, C.POINTER(C.c_uint32)]),
    "hs_db_from_arrays": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, u64p, u64p, u64p,
                                    C.POINTER(C.c_void_p)]),
    "hs_db_info": (C.c_int, [C.c_void_p, C.POINTER(DbInfo)]),
    "hs_db_ref": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), u64p, u64p]),
    "hs_db_free": (None, [C.c_void_p]),
    "hs_screen_new": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "hs_screen_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hs_screen_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "hs_screen_feed_fasta": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "hs_screen_feed_fasta_range": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64, C.c_uint64, C.c_int]),
    "hs_screen_feed_text": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "hs_screen_feed_packed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "hs_screen_feed_packed_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "hs_packed_words": (C.c_uint64, [C.c_uint64]),
    "hs_pack_text": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64, u64p,
                               C.POINTER(Stats)]),
    "hs_pack_text_device": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_uint64, u64p,
                                      C.POINTER(Stats)]),
    "hs_screen_flush": (C.c_int, [C.c_void_p]),
    "hs_screen_flush_async": (C.c_int, [C.c_void_p]),
    "hs_screen_counts_devptr": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), u64p]),
    "hs_screen_counts_compact": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, u32p]),
    "hs_screen_counts_compact_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "hs_screen_counts_scatter_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "hs_screen_counts_absorb": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "hs_screen_absorb_screen": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hs_screen_mixture_get": (C.c_int, [C.c_void_p, u64p, u32p]),
    "hs_screen_mixture_record": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hs_screen_mixture_merge_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "hs_screen_mixture_merge": (C.c_int, [C.c_void_p, u64p, C.c_uint32]),
    "hs_screen_segment_set_size": (C.c_int, [C.c_void_p, C.c_uint32, u64p]),
    "hs_screen_finish": (C.c_int, [C.c_void_p, C.c_int, u64p, u32p, f64p, f64p, C.POINTER(Stats)]),
    "hs_screen_finish_hits": (C.c_int, [C.c_void_p, C.c_int, u32p, C.POINTER(Stats)]),
    "hs_screen_hits_copy": (C.c_int, [C.c_void_p, C.c_uint32, u32p, u64p, u32p, f64p, f64p]),
    "hs_screen_reset": (C.c_int, [C.c_void_p]),
    "hs_screen_stats": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "hs_screen_free": (None, [C.c_void_p]),
    "hs_hash_packed": (C.c_int, [C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, u64p, u8p]),
    "hs_db_probe": (C.c_int, [C.c_void_p, u64p, C.c_uint64, u32p]),
    "hs_db_probe_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, u64p, u64p, C.POINTER(C.c_float)]),
    "hs_gather_bench": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(C.c_float)]),
    "hs_db_entry_ids": (C.c_int, [C.c_void_p, u32p]),
    "hs_stat_batch": (C.c_int, [C.c_uint32, C.c_uint64, C.c_uint64, u64p, u64p, f64p, f64p]),
    "hs_sketch_text": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t, u64p, u32p, u64p]),
    "hs_sketch_packed_device": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64,
                                          u64p, u32p]),
    "hs_pack_codes_device": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hs_lca_weighted": (C.c_int, [C.c_uint64, u64p, C.POINTER(C.c_int32), f64p, C.c_uint64, u32p, u32p, u32p, f64p, u8p]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB


def load(rebuild: bool = False) -> C.CDLL:
    """Load (building if the sources are newer) the CUDA library.  Raises if impossible."""
    global _lib
    if _lib is not None and not rebuild:
        return _lib
    path = _build.LIB
    if rebuild or not os.path.exists(path) or (os.path.exists(_build.CSRC) and _build.stale()
                                                and os.path.exists(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))):
        path = _build.build(force=rebuild)
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing and could not be built: the CUDA extension is required "
                           "(there is no CPU path)")
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != HS_OK:
        raise HsError(rc, load().hs_last_error().decode("utf-8", "replace"))


_tls = None


def init(device: int = 0) -> None:
    """Bind the CALLING THREAD to one B200 (hs_init is per thread: one thread per GPU can each own a
    database).  Raises HsError(HS_ENODEV) when there is none."""
    global _tls
    if _tls is None:
        import threading
        _tls = threading.local()
    if getattr(_tls, "device", None) == device:
        return
    check(load().hs_init(device))
    _tls.device = device

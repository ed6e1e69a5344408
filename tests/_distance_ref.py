"""`mash dist` references for the tests (TEST INFRASTRUCTURE): the CPU oracle's serial merge loop
(tests/distance_oracle/distance_oracle.c: orc_distance, orc_distance_write, orc_dist_pvalue) through
ctypes, a NumPy + scipy restatement of D1-D3 in closed form (DESIGN.md §5 "mash dist"), and a driver for
a real `mash dist` when one is installed."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
import time

import numpy as np

from tests import _oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "distance_oracle", "distance_oracle.c")
OUT = os.path.join(ROOT, "tests", "distance_oracle", "_build")
LIB = os.path.join(OUT, "libdistoracle.so")
BIN = os.path.join(OUT, "distance_oracle")
# the flags of oracle/Makefile: the distance oracle includes the screen oracle's source whole, so an orc_db
# made by tests/_oracle.py's liboracle.so is the same struct, built the same way, as one made here
CFLAGS = ["-O3", "-march=x86-64-v2", "-std=gnu11", "-Wall", "-Wextra", "-fPIC", "-pthread", "-fvisibility=hidden"]

_lib = None


def build() -> None:
    deps = [SRC, os.path.join(ROOT, "oracle", "mash_screen_oracle.c")]
    if all(os.path.exists(x) and os.path.getmtime(x) >= max(map(os.path.getmtime, deps)) for x in (LIB, BIN)):
        return
    os.makedirs(OUT, exist_ok=True)
    subprocess.run(["gcc", *CFLAGS, "-shared", "-o", LIB, SRC, "-lz", "-lm"], check=True)
    subprocess.run(["gcc", *CFLAGS, "-DDIST_ORACLE_MAIN", "-o", BIN, SRC, "-lz", "-lm"], check=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        orc.lib()
        build()
        L = C.CDLL(LIB)
        u64p, f64p = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
        L.orc_distance.argtypes = [C.c_void_p, C.c_void_p, u64p, C.c_uint64, C.c_uint32, C.c_int, u64p, u64p, f64p]
        L.orc_distance.restype = C.c_int
        L.orc_distance_write.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_double, C.c_double,
                                         C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_distance_write.restype = C.c_int
        L.orc_dist_pvalue.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64]
        L.orc_dist_pvalue.restype = C.c_double
        L.orc_dist_distance.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
        L.orc_dist_distance.restype = C.c_double
        _lib = L
    return _lib


def real_mash_dist(mash: str, ref: str, queries, threads: int, extra=()):
    """`mash dist -p threads [extra] ref queries...` of a real mash -> (TSV bytes, wall seconds, stderr)."""
    cmd = [mash, "dist", "-p", str(threads), *extra, ref, *queries]
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError("real mash failed (%d): %s" % (r.returncode, r.stderr.decode("utf-8", "replace")[-500:]))
    return r.stdout, dt, r.stderr.decode("utf-8", "replace")


def oracle_pairs(ref: orc.OracleDB, qry: orc.OracleDB, s_p: int, q_idx=None, threads: int = 8):
    """(common, denom, p-value), each [n_q, n_refs], from the oracle's serial merge."""
    q_idx = np.arange(qry.n_refs, dtype=np.uint64) if q_idx is None else np.ascontiguousarray(q_idx, np.uint64)
    n, N = len(q_idx), ref.n_refs
    common = np.zeros(max(n * N, 1), np.uint64); denom = np.zeros_like(common); pv = np.zeros(max(n * N, 1))
    p64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))
    assert lib().orc_distance(ref.h, qry.h, p64(q_idx), n, s_p, threads, p64(common), p64(denom),
                              pv.ctypes.data_as(C.POINTER(C.c_double))) == 0
    sh = (n, N)
    return common[:n * N].reshape(sh), denom[:n * N].reshape(sh), pv[:n * N].reshape(sh)


def oracle_tsv(ref: orc.OracleDB, qry: orc.OracleDB, s_p: int, max_d: float = 1.0, max_p: float = 1.0,
               table: bool = False, comments: bool = False, header: bool = True, threads: int = 8) -> bytes:
    with tempfile.TemporaryFile() as fh:
        assert lib().orc_distance_write(ref.h, qry.h, s_p, threads, max_d, max_p, int(table), int(comments),
                                        int(header), fh.fileno()) == 0
        fh.seek(0)
        return fh.read()


def r_of(len_ref: int, len_qry: int, k: int) -> float:
    kmer_space = 4.0 ** k
    px = 1. / (1. + kmer_space / len_ref)
    py = 1. / (1. + kmer_space / len_qry)
    return px * py / (px + py - px * py)


def closed_form(A: np.ndarray, B: np.ndarray, s_p: int):
    """D1 without a merge loop: a shared hash h counts iff #{x in A u B : x <= h} <= s_p."""
    A = np.asarray(A, np.uint64); B = np.asarray(B, np.uint64)
    shared = np.intersect1d(A, B, assume_unique=True)
    union = len(A) + len(B) - len(shared)
    rank = (np.searchsorted(A, shared, side="right") + np.searchsorted(B, shared, side="right")
            - np.arange(1, len(shared) + 1))
    return int(np.count_nonzero(rank <= s_p)), min(s_p, union)


def closed_pvalue(common: int, denom: int, len_ref: int, len_qry: int, k: int) -> float:
    from scipy.stats import binom
    if common == 0:
        return 1.0
    return float(binom.sf(common - 1, denom, r_of(len_ref, len_qry, k)))


def distance(common: int, denom: int, k: int) -> float:
    if common == denom:
        return 0.0
    if common == 0:
        return 1.0
    j = common / denom
    return min(-np.log(2 * j / (1. + j)) / k, 1.0)


def db_of(k: int, s: int, sketches, lengths=None, seed: int = 42) -> orc.OracleDB:
    offsets = np.concatenate([[0], np.cumsum([len(x) for x in sketches])]).astype(np.uint64)
    hashes = np.concatenate([np.asarray(x, np.uint64) for x in sketches]) if sketches else np.zeros(0, np.uint64)
    lengths = np.asarray(lengths if lengths is not None else [5_000_000] * len(sketches), np.uint64)
    return orc.OracleDB.from_arrays(k, s, seed, offsets, hashes if len(hashes) else np.zeros(1, np.uint64), lengths)


def distinct_hashes(rng: np.random.Generator, n: int) -> np.ndarray:
    """n distinct random 64-bit hashes, ascending."""
    h = np.unique(rng.integers(0, np.iinfo(np.uint64).max, size=n + 16, dtype=np.uint64, endpoint=True))
    return np.sort(rng.permutation(h)[:n])


def boundary_pairs(rng: np.random.Generator, s: int):
    """(A, B, s_p) cases at D1's edges: a shared hash at union rank s_p and s_p + 1, |A u B| < s, empty
    sketches, identical sketches, s_p below both sizes."""
    cases = []
    base = distinct_hashes(rng, 4 * s)
    A = base[0:2 * s:2][:s]; B = base[1:2 * s:2][:s]          # interleaved: union rank of element i is known
    for rank in (s - 1, s, s + 1):                              # put a shared hash at union rank `rank`
        a = A.copy(); b = B.copy()
        h = np.sort(np.concatenate([a, b]))[rank - 1]
        if h in a:
            b = np.sort(np.unique(np.concatenate([b[:-1], [h]])))
        else:
            a = np.sort(np.unique(np.concatenate([a[:-1], [h]])))
        cases.append((a, b, s))
    cases.append((A[: s // 4], B[: s // 3], s))                 # |A u B| < s
    cases.append((A[: s // 4], np.concatenate([A[: s // 8], B[: s // 8]]).astype(np.uint64), s))
    cases.append((np.zeros(0, np.uint64), B, s))                # one empty
    cases.append((np.zeros(0, np.uint64), np.zeros(0, np.uint64), s))   # both empty
    cases.append((A, A.copy(), s))                              # identical
    mixed = np.sort(np.concatenate([A[: s // 2], B[s // 2:]])).astype(np.uint64)
    cases.append((A, mixed, s // 2))                            # s_p below both sizes
    cases.append((A, mixed, s // 3))
    return [(np.sort(a).astype(np.uint64), np.sort(b).astype(np.uint64), sp) for a, b, sp in cases]

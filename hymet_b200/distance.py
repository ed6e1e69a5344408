"""`mash dist` on the GPU: ctypes binding of hs_distance_* (include/hymet_screen.h, DESIGN.md §5 "mash dist").

One reference .msh against query sketches: query .msh files as they are, FASTA/FASTQ files sketched
with the reference's k, s and seed by the GPU sketcher (screen.sketch_files).  The pairs that share a
hash are found and merged on the device; the library writes the TSV.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _abi
from ._abi import HsError, check


@dataclass
class MshHeader:
    """What decides whether two sketch files can be compared (read on the host, no GPU)."""
    k: int
    s: int
    seed: int
    use64: bool
    n_refs: int


class HostMsh:
    """A parsed .msh held by the library on the host (hs_msh)."""

    def __init__(self, path: str):
        self.path = path
        L = _abi.load()
        self.h = C.c_void_p()
        check(L.hs_msh_open(os.fsencode(path), C.byref(self.h)))
        info = _abi.DbInfo()
        check(L.hs_msh_info(self.h, C.byref(info)))
        self.header = MshHeader(int(info.k), int(info.s), int(info.seed), bool(info.use64), int(info.n_refs))

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            _abi.load().hs_msh_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def mismatch(ref: MshHeader, q: MshHeader) -> Optional[str]:
    """Why query sketches with header q cannot be compared with the reference's (None: they can)."""
    if q.k != ref.k:
        return "k-mer size %d differs from the reference's (%d)" % (q.k, ref.k)
    if q.seed != ref.seed:
        return "hash seed %d differs from the reference's (%d)" % (q.seed, ref.seed)
    if q.use64 != ref.use64:
        return "hash width differs from the reference's"
    return None


@dataclass
class Rows:
    """Candidate pairs (pairs that share a hash) in (query, reference) order."""
    q: np.ndarray
    r: np.ndarray
    common: np.ndarray
    denom: np.ndarray
    pvalue: np.ndarray      # < 0: not computed (farther than max_distance)


class Distance:
    """The reference side on one GPU; queries are queued, then `run` writes the output."""

    def __init__(self, ref: HostMsh, device: int = 0):
        _abi.init(device)
        self.ref = ref.header
        self.h = C.c_void_p()
        check(_abi.load().hs_distance_new(ref.h, C.byref(self.h)))

    def add_msh(self, m: HostMsh) -> None:
        check(_abi.load().hs_distance_add_msh(self.h, m.h))

    def add_sketch(self, name: str, comment: str, length: int, s: int, hashes: np.ndarray) -> None:
        hashes = np.ascontiguousarray(hashes, np.uint64)
        check(_abi.load().hs_distance_add_sketch(self.h, os.fsencode(name), comment.encode("utf-8", "surrogateescape"),
                                                 int(length), int(s), hashes.ctypes.data_as(_abi.u64p), len(hashes)))

    def run(self, fd: int, max_distance: float = 1.0, max_pvalue: float = 1.0, table: bool = False,
            comments: bool = False, threads: int = 1) -> None:
        check(_abi.load().hs_distance_run(self.h, fd, float(max_distance), float(max_pvalue), int(table),
                                          int(comments), int(threads)))

    def run_rows(self, max_distance: float = 1.0) -> Rows:
        L = _abi.load()
        n = C.c_uint64()
        check(L.hs_distance_run_rows(self.h, float(max_distance), C.byref(n)))
        m = n.value
        out = Rows(np.zeros(m, np.uint32), np.zeros(m, np.uint32), np.zeros(m, np.uint32), np.zeros(m, np.uint32),
                   np.zeros(m, np.float64))
        p32 = lambda a: a.ctypes.data_as(_abi.u32p)
        check(L.hs_distance_rows_copy(self.h, m, p32(out.q), p32(out.r), p32(out.common), p32(out.denom),
                                      out.pvalue.ctypes.data_as(_abi.f64p)))
        return out

    def stats(self) -> dict:
        st = _abi.DistanceStats()
        check(_abi.load().hs_distance_stats(self.h, C.byref(st)))
        return st.asdict()

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            _abi.load().hs_distance_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def sketch_comment(header: bytes, n_records: int) -> str:
    """Comment of a sketched file: its first header line; Mash's form for multi-record files."""
    first = header.decode("utf-8", "replace").strip()
    if n_records > 1:
        first = "[%d seqs] %s [...]" % (n_records, first)
    return first


def is_msh(path: str) -> bool:
    return path.endswith(".msh")


def add_queries(d: Distance, paths: List[str], threads: int = 1, device: int = 0, warn=None) -> None:
    """Queue the query files in order: .msh files whole, sequence files sketched (one sketch per file, named
    after the path as given) with the reference's k, s and seed.  `warn(msg)` hears about files whose
    sketch size differs from the reference's."""
    from . import screen
    ref = d.ref
    seq = [p for p in paths if not is_msh(p)]
    sketched = iter(screen.sketch_files(seq, ref.k, ref.s, ref.seed, threads, device)[0]) if seq else iter(())
    for p in paths:
        if is_msh(p):
            m = HostMsh(p)
            try:
                why = mismatch(ref, m.header)
                if why:
                    raise HsError(-7, "%s: %s" % (p, why))
                if m.header.s != ref.s and warn:
                    warn("The query sketch size of %s (%d) differs from the reference's (%d); distances use the "
                         "smaller one (%d)." % (p, m.header.s, ref.s, min(m.header.s, ref.s)))
                d.add_msh(m)
            finally:
                m.close()
        else:
            g = next(sketched)
            d.add_sketch(p, sketch_comment(g.header, g.n_records), g.length, ref.s, g.hashes)

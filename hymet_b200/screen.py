"""Host-side mirror of `mash screen` over the C ABI (include/hymet_screen.h).

The reference has no in-process API for this path: HYMET forks
``mash screen -p 8 -v 0.9 DB.msh input/*.fna`` (/root/reference/scripts/mash.sh:14).
``Database`` + ``Screen`` are the objects bin/mash (hymet_b200.cli) drives; their
method names follow the stages Mash prints on stderr (S20): load, stream, sum shared,
(reallocate to winners), coverage medians, output.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

from . import _abi
from ._abi import HsError, check  # noqa: F401  (re-exported)


def _ptr(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


@dataclass
class ScreenResult:
    shared: np.ndarray     # uint64 [N]
    median: np.ndarray     # uint32 [N]
    identity: np.ndarray   # float64 [N]
    pvalue: np.ndarray     # float64 [N]
    set_size: int
    stats: dict


@dataclass
class ScreenHits:
    """Only the references mash would print (shared > 0), ascending by reference index."""
    ref: np.ndarray        # uint32 [H]
    shared: np.ndarray     # uint64 [H]
    median: np.ndarray     # uint32 [H]
    identity: np.ndarray   # float64 [H]
    pvalue: np.ndarray     # float64 [H]
    set_size: int
    stats: dict

    def to_dense(self, n_refs: int) -> ScreenResult:
        """The columns hs_screen_finish would have returned (shared = 0 => identity 0, p-value 1)."""
        shared = np.zeros(n_refs, np.uint64); median = np.zeros(n_refs, np.uint32)
        ident = np.zeros(n_refs, np.float64); pv = np.ones(n_refs, np.float64)
        shared[self.ref] = self.shared; median[self.ref] = self.median
        ident[self.ref] = self.identity; pv[self.ref] = self.pvalue
        return ScreenResult(shared, median, ident, pv, self.set_size, self.stats)


class Database:
    """A sketch database resident in the HBM of one B200 (rows a4/a5)."""

    def __init__(self, handle: int, device: int):
        self._h = C.c_void_p(handle)
        self.device = device
        info = _abi.DbInfo()
        check(_abi.load().hs_db_info(self._h, C.byref(info)))
        self.info = info
        self.k, self.s, self.seed = info.k, info.s, info.seed
        self.use64 = bool(info.use64)
        self.n_refs, self.n_entries, self.n_distinct = info.n_refs, info.n_entries, info.n_distinct
        self._meta = None

    @classmethod
    def load_msh(cls, path: str, device: int = 0) -> "Database":
        """Parse the .msh on a helper thread (host only) while this thread creates the CUDA context."""
        import threading
        L = _abi.load()
        m, box = C.c_void_p(), {}

        def parse():
            try:
                check(L.hs_msh_open(path.encode(), C.byref(m)))     # hs_last_error() is thread local: check here
            except Exception as e:                                   # noqa: BLE001
                box["err"] = e

        th = threading.Thread(target=parse)
        th.start()
        try:
            _abi.init(device)
        finally:
            th.join()
        if "err" in box:
            raise box["err"]
        try:
            h = C.c_void_p()
            check(L.hs_db_from_msh(m, C.byref(h)))
        finally:
            L.hs_msh_free(m)
        return cls(h.value, device)

    def ref(self, i: int):
        """(name, comment, length, sketch size) of reference i."""
        nm, cm = C.c_char_p(), C.c_char_p()
        ln, nh = C.c_uint64(), C.c_uint64()
        check(_abi.load().hs_db_ref(self._h, i, C.byref(nm), C.byref(cm), C.byref(ln), C.byref(nh)))
        return ((nm.value or b"").decode("utf-8", "replace"), (cm.value or b"").decode("utf-8", "replace"), ln.value, nh.value)

    @classmethod
    def load_msh_multi(cls, paths, device: int = 0) -> "Database":
        """One table over several .msh files (row a3: run_hymet_cami.sh:85-97 screens sketch1-3.msh in
        turn); `segments` gives each file's reference range, `segment_s` its sketch size."""
        _abi.init(device)
        L = _abi.load()
        handles = []
        try:
            for p in paths:
                m = C.c_void_p()
                check(L.hs_msh_open(str(p).encode(), C.byref(m)))
                handles.append(m)
            arr = (C.c_void_p * len(handles))(*[m.value for m in handles])
            h = C.c_void_p()
            check(L.hs_db_from_msh_multi(arr, len(handles), C.byref(h)))
        finally:
            for m in handles:
                L.hs_msh_free(m)
        return cls(h.value, device)

    @property
    def segments(self):
        """[(first reference, one past the last)] per source file."""
        n = C.c_uint32()
        check(_abi.load().hs_db_segments(self._h, C.byref(n), None, None))
        rb = np.zeros(n.value + 1, np.uint64)
        ss = np.zeros(n.value, np.uint32)
        check(_abi.load().hs_db_segments(self._h, C.byref(n), _ptr(rb, C.c_uint64), _ptr(ss, C.c_uint32)))
        self.segment_s = [int(x) for x in ss]
        return [(int(rb[j]), int(rb[j + 1])) for j in range(n.value)]

    @classmethod
    def from_arrays(cls, k: int, s: int, seed: int, offsets, hashes, lengths=None, device: int = 0) -> "Database":
        _abi.init(device)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        hashes = np.ascontiguousarray(hashes, np.uint64)
        n = len(offsets) - 1
        ln = None if lengths is None else np.ascontiguousarray(lengths, np.uint64)
        h = C.c_void_p()
        check(_abi.load().hs_db_from_arrays(k, s, seed, n, _ptr(offsets, C.c_uint64),
                                            _ptr(hashes, C.c_uint64) if len(hashes) else None,
                                            _ptr(ln, C.c_uint64) if ln is not None else None, C.byref(h)))
        return cls(h.value, device)

    def _load_meta(self):
        if self._meta is None:
            L = _abi.load()
            names, comments = [], []
            lengths = np.zeros(self.n_refs, np.uint64)
            sizes = np.zeros(self.n_refs, np.uint64)
            nm, cm = C.c_char_p(), C.c_char_p()
            ln, nh = C.c_uint64(), C.c_uint64()
            for i in range(self.n_refs):
                check(L.hs_db_ref(self._h, i, C.byref(nm), C.byref(cm), C.byref(ln), C.byref(nh)))
                names.append((nm.value or b"").decode("utf-8", "replace"))
                comments.append((cm.value or b"").decode("utf-8", "replace"))
                lengths[i], sizes[i] = ln.value, nh.value
            self._meta = (names, comments, lengths, sizes)
        return self._meta

    @property
    def names(self) -> List[str]: return self._load_meta()[0]
    @property
    def comments(self) -> List[str]: return self._load_meta()[1]
    @property
    def lengths(self) -> np.ndarray: return self._load_meta()[2]
    @property
    def sizes(self) -> np.ndarray: return self._load_meta()[3]

    def entry_ids(self) -> np.ndarray:
        out = np.zeros(max(self.n_entries, 1), np.uint32)
        check(_abi.load().hs_db_entry_ids(self._h, _ptr(out, C.c_uint32)))
        return out[:self.n_entries]

    def probe(self, hashes) -> np.ndarray:
        """K2 alone: canonical entry id (or 0xFFFFFFFF) for each hash."""
        hashes = np.ascontiguousarray(hashes, np.uint64)
        out = np.zeros(max(len(hashes), 1), np.uint32)
        check(_abi.load().hs_db_probe(self._h, _ptr(hashes, C.c_uint64), len(hashes), _ptr(out, C.c_uint32)))
        return out[:len(hashes)]

    def probe_device(self, d_hashes_ptr: int, n: int):
        hits, reads, ms = C.c_uint64(), C.c_uint64(), C.c_float()
        check(_abi.load().hs_db_probe_device(self._h, C.c_void_p(d_hashes_ptr), n, C.byref(hits), C.byref(reads),
                                             C.byref(ms)))
        return hits.value, reads.value, ms.value

    def close(self):
        if self._h:
            _abi.load().hs_db_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Screen:
    """One query stream against a Database (rows a6-a15)."""

    def __init__(self, db: Database, *, stream_ptr: Optional[int] = None, probe_filter: bool = True):
        self.db = db
        self._h = C.c_void_p()
        check(_abi.load().hs_screen_new(db._h, C.byref(self._h)))
        if stream_ptr is not None:
            check(_abi.load().hs_screen_set_stream(self._h, C.c_void_p(stream_ptr)))
        if not probe_filter:
            self.set_option("filter", 0)
        self._keep = []  # keeps caller buffers of in-place device feeds alive

    def set_option(self, key: str, value: int):
        check(_abi.load().hs_screen_set_option(self._h, key.encode(), int(value)))

    def set_stream(self, stream_ptr: Optional[int]):
        check(_abi.load().hs_screen_set_stream(self._h, C.c_void_p(stream_ptr) if stream_ptr else None))

    # ---- streaming -------------------------------------------------------
    def feed_fasta(self, path: str, threads: int = 1):
        check(_abi.load().hs_screen_feed_fasta(self._h, path.encode(), threads))

    def feed_text(self, text, threads: int = 1):
        """FASTA/FASTQ text in host memory: bytes, bytearray, memoryview or uint8 ndarray."""
        if isinstance(text, np.ndarray):
            assert text.dtype == np.uint8 and text.flags.c_contiguous
            p, n = text.ctypes.data, text.size
        else:
            if not isinstance(text, bytes):
                text = bytes(text)
            keep = C.c_char_p(text)  # the call returns after the host packers are done with it
            p, n = C.cast(keep, C.c_void_p).value, len(text)
        check(_abi.load().hs_screen_feed_text(self._h, C.c_void_p(p), n, threads))

    def feed_text_ptr(self, ptr: int, n: int, threads: int = 1):
        check(_abi.load().hs_screen_feed_text(self._h, C.c_void_p(ptr), n, threads))

    def feed_packed(self, seq2: np.ndarray, inv: np.ndarray, n_bases: int):
        assert seq2.dtype == np.uint64 and inv.dtype == np.uint32
        assert len(seq2) * 32 >= n_bases and len(inv) * 32 >= n_bases
        check(_abi.load().hs_screen_feed_packed(self._h, C.c_void_p(seq2.ctypes.data), C.c_void_p(inv.ctypes.data),
                                                n_bases))

    def feed_packed_ptr(self, seq_ptr: int, inv_ptr: int, n_bases: int):
        """Packed HOST buffers given as raw addresses (e.g. pinned torch tensors)."""
        check(_abi.load().hs_screen_feed_packed(self._h, C.c_void_p(seq_ptr), C.c_void_p(inv_ptr), n_bases))

    def feed_packed_device(self, d_seq_ptr: int, d_inv_ptr: int, n_bases: int, keepalive=None):
        if keepalive is not None:
            self._keep.append(keepalive)
        check(_abi.load().hs_screen_feed_packed_device(self._h, C.c_void_p(d_seq_ptr), C.c_void_p(d_inv_ptr), n_bases))

    # ---- multi-GPU seam ----------------------------------------------------
    def flush(self):
        check(_abi.load().hs_screen_flush(self._h))

    def flush_async(self):
        """Enqueue the bottom-s selection without waiting; the next finish completes the flush."""
        check(_abi.load().hs_screen_flush_async(self._h))

    def counts_devptr(self):
        p, n = C.c_void_p(), C.c_uint64()
        check(_abi.load().hs_screen_counts_devptr(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def counts_compact_async(self, d_pairs_ptr: int, cap: int, d_n_out_ptr: int):
        check(_abi.load().hs_screen_counts_compact_async(self._h, C.c_void_p(d_pairs_ptr), cap, C.c_void_p(d_n_out_ptr)))

    def counts_absorb(self, d_rows_ptr: int, n_rows: int, cap: int, skip_row: int):
        """All ranks' pair records (device memory, after the all-gather) added in one launch."""
        check(_abi.load().hs_screen_counts_absorb(self._h, C.c_void_p(d_rows_ptr), n_rows, cap, skip_row))

    def mixture_record(self, d_record_ptr: int):
        """[length | s hashes] of the settled local mixture -> device memory ((s + 1) int64 words)."""
        check(_abi.load().hs_screen_mixture_record(self._h, C.c_void_p(d_record_ptr)))

    def mixture_merge_device(self, d_rows_ptr: int, n_rows: int):
        check(_abi.load().hs_screen_mixture_merge_device(self._h, C.c_void_p(d_rows_ptr), n_rows))

    def mixture(self) -> np.ndarray:
        out = np.zeros(max(self.db.s, 1), np.uint64)
        n = C.c_uint32()
        check(_abi.load().hs_screen_mixture_get(self._h, _ptr(out, C.c_uint64), C.byref(n)))
        return out[:n.value].copy()

    def segment_set_size(self, segment: int) -> int:
        v = C.c_uint64()
        check(_abi.load().hs_screen_segment_set_size(self._h, segment, C.byref(v)))
        return v.value

    # ---- reduction ---------------------------------------------------------
    def finish(self, wta: bool = False) -> ScreenResult:
        n = max(self.db.n_refs, 1)
        shared = np.zeros(n, np.uint64); median = np.zeros(n, np.uint32)
        ident = np.zeros(n, np.float64); pv = np.zeros(n, np.float64)
        st = _abi.Stats()
        check(_abi.load().hs_screen_finish(self._h, int(wta), _ptr(shared, C.c_uint64), _ptr(median, C.c_uint32),
                                           _ptr(ident, C.c_double), _ptr(pv, C.c_double), C.byref(st)))
        N = self.db.n_refs
        return ScreenResult(shared[:N], median[:N], ident[:N], pv[:N], int(st.set_size), st.asdict())

    def finish_hits(self, wta: bool = False) -> ScreenHits:
        """Rows a11-a16 for the references with shared > 0 only (what the TSV holds): O(hits) on the way home."""
        L = _abi.load()
        n, st = C.c_uint32(), _abi.Stats()
        check(L.hs_screen_finish_hits(self._h, int(wta), C.byref(n), C.byref(st)))
        h = max(n.value, 1)
        ref = np.zeros(h, np.uint32); shared = np.zeros(h, np.uint64); median = np.zeros(h, np.uint32)
        ident = np.zeros(h, np.float64); pv = np.zeros(h, np.float64)
        check(L.hs_screen_hits_copy(self._h, n.value, _ptr(ref, C.c_uint32), _ptr(shared, C.c_uint64), _ptr(median, C.c_uint32),
                                    _ptr(ident, C.c_double), _ptr(pv, C.c_double)))
        k = n.value
        return ScreenHits(ref[:k], shared[:k], median[:k], ident[:k], pv[:k], int(st.set_size), st.asdict())

    def stats(self) -> dict:
        st = _abi.Stats()
        check(_abi.load().hs_screen_stats(self._h, C.byref(st)))
        return st.asdict()

    def reset(self):
        check(_abi.load().hs_screen_reset(self._h))
        self._keep.clear()

    def close(self):
        if self._h:
            _abi.load().hs_screen_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def host_placement() -> dict:
    """Where hs_init left the calling thread: the GPU's NUMA node and the CPUs it may use."""
    node, cpus = C.c_int(), C.c_int()
    check(_abi.load().hs_host_placement(C.byref(node), C.byref(cpus)))
    return {"numa_node": node.value, "cpus_after_numa_binding": cpus.value}


# ---- single stages (parity tests, per-kernel measurement) ---------------------
def packed_words(n_bases: int) -> int:
    return int(_abi.load().hs_packed_words(n_bases))


def pack_text(text: bytes):
    """Host packer alone (no GPU): -> (seq2 uint64[], inv uint32[], n_positions, stats)."""
    L = _abi.load()
    cap = len(text) // 32 + 4
    seq = np.zeros(cap, np.uint64); inv = np.zeros(cap, np.uint32)
    n = C.c_uint64(); st = _abi.Stats()
    check(L.hs_pack_text(text, len(text), C.c_void_p(seq.ctypes.data), C.c_void_p(inv.ctypes.data), cap,
                         C.byref(n), C.byref(st)))
    words = (n.value + 31) // 32
    return seq[:words], inv[:words], int(n.value), st.asdict()


def pack_text_device(text: bytes, device: int = 0):
    """Device FASTA parser alone: same outputs as pack_text()."""
    _abi.init(device)
    cap = packed_words(len(text)) + 4
    seq = np.zeros(cap, np.uint64); inv = np.zeros(cap, np.uint32)
    n = C.c_uint64(); st = _abi.Stats()
    check(_abi.load().hs_pack_text_device(text, len(text), C.c_void_p(seq.ctypes.data), C.c_void_p(inv.ctypes.data), cap,
                                          C.byref(n), C.byref(st)))
    words = (n.value + 31) // 32
    return seq[:words], inv[:words], int(n.value), st.asdict()


def hash_packed(k: int, seed: int, seq2: np.ndarray, inv: np.ndarray, n_bases: int, device: int = 0):
    """K1 alone: (hash, valid) indexed by the position of each k-mer's last base."""
    _abi.init(device)
    h = np.zeros(max(n_bases, 1), np.uint64); v = np.zeros(max(n_bases, 1), np.uint8)
    check(_abi.load().hs_hash_packed(k, seed, C.c_void_p(seq2.ctypes.data), C.c_void_p(inv.ctypes.data), n_bases,
                                     _ptr(h, C.c_uint64), _ptr(v, C.c_uint8)))
    return h[:n_bases], v[:n_bases].astype(bool)


def stat_batch(k: int, set_size: int, shared, size, device: int = 0):
    """K6 alone: identity and p-value for (shared, sketch size) pairs."""
    _abi.init(device)
    shared = np.ascontiguousarray(shared, np.uint64); size = np.ascontiguousarray(size, np.uint64)
    n = len(shared)
    ident = np.zeros(max(n, 1), np.float64); pv = np.zeros(max(n, 1), np.float64)
    check(_abi.load().hs_stat_batch(k, set_size, n, _ptr(shared, C.c_uint64), _ptr(size, C.c_uint64),
                                    _ptr(ident, C.c_double), _ptr(pv, C.c_double)))
    return ident[:n], pv[:n]


def sketch_text(text: bytes, k: int, s: int, seed: int = 42, device: int = 0):
    """`mash sketch` of one genome (FASTA text): (s smallest distinct hashes, total bases)."""
    _abi.init(device)
    out = np.zeros(max(s, 1), np.uint64)
    n = C.c_uint32(); ln = C.c_uint64()
    check(_abi.load().hs_sketch_text(k, s, seed, text, len(text), _ptr(out, C.c_uint64), C.byref(n), C.byref(ln)))
    return out[:n.value].copy(), int(ln.value)


@dataclass
class GenomeSketch:
    """One input of `sketch_files`: what its .msh entry is made of."""
    hashes: np.ndarray     # uint64, ascending, <= s
    length: int            # sequence bases
    n_records: int         # occurrences of "\n>" plus one if the text starts with '>'
    header: bytes          # first header line after its '>' (empty unless the text starts with '>')


def sketch_files(paths: Sequence[str], k: int, s: int, seed: int = 42, threads: int = 1, device: int = 0):
    """`mash sketch` of a collection: one sketch per file (plain or gzip FASTA/FASTQ), many genomes per
    kernel pass, `threads` host threads reading and packing.  Returns ([GenomeSketch] in input order, stats)."""
    _abi.init(device)
    L = _abi.load()
    h = C.c_void_p()
    check(L.hs_sketcher_new(k, s, seed, threads, C.byref(h)))
    try:
        for p in paths:
            check(L.hs_sketcher_add_file(h, os.fsencode(p)))
        check(L.hs_sketcher_run(h))
        out = []
        hp, n, ln, nrec, hdr, hl = _abi.u64p(), C.c_uint32(), C.c_uint64(), C.c_uint64(), C.c_void_p(), C.c_uint64()
        for i in range(len(paths)):
            check(L.hs_sketcher_result(h, i, C.byref(hp), C.byref(n), C.byref(ln), C.byref(nrec), C.byref(hdr), C.byref(hl)))
            hashes = np.ctypeslib.as_array(hp, shape=(n.value,)).copy() if n.value else np.zeros(0, np.uint64)
            out.append(GenomeSketch(hashes, int(ln.value), int(nrec.value), C.string_at(hdr, hl.value) if hl.value else b""))
        st = _abi.SketchStats()
        check(L.hs_sketcher_stats(h, C.byref(st)))
        return out, st.asdict()
    finally:
        L.hs_sketcher_free(h)


def gather_bench(d_buf_ptr: int, nbytes: int, n_reads: int) -> float:
    """ms for n_reads independent random 32-byte sector reads over a device buffer."""
    ms = C.c_float()
    check(_abi.load().hs_gather_bench(C.c_void_p(d_buf_ptr), nbytes, n_reads, C.byref(ms)))
    return ms.value


def sketch_packed_device(d_seq_ptr: int, d_inv_ptr: int, n_bases: int, k: int, s: int, seed: int = 42):
    out = np.zeros(max(s, 1), np.uint64)
    n = C.c_uint32()
    check(_abi.load().hs_sketch_packed_device(k, s, seed, C.c_void_p(d_seq_ptr), C.c_void_p(d_inv_ptr), n_bases,
                                              _ptr(out, C.c_uint64), C.byref(n)))
    return out[:n.value].copy()


def pack_codes_device(d_codes_ptr: int, n: int, d_seq_ptr: int, d_inv_ptr: int, stream_ptr: int = 0):
    """uint8 base codes in HBM -> packed words in HBM (both caller-allocated)."""
    check(_abi.load().hs_pack_codes_device(C.c_void_p(d_codes_ptr), n, C.c_void_p(d_seq_ptr), C.c_void_p(d_inv_ptr),
                                           C.c_void_p(stream_ptr) if stream_ptr else None))


def read_msh_host(path: str):
    """The product's C++ .msh parser alone (no GPU): dict of arrays."""
    L = _abi.load()
    h = C.c_void_p()
    check(L.hs_msh_open(path.encode(), C.byref(h)))
    try:
        info = _abi.DbInfo()
        check(L.hs_msh_info(h, C.byref(info)))
        names, comments, lengths, hashes, offs = [], [], [], [], [0]
        nm, cm = C.c_char_p(), C.c_char_p()
        ln, nh = C.c_uint64(), C.c_uint64()
        hp = _abi.u64p()
        for i in range(info.n_refs):
            check(L.hs_msh_ref(h, i, C.byref(nm), C.byref(cm), C.byref(ln), C.byref(nh), C.byref(hp)))
            names.append((nm.value or b"").decode()); comments.append((cm.value or b"").decode())
            lengths.append(ln.value)
            hashes.append(np.ctypeslib.as_array(hp, shape=(nh.value,)).copy() if nh.value else np.zeros(0, np.uint64))
            offs.append(offs[-1] + nh.value)
        return dict(k=info.k, s=info.s, seed=info.seed, use64=bool(info.use64), names=names, comments=comments,
                    lengths=np.array(lengths, np.uint64), offsets=np.array(offs, np.uint64),
                    hashes=np.concatenate(hashes) if hashes else np.zeros(0, np.uint64), max_key=info.max_key)
    finally:
        L.hs_msh_free(h)

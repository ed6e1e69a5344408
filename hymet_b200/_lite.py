"""numpy-free binding for the one-shot `mash screen` process (hymet_b200/cli.py).

A `mash screen` invocation on C2 is about one second of wall clock, 0.1-0.4 s of which was
`import numpy`.  The CLI needs none of it: the four result columns are plain C arrays and the
TSV formatter walks them once.  Same C ABI, same reporting rules (S15/S16) as
hymet_b200/screen.py + hymet_b200/tsv.py; tests/test_gpu_parity.py compares the CLI's bytes with
the oracle CLI's.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import Iterator, List

from . import _abi
from ._abi import HsError, check  # noqa: F401  (re-exported)


DEVICE_ERRORS = (-2, -3, -6)     # HS_ENODEV, HS_ECUDA, HS_ENOMEM: the GPU path itself is unavailable (never a data problem)


class LiteMsh:
    """Sketch files parsed on the host (hs_msh_open): `handles` maps the index of every path that loaded to
    its handle, `errors` the others to messages (tolerate=True) -- one parse serves the tables of every GPU."""

    def __init__(self, paths, tolerate: bool = False):
        L = _abi.load()
        self.paths, self.handles, self.errors, self.fatal = list(paths), {}, {}, None
        for i, p in enumerate(self.paths):
            try:
                m = C.c_void_p()
                check(L.hs_msh_open(p.encode(), C.byref(m)))   # hs_last_error() is thread local: check on the parsing thread
                self.handles[i] = m
            except HsError as e:
                if not tolerate:
                    self.fatal = e
                    return
                self.errors[i] = e.msg

    def close(self):
        for m in self.handles.values():
            _abi.load().hs_msh_free(m)
        self.handles = {}


class LiteDb:
    def __init__(self, path, device: int, tolerate: bool = False, msh: LiteMsh = None):
        """`path`: one .msh, or a list of them for one table over several files (hs_db_from_msh_multi).
        The files are parsed on a helper thread (host only) while this thread creates the CUDA context.
        tolerate=True (list form): a file that cannot be opened or parsed is left out instead of failing
        the whole table; `loaded` lists the indices that made it, `errors` maps the others to messages.
        msh: files already parsed (several GPUs build their copy of the table from one parse)."""
        L = _abi.load()
        paths = [path] if isinstance(path, str) else list(path)
        box = {}
        own = msh is None

        def parse():
            box["msh"] = LiteMsh(paths, tolerate)

        if own:
            th = threading.Thread(target=parse)
            th.start()
            try:
                _abi.init(device)
            finally:
                th.join()
            msh = box["msh"]
        else:
            _abi.init(device)
        self.errors = dict(msh.errors)
        self._h = C.c_void_p()
        self.loaded = sorted(msh.handles)
        try:
            if msh.fatal is not None:
                raise msh.fatal
            if isinstance(path, str):
                check(L.hs_db_from_msh(msh.handles[0], C.byref(self._h)))
            elif self.loaded:
                arr = (C.c_void_p * len(self.loaded))(*[msh.handles[i].value for i in self.loaded])
                check(L.hs_db_from_msh_multi(arr, len(self.loaded), C.byref(self._h)))
        finally:
            if own:
                msh.close()
        self.info = _abi.DbInfo()
        self.n_refs = self.n_distinct = 0
        if self._h:
            check(L.hs_db_info(self._h, C.byref(self.info)))
            self.n_refs = int(self.info.n_refs)
            self.n_distinct = int(self.info.n_distinct)

    @property
    def segments(self):
        """[(first reference, one past the last)] per source file."""
        L = _abi.load()
        n = C.c_uint32()
        check(L.hs_db_segments(self._h, C.byref(n), None, None))
        rb = (C.c_uint64 * (n.value + 1))()
        check(L.hs_db_segments(self._h, C.byref(n), rb, None))
        return [(int(rb[j]), int(rb[j + 1])) for j in range(n.value)]

    def ref(self, i: int):
        nm, cm = C.c_char_p(), C.c_char_p()
        ln, nh = C.c_uint64(), C.c_uint64()
        check(_abi.load().hs_db_ref(self._h, i, C.byref(nm), C.byref(cm), C.byref(ln), C.byref(nh)))
        return ((nm.value or b"").decode("utf-8", "replace"), (cm.value or b"").decode("utf-8", "replace"), ln.value, nh.value)

    def close(self):
        if self._h:
            _abi.load().hs_db_free(self._h)
            self._h = C.c_void_p()


class LiteScreen:
    def __init__(self, db: LiteDb, probe_filter: bool = True):
        self.db = db
        self._cols = None
        self._hits = None
        self._h = C.c_void_p()
        check(_abi.load().hs_screen_new(db._h, C.byref(self._h)))
        if not probe_filter:
            check(_abi.load().hs_screen_set_option(self._h, b"filter", 0))

    def feed_fasta(self, path: str, threads: int):
        check(_abi.load().hs_screen_feed_fasta(self._h, path.encode(), threads))

    def feed_fasta_range(self, path: str, begin: int, end: int, threads: int):
        check(_abi.load().hs_screen_feed_fasta_range(self._h, path.encode(), begin, end, threads))

    def absorb(self, others: List["LiteScreen"]):
        """Add other GPUs' counts and mixtures (all flushed) into this screen, in one call."""
        arr = (C.c_void_p * len(others))(*[o._h.value for o in others])
        check(_abi.load().hs_screen_absorb_screens(self._h, arr, len(others)))

    def set_option(self, key: str, value: int):
        check(_abi.load().hs_screen_set_option(self._h, key.encode(), int(value)))

    def reset(self):
        """Forget the query; the handle (arena, pinned ring, result rows) stays allocated."""
        check(_abi.load().hs_screen_reset(self._h))
        self._cols = self._hits = None

    def close(self):
        if self._h:
            _abi.load().hs_screen_free(self._h)
            self._h = C.c_void_p()

    def flush(self):
        check(_abi.load().hs_screen_flush(self._h))

    def stats(self) -> dict:
        st = _abi.Stats()
        check(_abi.load().hs_screen_stats(self._h, C.byref(st)))
        return st.asdict()

    def finish_lines(self, wta: bool, min_identity: float, max_pvalue: float, begin: int = 0, end: int = None) -> Iterator[str]:
        """Rows a11-a16: reduce (once), then the TSV lines of references [begin, end) in sketch order
        (S15: keep iff (shared > 0 or -i < 0) and identity >= -i and p <= -v; numbers as C `%g`).
        Unless -i < 0 asks for every reference, only the rows with shared > 0 ever leave the GPU."""
        L = _abi.load()
        end = self.db.n_refs if end is None else end
        if min_identity < 0.0:
            if self._cols is None:
                n = max(self.db.n_refs, 1)
                cols = ((C.c_uint64 * n)(), (C.c_uint32 * n)(), (C.c_double * n)(), (C.c_double * n)())
                check(L.hs_screen_finish(self._h, int(wta), cols[0], cols[1], cols[2], cols[3], None))
                self._cols = cols
            shared, median, identity, pvalue = self._cols
            rows = ((i, i) for i in range(begin, end))
        else:
            if self._hits is None:
                n = C.c_uint32()
                check(L.hs_screen_finish_hits(self._h, int(wta), C.byref(n), None))
                h = max(n.value, 1)
                hits = ((C.c_uint32 * h)(), (C.c_uint64 * h)(), (C.c_uint32 * h)(), (C.c_double * h)(), (C.c_double * h)(), n.value)
                check(L.hs_screen_hits_copy(self._h, n.value, hits[0], hits[1], hits[2], hits[3], hits[4]))
                self._hits = hits
            ref, shared, median, identity, pvalue, n = self._hits
            rows = ((q, ref[q]) for q in range(n) if begin <= ref[q] < end)
        for q, i in rows:
            sh = shared[q]
            if not sh and min_identity >= 0.0:
                continue
            ident, p = identity[q], pvalue[q]
            if ident < min_identity or p > max_pvalue:
                continue
            name, comment, _, size = self.db.ref(i)
            yield "%s\t%d/%d\t%d\t%s\t%s\t%s\n" % ("%g" % ident, sh, size, median[q], "%g" % p, name, comment)


def is_plain_fasta_file(path: str) -> bool:
    """What hs_screen_feed_fasta_range accepts: a regular file whose first non-blank byte is '>'."""
    import os
    try:
        if path == "-" or not os.path.isfile(path):
            return False
        with open(path, "rb") as fh:
            head = fh.read(256).lstrip(b"\r\n")
        return head[:1] == b">"
    except OSError:
        return False


class MultiGpu:
    """HYMET_SCREEN_GPUS=N for the one-process drop-in (SURVEY.md 8b, 8e): the sketch files are parsed once,
    every GPU builds its own copy of the table (one thread per GPU), streams its byte range of every plain
    FASTA input -- records are never cut, inputs that cannot be cut (gzip, FASTQ, stdin) go whole to one
    GPU in turn -- and GPU 0 absorbs the others' counts and mixtures device to device, then reduces."""

    def __init__(self, path, devices, tolerate: bool = False):
        self.devices = list(devices)
        paths = [path] if isinstance(path, str) else list(path)
        box = {}
        th = threading.Thread(target=lambda: box.update(msh=LiteMsh(paths, tolerate)))
        th.start()
        try:
            _abi.init(self.devices[0])
        finally:
            th.join()
        msh = box["msh"]
        self.dbs = [None] * len(self.devices)
        errs = [None] * len(self.devices)

        def build(i):
            try:
                self.dbs[i] = LiteDb(path, self.devices[i], tolerate, msh=msh)
            except Exception as e:                                  # noqa: BLE001
                errs[i] = e

        ths = [threading.Thread(target=build, args=(i,)) for i in range(len(self.devices))]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        msh.close()
        for e in errs:
            if e is not None:
                raise e
        self.db = self.dbs[0]

    def screen(self, inputs: List[str], threads: int, probe_filter: bool = True) -> "LiteScreen":
        """Stream `inputs` across the GPUs; returns GPU 0's screen, flushed, holding everybody's counts."""
        import os
        n = len(self.devices)
        scrs = [None] * n
        errs = [None] * n
        per = max(1, threads // n)
        whole = [p for p in inputs if not is_plain_fasta_file(p)]

        def work(i):
            try:
                _abi.init(self.devices[i])
                scr = LiteScreen(self.dbs[i], probe_filter)
                scrs[i] = scr
                for p in inputs:
                    if p in whole:
                        if whole.index(p) % n == i:
                            scr.feed_fasta(p, per)
                        continue
                    size = os.path.getsize(p)
                    scr.feed_fasta_range(p, size * i // n, size * (i + 1) // n, per)
                scr.flush()
            except Exception as e:                                  # noqa: BLE001
                errs[i] = e

        ths = [threading.Thread(target=work, args=(i,)) for i in range(n)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        for e in errs:
            if e is not None:
                raise e
        if n > 1:
            scrs[0].absorb(scrs[1:])
        for scr in scrs[1:]:
            scr.close()
        return scrs[0]


def screen_lines(db_path: str, inputs: List[str], threads: int, wta: bool, min_identity: float, max_pvalue: float,
                 device: int, probe_filter: bool = True):
    """Convenience used by tests: the whole screen as a list of TSV lines."""
    db = LiteDb(db_path, device)
    scr = LiteScreen(db, probe_filter)
    for p in inputs:
        scr.feed_fasta(p, threads)
    return list(scr.finish_lines(wta, min_identity, max_pvalue))

#!/usr/bin/env python
"""Scratch: where does the end-to-end time go -- host packer rate per thread count, feed/finish wall
time per ingest mode and span size, and (HYMET_SCREEN_DEBUG_TIMING=1) the per-span timeline."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from hymet_b200 import screen as hs, workload

mbp = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
wl = workload.make_c2(0, mbp=mbp, n_sketches=50000, n_real=64, with_fasta=True, with_host_packed=False)
db = hs.Database.from_arrays(wl.k, wl.s, 42, wl.offsets, wl.hashes, wl.lengths)
scr = hs.Screen(db)
nthreads = len(os.sched_getaffinity(0))
print("cpus", nthreads, "text bytes", wl.fasta.numel(), flush=True)
for rep in range(3):
    scr.reset(); scr.feed_packed_device(wl.d_seq.data_ptr(), wl.d_inv.data_ptr(), wl.n_positions); r = scr.finish_hits()
print("resident: stream %.3f ms (%.1f Gbp/s) reduce %.3f" % (r.stats["ms_stream"], wl.n_bases / r.stats["ms_stream"] / 1e6, r.stats["ms_reduce"]), flush=True)

def run(label, thr, reps=4):
    best = None
    for rep in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        scr.reset()
        scr.feed_text_ptr(wl.fasta.data_ptr(), wl.fasta.numel(), thr)
        t1 = time.perf_counter()
        r = scr.finish_hits()
        t2 = time.perf_counter()
        if rep and (best is None or t2 - t0 < best[0]):
            best = (t2 - t0, t1 - t0, t2 - t1, r.stats)
    tot, feed, fin, st = best
    print("%-34s thr=%2d total %6.2f ms feed %6.2f finish %5.2f -> %6.1f Gbp/s  launches %4d stream %5.2f ms h2d %4d MB" % (
        label, thr, 1e3 * tot, 1e3 * feed, 1e3 * fin, wl.n_bases / tot / 1e9, st["n_launches"], st["ms_stream"], st["h2d_bytes"] >> 20), flush=True)

for mode, name in ((0, "host"), (2, "hybrid"), (1, "device")):
    scr.set_option("ingest", mode)
    for chunk in (16,):
        scr.set_option("chunk_bases", chunk << 20)
        for thr in (nthreads,):
            run("%s chunk %2d MB" % (name, chunk), thr)
        if mode == 1:
            break
scr.set_option("ingest", 2); scr.set_option("chunk_bases", 16 << 20)

# the same text as a FILE in the page cache
import tempfile
fdir = tempfile.mkdtemp(prefix="hs_e2e_")
fpath = os.path.join(fdir, "contigs.fna")
wl.fasta.numpy().tofile(fpath)
def run_file(label, thr, reps=4):
    best = None
    for rep in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        scr.reset()
        scr.feed_fasta(fpath, thr)
        t1 = time.perf_counter()
        r = scr.finish_hits()
        t2 = time.perf_counter()
        if rep and (best is None or t2 - t0 < best[0]):
            best = (t2 - t0, t1 - t0, t2 - t1, r.stats)
    tot, feed, fin, st = best
    print("%-34s thr=%2d total %6.2f ms feed %6.2f finish %5.2f -> %6.1f Gbp/s  launches %4d stream %5.2f ms h2d %4d MB" % (
        label, thr, 1e3 * tot, 1e3 * feed, 1e3 * fin, wl.n_bases / tot / 1e9, st["n_launches"], st["ms_stream"], st["h2d_bytes"] >> 20), flush=True)
scr.set_option("file_mode", 0); scr.set_option("file_readers", 8); scr.set_option("file_block_bytes", 16 << 20)
run_file("file: pread ring + device parser", nthreads)
scr.set_option("file_mode", 1)
for chunk in (8, 16):
    scr.set_option("chunk_bases", chunk << 20)
    run_file("file: mmap + host packers %d MB" % chunk, nthreads)
os.remove(fpath); os.rmdir(fdir)
scr.set_option("ingest", 0); scr.set_option("chunk_bases", 16 << 20)

# host packer alone on the pinned text, per thread count and level
import ctypes as C, threading
L = hs._abi.load()
txt = wl.fasta.numpy()
n = txt.size
def pack_range(b, e, out):
    cap = (e - b) // 32 + 4
    seq = np.empty(cap, np.uint64); inv = np.empty(cap, np.uint32); nb = C.c_uint64()
    seq[:] = 0; inv[:] = 0
    t0 = time.perf_counter()
    L.hs_pack_text(C.c_void_p(txt.ctypes.data + b), e - b, C.c_void_p(seq.ctypes.data), C.c_void_p(inv.ctypes.data), cap, C.byref(nb), None)
    out.append(time.perf_counter() - t0)
for thr in (1, 4, 8, nthreads):
    sl = n // 4 if thr < 8 else n       # keep the single-thread runs short
    outs = []; ths = []
    for i in range(thr):
        ths.append(threading.Thread(target=pack_range, args=(i * sl // thr, (i + 1) * sl // thr, outs)))
    t0 = time.perf_counter()
    [t.start() for t in ths]; [t.join() for t in ths]
    dt = time.perf_counter() - t0
    print("pack only, %2d threads: %.1f ms wall -> %.2f GB/s aggregate (slowest thread busy %.1f ms)" % (thr, 1e3 * dt, sl / dt / 1e9, 1e3 * max(outs)), flush=True)
if os.environ.get("HYMET_SCREEN_DEBUG_TIMING"):
    scr.reset(); scr.feed_text_ptr(wl.fasta.data_ptr(), wl.fasta.numel(), nthreads); scr.finish()

#!/usr/bin/env python3
"""`mash dist` on the GPU (DESIGN.md §5 "mash dist"): three seeded workloads, one JSON line each.

  W1  all-vs-all of a C2-shaped collection: 50 000 sketches at s = 1000 (500 clustered genomes sketched on
      the GPU plus decoys), -d 0.05.  Device ms per kernel, candidate pairs and pairs/s, the whole
      `bin/mash dist` process's wall clock, parity against the C oracle on a query sample and the
      oracle's CPU time on it (the oracle is a restatement of Mash, not Mash, unless a real mash ran).
  W2  every pair a candidate: 4 000 members of 20 clusters of one root.  Merge-bound: bytes the merges
      read (8 x (denom + common) per pair: both lists up to union rank s_p) over merge time.
  W3  unfiltered output, 5 000 x 5 000: writer lines/s at -p 1 and -p 16.

Sketch files go to a temporary directory.  The card name and power limit are read in the same process.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hymet_b200 import distance as dist  # noqa: E402
from hymet_b200 import msh as mshfmt  # noqa: E402
from hymet_b200 import screen as hs  # noqa: E402
from hymet_b200 import synth  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def write_db(path, k, s, sketches, lengths):
    offsets = np.concatenate([[0], np.cumsum([len(x) for x in sketches])]).astype(np.uint64)
    n = len(sketches)
    db = mshfmt.SketchDB(k=k, s=s, names=[synth.gcf_name(i) for i in range(n)], comments=[""] * n,
                         lengths=np.asarray(lengths, np.uint64), offsets=offsets,
                         hashes=np.concatenate([np.asarray(x, np.uint64) for x in sketches]))
    mshfmt.write_msh(path, db)
    return path


def perturb(rng, base, frac, s):
    keep = base[rng.random(len(base)) >= frac]
    fresh = np.unique(rng.integers(0, np.iinfo(np.uint64).max, size=s, dtype=np.uint64, endpoint=True))
    fresh = fresh[fresh < base[-1]][: s - len(keep)]
    return np.unique(np.concatenate([keep, fresh]))[:s]


def w1(rng, d, n, n_real, s):
    sk, lens = [], []
    per = 10
    for a in range(n_real // per):
        anc = synth.random_genome(rng, int(rng.integers(200_000, 400_000)))
        for m, rate in enumerate((0.0, 0.001, 0.003, 0.01, 0.02, 0.03, 0.05, 0.08, 0.12, 0.2)[:per]):
            g = synth.mutate(anc, rate, rng) if rate else anc
            sk.append(hs.sketch_text(synth.to_fasta([g], "g"), 21, s)[0])
            lens.append(len(g))
    h, G = synth.decoy_sketches(rng, n - len(sk), s)
    sk += list(h)
    lens += list(G)
    return write_db(os.path.join(d, "w1.msh"), 21, s, sk, lens)


def w2(rng, d, n, clusters, s):
    root, G = synth.decoy_sketches(rng, 1, s)
    sk = []
    for c in range(clusters):
        anc = perturb(rng, root[0], 0.5, s)
        sk += [perturb(rng, anc, float(rng.uniform(0.05, 0.3)), s) for _ in range(n // clusters)]
    return write_db(os.path.join(d, "w2.msh"), 21, s, sk, [int(G[0])] * len(sk))


def in_process(path, max_d, threads=16, rows=False, fd=None):
    ref = dist.HostMsh(path)
    dd = dist.Distance(ref)
    try:
        q = dist.HostMsh(path)
        dd.add_msh(q)
        q.close()
        t0 = time.perf_counter()
        out = dd.run_rows(max_d) if rows else dd.run(fd, max_d, 1.0, False, False, threads)
        wall = time.perf_counter() - t0
        return out, dd.stats(), wall
    finally:
        dd.close()
        ref.close()


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="w1,w2,w3")
    ap.add_argument("--sample", type=int, default=100, help="W1: queries checked against the oracle")
    args = ap.parse_args()
    card = gpu_info()
    rng = np.random.default_rng(2026)
    with tempfile.TemporaryDirectory() as d:
        null = os.open(os.devnull, os.O_WRONLY)
        if "w1" in args.only:
            p = w1(rng, d, 50_000, 500, 1000)
            in_process(p, 0.05, rows=True)                                   # warm-up
            rows, st, wall = in_process(p, 0.05, rows=True)
            t0 = time.perf_counter()
            r = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "mash"), "dist", "-p", "16", "-d", "0.05", p, p],
                               stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
            proc = time.perf_counter() - t0
            assert r.returncode == 0, r.stderr
            from tests import _distance_ref as dref
            from tests import _oracle as orc
            db = orc.OracleDB.load_msh(p)
            sample = np.sort(rng.choice(50_000, args.sample, replace=False))
            t0 = time.perf_counter()
            common, denom, _ = dref.oracle_pairs(db, db, 1000, sample, threads=os.cpu_count() or 8)
            t_orc = time.perf_counter() - t0
            pos = {int(q): i for i, q in enumerate(sample)}
            sel = np.isin(rows.q, sample)
            qi = np.array([pos[int(q)] for q in rows.q[sel]], np.int64)
            ok = (np.array_equal(common[qi, rows.r[sel]], rows.common[sel])
                  and np.array_equal(denom[qi, rows.r[sel]], rows.denom[sel])
                  and int((common > 0).sum()) == int(sel.sum()))
            print(json.dumps({"workload": "W1", "card": card, "n": 50_000, "s": 1000, "max_d": 0.05,
                              "candidates": st["n_candidates"], "blocks": st["n_blocks"], "splits": st["n_splits"],
                              "ms_mark": round(st["ms_mark"], 3), "ms_compact": round(st["ms_compact"], 3),
                              "ms_merge": round(st["ms_merge"], 3),
                              "pairs_per_s_device": 2.5e9 / ((st["ms_mark"] + st["ms_compact"] + st["ms_merge"]) / 1e3),
                              "candidates_per_s_merge": st["n_candidates"] / (st["ms_merge"] / 1e3),
                              "run_s": round(wall, 3), "process_wall_s": round(proc, 3),
                              "oracle_sample_queries": args.sample, "oracle_parity": bool(ok),
                              "oracle_cpu_s_sample": round(t_orc, 3), "oracle_threads": os.cpu_count(),
                              "oracle_is": "C restatement of Mash 2.3 CommandDistance (no real mash here)"}), flush=True)
        if "w2" in args.only:
            p = w2(rng, d, 4000, 20, 1000)
            in_process(p, 1.0, rows=True)
            rows, st, wall = in_process(p, 1.0, rows=True)
            nbytes = 8.0 * float(rows.denom.astype(np.float64).sum() + rows.common.astype(np.float64).sum())
            print(json.dumps({"workload": "W2", "card": card, "n": 4000, "clusters": 20, "s": 1000,
                              "candidates": st["n_candidates"], "all_pairs": st["n_candidates"] == 4000 * 4000,
                              "blocks": st["n_blocks"], "splits": st["n_splits"],
                              "ms_mark": round(st["ms_mark"], 3), "ms_compact": round(st["ms_compact"], 3),
                              "ms_merge": round(st["ms_merge"], 3),
                              "merge_bytes_per_pair": nbytes / max(1, st["n_candidates"]),
                              "merge_GBps": nbytes / (st["ms_merge"] / 1e3) / 1e9,
                              "candidates_per_s_merge": st["n_candidates"] / (st["ms_merge"] / 1e3)}), flush=True)
        if "w3" in args.only:
            h, G = synth.decoy_sketches(rng, 5000, 1000)
            p = write_db(os.path.join(d, "w3.msh"), 21, 1000, list(h), list(G))
            for threads in (1, 16):
                _, st, wall = in_process(p, 1.0, threads=threads, fd=null)
                print(json.dumps({"workload": "W3", "card": card, "n": 5000, "threads": threads, "lines": st["n_lines"],
                                  "write_s": round(st["t_write_s"], 3), "lines_per_s": st["n_lines"] / st["t_write_s"],
                                  "run_s": round(wall, 3)}), flush=True)
        os.close(null)
    return 0


if __name__ == "__main__":
    sys.exit(main())

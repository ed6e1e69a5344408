#!/usr/bin/env python3
"""End-to-end `mash sketch` throughput on seeded genome collections.

Writes each collection once (plain and gzip) to a temporary directory, then runs `bin/mash sketch -l`
of every tree given with --tree (e.g. this one and a copy of an older one), alternating trees, at each
-p.  Reports genomes/s and Gbp/s per run, and from this tree's sketcher statistics the device time of
the hashing launches per Gbp and the host thread-seconds spent inflating and packing.  Prints one JSON
line per measurement; the card name and power limit are read in the same process.
"""
from __future__ import annotations

import argparse
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hymet_b200 import screen as hs  # noqa: E402
from hymet_b200 import synth  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def make_collection(d, name, n, lo, hi, seed, gz):
    rng = np.random.default_rng(seed)
    paths, bases = [], 0
    os.makedirs(os.path.join(d, name), exist_ok=True)
    for i in range(n):
        g = synth.random_genome(rng, int(rng.integers(lo, hi + 1)))
        text = synth.to_fasta([g], "g%d" % i)
        p = os.path.join(d, name, "g%06d.fna" % i + (".gz" if gz else ""))
        with (gzip.open(p, "wb", compresslevel=1) if gz else open(p, "wb")) as fh:
            fh.write(text)
        paths.append(p)
        bases += len(g)
    lst = os.path.join(d, name + ".txt")
    with open(lst, "w") as fh:
        fh.write("\n".join(paths) + "\n")
    return lst, paths, bases


def run_tree(tree, lst, paths, threads, out):
    args = [sys.executable, os.path.join(tree, "bin", "mash"), "sketch", "-p", str(threads), "-o", out]
    # an older tree may not know -l: hand it the paths themselves
    has_l = "-l " in subprocess.run(args[:3] + ["-h"], capture_output=True, text=True).stdout
    args += ["-l", lst] if has_l else paths
    t0 = time.perf_counter()
    r = subprocess.run(args, capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError("%s failed: %s" % (tree, r.stderr[-2000:]))
    return dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", action="append", default=[], help="repository trees to compare (default: this one)")
    ap.add_argument("--big", type=int, default=5000, help="genomes of 2 Mbp")
    ap.add_argument("--small", type=int, default=20000, help="genomes of 5-50 kb")
    ap.add_argument("--threads", default="1,16")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None, help="JSON lines file")
    a = ap.parse_args()
    trees = a.tree or [ROOT]
    card = gpu_info()
    rows = []
    with tempfile.TemporaryDirectory() as d:
        sets = []
        for gz in (False, True):
            if a.big:
                sets.append(("2Mbp" + (".gz" if gz else ""),) + make_collection(d, "big%d" % gz, a.big, 2_000_000, 2_000_000, 1, gz))
            if a.small:
                sets.append(("5-50kb" + (".gz" if gz else ""),) + make_collection(d, "small%d" % gz, a.small, 5_000, 50_000, 2, gz))
        for name, lst, paths, bases in sets:
            for threads in [int(x) for x in a.threads.split(",")]:
                # this tree's sketcher statistics: device time per Gbp, host inflate + pack
                _, st = hs.sketch_files(paths, 21, 1000, threads=threads)
                for rep in range(a.reps):
                    for tree in trees:
                        dt = run_tree(tree, lst, paths, threads, os.path.join(d, "out"))
                        row = dict(collection=name, tree=tree, threads=threads, rep=rep, genomes=len(paths),
                                   gbp=bases / 1e9, seconds=dt, genomes_per_s=len(paths) / dt, gbp_per_s=bases / 1e9 / dt,
                                   gpu=card)
                        if tree == trees[0]:
                            row.update(api_seconds=st["t_total_s"], launches=st["n_launches"], passes=st["n_passes"],
                                       ms_stream_per_gbp=st["ms_stream"] / (st["n_bases"] / 1e9),
                                       ms_select=st["ms_select"], host_read_s=st["t_read_s"],
                                       host_pack_s=st["t_pack_s"], wait_for_host_s=st["t_wait_s"])
                        print(json.dumps(row), flush=True)
                        rows.append(row)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- `mash screen` query throughput (Mbp/s) on B200, per the driver contract.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA path)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU reference arm
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...  (one rank per GPU)

Workloads (BASELINE.json `configs`, SURVEY.md 8d):
  c2 (N = 1, `configs[1]`): synthetic 1 Gbp CAMI-shaped contig set (contigs cut from 500 x 2 Mb genomes at
      1 % substitutions, half reverse-complemented, Zymo-fitted lengths) vs a 50 000-sketch database
      (k=21, s=1000; 500 sketched from the genomes on the GPU + 49 500 decoy sketches).
  c3 (N > 1, `configs[2]`): ONE 10 Gbp contig set vs a 300 000-sketch database (sketch1+2+3 shape), the
      query sharded across the N GPUs, table replicated: STRONG scaling (total work fixed).  Rank 0
      also screens all N shards alone, in the same run: the single-GPU figure of the same job
      (`single_gpu_same_workload`) and the proof that sharding changes nothing (`parity_vs_single`).
  Second keys carry the other shape: `c3_single_gpu` at N = 1, `c2_weak` at N > 1 (1 Gbp per GPU, the
  round-1 scaling measurement), plus `tiny_db` (c2 with 10 000 viral/plasmid-sized sketches: the
  two-tier probe filter is the hot path there).

One step = one complete screen of the rank's contig shard: reset, stream (k-mer hash + probe +
mixture), mixture bottom-s, [N>1: all-gather of (hash id, count) pairs + all-gather of mixtures],
per-sketch reduction, identity/p-value, and the rows mash would print (shared > 0) back on the host.

  value  : device-resident (packed query already in HBM), whole job, CUDA-event timed, max over ranks.
  e2e    : same screen through the public API from FASTA TEXT in pinned host memory: host->device
           copies, FASTA parsing + 2-bit packing, kernels and the result copy inside the timed region.
One JSON line on stdout (rank 0).  --dump-outputs DIR also writes the last timed step's result columns
as DIR/*.npy; the inputs are generated from fixed seeds, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mash-screen query throughput"
UNIT = "Mbp/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c3"],
                    help="auto = c2 on one GPU, c3 (strong scaling) on several")
    ap.add_argument("--mbp", type=int, default=1000, help="c2: query Mbp per GPU")
    ap.add_argument("--sketches", type=int, default=50_000, help="c2: sketches in the database")
    ap.add_argument("--real", type=int, default=500, help="c2: sketches made from real (synthetic) genomes")
    ap.add_argument("--total-mbp", type=int, default=10_000, help="c3: query Mbp in total (sharded across the GPUs)")
    ap.add_argument("--c3-sketches", type=int, default=300_000)
    ap.add_argument("--c3-real", type=int, default=3000)
    ap.add_argument("--cpu-mbp", type=int, default=48, help="bounded sample for the CPU baseline")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the second-key measurements (c3_single_gpu / c2_weak / tiny_db)")
    ap.add_argument("--no-filter", action="store_true", help="probe the table for every k-mer (mash semantics, no range pre-filter)")
    ap.add_argument("--wta", action="store_true")
    ap.add_argument("--tiny", type=int, default=0,
                    help="this many decoy sketches come from tiny genomes (1.5-20 k k-mers): their hashes spread "
                         "over the whole range and defeat the range pre-filter (viral/plasmid-heavy databases)")
    ap.add_argument("--k", type=int, default=21)
    ap.add_argument("--s", type=int, default=1000)
    ap.add_argument("--clusters", type=int, default=0,
                    help="config 4: make this many of the real genomes 1-5 %% diverged copies of the others")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step as DIR/<column>.npy (float64), so that two builds "
                         "can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA arm's result")
    return args


def pick_workload(args) -> str:
    return args.workload if args.workload != "auto" else ("c2" if args.gpus <= 1 else "c3")


def workload_name(args, kind: str) -> str:
    if kind == "c3":
        return ("c3: ONE synthetic %d Mbp CAMI-shaped contig set sharded across the GPUs vs %d-sketch db (k=%d, s=%d)"
                % (args.total_mbp, args.c3_sketches, args.k, args.s))
    return ("c2: synthetic %d Mbp CAMI-shaped contig set per GPU vs %d-sketch db (k=%d, s=%d)"
            % (args.mbp, args.sketches, args.k, args.s))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def static_profile(key: str) -> dict:
    """Numbers that only a profiler can count (DRAM bytes, executed instructions), copied from the
    round's ncu captures into profiles/roofline_traffic.json; every use is labelled "static"."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json"))).get(key, {})
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, res) -> None:
    """The columns a caller of the timed step receives (ScreenHits: the references with shared > 0,
    ascending), as float64 .npy files; every count is below 2^53, so the conversion is exact.  Above
    DUMP_LIMIT_BYTES in all, a fixed seeded sample of the rows is written instead."""
    import numpy as np
    cols = {"ref": res.ref, "shared": res.shared, "median": res.median, "identity": res.identity, "pvalue": res.pvalue}
    rows = np.arange(len(res.ref))
    max_rows = (DUMP_LIMIT_BYTES - 4096) // (8 * len(cols))     # 4 KB: set_size and the .npy headers
    if len(rows) > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(len(rows), max_rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, col in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(col, dtype=np.float64)[rows])
    np.save(os.path.join(out_dir, "set_size.npy"), np.array([res.set_size], dtype=np.float64))


def n_host_threads() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------
# CPU side: the reference `mash screen` when a real binary is on the box, else the oracle port
# ---------------------------------------------------------------------------------------------
def write_case_files(tmpdir, k, s, offsets, hashes, lengths, fasta: bytes):
    """db.msh + contigs.fna for a real `mash` process (names shaped like RefSeq file names)."""
    import numpy as np

    from hymet_b200 import msh as mshfmt
    from hymet_b200 import synth
    n = len(offsets) - 1
    db = mshfmt.SketchDB(k=k, s=s, names=[synth.gcf_name(i) for i in range(n)], comments=["synthetic %d" % i for i in range(n)],
                         lengths=np.asarray(lengths, np.uint64), offsets=np.asarray(offsets, np.uint64),
                         hashes=np.asarray(hashes, np.uint64))
    dbp, fap = os.path.join(tmpdir, "db.msh"), os.path.join(tmpdir, "contigs.fna")
    mshfmt.write_msh(dbp, db)
    with open(fap, "wb") as fh:
        fh.write(fasta)
    return dbp, fap, db


class CpuSide:
    """The CPU leg for one table: real `mash screen` (a process per call, as scripts/mash.sh:14 runs it)
    when a binary exists on the box -- PATH, baseline/_ref/, $HYMET_REAL_MASH -- else the oracle port."""

    def __init__(self, k, s, offsets, hashes, lengths, threads):
        from oracle import real_mash
        self.k, self.s, self.offsets, self.hashes, self.lengths, self.threads = k, s, offsets, hashes, lengths, threads
        self.mash = real_mash.find_mash()
        self.table_build_s = None
        self._files = None
        if self.mash:
            self.kind = "mash"
            self.note = ("real %s (%s): wall clock of the whole process, which loads the .msh every time as scripts/mash.sh does"
                         % (self.mash, real_mash.version(self.mash)))
        else:
            from tests import _oracle as orc
            self.kind = "port"
            self.note = ("oracle/mash_screen_oracle.c (mash-semantics restatement, parity unpinned); no real mash on this box "
                         "(looked on PATH, in baseline/_ref and at $HYMET_REAL_MASH)")
            t0 = time.perf_counter()
            self.odb = orc.OracleDB.from_arrays(k, s, 42, offsets, hashes, lengths)
            self.table_build_s = time.perf_counter() - t0

    def screen(self, fasta: bytes, wta: bool):
        """-> (seconds, n_bases, result) where result is the oracle's arrays or the real binary's TSV bytes."""
        if self.kind == "port":
            t0 = time.perf_counter()
            r = self.odb.screen_text(fasta, threads=self.threads, wta=wta)
            return time.perf_counter() - t0, r.n_bases, r
        from oracle import real_mash
        if self._files is None or self._files[2] is not fasta:
            import tempfile
            d = tempfile.mkdtemp(prefix="hs_realmash_")
            dbp, fap, db = write_case_files(d, self.k, self.s, self.offsets, self.hashes, self.lengths, fasta)
            self._files, self.db = (dbp, fap, fasta), db
        tsv, dt, _ = real_mash.screen(self.mash, self._files[0], [self._files[1]], self.threads, ("-w",) if wta else ())
        n_bases = sum(len(l) for l in fasta.split(b"\n") if l and not l.startswith(b">"))
        return dt, n_bases, tsv

    def parity(self, result, g) -> str:
        """'bit-exact' / 'byte-identical TSV' / 'MISMATCH ...': CUDA result `g` of the same sample."""
        import numpy as np
        if self.kind == "port":
            r = result
            ok = (g.shared.tolist() == r.shared.tolist() and g.median.tolist() == r.median.tolist()
                  and g.set_size == r.set_size
                  and bool(np.all(np.abs(g.identity - r.identity) <= 1e-12 * np.abs(r.identity)))
                  and bool(np.all(np.abs(g.pvalue - r.pvalue) <= 1e-12 * np.abs(r.pvalue))))
            return "bit-exact" if ok else "MISMATCH vs oracle"
        from hymet_b200.tsv import screen_lines
        sizes = (self.db.offsets[1:] - self.db.offsets[:-1]).tolist()
        mine = "".join(screen_lines(g.shared, sizes, g.median, g.identity, g.pvalue, self.db.names, self.db.comments)).encode()
        return "byte-identical TSV" if mine == result else "MISMATCH vs real mash TSV"


def run_reference(args):
    """CPU arm: real `mash screen -p <all threads>` when a binary exists on the box, else the oracle
    restatement (the real binary is a third-party dependency that is not under /root/reference nor
    installable offline -- DESIGN.md), on a bounded sample of the same workload shape."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np

    from hymet_b200 import synth
    from tests import _oracle as orc

    kind = pick_workload(args)
    threads = n_host_threads()
    k, s = args.k, args.s
    n_sk = args.c3_sketches if kind == "c3" else args.sketches
    rng = np.random.default_rng(2)
    n_real = 24
    genomes = [synth.random_genome(rng, 2_000_000) for _ in range(n_real)]
    real = np.stack([orc.sketch_text(synth.to_fasta([g], "g", width=0), k, s, threads=threads)[0] for g in genomes])
    decoy, dlen = synth.decoy_sketches(rng, n_sk - n_real, s)
    hashes = np.concatenate([real.reshape(-1), decoy.reshape(-1)])
    lengths = np.concatenate([np.full(n_real, 2_000_000, np.uint64), dlen])
    offsets = np.arange(n_sk + 1, dtype=np.uint64) * np.uint64(s)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes, args.cpu_mbp * 1_000_000, 0.01), "c", width=80)
    cpu = CpuSide(k, s, offsets, hashes, lengths, threads)
    times, bases = [], 0
    for it in range(args.warmup + args.steps):
        dt, bases, _ = cpu.screen(fasta, args.wta)
        if it >= args.warmup:
            times.append(dt)
    total = sum(times)
    val = args.steps * bases / total / 1e6
    sample = "%d Mbp of contigs (%d bases) vs the full %d-sketch table, per step" % (args.cpu_mbp, bases, n_sk)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "strong" if kind == "c3" else "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        # the CUDA arm's workload, named and keyed the same way (a subset of its `config` with identical values);
        # what this arm actually timed -- a bounded sample of it -- is described in cpu_baseline
        "config": {"workload": workload_name(args, kind), "k": k, "s": s,
                   "sketches": n_sk, "mutation_rate": 0.01, "winner_take_all": bool(args.wta)},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": cpu.kind, "sample": sample,
                         "sample_mbp_per_step": args.cpu_mbp, "real_genome_sketches_in_sample_table": n_real,
                         "timing": "host wall clock around the CPU screen, all host threads",
                         "table_build_s": cpu.table_build_s, "note": cpu.note},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np  # noqa: F401
    import torch
    import torch.distributed as dist

    from hymet_b200 import dist as hd
    from hymet_b200 import screen as hs
    from hymet_b200 import workload

    rank, world, local = hd.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    kind = pick_workload(args)
    n_cpus = n_host_threads()
    host_threads = max(1, n_cpus // world)
    stream = torch.cuda.Stream(device=dev)   # explicit stream: the library launches on it, the events time it
    torch.cuda.set_stream(stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sample_clocks=False, collective=True):
        res = None
        for _ in range(warmup):
            res = fn()
        barrier() if collective else torch.cuda.synchronize()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
            time.sleep(0.25)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stats = []
        if sample_clocks:
            torch.cuda.profiler.start()   # `ncu --profile-from-start off` sees only the timed region
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            res = fn()
            stats.append(res.stats)
        e1.record(stream)
        barrier() if collective else torch.cuda.synchronize()
        if sample_clocks:
            torch.cuda.profiler.stop()
        wall = time.perf_counter() - t0
        n_timed = len(sampler.rows) if sampler else 0
        if sampler and n_timed < 25:
            # the timed region is only tens of ms: keep the same load running (untimed) until the
            # sampler has seen it for ~0.7 s, so the median clock is of the kernel, not of idle
            t_end = time.perf_counter() + 0.7
            while time.perf_counter() < t_end:
                fn()
            torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        if clocks is not None:
            clocks["samples_in_timed_region"] = n_timed
        ms = e0.elapsed_time(e1)
        if world > 1 and collective:
            t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms, wall, stats, res, clocks

    def all_sum(v: int) -> int:
        if world == 1:
            return int(v)
        t = torch.tensor([v], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        return int(t[0])

    def results_equal(a, b) -> bool:
        # the timed steps bring back only the references with hits (hs_screen_finish_hits); compare as full columns
        a = a.to_dense(n_sketches) if hasattr(a, "to_dense") else a
        b = b.to_dense(n_sketches) if hasattr(b, "to_dense") else b
        return (a.shared.tolist() == b.shared.tolist() and a.median.tolist() == b.median.tolist() and a.set_size == b.set_size
                and a.identity.tolist() == b.identity.tolist() and a.pvalue.tolist() == b.pvalue.tolist())

    # ---- the headline workload ------------------------------------------------------------------
    t_setup = time.perf_counter()
    want_host = not args.no_e2e
    sample_mbp = args.cpu_mbp if (rank == 0 and not args.no_cpu) else 0
    if kind == "c3":
        sk = workload.make_db(local, args.c3_sketches, args.c3_real, k=args.k, s=args.s, seed=3, tiny=args.tiny,
                              cluster_copies=args.clusters)
        wl = workload.make_query(sk, max(1, args.total_mbp // world), shard=rank, with_fasta=want_host,
                                 with_host_packed=False, fasta_sample_mbp=sample_mbp, name="c3")
    else:
        sk = workload.make_db(local, args.sketches, args.real, k=args.k, s=args.s, seed=2, tiny=args.tiny,
                              cluster_copies=args.clusters)
        wl = workload.make_query(sk, args.mbp, shard=rank, with_fasta=want_host, with_host_packed=want_host,
                                 fasta_sample_mbp=sample_mbp, name="c2")
    n_sketches = len(wl.offsets) - 1
    db = hs.Database.from_arrays(wl.k, wl.s, 42, wl.offsets, wl.hashes, wl.lengths, device=local)
    scr = hd.DistributedScreen(db, local, stream_ptr=stream.cuda_stream, probe_filter=not args.no_filter)
    t_setup = time.perf_counter() - t_setup

    def step_resident():
        scr.reset()
        scr.feed_packed_device(wl.d_seq.data_ptr(), wl.d_inv.data_ptr(), wl.n_positions)
        return scr.finish_hits(args.wta)

    text_wall = {}

    def step_text():
        t0 = time.perf_counter()
        scr.reset()
        t1 = time.perf_counter()
        scr.feed_text_ptr(wl.fasta.data_ptr(), wl.fasta.numel(), host_threads)
        t2 = time.perf_counter()
        r = scr.finish_hits(args.wta)
        t3 = time.perf_counter()
        text_wall.setdefault("steps", []).append([round(1e3 * (t1 - t0), 2), round(1e3 * (t2 - t1), 2),
                                                  round(1e3 * (t3 - t2), 2)])
        return r

    def step_packed_host():
        scr.reset()
        scr.feed_packed_ptr(wl.h_seq.data_ptr(), wl.h_inv.data_ptr(), wl.n_positions)
        return scr.finish_hits(args.wta)

    total_bases = all_sum(wl.n_bases)
    ms, wall, stats, res, clocks = timed(step_resident, args.steps, args.warmup, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)
    value = args.steps * total_bases / (ms * 1e-3) / 1e6
    st = stats[-1]
    launches = sum(s["n_launches"] for s in stats)

    # ---- roofline of the dominant kernel (k_stream), from its own CUDA events -------------------
    peak, peak_src = measured_peak_gbs()
    ms_stream = sum(s["ms_stream"] for s in stats) / len(stats)
    ms_reduce = sum(s["ms_reduce"] for s in stats) / len(stats)
    ms_reset = sum(s["ms_reset"] for s in stats) / len(stats)
    alg_bytes = st["n_positions"] * 3 / 8 + 128 * st["n_bucket_reads"] + 64 * st["n_hits"]
    sem_bytes = st["n_positions"] * 3 / 8 + 128 * st["n_valid_kmers"] + 64 * st["n_hits"]
    hbm_achieved = alg_bytes / (ms_stream * 1e-3) / 1e9
    prof = static_profile("k_stream")
    same_cfg = (prof.get("k") == args.k and bool(prof.get("filter", True)) == (not args.no_filter) and not args.tiny)
    inst_per_kmer = prof.get("warp_inst_per_kmer") if same_cfg else None      # warp-level instructions per k-mer (ncu)
    sm_clock_hz = 1e6 * ((clocks or {}).get("sm_mhz") or 1965.0)
    n_sm = hs._abi.load().hs_sm_count()
    kmers_per_s = st["n_valid_kmers"] / (ms_stream * 1e-3)
    issue_peak = n_sm * 4 * sm_clock_hz                                       # warp instructions per second
    traffic = None
    if same_cfg and prof.get("dram_bytes_per_gbp"):
        traffic = prof["dram_bytes_per_gbp"] * (st["n_positions"] / 1e9)
    if inst_per_kmer:
        issue_achieved = inst_per_kmer * kmers_per_s
        roofline = {"kernel": "k_stream<%d>" % args.k, "bound": "int-issue",
                    "achieved": issue_achieved / 1e12, "peak": issue_peak / 1e12, "unit": "T warp-inst/s",
                    "frac": issue_achieved / issue_peak,
                    "definition": "warp instructions per k-mer (static: %s) x k-mers/s measured here, over SMs x 4 schedulers x "
                                  "the SM clock sampled during this run" % prof.get("source", "profiles/"),
                    "warp_inst_per_kmer": inst_per_kmer, "sm_count": n_sm, "sm_clock_mhz": sm_clock_hz / 1e6,
                    "ncu_static": {"issue_active_frac": (prof.get("issue_active_pct") or 0) / 100.0,
                                   "alu_pipe_frac": (prof.get("alu_pipe_pct") or 0) / 100.0,
                                   "fma_pipe_frac": (prof.get("fma_pipe_pct") or 0) / 100.0,
                                   "note": "same kernel under ncu --set full: the half-rate ALU pipe (shifts, logic, carry adds) "
                                           "is the busiest unit; issue slots and ALU pipe bound the kernel at the same level"}}
    else:
        roofline = {"kernel": "k_stream<%d>" % args.k, "bound": "hbm", "achieved": hbm_achieved, "peak": peak, "unit": "GB/s",
                    "frac": hbm_achieved / peak,
                    "definition": "no instruction count on file for this configuration: HBM figure only"}
    roofline.update({
        "traffic": traffic, "traffic_source": ("static: " + prof.get("source", "")) if traffic else None,
        "ms_per_launch": ms_stream, "share_of_step": ms_stream / (ms / args.steps),
        "kmers_per_s": kmers_per_s,
        "hbm": {"achieved": hbm_achieved, "peak": peak, "unit": "GB/s", "frac": hbm_achieved / peak, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "bytes": "positions x 3/8 (2-bit base + validity bit) + 128 B per bucket line read + 64 B per count update",
                "semantic_bytes_per_launch": sem_bytes,
                "semantic_frac": sem_bytes / (ms_stream * 1e-3) / 1e9 / peak,
                "note": "semantic = every valid k-mer charged one bucket line, as a probe-everything design (CPU mash) would move; "
                        "the exact pre-filter removes almost all probes, so the HBM fraction is low by design"}})

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if kind == "c3" else "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(args, kind), "k": args.k, "s": args.s,
                   "query_mbp_per_gpu": wl.n_bases / 1e6, "query_mbp_total": total_bases / 1e6,
                   "contigs_per_gpu": wl.n_contigs, "sketches": n_sketches,
                   "real_genome_sketches": wl.n_real, "mutation_rate": 0.01, "probe_filter": not args.no_filter,
                   "winner_take_all": bool(args.wta), "parallelism": "query sharded x%d, table replicated" % world,
                   "count_exchange": scr.last_exchange,
                   "l2": "inputs larger than L2 (%.0f MB packed query + %.0f MB table per GPU)"
                         % (wl.n_positions * 0.375 / 1e6, db.info.device_bytes / 1e6),
                   "timing": "CUDA events on the launching stream, max over ranks"},
        "roofline": roofline,
        "gpu_launches": launches,
        "clocks": clocks,
        "step_breakdown_ms": {"stream_kernel": ms_stream, "mixture_and_reduce": ms_reduce, "reset": ms_reset,
                              "host_gaps_exchange_and_result_copy": ms / args.steps - ms_stream - ms_reduce - ms_reset,
                              "step_total": ms / args.steps, "wall_per_step": 1e3 * wall / args.steps},
        "reduce": {"path": "dense O(stored hashes)" if st["reduce_path"] else "sparse O(present hashes)",
                   "present_hashes": st["n_touched"], "refs_with_hits": st["n_hit_refs"], "pairs_walked": st["n_pairs"]},
        "counters": {k_: st[k_] for k_ in ("n_positions", "n_valid_kmers", "n_probes", "n_bucket_reads", "n_hits",
                                          "n_mix_inserts", "n_mix_passes", "set_size")},
        "db": {"distinct_hashes": int(db.n_distinct), "table_mb": db.info.device_bytes / 1e6,
               "bucket_bytes_per_key": db.info.n_buckets * 128.0 / max(1, db.info.n_entries),
               "tiny_genome_sketches": args.tiny, "bloom_mb": db.info.bloom_bytes / 1e6,
               "range_filter_pass_fraction": db.info.max_key / 2.0 ** 64,
               "dense_range_fraction": db.info.dense_max / 2.0 ** 64, "keys_in_bloom_tier": int(db.info.bloom_keys),
               "table_build_s": db.info.t_build_s},
        "setup_s": t_setup,
        "host": {"threads_visible_at_start": n_cpus, "threads_per_gpu": host_threads, **hs.host_placement()},
    }
    if world > 1:
        line["exchange"] = {"mode": scr.last_exchange, "pair_record_capacity": scr.cap, "largest_pair_count": st["exchange_max_pairs"],
                            "bytes_all_gathered_per_rank": 8 * (1 + scr.cap) * world + 8 * (1 + wl.s) * world}

    # ---- N > 1: the same job on ONE GPU, in this run (rank 0), and parity of the sharded result ----
    if world > 1:
        words = torch.tensor([wl.d_seq.numel(), wl.n_positions], dtype=torch.int64, device=dev)
        allw = [torch.zeros_like(words) for _ in range(world)]
        dist.all_gather(allw, words)
        maxw = max(int(w[0]) for w in allw)
        pad_seq = torch.zeros(maxw, dtype=torch.int64, device=dev); pad_seq[:wl.d_seq.numel()] = wl.d_seq
        pad_inv = torch.full((maxw,), -1, dtype=torch.int32, device=dev); pad_inv[:wl.d_inv.numel()] = wl.d_inv
        g_seq = [torch.empty_like(pad_seq) for _ in range(world)] if rank == 0 else None
        g_inv = [torch.empty_like(pad_inv) for _ in range(world)] if rank == 0 else None
        dist.gather(pad_seq, g_seq, dst=0)
        dist.gather(pad_inv, g_inv, dst=0)
        del pad_seq, pad_inv
        if rank == 0:
            solo = hs.Screen(db, stream_ptr=stream.cuda_stream, probe_filter=not args.no_filter)

            def step_solo():
                solo.reset()
                for r_ in range(world):
                    solo.feed_packed_device(g_seq[r_].data_ptr(), g_inv[r_].data_ptr(), int(allw[r_][1]))
                return solo.finish_hits(args.wta)

            n_solo = max(2, min(args.steps, 5))
            sms, _, sstats, sres, _ = timed(step_solo, n_solo, 2, collective=False)
            s_stream = sum(x["ms_stream"] for x in sstats) / len(sstats)
            s_fixed = sum(x["ms_reduce"] + x["ms_reset"] for x in sstats) / len(sstats)
            line["single_gpu_same_workload"] = {"value": n_solo * total_bases / (sms * 1e-3) / 1e6, "unit": UNIT,
                                                "ms_per_step": sms / n_solo, "steps": n_solo,
                                                "stream_kernel_ms": s_stream, "mixture_reduce_reset_ms": s_fixed,
                                                "what": "all %d shards screened by rank 0 alone, same table, same run" % world}
            # where the strong-scaling loss goes: step = T1 / N + (what does not divide by N)
            t1, tn = sms / n_solo, ms / args.steps
            line["scaling_loss"] = {
                "efficiency_vs_same_run_single_gpu": t1 / (world * tn),
                "ideal_ms_per_step": t1 / world, "actual_ms_per_step": tn, "excess_ms": tn - t1 / world,
                "attribution_ms": {
                    "stream_kernel_above_its_share": ms_stream - s_stream / world,
                    "replicated_mixture_reduce_reset (does not shrink with N; its single-GPU share is already in the ideal)":
                        (ms_reduce + ms_reset) - s_fixed / world,
                    "exchange_host_gaps_result_copy": (tn - ms_stream - ms_reduce - ms_reset) - (t1 - s_stream - s_fixed) / world},
                "note": "stream_kernel_above_its_share = smaller launches (tile quantisation over 592 CTAs, per-launch table fill) and "
                        "rank imbalance; the all-gather of (hash id, count) records runs underneath the mixture finaliser"}
            line["parity_vs_single"] = ("bit-exact (shared, median, set size, identity, p-value of all %d sketches; %d shared hashes)"
                                        % (n_sketches, int(res.shared.sum()))) if results_equal(sres, res) else "MISMATCH"
            solo.close()
            del g_seq, g_inv
        barrier()

    # ---- K2 alone: random probes against the HBM-resident table (the north-star probe roofline)
    if rank == 0:
        n_probe = 1 << 26
        hq = torch.randint(-(1 << 62), 1 << 62, (n_probe,), dtype=torch.int64, device=dev)
        best = None
        for it in range(4):
            if it == 3:
                torch.cuda.profiler.start()      # `ncu --profile-from-start off -k regex:k_probe` sees this launch
            hits, reads, pms = db.probe_device(hq.data_ptr(), n_probe)
            best = pms if best is None else min(best, pms)
        torch.cuda.profiler.stop()
        # what this GPU delivers for raw random 32-byte sector reads (no hashing), same footprint
        gbuf = torch.empty(int(db.info.n_buckets) * 16, dtype=torch.int64, device=dev)
        g_ms = min(hs.gather_bench(gbuf.data_ptr(), gbuf.numel() * 8, n_probe) for _ in range(3))
        del gbuf
        ent = static_profile("k_probe")
        p_traffic = ent.get("dram_bytes_per_launch") if (ent.get("probes") == n_probe and ent.get("sketches") == n_sketches) else None
        gbs = (128.0 * reads + 8.0 * n_probe) / (best * 1e-3) / 1e9
        line["probe_kernel"] = {"kernel": "k_probe (warp-cooperative, 8 lanes per 128-byte bucket)", "probes": n_probe,
                                "bucket_reads": int(reads), "ms": best,
                                "probes_per_s": n_probe / (best * 1e-3), "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s",
                                "frac": gbs / peak,
                                "bytes": "128 B bucket line per read (10 keys + their ids + overflow flag: everything a probe "
                                         "needs, hit or miss) + 8 B hash read per probe",
                                "traffic": p_traffic, "traffic_source": ("static: " + ent.get("source", "")) if p_traffic else None,
                                "dram_frac_with_measured_traffic": (p_traffic / (best * 1e-3) / 1e9 / peak) if p_traffic else None,
                                "table_bytes_per_key": db.info.n_buckets * 128.0 / max(1, db.info.n_entries),
                                "round1_layout": "32 B buckets of 4 keys + ids in a second array: 4.0e10 probes/s, 0.25 of peak in "
                                                 "useful bytes, 0.78 in moved bytes (B200 fills 128 B per 32 B read), 36 B per key",
                                "random_sector_reads_per_s_of_this_gpu": n_probe / (g_ms * 1e-3),
                                "frac_of_random_sector_rate": (reads / (best * 1e-3)) / (n_probe / (g_ms * 1e-3))}
        # "hash table or sorted array, chosen by measurement" (north star): the sorted-array form of the same
        # lookups, as a library binary search over the sorted stored hashes (reported, never used by the product)
        try:
            sign = torch.tensor(-(1 << 63), dtype=torch.int64, device=dev)
            sk_sorted = torch.sort(torch.from_numpy(wl.hashes.view(np.int64)).to(dev) ^ sign).values   # unsigned order
            # queries spread over the range the keys live in (what passes the range pre-filter): hashes above
            # the largest key would all walk the same, cached, right-most path of the search
            hq = (torch.rand(n_probe, device=dev, dtype=torch.float64) * float(db.info.max_key)).to(torch.int64) ^ sign
            s_best = None
            for _ in range(3):
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(stream)
                pos = torch.searchsorted(sk_sorted, hq)
                s1.record(stream)
                torch.cuda.synchronize()
                s_ms = s0.elapsed_time(s1)
                s_best = s_ms if s_best is None else min(s_best, s_ms)
            line["probe_kernel"]["sorted_array_alternative"] = {
                "what": "torch.searchsorted (library binary search) of 2^26 random values spread over [0, largest key] in the "
                        "sorted array of the %d stored hashes (8 B per key)" % sk_sorted.numel(),
                "ms": s_best, "probes_per_s": n_probe / (s_best * 1e-3),
                "bucket_table_speedup": s_best / best}
            del sk_sorted, pos
        except Exception as ex:      # a reported comparison must never cost the bench line
            line["probe_kernel"]["sorted_array_alternative"] = {"unavailable": repr(ex)[:200]}
        del hq

    # ---- e2e: FASTA text in pinned host memory -> TSV columns on the host --------------
    if not args.no_e2e:
        e_steps = max(3, min(args.steps, 10))
        # three ways to get FASTA text into HBM (option "ingest"): host AVX2 packer threads,
        # device parser fed by DMA of the raw text, or both competing for chunks (the default)
        modes = {}
        for mode, name in ((0, "host_packer"), (1, "device_parser"), (2, "hybrid")):
            scr.set_option("ingest", mode)
            mms, _, mstats, mres, _ = timed(step_text, 3, 2)
            modes[name] = {"value": 3 * total_bases / (mms * 1e-3) / 1e6, "ms_per_step": mms / 3,
                           "h2d_bytes_per_step": int(mstats[-1]["h2d_bytes"]),
                           "ok": bool(results_equal(mres, res))}
        scr.set_option("ingest", 2)
        ems, ewall, estats, eres, _ = timed(step_text, e_steps, 2)
        est = estats[-1]
        e_val = e_steps * total_bases / (ems * 1e-3) / 1e6
        line["e2e"] = {"value": e_val, "unit": UNIT, "h2d_bytes_per_step": int(est["h2d_bytes"]),
                       "d2h_bytes_per_step": int(est["d2h_bytes"]), "ms_per_step": ems / e_steps,
                       "input": "FASTA text (%d B per GPU, 80-column lines) in pinned host memory" % wl.fasta.numel(),
                       "host_threads_per_gpu": host_threads, "steps": e_steps, "ingest": "hybrid (default)",
                       "ingest_modes": modes,
                       "host_wall_ms_reset_feed_finish": text_wall["steps"][-e_steps:],
                       "stream_kernel_ms_per_step": est["ms_stream"], "launches_per_step": est["n_launches"],
                       "includes": "host FASTA parse + 2-bit pack, H2D, all kernels, D2H of the result columns"}
        same = results_equal(eres, res)
        if wl.h_seq is not None:
            pms, pwall, pstats, pres, _ = timed(step_packed_host, 3, 1)
            line["e2e_packed"] = {"value": 3 * total_bases / (pms * 1e-3) / 1e6, "unit": UNIT,
                                  "h2d_bytes_per_step": int(pstats[-1]["h2d_bytes"]),
                                  "d2h_bytes_per_step": int(pstats[-1]["d2h_bytes"]), "ms_per_step": pms / 3,
                                  "input": "pre-packed 2-bit + mask words in pinned host memory"}
            same = same and results_equal(pres, res)
        # SURVEY 8d's end-to-end: the FASTA is a FILE in the page cache, read by hs_screen_feed_fasta (reader
        # threads pread() record-aligned blocks into a pinned ring, the device parses them)
        import tempfile
        fdir = tempfile.mkdtemp(prefix="hs_bench_%d_" % rank)
        fpath = os.path.join(fdir, "contigs.fna")
        wl.fasta.numpy().tofile(fpath)
        def step_file():
            scr.reset()
            scr.feed_fasta(fpath, host_threads)
            return scr.finish_hits(args.wta)

        best_file = None
        for readers in sorted({max(1, min(8, host_threads)), max(1, min(16, host_threads))}):
            scr.set_option("file_readers", readers)
            scr.set_option("file_block_bytes", 16 << 20)
            fms, fwall, fstats, fres, _ = timed(step_file, 3, 2)
            ent = {"value": 3 * total_bases / (fms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": fms / 3,
                   "h2d_bytes_per_step": int(fstats[-1]["h2d_bytes"]), "d2h_bytes_per_step": int(fstats[-1]["d2h_bytes"]),
                   "input": "the same FASTA as a file in the page cache (%d B per GPU)" % wl.fasta.numel(),
                   "reader_threads_per_gpu": readers, "ok": bool(results_equal(fres, res))}
            if best_file is None or ent["value"] > best_file["value"]:
                ent["other_reader_counts"] = (best_file or {}).get("other_reader_counts", []) + \
                    ([{"readers": best_file["reader_threads_per_gpu"], "value": best_file["value"]}] if best_file else [])
                best_file = ent
            else:
                best_file.setdefault("other_reader_counts", []).append({"readers": readers, "value": ent["value"]})
        line["e2e_file"] = best_file
        try:
            os.remove(fpath)
            os.rmdir(fdir)
        except OSError:
            pass
        line["e2e"]["matches_device_resident"] = bool(same)
    else:
        line["e2e"] = None

    # ---- CPU baseline on a bounded sample (rank 0) + parity of that sample ----------
    if rank == 0 and not args.no_cpu and wl.fasta_sample:
        cpu = CpuSide(wl.k, wl.s, wl.offsets, wl.hashes, wl.lengths, n_cpus)
        reps = 2 if world == 1 else 1
        best, cres, cbases = None, None, 0
        for _ in range(reps):
            dt, cbases, cres = cpu.screen(wl.fasta_sample, args.wta)
            best = dt if best is None else min(best, dt)
        chk = hs.Screen(db, stream_ptr=stream.cuda_stream, probe_filter=not args.no_filter)
        chk.feed_text(wl.fasta_sample, host_threads)
        g = chk.finish(args.wta)
        chk.close()
        entry = {"value": cbases / best / 1e6, "unit": UNIT, "cores": n_cpus, "kind": cpu.kind,
                 "sample": "first %d bases of rank 0's contigs vs the same %d-sketch table, best of %d" % (cbases, n_sketches, reps),
                 "table_build_s": cpu.table_build_s, "parity_on_sample": cpu.parity(cres, g),
                 "sample_shared_hashes": int(g.shared.sum()), "note": cpu.note}
        if world == 1:
            line["cpu_baseline"] = entry
        else:
            line["cpu_parity"] = entry      # the contract asks for cpu_baseline at N = 1 only; the parity check stays
        del cpu

    scr.scr.close()
    db.close()
    del wl, sk, scr, db
    torch.cuda.empty_cache()

    # ---- second keys: the other shape of BASELINE.json, and the viral/plasmid-bearing database ----
    if not args.no_extras:
        def quick(name, n_sk, n_real, mbp, seed, tiny=0, steps=5):
            sk2 = workload.make_db(local, n_sk, n_real, k=args.k, s=args.s, seed=seed, tiny=tiny)
            wl2 = workload.make_query(sk2, mbp, shard=rank, name=name)
            db2 = hs.Database.from_arrays(wl2.k, wl2.s, 42, wl2.offsets, wl2.hashes, wl2.lengths, device=local)
            scr2 = hd.DistributedScreen(db2, local, stream_ptr=stream.cuda_stream)

            def step2():
                scr2.reset()
                scr2.feed_packed_device(wl2.d_seq.data_ptr(), wl2.d_inv.data_ptr(), wl2.n_positions)
                return scr2.finish_hits(False)

            ms2, _, st2, _, _ = timed(step2, steps, 3)
            tot = all_sum(wl2.n_bases)
            out = {"value": steps * tot / (ms2 * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms2 / steps, "steps": steps,
                   "sketches": n_sk, "query_mbp_total": tot / 1e6, "n_gpus": world,
                   "stream_kernel_ms": sum(s["ms_stream"] for s in st2) / len(st2),
                   "mixture_and_reduce_ms": sum(s["ms_reduce"] for s in st2) / len(st2),
                   "reset_ms": sum(s["ms_reset"] for s in st2) / len(st2),
                   "table_mb": db2.info.device_bytes / 1e6, "probes": st2[-1]["n_probes"], "hits": st2[-1]["n_hits"],
                   "bloom_mb": db2.info.bloom_bytes / 1e6, "dense_range_fraction": db2.info.dense_max / 2.0 ** 64,
                   "range_filter_pass_fraction": db2.info.max_key / 2.0 ** 64}
            scr2.scr.close()
            db2.close()
            del wl2, sk2, scr2, db2
            torch.cuda.empty_cache()
            return out

        if kind == "c2" and world == 1:
            line["c3_single_gpu"] = dict(quick("c3", args.c3_sketches, args.c3_real, args.total_mbp, 3, steps=3),
                                         workload=workload_name(args, "c3"), scaling="the N = 1 point of the strong-scaling line")
        if kind == "c3":
            line["c2_weak"] = dict(quick("c2", args.sketches, args.real, args.mbp, 2), workload=workload_name(args, "c2"), scaling="weak")
        if not args.tiny:
            line["tiny_db"] = dict(quick("c2", args.sketches, args.real, args.mbp, 2, tiny=10_000),
                                   workload="c2 with 10 000 of the sketches drawn from 1.5-20 k-k-mer genomes (viral/plasmid-sized): "
                                            "their hashes cover the hash range, the two-tier probe filter is the hot path")
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_OUT = None


def emit(line) -> None:
    _OUT.write(json.dumps(line) + "\n")
    _OUT.flush()


def main():
    global _OUT
    args = parse_args()
    # libraries (NCCL's version banner) write to fd 1; the contract is ONE JSON line on stdout
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

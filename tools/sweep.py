#!/usr/bin/env python
"""Run bench.py over the BASELINE.json configs (3, 4, 5) and collect the JSON lines, each with a CPU-oracle
parity check on a bounded sample of its own contigs (SWEEP_NO_CPU=1 skips that).
Usage: python tools/sweep.py out.jsonl  (on a GPU box)"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "sweep.jsonl")
runs = [
    ("c2_default", []),
    ("c2_probe_all", ["--no-filter"]),
    ("c3_300k_sketches_1250mbp", ["--sketches", "300000", "--real", "3000", "--mbp", "1250"]),
    ("c4_wta_clusters", ["--wta", "--clusters", "250"]),
    ("c4_plain_clusters", ["--clusters", "250"]),
    ("c2_tiny10k_bloom", ["--tiny", "10000"]),
    ("c5_k21_s5000", ["--s", "5000"]),
    ("c5_k21_s10000", ["--s", "10000"]),
    ("c5_k31_s1000", ["--k", "31"]),
    ("c5_k31_s5000", ["--k", "31", "--s", "5000"]),
    ("c5_k31_s10000", ["--k", "31", "--s", "10000"]),
]
only = set(sys.argv[2].split(",")) if len(sys.argv) > 2 else None
with open(out, "a") as fh:
    for name, extra in runs:
        if only and name not in only:
            continue
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--no-e2e", "--no-extras", "--workload", "c2"] + extra + (["--no-cpu"] if os.environ.get("SWEEP_NO_CPU") else [])
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
        line = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else ""
        try:
            d = json.loads(line)
            d["sweep_name"] = name
            fh.write(json.dumps(d) + "\n"); fh.flush()
            print(name, "value %.0f Mbp/s  step %.2f ms  stream %.2f ms  reduce %.2f ms  reset %.3f ms  kmers/s %.3g  probes %d  hits %d  table %.0f MB  cpu-parity %s" % (
                d["value"], d["ms_per_step"], d["step_breakdown_ms"]["stream_kernel"], d["step_breakdown_ms"]["mixture_and_reduce"],
                d["step_breakdown_ms"]["reset"], d["roofline"]["kmers_per_s"], d["counters"]["n_probes"], d["counters"]["n_hits"],
                d["db"]["table_mb"], (d.get("cpu_baseline") or {}).get("parity_on_sample")), flush=True)
        except Exception as e:
            print(name, "FAILED", e, r.stderr[-800:], flush=True)

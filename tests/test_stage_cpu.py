"""Rows a2/a3 on the CPU: hymet_b200.stage restates what scripts/mash.sh:15-55 does to the TSV
(`sort -u -k5,5`, `sort -gr`, the bc/awk threshold loop, `cut -f5`) and run_hymet_cami.sh's merge.
Checked here against the real coreutils/awk of this image and against HYMET's own unmodified
scripts/mash.sh (stored verbatim in tests/golden/mash_sh_fixture.json) with the oracle CLI standing in
for `mash`."""
import base64
import gzip
import hashlib
import json
import os
import stat
import subprocess
import sys

import numpy as np
import pytest

from hymet_b200 import msh as mshfmt
from hymet_b200 import stage, synth
from tests import _oracle as orc

C_ENV = dict(os.environ, LC_ALL="C")

# `bc` is not in this image; mash.sh needs three kinds of expression from it.  Exact decimals,
# bc's scale rules (product: min(a+b, max(scale, a, b))) and its print format.
FAKE_BC = r'''#!%s
import sys
from decimal import Decimal
scale = 20 if "-l" in sys.argv[1:] else 0
def dp(x): return max(0, -Decimal(x).as_tuple().exponent)
def show(d):
    if d == 0: return "0"
    s = format(d, "f")
    if s.startswith("0."): s = s[1:]
    elif s.startswith("-0."): s = "-" + s[2:]
    return s
for line in sys.stdin:
    t = line.split()
    if not t: continue
    a, op, b = t[0], t[1], t[2]
    if op == ">=": print(1 if Decimal(a) >= Decimal(b) else 0)
    elif op == "-": print(show(Decimal(a) - Decimal(b)))
    elif op == "*":
        r = Decimal(a) * Decimal(b)
        sc = min(dp(a) + dp(b), max(scale, dp(a), dp(b)))
        print(show(r.quantize(Decimal(1).scaleb(-sc), rounding="ROUND_DOWN")))
    else: sys.exit("fake bc: unsupported " + line)
''' % sys.executable


def random_tsv(rng, n):
    lines = []
    names = ["GCF_%09d.1_ASM%d_genomic.fna" % (rng.integers(0, n // 2 + 2), i) if i % 3 else "GCF_dup_%d" % (i % 7)
             for i in range(n)]
    for i in range(n):
        shared = int(rng.integers(1, 1001))
        ident = [1.0, (shared / 1000.0) ** (1 / 21.0), 10.0 ** -rng.integers(1, 8), 0.0][int(rng.integers(0, 4)) if i % 5 == 0 else 1]
        name = names[i] if i % 11 else "name with blank %d" % (i % 3)
        comment = ["", "Escherichia coli str. K-12", "[12 seqs] NZ_X [...]", "\tleading tab"][i % 4]
        lines.append(("%g\t%d/1000\t%d\t%g\t%s\t%s" % (ident, shared, rng.integers(1, 9), 10.0 ** -rng.integers(0, 30), name,
                                                   comment)).encode())
    return lines


def run_tool(cmd, data):
    return subprocess.run(cmd, input=data, capture_output=True, env=C_ENV, check=True).stdout


def reference_mash_sh(tmp_path, golden_dir):
    """HYMET's scripts/mash.sh, byte for byte, from the compressed fixture."""
    fx = json.load(open(os.path.join(golden_dir, "mash_sh_fixture.json")))
    raw = gzip.decompress(base64.b64decode(fx["gzip_base64"]))
    assert hashlib.sha256(raw).hexdigest() == fx["sha256"]
    sh = tmp_path / "mash.sh"
    sh.write_bytes(raw)
    return str(sh)


def test_text_tools_match_coreutils_and_awk():
    rng = np.random.default_rng(5)
    for n in (0, 1, 40, 700):
        lines = random_tsv(rng, n)
        blob = b"".join(l + b"\n" for l in lines)
        j = lambda ls: b"".join(l + b"\n" for l in ls)
        filt = stage.sort_u_k5(lines)
        assert j(filt) == run_tool(["sort", "-u", "-k5,5"], blob)
        srt = stage.sort_gr(filt)
        assert j(srt) == run_tool(["sort", "-gr"], j(filt))
        assert j(stage.sort_gr(lines)) == run_tool(["sort", "-gr"], blob)       # ties + duplicates included
        for t in ("0.9", ".88", "0.71", "0.5", "1"):
            assert j(stage.awk_gt(srt, t)) == run_tool(["awk", "-v", "t=" + t, "$1 > t"], j(srt))
        assert j(stage.cut_f5(srt)) == run_tool(["cut", "-f5"], j(srt))
        assert stage.merge_selected([j(stage.cut_f5(srt)), j(stage.cut_f5(lines))]) == \
            run_tool(["sort", "-u"], j(stage.cut_f5(srt)) + j(stage.cut_f5(lines)))


def test_threshold_arithmetic():
    assert [stage.min_candidates(n) for n in (0, 1, 2, 3, 4, 10)] == [5, 5, 7, 10, 13, 33]
    from decimal import Decimal
    assert stage._bc(Decimal("0.90") - Decimal("0.02")) == ".88"
    assert stage._bc(Decimal("0.9") - Decimal("0.02")) == ".88"
    assert stage._bc(Decimal("1.00") - Decimal("0.02")) == ".98"
    assert stage._bc(Decimal("1.5")) == "1.5" and stage._bc(Decimal("0.00")) == "0"
    # every sketch below 0.70: the loop runs out and 0.71 is used (mash.sh:46-50)
    tab = b"0.65\t1/1000\t1\t0.1\tA\t\n0.72\t2/1000\t1\t0.1\tB\t\n"
    r = stage.select(tab, 1, "0.9")
    assert r["threshold"] == "0.71" and r["selected"] == b"B\n" and "Using 0.70" in r["log"]
    assert r["log"].count("Testing threshold") == 11 and "Testing threshold: .70\n" in r["log"]


def test_input_files_glob_and_find(tmp_path):
    for n in ("b.fna", "a.fna", ".hidden.fna", "c.fasta", "B.fna"):
        (tmp_path / n).write_text(">x\nACGT\n")
    files, n_find = stage.input_files(str(tmp_path))
    assert [os.path.basename(f) for f in files] == ["B.fna", "a.fna", "b.fna"] and n_find == 4
    out = subprocess.run(["bash", "-c", 'echo "$1"/*.fna; find "$1" -maxdepth 1 -name "*.fna" | wc -l', "_", str(tmp_path)],
                         capture_output=True, text=True, env=C_ENV).stdout.split("\n")
    assert out[0].split() == files and int(out[1]) == n_find


def make_case(tmp_path, seed, n_genomes, n_files, glen=30_000, rates=(0.0, 0.02, 0.05, 0.08), per_file=5):
    rng = np.random.default_rng(seed)
    genomes = [synth.random_genome(rng, glen) for _ in range(n_genomes)]
    genomes += [synth.mutate(genomes[i], 0.03, rng) for i in range(min(6, n_genomes))]
    sk = [orc.sketch_text(synth.to_fasta([g], "g"), 21, 1000)[0] for g in genomes]
    offs = np.concatenate([[0], np.cumsum([len(x) for x in sk])]).astype(np.uint64)
    names = ["GCF_%09d.%d_ASM%d_genomic.fna" % (i // 2, 1 + i % 2, i) for i in range(len(genomes))]
    names[-1] = names[0]                                   # a duplicated query-ID: `sort -u -k5,5` must drop one
    db = mshfmt.SketchDB(k=21, s=1000, names=names, comments=["c %d" % i if i % 2 else "" for i in range(len(genomes))],
                         lengths=np.array([len(g) for g in genomes], np.uint64), offsets=offs, hashes=np.concatenate(sk))
    dbp = str(tmp_path / "db.msh")
    mshfmt.write_msh(dbp, db)
    indir = tmp_path / "input"
    indir.mkdir()
    for f in range(n_files):
        rate = rates[f % len(rates)]
        (indir / ("sample_%d.fna" % f)).write_bytes(
            synth.to_fasta(synth.cut_contigs(rng, genomes[2 * f:2 * f + per_file], 120_000, rate, median=4000.0), "s%d" % f))
    return dbp, str(indir)


@pytest.mark.parametrize("seed,n_genomes,n_files,thr,rates,per_file", [
    (1, 24, 1, "0.9", (0.0,), 5),                        # first threshold is enough
    (3, 12, 2, "0.95", (0.0, 0.02), 5),
    (5, 10, 3, "0.9", (0.0, 0.12, 0.2), 2),              # steps down to .78
    (6, 14, 2, "0.9", (0.15, 0.2), 4),                   # .80
    (8, 20, 4, "0.97", (0.05, 0.1, 0.15, 0.22), 3),      # ten steps
    (7, 3, 1, "0.9", (0.1,), 2),                         # never enough candidates: 0.71 fallback
])
def test_select_equals_unmodified_reference_mash_sh(tmp_path, golden_dir, seed, n_genomes, n_files, thr, rates, per_file):
    script = reference_mash_sh(tmp_path, golden_dir)
    orc.build()
    dbp, indir = make_case(tmp_path, seed, n_genomes, n_files, rates=rates, per_file=per_file)
    bindir = tmp_path / "bin"
    bindir.mkdir()
    os.symlink(orc.BIN, bindir / "mash")
    bc = bindir / "bc"
    bc.write_text(FAKE_BC)
    bc.chmod(bc.stat().st_mode | stat.S_IXUSR)
    od = tmp_path / "out"
    od.mkdir()
    files = [str(od / f) for f in ("screen.tab", "filtered.tab", "sorted.tab", "top_hits.tab", "selected.txt")]
    env = dict(C_ENV, PATH=str(bindir) + os.pathsep + os.environ["PATH"])
    p = subprocess.run(["bash", script, indir, dbp] + files + [thr], capture_output=True, env=env, check=True)
    got = [open(f, "rb").read() for f in files]
    assert got[0].count(b"\n") >= 3
    _, n_find = stage.input_files(indir)
    r = stage.select(got[0], n_find, thr)
    assert [r["filtered"], r["sorted"], r["top_hits"], r["selected"]] == got[1:]
    assert r["log"] == p.stdout.decode()


def test_select_on_real_genome_golden():
    """tests/golden/zymo_mash_sh.json = what the unmodified scripts/mash.sh left behind for the real-genome
    fixture (made by tests/golden/make_zymo_mash_sh_golden.py where /root/reference exists): the restated
    post-processing reproduces it on any box, including the threshold that had to step down."""
    import json
    g = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    want = json.load(open(os.path.join(g, "zymo_mash_sh.json")))
    tab = open(os.path.join(g, "zymo_screen.tsv"), "rb").read()
    for thr, w in want.items():
        r = stage.select(tab, 1, thr)
        for key in ("filtered", "sorted", "top_hits", "selected"):
            assert r[key] == w[key].encode(), (thr, key)
        assert r["log"] == w["log"]
    assert want["0.9"]["log"].count("Testing threshold") > 1      # 0.9 is not reached by five sketches: the loop steps


def test_stage_cli_usage_and_no_silent_cpu_result(tmp_path):
    exe = [sys.executable, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin", "hymet-mash-stage")]
    r = subprocess.run(exe + ["input", "0.9", "db.msh"], capture_output=True, text=True)
    assert r.returncode == 2 and "hymet-mash-stage" in r.stderr
    r = subprocess.run(exe + ["-h"], capture_output=True, text=True)
    assert r.returncode == 0 and "THRESHOLD" in r.stdout
    import torch
    gpu = torch.cuda.is_available()
    outs = [str(tmp_path / f) for f in ("a", "b", "c", "d", "e")]
    r = subprocess.run(exe + [str(tmp_path), "0.9", "notasketch.txt"] + outs, capture_output=True, text=True)
    assert "does not look like a sketch" in r.stderr
    if gpu:      # a bad sketch file is a data error, as in scripts/mash.sh (no `set -e`): status 0, empty files
        assert r.returncode == 0 and all(open(o, "rb").read() == b"" for o in outs)
    else:
        assert r.returncode == 1
    r = subprocess.run(exe + [str(tmp_path), "abc", "x.msh"] + outs, capture_output=True, text=True)
    assert r.returncode == 1 and "threshold" in r.stderr
    if not gpu:                            # without a B200 the stage fails loudly and writes nothing
        db = mshfmt.SketchDB(k=21, s=10, names=["a"], comments=[""], lengths=np.array([5], np.uint64),
                             offsets=np.array([0, 2], np.uint64), hashes=np.array([1, 2], np.uint64))
        p = str(tmp_path / "d.msh")
        mshfmt.write_msh(p, db)
        (tmp_path / "x.fna").write_text(">a\nACGT\n")
        r = subprocess.run(exe + [str(tmp_path), "0.9", p] + outs, capture_output=True, text=True)
        assert r.returncode == 1 and "ERROR" in r.stderr and not any(os.path.exists(o) for o in outs)

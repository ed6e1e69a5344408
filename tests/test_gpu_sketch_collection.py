"""`mash sketch` of whole genome collections: many genomes per kernel pass (k_stream MODE 4), `-l` input
lists, `-p` host threads.  Every sketch must equal the CPU oracle's on the same bytes, and the CLI's .msh
must be byte-identical to one written here with msh.write_msh from oracle sketches and the comment rule."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

from hymet_b200 import msh as mshfmt
from hymet_b200 import screen as hs
from hymet_b200 import synth
from tests import _oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASH = [sys.executable, os.path.join(ROOT, "bin", "mash")]
BATCH_POSITIONS = 4096 * 8192   # kSketchBatchTiles tiles of 8192 positions (abi.cu)


def read_text(p):
    with (gzip.open(p, "rb") if p.endswith(".gz") else open(p, "rb")) as fh:
        return fh.read()


def comment_of(text):
    n_rec = text.count(b"\n>") + (1 if text.startswith(b">") else 0)
    first = text[1:text.find(b"\n")].decode("utf-8", "replace").strip() if text.startswith(b">") else ""
    return "[%d seqs] %s [...]" % (n_rec, first) if n_rec > 1 else first


def expected_msh(out, paths, k, s, seed=42):
    texts = [read_text(p) for p in paths]
    sk = [orc.sketch_text(t, k, s, seed, threads=4) for t in texts]
    offsets = np.concatenate([[0], np.cumsum([len(h) for h, _ in sk])]).astype(np.uint64)
    db = mshfmt.SketchDB(k=k, s=s, seed=seed, names=list(paths), comments=[comment_of(t) for t in texts],
                         lengths=np.array([ln for _, ln in sk], np.uint64), offsets=offsets,
                         hashes=np.concatenate([h for h, _ in sk]) if sk else np.zeros(0, np.uint64))
    mshfmt.write_msh(out, db)
    return sk


def to_fastq(records, prefix):
    parts = []
    for i, c in enumerate(records):
        seq = synth.ASCII[c].tobytes()
        parts.append(b"@%s_%d\n%s\n+\n%s\n" % (prefix.encode(), i, seq, b"I" * len(seq)))
    return b"".join(parts)


def write(path, data):
    if str(path).endswith(".gz"):
        with gzip.open(path, "wb") as fh:
            fh.write(data)
    else:
        with open(path, "wb") as fh:
            fh.write(data)
    return str(path)


def run_cli(args):
    return subprocess.run(MASH + ["sketch"] + args, capture_output=True)


def check_cli(tmp_path, paths, k, s, extra=()):
    """sketch `paths` through `-l` and compare the file with the oracle's, byte for byte"""
    lst = tmp_path / "inputs.txt"
    lst.write_bytes(b"\n".join(p.encode() for p in paths) + b"\n")
    out = str(tmp_path / "cli")
    r = run_cli(["-l", "-k", str(k), "-s", str(s), "-o", out] + list(extra) + [str(lst)])
    assert r.returncode == 0, r.stderr.decode()
    want = str(tmp_path / "want.msh")
    sk = expected_msh(want, paths, k, s)
    assert open(out + ".msh", "rb").read() == open(want, "rb").read()
    return sk


def test_two_thousand_genomes_in_few_launches(tmp_path):
    rng = np.random.default_rng(2000)
    paths = []
    for i in range(2000):
        g = synth.random_genome(rng, int(rng.integers(5_000, 50_001)), n_frac=0.001)
        cut = int(rng.integers(1, len(g)))
        paths.append(write(tmp_path / ("g%04d.fna" % i), synth.to_fasta([g[:cut], g[cut:]], "g%d" % i)))
    got, st = hs.sketch_files(paths, 21, 1000, threads=8)
    assert st["n_genomes"] == 2000 and st["n_launches"] <= 20, st
    for p, g in zip(paths, got):
        want, ln = orc.sketch_text(read_text(p), 21, 1000)
        assert g.hashes.tolist() == want.tolist() and g.length == ln
    check_cli(tmp_path, paths, 21, 1000, ["-p", "16"])


def test_mixed_formats_edge_files_and_repeats(tmp_path):
    rng = np.random.default_rng(7)
    g = [synth.random_genome(rng, n) for n in (60_000, 45_000, 30_000, 800)]
    unit = synth.random_genome(rng, 20_000)
    paths = [
        write(tmp_path / "plain.fna", synth.to_fasta([g[0]], "plain")),
        write(tmp_path / "zipped.fna.gz", synth.to_fasta([g[1][:20_000], g[1][20_000:]], "zipped")),
        write(tmp_path / "reads.fastq", to_fastq([g[2][i:i + 150] for i in range(0, 29_000, 100)], "read")),
        write(tmp_path / "reads.fastq.gz", to_fastq([g[2][i:i + 150] for i in range(50, 29_000, 100)], "read")),
        write(tmp_path / "small.fna", synth.to_fasta([g[3]], "small")),                       # < s distinct k-mers
        write(tmp_path / "repeat.fna", synth.to_fasta([np.tile(unit, 50)], "repeat", width=0)),  # 1 Mbp, 20 kb distinct
        write(tmp_path / "empty.fna", b""),
        write(tmp_path / "allN.fna", b">nothing\n" + b"N" * 5000 + b"\n"),
        write(tmp_path / "norecords.txt", b"ACGTACGTACGTACGTACGTACGTACGTACGT\n"),
        write(tmp_path / "noheader_newline.fna", b">only a header"),
    ]
    paths.append(paths[0])   # the same path twice
    got, st = hs.sketch_files(paths, 21, 1000, threads=4)
    assert st["n_passes"] > 0, st          # the repeat genome needed its threshold raised
    for p, sk in zip(paths, got):
        want, ln = orc.sketch_text(read_text(p), 21, 1000)
        assert sk.hashes.tolist() == want.tolist() and sk.length == ln, p
    assert len(got[4].hashes) < 1000 and len(got[4].hashes) == 800 - 20
    assert len(got[6].hashes) == len(got[7].hashes) == 0
    check_cli(tmp_path, paths, 21, 1000, ["-p", "3"])


@pytest.mark.parametrize("k", [12, 16, 21, 31, 32])
@pytest.mark.parametrize("s", [1, 64, 1000, 10000])
def test_k_and_s(k, s):
    rng = np.random.default_rng(k * 100_003 + s)
    texts = [synth.to_fasta([synth.random_genome(rng, n, n_frac=0.002)], "g")
             for n in (5_000, 40_000, 300_000, 12_000)]
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        paths = [write(os.path.join(d, "g%d.fa" % i), t) for i, t in enumerate(texts)]
        got, _ = hs.sketch_files(paths, k, s, threads=2)
    for t, sk in zip(texts, got):
        want, ln = orc.sketch_text(t, k, s)
        assert sk.hashes.tolist() == want.tolist() and sk.length == ln


def test_genome_larger_than_a_batch(tmp_path):
    rng = np.random.default_rng(99)
    big = synth.random_genome(rng, BATCH_POSITIONS + 3_000_000, n_frac=0.0005)
    paths = [write(tmp_path / "a.fna", synth.to_fasta([synth.random_genome(rng, 30_000)], "a")),
             write(tmp_path / "big.fna", synth.to_fasta([big[:1_000_000], big[1_000_000:]], "big", width=0)),
             write(tmp_path / "b.fna", synth.to_fasta([synth.random_genome(rng, 30_000)], "b"))]
    got, st = hs.sketch_files(paths, 21, 1000, threads=3)
    assert st["n_launches"] >= 4, st        # two pieces for the big genome, one launch around it, selections
    for p, sk in zip(paths, got):
        want, ln = orc.sketch_text(read_text(p), 21, 1000, threads=8)
        assert sk.hashes.tolist() == want.tolist() and sk.length == ln


def test_list_with_empty_lines_and_missing_path(tmp_path):
    rng = np.random.default_rng(3)
    paths = [write(tmp_path / ("x%d.fna" % i), synth.to_fasta([synth.random_genome(rng, 20_000)], "x")) for i in range(3)]
    lst = tmp_path / "list.txt"
    lst.write_bytes(b"\n" + paths[0].encode() + b"\n\n" + paths[1].encode() + b"\n" + paths[2].encode())
    r = run_cli(["-l", "-s", "200", str(lst)])
    assert r.returncode == 0, r.stderr.decode()
    want = str(tmp_path / "want.msh")
    expected_msh(want, paths, 21, 200)
    assert open(str(lst) + ".msh", "rb").read() == open(want, "rb").read()   # default prefix: first positional
    missing = str(tmp_path / "nope.fna")
    lst.write_bytes((paths[0] + "\n" + missing + "\n").encode())
    r = run_cli(["-l", "-o", str(tmp_path / "m"), str(lst)])
    assert r.returncode == 1 and ("ERROR: could not open %s for reading." % missing).encode() in r.stderr
    assert not os.path.exists(str(tmp_path / "m.msh"))


def test_screen_finds_genomes_of_collection_sketch(tmp_path):
    rng = np.random.default_rng(21)
    genomes = [synth.random_genome(rng, 80_000) for _ in range(40)]
    paths = [write(tmp_path / synth.gcf_name(i), synth.to_fasta([g], "chr")) for i, g in enumerate(genomes)]
    out = str(tmp_path / "db")
    r = run_cli(["-s", "500", "-p", "4", "-o", out] + paths)
    assert r.returncode == 0, r.stderr.decode()
    q = tmp_path / "q.fna"
    q.write_bytes(synth.to_fasta(synth.cut_contigs(rng, [genomes[3], genomes[17]], 200_000, 0.005, median=5000.0), "c"))
    r = subprocess.run(MASH + ["screen", "-v", "0.9", out + ".msh", str(q)], capture_output=True)
    assert r.returncode == 0
    assert [l.split(b"\t")[4].decode() for l in r.stdout.splitlines()] == [paths[3], paths[17]]

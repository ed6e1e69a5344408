"""CUDA path vs the CPU oracle, through the C ABI (needs a B200: `pytest -m gpu`).

Bit-exact: k-mer hashes, table membership, per-hash counts, shared counts, median
multiplicities, winner-take-all assignment, mixture bottom-s, set size.
Floating point: identity and p-value within 1e-12 relative (north_star).
"""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from hymet_b200 import msh as mshfmt
from hymet_b200 import screen as hs
from hymet_b200 import synth
from hymet_b200.tsv import screen_lines
from oracle import py_micro_oracle as po
from tests import _oracle as orc
from tests.test_stage_cpu import reference_mash_sh

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-12  # north_star tolerance for identity / p-value


def rel_close(a, b, rtol=RTOL):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.all(np.abs(a - b) <= rtol * np.abs(b))


def build_db(genomes, k, s, seed=42):
    """Sketch genomes with the ORACLE (checker side) -> flat arrays."""
    hs_list, lens = [], []
    for g in genomes:
        h, ln = orc.sketch_text(synth.to_fasta([g], "g"), k, s, seed)
        hs_list.append(h); lens.append(ln)
    offsets = np.concatenate([[0], np.cumsum([len(h) for h in hs_list])]).astype(np.uint64)
    hashes = np.concatenate(hs_list) if hs_list else np.zeros(0, np.uint64)
    return offsets, hashes, np.array(lens, np.uint64)


def compare_screen(db_gpu, db_orc, fasta: bytes, wta: bool, threads=2, feed="text", probe_filter=True):
    scr = hs.Screen(db_gpu, probe_filter=probe_filter)
    if feed == "text":
        scr.feed_text(fasta, threads)
    else:
        seq, inv, n, _ = hs.pack_text(fasta)
        scr.feed_packed(seq, inv, n)
    res = scr.finish(wta)
    want = db_orc.screen_text(fasta, threads=2, wta=wta)
    assert res.shared.tolist() == want.shared.tolist()
    assert res.median.tolist() == want.median.tolist()
    assert res.set_size == want.set_size
    assert scr.mixture().tolist() == want.mixture.tolist()
    assert res.stats["n_valid_kmers"] == want.n_kmers
    assert rel_close(res.identity, want.identity)
    assert rel_close(res.pvalue, want.pvalue)
    scr.close()
    return res, want


# ---------------------------------------------------------------- K1 ----------
@pytest.mark.parametrize("k", [7, 15, 16, 17, 21, 27, 31, 32])
def test_k1_hashes_every_kmer(k):
    rng = random.Random(k)
    text = ""
    for r in range(9):
        L = rng.choice([0, 5, k - 1, k, k + 1, 300, 8191, 8193, 20000])
        s = "".join(rng.choice("ACGTacgtNRY") if rng.random() < 0.01 else rng.choice("ACGT") for _ in range(L))
        text += ">r%d\n%s\n" % (r, s)
    seq, inv, n, st = hs.pack_text(text.encode())
    h, v = hs.hash_packed(k, 42, seq, inv, n)
    # oracle: per record, window start i <-> packed position of last base
    pos = 0
    want_h = np.zeros(n, np.uint64); want_v = np.zeros(n, bool)
    for _, s in po.parse_fasta(text):
        pos += 1  # separator
        oh, ov = orc.hash_sequence(s.encode(), k)
        for i in np.nonzero(ov)[0]:
            want_h[pos + i + k - 1] = oh[i]; want_v[pos + i + k - 1] = True
        pos += len(s)
    assert pos == n
    assert np.array_equal(v, want_v)
    assert np.array_equal(h[v], want_h[want_v])


def test_k1_golden_murmur_vectors(golden_dir):
    # every ACGT-only golden string of length <= 32 hashed as a (forward-canonical or not) k-mer
    for vec in json.load(open(os.path.join(golden_dir, "murmur_kat.json"))):
        data = bytes.fromhex(vec["hex"])
        if vec["seed"] != 42 or not (1 <= len(data) <= 32) or any(c not in b"ACGT" for c in data):
            continue
        k = len(data)
        rc = data.translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1]
        if data > rc:
            continue  # the k-mer hashed by mash is the canonical one
        seq, inv, n, _ = hs.pack_text(b">x\n" + data + b"\n")
        h, v = hs.hash_packed(k, 42, seq, inv, n)
        assert v.sum() == 1
        want = int(vec["h1"], 16)
        assert int(h[v][0]) == (want if k > 16 else want & 0xFFFFFFFF)


def test_k1_empty_and_padding():
    seq, inv, n, _ = hs.pack_text(b"")
    assert n == 0
    seq, inv, n, _ = hs.pack_text(b">a\n" + b"N" * 100 + b"\n")
    h, v = hs.hash_packed(21, 42, seq, inv, n)
    assert not v.any()


# ------------------------------------------------ device FASTA parser (row a6) ---
def test_device_parser_equals_host_packer():
    rng = random.Random(61)
    cases = [
        b">only_header\n",
        b">short\nACGT\n",
        b">a\n" + b"A" * 64 + b"\n>b\n" + b"C" * 64 + b"\n",
        b">crlf\r\nACGTACGTACGTACGTACGTACGT\r\nACGTACGT\r\n>x\r\nAC\r\rGT\r\n",
        b">nonl\nACGTACGTACGTACGTACGTACGTACG",
        b">nonl_cr\nACGTACGT\r",
        b">x\nACGTACGTACGT ACGTACGTACGTACG\tTACGTACGT\n",
        b"junk before header\nmore junk\n>x\n" + b"GATTACA" * 9 + b"\n\n\n>y\n\n" + b"TTGACCA" * 9 + b"\n",
        b"\n\n>lead\nACGT>notheader\n>real header > with gt\nGG>CC\n",
        b">plus\nACGTACGT\n+\nIIIIIIII\nACGT\n>next\nTTTT\n",
        b">big\n" + bytes(rng.choice(b"ACGTacgtNn") for _ in range(100_000)) + b"\n",
    ]
    text = ""
    for r in range(300):
        L = rng.choice([0, 1, 31, 32, 33, 79, 80, 81, 500, 8191, 8192, 8193, 30000])
        s = "".join(rng.choice("ACGTacgtNRY") if rng.random() < 0.01 else rng.choice("ACGT") for _ in range(L))
        w = rng.choice([60, 70, 80, 10 ** 9])
        text += ">r%d some text\n" % r + "\n".join(s[i:i + w] for i in range(0, len(s), w)) + "\n"
    cases.append(text.encode())
    for t in cases:
        hs_, hi, hn, hst = hs.pack_text(t)
        ds, di, dn, dst = hs.pack_text_device(t)
        assert dn == hn, t[:40]
        assert (dst["n_records"], dst["n_bases"]) == (hst["n_records"], hst["n_bases"])
        assert np.array_equal(di, hi) and np.array_equal(ds, hs_), t[:40]


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_ingest_modes_agree_on_pinned_text(c1_case, mode):
    import torch
    offsets, hashes, lengths, fasta = c1_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    want = odb.screen_text(fasta, threads=2)
    pinned = torch.empty(len(fasta), dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = np.frombuffer(fasta, np.uint8)
    scr = hs.Screen(db)
    scr.set_option("ingest", mode)
    scr.set_option("chunk_bases", 300_000)
    scr.feed_text_ptr(pinned.data_ptr(), pinned.numel(), 6)   # >= 6 threads: packer threads and the device parser compete in mode 2
    res = scr.finish(False)
    assert res.shared.tolist() == want.shared.tolist() and res.median.tolist() == want.median.tolist()
    assert res.set_size == want.set_size
    assert res.stats["n_bases"] == want.n_bases and res.stats["n_valid_kmers"] == want.n_kmers


# ---------------------------------------------------------------- K2 ----------
def test_k2_probe_membership_and_canonical_ids():
    rng = np.random.default_rng(5)
    n_refs, s = 300, 200
    pool = rng.integers(0, 2 ** 62, size=20000, dtype=np.uint64)
    pool[0] = 0; pool[1] = np.uint64(2 ** 64 - 1); pool[2] = np.uint64(2 ** 64 - 2)
    sk = [np.unique(rng.choice(pool, size=s, replace=False)) for _ in range(n_refs)]
    sk[0] = np.unique(np.concatenate([sk[0], pool[:3]]))
    offsets = np.concatenate([[0], np.cumsum([len(x) for x in sk])]).astype(np.uint64)
    hashes = np.concatenate(sk)
    db = hs.Database.from_arrays(21, s, 42, offsets, hashes, np.ones(n_refs, np.uint64))
    first = {}
    for e, h in enumerate(hashes.tolist()):
        first.setdefault(h, e)
    assert db.n_distinct == len(first)
    assert db.entry_ids().tolist() == [first[h] for h in hashes.tolist()]
    q = np.concatenate([pool, rng.integers(0, 2 ** 64, size=50000, dtype=np.uint64)])
    got = db.probe(q)
    want = np.array([first.get(h, 0xFFFFFFFF) for h in q.tolist()], np.uint32)
    assert np.array_equal(got, want)


# ---------------------------------------------------------------- K6 ----------
def test_k6_identity_pvalue_golden(golden_dir):
    vecs = json.load(open(os.path.join(golden_dir, "pvalue_kat.json")))
    for key in sorted({(v["k"], v["set_size"]) for v in vecs}):
        grp = [v for v in vecs if (v["k"], v["set_size"]) == key]
        ident, pv = hs.stat_batch(key[0], key[1], [v["x"] for v in grp], [v["n"] for v in grp])
        for v, i_, p_ in zip(grp, ident, pv):
            want_p, want_i = float(v["p"]), float(v["identity"])
            assert abs(i_ - want_i) <= RTOL * want_i, v
            if want_p < 1e-300:
                assert p_ == pytest.approx(want_p, rel=1e-6, abs=1e-320), v
            else:
                assert abs(p_ - want_p) <= RTOL * want_p, (v, p_)


def test_k6_matches_oracle_dense_grid():
    rng = np.random.default_rng(11)
    for k, ss in [(21, 10 ** 9), (21, 3 * 10 ** 6), (31, 10 ** 10), (16, 10 ** 6), (11, 5 * 10 ** 5)]:
        n = rng.choice([1000, 1000, 5000, 10000, 437], size=400).astype(np.uint64)
        x = (rng.random(400) ** 2 * n).astype(np.uint64)
        x[:20] = 0; x[20:40] = n[20:40]
        ident, pv = hs.stat_batch(k, ss, x, n)
        L = orc.lib()
        for i in range(400):
            wi = L.orc_identity(int(x[i]), int(n[i]), k)
            wp = L.orc_pvalue(int(x[i]), ss, 4.0 ** k, int(n[i]))
            assert abs(ident[i] - wi) <= RTOL * wi
            if wp < 1e-300:
                assert pv[i] < 1e-299
            else:
                assert abs(pv[i] - wp) <= RTOL * wp, (k, ss, int(x[i]), int(n[i]), pv[i], wp)


# ------------------------------------------------------- mixture / sketch -------
@pytest.mark.parametrize("k,s", [(21, 1000), (16, 500), (31, 64)])
def test_gpu_sketch_equals_oracle_sketch(k, s):
    rng = np.random.default_rng(k)
    g = synth.random_genome(rng, 300_000, n_frac=0.001)
    fa = synth.to_fasta([g[:120_000], g[120_000:]], "chr")
    got, ln = hs.sketch_text(fa, k, s)
    want, wln = orc.sketch_text(fa, k, s)
    assert ln == wln == 300_000
    assert got.tolist() == want.tolist()


def test_mixture_fewer_than_s_and_repetitive():
    # S9: fewer than s distinct k-mers -> all of them; heavy duplication -> re-thresholding path
    unit = synth.random_genome(np.random.default_rng(1), 700)
    fa = synth.to_fasta([unit] * 3, "dup")
    got, _ = hs.sketch_text(fa, 21, 1000)
    want, _ = orc.sketch_text(fa, 21, 1000)
    assert len(want) == 680 and got.tolist() == want.tolist()
    big = synth.to_fasta([np.tile(synth.random_genome(np.random.default_rng(2), 5000), 400)], "rep", width=0)
    got, _ = hs.sketch_text(big, 21, 1000)   # 2 Mbp but only ~5000 distinct k-mers
    want, _ = orc.sketch_text(big, 21, 1000)
    assert got.tolist() == want.tolist()


# ---------------------------------------------------------------- full screen ---
def golden_db(g):
    hsl = [np.array([int(h) for h in r["hashes"]], np.uint64) for r in g["db"]]
    offsets = np.concatenate([[0], np.cumsum([len(h) for h in hsl])]).astype(np.uint64)
    return offsets, np.concatenate(hsl), np.array([r["length"] for r in g["db"]], np.uint64)


@pytest.mark.parametrize("mode", ["plain", "wta"])
def test_screen_small_golden(golden_dir, mode):
    g = json.load(open(os.path.join(golden_dir, "screen_small.json")))
    offsets, hashes, lengths = golden_db(g)
    db = hs.Database.from_arrays(g["k"], g["s"], g["seed"], offsets, hashes, lengths)
    scr = hs.Screen(db)
    scr.feed_text(g["fasta"].encode(), 1)
    res = scr.finish(mode == "wta")
    want = g["results"][mode]
    assert res.shared.tolist() == want["shared"]
    assert res.median.tolist() == want["median"]
    assert res.set_size == want["set_size"]
    assert [str(int(h)) for h in scr.mixture()] == want["mixture"]
    assert rel_close(res.identity, want["identity"])
    assert rel_close(res.pvalue, want["pvalue"])


@pytest.fixture(scope="module")
def c1_case():
    """Config 1 shape, scaled to seconds of oracle time: 200 genomes x 50 kb, k=21 s=1000,
    2 Mbp of contigs cut from 20 of them at m in {0, 0.01, 0.05}."""
    rng = np.random.default_rng(1)
    genomes = [synth.random_genome(rng, 50_000, n_frac=0.001) for _ in range(200)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    contigs = []
    for m in (0.0, 0.01, 0.05):
        contigs += synth.cut_contigs(rng, genomes[:20], 700_000, m, median=6000.0)
    fasta = synth.to_fasta(contigs, "contig", lower_frac=0.05, rng=rng)
    return offsets, hashes, lengths, fasta


@pytest.mark.parametrize("wta", [False, True])
@pytest.mark.parametrize("feed", ["text", "packed"])
def test_screen_c1_shape(c1_case, wta, feed):
    offsets, hashes, lengths, fasta = c1_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    res, want = compare_screen(db, odb, fasta, wta, threads=3, feed=feed)
    assert int(res.shared.sum()) > 10_000  # the case really exercises hits


def test_filter_off_is_identical_and_probes_everything(c1_case):
    offsets, hashes, lengths, fasta = c1_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    on, _ = compare_screen(db, odb, fasta, False, probe_filter=True)
    off, _ = compare_screen(db, odb, fasta, False, probe_filter=False)
    assert off.stats["n_probes"] == off.stats["n_valid_kmers"]
    assert on.stats["n_probes"] <= off.stats["n_probes"]
    assert on.stats["n_hits"] == off.stats["n_hits"]


@pytest.mark.parametrize("k,s", [(16, 400), (31, 1000), (21, 5000)])
def test_screen_other_k_and_s(k, s):
    rng = np.random.default_rng(100 + k)
    genomes = [synth.random_genome(rng, 40_000) for _ in range(30)]
    offsets, hashes, lengths = build_db(genomes, k, s)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[:10], 400_000, 0.02, median=5000.0), "c")
    db = hs.Database.from_arrays(k, s, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(k, s, 42, offsets, hashes, lengths)
    compare_screen(db, odb, fasta, False)
    compare_screen(db, odb, fasta, True)


def test_wta_clusters_with_ties():
    """Config 4 shape: clusters of near-identical references (1-5 % divergence), equal-length
    members (exact (score, length) ties -> highest index) and length-perturbed ones."""
    rng = np.random.default_rng(4)
    genomes = []
    for c in range(12):
        anc = synth.random_genome(rng, 60_000)
        for m in range(6):
            g = synth.mutate(anc, float(rng.uniform(0.01, 0.05)), rng)
            genomes.append(g if m < 2 else g[:60_000 - int(rng.integers(1, 999))])
        genomes.append(genomes[-1].copy())  # exact duplicate sketch: full tie
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[::7], 600_000, 0.0, median=8000.0), "c")
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    plain, _ = compare_screen(db, odb, fasta, False)
    wta, _ = compare_screen(db, odb, fasta, True)
    assert wta.shared.sum() < plain.shared.sum()          # reassignment removed shared credit
    dup = [i for i in range(len(genomes)) if i % 7 == 6]
    assert all(wta.shared[i - 1] == 0 or wta.shared[i] >= wta.shared[i - 1] for i in dup)


def test_reset_and_chunked_feeds_agree(c1_case):
    offsets, hashes, lengths, fasta = c1_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    scr = hs.Screen(db)
    scr.set_option("chunk_bases", 70_000)   # many small chunks, several packer threads
    scr.feed_text(fasta, 4)
    a = scr.finish(False)
    scr.reset()
    half = fasta.rfind(b"\n>", 0, len(fasta) // 2) + 1
    scr.feed_text(fasta[:half], 1); scr.feed_text(fasta[half:], 2)
    b = scr.finish(False)
    assert a.shared.tolist() == b.shared.tolist() and a.median.tolist() == b.median.tolist()
    assert a.set_size == b.set_size
    # idempotence of multiplicity: the same query twice doubles every median, keeps shared
    scr.reset()
    scr.feed_text(fasta, 2); scr.feed_text(fasta, 2)
    c = scr.finish(False)
    assert c.shared.tolist() == a.shared.tolist()
    assert c.median.tolist() == (2 * a.median).tolist()


@pytest.mark.parametrize("wta", [False, True])
def test_flush_async_completes_in_finish(c1_case, wta, monkeypatch):
    """hs_screen_flush_async: the bottom-s selection is enqueued and the next finish completes the flush
    with its single synchronisation -- same mixture, set size and rows as the waiting flush; and when the
    selection is made to report "not settled" a single process falls back to the iterative finaliser."""
    offsets, hashes, lengths, fasta = c1_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    ref = hs.Screen(db)
    ref.feed_text(fasta, 2)
    want = ref.finish(wta)
    want_mix = ref.mixture().tolist()
    ref.close()
    for forced in (False, True):
        if forced:
            monkeypatch.setenv("HYMET_SCREEN_FORCE_UNSETTLED", "1")
        scr = hs.Screen(db)
        monkeypatch.delenv("HYMET_SCREEN_FORCE_UNSETTLED", raising=False)
        for rep in range(2):          # the same handle again after a reset
            scr.feed_text(fasta, 2)
            scr.flush_async()
            got = scr.finish(wta)
            assert got.shared.tolist() == want.shared.tolist() and got.median.tolist() == want.median.tolist()
            assert got.set_size == want.set_size and scr.mixture().tolist() == want_mix
            assert got.identity.tolist() == want.identity.tolist() and got.pvalue.tolist() == want.pvalue.tolist()
            assert got.stats["n_valid_kmers"] == want.stats["n_valid_kmers"] and got.stats["n_bases"] == want.stats["n_bases"]
            scr.reset()
        scr.close()


# ---------------------------------------------------------------- drop-in -------
def write_db(tmp_path, genomes, k, s, **kw):
    offsets, hashes, lengths = build_db(genomes, k, s)
    db = mshfmt.SketchDB(k=k, s=s, names=[synth.gcf_name(i) for i in range(len(genomes))],
                         comments=["synthetic genome %d" % i for i in range(len(genomes))],
                         lengths=lengths, offsets=offsets, hashes=hashes)
    p = str(tmp_path / "db.msh")
    mshfmt.write_msh(p, db, **kw)
    return p


def test_cli_tsv_byte_identical_to_oracle_cli(tmp_path):
    rng = np.random.default_rng(8)
    genomes = [synth.random_genome(rng, 30_000) for _ in range(40)]
    dbp = write_db(tmp_path, genomes, 21, 1000, seg_cap_words=1 << 13, double_far_refs=[3])
    fa1, fa2 = str(tmp_path / "a.fna"), str(tmp_path / "b.fna.gz")
    open(fa1, "wb").write(synth.to_fasta(synth.cut_contigs(rng, genomes[:8], 200_000, 0.01, median=4000.0), "a"))
    import gzip
    gzip.open(fa2, "wb").write(synth.to_fasta(synth.cut_contigs(rng, genomes[5:12], 150_000, 0.03, median=4000.0), "b"))
    orc.build()
    for extra in ([], ["-w"], ["-i", "0.8"], ["-i", "-1", "-v", "0.9"]):
        args = ["screen", "-p", "4"] + extra + [dbp, fa1, fa2]
        got = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "mash")] + args, capture_output=True)
        want = subprocess.run([orc.BIN] + args, capture_output=True)
        assert got.returncode == 0 and want.returncode == 0, got.stderr.decode()
        assert got.stdout == want.stdout
        assert len(got.stdout.splitlines()) > 5
    # S21: errors
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "mash"), "screen", dbp, str(tmp_path / "none.fna")],
                       capture_output=True)
    assert r.returncode == 1 and b"ERROR" in r.stderr and r.stdout == b""


def run_mash_sh(tmp_path, script, mash_exe, tag, indir, dbp, thr):
    import stat

    from tests.test_stage_cpu import FAKE_BC
    bindir = tmp_path / ("bin_" + tag); bindir.mkdir()
    os.symlink(mash_exe, bindir / "mash")
    bc = bindir / "bc"                       # no bc in the image: exact-decimal stand-in (tests/test_stage_cpu.py)
    bc.write_text(FAKE_BC)
    bc.chmod(bc.stat().st_mode | stat.S_IXUSR)
    od = tmp_path / ("out_" + tag); od.mkdir()
    files = [str(od / f) for f in ("screen.tab", "filtered.tab", "sorted.tab", "top_hits.tab", "selected.txt")]
    env = dict(os.environ, PATH=str(bindir) + os.pathsep + os.environ["PATH"], LC_ALL="C")
    p = subprocess.run(["bash", script, str(indir), dbp] + files + [thr], capture_output=True, env=env)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return [open(f, "rb").read() for f in files], p.stdout.decode()


@pytest.mark.parametrize("seed,n_genomes,n_files,thr,rates,per_file", [
    (1, 24, 1, "0.9", (0.0,), 5),                        # first threshold is enough
    (5, 10, 3, "0.9", (0.0, 0.12, 0.2), 2),              # the bc/awk loop steps down to .78
    (7, 3, 1, "0.9", (0.1,), 2),                         # never enough candidates: the 0.71 fallback
])
def test_full_reference_mash_sh_with_gpu_mash(tmp_path, golden_dir, seed, n_genomes, n_files, thr, rates, per_file):
    """/root/reference/scripts/mash.sh:1-59, UNMODIFIED (fixture), with bin/mash first on PATH: the
    screen (line 14), both sorts, the min-candidates arithmetic, the threshold loop and the fallback
    (lines 19-51) leave the same five files and the same log as with the oracle CLI as `mash`, and as
    hymet_b200.stage.select computes."""
    from hymet_b200 import stage
    from tests.test_stage_cpu import make_case
    script = reference_mash_sh(tmp_path, golden_dir)
    dbp, indir = make_case(tmp_path, seed, n_genomes, n_files, rates=rates, per_file=per_file)
    orc.build()
    gpu, gpu_log = run_mash_sh(tmp_path, script, os.path.join(ROOT, "bin", "mash"), "gpu", indir, dbp, thr)
    ora, ora_log = run_mash_sh(tmp_path, script, orc.BIN, "oracle", indir, dbp, thr)
    assert gpu == ora and gpu_log == ora_log
    assert gpu[0].count(b"\n") >= 3
    _, n_find = stage.input_files(indir)
    r = stage.select(gpu[0], n_find, thr)
    assert [r["filtered"], r["sorted"], r["top_hits"], r["selected"]] == gpu[1:] and r["log"] == gpu_log
    if seed == 5:
        assert gpu_log.count("Testing threshold") > 3
    if seed == 7:
        assert "No suitable threshold found" in gpu_log


@pytest.mark.parametrize("thr", ["0.9", "0.82"])
def test_full_reference_mash_sh_on_real_genomes(tmp_path, golden_dir, thr):
    """Same, on the Zymo fixture: the files the unmodified script left behind in the build container
    (tests/golden/zymo_mash_sh.json, oracle CLI as `mash`) are reproduced with the GPU `mash`."""
    import gzip
    script = reference_mash_sh(tmp_path, golden_dir)
    indir = tmp_path / "input"; indir.mkdir()
    (indir / "sample_0.fna").write_bytes(gzip.open(os.path.join(golden_dir, "zymo_query.fna.gz"), "rb").read())
    got, log = run_mash_sh(tmp_path, script, os.path.join(ROOT, "bin", "mash"), "gpu", indir,
                           os.path.join(golden_dir, "zymo25.msh"), thr)
    want = json.load(open(os.path.join(golden_dir, "zymo_mash_sh.json")))[thr]
    assert got[0] == open(os.path.join(golden_dir, "zymo_screen.tsv"), "rb").read()
    assert [g.decode() for g in got[1:]] == [want["filtered"], want["sorted"], want["top_hits"], want["selected"]]
    assert log == want["log"]


# ------------------------------------------------- BASELINE-size properties -------
def test_baseline_shape_properties():
    """Config-2 shape (50 000 sketches, CAMI-shaped contigs, here 300 Mbp to stay within seconds):
    results that do not need the oracle -- the three entry points agree, the exact pre-filter
    changes nothing, multiplicities are linear in the input, planted genomes are found and
    decoys are not, counts add up, winner-take-all assigns every present hash exactly once."""
    import torch

    from hymet_b200 import dist as hd
    from hymet_b200 import workload
    wl = workload.make_c2(0, mbp=300, n_sketches=50_000, n_real=120, with_fasta=True, with_host_packed=True)
    db = hs.Database.from_arrays(wl.k, wl.s, 42, wl.offsets, wl.hashes, wl.lengths)
    scr = hs.Screen(db)

    def run(feed, wta=False, twice=False, probe_filter=True):
        scr.reset()
        scr.set_option("filter", int(probe_filter))
        for _ in range(2 if twice else 1):
            feed()
        r = scr.finish(wta)
        return r

    dev = lambda: scr.feed_packed_device(wl.d_seq.data_ptr(), wl.d_inv.data_ptr(), wl.n_positions)
    host = lambda: scr.feed_packed_ptr(wl.h_seq.data_ptr(), wl.h_inv.data_ptr(), wl.n_positions)
    text = lambda: scr.feed_text_ptr(wl.fasta.data_ptr(), wl.fasta.numel(), 8)
    a = run(dev)
    assert a.stats["n_valid_kmers"] > 0.99 * wl.n_bases
    for other in (run(host), run(text), run(dev, probe_filter=False)):
        assert other.shared.tolist() == a.shared.tolist() and other.median.tolist() == a.median.tolist()
        assert other.set_size == a.set_size
    assert run(dev, probe_filter=False).stats["n_probes"] == a.stats["n_valid_kmers"]
    # probe-everything keeps the load/store pipe saturated: the regime in which a missing proxy fence
    # in the TMA tile pipeline corrupted ~1 word per 1e9 (DESIGN.md 5).  Counts must be identical.
    ref_counts = None
    for _ in range(3):
        r = run(dev, probe_filter=False)
        c = hd.counts_tensor(scr, 0).clone()
        torch.cuda.synchronize()
        assert r.stats["n_hits"] == a.stats["n_hits"]
        assert ref_counts is None or bool(torch.equal(c, ref_counts))
        ref_counts = c
    # linearity: the same contigs twice -> same shared hashes, doubled multiplicities, same mixture
    b = run(dev, twice=True)
    assert b.shared.tolist() == a.shared.tolist() and b.median.tolist() == (2 * a.median).tolist()
    assert b.set_size == a.set_size
    # planted truth: contigs come from the first 120 sketches at 1 % substitutions; decoys are random hashes
    real, decoy = a.shared[:wl.n_real], a.shared[wl.n_real:]
    assert int(decoy.sum()) == 0
    assert (real > 0.5 * wl.s).sum() >= 0.9 * wl.n_real          # expected containment ~ 0.99^21 = 0.81
    assert np.all(a.identity[:wl.n_real][real > 0] > 0.9) and np.all(a.pvalue[:wl.n_real][real > 100] < 1e-50)
    # counts add up to the kernel's own hit counter
    run(dev)
    counts = hd.counts_tensor(scr, 0)
    torch.cuda.synchronize()
    assert int(counts.to(torch.int64).sum()) == a.stats["n_hits"]
    present = int((counts != 0).sum())
    # winner-take-all: every present hash credited to exactly one sketch
    w = run(dev, wta=True)
    assert int(w.shared.sum()) == present
    assert int(w.shared.sum()) <= int(a.shared.sum())
    scr.close()


def test_cli_sketch_then_screen(tmp_path):
    """`mash sketch` on the GPU writes a .msh that all three readers accept, equal to the oracle's
    sketches, and `mash screen` against it finds the genomes the contigs came from."""
    rng = np.random.default_rng(12)
    genomes = [synth.random_genome(rng, 80_000) for _ in range(6)]
    paths = []
    for i, g in enumerate(genomes):
        p = tmp_path / (synth.gcf_name(i)); paths.append(str(p))
        p.write_bytes(synth.to_fasta([g[:50_000], g[50_000:]], "chr"))
    mash = [sys.executable, os.path.join(ROOT, "bin", "mash")]
    out = str(tmp_path / "db")
    r = subprocess.run(mash + ["sketch", "-k", "21", "-s", "500", "-o", out] + paths, capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    db = mshfmt.read_msh(out + ".msh")
    assert (db.k, db.s, db.n_refs) == (21, 500, 6) and db.names == paths
    assert db.comments[0].startswith("[2 seqs] chr_0")
    odb = orc.OracleDB.load_msh(out + ".msh")
    for i, p in enumerate(paths):
        want, ln = orc.sketch_text(open(p, "rb").read(), 21, 500)
        assert db.ref_hashes(i).tolist() == want.tolist() and int(db.lengths[i]) == ln == 80_000
        assert odb.hashes(i).tolist() == want.tolist()
    q = tmp_path / "q.fna"
    q.write_bytes(synth.to_fasta(synth.cut_contigs(rng, genomes[:2], 200_000, 0.005, median=5000.0), "c"))
    r = subprocess.run(mash + ["screen", "-v", "0.9", out + ".msh", str(q)], capture_output=True)
    assert r.returncode == 0
    hits = [l.split(b"\t")[4].decode() for l in r.stdout.splitlines()]
    assert hits == paths[:2]


def test_bloom_second_level_filter_is_exact():
    """A database with tiny genomes keeps ALL their k-mer hashes, so max_key ~ 2^64 and the range
    test passes everything; the Bloom second level is built and must not change any result."""
    rng = np.random.default_rng(77)
    genomes = [synth.random_genome(rng, 40_000) for _ in range(20)]
    genomes += [synth.random_genome(rng, int(n)) for n in rng.integers(300, 3000, size=40)]   # < s k-mers each
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[:6] + genomes[20:30], 500_000, 0.01, median=2500.0, lo=300), "c")
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    assert db.info.max_key > 2 ** 63 and db.info.bloom_bytes > 0
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    res, want = compare_screen(db, odb, fasta, False)
    compare_screen(db, odb, fasta, True)
    off, _ = compare_screen(db, odb, fasta, False, probe_filter=False)
    assert res.stats["n_hits"] == off.stats["n_hits"] and res.stats["n_probes"] < 0.2 * off.stats["n_probes"]
    assert int(res.shared[20:30].min()) > 100     # the tiny genomes in the query are found


# ------------------------------------------------- rows a2/a3: three sketch files, one pass -------
def _three_dbs(tmp_path, rng):
    """sketch1-3.msh stand-ins: overlapping reference sets (a hash may live in all three), the
    third with a different sketch size; returns paths + the genomes."""
    genomes = [synth.random_genome(rng, 30_000) for _ in range(36)]
    genomes += [synth.mutate(genomes[i], 0.02, rng) for i in range(6)]          # relatives: -w has work to do
    sets = [(list(range(0, 20)) + [36, 37], 1000), (list(range(10, 30)) + [38, 39, 0], 1000),
            (list(range(25, 36)) + [40, 41, 5, 12], 500)]
    paths = []
    for j, (idx, s) in enumerate(sets):
        offsets, hashes, lengths = build_db([genomes[i] for i in idx], 21, s)
        db = mshfmt.SketchDB(k=21, s=s, names=[synth.gcf_name(i) for i in idx], comments=["db%d genome %d" % (j, i) for i in idx],
                             lengths=lengths - np.arange(len(idx), dtype=np.uint64) % np.uint64(3), offsets=offsets, hashes=hashes)
        p = str(tmp_path / ("sketch%d.msh" % (j + 1)))
        mshfmt.write_msh(p, db)
        paths.append(p)
    return paths, genomes


@pytest.mark.parametrize("wta", [False, True])
def test_multi_file_db_equals_one_screen_per_file(tmp_path, wta):
    rng = np.random.default_rng(21)
    paths, genomes = _three_dbs(tmp_path, rng)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[:32:3] + genomes[36:40], 400_000, 0.01, median=5000.0), "q")
    db = hs.Database.load_msh_multi(paths)
    segs = db.segments
    assert len(segs) == 3 and db.segment_s == [1000, 1000, 500] and db.s == 1000 and segs[-1][1] == db.n_refs
    scr = hs.Screen(db)
    scr.feed_text(fasta, 2)
    res = scr.finish(wta)
    for j, (p, (b, e)) in enumerate(zip(paths, segs)):
        odb = orc.OracleDB.load_msh(p)
        want = odb.screen_text(fasta, threads=2, wta=wta)
        assert e - b == odb.n_refs
        assert res.shared[b:e].tolist() == want.shared.tolist()
        assert res.median[b:e].tolist() == want.median.tolist()
        assert scr.segment_set_size(j) == want.set_size
        assert scr.mixture()[:db.segment_s[j]].tolist() == want.mixture.tolist()
        assert rel_close(res.identity[b:e], want.identity) and rel_close(res.pvalue[b:e], want.pvalue)
        assert [db.names[i] for i in range(b, e)] == [odb.name(i) for i in range(odb.n_refs)]
        if wta:
            assert int(want.shared.sum()) > 0
    scr.close()
    # files that disagree in k cannot share a table
    offsets, hashes, lengths = build_db(genomes[:3], 16, 200)
    other = str(tmp_path / "k16.msh")
    mshfmt.write_msh(other, mshfmt.SketchDB(k=16, s=200, names=list("abc"), comments=[""] * 3, lengths=lengths,
                                            offsets=offsets, hashes=hashes))
    with pytest.raises(hs.HsError, match="one at a time"):
        hs.Database.load_msh_multi([paths[0], other])


def test_fused_mash_stage_equals_three_reference_runs(tmp_path):
    """bin/hymet-mash-stage (one pass over the contigs for sketch1-3) leaves the same fifteen files and
    the same merged candidate list as run_hymet_cami.sh:85-97 = three mash.sh runs; the per-file `mash
    screen` output comes from the oracle CLI, mash.sh:15-55 from hymet_b200.stage.select, which
    tests/test_stage_cpu.py pins against the unmodified reference script."""
    from hymet_b200 import stage
    rng = np.random.default_rng(22)
    paths, genomes = _three_dbs(tmp_path, rng)
    indir = tmp_path / "input"; indir.mkdir()
    (indir / "sample_0.fna").write_bytes(synth.to_fasta(synth.cut_contigs(rng, genomes[:30:2], 300_000, 0.01, median=5000.0), "s"))
    (indir / "sample_1.fna").write_bytes(synth.to_fasta(synth.cut_contigs(rng, genomes[20:40], 200_000, 0.06, median=3000.0), "t"))
    (indir / "notes.txt").write_text("not a contig file\n")
    orc.build()
    files, n_fna = stage.input_files(str(indir))
    assert n_fna == 2
    od = tmp_path / "out"; od.mkdir()
    tags = ("", "gtdb_", "custom_")
    outs = [[str(od / (t + f)) for f in ("screen.tab", "filtered.tab", "sorted.tab", "top_hits.tab", "selected_genomes.txt")]
            for t in tags]
    argv = ["--merge", "-p", "4", str(indir), "0.9"]
    for p, o in zip(paths, outs):
        argv += [p] + o
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "hymet-mash-stage")] + argv, capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    want_sel, want_log = [], ""
    for p, o in zip(paths, outs):
        tab = subprocess.run([orc.BIN, "screen", "-p", "8", "-v", "0.9", p] + files, capture_output=True, check=True).stdout
        assert tab.count(b"\n") >= 5
        w = stage.select(tab, n_fna, "0.9")
        assert open(o[0], "rb").read() == tab
        for path, key in zip(o[1:4], ("filtered", "sorted", "top_hits")):
            assert open(path, "rb").read() == w[key], path
        want_sel.append(w["selected"])
        want_log += w["log"]
    assert open(outs[1][4], "rb").read() == want_sel[1] and open(outs[2][4], "rb").read() == want_sel[2]
    assert open(outs[0][4], "rb").read() == stage.merge_selected(want_sel)       # run_hymet_cami.sh:91,96,97
    assert r.stdout.decode() == want_log
    # and the one-file drop-in prints what the fused pass wrote for that file
    one = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "mash"), "screen", "-p", "8", "-v", "0.9", paths[2]] + files,
                         capture_output=True, check=True).stdout
    assert one == open(outs[2][0], "rb").read()


def test_fused_stage_survives_missing_and_broken_sketch_files(tmp_path, golden_dir):
    """run_hymet_cami.sh:85-97 with data/sketch3.msh absent and sketch2.msh unreadable: scripts/mash.sh has
    no `set -e`, so the failed `mash screen` leaves an empty screen.tab, lines 15-55 still write their
    (empty) files and log, and the run goes on with sketch1's candidates.  The fused stage must leave
    exactly what the three UNMODIFIED mash.sh runs leave (oracle CLI as `mash`)."""
    from hymet_b200 import stage
    rng = np.random.default_rng(23)
    paths, genomes = _three_dbs(tmp_path, rng)
    open(paths[1], "wb").write(b"this is not a capnp message" * 10)       # sketch2: malformed
    os.remove(paths[2])                                                   # sketch3: absent
    indir = tmp_path / "input"; indir.mkdir()
    (indir / "sample_0.fna").write_bytes(synth.to_fasta(synth.cut_contigs(rng, genomes[:30:2], 300_000, 0.01, median=5000.0), "s"))
    script = reference_mash_sh(tmp_path, golden_dir)
    orc.build()
    tags = ("", "gtdb_", "custom_")
    od = tmp_path / "out"; od.mkdir()
    outs = [[str(od / (t + f)) for f in ("screen.tab", "filtered.tab", "sorted.tab", "top_hits.tab", "selected_genomes.txt")]
            for t in tags]
    argv = ["--merge", "-p", "4", str(indir), "0.9"]
    for p, o in zip(paths, outs):
        argv += [p] + o
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "hymet-mash-stage")] + argv, capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    assert r.stderr.count(b"ERROR") >= 2
    want_log, want_sel = "", []
    for j, p in enumerate(paths):
        got, log = run_mash_sh(tmp_path, script, orc.BIN, "ref%d" % j, indir, p, "0.9")
        for path, data in zip(outs[j][:4], got[:4]):
            assert open(path, "rb").read() == data, path
        want_sel.append(got[4])
        want_log += log
    assert want_sel[1] == b"" and want_sel[2] == b"" and want_sel[0].count(b"\n") >= 3
    assert open(outs[1][4], "rb").read() == b"" and open(outs[2][4], "rb").read() == b""
    assert open(outs[0][4], "rb").read() == stage.merge_selected(want_sel)
    assert r.stdout.decode() == want_log


# ------------------------------------------------- row a6: plain FASTA files streamed through the pinned ring -------
@pytest.mark.parametrize("variant", ["plain", "crlf_no_final_newline", "leading_blank_lines", "one_record"])
def test_file_streaming_blocks_and_giant_records(tmp_path, variant):
    """hs_screen_feed_fasta on a plain FASTA file: reader threads cut the file into blocks of whole
    records for the device parser.  Tiny blocks (64 KiB) put hundreds of block boundaries inside the
    file, records longer than a ring slot (the 300 kb ones) take the host path; the result must not
    depend on any of it."""
    rng = np.random.default_rng(33)
    genomes = [synth.random_genome(rng, 300_000) for _ in range(6)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    contigs = synth.cut_contigs(rng, genomes, 3_000_000, 0.01, median=9000.0) + [genomes[2], synth.revcomp(genomes[4])]
    order = rng.permutation(len(contigs))
    text = synth.to_fasta([contigs[i] for i in order], "c")
    if variant == "crlf_no_final_newline":
        text = text.replace(b"\n", b"\r\n").rstrip(b"\r\n")
    elif variant == "leading_blank_lines":
        text = b"\n\n" + text
    elif variant == "one_record":
        text = synth.to_fasta([genomes[1]], "whole")
    path = str(tmp_path / "contigs.fna")
    open(path, "wb").write(text)
    want = odb.screen_text(text, threads=2)
    assert int(want.shared.sum()) >= 1000
    # file_mode 0: pread ring -> device parser; 1: the file mapped and packed by the host threads (16 KiB spans:
    # hundreds of them, so both the 64-byte block path of the packer and its line path meet every boundary)
    # (mode -1: "ingest" 0 = host packers only, which takes the mapped form whatever file_mode says)
    for mode, block, readers in ((0, 65536, 3), (0, 1 << 20, 2), (0, 16 << 20, 4), (1, 0, 4), (1, 16384, 5), (-1, 50_000, 2)):
        scr = hs.Screen(db)
        if mode < 0:
            scr.set_option("ingest", 0)
        scr.set_option("file_mode", max(mode, 0))
        if mode == 0:
            scr.set_option("file_block_bytes", block)
            scr.set_option("file_readers", readers)
        elif block:
            scr.set_option("chunk_bases", block)
        scr.feed_fasta(path, readers if mode else 4)
        res = scr.finish(False)
        assert res.shared.tolist() == want.shared.tolist(), (variant, block)
        assert res.median.tolist() == want.median.tolist()
        assert res.set_size == want.set_size and scr.mixture().tolist() == want.mixture.tolist()
        assert res.stats["n_valid_kmers"] == want.n_kmers
        assert res.stats["n_records"] == text.count(b">")
        scr.close()


def test_cli_fastq_gzip_and_stdin_inputs(tmp_path):
    """Row a6's other input forms through the drop-in: FASTQ (single- and multi-line, quality lines that
    start with '@' / '>' / '+'), gzip, "-" = stdin, and several of them pooled into one mixture --
    byte-identical TSV to the oracle CLI."""
    import gzip
    from tests.test_host_emul import make_fastq
    rng = np.random.default_rng(41)
    genomes = [synth.random_genome(rng, 30_000) for _ in range(12)]
    dbp = write_db(tmp_path, genomes, 21, 1000)
    contigs = synth.cut_contigs(rng, genomes[:7], 160_000, 0.01, median=3000.0)
    seqs = [synth.ASCII[c].tobytes().decode() for c in contigs]
    half = len(seqs) // 2
    fq1, fq2 = str(tmp_path / "reads.fq"), str(tmp_path / "more.fastq.gz")
    fa3 = str(tmp_path / "rest.fna")
    open(fq1, "w").write(make_fastq(seqs[:half], multiline=False))
    with gzip.open(fq2, "wb") as fh:
        fh.write(make_fastq(seqs[half:], multiline=True, crlf=True).encode())
    open(fa3, "wb").write(synth.to_fasta(synth.cut_contigs(rng, genomes[6:10], 90_000, 0.02, median=3000.0), "x"))
    orc.build()
    mash = [sys.executable, os.path.join(ROOT, "bin", "mash")]
    for inputs, stdin in (([fq1], None), ([fq2], None), ([fq1, fq2, fa3], None), (["-"], open(fq1, "rb").read()),
                          (["-", fa3], open(fa3, "rb").read())):
        args = ["screen", "-p", "3", "-v", "0.9", dbp] + inputs
        got = subprocess.run(mash + args, input=stdin, capture_output=True)
        want = subprocess.run([orc.BIN] + args, input=stdin, capture_output=True)
        assert got.returncode == 0 and want.returncode == 0, (inputs, got.stderr.decode()[-400:], want.stderr.decode()[-200:])
        assert got.stdout == want.stdout, inputs
        assert got.stdout.count(b"\n") >= 2, (inputs, got.stdout)
    # the FASTQ of a set of sequences screens like their FASTA
    fa1 = str(tmp_path / "reads.fna")
    open(fa1, "w").write("".join(">r%d\n%s\n" % (i, s) for i, s in enumerate(seqs[:half])))
    a = subprocess.run(mash + ["screen", dbp, fq1], capture_output=True).stdout
    b = subprocess.run(mash + ["screen", dbp, fa1], capture_output=True).stdout
    assert a == b and a


@pytest.mark.parametrize("extra,name", [([], "zymo_screen.tsv"), (["-w"], "zymo_screen_w.tsv")])
def test_real_genome_golden_tsv(golden_dir, extra, name):
    """Real sequence instead of random bases: 25 RefSeq assemblies of the reference's Zymo case study
    (strain triplets, plasmids, rRNA repeats, soft-masked and N bases), sketched and screened by the
    oracle in the build container (tests/golden/make_zymo_golden.py).  The drop-in prints the committed
    TSV byte for byte, with and without -w."""
    msh, q = os.path.join(golden_dir, "zymo25.msh"), os.path.join(golden_dir, "zymo_query.fna.gz")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "mash"), "screen", "-p", "4", "-v", "0.9"] + extra + [msh, q],
                       capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    assert r.stdout == open(os.path.join(golden_dir, name), "rb").read()


def test_gzip_input_is_inflated_in_chunks_of_whole_records(tmp_path):
    """gzip (and stdin) FASTA is inflated chunk by chunk and handed to the packers in whole records:
    tiny chunks (records larger than a chunk included) give the result of the plain file."""
    import gzip
    rng = np.random.default_rng(52)
    genomes = [synth.random_genome(rng, 150_000) for _ in range(5)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    contigs = synth.cut_contigs(rng, genomes, 1_200_000, 0.01, median=6000.0) + [genomes[3]]   # one 150 kb record
    text = synth.to_fasta([contigs[i] for i in rng.permutation(len(contigs))], "c")
    path = str(tmp_path / "c.fna.gz")
    with gzip.open(path, "wb") as fh:
        fh.write(text)
    want = odb.screen_text(text, threads=2)
    for chunk in (4096, 100_000, 1 << 28):
        scr = hs.Screen(db)
        scr.set_option("text_chunk_bytes", chunk)
        scr.feed_fasta(path, 3)
        res = scr.finish(False)
        assert res.shared.tolist() == want.shared.tolist() and res.median.tolist() == want.median.tolist(), chunk
        assert res.set_size == want.set_size and res.stats["n_valid_kmers"] == want.n_kmers
        assert res.stats["n_records"] == text.count(b">")
        scr.close()


@pytest.mark.parametrize("multiline", [False, True])
def test_fastq_is_cut_at_whole_records_and_packed_by_all_threads(tmp_path, multiline):
    """A read set (FASTQ: plain, gzip) is inflated in bounded chunks and split across the packer threads at
    record headers found by the packer's own walk -- quality lines that start with '@', '>' or '+' included:
    same result as the equivalent FASTA, for every chunk size."""
    import gzip
    from tests.test_host_emul import make_fastq
    rng = np.random.default_rng(53)
    genomes = [synth.random_genome(rng, 60_000) for _ in range(6)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    reads = synth.cut_contigs(rng, genomes[:4], 500_000, 0.01, median=300.0)
    seqs = [synth.ASCII[c].tobytes().decode() for c in reads]
    fq = make_fastq(seqs, multiline=multiline).encode()
    fa = "".join(">r%d\n%s\n" % (i, q) for i, q in enumerate(seqs)).encode()
    want = odb.screen_text(fa, threads=2)
    plain, gz = str(tmp_path / "reads.fq"), str(tmp_path / "reads.fq.gz")
    open(plain, "wb").write(fq)
    with gzip.open(gz, "wb") as fh:
        fh.write(fq)
    for path, chunk, threads in ((plain, 1 << 28, 4), (gz, 3000, 3), (gz, 70_000, 5)):
        scr = hs.Screen(db)
        scr.set_option("text_chunk_bytes", chunk)
        scr.set_option("chunk_bases", 20_000)       # dozens of spans per chunk
        scr.feed_fasta(path, threads)
        res = scr.finish(False)
        assert res.shared.tolist() == want.shared.tolist() and res.median.tolist() == want.median.tolist(), (path, chunk)
        assert res.set_size == want.set_size and res.stats["n_valid_kmers"] == want.n_kmers
        assert res.stats["n_records"] == len(seqs) and res.stats["n_bases"] == sum(len(q) for q in seqs)
        scr.close()


@pytest.mark.parametrize("k,s", [(21, 1000), (31, 5000), (16, 400)])
def test_gpu_sketch_of_real_sequence(golden_dir, k, s):
    """`mash sketch` on the GPU against the oracle on real contigs (60 records of the Zymo fixture:
    soft-masked stretches, rRNA repeats, a few N): same bottom-s hashes, same total length."""
    import gzip
    text = gzip.open(os.path.join(golden_dir, "zymo_query.fna.gz"), "rb").read()
    h, total = hs.sketch_text(text, k, s)
    want, wtotal = orc.sketch_text(text, k, s, threads=2)
    assert h.tolist() == want.tolist() and total == wtotal and len(h) == s

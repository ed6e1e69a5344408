"""`mash dist` on the B200 (DESIGN.md §5 "mash dist"): every candidate pair's (common, denom) and p-value against the
C oracle's serial merge, the TSV byte for byte against the oracle's and the goldens, query blocks that split
on result-buffer overflow, sequence queries sketched on the fly, and a 20 000 x 20 000 collection."""
import gzip
import os
import subprocess
import sys

import numpy as np
import pytest

from hymet_b200 import distance as dist
from hymet_b200 import msh as mshfmt
from hymet_b200 import screen as hs
from hymet_b200 import synth
from oracle import real_mash
from tests import _distance_ref as dref
from tests import _oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASH = [sys.executable, os.path.join(ROOT, "bin", "mash")]


def mash(*args, **kw):
    return subprocess.run(MASH + [str(a) for a in args], capture_output=True, **kw)


def write_db(path, k, s, sketches, lengths, names=None, comments=None, seed=42):
    offsets = np.concatenate([[0], np.cumsum([len(x) for x in sketches])]).astype(np.uint64)
    n = len(sketches)
    db = mshfmt.SketchDB(k=k, s=s, seed=seed, names=names or ["seq%d" % i for i in range(n)],
                         comments=comments or ["comment %d" % i for i in range(n)],
                         lengths=np.asarray(lengths, np.uint64), offsets=offsets,
                         hashes=np.concatenate([np.asarray(x, np.uint64) for x in sketches]) if n else np.zeros(0, np.uint64))
    mshfmt.write_msh(str(path), db)
    return str(path)


def gpu_rows(ref_path, qry_path, max_d=1.0):
    ref = dist.HostMsh(ref_path)
    d = dist.Distance(ref)
    try:
        q = dist.HostMsh(qry_path)
        d.add_msh(q)
        q.close()
        return d.run_rows(max_d), d.stats()
    finally:
        d.close()
        ref.close()


def gpu_tsv(tmp_path, ref_path, qry_paths, *opts):
    r = mash("dist", *opts, ref_path, *qry_paths)
    assert r.returncode == 0, r.stderr.decode()
    return r.stdout


def assert_rows_match_oracle(rows, ref_db, qry_db, s_p, q_sample=None, max_d=1.0):
    q_idx = np.arange(qry_db.n_refs) if q_sample is None else np.asarray(q_sample)
    common, denom, pv = dref.oracle_pairs(ref_db, qry_db, s_p, q_idx)
    pos = {int(q): i for i, q in enumerate(q_idx)}
    sel = np.isin(rows.q, q_idx)
    got_c = np.zeros_like(common); got_d = np.zeros_like(denom)
    cand = np.zeros(common.shape, bool)
    qi = np.array([pos[int(q)] for q in rows.q[sel]], np.int64)
    ri = rows.r[sel].astype(np.int64)
    got_c[qi, ri] = rows.common[sel]; got_d[qi, ri] = rows.denom[sel]; cand[qi, ri] = True
    assert np.array_equal(got_c[cand], common[cand]) and np.array_equal(got_d[cand], denom[cand])
    # pairs that are not candidates share no hash at all
    assert np.all(common[~cand] == 0)
    p = rows.pvalue[sel]
    want = pv[qi, ri]
    have = p >= 0
    assert np.all(np.abs(p[have] - want[have]) <= 1e-12 * np.abs(want[have]))
    # a p-value is skipped only for pairs the host drops
    dd = np.array([dref.distance(int(c), int(d), ref_db.k) for c, d in zip(rows.common[sel][~have], rows.denom[sel][~have])])
    assert np.all(dd > max_d)
    return int(cand.sum())


# ---- zymo goldens ---------------------------------------------------------------------------------------------
def test_zymo_goldens(golden_dir, tmp_path):
    z = os.path.join(golden_dir, "zymo25.msh")
    assert mash("dist", z, z).stdout == open(os.path.join(golden_dir, "zymo_dist.tsv"), "rb").read()
    assert mash("dist", "-t", z, z).stdout == open(os.path.join(golden_dir, "zymo_dist_table.tsv"), "rb").read()
    db = orc.OracleDB.load_msh(z)
    for opts, kw in ((["-C"], dict(comments=True)), (["-d", "0.05"], dict(max_d=0.05)),
                     (["-v", "1e-10"], dict(max_p=1e-10)), (["-t", "-C", "-d", "0.3"], dict(table=True, comments=True, max_d=0.3)),
                     (["-p", "4", "-d", "0.2", "-v", "1e-40"], dict(max_d=0.2, max_p=1e-40))):
        assert mash("dist", *opts, z, z).stdout == dref.oracle_tsv(db, db, db.s, **kw), opts


# ---- synthetic clusters ---------------------------------------------------------------------------------------
def cluster_collection(rng, k, s, tmp_path):
    n_anc, rates = 3, (0.001, 0.01, 0.05, 0.1, 0.2)
    genomes = []
    for _ in range(n_anc):
        a = synth.random_genome(rng, 150_000)
        genomes.append(a)
        genomes += [synth.mutate(a, r, rng) for r in rates]
    genomes += [synth.random_genome(rng, 120_000) for _ in range(3)]        # decoys
    genomes += [synth.random_genome(rng, int(n)) for n in (600, 3_000, 8_000)]   # fewer k-mers than s
    genomes.append(genomes[0].copy())                                       # an exact duplicate
    sk = [hs.sketch_text(synth.to_fasta([g], "g"), k, s)[0] for g in genomes]
    return write_db(tmp_path / ("c%d_%d.msh" % (k, s)), k, s, sk, [len(g) for g in genomes])


@pytest.mark.parametrize("k", [12, 16, 21, 31])
@pytest.mark.parametrize("s", [1000, 10000])
def test_synthetic_clusters(k, s, tmp_path):
    rng = np.random.default_rng(100 + k + s)
    p = cluster_collection(rng, k, s, tmp_path)
    db = orc.OracleDB.load_msh(p)
    rows, st = gpu_rows(p, p)
    n_cand = assert_rows_match_oracle(rows, db, db, s)
    assert st["n_candidates"] == n_cand == len(rows.q)
    for opts, kw in (([], {}), (["-d", "0.1"], dict(max_d=0.1)), (["-t"], dict(table=True))):
        assert gpu_tsv(tmp_path, p, [p], *opts) == dref.oracle_tsv(db, db, s, **kw), (k, s, opts)


# ---- D1 boundaries --------------------------------------------------------------------------------------------
def test_boundaries(tmp_path):
    rng = np.random.default_rng(3)
    for i, (A, B, sp) in enumerate(dref.boundary_pairs(rng, 100)):
        rp = write_db(tmp_path / ("r%d.msh" % i), 21, sp, [A], [3_000_000])
        qp = write_db(tmp_path / ("q%d.msh" % i), 21, sp, [B], [4_000_000])
        rows, _ = gpu_rows(rp, qp)
        c, d = dref.closed_form(A, B, sp)
        if len(np.intersect1d(A, B)):
            assert (len(rows.q), int(rows.common[0]), int(rows.denom[0])) == (1, c, d), i
        else:
            assert len(rows.q) == 0
        rdb, qdb = orc.OracleDB.load_msh(rp), orc.OracleDB.load_msh(qp)
        for opts, kw in (([], {}), (["-v", "0.5"], dict(max_p=0.5)), (["-t"], dict(table=True)), (["-d", "0.5"], dict(max_d=0.5))):
            assert gpu_tsv(tmp_path, rp, [qp], *opts) == dref.oracle_tsv(rdb, qdb, sp, **kw), (i, opts)


# ---- blocks, a query that hits everything, a split on overflow ------------------------------------------------
def test_blocks_and_overflow_split(tmp_path):
    rng = np.random.default_rng(17)
    s = 10000
    ident = dref.distinct_hashes(rng, s)
    n_ident, n_other = 900, 1100
    pool = dref.distinct_hashes(rng, 4 * s)
    others = [np.sort(rng.choice(pool, size=s, replace=False)) for _ in range(n_other)]
    sk = [ident] * n_ident + others
    universal = np.unique(np.array([x[0] for x in sk], np.uint64))       # shares a hash with every sketch
    sk.append(universal)
    lens = [5_000_000] * len(sk)
    p = write_db(tmp_path / "blocks.msh", 21, s, sk, lens)
    rows, st = gpu_rows(p, p)
    assert st["n_blocks"] >= 3 and st["n_splits"] >= 1, st
    assert st["block_queries"] * 3 <= len(sk) and st["block_queries"] * n_ident > st["result_cap"], st
    key = rows.q.astype(np.uint64) << np.uint64(32) | rows.r.astype(np.uint64)
    assert np.all(np.diff(key.astype(np.int64)) > 0)                      # (q, r) order, nothing twice
    u = len(sk) - 1
    assert np.array_equal(np.sort(rows.r[rows.q == u]), np.arange(len(sk)))
    blk = (rows.q < n_ident) & (rows.r < n_ident)
    assert blk.sum() == n_ident * n_ident and np.all(rows.common[blk] == s) and np.all(rows.denom[blk] == s)
    db = orc.OracleDB.load_msh(p)
    sample = np.concatenate([[0, n_ident - 1, n_ident, u], rng.choice(len(sk), 40, replace=False)])
    assert_rows_match_oracle(rows, db, db, s, np.unique(sample))


# ---- sequence queries -----------------------------------------------------------------------------------------
def test_sequence_queries_and_lists(tmp_path):
    rng = np.random.default_rng(23)
    anc = synth.random_genome(rng, 200_000)
    gs = [anc] + [synth.mutate(anc, r, rng) for r in (0.002, 0.02, 0.08)] + [synth.random_genome(rng, 90_000)]
    paths = []
    for i, g in enumerate(gs):
        if i % 2:
            p = tmp_path / ("g%d.fq.gz" % i)
            seq = synth.ASCII[g].tobytes()
            with gzip.open(p, "wb") as fh:
                for j in range(0, len(seq), 5000):
                    fh.write(b"@r%d_%d\n%s\n+\n%s\n" % (i, j, seq[j:j + 5000], b"I" * len(seq[j:j + 5000])))
        else:
            p = tmp_path / ("g%d.fna" % i)
            p.write_bytes(synth.to_fasta([g[: len(g) // 2], g[len(g) // 2:]], "g%d" % i))
        paths.append(str(p))
    ref = str(tmp_path / "ref")
    assert mash("sketch", "-o", ref, *paths).returncode == 0
    qm = str(tmp_path / "q")
    assert mash("sketch", "-o", qm, *paths[::-1]).returncode == 0
    want = gpu_tsv(tmp_path, ref + ".msh", [qm + ".msh"])
    assert gpu_tsv(tmp_path, ref + ".msh", paths[::-1]) == want
    assert gpu_tsv(tmp_path, ref + ".msh", paths[::-1], "-p", "3") == want
    lst = tmp_path / "list.txt"
    lst.write_text("\n".join(paths[::-1]) + "\n\n")
    assert gpu_tsv(tmp_path, ref + ".msh", [str(lst)], "-l") == want
    assert len(want.splitlines()) == len(paths) ** 2
    # a query file with a smaller sketch size: s_p = the smaller one, and a WARNING
    small = str(tmp_path / "small")
    assert mash("sketch", "-s", "300", "-o", small, *paths).returncode == 0
    r = mash("dist", ref + ".msh", small + ".msh")
    assert r.returncode == 0 and b"WARNING" in r.stderr
    rdb, sdb = orc.OracleDB.load_msh(ref + ".msh"), orc.OracleDB.load_msh(small + ".msh")
    assert r.stdout == dref.oracle_tsv(rdb, sdb, 300)
    assert all(ln.split(b"\t")[4].endswith(b"/300") for ln in r.stdout.splitlines())


# ---- scale ----------------------------------------------------------------------------------------------------
def test_scale_20000_symmetric(tmp_path):
    rng = np.random.default_rng(29)
    s, n = 1000, 20000
    anc, G = synth.decoy_sketches(rng, 400, s)
    sk, lens = [], []
    for i in range(n):
        a = anc[i % 400]
        keep = rng.random(s) > rng.choice([0.0, 0.05, 0.2, 0.5, 1.0])
        fresh = dref.distinct_hashes(rng, s)[: s - int(keep.sum())] >> np.uint64(int(rng.integers(0, 4)))
        sk.append(np.unique(np.concatenate([a[keep], fresh]))[:s])
        lens.append(int(G[i % 400]))
    p = write_db(tmp_path / "scale.msh", 21, s, sk, lens)
    rows, st = gpu_rows(p, p, max_d=0.3)
    assert st["n_blocks"] >= 3
    db = orc.OracleDB.load_msh(p)
    assert_rows_match_oracle(rows, db, db, s, rng.choice(n, 200, replace=False), max_d=0.3)
    fwd = np.stack([rows.q, rows.r, rows.common, rows.denom]).T
    bwd = np.stack([rows.r, rows.q, rows.common, rows.denom]).T
    o1, o2 = np.lexsort(fwd.T[::-1]), np.lexsort(bwd.T[::-1])
    assert np.array_equal(fwd[o1], bwd[o2])
    p1, p2 = rows.pvalue[o1], rows.pvalue[o2]
    assert np.array_equal(p1 < 0, p2 < 0) and np.all(np.abs(p1 - p2) <= 1e-12 * np.abs(p1))


# ---- a real mash, when one is installed -----------------------------------------------------------------------
@pytest.mark.skipif(real_mash.find_mash() is None, reason="no real mash binary on this machine")
def test_real_mash_pins_goldens_and_cli(golden_dir):
    m = real_mash.find_mash()
    z = os.path.join(golden_dir, "zymo25.msh")
    for opts, golden in (([], "zymo_dist.tsv"), (["-t"], "zymo_dist_table.tsv")):
        out, _, _ = dref.real_mash_dist(m, z, [z], 4, tuple(opts))
        assert out == open(os.path.join(golden_dir, golden), "rb").read()
    for opts in ([], ["-C"], ["-d", "0.05"], ["-v", "1e-10"], ["-t"]):
        assert mash("dist", *opts, z, z).stdout == dref.real_mash_dist(m, z, [z], 4, tuple(opts))[0], opts

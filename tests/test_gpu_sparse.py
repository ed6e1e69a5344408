"""O(present hashes) reduction, reset and exchange vs their dense forms and vs the oracle
(needs a B200: `pytest -m gpu`).  Everything here is bit-exact integer work."""
import os
import subprocess
import sys

import numpy as np
import pytest

from hymet_b200 import screen as hs
from hymet_b200 import synth
from tests import _oracle as orc
from tests.test_gpu_parity import build_db, rel_close

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def cluster_case():
    """References with shared hashes (relatives 1-5 % apart, exact duplicates), so that the chains of
    the inverted index are longer than one and -w has ties to break."""
    rng = np.random.default_rng(11)
    genomes = []
    for c in range(10):
        anc = synth.random_genome(rng, 50_000)
        for m in range(5):
            g = synth.mutate(anc, float(rng.uniform(0.01, 0.05)), rng)
            genomes.append(g if m < 2 else g[:50_000 - int(rng.integers(1, 999))])
        genomes.append(genomes[-1].copy())
    genomes += [synth.random_genome(rng, 50_000) for _ in range(40)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[::6] + genomes[60:70], 900_000, 0.005, median=6000.0), "c")
    return offsets, hashes, lengths, fasta


def same(a, b):
    return (a.shared.tolist() == b.shared.tolist() and a.median.tolist() == b.median.tolist() and a.set_size == b.set_size
            and a.identity.tolist() == b.identity.tolist() and a.pvalue.tolist() == b.pvalue.tolist())


def check_oracle(res, want):
    assert res.shared.tolist() == want.shared.tolist()
    assert res.median.tolist() == want.median.tolist()
    assert res.set_size == want.set_size
    assert rel_close(res.identity, want.identity) and rel_close(res.pvalue, want.pvalue)


@pytest.mark.parametrize("wta", [False, True])
def test_sparse_reduction_equals_dense_and_oracle(cluster_case, wta):
    offsets, hashes, lengths, fasta = cluster_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    want = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths).screen_text(fasta, threads=2, wta=wta)
    scr = hs.Screen(db)
    scr.feed_text(fasta, 2)
    sp = scr.finish(wta)
    assert sp.stats["reduce_path"] == 0 and sp.stats["n_touched"] > 1000
    assert sp.stats["n_hit_refs"] == int((want.shared > 0).sum()) if not wta else sp.stats["n_hit_refs"] > 0
    assert sp.stats["n_pairs"] == int(want.shared.sum())
    check_oracle(sp, want)
    scr.set_option("sparse", 0)      # takes effect with the next reset
    scr.reset()
    scr.feed_text(fasta, 2)
    de = scr.finish(wta)
    assert de.stats["reduce_path"] == 1
    assert same(sp, de)
    # back to the sparse path on the same handle: the dense screen left no stale record behind
    scr.set_option("sparse", 1)
    scr.reset()
    scr.feed_text(fasta, 2)
    again = scr.finish(wta)
    assert again.stats["reduce_path"] == 0 and same(sp, again)
    scr.close()


@pytest.mark.parametrize("env", [{"HYMET_SCREEN_TOUCHED_CAP": "64"}, {"HYMET_SCREEN_PAIR_CAP": "100"}])
def test_sparse_buffers_too_small_fall_back_to_dense(cluster_case, env):
    """Run in a child process (the caps are read when a screen is created): the fallback gives the
    same numbers, says so in reduce_path, and the handle stays usable (the next reset clears every
    count when the touched list was incomplete)."""
    code = r'''
import sys
sys.path.insert(0, %r)
import numpy as np
from hymet_b200 import screen as hs, synth
from tests import _oracle as orc
from tests.test_gpu_parity import build_db
rng = np.random.default_rng(12)
genomes = [synth.random_genome(rng, 40_000) for _ in range(30)]
genomes += [synth.mutate(genomes[i], 0.02, rng) for i in range(6)]
offsets, hashes, lengths = build_db(genomes, 21, 1000)
f1 = synth.to_fasta(synth.cut_contigs(rng, genomes[:8] + genomes[30:33], 500_000, 0.01, median=5000.0), "a")
f2 = synth.to_fasta(synth.cut_contigs(rng, genomes[10:14], 200_000, 0.0, median=5000.0), "b")
db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
scr = hs.Screen(db)
for fasta, wta in ((f1, False), (f2, True), (f1, True), (f2, False)):
    scr.reset()
    scr.feed_text(fasta, 2)
    r = scr.finish(wta)
    w = odb.screen_text(fasta, threads=2, wta=wta)
    assert r.stats["reduce_path"] == 1, r.stats
    assert r.shared.tolist() == w.shared.tolist() and r.median.tolist() == w.median.tolist() and r.set_size == w.set_size
print("FALLBACK-OK")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, **env), timeout=600)
    assert r.returncode == 0 and "FALLBACK-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]


def test_one_handle_many_queries_reset_is_exact(cluster_case):
    """The sparse reset zeroes only the counts the previous query touched: three different queries
    on one handle must each equal a fresh oracle run."""
    offsets, hashes, lengths, fasta = cluster_case
    rng = np.random.default_rng(5)
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    odb = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    recs = fasta.split(b"\n>")
    parts = [b">" + b"\n>".join(recs[i::3]).lstrip(b">") + b"\n" for i in range(3)]
    scr = hs.Screen(db)
    for i, (q, wta) in enumerate(zip(parts + [fasta], (False, True, False, True))):
        if i:
            scr.reset()
        scr.feed_text(q, 2)
        r = scr.finish(wta)
        assert r.stats["reduce_path"] == 0
        check_oracle(r, odb.screen_text(q, threads=2, wta=wta))
    scr.close()


def test_two_tier_filter_equals_unfiltered_and_oracle():
    """Tiny genomes put keys all over the hash range: the build picks a dense range + a Bloom tier above
    it.  The tier, whose reads are issued a group of k-mers at a time, may not change a result."""
    rng = np.random.default_rng(78)
    genomes = [synth.random_genome(rng, 40_000) for _ in range(24)]
    genomes += [synth.random_genome(rng, int(n)) for n in rng.integers(300, 3000, size=60)]   # < s k-mers each
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[:6] + genomes[24:40], 600_000, 0.01, median=2500.0, lo=300), "c")
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    info = db.info
    assert info.bloom_bytes > 0 and info.dense_max < info.max_key and info.max_key > 2 ** 63
    assert info.dense_max < 2 ** 64 * 0.2          # the dense range is a sliver: 40 kb genomes keep hashes below 2^64 * 1000/40000
    want = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths).screen_text(fasta, threads=2)
    out = {}
    for name, opts in (("batched", {}), ("no_filter", {"filter": 0})):
        scr = hs.Screen(db)
        for k_, v in opts.items():
            scr.set_option(k_, v)
        scr.feed_text(fasta, 2)
        out[name] = scr.finish(False)
        check_oracle(out[name], want)
        scr.close()
    assert out["batched"].stats["n_hits"] == out["no_filter"].stats["n_hits"]
    assert out["batched"].stats["n_probes"] < 0.5 * out["no_filter"].stats["n_probes"]
    assert int(out["batched"].shared[24:40].min()) > 100     # the tiny genomes in the query are found


def test_32bit_hashes_need_one_mixture_pass():
    """k = 16: hashes live in [0, 2^32).  The per-launch mixture cap must be scaled to that space, or the
    first big launch floods the set and the finaliser needs extra passes over the query (ADVICE r1)."""
    rng = np.random.default_rng(16)
    genomes = [synth.random_genome(rng, 400_000) for _ in range(12)]
    offsets, hashes, lengths = build_db(genomes, 16, 1000)
    fasta = synth.to_fasta(genomes, "g", width=0)          # 4.8 M distinct-ish 16-mers in one feed
    db = hs.Database.from_arrays(16, 1000, 42, offsets, hashes, lengths)
    want = orc.OracleDB.from_arrays(16, 1000, 42, offsets, hashes, lengths).screen_text(fasta, threads=2)
    scr = hs.Screen(db)
    scr.feed_text(fasta, 2)
    r = scr.finish(False)
    check_oracle(r, want)
    assert r.stats["n_mix_passes"] == 1
    scr.close()


def test_exchange_absorb_and_device_mixture_merge_on_one_gpu(cluster_case):
    """The multi-GPU exchange, rehearsed on one GPU: two screens each stream half of the contigs, their
    pair records and mixture records are laid out as an all-gather would leave them, and screen 0
    absorbs them in one launch + merges the mixtures on the device.  Result == one screen over all."""
    import torch
    offsets, hashes, lengths, fasta = cluster_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    half = fasta.rfind(b"\n>", 0, len(fasta) // 2) + 1
    shards = [fasta[:half], fasta[half:]]
    want = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    for wta in (False, True):
        scrs = [hs.Screen(db) for _ in shards]
        cap, s = 1 << 16, db.s
        rows = torch.zeros((2, 1 + cap), dtype=torch.int64, device="cuda")
        mix = torch.zeros((2, 1 + s), dtype=torch.int64, device="cuda")
        for r, (scr, text) in enumerate(zip(scrs, shards)):
            scr.feed_text(text, 2)
            scr.counts_compact_async(rows[r, 1:].data_ptr(), cap, rows[r].data_ptr())
            scr.flush()
            scr.mixture_record(mix[r].data_ptr())
        torch.cuda.synchronize()
        assert 0 < int(rows[0, 0]) <= cap and 0 < int(rows[1, 0]) <= cap
        scrs[0].counts_absorb(rows.data_ptr(), 2, cap, 0)
        scrs[0].mixture_merge_device(mix.data_ptr(), 2)
        res = scrs[0].finish(wta)
        w = want.screen_text(fasta, threads=2, wta=wta)
        assert res.stats["exchange_overflow"] == 0 and res.stats["reduce_path"] == 0
        check_oracle(res, w)
        assert scrs[0].mixture().tolist() == w.mixture.tolist()
        # a record that is too small: nothing is added, the flag comes back
        scrs[1].counts_absorb(rows.data_ptr(), 2, 8, 1)
        res1 = scrs[1].finish(wta)
        assert res1.stats["exchange_overflow"] == 1
        for scr in scrs:
            scr.close()


@pytest.mark.parametrize("wta", [False, True])
def test_finish_hits_equals_dense_columns(cluster_case, wta):
    """hs_screen_finish_hits brings back only the references with shared > 0 (rows written by the GPU
    into host-mapped memory): expanded to columns they equal hs_screen_finish bit for bit, both on the
    sparse reduction path and on the dense one."""
    offsets, hashes, lengths, fasta = cluster_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    for sparse in (1, 0):
        scr = hs.Screen(db)
        scr.set_option("sparse", sparse)
        scr.reset()
        scr.feed_text(fasta, 2)
        hits = scr.finish_hits(wta)
        dense = scr.finish(wta)
        assert hits.stats["reduce_path"] == (0 if sparse else 1)
        assert np.all(np.diff(hits.ref.astype(np.int64)) > 0) and np.all(hits.shared > 0)
        assert len(hits.ref) == int((dense.shared > 0).sum())
        assert same(hits.to_dense(db.n_refs), dense)
        scr.close()


def test_cooperative_probe_all_equals_filtered(cluster_case):
    """filter = 0 probes the table for every k-mer.  The warp-cooperative kernel (coop_probe, MODE 3) gives
    the same counts as the filtered screen and the oracle."""
    offsets, hashes, lengths, fasta = cluster_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    want = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths).screen_text(fasta, threads=2)
    out = []
    for opts in ({"filter": 0}, {}):
        scr = hs.Screen(db)
        for k_, v in opts.items():
            scr.set_option(k_, v)
        scr.feed_text(fasta, 2)
        r = scr.finish(False)
        check_oracle(r, want)
        out.append(r.stats)
        scr.close()
    assert out[0]["n_probes"] == out[0]["n_valid_kmers"]
    assert out[0]["n_hits"] == out[1]["n_hits"]


def test_retired_options_are_unknown(cluster_case):
    """Options that used to pick a code path by hand are gone: setting one is an unknown option
    (HS_EINVAL) and leaves the handle usable."""
    offsets, hashes, lengths, _ = cluster_case
    db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
    scr = hs.Screen(db)
    for key in ("batch_bloom", "coop_probe", "piece_bases", "ingest_slots", "ingest_batch", "keep_query"):
        with pytest.raises(hs.HsError, match="unknown option") as e:
            scr.set_option(key, 1)
        assert e.value.code == -1, key        # HS_EINVAL
    scr.set_option("filter", 1)
    scr.close()


def test_iterative_mixture_finaliser_still_exact():
    """HYMET_SCREEN_FAST_SELECT=0 disables the one-synchronisation selection: the iterative finaliser
    (the fallback for overflow / repetitive input) must give the same mixture."""
    code = r'''
import sys
sys.path.insert(0, %r)
import numpy as np
from hymet_b200 import screen as hs, synth
from tests import _oracle as orc
from tests.test_gpu_parity import build_db
rng = np.random.default_rng(3)
genomes = [synth.random_genome(rng, 60_000) for _ in range(10)]
offsets, hashes, lengths = build_db(genomes, 21, 1000)
fasta = synth.to_fasta(synth.cut_contigs(rng, genomes, 900_000, 0.02, median=7000.0), "c")
db = hs.Database.from_arrays(21, 1000, 42, offsets, hashes, lengths)
w = orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths).screen_text(fasta, threads=2)
scr = hs.Screen(db)
scr.feed_text(fasta, 2)
r = scr.finish(False)
assert scr.mixture().tolist() == w.mixture.tolist() and r.set_size == w.set_size and r.shared.tolist() == w.shared.tolist()
print("ITERATIVE-OK")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       env=dict(os.environ, HYMET_SCREEN_FAST_SELECT="0"), timeout=600)
    assert r.returncode == 0 and "ITERATIVE-OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]

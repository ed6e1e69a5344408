"""N>1 on real GPUs (needs >= 2 B200 on the box; skipped otherwise): the NCCL all-reduce of
counts + all-gather of mixtures reproduce the single-process oracle bit for bit."""
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_rank_screen_matches_oracle():
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    world = 2 if n < 4 else 4
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tools", "dist_parity.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "parity=True" in r.stdout and "parity=False" not in r.stdout


def _case(tmp_path):
    """A 35-reference table (.msh) and a plain FASTA query of contigs from 12 of them."""
    import numpy as np

    from hymet_b200 import msh as mshfmt, synth
    from tests import _oracle as orc
    from tests.test_gpu_parity import build_db
    rng = np.random.default_rng(51)
    genomes = [synth.random_genome(rng, 40_000) for _ in range(30)]
    genomes += [synth.mutate(genomes[i], 0.02, rng) for i in range(5)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    dbp = str(tmp_path / "db.msh")
    mshfmt.write_msh(dbp, mshfmt.SketchDB(k=21, s=1000, names=[synth.gcf_name(i) for i in range(len(genomes))],
                                          comments=[""] * len(genomes), lengths=lengths, offsets=offsets, hashes=hashes))
    fasta = synth.to_fasta(synth.cut_contigs(rng, genomes[:9] + genomes[30:33], 900_000, 0.01, median=7000.0), "c")
    fap = str(tmp_path / "q.fna")
    open(fap, "wb").write(fasta)
    return dbp, fap, fasta, orc.OracleDB.from_arrays(21, 1000, 42, offsets, hashes, lengths)


def _range_screens(db, fap, n):
    """n screens over one table, screen i fed the records that start in the i-th n-th of the file's bytes."""
    from hymet_b200 import _lite
    size = os.path.getsize(fap)
    scrs = [_lite.LiteScreen(db) for _ in range(n)]
    for i, scr in enumerate(scrs):
        scr.set_option("file_block_bytes", 65536)          # several blocks per range
        scr.feed_fasta_range(fap, size * i // n, size * (i + 1) // n, 2)
    return scrs


def _whole(db, fap, wta):
    """TSV lines and stats of one screen of the whole file."""
    from hymet_b200 import _lite
    scr = _lite.LiteScreen(db)
    scr.feed_fasta(fap, 2)
    scr.flush()
    lines = "".join(scr.finish_lines(wta, 0.0, 1.0))
    st = scr.stats()
    scr.close()
    return lines, st


def test_byte_ranges_and_absorb_screens_rehearsed_on_one_gpu(tmp_path):
    """HYMET_SCREEN_GPUS's building blocks on ONE GPU: three screens over the same table each stream
    the records that start in a third of the file's bytes (hs_screen_feed_fasta_range), screen 0
    absorbs the other two in one call (hs_screen_absorb_screens): the result equals one screen of the
    whole file and the oracle, for -w too."""
    from hymet_b200 import _lite
    dbp, fap, fasta, odb = _case(tmp_path)
    db = _lite.LiteDb(dbp, 0)
    for wta in (False, True):
        scrs = _range_screens(db, fap, 3)
        for scr in scrs:
            scr.flush()
        parts = [scr.stats()["n_records"] for scr in scrs]
        assert sum(parts) == fasta.count(b">") and all(p > 0 for p in parts)
        scrs[0].absorb([scrs[1], scrs[2]])
        got = "".join(scrs[0].finish_lines(wta, 0.0, 1.0))
        want = odb.screen_text(fasta, threads=2, wta=wta)
        assert got == _whole(db, fap, wta)[0] and got.count("\n") == int((want.shared > 0).sum())
        assert scrs[0].stats()["set_size"] == want.set_size and scrs[0].stats()["n_bases"] == want.n_bases
        for scr in scrs:
            scr.close()
    # ranges need a plain FASTA file
    import gzip
    gz = str(tmp_path / "q.fna.gz")
    gzip.open(gz, "wb").write(fasta)
    scr = _lite.LiteScreen(db)
    with pytest.raises(_lite.HsError, match="plain FASTA"):
        scr.feed_fasta_range(gz, 0, 100, 1)
    scr.close()


def test_absorb_over_two_sketch_files_with_different_s(tmp_path):
    """One table over two .msh files of different sketch sizes (what hymet-mash-stage builds): each file's
    p-values use the set size of its own s, which the fold takes from the device merge of the mixtures."""
    import numpy as np

    from hymet_b200 import _lite, msh as mshfmt, synth
    from tests.test_gpu_parity import build_db
    rng = np.random.default_rng(53)
    genomes = [synth.random_genome(rng, 40_000) for _ in range(24)]
    paths = []
    for j, s in enumerate((1000, 300)):
        part = genomes[12 * j:12 * (j + 1)]
        offsets, hashes, lengths = build_db(part, 21, s)
        paths.append(str(tmp_path / ("f%d.msh" % j)))
        mshfmt.write_msh(paths[-1], mshfmt.SketchDB(k=21, s=s, names=[synth.gcf_name(12 * j + i) for i in range(12)],
                                                    comments=[""] * 12, lengths=lengths, offsets=offsets, hashes=hashes))
    fap = str(tmp_path / "q.fna")
    open(fap, "wb").write(synth.to_fasta(synth.cut_contigs(rng, genomes[:5] + genomes[12:17], 700_000, 0.01, median=7000.0), "c"))
    db = _lite.LiteDb(paths, 0)
    assert [e - b for b, e in db.segments] == [12, 12]
    for wta in (False, True):
        scrs = _range_screens(db, fap, 3)
        for scr in scrs:
            scr.flush()
        scrs[0].absorb(scrs[1:])
        before = scrs[0].stats()["set_size"]          # what `mash screen` reports before the reduction
        got = "".join(scrs[0].finish_lines(wta, 0.0, 1.0))
        want, st = _whole(db, fap, wta)
        hit = {ln.split("\t")[4] for ln in got.splitlines()}
        assert got == want and all(hit & {synth.gcf_name(12 * j + i) for i in range(12)} for j in (0, 1))
        assert before == scrs[0].stats()["set_size"] == st["set_size"]
        for scr in scrs:
            scr.close()


def test_absorb_when_the_touched_lists_overflow(tmp_path, monkeypatch):
    """Every screen's record of touched counts overflows (HYMET_SCREEN_TOUCHED_CAP, read when a screen is
    created): each source's pairs come from a scan of all its counts, and the fold still equals one screen."""
    from hymet_b200 import _lite
    monkeypatch.setenv("HYMET_SCREEN_TOUCHED_CAP", "64")
    dbp, fap, _, _ = _case(tmp_path)
    db = _lite.LiteDb(dbp, 0)
    for wta in (False, True):
        scrs = _range_screens(db, fap, 3)
        for scr in scrs:
            scr.flush()
        scrs[0].absorb(scrs[1:])
        got = "".join(scrs[0].finish_lines(wta, 0.0, 1.0))
        st = scrs[0].stats()
        assert st["n_touched"] > 64 and st["reduce_path"] == 1
        assert got == _whole(db, fap, wta)[0] and got.count("\n") >= 10
        for scr in scrs:
            scr.close()


def test_absorb_refusals_leave_the_screens_usable(tmp_path):
    """dst among its sources, a source listed twice, no source, an unflushed source and a second absorb
    before reset are refused without touching any handle: a valid absorb afterwards is still exact."""
    from hymet_b200 import _lite
    HS_EINVAL, HS_ESTATE = -1, -9
    dbp, fap, _, _ = _case(tmp_path)
    db = _lite.LiteDb(dbp, 0)
    scrs = _range_screens(db, fap, 3)
    scrs[0].flush(); scrs[1].flush()

    def refused(code, others):
        with pytest.raises(_lite.HsError) as e:
            scrs[0].absorb(others)
        assert e.value.code == code, e.value

    refused(HS_ESTATE, [scrs[1], scrs[2]])
    scrs[2].flush()
    refused(HS_EINVAL, [scrs[1], scrs[0]])
    refused(HS_EINVAL, [scrs[1], scrs[2], scrs[1]])
    refused(HS_EINVAL, [])
    scrs[0].absorb([scrs[1], scrs[2]])
    refused(HS_ESTATE, [scrs[1], scrs[2]])
    got = "".join(scrs[0].finish_lines(False, 0.0, 1.0))
    assert got == _whole(db, fap, False)[0] and got.count("\n") >= 10
    for scr in scrs:
        scr.close()


def test_drop_in_with_two_gpus_in_one_process(tmp_path):
    """HYMET_SCREEN_GPUS=2 bin/mash screen ... prints the same bytes as one GPU (needs >= 2 GPUs)."""
    import numpy as np
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    from hymet_b200 import msh as mshfmt, synth
    from tests.test_gpu_parity import build_db
    rng = np.random.default_rng(52)
    genomes = [synth.random_genome(rng, 40_000) for _ in range(24)]
    offsets, hashes, lengths = build_db(genomes, 21, 1000)
    dbp = str(tmp_path / "db.msh")
    mshfmt.write_msh(dbp, mshfmt.SketchDB(k=21, s=1000, names=[synth.gcf_name(i) for i in range(24)], comments=["c"] * 24,
                                          lengths=lengths, offsets=offsets, hashes=hashes))
    a, b = str(tmp_path / "a.fna"), str(tmp_path / "b.fna.gz")
    open(a, "wb").write(synth.to_fasta(synth.cut_contigs(rng, genomes[:8], 700_000, 0.01, median=6000.0), "a"))
    import gzip
    gzip.open(b, "wb").write(synth.to_fasta(synth.cut_contigs(rng, genomes[10:14], 200_000, 0.02, median=6000.0), "b"))
    exe = [sys.executable, os.path.join(ROOT, "bin", "mash"), "screen", "-p", "8", "-v", "0.9"]
    for extra in ([], ["-w"]):
        one = subprocess.run(exe + extra + [dbp, a, b], capture_output=True, env=dict(os.environ, HYMET_SCREEN_GPUS="1"))
        two = subprocess.run(exe + extra + [dbp, a, b], capture_output=True, env=dict(os.environ, HYMET_SCREEN_GPUS="2"))
        assert one.returncode == 0 and two.returncode == 0, two.stderr.decode()[-2000:]
        assert one.stdout == two.stdout and one.stdout.count(b"\n") >= 5

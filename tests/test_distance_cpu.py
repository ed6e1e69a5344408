"""`mash dist` without a GPU (DESIGN.md §5 "mash dist"): the C oracle's merge loop against the closed form of D1-D3
(NumPy + scipy), its p-values against mpmath, and the CLI's option handling and error exits."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from hymet_b200 import msh as mshfmt
from tests import _distance_ref as dref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASH = os.path.join(ROOT, "bin", "mash")


def run(*args, env=None):
    return subprocess.run([sys.executable, MASH] + list(args), capture_output=True, text=True, env=env)


def check_pairs(k, refs, qrys, s_p, lr, lq):
    ref = dref.db_of(k, s_p, refs, lr)
    qry = dref.db_of(k, s_p, qrys, lq)
    common, denom, pv = dref.oracle_pairs(ref, qry, s_p)
    for qi, B in enumerate(qrys):
        for ri, A in enumerate(refs):
            c, d = dref.closed_form(A, B, s_p)
            assert (int(common[qi, ri]), int(denom[qi, ri])) == (c, d), (qi, ri)
            want = dref.closed_pvalue(c, d, lr[ri], lq[qi], k)
            got = float(pv[qi, ri])
            assert abs(got - want) <= 1e-9 * abs(want) + 1e-300, (qi, ri, got, want)
    return common, denom


def test_oracle_random_pairs_match_closed_form():
    rng = np.random.default_rng(5)
    s = 200
    pool = dref.distinct_hashes(rng, 3 * s)
    sk = []
    for i in range(12):
        n = int(rng.integers(s // 2, s + 1)) if i % 4 else s
        sk.append(np.sort(rng.choice(pool, size=n, replace=False)))
    lens = [int(x) for x in rng.integers(200_000, 6_000_000, size=len(sk))]
    for k in (12, 21):
        common, denom = check_pairs(k, sk, sk, s, lens, lens)
        assert np.array_equal(common, common.T) and np.array_equal(denom, denom.T)
        assert (common > 0).mean() > 0.9


def test_oracle_boundaries_match_closed_form():
    rng = np.random.default_rng(11)
    for A, B, sp in dref.boundary_pairs(rng, 100):
        check_pairs(21, [A], [B], sp, [3_000_000], [4_000_000])


def test_boundary_at_rank_s():
    # A = {1..10}, B = {11..19, h}: h shared at union rank r counts iff r <= s
    A = np.arange(1, 11, dtype=np.uint64)
    for h, s, want in ((5, 10, 1), (10, 10, 1), (10, 9, 0), (10, 5, 0), (3, 3, 1), (3, 2, 0)):
        B = np.sort(np.concatenate([np.arange(100, 109, dtype=np.uint64), [h]])).astype(np.uint64)
        c, d = dref.closed_form(A, B, s)
        assert c == want and d == min(s, 19), (h, s)
        common, denom = check_pairs(21, [A], [B], s, [1_000_000], [1_000_000])
        assert (int(common[0, 0]), int(denom[0, 0])) == (want, min(s, 19))


def test_distance_rules():
    assert dref.distance(0, 0, 21) == 0.0 and dref.distance(5, 5, 21) == 0.0
    assert dref.distance(0, 1000, 21) == 1.0
    assert dref.distance(1, 1000, 2) == 1.0                      # small k: capped at 1
    L = dref.lib()
    for c, d, k in ((1, 1000, 2), (1, 1000, 21), (500, 1000, 21), (999, 1000, 31), (0, 7, 9), (3, 3, 9), (0, 0, 9)):
        assert L.orc_dist_distance(c, d, k) == dref.distance(c, d, k)


def test_oracle_pvalue_kats(golden_dir):
    kats = json.load(open(os.path.join(golden_dir, "distance_pvalue_kat.json")))
    L = dref.lib()
    for e in kats:
        assert float.fromhex(e["r"]) == dref.r_of(e["len_ref"], e["len_qry"], e["k"])
        got = L.orc_dist_pvalue(e["common"], e["len_ref"], e["len_qry"], e["k"], e["denom"])
        want = float(e["pvalue"])
        assert abs(got - want) <= 1e-13 * abs(want), (e, got)
    assert L.orc_dist_pvalue(0, 1000, 1000, 21, 1000) == 1.0


def test_zymo_goldens_are_the_oracle(golden_dir):
    from tests import _oracle as orc
    db = orc.OracleDB.load_msh(os.path.join(golden_dir, "zymo25.msh"))
    for name, table in (("zymo_dist.tsv", False), ("zymo_dist_table.tsv", True)):
        assert dref.oracle_tsv(db, db, db.s, table=table) == open(os.path.join(golden_dir, name), "rb").read()


def _msh(path, k=21, s=10, seed=42, hashes=(1, 2, 3)):
    db = mshfmt.SketchDB(k=k, s=s, seed=seed, names=["a"], comments=["c"], lengths=np.array([5000], np.uint64),
                         offsets=np.array([0, len(hashes)], np.uint64), hashes=np.array(hashes, np.uint64))
    mshfmt.write_msh(str(path), db)
    return str(path)


def test_usage():
    for args in (["dist", "-h"], ["dist", "-h", "x.msh"]):
        r = run(*args)
        assert r.returncode == 0 and "mash dist [options] <reference>.msh <query>" in r.stdout, args
        assert "-d <num>" in r.stdout and "-t " in r.stdout and "-C " in r.stdout
    r = run("-h")
    assert r.returncode == 0 and "`dist`" in r.stdout


def test_non_sketch_reference_keeps_the_old_route(tmp_path):
    env = dict(os.environ, PATH=str(tmp_path))           # no mash further down PATH
    for args in (["dist", "a", "b"], ["dist", "-p", "2", "ref.fna", "q.msh"]):
        r = run(*args, env=env)
        assert r.returncode == 2 and "not provided by this drop-in" in r.stderr, args


def test_option_errors(tmp_path):
    ref = _msh(tmp_path / "ref.msh")
    q = _msh(tmp_path / "q.msh")
    for args, msg in [(["-v", "x"], "malformed numeric option value"), (["-d", "1e"], "malformed numeric option value"),
                      (["-v", "1.5"], "option value out of range"), (["-v", "-0.1"], "option value out of range"),
                      (["-d", "2"], "option value out of range"), (["-d", "-1"], "option value out of range"),
                      (["-p", "0"], "option value out of range"), (["-q"], "Unrecognized option: -q"),
                      (["-k", "21"], "Sketching option -k cannot be used"), (["-s", "500"], "Sketching option -s cannot be used")]:
        r = run("dist", *args, ref, q)
        assert r.returncode == 1 and ("ERROR: " + msg) in r.stderr and r.stdout == "", (args, r.stderr)
    r = run("dist", ref, q, "-d")
    assert r.returncode == 1 and "ERROR: -d requires an argument" in r.stderr


def test_missing_query_and_mismatched_sketches(tmp_path):
    ref = _msh(tmp_path / "ref.msh")
    missing = str(tmp_path / "nope.fna")
    r = run("dist", ref, missing)
    assert r.returncode == 1 and ("ERROR: could not open %s for reading." % missing) in r.stderr and r.stdout == ""
    lst = tmp_path / "list.txt"
    lst.write_text("%s\n" % missing)
    r = run("dist", "-l", ref, str(lst))
    assert r.returncode == 1 and ("ERROR: could not open %s for reading." % missing) in r.stderr
    for kw, what in (({"k": 15}, "k-mer size 15 differs"), ({"seed": 7}, "hash seed 7 differs")):
        q = _msh(tmp_path / ("q_%s.msh" % what.split()[0]), **kw)
        r = run("dist", ref, q)
        assert r.returncode == 1 and "ERROR: " in r.stderr and what in r.stderr and r.stdout == "", r.stderr


def test_without_a_usable_gpu_fails_loudly(tmp_path):
    ref = _msh(tmp_path / "ref.msh")
    q = _msh(tmp_path / "q.msh", hashes=(2, 3, 4))
    env = dict(os.environ, HYMET_SCREEN_DEVICE="99")   # no such device, here or on any single-node box
    r = run("dist", ref, q, env=env)
    assert r.returncode == 1 and "ERROR: " in r.stderr and r.stdout == "" and "Traceback" not in r.stderr

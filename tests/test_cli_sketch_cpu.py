"""`mash sketch` option handling that needs no GPU: usage, option errors, `-l` list files, and that a
sketch that cannot run on a GPU fails with ERROR: and leaves no .msh behind."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MASH = os.path.join(ROOT, "bin", "mash")


def run(*args, env=None):
    return subprocess.run([sys.executable, MASH, "sketch"] + list(args), capture_output=True, text=True, env=env)


def test_usage():
    for r in (run(), run("-h")):
        assert r.returncode == 0 and "mash sketch [options] <input>" in r.stdout
        assert "-l " in r.stdout and "-p <int>" in r.stdout and "-i " not in r.stdout


def test_option_errors(tmp_path):
    fa = tmp_path / "a.fna"
    fa.write_bytes(b">a\nACGTACGTACGTACGTACGTACGTACGT\n")
    for args, msg in [(["-k", "0"], "k-mer size must be 1-32"), (["-k", "33"], "k-mer size must be 1-32"),
                      (["-s", "0"], "k-mer size must be 1-32 and sketch size positive"), (["-p", "0"], "option value out of range"),
                      (["-p", "two"], "malformed numeric option value"), (["-x"], "Unrecognized option: -x"),
                      (["-q", "3"], "Unrecognized option: -q")]:
        r = run(*args, str(fa))
        assert r.returncode == 1 and ("ERROR: " + msg) in r.stderr and r.stdout == "", (args, r.stderr)
    r = run(str(fa), "-o")
    assert r.returncode == 1 and "ERROR: -o requires an argument" in r.stderr
    assert not os.path.exists(str(fa) + ".msh")


def test_list_files_are_read_before_any_sketching(tmp_path):
    fa = tmp_path / "a.fna"
    fa.write_bytes(b">a\nACGTACGTACGTACGTACGTACGTACGT\n")
    missing = str(tmp_path / "missing.fna")
    lst = tmp_path / "list.txt"
    lst.write_text("\n%s\n\n%s\n" % (fa, missing))
    r = run("-l", "-o", str(tmp_path / "out"), str(lst))
    assert r.returncode == 1 and ("ERROR: could not open %s for reading." % missing) in r.stderr
    assert not os.path.exists(str(tmp_path / "out.msh"))
    r = run("-l", "-o", str(tmp_path / "out"), str(tmp_path / "no_list.txt"))
    assert r.returncode == 1 and "ERROR: could not open %s for reading." % (tmp_path / "no_list.txt") in r.stderr
    empty = tmp_path / "empty.txt"
    empty.write_text("\n\n")
    r = run("-l", "-o", str(tmp_path / "out"), str(empty))
    assert r.returncode == 1 and "ERROR: no input files listed" in r.stderr
    assert not os.path.exists(str(tmp_path / "out.msh"))


def test_without_a_usable_gpu_fails_and_writes_nothing(tmp_path):
    fa = tmp_path / "a.fna"
    fa.write_bytes(b">a\nACGTACGTACGTACGTACGTACGTACGT\n")
    env = dict(os.environ, HYMET_SCREEN_DEVICE="99")   # no such device, here or on any single-node box
    r = run("-o", str(tmp_path / "out"), str(fa), env=env)
    assert r.returncode == 1 and "ERROR: " in r.stderr and "Traceback" not in r.stderr
    assert not os.path.exists(str(tmp_path / "out.msh"))

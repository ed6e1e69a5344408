"""`mash`-compatible command line: the process-level drop-in (SURVEY.md 8b #1).

HYMET only ever runs ``mash screen -p 8 -v 0.9 DB.msh dir/*.fna``
(/root/reference/scripts/mash.sh:14; presence check run_hymet_cami.sh:72).  Put
bin/mash first on PATH and the unmodified scripts keep working: same options
(-p -v -i -w -h), same stdout TSV, same exit codes, progress on stderr (S20/S21).
"""
from __future__ import annotations

import os
import sys
from typing import List, Optional

USAGE = """
Version: hymet-screen-b200 (mash screen drop-in, B200)

Usage:

  mash screen [options] <queries>.msh <mixture> [<mixture>] ...

Description:

  Determine how well query sequences are contained within a mixture of
  sequences. The queries must be formatted as a single Mash sketch file (.msh).
  The mixture files can be contigs or reads, in fasta or fastq, gzipped or not,
  and "-" can be given for <mixture> to read from standard input. The output
  fields are [identity, shared-hashes, median-multiplicity, p-value, query-ID,
  query-comment], where median-multiplicity is computed for shared hashes.

Options:

  -h          Help
  -p <int>    Host packer threads [1]
  -w          Winner-takes-all strategy for identity estimates.
  -i <num>    Minimum identity to report. Inclusive unless set to zero. -1 to
              include all. [0]
  -v <num>    Maximum p-value to report. (0-1) [1.0]
"""


def _err(msg: str, stderr=None) -> None:
    (stderr or sys.stderr).write("ERROR: %s\n" % msg)


def screen_main(args: List[str], stdout=None, stderr=None, cwd: Optional[str] = None, server=None) -> int:
    """`mash screen`.  In-process by default; `server` is the resident table server when this runs inside
    it (hymet_b200/server.py): tables and screens then outlive the call, relative paths are the
    client's (`cwd`), and stdout/stderr are the client's too."""
    stdout = stdout or sys.stdout
    stderr = stderr or sys.stderr
    _e = lambda msg: _err(msg, stderr)
    threads, wta, imin, pmax = 1, False, 0.0, 1.0
    pos: List[str] = []
    i = 0
    try:
        while i < len(args):
            a = args[i]
            if a == "-h":
                stdout.write(USAGE)
                return 0
            if a == "-w":
                wta = True
            elif a in ("-p", "-i", "-v"):
                if i + 1 >= len(args):
                    _e("-%s requires an argument" % a[1])
                    return 1
                v = args[i + 1]
                i += 1
                if a == "-p":
                    threads = int(v)
                elif a == "-i":
                    imin = float(v)
                else:
                    pmax = float(v)
            elif a.startswith("-") and a != "-":
                _e("Unrecognized option: %s" % a)
                return 1
            else:
                pos.append(a)
            i += 1
    except ValueError:
        _e("malformed numeric option value")
        return 1
    if len(pos) < 2:
        stdout.write(USAGE)
        return 0
    db_path, inputs = pos[0], pos[1:]
    if cwd:
        rel = lambda p: p if (p == "-" or os.path.isabs(p)) else os.path.join(cwd, p)
        shown_db, db_path, inputs = db_path, rel(db_path), [rel(p) for p in inputs]
    else:
        shown_db = db_path
    if not db_path.endswith(".msh"):
        _e("%s does not look like a sketch (.msh)" % shown_db)
        return 1
    if threads < 1 or not (0.0 <= pmax <= 1.0) or imin > 1.0:
        _e("option value out of range")
        return 1

    import time
    t0 = time.perf_counter()
    marks = []
    mark = lambda what: marks.append((what, time.perf_counter()))
    from . import _lite as hs    # ctypes only: neither torch nor numpy on the one-shot CLI path
    mark("imports")

    device = int(os.environ.get("HYMET_SCREEN_DEVICE", "0"))
    try:
        stderr.write("Loading %s...\n" % shown_db)
        if server is not None:
            if "-" in inputs:
                _e("the screen server cannot read the client's standard input")
                return 1
            ent = server.table([db_path])                # resident: built on first use only
            db, scr = ent["db"], server.screen_for(ent)
            multi = None
        else:
            # HYMET_SCREEN_GPUS=N (SURVEY.md 8b): N GPUs of this box, one table copy each, the inputs cut by bytes
            n_gpus = max(1, int(os.environ.get("HYMET_SCREEN_GPUS", "1") or "1"))
            multi = hs.MultiGpu(db_path, range(device, device + n_gpus)) if n_gpus > 1 else None
            if multi is not None:
                db = multi.db
            else:
                db = hs.LiteDb(db_path, device)          # CUDA context creation overlaps the .msh parse
                scr = hs.LiteScreen(db, probe_filter=os.environ.get("HYMET_SCREEN_FILTER", "1") != "0")
        mark("cuda_init + load_db(parse %.3f build %.3f)" % (db.info.t_parse_s, db.info.t_build_s))
        stderr.write("   %d distinct hashes.\n" % db.n_distinct)
        stderr.write("Streaming from %s...\n" % (inputs[0] if len(inputs) == 1 else "%d inputs" % len(inputs)))
        for p in inputs:
            if p != "-" and not os.path.exists(p):
                _e("could not open %s for reading." % p)
                return 1
        if multi is not None:
            scr = multi.screen(inputs, threads, probe_filter=os.environ.get("HYMET_SCREEN_FILTER", "1") != "0")
        else:
            for p in inputs:
                scr.feed_fasta(p, threads)
        mark("feed")
        scr.flush()
        mark("flush")
        st = scr.stats()
        if st["n_records"] == 0:
            _e("Did not find sequence records in inputs.")
            return 1
        stderr.write("   Estimated distinct k-mers in mixture: %d\n" % st["set_size"])
        if st["set_size"] == 0:
            stderr.write("WARNING: no valid k-mers in input.\n")
        stderr.write("Summing shared...\n")
        if wta:
            stderr.write("Reallocating to winners...\n")
        stderr.write("Computing coverage medians...\n")
        lines = scr.finish_lines(wta, imin, pmax)
        first = next(lines, None)                 # the reduction runs on the first pull
        mark("finish")
        stderr.write("Writing output...\n")
        if first is not None:
            stdout.write(first)
        for ln in lines:
            stdout.write(ln)
        stdout.flush()
        mark("write")
        if os.environ.get("HYMET_SCREEN_TIMING"):
            prev = t0
            for what, t in marks:
                stderr.write("[timing] %-40s %8.3f s\n" % (what, t - prev))
                prev = t
            stderr.write("[timing] %-40s %8.3f s\n" % ("total inside screen_main", prev - t0))
        return 0
    except hs.HsError as e:
        _e(e.msg)
        return 1


SKETCH_USAGE = """
Usage:

  mash sketch [options] <input> [<input>] ...

Description:

  Create a sketch file (.msh): for every input file the s smallest distinct
  canonical k-mer hashes of all its records (one reference per file, named after
  the file).  Inputs are FASTA or FASTQ, gzipped or not.  Computed on the GPU
  with the same hash kernel as `mash screen`, many genomes per kernel pass.

Options:

  -h          Help
  -l          List input. Each positional argument is a file that lists one
              input path per line (empty lines are ignored).
  -o <path>   Output prefix (".msh" is appended unless present) [first input]
  -p <int>    Host threads reading, inflating and packing input files [1]
  -k <int>    K-mer size, 1-32 [21]
  -s <int>    Sketch size [1000]
  -S <int>    Hash seed [42]
"""


def sketch_main(args: List[str], stdout=None) -> int:
    """`mash sketch` (SURVEY.md 8f rank 1): HYMET never runs it (its three databases are
    downloaded pre-built, README.md:164-169) but a drop-in without it cannot refresh them."""
    stdout = stdout or sys.stdout
    k, s, seed, threads, out, lists = 21, 1000, 42, 1, None, False
    pos: List[str] = []
    i = 0
    try:
        while i < len(args):
            a = args[i]
            if a == "-h":
                stdout.write(SKETCH_USAGE)
                return 0
            if a == "-l":
                lists = True
            elif a in ("-o", "-k", "-s", "-S", "-p"):
                if i + 1 >= len(args):
                    _err("-%s requires an argument" % a[1])
                    return 1
                v = args[i + 1]
                i += 1
                if a == "-o":
                    out = v
                elif a == "-k":
                    k = int(v)
                elif a == "-s":
                    s = int(v)
                elif a == "-S":
                    seed = int(v)
                else:
                    threads = int(v)
            elif a.startswith("-") and a != "-":
                _err("Unrecognized option: %s" % a)
                return 1
            else:
                pos.append(a)
            i += 1
    except ValueError:
        _err("malformed numeric option value")
        return 1
    if not pos:
        stdout.write(SKETCH_USAGE)
        return 0
    if not (1 <= k <= 32) or s < 1:
        _err("k-mer size must be 1-32 and sketch size positive")
        return 1
    if threads < 1:
        _err("option value out of range")
        return 1
    paths: List[str] = []
    if lists:
        for lf in pos:
            try:
                with open(lf, "rb") as fh:
                    listed = fh.read()
            except OSError:
                _err("could not open %s for reading." % lf)
                return 1
            paths += [os.fsdecode(ln) for ln in listed.split(b"\n") if ln]
        if not paths:
            _err("no input files listed in %s" % " ".join(pos))
            return 1
    else:
        paths = pos
    for p in paths:
        if not os.path.exists(p):
            _err("could not open %s for reading." % p)
            return 1
    import numpy as np

    from . import msh as mshfmt
    from . import screen as hs
    device = int(os.environ.get("HYMET_SCREEN_DEVICE", "0"))
    sys.stderr.write("Sketching %d file%s...\n" % (len(paths), "" if len(paths) == 1 else "s"))
    try:
        sketches, _ = hs.sketch_files(paths, k, s, seed, threads, device)
    except hs.HsError as e:
        _err(e.msg)
        return 1
    from .distance import sketch_comment
    comments = [sketch_comment(g.header, g.n_records) for g in sketches]
    offsets = np.concatenate([[0], np.cumsum([len(g.hashes) for g in sketches])]).astype(np.uint64)
    db = mshfmt.SketchDB(k=k, s=s, seed=seed, names=list(paths), comments=comments,
                         lengths=np.array([g.length for g in sketches], np.uint64), offsets=offsets,
                         hashes=np.concatenate([g.hashes for g in sketches]) if sketches else np.zeros(0, np.uint64))
    out = out or pos[0]
    if not out.endswith(".msh"):
        out += ".msh"
    sys.stderr.write("Writing to %s...\n" % out)
    mshfmt.write_msh(out, db)
    return 0


DIST_USAGE = """
Usage:

  mash dist [options] <reference>.msh <query> [<query>] ...

Description:

  Estimate the distance of each query sequence to each reference sketch.  The
  reference is one sketch file (.msh); queries are sketch files (.msh) or
  FASTA/FASTQ files, gzipped or not, which are sketched with the reference's
  k-mer size, sketch size and seed (one sketch per file).  The output fields are
  [reference-ID, query-ID, distance, p-value, shared-hashes].  Computed on the
  GPU, exactly as Mash 2.3 computes it.

Options:

  -h          Help
  -p <int>    Host threads sketching sequence queries and formatting output [1]
  -l          List input. Each query is a file that lists one input path per
              line (empty lines are ignored).
  -t          Table output (one row per query, distances only).
  -C          Show comments for sequences (name:comment).
  -v <num>    Maximum p-value to report. (0-1) [1.0]
  -d <num>    Maximum distance to report. (0-1) [1.0]
"""

# sketching options of `mash dist`: Mash refuses them when the reference is a sketch (its parameters win)
_DIST_SKETCH_OPTS = {"-k", "-s", "-S", "-w", "-a", "-z", "-n", "-Z", "-r", "-b", "-c", "-m", "-g", "-i"}
_DIST_VALUE_OPTS = {"-p", "-v", "-d", "-k", "-s", "-S", "-w", "-z", "-b", "-c", "-m", "-g"}


def _dist_first_positional(args: List[str]) -> Optional[str]:
    i = 0
    while i < len(args):
        a = args[i]
        if a.startswith("-") and len(a) > 1:
            i += 2 if a in _DIST_VALUE_OPTS else 1
            continue
        return a
    return None


def distance_main(args: List[str], stdout=None, stderr=None) -> int:
    """`mash dist` against a reference sketch file (DESIGN.md §5 "mash dist"): exact Mash 2.3 distances on the GPU."""
    stdout = stdout or sys.stdout
    stderr = stderr or sys.stderr
    _e = lambda msg: _err(msg, stderr)
    threads, lists, table, comments, pmax, dmax = 1, False, False, False, 1.0, 1.0
    pos: List[str] = []
    i = 0
    try:
        while i < len(args):
            a = args[i]
            if a == "-h":
                stdout.write(DIST_USAGE)
                return 0
            if a == "-l":
                lists = True
            elif a == "-t":
                table = True
            elif a == "-C":
                comments = True
            elif a in ("-p", "-v", "-d"):
                if i + 1 >= len(args):
                    _e("-%s requires an argument" % a[1])
                    return 1
                v = args[i + 1]
                i += 1
                if a == "-p":
                    threads = int(v)
                elif a == "-v":
                    pmax = float(v)
                else:
                    dmax = float(v)
            elif a in _DIST_SKETCH_OPTS:
                _e("Sketching option %s cannot be used when the reference is a sketch (.msh): its parameters are used" % a)
                return 1
            elif a.startswith("-") and a != "-":
                _e("Unrecognized option: %s" % a)
                return 1
            else:
                pos.append(a)
            i += 1
    except ValueError:
        _e("malformed numeric option value")
        return 1
    if len(pos) < 2:
        stdout.write(DIST_USAGE)
        return 0
    if threads < 1 or not (0.0 <= pmax <= 1.0) or not (0.0 <= dmax <= 1.0):
        _e("option value out of range")
        return 1
    ref_path, queries = pos[0], pos[1:]
    if not ref_path.endswith(".msh"):
        _e("%s does not look like a sketch (.msh)" % ref_path)
        return 1
    if lists:
        listed: List[str] = []
        for lf in queries:
            try:
                with open(lf, "rb") as fh:
                    listed += [os.fsdecode(ln) for ln in fh.read().split(b"\n") if ln]
            except OSError:
                _e("could not open %s for reading." % lf)
                return 1
        if not listed:
            _e("no input files listed in %s" % " ".join(queries))
            return 1
        queries = listed
    for p in [ref_path] + queries:
        if not os.path.isfile(p):
            _e("could not open %s for reading." % p)
            return 1

    from . import distance as dist
    from ._abi import HsError
    try:
        ref = dist.HostMsh(ref_path)
        for p in queries:                      # every query sketch file is checked before the GPU is touched
            if dist.is_msh(p):
                m = dist.HostMsh(p)
                why = dist.mismatch(ref.header, m.header)
                m.close()
                if why:
                    _e("%s: %s" % (p, why))
                    return 1
        d = dist.Distance(ref, int(os.environ.get("HYMET_SCREEN_DEVICE", "0")))
        try:
            dist.add_queries(d, queries, threads, int(os.environ.get("HYMET_SCREEN_DEVICE", "0")),
                             warn=lambda msg: stderr.write("WARNING: %s\n" % msg))
            stdout.flush()
            d.run(stdout.fileno(), dmax, pmax, table, comments, threads)
        finally:
            d.close()
            ref.close()
    except HsError as e:
        _e(e.msg)
        return 1
    return 0


def _via_server(args: List[str]) -> Optional[int]:
    """Hand `mash screen args` to the resident table server (hymet_b200/server.py) when
    HYMET_SCREEN_SERVER is 1 (use it if it answers) or auto (start it first if it does not).  None =
    no server took the request: the caller screens in-process, exactly as without the variable."""
    if "-" in args or "-h" in args:
        return None                      # standard input belongs to this process
    from . import server
    path = server.default_socket_path()
    req = {"op": "screen", "argv": list(args), "cwd": os.getcwd()}
    try:
        return server.request(path, req)
    except OSError:
        pass
    if os.environ.get("HYMET_SCREEN_SERVER") != "auto":
        return None
    try:
        server.spawn_detached(path, int(os.environ.get("HYMET_SCREEN_DEVICE", "0")))
        return server.request(path, req)
    except OSError as e:
        sys.stderr.write("WARNING: no screen server (%s); screening in-process\n" % e)
        return None


def main(argv: Optional[List[str]] = None) -> int:
    argv = sys.argv[1:] if argv is None else argv
    if not argv or argv[0] in ("-h", "--help", "help"):
        sys.stdout.write("mash (hymet-screen-b200): commands `screen`, `sketch` and `dist` (against a .msh reference) "
                         "are provided.\n" + USAGE)
        return 0
    if argv[0] == "--version":
        sys.stdout.write("2.3-hymet-screen-b200\n")
        return 0
    if argv[0] == "sketch":
        return sketch_main(argv[1:])
    if argv[0] == "dist":
        first = _dist_first_positional(argv[1:])
        if (first is None and "-h" in argv[1:]) or (first is not None and first.endswith(".msh")):
            return distance_main(argv[1:])
    if argv[0] == "screen" and os.environ.get("HYMET_SCREEN_SERVER", "0") not in ("", "0"):
        rc = _via_server(argv[1:])
        if rc is not None:
            return rc
    if argv[0] != "screen":
        # HYMET uses nothing else (SURVEY.md 8b); hand over to a real mash when one exists further down PATH
        me = os.path.realpath(sys.argv[0])
        for d in os.environ.get("PATH", "").split(os.pathsep):
            cand = os.path.join(d, "mash")
            if os.path.isfile(cand) and os.access(cand, os.X_OK) and os.path.realpath(cand) != me:
                os.execv(cand, [cand] + argv)
        sys.stderr.write("mash (hymet-screen-b200): command '%s' is not provided by this drop-in\n" % argv[0])
        return 2
    return screen_main(argv[1:])


if __name__ == "__main__":
    sys.exit(main())

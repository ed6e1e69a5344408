"""Regenerate the `mash dist` goldens (DESIGN.md §5 "mash dist"):

  distance_pvalue_kat.json   D3 p-values at 40 digits (mpmath), r computed with Mash's double expression
  zymo_dist.tsv              zymo25.msh against itself, default options, written by the CPU oracle
                             (tests/distance_oracle/distance_oracle.c)
  zymo_dist_table.tsv        the same with -t

    python tests/golden/make_distance_golden.py
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

# (common, reference length, query length, k, denom): small and large k, tails on both sides of the mean,
# the full sketch, a single shared hash, unequal lengths
KAT_CASES = [
    (1, 5_000_000, 5_000_000, 21, 1000), (2, 5_000_000, 4_000_000, 21, 1000), (10, 3_000_000, 6_000_000, 21, 1000),
    (100, 5_000_000, 5_000_000, 21, 1000), (999, 5_000_000, 5_000_000, 21, 1000), (1000, 5_000_000, 5_000_000, 21, 1000),
    (5, 50_000, 80_000, 12, 1000), (40, 2_000_000, 2_000_000, 12, 1000), (300, 2_000_000, 2_000_000, 12, 1000),
    (3, 100_000, 100_000, 16, 10_000), (1234, 4_500_000, 4_600_000, 31, 10_000), (7, 40_000, 9_000_000, 31, 137),
    (2, 1_000, 1_500, 8, 50), (20, 1_000, 1_500, 8, 50), (49, 1_000, 1_500, 8, 50),
]


def r_of(len_ref: int, len_qry: int, k: int) -> float:
    kmer_space = 4.0 ** k
    px = 1. / (1. + kmer_space / len_ref)
    py = 1. / (1. + kmer_space / len_qry)
    return px * py / (px + py - px * py)


def kats():
    import mpmath
    mpmath.mp.dps = 60
    out = []
    for x, lr, lq, k, n in KAT_CASES:
        r = r_of(lr, lq, k)
        p = mpmath.betainc(x, n - x + 1, 0, mpmath.mpf(r), regularized=True)
        out.append({"common": x, "len_ref": lr, "len_qry": lq, "k": k, "denom": n, "r": r.hex(),
                    "pvalue": mpmath.nstr(p, 40)})
    return out


def main() -> int:
    with open(os.path.join(HERE, "distance_pvalue_kat.json"), "w") as fh:
        json.dump(kats(), fh, indent=1)
        fh.write("\n")
    sys.path.insert(0, ROOT)
    from tests import _distance_ref as dref
    dref.build()
    msh = os.path.join(HERE, "zymo25.msh")
    for name, extra in (("zymo_dist.tsv", []), ("zymo_dist_table.tsv", ["-t"])):
        r = subprocess.run([dref.BIN, "dist", "-p", "4", *extra, msh, msh], check=True, capture_output=True)
        with open(os.path.join(HERE, name), "wb") as fh:
            fh.write(r.stdout)
    return 0


if __name__ == "__main__":
    sys.exit(main())

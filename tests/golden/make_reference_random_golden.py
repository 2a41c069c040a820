#!/usr/bin/env python
"""Regenerate reference_random.json.gz: the answers of the compiled, unmodified reference (oracle/_ref/libssw_ref.so, built
by `make -C oracle` with REF= the reference's src directory) to the seeded random cases of test_oracle.random_case --
s_align fields, CIGAR, and mark_mismatch's NM and marked CIGAR; null where ssw_align returns NULL."""
import gzip
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import common as C  # noqa: E402
from test_oracle import RANDOM_SETS, random_case  # noqa: E402


def main():
    if not C.have_ref():
        raise SystemExit("oracle/_ref/libssw_ref.so not built: make -C oracle REF=<reference>/src")
    ref = C.load_ref()
    out = {}
    for seed, count in RANDOM_SETS:
        rng = np.random.default_rng(seed)
        out[str(seed)] = [ref.align(mark=True, **random_case(rng)) for _ in range(count)]
    with gzip.GzipFile(os.path.join(HERE, "reference_random.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(out, separators=(",", ":"), sort_keys=True).encode())


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Regenerate parity_full.json: the compiled, unmodified reference (oracle/_ref/libssw_ref.so, built by `make -C oracle`
with REF= the reference's src directory) aligns every pair of every case of test_gpu_parity_full.py on all usable host
cores; the answers are stored as per-block digests (common.record_digests).  CPU-bound: ~10 minutes on 8 cores."""
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import common as C  # noqa: E402
import test_gpu_parity_full as T  # noqa: E402


def main():
    if not C.have_ref():
        raise SystemExit("oracle/_ref/libssw_ref.so not built: make -C oracle REF=<reference>/src")
    out = {}
    for name in T.CASES:
        c = T.case(name)
        t0 = time.time()
        rec, pool, _, _, kind = C.cpu_batch(c["queries"], c["refs"], c["pair_q"], c["pair_r"], c["mat"], c["n"], impl="reference", **c["kw"])
        assert kind == "reference"
        block = T.block_size(len(rec))
        out[name] = {"pairs": int(len(rec)), "block": block, "digests": C.record_digests(rec, pool, block)}
        print("%s: %d pairs, %.0f s" % (name, len(rec), time.time() - t0), file=sys.stderr)
    with open(T.GOLDEN_FILE, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()

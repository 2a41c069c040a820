"""CPU tests of the PRODUCT's kernel and engine sources, compiled for the fiber emulator
(tests/cuda_emu, test infrastructure) and compared with the oracle.  This is how kernel
logic is validated in the GPU-less build container; the same comparisons run against the
real CUDA library in test_gpu_parity.py.  libssw_emu.so is never used by the product.
"""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import common as C
from test_oracle import golden_inputs, random_case, run_golden

EMU_DIR = os.path.join(C.ROOT, "tests", "cuda_emu")


def _pkg():
    spec = importlib.util.spec_from_file_location("ssw_b200_lib", os.path.join(C.PKG, "ssw_lib.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    return C.SswLib(os.path.join(EMU_DIR, "libssw_emu.so"))


@pytest.fixture(scope="module")
def oracle():
    return C.load_oracle()


def test_emulated_goldens(emu, capfd):
    _latency_instances(True)
    with open(os.path.join(C.GOLDEN, "goldens.json")) as f:
        goldens = json.load(f)
    for case in goldens:
        if "refs_npz" in case:
            continue                       # 1 Mbp reference: GPU test only
        limit = 6 if len(case["reads"]) > 6 else None
        assert run_golden(emu, case, limit) == []


def _latency_instances(on):
    """Small passes use the 32-lane kernel instances ("latency_cols" option, here set on the engines behind ssw_align:
    engine NULL); off = the layouts a large batch gets, so that the small CPU cases cover both families."""
    import ctypes as ct
    lib = ct.CDLL(os.path.join(EMU_DIR, "libssw_emu.so"))
    lib.ssw_engine_set_option.argtypes = [ct.c_void_p, ct.c_char_p, ct.c_int64]
    lib.ssw_engine_set_option.restype = ct.c_int
    assert lib.ssw_engine_set_option(None, b"latency_cols", (1 << 20) if on else 0) == 0
    assert lib.ssw_engine_set_option(None, b"no such option", 1) != 0


@pytest.mark.parametrize("latency", [True, False])
def test_emulated_random_vs_oracle(emu, oracle, latency, capfd):
    _latency_instances(latency)
    rng = np.random.default_rng(424242 + int(latency))
    bad = []
    n = 0
    while n < 80:
        c = random_case(rng)           # every gap regime, incl. gapO <= gapE (lane-literal kernel)
        n += 1
        d = C.diff_results(emu.align(**c), oracle.align(**c))
        if d:
            bad.append((n, d))
    _latency_instances(False)          # the remaining tests of this module exercise the batch layouts
    assert bad == []


def test_emulated_chunked_reference(oracle, capfd):
    """Reference chunking with warm-up overlap (forced small chunks) must not change any field."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    eng.set_option("chunk", 64)
    rng = np.random.default_rng(99)
    mat = C.dna_matrix(2, 2)
    ref = rng.integers(0, 4, size=1500).astype(np.int8)
    reads = [C.mutate_read(rng, ref, int(rng.integers(0, 1400)), int(rng.integers(20, 41)), 0.1, 0.02, 0.02) for _ in range(7)]
    reads.append(rng.integers(0, 4, size=33).astype(np.int8))
    eng.set_sequences(reads, [ref])
    for flag in (0, 0x0f, 1):
        eng.set_option("tb_maxbw", 0 if flag == 1 else -1)      # flag 1: the single-warp traceback kernel
        res, pool = eng.align(mat, 5, 3, 2, flag=flag, filterd=32767, mask_len=15, score_size=2)
        for i, q in enumerate(reads):
            exp = oracle.align(q, ref, mat, 5, 3, 2, flag, 0, 32767, 15, 2)
            r = res[i]
            got = {k: int(r[k]) for k in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")}
            got["cigar"] = [int(x) for x in pool[r["cigar_off"]: r["cigar_off"] + r["cigar_len"]]] if r["cigar_off"] >= 0 else []
            assert C.diff_results(got, exp) == [], (flag, i)
    eng.set_option("tb_maxbw", -1)
    eng.close()


def test_emulated_long_queries_strip_pipeline(oracle, capfd):
    """Queries longer than one 512-row strip: strip-pipelined kernel, forward and reverse (early termination,
    several super-blocks with parked registers), paired and unpaired, followed by the traceback."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    eng.set_option("tb_spec", 0)               # band-doubling rounds one after the other: the emulator runs warps serially, and the
                                               # side-by-side rounds are covered by the random and wide-band cases
    eng.set_option("super", 256)
    rng = np.random.default_rng(515)
    mat = C.dna_matrix(2, 2)
    ref = rng.integers(0, 4, size=1800).astype(np.int8)
    reads = [C.mutate_read(rng, ref, int(rng.integers(0, 600)), n, 0.08, 0.02, 0.02) for n in (600, 1100, 530)]
    reads.append(C.mutate_read(rng, np.concatenate([ref, ref[::-1]]), 100, 2100, 0.08, 0.02, 0.02))      # 7 strips: splits 4+3 and 2+2+2+1
    eng.set_sequences(reads, [ref])
    for flag, parts in ((0x0f, 1), (0x0f, 2), (0, 4)):      # parts: strips of a task split over CTAs
        eng.set_option("parts", parts)
        res, pool = eng.align(mat, 5, 3, 1, flag=flag, filterd=32767, mask_len=100, score_size=2)
        for i, q in enumerate(reads):
            exp = oracle.align(q, ref, mat, 5, 3, 1, flag, 0, 32767, 100, 2)
            r = res[i]
            got = {k: int(r[k]) for k in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")}
            got["cigar"] = [int(x) for x in pool[r["cigar_off"]: r["cigar_off"] + r["cigar_len"]]] if r["cigar_off"] >= 0 else []
            assert C.diff_results(got, exp) == [], (flag, parts, i)
    eng.set_option("parts", 0)
    # reverse pass with two unrelated alignments per strip task: different references, end columns and scan lengths
    ref2 = np.concatenate([rng.integers(0, 4, size=700).astype(np.int8), ref[900:1500], rng.integers(0, 4, size=150).astype(np.int8)])
    refs2 = [ref, ref2, ref[:900].copy()]
    eng.set_sequences(reads, refs2)
    # the same batch cut into slices that run on helper engines (views of the resident sequences, own scratch)
    base_res, base_pool = eng.align(mat, 5, 3, 1, flag=0x0f, filterd=32767, mask_len=100, score_size=2)
    k = 0
    for q in reads:
        for rr in refs2:
            exp = oracle.align(q, rr, mat, 5, 3, 1, 0x0f, 0, 32767, 100, 2)
            r = base_res[k]
            got = {f: int(r[f]) for f in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")}
            got["cigar"] = [int(x) for x in base_pool[r["cigar_off"]: r["cigar_off"] + r["cigar_len"]]] if r["cigar_off"] >= 0 else []
            assert C.diff_results(got, exp) == [], k
            k += 1
    for slices, taper in ((3, 0), (5, 60)):      # equal slices; five slices, each 60 % of the one before it
        eng.set_option("slices", slices)
        eng.set_option("slice_taper", taper)
        res, pool = eng.align(mat, 5, 3, 1, flag=0x0f, filterd=32767, mask_len=100, score_size=2)
        assert len(pool) == len(base_pool)
        for a, b in zip(res, base_res):
            for f in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag", "cigar_len"):
                assert int(a[f]) == int(b[f]), (slices, f)
            if a["cigar_len"] > 0:
                assert list(pool[a["cigar_off"]: a["cigar_off"] + a["cigar_len"]]) == list(base_pool[b["cigar_off"]: b["cigar_off"] + b["cigar_len"]])
    eng.set_option("slices", 0)
    eng.set_option("slice_taper", 0)
    eng.set_option("super", 0)
    eng.close()


def test_emulated_batch_grid_mixed_lengths(oracle, capfd):
    """The batch ABI on a queries x references grid with ragged lengths: pair-task formation, CTA-shared profiles,
    word-first prediction (long queries) with fall-back to byte semantics, byte->word re-resolve and re-fill."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    rng = np.random.default_rng(2024)
    mat = C.dna_matrix(2, 2)
    refs = [rng.integers(0, 4, size=n).astype(np.int8) for n in (300, 517, 90)]
    qlens = (16, 40, 40, 150, 152, 260, 272, 300, 33, 7)
    queries = []
    for i, n in enumerate(qlens):
        r = refs[i % len(refs)]
        if len(r) > n + 20 and i % 3 != 2:
            queries.append(C.mutate_read(rng, r, int(rng.integers(0, len(r) - n - 10)), n, 0.04 if n > 200 else 0.12, 0.01, 0.01))
        else:
            queries.append(rng.integers(0, 4, size=n).astype(np.int8))
    eng.set_sequences(queries, refs)
    for score_size in (2, 1, 0):
        for flag in (0, 9):
            res, pool = eng.align(mat, 5, 3, 1, flag=flag, filterd=32767, mask_len=-1, score_size=score_size)
            k = 0
            for q in queries:
                for r in refs:
                    exp = oracle.align(q, r, mat, 5, 3, 1, flag, 0, 32767, len(q) // 2, score_size)
                    rr = res[k]
                    if exp is None:
                        assert int(rr["status"]) == 1, (score_size, flag, k)
                    else:
                        got = {f: int(rr[f]) for f in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")}
                        got["cigar"] = [int(x) for x in pool[rr["cigar_off"]: rr["cigar_off"] + rr["cigar_len"]]] if rr["cigar_off"] >= 0 else []
                        assert int(rr["status"]) == 0 and C.diff_results(got, exp) == [], (score_size, flag, k)
                    k += 1
    eng.close()


def test_emulated_word_saturation(emu, oracle, capfd):
    """Scores that reach the reference's signed 16-bit saturation (ssw.c:483) go through the lane-literal kernel."""
    rng = np.random.default_rng(1)
    mat = C.dna_matrix(127, 100)
    r = rng.integers(0, 4, size=500).astype(np.int8)
    for qlen, flag, ss in ((300, 0, 1), (290, 15, 2), (256, 1, 2)):
        q = r[60:60 + qlen].copy()
        q[qlen // 2] = (q[qlen // 2] + 1) % 4
        a = emu.align(q, r, mat, 5, 40, 3, flag, 0, 32767, 50, ss)
        b = oracle.align(q, r, mat, 5, 40, 3, flag, 0, 32767, 50, ss)
        assert b["score1"] >= 32000 and C.diff_results(a, b) == [], (qlen, flag, ss)


def test_emulated_device_planned_grid(oracle, capfd):
    """Full grids with flag 0 are planned on the device (ssw_grid.cuh); byte overflows come back through the general
    path.  Forced here for a small grid with the "grid_min" option."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    eng.set_option("grid_min", 1)
    rng = np.random.default_rng(31)
    mat = C.dna_matrix(2, 2)
    refs = [rng.integers(0, 4, size=n).astype(np.int8) for n in (260, 97, 400, 33, 180)]
    queries = []
    for i, n in enumerate((150, 150, 140, 33, 64, 17, 150, 100, 1)):
        r = refs[(2 * i) % len(refs)]
        if len(r) > n + 10 and i % 4 != 3:
            queries.append(C.mutate_read(rng, r, int(rng.integers(0, len(r) - n - 5)), n, 0.02 if i < 3 else 0.1, 0.005, 0.005))
        else:
            queries.append(rng.integers(0, 4, size=n).astype(np.int8))
    eng.set_sequences(queries, refs)
    for score_size in (2, 1, 0):
        res, _ = eng.align(mat, 5, 3, 1, flag=0, mask_len=-1, score_size=score_size)
        k = 0
        n_over = 0
        for q in queries:
            for r in refs:
                exp = oracle.align(q, r, mat, 5, 3, 1, 0, 0, 0, len(q) // 2, score_size)
                rr = res[k]
                if exp is None:
                    assert int(rr["status"]) == 1, (score_size, k)
                    n_over += 1
                else:
                    got = {f: int(rr[f]) for f in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")}
                    got["cigar"] = []
                    assert int(rr["status"]) == 0 and C.diff_results(got, exp) == [], (score_size, k)
                k += 1
        if score_size == 0:
            assert n_over > 0          # the high-identity 150-mers overflow 8-bit scores
    # protein grid (BLOSUM50, 24 letters): the CTA-shared profile is 64 KB, so the launch uses eight warps per CTA
    W = C.config_workload(4, n_queries=5, n_targets=37)
    pq, pr = np.repeat(np.arange(5), 37), np.tile(np.arange(37), 5)
    # equal-length queries, forced into launch groups of one query pair: the records come back group by group
    eng.set_option("grid_split", 1)
    eng.set_option("grid_group", 1)
    eng.set_sequences(W["queries"], W["refs"])
    res, pool = eng.align(C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1)
    exp, exp_pool, _, _, _ = C.cpu_batch(W["queries"], W["refs"], pq, pr, C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1, threads=4)
    assert C.compare_records(res, pool, exp, exp_pool) == []
    assert eng.timing()["fill_forward_launches"] == 3
    W["queries"][3] = W["queries"][3][:170]              # another kernel instance and a ragged grid (groups not contiguous: one copy at the end)
    eng.set_sequences(W["queries"], W["refs"])
    res, pool = eng.align(C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1)
    exp, exp_pool, _, _, _ = C.cpu_batch(W["queries"], W["refs"], pq, pr, C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1, threads=4)
    assert C.compare_records(res, pool, exp, exp_pool) == []
    # late arming of the best-cell bookkeeping: a tail so short that many maxima lie before it (those pairs are re-done by the general
    # path), a generous one, and the automatic choice (pilot group first)
    W = C.config_workload(4, n_queries=6, n_targets=41)
    pq6, pr6 = np.repeat(np.arange(6), 41), np.tile(np.arange(41), 6)
    eng.set_sequences(W["queries"], W["refs"])
    exp, exp_pool, _, _, _ = C.cpu_batch(W["queries"], W["refs"], pq6, pr6, C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1, threads=4)
    redone = []
    for arm in (30, 250, -1, 0):
        eng.set_option("grid_arm", arm)
        res, pool = eng.align(C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1)
        assert C.compare_records(res, pool, exp, exp_pool) == [], arm
        redone.append(eng.timing()["byte_overflows"])
    assert redone[0] > 20 and redone[3] == 0, redone          # tail 30: most maxima lie earlier; armed everywhere: nothing to re-do
    eng.set_option("grid_arm", -1)
    # automatic arming where it cannot pay: short queries inside long targets (the best cell lies anywhere): the pilot group is
    # rejected and recomputed armed from column 0 -- nothing is re-done by the general path
    rng2 = np.random.default_rng(99)
    tq = [rng2.integers(0, 20, size=40).astype(np.int8) for _ in range(6)]
    tt = []
    for k in range(30):
        t = rng2.integers(0, 20, size=260).astype(np.int8)
        a = int(rng2.integers(0, 200))
        t[a: a + 40] = tq[k % 6]
        tt.append(t)
    eng.set_sequences(tq, tt)
    res, pool = eng.align(C.BLOSUM50, 24, 12, 2, flag=0, mask_len=20, score_size=1)
    exp, exp_pool, _, _, _ = C.cpu_batch(tq, tt, np.repeat(np.arange(6), 30), np.tile(np.arange(30), 6), C.BLOSUM50, 24, 12, 2, flag=0, mask_len=20,
                                        score_size=1, threads=4)
    assert C.compare_records(res, pool, exp, exp_pool) == []
    assert eng.timing()["byte_overflows"] == 0
    eng.set_option("grid_split", -1)
    eng.set_option("grid_group", -1)
    eng.set_option("grid_min", -1)
    eng.close()


def test_emulated_wide_bands_multi_tile(oracle, capfd):
    """Traceback bands of several 32-column tiles per row (long deletions / insertions): the multi-tile row groups of
    the shared-memory kernel (4-, 2- and 1-tile groups), band doubling inside the kernel, and the global-memory kernel."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    rng = np.random.default_rng(2718)
    mat = C.dna_matrix(2, 2)
    ref = rng.integers(0, 4, size=1600).astype(np.int8)
    ins = rng.integers(0, 4, size=70).astype(np.int8)
    reads = [
        np.concatenate([ref[100:330], ref[450:700]]),            # 120-base deletion: band 121 -> 8 tiles per row
        np.concatenate([ref[800:950], ins, ref[950:1150]]),      # 70-base insertion
        np.concatenate([ref[200:300], ref[345:520]]),            # 45-base deletion: 3 tiles
        C.mutate_read(rng, ref, 900, 260, 0.05, 0.03, 0.03),
    ]
    eng.set_sequences(reads, [ref])
    for tb in (-1, 0):
        eng.set_option("tb_maxbw", tb)
        res, pool = eng.align(mat, 5, 3, 1, flag=0x0f, filterd=32767, mask_len=60, score_size=2)
        for i, q in enumerate(reads):
            exp = oracle.align(q, ref, mat, 5, 3, 1, 0x0f, 0, 32767, 60, 2)
            r = res[i]
            got = {k: int(r[k]) for k in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")}
            got["cigar"] = [int(x) for x in pool[r["cigar_off"]: r["cigar_off"] + r["cigar_len"]]] if r["cigar_off"] >= 0 else []
            assert C.diff_results(got, exp) == [], (tb, i)
            assert len(got["cigar"]) >= 1
    eng.set_option("tb_maxbw", -1)
    eng.close()


def test_emulated_text_sequences(oracle, capfd):
    """ssw_engine_set_sequences_text: letter -> code translation, reverse complements and the padded reference layout
    made on the device give the same records as host-translated codes (incl. N, lower case and other letters)."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    rng = np.random.default_rng(4242)
    letters = np.frombuffer(b"ACGTacgtNnUuRY-", dtype=np.uint8)
    weights = np.array([20, 20, 20, 20, 3, 3, 3, 3, 1, 1, 1, 1, 1, 1, 1], dtype=float)
    weights /= weights.sum()
    refs = [bytes(rng.choice(letters, size=int(n), p=weights)) for n in (700, 301, 64)]
    reads = []
    for k in range(9):
        r = refs[k % 3]
        a = int(rng.integers(0, max(1, len(r) - 60)))
        reads.append(r[a: a + int(rng.integers(20, 60))])
    table = np.full(128, 4, dtype=np.int8)
    for i, c in enumerate("ACGT"):
        table[ord(c)] = i
        table[ord(c.lower())] = i
    table[ord("U")] = table[ord("u")] = 3
    comp = {ord("A"): "T", ord("a"): "T", ord("C"): "G", ord("c"): "G", ord("G"): "C", ord("g"): "C", ord("T"): "A", ord("t"): "A",
            ord("U"): "A", ord("u"): "A", ord("N"): "N", ord("n"): "N"}
    def rc(b):
        return bytes(ord(comp[c]) if c in comp else 4 for c in reversed(b))
    def codes(b):
        return table[np.frombuffer(b, dtype=np.uint8) & 127].astype(np.int8)
    mat = C.dna_matrix(2, 2)
    eng.set_sequences_text(reads, refs, table, 5, add_reverse_complement=True)
    res_t, pool_t = eng.align(mat, 5, 3, 1, flag=0x0f, filterd=32767, mask_len=15, score_size=2)
    eng.set_sequences([codes(q) for q in reads] + [codes(rc(q)) for q in reads], [codes(r) for r in refs])
    res_c, pool_c = eng.align(mat, 5, 3, 1, flag=0x0f, filterd=32767, mask_len=15, score_size=2)
    assert len(res_t) == 2 * len(reads) * len(refs)
    for i in range(len(res_t)):
        a, b = res_t[i], res_c[i]
        for k in ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag", "cigar_len"):
            assert int(a[k]) == int(b[k]), (i, k)
        if a["cigar_len"] > 0:
            assert list(pool_t[a["cigar_off"]: a["cigar_off"] + a["cigar_len"]]) == list(pool_c[b["cigar_off"]: b["cigar_off"] + b["cigar_len"]])
    q0 = codes(reads[0]); r0 = codes(refs[0])
    exp = oracle.align(q0, r0, mat, 5, 3, 1, 0x0f, 0, 32767, 15, 2)
    assert int(res_t[0]["score1"]) == exp["score1"] and int(res_t[0]["ref_end1"]) == exp["ref_end1"]
    # a different alphabet size than the one given with the text is refused (no host copy to re-pad from)
    eng.set_sequences_text(reads, refs, table, 5)
    with pytest.raises(RuntimeError):
        eng.align(C.BLOSUM50, 24, 3, 1, flag=0, mask_len=15, score_size=2)
    eng.close()


def test_emulated_align_batch_c_entry(oracle, capfd):
    """ssw_align_batch (host buffers in, heap s_align records out) on the emulator build."""
    import ctypes as ct
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    lib = eng.lib
    rng = np.random.default_rng(3)
    ref = rng.integers(0, 4, size=400, dtype=np.int8)
    reads = [C.mutate_read(rng, ref, int(rng.integers(0, 300)), 60, 0.05, 0.02, 0.02) for _ in range(5)]
    qc, qo = L.concat(reads)
    rc, ro = L.concat([ref])
    mat = np.ascontiguousarray(C.dna_matrix(2, 2), dtype=np.int8)
    P = L.BatchParams(mat.ctypes.data_as(ct.POINTER(ct.c_int8)), 5, 3, 1, 2, 0, 0, 30, 2)
    out = (ct.c_void_p * len(reads))()
    lib.ssw_align_batch.argtypes = [ct.c_void_p, ct.POINTER(L.BatchParams), ct.c_int32, ct.POINTER(ct.c_int8), ct.POINTER(ct.c_int64),
                                    ct.c_int32, ct.POINTER(ct.c_int8), ct.POINTER(ct.c_int64), ct.c_int64, ct.c_void_p, ct.c_void_p, ct.c_void_p]
    lib.ssw_align_batch.restype = ct.c_int
    lib.align_destroy.argtypes = [ct.c_void_p]
    assert lib.ssw_align_batch(eng.h, ct.byref(P), len(reads), qc.ctypes.data_as(ct.POINTER(ct.c_int8)), qo.ctypes.data_as(ct.POINTER(ct.c_int64)),
                               1, rc.ctypes.data_as(ct.POINTER(ct.c_int8)), ro.ctypes.data_as(ct.POINTER(ct.c_int64)), len(reads), None, None, out) == 0
    for i, q in enumerate(reads):
        a = ct.cast(out[i], ct.POINTER(C.SAlign)).contents
        exp = oracle.align(q, ref, mat, 5, 3, 1, 2, 0, 0, 30, 2)
        assert (a.score1, a.ref_begin1, a.ref_end1, a.read_begin1, a.read_end1) == (exp["score1"], exp["ref_begin1"], exp["ref_end1"], exp["read_begin1"], exp["read_end1"])
        assert [int(a.cigar[k]) for k in range(a.cigarLen)] == exp["cigar"]
        lib.align_destroy(out[i])
    eng.close()


def _prebuilt(name):
    """A program of the reference that build() puts in oracle/_ref (made where the reference's source is at hand)."""
    path = os.path.join(C.ORACLE_DIR, "_ref", name)
    if not os.path.exists(path):
        pytest.skip("oracle/_ref/%s not built: the reference's source was not at hand when the checkers were built" % name)
    return path


def _consumer_files(tmp_path):
    """Writes the demo inputs frozen in consumer_outputs.json into tmp_path; returns the frozen runs."""
    with open(os.path.join(C.GOLDEN, "consumer_outputs.json")) as f:
        G = json.load(f)
    for name, text in G["files"].items():
        (tmp_path / name).write_text(text)
    return G


def test_reference_python_driver_unmodified(tmp_path):
    """The reference's own pyssw.py + ssw_lib.py (ctypes) load a library by the name libssw.so: given the emulator build
    of our sources they print what they print with the reference's ssw.c (the ctypes struct mirrors stay compatible)."""
    pyssw = _prebuilt("pyssw.py")
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    if not C.have_ref():
        pytest.skip("compiled reference not available")
    _consumer_files(tmp_path)
    outs = []
    for name, lib in (("ours", os.path.join(EMU_DIR, "libssw_emu.so")), ("ref", C.LIB_REF)):
        d = tmp_path / name
        d.mkdir()
        os.symlink(lib, d / "libssw.so")
        r = subprocess.run([sys.executable, pyssw, "-l", str(d), "-c", "r1.fa", "r1_query.fq"], capture_output=True, text=True, timeout=300,
                           cwd=str(tmp_path), env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
        assert r.returncode == 0, r.stderr[-500:]
        outs.append("\n".join(l for l in r.stdout.splitlines() if not l.startswith("CPU time")))
    assert outs[0] == outs[1] and "optimal_alignment_score: 52" in outs[0]


def test_reference_c_consumers_unmodified_on_emulator_build(tmp_path):
    """CPU replica of test_gpu_parity.py::test_unmodified_reference_consumers_on_our_library: the reference's ssw_test,
    example_c and example_cpp, built unmodified against libssw.so (oracle/_ref/*_b200), run over the emulator build of our
    sources (found through LD_LIBRARY_PATH, which comes before their run path) and reproduce the frozen outputs."""
    exe = {name: _prebuilt(name + "_b200") for name in ("ssw_test", "example_c", "example_cpp")}
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    lib = tmp_path / "lib"
    lib.mkdir()
    os.symlink(os.path.join(EMU_DIR, "libssw_emu.so"), lib / "libssw.so")
    env = dict(os.environ, LD_LIBRARY_PATH=os.pathsep.join(p for p in (str(lib), os.environ.get("LD_LIBRARY_PATH")) if p))
    G = _consumer_files(tmp_path)
    n = 0
    for run in G["runs"]:
        if "1k.fa" in run["args"]:
            continue                       # 100 reads per run: minutes on the emulator; the GPU suite runs them
        out = subprocess.run([exe[run["exe"]]] + run["args"], capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=env)
        got = "\n".join(l for l in out.stdout.splitlines() if not l.startswith("CPU time"))
        assert got == run["stdout"], (run["exe"], run["args"])
        n += 1
    assert n >= 8


def test_emulated_block_column_maxima(capfd):
    """Block-maximum mode of the forward fill (one word per 64 columns + re-fill of the three blocks per alignment whose single
    columns matter) against the one-word-per-column mode and the compiled reference / oracle: second-best score and position
    with the mask window at the start, in the middle, at the end of the reference, repeats (ties broken by the first column),
    window edges on and off block boundaries, several chunk lengths."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    eng.set_option("latency_cols", 0)          # batch layouts (options are per engine)
    eng.set_option("latency_cols", 0)
    rng = np.random.default_rng(2024)
    mat = C.dna_matrix(2, 2)
    motif = rng.integers(0, 4, size=48).astype(np.int8)
    ref = rng.integers(0, 4, size=1700).astype(np.int8)
    for at in (0, 130, 333, 640, 704, 1011, 1652):             # the same motif many times: equal second-best candidates
        ref[at: at + 48] = motif
    ref[400:430] = motif[:30]                                   # a weaker copy
    reads = [motif.copy(), motif[4:44].copy(), np.concatenate([motif[:24], rng.integers(0, 4, size=6).astype(np.int8), motif[24:]])]
    reads += [C.mutate_read(rng, ref, int(rng.integers(0, 1600)), int(rng.integers(25, 60)), 0.08, 0.02, 0.02) for _ in range(9)]
    reads.append(rng.integers(0, 4, size=40).astype(np.int8))
    eng.set_sequences(reads, [ref])
    n = len(reads)
    exp, exp_pool, _, _, _ = C.cpu_batch(reads, [ref], np.arange(n), np.zeros(n), mat, 5, 3, 1, flag=0, mask_len=20, score_size=2,
                                        threads=4)
    assert len(set(int(x) for x in exp["score2"])) > 3 and int((exp["score2"] > 0).sum()) >= n - 2
    for mask_len in (20, 15, 64, 100):
        exp, exp_pool, _, _, _ = C.cpu_batch(reads, [ref], np.arange(n), np.zeros(n), mat, 5, 3, 1, flag=0, mask_len=mask_len,
                                            score_size=2, threads=4)
        for cm_block, chunk in ((1, 0), (1, 64), (1, 128), (1, 320), (0, 64)):
            eng.set_option("cm_block", cm_block)
            eng.set_option("chunk", chunk)
            res, pool = eng.align(mat, 5, 3, 1, flag=0, mask_len=mask_len, score_size=2)
            bad = C.compare_records(res, pool, exp, exp_pool)
            assert bad == [], (mask_len, cm_block, chunk, bad, [(res[i], exp[i]) for i in bad[:2]])
    eng.set_option("cm_block", -1)
    eng.set_option("chunk", 0)
    eng.close()


def test_emulated_resident_reference_cache(emu, oracle, capfd):
    """ssw_align re-uses the resident reference while length and content hash are unchanged; rewriting the caller's buffer in
    place (same pointer, same length) must be noticed.  Also: alphabet changes between calls (the null letter of the pads)."""
    rng = np.random.default_rng(77)
    mat = C.dna_matrix(2, 2)
    ref = rng.integers(0, 4, size=900, dtype=np.int8)
    reads = [C.mutate_read(rng, ref, int(rng.integers(0, 800)), 40, 0.05, 0.01, 0.01) for _ in range(3)]
    for rnd in range(3):
        for q in reads:
            kw = dict(read=q, ref=ref, mat=mat, n=5, gapO=3, gapE=1, flag=0x0f, filters=0, filterd=32767, maskLen=20, score_size=2)
            assert C.diff_results(emu.align(**kw), oracle.align(**kw)) == []
        ref[:] = np.roll(ref, 131)
        ref[int(rng.integers(0, 900))] ^= 1
    # same reference bytes, other alphabet size: the pads must be rewritten with the new null letter
    mat8 = np.zeros((8, 8), dtype=np.int8) - 3
    np.fill_diagonal(mat8, 4)
    kw = dict(read=reads[0], ref=ref, mat=mat8.reshape(-1).copy(), n=8, gapO=5, gapE=2, flag=8, filters=0, filterd=0, maskLen=20, score_size=2)
    assert C.diff_results(emu.align(**kw), oracle.align(**kw)) == []
    kw = dict(read=reads[1], ref=ref, mat=mat, n=5, gapO=3, gapE=1, flag=8, filters=0, filterd=0, maskLen=20, score_size=2)
    assert C.diff_results(emu.align(**kw), oracle.align(**kw)) == []


def test_emulated_argument_validation(capfd):
    """The C ABI rejects malformed input with -1 instead of reading out of bounds, dividing by zero or letting a C++ exception
    escape (round-1 advisor findings): decreasing offsets, offsets that do not start at 0, NULL offset arrays, a full grid over an
    empty reference set, pair indices out of range; an empty batch is fine."""
    import ctypes as ct
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    lib = eng.lib
    I64P, I8P = ct.POINTER(ct.c_int64), ct.POINTER(ct.c_int8)
    q = np.array([0, 1, 2, 3, 0, 1, 2, 3], dtype=np.int8)
    r = np.array([0, 1, 2, 3] * 8, dtype=np.int8)

    def set_seq(nq, qoff, nr, roff):
        qo = np.array(qoff, dtype=np.int64) if qoff is not None else None
        ro = np.array(roff, dtype=np.int64) if roff is not None else None
        return lib.ssw_engine_set_sequences(eng.h, nq, q.ctypes.data_as(I8P), qo.ctypes.data_as(I64P) if qo is not None else None,
                                            nr, r.ctypes.data_as(I8P), ro.ctypes.data_as(I64P) if ro is not None else None)

    assert set_seq(2, [0, 4, 8], 1, [0, 32]) == 0
    assert set_seq(2, [0, 6, 4], 1, [0, 32]) == -1            # decreasing
    assert set_seq(2, [1, 4, 8], 1, [0, 32]) == -1            # does not start at 0
    assert set_seq(2, None, 1, [0, 32]) == -1                 # NULL offsets with sequences
    assert set_seq(2, [0, 4, 8], 1, [0, -5]) == -1            # negative length
    assert set_seq(2, [0, 4, 8], 0, None) == 0                # no references at all is a valid resident set ...
    mat = C.dna_matrix(2, 2)
    P = L.BatchParams(mat.ctypes.data_as(I8P), 5, 3, 1, 0, 0, 0, 15, 2)
    res = np.zeros(4, dtype=L.RESULT_DTYPE)
    used = ct.c_int64(0)
    # ... but a grid over it is not
    assert lib.ssw_engine_align(eng.h, ct.byref(P), 2, None, None, res.ctypes.data_as(ct.c_void_p), None, 0, ct.byref(used)) == -1
    assert lib.ssw_engine_align(eng.h, ct.byref(P), 0, None, None, None, None, 0, ct.byref(used)) == 0
    assert set_seq(2, [0, 4, 8], 1, [0, 32]) == 0
    pq = np.array([0, 5], dtype=np.int32)
    pr = np.array([0, 0], dtype=np.int32)
    assert lib.ssw_engine_align(eng.h, ct.byref(P), 2, pq.ctypes.data_as(ct.POINTER(ct.c_int32)), pr.ctypes.data_as(ct.POINTER(ct.c_int32)),
                                res.ctypes.data_as(ct.c_void_p), None, 0, ct.byref(used)) == -1
    eng.close()


def test_emulated_device_mark_mismatch(oracle, capfd):
    """ssw_engine_mark_mismatch (device) against the exported host mark_mismatch of the checker: soft clips, '=' / 'X' runs that
    span several 32-column groups, insertions and deletions, NM; reads on both strands of the pair list, records without CIGAR."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    rng = np.random.default_rng(8)
    mat = C.dna_matrix(2, 2)
    refs = [rng.integers(0, 4, size=n).astype(np.int8) for n in (900, 400)]
    reads = []
    for k in range(10):
        r = refs[k % 2]
        core = C.mutate_read(rng, r, int(rng.integers(0, len(r) - 260)), int(rng.integers(40, 200)), 0.06, 0.03, 0.03)
        reads.append(np.concatenate([rng.integers(0, 4, size=int(rng.integers(0, 9))).astype(np.int8), core,
                                     rng.integers(0, 4, size=int(rng.integers(0, 9))).astype(np.int8)]))     # unaligned ends -> soft clips
    reads.append(rng.integers(0, 4, size=30).astype(np.int8))
    pq = np.array(list(range(len(reads))) * 2, dtype=np.int32)
    pr = np.array([k % 2 for k in range(len(reads))] + [(k + 1) % 2 for k in range(len(reads))], dtype=np.int32)
    eng.set_sequences(reads, refs)
    res, pool = eng.align(mat, 5, 3, 1, flag=2, filters=30, filterd=32767, mask_len=20, score_size=2, pair_query=pq, pair_ref=pr)
    assert int((res["cigar_len"] > 0).sum()) >= 8 and int((res["cigar_len"] == 0).sum()) >= 2     # filters: some pairs carry no path
    out, marked, nm = eng.mark_mismatch(res, pool, pq, pr)
    n_x = 0
    for p in range(len(pq)):
        q, r = reads[pq[p]], refs[pr[p]]
        exp = oracle.align(q, r, mat, 5, 3, 1, 2, 30, 32767, 20, 2, mark=True)
        if int(res[p]["cigar_len"]) == 0:
            assert int(out[p]["cigar_len"]) == 0 and int(nm[p]) == 0
            continue
        got = [int(x) for x in marked[out[p]["cigar_off"]: out[p]["cigar_off"] + out[p]["cigar_len"]]]
        assert got == exp["cigar_marked"] and int(nm[p]) == exp["nm"], (p, C.cigar_string(got), C.cigar_string(exp["cigar_marked"]))
        n_x += sum(1 for w in got if (w & 15) == 8)
    assert n_x > 5
    eng.close()


def test_emulated_packed_references(capfd):
    """References delivered as a 4-bit (codes 0..4 incl. N) or 2-bit (N-free) packed stream, unpacked on the device, give the
    results of the plain one-byte-per-base input: several references of odd lengths (bases straddling bytes), CIGARs."""
    subprocess.run(["make", "-s", "-C", EMU_DIR], check=True)
    L = _pkg()
    eng = L.BatchAligner(lib_dir=EMU_DIR, lib_name="libssw_emu.so")
    rng = np.random.default_rng(12)
    mat = C.dna_matrix(2, 2)
    for bits, top in ((4, 5), (2, 4)):
        refs = [rng.integers(0, top, size=n).astype(np.int8) for n in (301, 77, 1, 514)]
        reads = [C.mutate_read(rng, refs[k % 4] if len(refs[k % 4]) > 60 else refs[0], 3, 50, 0.05, 0.02, 0.02) for k in range(6)]
        pq = np.repeat(np.arange(6), 4)
        pr = np.tile(np.arange(4), 6)
        eng.set_sequences(reads, refs)
        want, want_pool = eng.align(mat, 5, 3, 1, flag=2, filters=0, filterd=32767, mask_len=25, score_size=2, pair_query=pq, pair_ref=pr)
        nbytes = eng.set_sequences_packed(reads, refs, bits, 5)
        assert nbytes == (sum(len(r) for r in refs) * bits + 7) // 8
        got, got_pool = eng.align(mat, 5, 3, 1, flag=2, filters=0, filterd=32767, mask_len=25, score_size=2, pair_query=pq, pair_ref=pr)
        assert C.compare_records(got, got_pool, want, want_pool) == [] and int((want["cigar_len"] > 0).sum()) >= 6
    eng.close()

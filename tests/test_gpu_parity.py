"""GPU parity tests (run on the B200 box): the CUDA library, called through its C ABI,
must return bit-identical s_align records to the oracle (and to the unmodified reference
library oracle/_ref/libssw_ref.so when that prebuilt checker travelled with the snapshot).
Nothing here reads the reference's source tree."""
import json
import os
import subprocess

import numpy as np
import pytest

import common as C
from test_oracle import RANDOM_SETS, golden_inputs, random_vs_reference, run_golden

pytestmark = pytest.mark.gpu

FIELDS8 = ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag")


def _pkg():
    import importlib.util
    spec = importlib.util.spec_from_file_location("ssw_b200_lib", os.path.join(C.PKG, "ssw_lib.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.fixture(scope="module")
def ours():
    assert os.path.exists(C.LIB_OURS), "libssw.so missing: the CUDA extension must be built in-tree (no fallback)"
    return C.load_ours()


@pytest.fixture(scope="module")
def checker():
    """The strongest checker available: the compiled reference if it travelled, else the oracle port."""
    return C.load_ref() if C.have_ref() else C.load_oracle()


@pytest.fixture(scope="module")
def oracle():
    return C.load_oracle()


@pytest.fixture(scope="module")
def engine():
    L = _pkg()
    e = L.BatchAligner(device=0)
    yield e
    e.close()


def batch_dict(res, pool, i):
    r = res[i]
    d = {k: int(r[k]) for k in FIELDS8}
    d["cigar"] = [int(x) for x in pool[r["cigar_off"]: r["cigar_off"] + r["cigar_len"]]] if r["cigar_off"] >= 0 else []
    return d


def test_goldens_through_ssw_h(ours, capfd):
    """Every frozen golden (demo/old.txt, README sample, config 1, protein, example.c) through ssw_init/ssw_align."""
    with open(os.path.join(C.GOLDEN, "goldens.json")) as f:
        goldens = json.load(f)
    for case in goldens:
        limit = 10 if "refs_npz" in case else None
        assert run_golden(ours, case, limit) == [], case["name"]


def test_demo_golden_1M_batched(engine):
    """The reference's shipped regression golden (100 x 54 bp vs 1 Mbp, demo/old.txt) through the batch ABI."""
    with open(os.path.join(C.GOLDEN, "goldens.json")) as f:
        case = [c for c in json.load(f) if "refs_npz" in c][0]
    mat, refs, reads = golden_inputs(case)
    engine.set_sequences(reads, refs)
    res, pool = engine.align(mat, 5, 3, 1, flag=0, mask_len=-1, score_size=2)
    for i, exp in enumerate(case["expected"]):
        assert C.diff_results(batch_dict(res, pool, i), exp) == [], i


def test_random_pairs_vs_checker(ours, capfd):
    """1,500 random cases of every gap regime, incl. gapO <= gapE (lane-literal kernel), against the stored answers of the
    unmodified reference (fields, CIGAR, NM and marked CIGAR)."""
    assert random_vs_reference(ours, RANDOM_SETS[1][0]) == []


@pytest.mark.parametrize("flag", [0, 8, 2, 0x0f])
def test_config2_shape_reduced(engine, checker, flag, capfd):
    """Config 2 shape at a size the checker finishes in seconds: 150 bp reads vs a 300 kbp reference, all flags."""
    ref, reads = C.make_dna_workload(300_000, 96, 150, seed_ref=1001, seed_reads=2002)
    mat = C.dna_matrix(2, 2)
    engine.set_sequences(reads, [ref])
    res, pool = engine.align(mat, 5, 3, 1, flag=flag, filters=0, filterd=32767, mask_len=75, score_size=2)
    n_check = len(reads) if C.have_ref() else 12
    for i in range(n_check):
        exp = checker.align(reads[i], ref, mat, 5, 3, 1, flag, 0, 32767, 75, 2)
        assert C.diff_results(batch_dict(res, pool, i), exp) == [], (flag, i)


def test_config2_full_size_properties(engine, checker, capfd):
    """BASELINE config 2 at full size (1,000 x 150 bp vs 5 Mbp): chunk-size invariance of every field, agreement of a
    fixed subsample with the checker, and the score bounds the workload model implies."""
    ref, reads = C.make_dna_workload(5_000_000, 1000, 150, seed_ref=1001, seed_reads=2002)
    mat = C.dna_matrix(2, 2)
    engine.set_sequences(reads, [ref])
    res_a, _ = engine.align(mat, 5, 3, 1, flag=0, mask_len=75, score_size=2)
    engine.set_option("chunk", 20000)
    res_b, _ = engine.align(mat, 5, 3, 1, flag=0, mask_len=75, score_size=2)
    engine.set_option("chunk", 0)
    assert (res_a == res_b).all()
    assert int(res_a["score1"].max()) <= 300 and int(res_a["score1"].min()) > 0
    assert (res_a["ref_end1"] < 5_000_000).all() and (res_a["read_end1"] < 150).all()
    assert engine.timing()["byte_overflows"] >= 0
    sub = list(range(0, 1000, 64)) if C.have_ref() else [0]
    for i in sub:
        exp = checker.align(reads[i], ref, mat, 5, 3, 1, 0, 0, 0, 75, 2)
        got = {k: int(res_a[i][k]) for k in FIELDS8}
        got["cigar"] = []
        assert C.diff_results(got, exp) == [], i


def test_protein_word_path(engine, checker, capfd):
    """Config 4 shape reduced: BLOSUM50, 300 aa queries x 400 aa targets, score_size 1 (word semantics)."""
    rng = np.random.default_rng(4004)
    queries = [rng.integers(0, 20, size=300).astype(np.int8) for _ in range(12)]
    targets = []
    for t in range(40):
        s = rng.integers(0, 20, size=400).astype(np.int8)
        if t % 4 == 0:
            q = queries[int(rng.integers(0, len(queries)))]
            seg = q[50:250].copy()
            m = rng.random(len(seg)) < 0.2
            seg[m] = rng.integers(0, 20, size=int(m.sum()))
            s[100:300] = seg
        targets.append(s)
    engine.set_sequences(queries, targets)
    res, pool = engine.align(C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1)
    k = 0
    for q in queries:
        for t in targets:
            exp = checker.align(q, t, C.BLOSUM50, 24, 3, 1, 0, 0, 0, 150, 1)
            assert C.diff_results(batch_dict(res, pool, k), exp) == [], k
            k += 1


def test_device_planned_grid(engine, checker, capfd):
    """Config 4 shape through the device-planned grid path (ssw_grid.cuh; forced with grid_min = 1): BLOSUM50 word
    scores, and a DNA byte-score grid whose overflows are re-done by the general path."""
    engine.set_option("grid_min", 1)
    try:
        rng = np.random.default_rng(4004)
        queries = [rng.integers(0, 20, size=int(n)).astype(np.int8) for n in (300, 300, 299, 301, 120, 77, 300)]
        targets = []
        for t_i in range(60):
            s = rng.integers(0, 20, size=int(rng.integers(350, 450))).astype(np.int8)
            if t_i % 5 == 0:
                q = queries[int(rng.integers(0, 4))]
                seg = q[40:240].copy()
                m = rng.random(len(seg)) < 0.2
                seg[m] = rng.integers(0, 20, size=int(m.sum()))
                s[60:260] = seg
            targets.append(s)
        engine.set_sequences(queries, targets)
        res, pool = engine.align(C.BLOSUM50, 24, 3, 1, flag=0, mask_len=150, score_size=1)
        k = 0
        for q in queries:
            for t_ in targets:
                exp = checker.align(q, t_, C.BLOSUM50, 24, 3, 1, 0, 0, 0, 150, 1)
                assert C.diff_results(batch_dict(res, pool, k), exp) == [], k
                k += 1
        ref, reads = C.make_dna_workload(3000, 40, 150, seed_ref=9, seed_reads=10, p_sub=0.03)
        refs = [ref[:1500].copy(), ref[1000:].copy(), ref[500:2600].copy()]
        mat = C.dna_matrix(2, 2)
        engine.set_sequences(reads, refs)
        res, pool = engine.align(mat, 5, 3, 1, flag=0, mask_len=-1, score_size=2)
        assert engine.timing()["byte_overflows"] > 0
        k = 0
        for q in reads:
            for r in refs:
                exp = checker.align(q, r, mat, 5, 3, 1, 0, 0, 0, 75, 2)
                assert C.diff_results(batch_dict(res, pool, k), exp) == [], k
                k += 1
    finally:
        engine.set_option("grid_min", -1)


def test_byte_overflow_falls_back_to_word(engine, ours, checker, capfd):
    """Scores >= 255 - bias: score_size 2 re-runs with word semantics (ssw.c:883-886); score_size 0 returns NULL (:887-890)."""
    rng = np.random.default_rng(5)
    ref = rng.integers(0, 4, size=4000).astype(np.int8)
    reads = [C.mutate_read(rng, ref, int(rng.integers(0, 3000)), 400, 0.03, 0.005, 0.005) for _ in range(8)]
    reads.append(rng.integers(0, 4, size=400).astype(np.int8))
    mat = C.dna_matrix(2, 2)
    engine.set_sequences(reads, [ref])
    for flag in (0, 0x0f):
        res, pool = engine.align(mat, 5, 3, 1, flag=flag, filterd=32767, mask_len=200, score_size=2)
        assert engine.timing()["byte_overflows"] >= 8
        for i, q in enumerate(reads):
            exp = checker.align(q, ref, mat, 5, 3, 1, flag, 0, 32767, 200, 2)
            assert C.diff_results(batch_dict(res, pool, i), exp) == [], (flag, i)
    assert ours.align(reads[0], ref, mat, 5, 3, 1, 0, 0, 0, 200, score_size=0) is None
    assert checker.align(reads[0], ref, mat, 5, 3, 1, 0, 0, 0, 200, score_size=0) is None


@pytest.mark.parametrize("flag", [2, 0x0f])
def test_config5_shape_long_reads(engine, checker, flag, capfd):
    """Config 5 shape: 10 kbp reads x 100 kbp reference (byte pass overflows -> word), strip-pipelined fill, reverse
    pass with early termination, banded traceback; every field and every CIGAR word."""
    ref, reads = C.make_dna_workload(100_000, 12 if C.have_ref() else 2, 10_000, seed_ref=5005, seed_reads=5006,
                                     decoy_frac=0.0, p_sub=0.05, p_ins=0.02, p_del=0.02)
    reads.append(reads[0][:3000].copy())                       # ragged batch: a shorter long read
    reads.append(reads[1][:700].copy())
    mat = C.dna_matrix(2, 2)
    engine.set_sequences(reads, [ref])
    res, pool = engine.align(mat, 5, 3, 1, flag=flag, filters=0, filterd=32767, mask_len=5000, score_size=2)
    for i, q in enumerate(reads):
        exp = checker.align(q, ref, mat, 5, 3, 1, flag, 0, 32767, 5000, 2)
        assert C.diff_results(batch_dict(res, pool, i), exp) == [], (flag, i)


def test_word_saturation_and_linear_gaps(ours, engine, checker, capfd):
    """(i) scores at the reference's signed 16-bit saturation (ssw.c:483); (ii) gapO == gapE on the config-2 shape:
    both are served by the lane-literal kernel and must match the reference exactly."""
    rng = np.random.default_rng(1)
    mat = C.dna_matrix(127, 100)
    r = rng.integers(0, 4, size=700).astype(np.int8)
    for qlen, flag, ss in ((300, 0, 1), (300, 15, 2), (280, 8, 1), (256, 1, 2), (330, 0, 2)):
        q = r[100:100 + qlen].copy()
        q[qlen // 2] = (q[qlen // 2] + 1) % 4
        a = ours.align(q, r, mat, 5, 40, 3, flag, 0, 32767, 50, ss)
        b = checker.align(q, r, mat, 5, 40, 3, flag, 0, 32767, 50, ss)
        assert C.diff_results(a, b) == [], (qlen, flag, ss)
    ref, reads = C.make_dna_workload(60_000, 24, 150, seed_ref=77, seed_reads=78)
    m2 = C.dna_matrix(2, 2)
    engine.set_sequences(reads, [ref])
    for gapO, gapE in ((2, 2), (1, 3)):
        res, pool = engine.align(m2, 5, gapO, gapE, flag=0x0f, filterd=32767, mask_len=75, score_size=2)
        for i, q in enumerate(reads):
            exp = checker.align(q, ref, m2, 5, gapO, gapE, 0x0f, 0, 32767, 75, 2)
            assert C.diff_results(batch_dict(res, pool, i), exp) == [], (gapO, gapE, i)


@pytest.mark.parametrize("score_size,flag", [(2, 0), (2, 0x0f), (1, 9), (0, 1)])
def test_ragged_grid_batch(engine, checker, score_size, flag, capfd):
    """A queries x references grid with ragged lengths (1..1,300 rows, 40..4,000 columns) through the batch ABI:
    exercises pair-task formation, CTA-shared and per-warp profiles, every kernel instance, the strip kernel,
    word-first prediction, byte<->word re-resolve / re-fill, NULL results (score_size 0 overflow)."""
    rng = np.random.default_rng(777 + score_size * 16 + flag)
    mat = C.dna_matrix(2, 2)
    refs = [rng.integers(0, 4, size=int(n)).astype(np.int8) for n in (40, 333, 1000, 2048, 4000, 77, 512)]
    queries = []
    for i in range(96):
        n = int(rng.choice([1, 7, 15, 16, 17, 31, 33, 40, 64, 65, 100, 128, 150, 151, 160, 161, 250, 256, 300, 320, 333, 500, 512, 513, 700, 1300]))
        r = refs[int(rng.integers(0, len(refs)))]
        if len(r) > n + 10 and rng.random() < 0.7:
            queries.append(C.mutate_read(rng, r, int(rng.integers(0, len(r) - n - 5)), n, 0.06 if n > 128 else 0.12, 0.01, 0.01))
        else:
            queries.append(rng.integers(0, 4, size=n).astype(np.int8))
    engine.set_sequences(queries, refs)
    res, pool = engine.align(mat, 5, 3, 1, flag=flag, filters=20, filterd=32767, mask_len=-1, score_size=score_size)
    k = 0
    for q in queries:
        for r in refs:
            exp = checker.align(q, r, mat, 5, 3, 1, flag, 20, 32767, len(q) // 2, score_size)
            if exp is None:
                assert int(res[k]["status"]) == 1, (k, len(q), len(r))
            else:
                assert int(res[k]["status"]) == 0 and C.diff_results(batch_dict(res, pool, k), exp) == [], (k, len(q), len(r))
            k += 1


def test_edge_cases(ours, checker, capfd):
    """Length-1 sequences, all-N queries, zero score, maskLen < 15, ragged batch."""
    mat = C.dna_matrix(2, 2)
    cases = [
        (np.array([0], np.int8), np.array([0], np.int8)),
        (np.array([0], np.int8), np.array([1], np.int8)),
        (np.full(40, 4, np.int8), np.arange(100, dtype=np.int8) % 4),
        (np.arange(17, dtype=np.int8) % 4, np.array([2], np.int8)),
        (np.zeros(16, np.int8), np.zeros(16, np.int8)),
        (np.zeros(15, np.int8), np.zeros(400, np.int8)),
    ]
    for q, r in cases:
        for flag in (0, 1, 0x0f):
            for ml in (5, 15):
                a = ours.align(q, r, mat, 5, 3, 1, flag, 0, 32767, ml, 2)
                b = checker.align(q, r, mat, 5, 3, 1, flag, 0, 32767, ml, 2)
                assert C.diff_results(a, b) == [], (len(q), len(r), flag, ml)


def test_unmodified_reference_consumers_on_our_library(tmp_path, capfd):
    """The reference's own ssw_test / example_c / example_cpp (built UNMODIFIED in the build container against our
    libssw.so) reproduce the outputs the reference produces with its own ssw.c (frozen in consumer_outputs.json)."""
    gold = os.path.join(C.GOLDEN, "consumer_outputs.json")
    bindir = os.path.join(C.ORACLE_DIR, "_ref")
    if not (os.path.exists(gold) and os.path.exists(os.path.join(bindir, "ssw_test_b200"))):
        pytest.skip("prebuilt consumers not present")
    with open(gold) as f:
        G = json.load(f)
    for name, seqs in G["files"].items():
        (tmp_path / name).write_text(seqs)
    for run in G["runs"]:
        exe = os.path.join(bindir, run["exe"] + "_b200")
        out = subprocess.run([exe] + run["args"], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        got = "\n".join(l for l in out.stdout.splitlines() if not l.startswith("CPU time"))
        assert got == run["stdout"], (run["exe"], run["args"])
        native = os.path.join(bindir, run["exe"] + "_native_b200")      # example.cpp over include/ssw_cpp.h
        if os.path.exists(native):
            out = subprocess.run([native], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
            assert "\n".join(out.stdout.splitlines()) == run["stdout"], native


def test_batch_cli_matches_reference_driver(tmp_path):
    """ssw_batch_cli (one ssw_align_batch call for all read x reference x strand pairs) prints, byte for byte, what the
    reference's ssw_test prints (main.c:129-244, :462-532) for the same command lines -- frozen in consumer_outputs.json."""
    exe = os.path.join(C.PKG, "ssw_batch_cli")
    assert os.path.exists(exe), "ssw_batch_cli not built (make -C complete-striped-smith-waterman-library_b200)"
    with open(os.path.join(C.GOLDEN, "consumer_outputs.json")) as f:
        G = json.load(f)
    for name, seqs in G["files"].items():
        (tmp_path / name).write_text(seqs)
    n = 0
    for run in G["runs"]:
        if run["exe"] != "ssw_test":
            continue
        out = subprocess.run([exe] + run["args"], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        assert out.returncode == 0, out.stderr[-500:]
        assert "\n".join(out.stdout.splitlines()) == run["stdout"], run["args"]
        n += 1
    assert n >= 10


def test_cpp_wrapper_matches_reference_wrapper(tmp_path):
    """include/ssw_cpp.h + libssw.so (Align overloads, filters, ReBuild, custom alphabets, AlignBatch) print what the same
    driver prints over the unmodified reference wrapper and ssw.c (tests/golden/cpp_wrapper.txt)."""
    exe = str(tmp_path / "driver_gpu")
    subprocess.run(["g++", "-O2", "-std=c++17", "-DWITH_BATCH", "-I" + os.path.join(C.ROOT, "include"), "-o", exe,
                    os.path.join(C.ROOT, "tests", "cpp_wrapper", "driver.cpp"), "-L" + C.PKG, "-lssw", "-Wl,-rpath," + C.PKG, "-lm"],
                   check=True)
    got = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert got.returncode == 0, got.stderr[-500:]
    assert got.stdout == open(os.path.join(C.GOLDEN, "cpp_wrapper.txt")).read()


def test_concurrent_callers(ours, checker, capfd):
    """ssw_align is called from several host threads at once (the reference is re-entrant, SURVEY 8(b) Threading): every
    caller gets its own, correct record; the calls run side by side (engine pool: own stream and scratch per call, no
    process-wide lock around a call)."""
    import time
    from concurrent.futures import ThreadPoolExecutor
    rng = np.random.default_rng(31337)
    mat = C.dna_matrix(2, 2)
    cases = []
    for _ in range(192):
        ref = rng.integers(0, 4, size=int(rng.integers(20_000, 60_000)), dtype=np.int8)
        start = int(rng.integers(0, len(ref) - 120))
        q = C.mutate_read(rng, ref, start, int(rng.integers(30, 110)), 0.08, 0.02, 0.02)
        cases.append((q, ref, int(rng.choice([0, 1, 2, 8, 0x0f]))))

    def run(c):
        q, ref, flag = c
        return ours.align(q, ref, mat, 5, 3, 1, flag, 0, 32767, max(15, len(q) // 2), 2)

    with ThreadPoolExecutor(8) as ex:                 # warm-up: creates the pool's engines and their scratch
        list(ex.map(run, cases[:32]))
    t0 = time.perf_counter()
    serial = [run(c) for c in cases]
    t_serial = time.perf_counter() - t0
    t0 = time.perf_counter()
    with ThreadPoolExecutor(8) as ex:
        got = list(ex.map(run, cases))
    t_conc = time.perf_counter() - t0
    for c, g, s1 in zip(cases, got, serial):
        q, ref, flag = c
        exp = checker.align(q, ref, mat, 5, 3, 1, flag, 0, 32767, max(15, len(q) // 2), 2)
        assert C.diff_results(g, exp) == [], flag
        assert C.diff_results(s1, exp) == [], flag
    with capfd.disabled():
        print("\n[concurrent callers] 192 ssw_align calls: one thread %.1f ms, eight threads %.1f ms" % (t_serial * 1e3, t_conc * 1e3))
    # correctness is the assertion; the wall times are evidence (tools/call_bench measures the same from C, without the GIL).
    # Calls this small are bound by host-side driver work, which threads contend for; overlap shows once a call carries
    # enough device work (profiles/call_latency_r2.md).
    assert t_conc < 4 * t_serial, (t_serial, t_conc)


def test_resident_reference_is_reused_only_while_its_bytes_are_unchanged(ours, checker, capfd):
    """ssw_align keeps the last reference resident (length + content hash) so that a loop of reads over one reference
    (main.c:462-532) uploads it once; a caller that rewrites the buffer in place must still get answers for the new bytes."""
    rng = np.random.default_rng(99)
    mat = C.dna_matrix(2, 2)
    ref = rng.integers(0, 4, size=50_000, dtype=np.int8)
    reads = [C.mutate_read(rng, ref, int(rng.integers(0, 49_000)), 80, 0.05, 0.01, 0.01) for _ in range(6)]
    for rnd in range(3):
        for q in reads:
            g = ours.align(q, ref, mat, 5, 3, 1, 0x0f, 0, 32767, 40, 2)
            assert C.diff_results(g, checker.align(q, ref, mat, 5, 3, 1, 0x0f, 0, 32767, 40, 2)) == []
        ref[:] = np.roll(ref, 7777)                    # same pointer, same length, different content
        ref[int(rng.integers(0, 50_000))] ^= 1


def test_text_sequences_on_device(engine, checker, capfd):
    """Letters translated, reverse-complemented and padded on the device (ssw_engine_set_sequences_text) against the
    checker run on host-translated codes: both strands of 60 reads x 3 references, every field and CIGAR word."""
    rng = np.random.default_rng(777)
    letters = np.frombuffer(b"ACGTacgtNnUuRY", dtype=np.uint8)
    w = np.array([24, 24, 24, 24, 3, 3, 3, 3, 1, 1, 1, 1, 1, 1], dtype=float)
    w /= w.sum()
    refs = [bytes(rng.choice(letters, size=int(n), p=w)) for n in (20000, 3001, 257)]
    reads = []
    for k in range(60):
        r = refs[k % 3]
        a = int(rng.integers(0, len(r) - 200))
        q = bytearray(r[a: a + int(rng.integers(40, 200))])
        for _ in range(len(q) // 12):
            q[int(rng.integers(0, len(q)))] = int(rng.choice(letters))
        reads.append(bytes(q))
    table = np.full(128, 4, dtype=np.int8)
    for i, c in enumerate("ACGT"):
        table[ord(c)] = i
        table[ord(c.lower())] = i
    table[ord("U")] = table[ord("u")] = 3
    comp = {"A": "T", "a": "T", "C": "G", "c": "G", "G": "C", "g": "C", "T": "A", "t": "A", "U": "A", "u": "A", "N": "N", "n": "N"}

    def rc(b):
        return bytes(ord(comp[chr(c)]) if chr(c) in comp else 4 for c in reversed(b))

    def codes(b):
        return table[np.frombuffer(b, dtype=np.uint8) & 127].astype(np.int8)

    mat = C.dna_matrix(2, 2)
    engine.set_sequences_text(reads, refs, table, 5, add_reverse_complement=True)
    res, pool = engine.align(mat, 5, 3, 1, flag=0x0f, filters=0, filterd=32767, mask_len=20, score_size=2)
    both = reads + [rc(q) for q in reads]
    k = 0
    for q in both:
        for r in refs:
            exp = checker.align(codes(q), codes(r), mat, 5, 3, 1, 0x0f, 0, 32767, 20, 2)
            assert C.diff_results(batch_dict(res, pool, k), exp) == [], k
            k += 1


def test_large_result_array_staged_copy(engine, checker, capfd):
    """A grid whose records exceed the staged-copy threshold (2 x 8 MB): 520,000 pairs of short sequences; pairs sampled
    across every staging chunk are compared with the checker and the whole array with a second, independent call."""
    rng = np.random.default_rng(86420)
    refs = [rng.integers(0, 4, size=int(rng.integers(40, 70)), dtype=np.int8) for _ in range(5200)]
    queries = [rng.integers(0, 4, size=int(rng.integers(24, 40)), dtype=np.int8) for _ in range(100)]
    mat = C.dna_matrix(2, 2)
    engine.set_sequences(queries, refs)
    res, _ = engine.align(mat, 5, 3, 1, flag=0, mask_len=15, score_size=2)
    assert res.nbytes > 2 * (8 << 20)
    pq = np.repeat(np.arange(100, dtype=np.int32), 5200)
    pr = np.tile(np.arange(5200, dtype=np.int32), 100)
    res2, _ = engine.align(mat, 5, 3, 1, flag=0, mask_len=15, score_size=2, pair_query=pq, pair_ref=pr)   # general path, explicit pairs
    for f in ("score1", "score2", "ref_end1", "read_end1", "ref_end2"):
        assert (res[f] == res2[f]).all(), f
    for p in range(0, len(res), 4999):
        q, r = queries[p // 5200], refs[p % 5200]
        exp = checker.align(q, r, mat, 5, 3, 1, 0, 0, 0, 15, 2)
        got = {k: int(res[p][k]) for k in FIELDS8}
        got["cigar"] = []
        assert C.diff_results(got, exp) == [], p


def test_device_mark_mismatch(engine, checker, capfd):
    """ssw_engine_mark_mismatch: '=' / 'X' expansion, soft clips and NM of a batch on the device against the checker's own
    mark_mismatch (ssw.c:1019-1074), for short reads with clipped ends and for 5 kbp reads (thousands of runs per CIGAR)."""
    rng = np.random.default_rng(4242)
    mat = C.dna_matrix(2, 2)
    ref = rng.integers(0, 4, size=60_000).astype(np.int8)
    reads = []
    for k in range(40):
        core = C.mutate_read(rng, ref, int(rng.integers(0, 59_000)), int(rng.integers(60, 240)), 0.06, 0.02, 0.02)
        reads.append(np.concatenate([rng.integers(0, 4, size=int(rng.integers(0, 12))).astype(np.int8), core,
                                     rng.integers(0, 4, size=int(rng.integers(0, 12))).astype(np.int8)]))
    for k in range(8):
        reads.append(C.mutate_read(rng, ref, int(rng.integers(0, 50_000)), 5000, 0.05, 0.02, 0.02))
    engine.set_sequences(reads, [ref])
    res, pool = engine.align(mat, 5, 3, 1, flag=2, filters=0, filterd=32767, mask_len=30, score_size=2)
    out, marked, nm = engine.mark_mismatch(res, pool)
    assert int((out["cigar_len"] > 0).sum()) == len(reads)
    for i, q in enumerate(reads):
        exp = checker.align(q, ref, mat, 5, 3, 1, 2, 0, 32767, 30, 2, mark=True)
        got = [int(x) for x in marked[out[i]["cigar_off"]: out[i]["cigar_off"] + out[i]["cigar_len"]]]
        assert got == exp["cigar_marked"] and int(nm[i]) == exp["nm"], i


def test_packed_reference_input(engine, capfd):
    """A 3 Mbp reference delivered as a 4-bit and as a 2-bit packed stream (unpacked on the device) gives the records of the
    plain one-byte-per-base input, block column maxima and all."""
    ref, reads = C.make_dna_workload(3_000_000, 96, 150, seed_ref=77, seed_reads=78)
    mat = C.dna_matrix(2, 2)
    engine.set_sequences(reads, [ref])
    want, want_pool = engine.align(mat, 5, 3, 1, flag=0, mask_len=75, score_size=2)
    for bits in (4, 2):
        nbytes = engine.set_sequences_packed(reads, [ref], bits, 5)
        assert nbytes == len(ref) * bits // 8
        got, got_pool = engine.align(mat, 5, 3, 1, flag=0, mask_len=75, score_size=2)
        assert C.compare_records(got, got_pool, want, want_pool) == []


def test_two_engines_in_two_threads(capfd):
    """Independent engines (own stream, own scratch) used from two host threads at the same time give the results of a
    lone engine -- the way a caller drives several batches (or several GPUs) from one process."""
    from concurrent.futures import ThreadPoolExecutor
    L = _pkg()
    mat = C.dna_matrix(2, 2)
    work = []
    for seed in (1, 2):
        ref, reads = C.make_dna_workload(200_000, 64, 150, seed_ref=100 + seed, seed_reads=200 + seed)
        long_ref, long_reads = C.make_dna_workload(30_000, 3, 2500, seed_ref=300 + seed, seed_reads=400 + seed, decoy_frac=0.0, p_sub=0.05, p_ins=0.02, p_del=0.02)
        work.append((reads, ref, long_reads, long_ref))

    def run(w):
        reads, ref, long_reads, long_ref = w
        eng = L.BatchAligner(device=0)
        out = []
        for _ in range(2):
            eng.set_sequences(reads, [ref])
            out.append(eng.align(mat, 5, 3, 1, flag=0x0f, filters=0, filterd=32767, mask_len=75, score_size=2))
            eng.set_sequences(long_reads, [long_ref])
            out.append(eng.align(mat, 5, 3, 1, flag=2, filters=0, filterd=32767, mask_len=1000, score_size=2))
        eng.close()
        return out

    solo = [run(w) for w in work]
    with ThreadPoolExecutor(2) as ex:
        both = list(ex.map(run, work))
    for a, b in zip(solo, both):
        for (ra, pa), (rb, pb) in zip(a, b):
            assert (ra == rb).all() and (pa == pb).all()

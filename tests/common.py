"""Shared helpers for the test-suite: ctypes bindings for the three
implementations of the ssw.h ABI (ours, the scalar oracle, the compiled
reference), input generators for the BASELINE.json configurations, and a
field-by-field comparison of s_align records.

Reference interface mirrored by the bindings: src/ssw.h:55-66 (s_align),
:86 ssw_init, :91 init_destroy, :126-134 ssw_align, :139 align_destroy,
:157-164 mark_mismatch.
"""
import ctypes as ct
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "complete-striped-smith-waterman-library_b200")
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_OURS = os.path.join(PKG, "libssw.so")
LIB_ORACLE = os.path.join(ORACLE_DIR, "libssw_oracle.so")
LIB_REF = os.path.join(ORACLE_DIR, "_ref", "libssw_ref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")


class SAlign(ct.Structure):
    """s_align, ssw.h:55-66 (LP64: 40 bytes)."""
    _fields_ = [("score1", ct.c_uint16), ("score2", ct.c_uint16),
                ("ref_begin1", ct.c_int32), ("ref_end1", ct.c_int32),
                ("read_begin1", ct.c_int32), ("read_end1", ct.c_int32),
                ("ref_end2", ct.c_int32), ("cigar", ct.POINTER(ct.c_uint32)),
                ("cigarLen", ct.c_int32), ("flag", ct.c_uint16)]


assert ct.sizeof(SAlign) == 40

I8P = ct.POINTER(ct.c_int8)


def i8ptr(a):
    assert a.dtype == np.int8 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(I8P)


class SswLib:
    """One loaded implementation of the ssw.h ABI (prefix '' or 'oracle_')."""

    def __init__(self, path, prefix=""):
        self.path = path
        self.lib = ct.CDLL(path)
        g = lambda name: getattr(self.lib, prefix + name)
        self.ssw_init = g("ssw_init")
        self.ssw_init.argtypes = [I8P, ct.c_int32, I8P, ct.c_int32, ct.c_int8]
        self.ssw_init.restype = ct.c_void_p
        self.init_destroy = g("init_destroy")
        self.init_destroy.argtypes = [ct.c_void_p]
        self.init_destroy.restype = None
        self.ssw_align = g("ssw_align")
        self.ssw_align.argtypes = [ct.c_void_p, I8P, ct.c_int32, ct.c_uint8, ct.c_uint8, ct.c_uint8,
                                   ct.c_uint16, ct.c_int32, ct.c_int32]
        self.ssw_align.restype = ct.POINTER(SAlign)
        self.align_destroy = g("align_destroy")
        self.align_destroy.argtypes = [ct.POINTER(SAlign)]
        self.align_destroy.restype = None
        self.mark_mismatch = g("mark_mismatch")
        self.mark_mismatch.argtypes = [ct.c_int32, ct.c_int32, ct.c_int32, I8P, I8P, ct.c_int32,
                                       ct.POINTER(ct.POINTER(ct.c_uint32)), ct.POINTER(ct.c_int32)]
        self.mark_mismatch.restype = ct.c_int32

    def align(self, read, ref, mat, n, gapO=3, gapE=1, flag=0, filters=0, filterd=0, maskLen=15,
              score_size=2, mark=False):
        """Run ssw_init + ssw_align (+ optional mark_mismatch) and return a dict, or None for a NULL result."""
        read = np.ascontiguousarray(read, dtype=np.int8)
        ref = np.ascontiguousarray(ref, dtype=np.int8)
        mat = np.ascontiguousarray(mat, dtype=np.int8)
        p = self.ssw_init(i8ptr(read), len(read), i8ptr(mat), n, score_size)
        try:
            r = self.ssw_align(p, i8ptr(ref), len(ref), gapO, gapE, flag, filters, filterd, maskLen)
            if not r:
                return None
            try:
                out = result_dict(r.contents)
                if mark and r.contents.cigarLen > 0:
                    base = ct.addressof(r.contents)
                    cig_pp = ct.cast(base + SAlign.cigar.offset, ct.POINTER(ct.POINTER(ct.c_uint32)))
                    len_p = ct.cast(base + SAlign.cigarLen.offset, ct.POINTER(ct.c_int32))
                    nm = self.mark_mismatch(r.contents.ref_begin1, r.contents.read_begin1, r.contents.read_end1,
                                            i8ptr(ref), i8ptr(read), len(read), cig_pp, len_p)
                    out["nm"] = nm
                    out["cigar_marked"] = [int(r.contents.cigar[i]) for i in range(r.contents.cigarLen)]
                return out
            finally:
                self.align_destroy(r)
        finally:
            self.init_destroy(p)


def result_dict(a):
    return {
        "score1": int(a.score1), "score2": int(a.score2),
        "ref_begin1": int(a.ref_begin1), "ref_end1": int(a.ref_end1),
        "read_begin1": int(a.read_begin1), "read_end1": int(a.read_end1),
        "ref_end2": int(a.ref_end2), "flag": int(a.flag),
        "cigar": [int(a.cigar[i]) for i in range(a.cigarLen)] if a.cigarLen > 0 and a.cigar else [],
    }


def cigar_string(words):
    return "".join("%d%s" % (w >> 4, "MIDNSHP=X"[w & 15] if (w & 15) <= 8 else "M") for w in words)


_built = {}


def build_oracle():
    """Compile the checkers (oracle restatement; the reference too when its tree is present)."""
    if "oracle" not in _built:
        # make's chatter goes to stderr: bench.py prints exactly one JSON line on stdout
        subprocess.run(["make", "-s", "-C", ORACLE_DIR, "all"], check=True, stdout=sys.stderr)
        _built["oracle"] = True


def load_oracle():
    build_oracle()
    return SswLib(LIB_ORACLE, "oracle_")


def have_ref():
    build_oracle()
    return os.path.exists(LIB_REF)


def load_ref():
    build_oracle()
    return SswLib(LIB_REF)


def load_ours():
    return SswLib(LIB_OURS)


# --------------------------------------------------------------------------
# scoring matrices (values restated from the reference drivers)
# --------------------------------------------------------------------------

def dna_matrix(match=2, mismatch=2, n_score=0):
    """5x5 A,C,G,T,N matrix as built by the CLI (main.c:328-335): N row/column = 0."""
    m = np.full((5, 5), -mismatch, dtype=np.int8)
    for i in range(4):
        m[i, i] = match
    m[4, :] = n_score
    m[:, 4] = n_score
    return m.reshape(-1).copy()


def dna_matrix_cpp(match=2, mismatch=2):
    """5x5 matrix as built by the C++ wrapper (ssw_cpp.cpp:26-50): N scores -mismatch."""
    m = np.full((5, 5), -mismatch, dtype=np.int8)
    for i in range(4):
        m[i, i] = match
    return m.reshape(-1).copy()


# BLOSUM50 over "ARNDCQEGHILKMFPSTWYVBZX*" (the CLI's protein default, main.c:43-69)
BLOSUM50 = np.array([
    5, -2, -1, -2, -1, -1, -1, 0, -2, -1, -2, -1, -1, -3, -1, 1, 0, -3, -2, 0, -2, -1, -1, -5,
    -2, 7, -1, -2, -4, 1, 0, -3, 0, -4, -3, 3, -2, -3, -3, -1, -1, -3, -1, -3, -1, 0, -1, -5,
    -1, -1, 7, 2, -2, 0, 0, 0, 1, -3, -4, 0, -2, -4, -2, 1, 0, -4, -2, -3, 5, 0, -1, -5,
    -2, -2, 2, 8, -4, 0, 2, -1, -1, -4, -4, -1, -4, -5, -1, 0, -1, -5, -3, -4, 6, 1, -1, -5,
    -1, -4, -2, -4, 13, -3, -3, -3, -3, -2, -2, -3, -2, -2, -4, -1, -1, -5, -3, -1, -3, -3, -1, -5,
    -1, 1, 0, 0, -3, 7, 2, -2, 1, -3, -2, 2, 0, -4, -1, 0, -1, -1, -1, -3, 0, 4, -1, -5,
    -1, 0, 0, 2, -3, 2, 6, -3, 0, -4, -3, 1, -2, -3, -1, -1, -1, -3, -2, -3, 1, 5, -1, -5,
    0, -3, 0, -1, -3, -2, -3, 8, -2, -4, -4, -2, -3, -4, -2, 0, -2, -3, -3, -4, -1, -2, -1, -5,
    -2, 0, 1, -1, -3, 1, 0, -2, 10, -4, -3, 0, -1, -1, -2, -1, -2, -3, 2, -4, 0, 0, -1, -5,
    -1, -4, -3, -4, -2, -3, -4, -4, -4, 5, 2, -3, 2, 0, -3, -3, -1, -3, -1, 4, -4, -3, -1, -5,
    -2, -3, -4, -4, -2, -2, -3, -4, -3, 2, 5, -3, 3, 1, -4, -3, -1, -2, -1, 1, -4, -3, -1, -5,
    -1, 3, 0, -1, -3, 2, 1, -2, 0, -3, -3, 6, -2, -4, -1, 0, -1, -3, -2, -3, 0, 1, -1, -5,
    -1, -2, -2, -4, -2, 0, -2, -3, -1, 2, 3, -2, 7, 0, -3, -2, -1, -1, 0, 1, -3, -1, -1, -5,
    -3, -3, -4, -5, -2, -4, -3, -4, -1, 0, 1, -4, 0, 8, -4, -3, -2, 1, 4, -1, -4, -4, -1, -5,
    -1, -3, -2, -1, -4, -1, -1, -2, -2, -3, -4, -1, -3, -4, 10, -1, -1, -4, -3, -3, -2, -1, -1, -5,
    1, -1, 1, 0, -1, 0, -1, 0, -1, -3, -3, 0, -2, -3, -1, 5, 2, -4, -2, -2, 0, 0, -1, -5,
    0, -1, 0, -1, -1, -1, -1, -2, -2, -1, -1, -1, -1, -2, -1, 2, 5, -3, -2, 0, 0, -1, -1, -5,
    -3, -3, -4, -5, -5, -1, -3, -3, -3, -3, -2, -3, -1, 1, -4, -4, -3, 15, 2, -3, -5, -2, -1, -5,
    -2, -1, -2, -3, -3, -1, -2, -3, 2, -1, -1, -2, 0, 4, -3, -2, -2, 2, 8, -1, -3, -2, -1, -5,
    0, -3, -3, -4, -1, -3, -3, -4, -4, 4, 1, -3, 1, -1, -3, -2, 0, -3, -1, 5, -3, -3, -1, -5,
    -2, -1, 5, 6, -3, 0, 1, -1, 0, -4, -4, 0, -3, -4, -2, 0, 0, -5, -3, -3, 6, 1, -1, -5,
    -1, 0, 0, 1, -3, 4, 5, -2, 0, -3, -3, 1, -1, -4, -1, 0, -1, -2, -2, -3, 1, 5, -1, -5,
    -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -5,
    -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, -5, 1,
], dtype=np.int8)
assert BLOSUM50.size == 576

NT_CODE = {c: i for i, c in enumerate("ACGT")}
AA_ORDER = "ARNDCQEGHILKMFPSTWYVBZX*"


def encode_dna(s):
    """ASCII -> codes as the CLI's nt_table does (main.c:84-93): A0 C1 G2 T/U3, everything else 4."""
    out = np.full(len(s), 4, dtype=np.int8)
    for i, c in enumerate(s.upper()):
        if c in NT_CODE:
            out[i] = NT_CODE[c]
        elif c == "U":
            out[i] = 3
    return out


def encode_aa(s):
    """ASCII -> codes per the CLI's aa_table (main.c:72-81): unknown letters map to X (22)."""
    idx = {c: i for i, c in enumerate(AA_ORDER)}
    out = np.empty(len(s), dtype=np.int8)
    for i, c in enumerate(s.upper()):
        out[i] = idx.get(c, 23)
    return out


# --------------------------------------------------------------------------
# synthetic workloads (SURVEY.md section 8(d))
# --------------------------------------------------------------------------

def mutate_read(rng, ref, start, length, p_sub=0.15, p_ins=0.01, p_del=0.01, alphabet=4):
    """Copy `length` bases from ref[start:], with deletions, insertions and resampled bases."""
    out = np.empty(length, dtype=np.int8)
    k = 0
    pos = start
    L = len(ref)
    while k < length:
        u = rng.random()
        if u < p_del:
            pos += 1
            continue
        if u < p_del + p_ins:
            out[k] = rng.integers(0, alphabet)
            k += 1
            continue
        b = ref[pos % L]
        pos += 1
        if rng.random() < p_sub:
            b = rng.integers(0, alphabet)
        out[k] = b
        k += 1
    return out


def make_dna_workload(ref_len, n_reads, read_len, seed_ref=1001, seed_reads=2002, decoy_frac=0.05,
                      p_sub=0.15, p_ins=0.01, p_del=0.01):
    """Config 2/3/5-style workload: one random reference + reads sampled from it."""
    ref = np.random.default_rng(seed_ref).integers(0, 4, size=ref_len, dtype=np.int8)
    rng = np.random.default_rng(seed_reads)
    reads = []
    span = max(1, ref_len - read_len - read_len // 3 - 1)
    for _ in range(n_reads):
        if rng.random() < decoy_frac:
            reads.append(rng.integers(0, 4, size=read_len, dtype=np.int8))
        else:
            reads.append(mutate_read(rng, ref, int(rng.integers(0, span)), read_len, p_sub, p_ins, p_del))
    return ref, reads


FIELDS = ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag", "cigar")


def diff_results(a, b, fields=FIELDS):
    """Return a list of (field, a, b) for every differing field (None results compare equal to None)."""
    if a is None or b is None:
        return [] if a is b else [("null", a, b)]
    return [(f, a[f], b[f]) for f in fields if a[f] != b[f]]


# --------------------------------------------------------------------------
# the BASELINE.json configurations as (queries, refs, params) -- shared by the parity tests and bench.py
# --------------------------------------------------------------------------

def config_workload(cfg, n_reads=None, n_queries=None, n_targets=None, ref_len=None, read_len=None):
    """SURVEY 8(d) workloads.  Returns dict(queries, refs, mat, n, gapO, gapE, flag, filters, filterd, mask_len, score_size, name).
    cfg 2: 1,000 x 150 bp vs 5 Mbp (seeds 1001/2002);  cfg 3: 100,000 x 150 bp vs the same reference (seed 3003);
    cfg 4: protein grid, 300 aa queries (seed 4004) x 400 aa targets (seed 4005, every 10th target embeds a mutated
    query segment), BLOSUM50, word scores;  cfg 5: 1,000 x 10 kbp vs 100 kbp (seeds 5005/5006), flag 2 (CIGAR)."""
    if cfg in (2, 3):
        n = n_reads or (1000 if cfg == 2 else 100_000)
        ref, reads = make_dna_workload(ref_len or 5_000_000, n, read_len or 150, seed_ref=1001, seed_reads=2002 if cfg == 2 else 3003)
        return dict(queries=reads, refs=[ref], mat=dna_matrix(2, 2), n=5, gapO=3, gapE=1, flag=0, filters=0, filterd=0,
                    mask_len=(read_len or 150) // 2, score_size=2, name="config%d" % cfg)
    if cfg == 4:
        nq, nt = n_queries or 10_000, n_targets or 50_000
        rq, rt = np.random.default_rng(4004), np.random.default_rng(4005)
        queries = [rq.integers(0, 20, size=300).astype(np.int8) for _ in range(nq)]
        targets = []
        for t in range(nt):
            s = rt.integers(0, 20, size=400).astype(np.int8)
            if t % 10 == 0:
                q = queries[int(rt.integers(0, len(queries)))]
                a = int(rt.integers(0, 100))
                seg = q[a: a + 200].copy()
                m = rt.random(len(seg)) < 0.2
                seg[m] = rt.integers(0, 20, size=int(m.sum()))
                b = int(rt.integers(0, 200))
                s[b: b + 200] = seg
            targets.append(s)
        return dict(queries=queries, refs=targets, mat=BLOSUM50, n=24, gapO=3, gapE=1, flag=0, filters=0, filterd=0,
                    mask_len=150, score_size=1, name="config4")
    if cfg == 5:
        n = n_reads or 1000
        ref, reads = make_dna_workload(ref_len or 100_000, n, read_len or 10_000, seed_ref=5005, seed_reads=5006, decoy_frac=0.0, p_sub=0.05, p_ins=0.02, p_del=0.02)
        return dict(queries=reads, refs=[ref], mat=dna_matrix(2, 2), n=5, gapO=3, gapE=1, flag=2, filters=0, filterd=32767,
                    mask_len=(read_len or 10_000) // 2, score_size=2, name="config5")
    raise ValueError(cfg)


# --------------------------------------------------------------------------
# many pairs on all host cores through a CPU implementation (oracle/ssw_harness.c; test infrastructure)
# --------------------------------------------------------------------------

LIB_HARNESS = os.path.join(ORACLE_DIR, "libssw_harness.so")

HARNESS_DTYPE = np.dtype([("score1", "<u2"), ("score2", "<u2"), ("ref_begin1", "<i4"), ("ref_end1", "<i4"),
                          ("read_begin1", "<i4"), ("read_end1", "<i4"), ("ref_end2", "<i4"),
                          ("cigar_off", "<i4"), ("cigar_len", "<i4"), ("flag", "<u2"), ("status", "<u2")])
assert HARNESS_DTYPE.itemsize == 36


def effective_cores():
    """Host cores this process may really use: scheduler affinity capped by the cgroup CPU quota (a 1-GPU lease of a
    big node reports all of the node's CPUs through os.cpu_count())."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    info = {"affinity": n, "cpu_count": os.cpu_count() or 1, "cgroup_quota": None}
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                      # cgroup v2
            a, b = f.read().split()[:2]
            if a != "max":
                quota = float(a) / float(b)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:      # cgroup v1
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota is not None:
        info["cgroup_quota"] = quota
        n = max(1, min(n, int(np.ceil(quota))))
    info["effective"] = n
    return n, info


def _concat(seqs):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    if len(seqs):
        off[1:] = np.cumsum([len(s) for s in seqs])
    cat = np.concatenate([np.asarray(s, dtype=np.int8) for s in seqs]) if len(seqs) else np.zeros(0, np.int8)
    return np.ascontiguousarray(cat, dtype=np.int8), off


def cpu_batch(queries, refs, pair_q, pair_r, mat, n, gapO=3, gapE=1, flag=0, filters=0, filterd=0, mask_len=-1,
              score_size=2, threads=None, want_cigar=None, impl=None):
    """Align pairs (pair_q[i], pair_r[i]) with a CPU implementation on `threads` host threads (pthread harness).
    impl: "reference" (oracle/_ref/libssw_ref.so), "port" (scalar oracle) or None = reference if present.
    Returns (records[HARNESS_DTYPE], pool[uint32], seconds, cells, kind)."""
    build_oracle()
    if impl is None:
        impl = "reference" if have_ref() else "port"
    path, prefix = (LIB_REF, b"") if impl == "reference" else (LIB_ORACLE, b"oracle_")
    H = ct.CDLL(LIB_HARNESS)
    f = H.ssw_harness_run
    f.restype = ct.c_int
    f.argtypes = [ct.c_char_p, ct.c_char_p, ct.c_int32, ct.c_int64, I8P, ct.POINTER(ct.c_int64), ct.POINTER(ct.c_int32),
                  I8P, ct.POINTER(ct.c_int64), ct.POINTER(ct.c_int32), I8P, ct.c_int32, ct.c_int32, ct.c_int32, ct.c_int32,
                  ct.c_int32, ct.c_int32, ct.c_int32, ct.c_int32, ct.c_void_p, ct.POINTER(ct.c_uint32), ct.c_int64,
                  ct.POINTER(ct.c_int64), ct.POINTER(ct.c_double), ct.POINTER(ct.c_int64)]
    qc, qo = _concat(queries)
    rc, ro = _concat(refs)
    pq = np.ascontiguousarray(pair_q, dtype=np.int32)
    pr = np.ascontiguousarray(pair_r, dtype=np.int32)
    m = np.ascontiguousarray(mat, dtype=np.int8)
    out = np.zeros(len(pq), dtype=HARNESS_DTYPE)
    if want_cigar is None:
        want_cigar = bool(flag & 7)
    cap = 1
    if want_cigar:
        ql, rl = np.diff(qo), np.diff(ro)
        cap = int(np.sum(ql[pq] + np.minimum(rl[pr], ql[pq] * 128) + 4))
    pool = np.zeros(cap, dtype=np.uint32)
    used, secs, cells = ct.c_int64(0), ct.c_double(0), ct.c_int64(0)
    if threads is None:
        threads = effective_cores()[0]
    rv = f(path.encode(), prefix, int(threads), len(pq), i8ptr(qc), qo.ctypes.data_as(ct.POINTER(ct.c_int64)),
           pq.ctypes.data_as(ct.POINTER(ct.c_int32)), i8ptr(rc), ro.ctypes.data_as(ct.POINTER(ct.c_int64)),
           pr.ctypes.data_as(ct.POINTER(ct.c_int32)), i8ptr(m), n, gapO, gapE, flag, filters, filterd, mask_len, score_size,
           out.ctypes.data_as(ct.c_void_p), pool.ctypes.data_as(ct.POINTER(ct.c_uint32)) if want_cigar else None, cap,
           ct.byref(used), ct.byref(secs), ct.byref(cells))
    if rv:
        raise RuntimeError("ssw_harness_run failed (%d)" % rv)
    return out, pool[: used.value], secs.value, cells.value, impl


CMP_FIELDS = ("score1", "score2", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "ref_end2", "flag", "status")


def compare_records(got, got_pool, exp, exp_pool, idx=None):
    """Field-by-field comparison of batch records (ssw_batch_result layout) incl. every CIGAR word.
    got[idx[i]] is compared with exp[i].  Returns the list of mismatching positions i."""
    bad = []
    for i in range(len(exp)):
        g = got[idx[i]] if idx is not None else got[i]
        e = exp[i]
        if int(g["status"]) == 1 and int(e["status"]) == 1:
            continue                      # both sides: ssw_align returns NULL (no record to compare)
        if any(int(g[f]) != int(e[f]) for f in CMP_FIELDS) or int(g["cigar_len"]) != int(e["cigar_len"]):
            bad.append(i)
            continue
        if int(e["cigar_len"]) > 0 and int(e["cigar_off"]) >= 0:
            gw = got_pool[int(g["cigar_off"]): int(g["cigar_off"]) + int(g["cigar_len"])]
            ew = exp_pool[int(e["cigar_off"]): int(e["cigar_off"]) + int(e["cigar_len"])]
            if len(gw) != len(ew) or not np.array_equal(np.asarray(gw), np.asarray(ew)):
                bad.append(i)
    return bad


def record_digests(recs, pool, block):
    """One SHA-256 (first 16 hex digits) per block of `block` consecutive pairs over what compare_records compares: the
    fields of CMP_FIELDS, cigar_len and every CIGAR word (a NULL record, status 1, counts as its status alone).  Equal digest
    lists mean equal answers for every pair, so a large reference answer can be stored as a few kilobytes."""
    import hashlib
    cols = CMP_FIELDS + ("cigar_len",)
    F = np.stack([np.asarray(recs[f], dtype=np.int64) for f in cols], axis=1)
    null = F[:, cols.index("status")] == 1
    F[null] = 0
    F[null, cols.index("status")] = 1
    lens = np.where(null | (np.asarray(recs["cigar_off"]) < 0), 0, F[:, -1])
    offs = np.asarray(recs["cigar_off"], dtype=np.int64)
    starts = np.zeros(len(lens) + 1, dtype=np.int64)
    starts[1:] = np.cumsum(lens)
    idx = np.repeat(offs - starts[:-1], lens) + np.arange(starts[-1])
    words = np.asarray(pool, dtype=np.uint32)[idx].astype("<u4")
    out = []
    for b in range(0, len(F), block):
        e = min(b + block, len(F))
        h = hashlib.sha256(np.ascontiguousarray(F[b:e]).astype("<i8").tobytes())
        h.update(words[starts[b]: starts[e]].tobytes())
        out.append(h.hexdigest()[:16])
    return out

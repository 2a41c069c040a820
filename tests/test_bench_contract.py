"""bench.py's output contract on the CPU: (a) the `--impl reference` arm (the reference's own SSE2 path on the host
cores through the pthread harness) and (b) a dry run of OUR arm's orchestration -- sharding, timing loop, two-phase
gather, parity self-check, sub-results -- on the emulator build of the kernels with tiny shapes, at world size 1 and
under torchrun with two gloo ranks.  Exactly one line on stdout, a JSON object with the keys the driver reads."""
import json
import os
import subprocess
import sys

import common as C

BASE_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e")


def _one_line(out):
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[:500]
    return json.loads(lines[0])


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(C.ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample", "2"], capture_output=True, text=True, timeout=600)
    d = _one_line(out)
    assert d["impl"] == "reference"
    for k in BASE_KEYS + ("cpu_baseline",):
        assert k in d, k
    assert d["unit"] == "GCUPS" and d["value"] > 0 and d["higher_is_better"] is True and d["scaling"] == "strong"
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] in ("reference", "port")
    assert d["cpu_baseline"]["cores"] == C.effective_cores()[0]
    assert "workload" in d["config"] and d["config"]["workload"].startswith("config3")


DRY = ["--dry-run-emu", "--reads", "7", "--steps", "1", "--warmup", "1", "--c4-queries", "3", "--c4-targets", "5", "--parity", "7",
       "--e2e-reps", "1", "--sub-steps", "1"]


def _check_b200_line(d, world):
    for k in BASE_KEYS + ("clocks", "gpu_launches", "roofline", "alu_roofline", "parity", "parity_checked", "mismatches", "config2", "config4", "config5"):
        assert k in d, k
    assert d["n_gpus"] == world and d["scaling"] == "strong" and d["mismatches"] == 0 and d["parity_checked"] >= 7 + 4 + 15 + 3
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    for c in ("config2", "config4", "config5"):
        assert {"value", "e2e", "phases_ms", "alu_roofline", "parity"} <= set(d[c]) and d[c]["parity"]["mismatches"] == 0
    assert d["config5"]["cigar_words"] > 0
    if world == 1:
        assert d["cpu_baseline"]["kind"] in ("reference", "port") and "cpu_baseline" in d["config4"]


def test_b200_arm_dry_run_on_emulator_world1(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(C.ROOT, "bench.py"), "--gpus", "1", "--dump-outputs", str(tmp_path)] + DRY,
                         capture_output=True, text=True, timeout=900)
    d = _one_line(out)
    _check_b200_line(d, 1)
    import numpy as np
    for shape, pairs in (("config3", 7), ("config2", 4), ("config4", 15), ("config5", 3)):
        a = {f: np.load(tmp_path / ("%s_%s.npy" % (shape, f))) for f in ("score1", "ref_end1", "status", "cigar_len")}
        assert len(a["score1"]) == len(a["ref_end1"]) == pairs and (a["score1"] > 0).any()
        cigar = tmp_path / ("%s_cigar.npy" % shape)
        assert cigar.exists() == (shape == "config5")          # flag 2: CIGARs; the other shapes run flag 0
        if cigar.exists():
            a["cigar"] = np.load(cigar)
            assert len(a["cigar"]) == a["cigar_len"].sum() > 0
        assert all(x.dtype == np.float64 for x in a.values())
    files = list(tmp_path.iterdir())
    assert all(np.load(p).size > 0 for p in files)
    total = sum(os.path.getsize(p) for p in files)
    assert 0 < d["dumped_bytes"] <= total <= 64 << 20


def test_b200_arm_dry_run_on_emulator_torchrun_world2():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), os.path.join(C.ROOT, "bench.py"), "--gpus", "2"] + DRY,
                         capture_output=True, text=True, timeout=1200)
    _check_b200_line(_one_line(out), 2)

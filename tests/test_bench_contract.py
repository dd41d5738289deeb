"""The reference arm of bench.py runs on the CPU alone (it times the oracle, the C++ restatement of the reference), so its
JSON contract can be checked without a GPU.  The GPU arm's line carries the same keys plus roofline / e2e details; its
static shape is checked here from the source, and what --dump-outputs writes is checked on the GPU."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "e2e", "cpu_baseline")


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-sample", "1500"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for k in REQUIRED:
        assert k in j, k
    assert j["impl"] == "reference" and j["metric"] == "plonk_by_hand_prove_plus_verify_throughput" and j["unit"] == "proof+verify/s"
    assert j["steps"] == 2 and j["value"] > 0 and j["higher_is_better"] is True and j["vs_baseline"] is None
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in j["config"] and "model" not in j["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_gpu_arm_line_has_the_contract_keys():
    src = open(os.path.join(ROOT, "bench.py")).read()
    body = src[src.index("    line = {\n        \"metric\": METRIC"):]
    for k in REQUIRED + ("clocks", "gpu_launches", "roofline"):
        assert re.search(r'"%s":' % k, body), k
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert re.search(r'"%s":' % k, body[body.index('"roofline"'):]), k
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert re.search(r'"%s":' % k, src[src.index("cpu = {"):]), k


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps" in out.stderr and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(gpu_ctx, tmp_path):
    """--dump-outputs writes what the last timed step computed: with 2 steps on a 2-slot ring that is ring slot 1 (global
    items n .. 2n - 1), recomputed here with the plain prove / verify / bitmap / digest calls."""
    import pbh_b200
    n = 1 << 16
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--reps", "1",
                          "--items", str(n), "--ring", "2", "--no-cpu", "--no-arith", "--no-fs", "--no-uniform", "--no-sweeps",
                          "--no-config2", "--no-config4", "--e2e-steps", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert set(got) == {"item_index", "proof", "status", "result", "verdict_bitmap", "proof_digest"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    ctx = gpu_ctx["table"]
    w, r, c, u = ctx.generate_inputs(n, first_index=n, seed=0xB200, dist=pbh_b200.DIST_FULLPATH)
    p, s = ctx.prove_batch(w, r, c)
    v = ctx.verify_batch(p, c, u)
    bm = ctx.pack_verdicts(v)
    dg = int(ctx.digest(p, first_index=n).item()) & (2**64 - 1)
    ctx.sync()
    assert np.array_equal(got["item_index"], np.arange(n))
    assert np.array_equal(got["proof"], p.cpu().numpy()) and np.array_equal(got["status"], s.cpu().numpy())
    assert np.array_equal(got["result"], v.cpu().numpy()) and np.array_equal(got["verdict_bitmap"], bm.cpu().numpy())
    assert got["proof_digest"].tolist() == [dg & 0xFFFFFFFF, dg >> 32]

"""bench.py's output contract, checked on CPU through the reference arm (the one leg that needs no GPU): exactly one JSON line
on stdout with the keys a caller reads; the N > 1 reference arm prints from rank 0 only.  Without the reference compiled in
place (oracle/_ref) the arm times the oracle's C restatement instead, and the contract is checked on that.  On the GPU: what
`--dump-outputs` writes after the timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "libdelphy_ref.so")
HAVE_REF = os.path.exists(REF)


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1", "--steps", "1",
                           "--warmup", "0", "--cpu-seconds", "0.3", "--spr-studies", "2", "--mcmc-tips", "300", "--mcmc-steps", "20000"],
                          capture_output=True, text=True, timeout=300, env=env)


def test_reference_arm_prints_one_json_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == ("reference" if HAVE_REF else "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["ms_per_step"] > 0
    if HAVE_REF:
        # the reference's own multithreaded scheme (tree cut into one part per thread) and its own CLI's MCMC throughput
        assert d["partitioned"]["kind"] == "reference" and d["partitioned"]["value"] > 0
        stock = os.path.join(ROOT, "oracle", "_ref", "delphy")
        if os.path.exists(stock):
            for case in ("cfg1_200_tips", "cfg3_300_tips"):
                assert d["mcmc"][case]["returncode"] == 0 and d["mcmc"][case]["steps_per_s"] > 0
    # the reference arm loads no product code: its inputs come from libdphy_synth.so
    assert "libdelphy_b200" not in r.stderr


def test_reference_arm_other_ranks_stay_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def _dump(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--chains", "3", "--steps", str(steps), "--warmup", "1",
                        "--evals-per-step", "2", "--spr-studies", "4", "--spr-batches-per-step", "1", "--e2e-chains", "2", "--e2e-threads", "1",
                        "--no-secondary", "--no-partitioned", "--no-mcmc", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["steps"] == steps
    return d, {p.stem: np.load(p) for p in out.glob("*.npy")}


@pytest.mark.gpu
def test_dump_outputs_writes_what_the_timed_steps_computed(tmp_path):
    d, got = _dump(tmp_path / "one_step", 1)
    assert {"log_root_prior", "log_G_below_root", "log_G", "lambda_i", "log_G_general_schedule", "spr_summary_num_regions",
            "spr_region_branch", "spr_region_W_over_Wmax"} <= set(got)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["log_G"].shape == (3,) and float(np.sum(got["log_G"])) == d["log_G_checksum"]
    np.testing.assert_allclose(got["log_G"], got["log_root_prior"] + got["log_G_below_root"], rtol=1e-12)
    np.testing.assert_allclose(got["log_G_general_schedule"], got["log_G"], rtol=1e-11)
    assert got["lambda_i"].size == 3 * d["workload_detail"]["nodes_per_chain"]
    assert got["spr_summary_num_regions"].sum() == d["spr_regions_per_batch"] == got["spr_region_branch"].size
    # same arguments but the step count: the same inputs, so the same arrays, bit for bit
    _, again = _dump(tmp_path / "two_steps", 2)
    assert sorted(again) == sorted(got)
    for k in got:
        assert np.array_equal(again[k], got[k], equal_nan=True), k

"""bench.py's output contract.  Without a GPU: `--impl reference` times the oracle port of the reference's CPU
path and must print exactly ONE JSON line on stdout with the agreed keys; the B200 arm must refuse to run
without a device instead of falling back.  On the GPU: `--steps` sets the timed window and `--dump-outputs`
writes what its last step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "impl"}


def _run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=280, env=dict(os.environ, **(env or {})))


@pytest.mark.timeout(300)
def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--workload", "tiny", "--steps", "2", "--warmup", "1", "--cpu-seconds", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    j = json.loads(lines[0])
    assert KEYS <= set(j), KEYS - set(j)
    assert j["impl"] == "reference" and j["unit"] == "pairs/s" and j["higher_is_better"] is True
    assert j["vs_baseline"] is None and j["steps"] == 2 and j["value"] > 0
    assert "workload" in j["config"] and "model" not in j["config"]
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "candidates" in cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.timeout(300)
def test_reference_arm_non_zero_ranks_exit_quietly():
    r = _run("--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "1", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device behaviour")
@pytest.mark.timeout(120)
def test_b200_arm_has_no_cpu_fallback():
    r = _run("--workload", "tiny", "--steps", "1")
    assert r.returncode != 0 and r.stdout.strip() == ""
    assert "no CUDA device" in r.stderr


@pytest.mark.timeout(240)
def test_dump_outputs_cuts_long_lists_at_fixed_positions(tmp_path):
    """A list over its share of the byte budget keeps the rows at seeded positions, ascending, the same in every
    run; a list within it is written whole.  (Importing bench.py redirects fd 1, hence the subprocess.)"""
    code = ("import sys, torch, bench; "
            "bench.dump_outputs([torch.arange(3000.).reshape(1000, 3), torch.arange(30.).reshape(10, 3)], sys.argv[1], "
            "budget=2 * 100 * 12)")
    got = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, "-c", code, str(tmp_path / d)], cwd=ROOT, capture_output=True, text=True,
                           timeout=200)
        assert r.returncode == 0, r.stderr[-2000:]
        got.append({m: np.load(tmp_path / d / f"{m}.npy") for m in ("adamic_ogb", "gcn")})
    a = got[0]["adamic_ogb"]
    rows = (a[:, 0] / 3).astype(np.int64)                      # input row i is (3i, 3i+1, 3i+2)
    assert a.dtype == np.float32 and a.shape == (100, 3) and np.all(np.diff(rows) > 0)
    assert np.array_equal(a, np.arange(3000, dtype=np.float32).reshape(1000, 3)[rows])
    assert np.array_equal(got[0]["gcn"], np.arange(30, dtype=np.float32).reshape(10, 3))
    for m in got[0]:
        assert np.array_equal(got[0][m], got[1][m]), m


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_b200_arm_dumps_the_last_timed_step(tmp_path):
    """Twice the steps, twice the launches in the timed window; the inputs are seeded, so runs with different
    --steps dump the same lists, and the Adamic-Adar list holds the oracle's scores of its pairs."""
    from edge_proposal_sets_b200 import synth
    from oracle import graph as og, heuristics as oh
    runs = {}
    for steps in (1, 2):
        out = tmp_path / str(steps)
        r = _run("--workload", "tiny", "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-extras",
                 "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-2000:]
        j = json.loads(r.stdout)
        assert j["steps"] == steps
        runs[steps] = j["gpu_launches"], {m: np.load(out / f"{m}.npy") for m in ("adamic_ogb", "gcn")}
    assert runs[2][0] == 2 * runs[1][0] > 0
    for m, a in runs[1][1].items():
        assert a.dtype == np.float32 and a.shape == (500, 3) and np.all(np.diff(a[:, 2]) <= 0), m
        assert np.array_equal(a, runs[2][1][m]), m
    s = synth.make_shape("tiny")
    ei = synth.undirected_edge_index(s["train_edges"])
    g = og.add_edges("tiny", ei, np.ones(ei.shape[1], np.float32), np.zeros((2, 0), np.int64), s["n"])
    aa = runs[1][1]["adamic_ogb"]
    np.testing.assert_allclose(aa[:, 2], oh.aa_ogb_pairs(g, aa[:, :2].astype(np.int64).T), rtol=1e-5)

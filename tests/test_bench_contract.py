"""bench.py's reference arm runs on the host cores only, so its JSON contract can be checked without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from limo_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_dir(path):
    return {f[:-4]: np.load(os.path.join(path, f)) for f in os.listdir(path)}


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "windows/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("BA windows/s") and d["dtype"] == "f64" and d["scaling"] == "weak"
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "config 2" in d["config"]["workload"]


def test_b200_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_format(tmp_path, monkeypatch, oracle):
    """--dump-outputs: one float .npy per array a caller of the batch solve receives, windows along the first axis; over the
    size limit, a seeded sample of whole windows"""
    import bench
    wins = [synth.make_window(1, seed=s) for s in (1, 2, 3)]
    res = [oracle.solve_window(w) for w in wins]
    bench.dump_outputs(str(tmp_path / "all"), res, wins)
    d = _load_dir(tmp_path / "all")
    assert all(a.dtype in (np.float32, np.float64) and len(a) == 3 for a in d.values())
    assert d["kf_pose"].shape == (3, wins[0].n_kf, 7) and d["lm_pos"].shape == (3, wins[0].n_lm, 3)
    assert np.array_equal(d["lm_pos"][1], res[1].lm_pos[:wins[1].n_lm])
    assert np.array_equal(d["lm_rejected"][2], res[2].lm_rejected[:wins[2].n_lm])
    assert np.array_equal(d["final_cost"], [r.c.final_cost for r in res])
    n = res[2].c.num_solves
    assert np.array_equal(d["solve_num_iterations"][2, :n], [s.num_iterations for s in res[2].solves])
    assert not d["solve_final_cost"][2, n:].any()
    total = sum(a.nbytes for a in d.values())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", total * 4)
    bench.dump_outputs(str(tmp_path / "sample"), res * 10, wins * 10)
    s = _load_dir(tmp_path / "sample")
    assert sum(a.nbytes for a in s.values()) <= total * 4 and len(s["window_index"]) == 12
    for k, i in enumerate(s["window_index"].astype(int)):
        assert np.array_equal(s["lm_pos"][k], d["lm_pos"][i % 3])
    bench.dump_outputs(str(tmp_path / "again"), res * 10, wins * 10)
    assert all(np.array_equal(a, np.load(tmp_path / "again" / (k + ".npy"))) for k, a in s.items())


@pytest.mark.gpu
def test_dump_outputs_are_the_solved_batch(tmp_path):
    """the dumped arrays are the results of the timed batch: the same windows solved through the C ABI give them back"""
    from limo_b200 import capi, parallel
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "3",
                        "--distinct", "3", "--cpu-sample", "0", "--no-sub", "--in-flight", "1", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == 2
    d = _load_dir(tmp_path)
    wins = parallel.windows_for_rank(3, 0)
    h = capi.Handle(0)
    ref = h.solve_batch(wins)
    h.close()
    assert np.array_equal(d["window_index"], [0, 1, 2]) and np.array_equal(d["status"], [0, 0, 0])
    for i, (x, w) in enumerate(zip(ref, wins)):
        assert np.array_equal(d["lm_rejected"][i], x.lm_rejected[:w.n_lm])
        assert np.abs(d["kf_pose"][i] - x.kf_pose).max() <= 1e-9
        assert np.percentile(np.abs(d["lm_pos"][i] - x.lm_pos[:w.n_lm]), 95) <= 1e-9
        assert d["final_cost"][i] == pytest.approx(x.c.final_cost, rel=1e-10)
        assert list(d["solve_num_iterations"][i, :x.c.num_solves]) == [s.num_iterations for s in x.solves]

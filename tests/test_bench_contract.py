"""bench.py contract: the reference arm (CPU restatement on the host cores) prints ONE JSON line with the keys its readers
use; under torchrun only rank 0 prints; the GPU arm refuses to run without a device instead of falling back to the CPU;
--dump-outputs writes what the last timed step computed.  Only the last test needs a GPU."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--scale", "0.02"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "ms/LM-iter" and d["higher_is_better"] is False
    assert d["metric"] == json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] == d["value"]
    assert d["config"]["workload"].startswith("synthetic ladybug-1723")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "ms/LM-iter", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert len(d["cg_iterations"]) == 2 and d["steps_timed"] == 2
    op = d["cpu_operator"]  # SURVEY 8(d): T = all cores and T = 1, on the PCG operator
    assert op["ms_1_thread"] > 0


def test_workload_follows_the_gpu_count():
    """N = 1 -> BASELINE configs[1] (ladybug-1723); N > 1 -> configs[3] (venice-1778); both arms print the same config label"""
    sys.path.insert(0, ROOT)
    import bench
    assert bench.default_workload(1) == "ladybug-1723" and bench.default_workload(8) == "venice-1778"
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--scale", "0.002", "--gpus", "8", "--no-single-thread"], env={"RANK": "0"})
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    assert d["config"]["workload"] == bench.WORKLOAD_LABEL["venice-1778"] and d["n_gpus"] == 8


def test_lm_stepper_restarts_after_the_reference_stopping_rule():
    """the timed steps never run past convergence: a terminated solve is followed by a new solve from the initial point"""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from oracle import oracle_py as orc
    from rootba_b200.synthetic import synth_bal
    o = orc.Oracle(synth_bal(12, 300, 4.1, seed=1), np.float64, orc.default_options(num_threads=1))
    secs, wall, st, done = bench.run_lm(bench.OracleBackend(o), np.float64, 2, 30)
    assert done == 30 and len(st.log) == 30
    ends = [i for i, r in enumerate(st.log) if r["terminated"]]
    assert len(ends) >= 2 and st.log[0]["it"] == 1
    for e in ends[:-1]:
        assert st.log[e + 1]["it"] == 1 and st.log[e + 1]["lambda"] == st.log[0]["lambda"]
    # the solves are identical repetitions of the same trajectory
    n = ends[0] + 1
    assert [r["cg_iterations"] for r in st.log[:n]] == [r["cg_iterations"] for r in st.log[n:2 * n]]


def test_reference_arm_other_ranks_stay_silent():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--scale", "0.02", "--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_has_no_cpu_fallback():
    r = _run(["--steps", "1", "--warmup", "1", "--scale", "0.02"], env={"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_bench_rejects_arguments_it_cannot_honour(tmp_path):
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = _run(["--scale", "0.002"] + args)
        assert r.returncode == 2 and "error" in r.stderr, args
    assert not any(tmp_path.iterdir())


def test_dump_outputs_writes_state_and_last_step(tmp_path, monkeypatch):
    """--dump-outputs: cameras, this rank's landmark shard and the last step's record; landmarks over the byte budget are
    cut to the same seeded rows in every run"""
    sys.path.insert(0, ROOT)
    import types
    import numpy as np
    import bench
    rng = np.random.default_rng(5)
    final = (rng.normal(size=(7, 10)).astype(np.float32), rng.normal(size=(500, 3)).astype(np.float32))
    bp = types.SimpleNamespace(cams=np.zeros((7, 10), np.float32), lms=np.zeros((500, 3), np.float32))

    def download_state():
        bp.cams[:], bp.lms[:] = final
    lin = types.SimpleNamespace(bal_problem=bp, download_state=download_state,
                                stats=lambda: {"landmark_begin": 100, "landmark_end": 400})
    last = {"lambda": 1e-4, "cost": 12.5, "l_diff": 3.0, "relative_decrease": 0.9, "cg_iterations": 17, "accepted": True,
            "terminated": False, "device_seconds": 0.01}
    bench.dump_outputs(str(tmp_path / "all"), lin, last)
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in ("cameras", "landmarks", "last_step")}
    assert sorted(p.name for p in (tmp_path / "all").iterdir()) == ["cameras.npy", "landmarks.npy", "last_step.npy"]
    assert got["cameras"].dtype == np.float32 and np.array_equal(got["cameras"], final[0])
    assert np.array_equal(got["landmarks"], final[1][100:400])
    assert got["last_step"].dtype == np.float64 and got["last_step"].tolist() == [1e-4, 12.5, 3.0, 0.9, 17, 1, 0]
    budget = final[0].nbytes + 4096 + 50 * 12
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", budget)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), lin, last)
    a, b = np.load(tmp_path / "a" / "landmarks.npy"), np.load(tmp_path / "b" / "landmarks.npy")
    assert a.shape == (50, 3) and np.array_equal(a, b)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= budget
    rows = {tuple(r) for r in final[1][100:400]}
    assert all(tuple(r) in rows for r in a)


@pytest.mark.gpu
def test_dump_outputs_of_the_gpu_arm(tmp_path):
    """the dumped last step is the last step of the timed trajectory that the JSON line reports"""
    import numpy as np
    r = _run(["--steps", "3", "--warmup", "1", "--scale", "0.02", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
    cams, lms, last = (np.load(tmp_path / f"{n}.npy") for n in ("cameras", "landmarks", "last_step"))
    assert cams.dtype == lms.dtype == np.float32 and cams.shape == (d["config"]["num_cameras"], 10) and lms.shape == (d["config"]["num_landmarks"], 3)
    assert np.all(np.isfinite(cams)) and np.all(np.isfinite(lms))
    assert last[4] == d["cg_iterations"][-1] and bool(last[5]) == d["accepted"][-1]

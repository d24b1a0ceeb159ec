"""bench.py's output contract.  CPU: on the arm that runs without a GPU (`--impl reference`),
exactly ONE line on stdout, valid JSON, every key a consumer of the line reads; the format of
`--dump-outputs`.  GPU: the engine arm dumps the same outputs for the same arguments."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    proc = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--arch", "tiny-gqa",
         "--exit-layer", "3", "--num-speculations", "4", "--steps", "1", "--warmup", "1",
         "--prompt-len", "12", "--cpu-max-steps", "8"],
        capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, proc.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "tokens/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "sample" in cb and cb["value"] == d["value"]
    assert "workload" in d["config"]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                          capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert proc.returncode == 0 and proc.stdout.strip() == ""


def test_dump_outputs_writes_float_arrays_within_budget(tmp_path):
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from layerskip_b200.engine import RoundOutput
    rounds = [RoundOutput(n_drafted=3, n_matches=1, emitted=[7, 8], draft=[7, 9, 9],
                          verified=[7, 8, 4, 4], kv_len=14),
              RoundOutput(n_drafted=2, n_matches=2, emitted=[5, 6, 2], draft=[5, 6],
                          verified=[5, 6, 2], kv_len=17)]
    bench.dump_outputs(str(tmp_path), dict(streams=[[1], [7, 8, 5, 6, 2]], accs=[0.0, 0.6],
                                           last_rounds=rounds))
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["tokens"].tolist() == [7, 8, 5, 6, 2] and got["acceptance_rate"].tolist() == [0.6]
    assert got["round_n_matches"].tolist() == [1, 2] and got["round_kv_len"].tolist() == [14, 17]
    assert got["round_verified_ids"].tolist() == [7, 8, 4, 4, 5, 6, 2]


@pytest.mark.gpu
def test_engine_arm_dumps_identical_outputs_for_identical_arguments(tmp_path):
    import numpy as np
    outs = []
    for run in ("a", "b"):
        proc = subprocess.run(
            [sys.executable, os.path.join(ROOT, "bench.py"), "--arch", "tiny-gqa", "--exit-layer", "3",
             "--num-speculations", "4", "--prompt-len", "12", "--max-steps", "40", "--steps", "3",
             "--warmup", "1", "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path / run)],
            capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert proc.returncode == 0, proc.stderr[-2000:]
        d = json.loads(proc.stdout)
        assert d["steps"] == 3 and d["value"] > 0
        outs.append({p.stem: np.load(p) for p in (tmp_path / run).iterdir()})
    assert outs[0].keys() == outs[1].keys() and "tokens" in outs[0]
    assert 0 < len(outs[0]["tokens"]) <= 40
    for name in outs[0]:
        assert np.array_equal(outs[0][name], outs[1][name]), name


def test_usable_cpu_detection_is_sane():
    sys.path.insert(0, ROOT)
    import bench
    n = bench.usable_cpus()
    assert 1 <= n <= (os.cpu_count() or 1)
    assert 1 <= bench.cpu_threads() <= 32

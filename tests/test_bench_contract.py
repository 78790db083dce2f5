"""bench.py contract checks that do not need a GPU: the reference arm's JSON line."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_schema():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["data"] == "synthetic"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "config", "e2e", "cpu_baseline"):
        assert k in line, k
    assert line["value"] > 0 and line["dtype"] == "f32" and line["vs_baseline"] is None
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    assert "workload" in line["config"]


def test_reference_arm_non_root_rank_exits_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_bad_arguments_are_refused():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr)


def test_dump_blocks_sample():
    bench = _bench_module()
    assert bench.dump_blocks(64, 2, 512).tolist() == list(range(64))          # small outputs are written whole
    T, C, B = bench.T_METRIC, 2, 512
    s = bench.dump_blocks(T, C, B)
    assert np.array_equal(s, bench.dump_blocks(T, C, B))                      # fixed from run to run
    assert s[0] == 0 and s[-1] == T - 1 and np.all(np.diff(s) > 0)
    assert s.size * C * B * 4 <= bench.DUMP_BYTES <= 64 << 20


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """--dump-outputs writes what the last timed call returned: with --blocks T the engine has seen warmup + steps
    calls of the same T-block input, so y is the CPU oracle's output for the last T blocks of that stream."""
    from oracle import oracle as orc
    T, steps, warm = 64, 2, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warm),
                          "--blocks", str(T), "--no-cpu", "--no-e2e", "--no-stream", "--no-traffic", "--no-ir120", "--no-parity",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["warmup"] == warm
    y = np.load(tmp_path / "y.npy")
    assert y.dtype == np.float32 and y.shape == (2, T, 512)
    for c in range(2):
        o = orc.OracleUniform()
        assert o.init(512, orc.synth_ir(480000, c))
        ref = o.run(np.tile(orc.synth_input(T * 512, c), warm + steps), 512)[-T * 512:]
        err = np.max(np.abs(y[c].reshape(-1) - ref)) / np.max(np.abs(ref))
        assert err <= 1e-5, (c, err)

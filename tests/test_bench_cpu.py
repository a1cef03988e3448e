"""bench.py on a box without a GPU: the reference arm (the unmodified reference on the host cores) prints the contract's
JSON line, both arms describe the workload with the same `config` object, and the product arm refuses to run without a
CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _run(*args, timeout=600):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, env=env,
                          cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    if not (os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libopal_ref.so")) or os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so"))):
        pytest.skip("no CPU library built (run __graft_entry__.build() first)")
    r = _run("--impl", "reference", "--workload", "config2", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "GCUPS" and line["unit"] == "GCUPS"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the same `config` object as the product arm's (same function, same workload): the driver compares them
    import bench
    w = bench.make_workload("config2", 0, 1)
    assert line["config"] == bench.config_of(w)
    assert set(line["config"]) == {"workload", "modes", "search", "query_lengths", "matrix", "gap_open", "gap_ext", "db_sequences"}


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "config2"],
                       capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.parametrize("shape", [(1000,), (60, 100000)])
def test_dump_outputs_writes_the_same_float64_sample_every_run(tmp_path, shape):
    import bench
    n = shape[-1]
    rng = np.random.default_rng(5)
    arrays = {name: rng.integers(-2 ** 20, 2 ** 20, shape, dtype=np.int32) for name in ("score", "end_query", "end_target")}
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, n)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["end_query.npy", "end_target.npy", "score.npy", "target_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    cols = np.load(tmp_path / "a" / "target_index.npy").astype(np.int64)
    assert len(cols) == min(n, bench.DUMP_TARGETS) and (np.diff(cols) > 0).all()
    for f in files:
        got = np.load(tmp_path / "a" / f)
        assert got.dtype == np.float64 and (got == np.load(tmp_path / "b" / f)).all()
    for name, a in arrays.items():
        assert (np.load(tmp_path / "a" / f"{name}.npy") == a[..., cols]).all()


def test_product_arm_fails_loudly_without_a_gpu():
    r = _run("--workload", "config2", "--steps", "1", "--warmup", "1", timeout=300)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout) or "no CPU path" in (r.stderr + r.stdout)

"""bench.py's contract on the CPU (the arm that runs without a GPU): `--impl reference` prints exactly ONE line on stdout,
a JSON object with the keys the driver reads, whatever else libraries write to file descriptor 1 during the run; ranks
other than 0 exit 0 without a line; and both arms describe the same workload configuration."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def _run(extra_env=None, args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                           "--steps", "2", "--warmup", "1", *args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.splitlines()
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "path-contexts/sec" and d["unit"] == "ctx/s"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["config"]["workload"] == "tiny"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "ctx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # value is what the line says it is: bags x contexts x steps / time
    B, L = d["config"]["batch_per_gpu"], d["config"]["bag"]
    assert abs(d["value"] - B * L / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]


def test_reference_arm_times_the_steps_it_is_given_and_refuses_dump_outputs(tmp_path):
    r = _run(args=("--steps", "2000", "--warmup", "0"))         # 2000 is the GPU arm's default, not a sentinel here
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2000
    r = _run(args=("--dump-outputs", str(tmp_path / "d")))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and r.stdout == ""
    assert not (tmp_path / "d").exists()


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_dump_outputs_writes_floats_within_the_budget_and_samples_the_same_rows(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 16 << 10)
    g = torch.Generator().manual_seed(0)
    t = {"outputs": torch.randn(64, 100, generator=g), "code_vector": torch.randn(64, 8, generator=g),
         "predicted_label": torch.randint(0, 100, (64,), generator=g)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), t)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["code_vector.npy", "outputs.npy", "outputs_rows.npy", "predicted_label.npy"]
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert sum(os.path.getsize(tmp_path / "a" / f) - 128 for f in files) <= bench.DUMP_BYTES   # 128: the .npy header
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    rows = got["outputs_rows"].astype(np.int64)
    assert 0 < len(rows) < 64 and (np.diff(rows) > 0).all()
    assert np.array_equal(got["outputs"], t["outputs"].numpy()[rows])
    assert np.array_equal(got["code_vector"], t["code_vector"].numpy())
    assert np.array_equal(got["predicted_label"], t["predicted_label"].numpy().astype(np.float64))
    for f in files:
        assert np.array_equal(np.load(tmp_path / "b" / f), got[f[:-4]]), f


def test_stdout_is_protected_from_library_banners():
    """whatever is written to fd 1 while main() runs (NCCL prints its version banner there) ends up on stderr"""
    code = ("import os, runpy, sys; sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'tiny', '--steps', '1', '--warmup', '0'];"
            "import torch; _sp = torch.set_num_threads;"
            "torch.set_num_threads = lambda n: (os.write(1, b'BANNER on fd 1\\n'), _sp(n))[1];"
            "runpy.run_path('bench.py', run_name='__main__')")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.splitlines()
    assert len(lines) == 1 and json.loads(lines[0])["impl"] == "reference", lines
    assert "BANNER on fd 1" in r.stderr

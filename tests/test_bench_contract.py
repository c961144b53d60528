"""bench.py's output contract on the arm that runs without a GPU (`--impl reference`: the oracle timed on the host cores): exactly
ONE line on stdout, a JSON object with the driver's keys on the engine arm's metric / unit / config; under torchrun only rank 0 works.
--dump-outputs on both arms (the engine arm's test needs a GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(extra_env, *args):
    env = dict(os.environ)
    env.update(extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"] + list(args),
                          capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    r = run_bench({})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stdout.splitlines()
    assert len(lines) == 1, r.stdout[:500]          # nothing but the JSON line reaches stdout (library chatter goes to stderr)
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "frames/sec at 656x368 COCO-18" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("C2: COCO 656x368")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "full" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_do_no_work():
    r = run_bench({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout == ""


def check_dump(path, frames, scales):
    """--dump-outputs: float32 arrays of the last step's frames, 64 MB at most, joints consistent with the person counts."""
    files = sorted(os.listdir(path))
    assert files == ["joints.npy", "maps.npy", "num_people.npy", "peaks.npy"]
    a = {f[:-4]: np.load(os.path.join(path, f)) for f in files}
    assert all(v.dtype == np.float32 for v in a.values())
    assert sum(os.path.getsize(os.path.join(path, f)) for f in files) <= 64 << 20
    assert a["num_people"].shape == (frames,) and a["joints"].shape == (frames, 96, 18, 3) and a["peaks"].shape == (frames, 18, 65, 3)
    assert a["maps"].shape == (frames * scales, 57, 46, 82) and np.isfinite(a["maps"]).all() and np.abs(a["maps"]).max() > 0
    for k, n in enumerate(a["num_people"].astype(int)):
        assert (a["joints"][k, n:] == 0).all()
    return a


def test_reference_arm_dumps_its_last_step(tmp_path):
    r = run_bench({}, "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 0, r.stderr[-2000:]
    assert len(r.stdout.splitlines()) == 1
    check_dump(str(tmp_path / "out"), 1, 1)


@pytest.mark.gpu
def test_engine_arm_dumps_its_last_step(tmp_path):
    """The engine arm times exactly --steps steps and writes what the last one computed (9 frames of C2 per step)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.splitlines()[-1])
    assert d["steps"] == 3 and d["config"]["frames_per_step_per_gpu"] == 9
    a = check_dump(str(tmp_path / "out"), 9, 1)
    assert a["num_people"].max() > 0

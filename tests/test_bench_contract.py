"""bench.py contract checks: the reference arm (`--impl reference`) prints ONE JSON line with the agreed keys, the
product arm refuses to run without a CUDA device instead of falling back to the CPU, and (on the GPU) `--dump-outputs`
writes the last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")  # the reference arm is a CPU arm; the product arm must refuse
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, env=env, cwd=ROOT)


def test_reference_arm_json_line():
    p = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "chamfer_pairs_per_s_10k" and d["unit"] == "pairs/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "fp32"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_product_arm_refuses_without_gpu():
    p = _run("--steps", "1", "--warmup", "0")
    assert "no CUDA device" in (p.stdout + p.stderr)
    assert not any(l.strip().startswith("{") for l in p.stdout.splitlines()), "no result line without a GPU"


def test_bad_steps_and_dump_arguments_are_refused(tmp_path):
    for args in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", str(tmp_path / "d"))):
        p = _run(*args)
        assert p.returncode == 2 and "error" in p.stderr and not p.stdout.strip(), args


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    d = tmp_path / "dump"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-extra",
                        "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout)["steps"] == 2
    out = {f[:-4]: np.load(d / f) for f in os.listdir(d)}
    assert sorted(out) == ["cham", "grad_x", "grad_y", "idx_x", "idx_y"]
    assert sum(os.path.getsize(d / (k + ".npy")) for k in out) <= 64 << 20
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in out.values())
    assert out["cham"].shape == (256,) and (out["cham"] > 0).all()
    n = out["idx_x"].shape[0]
    assert n > 0 and out["idx_y"].shape == (n,) and out["grad_x"].shape == out["grad_y"].shape == (n, 3)
    for k in ("idx_x", "idx_y"):
        assert (out[k] == np.round(out[k])).all() and out[k].min() >= 0 and out[k].max() < 10000

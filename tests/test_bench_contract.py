"""CPU: the reference arm of bench.py (`--impl reference`) prints exactly one JSON line with the contract's keys, and the
committed bench lines under profiles/ carry the keys the measurement contract names.  GPU: --dump-outputs writes what
the timed step computed."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and d["steps"] == 1


def test_committed_bench_lines_follow_the_contract():
    for name, n in [("r%d_bench_n%d.json" % (r, n), n) for r in (1, 2) for n in (1, 2, 4, 8)]:
        path = os.path.join(ROOT, "profiles", name)
        with open(path) as f:
            d = json.loads(f.read())
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                    "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"):
            assert key in d, (name, key)
        assert d["n_gpus"] == n and d["scaling"] == "weak" and d["dtype"] == "f32"
        r = d["roofline"]
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
        assert d["gpu_launches"] > 0 and "workload" in d["config"]
    with open(os.path.join(ROOT, "profiles", "r1_bench_n1.json")) as f:
        d = json.loads(f.read())
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    # round 2: the CPU baseline is the reference's own implementation, staged into oracle/_ref by build()
    with open(os.path.join(ROOT, "profiles", "r2_bench_n1.json")) as f:
        d = json.loads(f.read())
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["value"] > 0 and d["cpu_baseline"]["cores"] == 1
    with open(os.path.join(ROOT, "profiles", "r2_bench_reference_n1.json")) as f:
        ref = json.loads(f.read())
    assert ref["impl"] == "reference" and ref["config"] == d["config"] and ref["metric"] == d["metric"]


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_steps_outputs(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--e2e-steps", "1",
                          "--no-cpu-baseline", "--no-kernel-loop", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["grad_rows.npy", "loss.npy"]
    assert sum(os.path.getsize(os.path.join(tmp_path, n)) for n in os.listdir(tmp_path)) <= 64 << 20
    loss = np.load(os.path.join(tmp_path, "loss.npy"))
    rows = np.load(os.path.join(tmp_path, "grad_rows.npy"))
    assert loss.dtype == np.float32 and loss.shape == () and rows.dtype == np.float32
    assert abs(float(loss) - d["loss"]) <= 1e-6 * abs(d["loss"])
    # the same seeded workload through the float64 oracle: reduce="mean" scales every utterance's gradient by 1/B
    bench = importlib.import_module("bench")
    W = bench.WORKLOAD
    prob = importlib.import_module("chainer-speech-recognition_b200.synth").ctc_problem(W["B"], W["T"], W["V"], W["L"], seed=0)
    from oracle import c_oracle
    ref = c_oracle.run(0, prob["x"], prob["labels"], None, prob["input_length"], prob["label_length"], 0,
                       grad_scale=np.full(W["B"], 1.0 / W["B"]))
    assert abs(float(loss) - ref["loss"].mean()) <= 1e-5 * abs(ref["loss"].mean())
    frames = bench.dump_frames(W["T"], W["B"])
    assert rows.shape == (len(frames), W["V"])
    assert np.abs(rows - ref["grad"].reshape(W["T"] * W["B"], W["V"])[frames]).max() <= 1e-5

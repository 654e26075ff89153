"""bench.py's reference arm runs on host cores only, so its JSON line can be checked without a GPU; the GPU arm
must refuse to run without a device (there is no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, timeout=600):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=env, timeout=timeout,
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)


def test_reference_arm_json_line():
    p = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-seconds", "0.5"])
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "eddsa_poseidon_verifies_per_sec" and d["unit"] == "verifies/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_dump_outputs_full_and_sampled(tmp_path):
    """--dump-outputs writes float32 .npy files; an output too large for the budget is replaced by the same seeded sample
    on every run"""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    ok = (np.arange(1000) % 3 == 0).astype(np.uint8)
    bench.dump_outputs(str(tmp_path / "a"), "verify_ok", ok, 0, 1)
    got = np.load(tmp_path / "a" / "verify_ok.npy")
    assert got.dtype == np.float32 and np.array_equal(got, ok)
    big = np.arange(bench.DUMP_BUDGET // 16, dtype=np.uint32) % 2
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), "verify_ok", big, 3, 8)
    a, b = np.load(tmp_path / "b" / "verify_ok_rank3.npy"), np.load(tmp_path / "c" / "verify_ok_rank3.npy")
    assert 8 * a.nbytes <= bench.DUMP_BUDGET and len(a) < len(big) and np.array_equal(a, b)
    p = _run(["--impl", "reference", "--dump-outputs", str(tmp_path / "r")], timeout=120)
    assert p.returncode != 0 and not (tmp_path / "r").exists()


def test_gpu_arm_refuses_to_run_without_a_device():
    p = _run(["--steps", "1", "--warmup", "1"], timeout=300)
    assert p.returncode != 0
    assert "no CPU fallback" in (p.stderr + p.stdout)

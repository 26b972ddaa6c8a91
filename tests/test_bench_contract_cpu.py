"""bench.py's reference arm (the oracle port on host cores) runs without a GPU: check its JSON line against the
driver's contract, single process and under torchrun (rank 0 prints, the other ranks exit 0 without work)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _json_lines(out):
    return [json.loads(l) for l in out.splitlines() if l.startswith("{")]


def _check(line, n_gpus):
    assert REQUIRED <= set(line), sorted(REQUIRED - set(line))
    assert line["impl"] == "reference" and line["metric"] == "tps_pp_rectified_img_per_s" and line["unit"] == "img/s"
    assert line["n_gpus"] == n_gpus and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["value"] > 0 and line["ms_per_step"] > 0 and "workload" in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e = line["e2e"]
    assert e["value"] == line["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_single_process():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--batch", "32"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1
    _check(lines[0], 1)
    # --steps / --warmup / --batch are honoured exactly (the driver compares them with our arm: same_config)
    assert lines[0]["steps"] == 2 and lines[0]["warmup"] == 1 and lines[0]["config"]["global_batch"] == 32


def test_dump_outputs_keeps_a_fixed_sample_under_the_limit(tmp_path):
    """--dump-outputs: float32 .npy per returned array; above 64 MB the same seeded images are kept from every array."""
    import numpy as np
    import torch
    import bench
    item = torch.arange(256, dtype=torch.float32)          # every element of image i holds i
    r = {"output": item[:, None, None, None].expand(256, 64, 16, 64), "pc_score": item[:, None, None].expand(256, 1024, 32)}
    for d in ("a", "b"):
        bench._dump_outputs(str(tmp_path / d), r)
    out, sc = (np.load(tmp_path / "a" / f"{k}.npy") for k in ("output", "pc_score"))
    assert out.dtype == sc.dtype == np.float32 and out.shape[1:] == (64, 16, 64) and sc.shape[1:] == (1024, 32)
    assert 0 < out.shape[0] == sc.shape[0] < 256 and sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 * 10 ** 6
    # whole images, distinct and in batch order, the same ones in both arrays and in both runs
    i = out[:, 0, 0, 0]
    assert np.all(np.diff(i) > 0) and np.all(out == i[:, None, None, None]) and np.all(sc == i[:, None, None])
    for k in ("output", "pc_score"):
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy"))
    small = {"output": torch.randn((4, 3, 8, 8), dtype=torch.float64)}
    bench._dump_outputs(str(tmp_path / "c"), small)
    assert np.array_equal(np.load(tmp_path / "c" / "output.npy"), small["output"].float().numpy())


def test_bench_rejects_zero_steps_and_dump_on_the_reference_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300,
                           cwd=ROOT)
        assert r.returncode == 2 and not _json_lines(r.stdout), extra
    assert not os.listdir(tmp_path)


def test_reference_arm_under_torchrun_prints_once():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29571", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
           "--warmup", "1", "--batch", "32"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = _json_lines(r.stdout)
    assert len(lines) == 1
    _check(lines[0], 2)

"""bench.py's contract, as far as a box without a GPU can check it: the reference arm prints ONE JSON line with the
keys the driver reads, and the product arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("config", ["c2", "c3"])
def test_reference_arm_line(config):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", config,
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "riccati_knots_per_sec" and d["unit"] == "knots/s"
    assert d["higher_is_better"] is True and d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1 and d["gpu_launches"] == 0
    assert d["steps"] == 2
    assert "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "instances per step" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "knots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "needs a CUDA device" in (r.stderr + r.stdout)


@pytest.mark.parametrize("args,message", [
    (["--steps", "0"], "--steps must be at least 1"),
    (["--impl", "reference", "--dump-outputs", "out"], "--impl reference has none to write"),
])
def test_bad_arguments_are_refused(args, message):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args,
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and message in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_same_from_run_to_run(tmp_path):
    """--dump-outputs writes the last timed sweep's outputs (a seeded sample of the batch, 64 MB at most);
    the inputs are seeded, so two runs -- with different step counts -- write the same arrays, and the sampled
    instances named by idx.npy hold what the CPU oracle computes for those instances of the same inputs."""
    import numpy as np
    import torch
    import bench
    import gen
    from oracle import gar_oracle as orc
    dumps = []
    for steps in (2, 3):
        out = tmp_path / ("steps%d" % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                            "--warmup", "1", "--no-cpu", "--no-e2e", "--no-parity", "--strong", "none",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({p.stem: np.load(p) for p in sorted(out.glob("*.npy"))})
    a, b = dumps
    assert set(a) == {"idx", "ff", "fb", "Vxx", "vx", "xs", "us", "lbd0", "lbdas"}
    assert sum(p.stat().st_size for p in (tmp_path / "steps2").glob("*.npy")) <= 64 * 10 ** 6
    n = a["xs"].shape[0]
    assert n >= 16 and a["xs"].shape == (n, 101, 12) and a["fb"].shape == (n, 100, 18, 12)
    for k in a:
        assert a[k].dtype == np.float64 and np.isfinite(a[k]).all() and np.array_equal(a[k], b[k]), k
    idx = a["idx"].astype(np.int64)
    assert idx.shape == (n,) and np.array_equal(idx, a["idx"]) and np.all(np.diff(idx) > 0) and idx[-1] < bench.BATCH
    # the first, a middle and the last sampled instance against the oracle on the same seeded inputs
    pick = [0, n // 2, n - 1]
    inputs = bench.synth_batch_torch(torch, bench.BATCH, bench.HORIZON, bench.NX, bench.NU, torch.device("cuda", 0),
                                     1234, bench.NC)
    host = [x[torch.as_tensor(idx[pick], device=x.device)].cpu().numpy() for x in inputs]
    bo = orc.BatchedOracle(bench.NX, bench.NU, bench.NC, bench.NCT, bench.NX, bench.HORIZON, len(pick), *host)
    bo.sweep(bench.MUEQ, nthreads=1)
    assert bool((bo.status == 1).all())
    ref = bo.get()
    nu = bench.NU
    for j, i in enumerate(pick):
        assert gen.rel_fro(a["fb"][i][:, :nu], ref["fb"][j][:, :nu]) <= 1e-9
        assert gen.rel_fro(a["ff"][i][:, :nu], ref["ff"][j][:, :nu]) <= 1e-9
        for k in ("Vxx", "xs", "us"):
            assert gen.rel_fro(a[k][i], ref[k][j]) <= 1e-9, k

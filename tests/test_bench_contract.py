"""bench.py prints ONE JSON line on stdout with the keys the driver reads (CPU: the reference arm; GPU: our arm)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT

BASE_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e")


def run_bench(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                       cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "stdout must hold exactly one line, got %d" % len(lines)
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--envs", "512")
    for k in BASE_KEYS + ("impl", "cpu_baseline"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "shielded agent-steps/s" and d["unit"] == "agent-steps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_our_arm_line():
    d = run_bench("--envs", "8192", "--steps", "3", "--warmup", "3", "--cpu-seconds", "1")
    for k in BASE_KEYS + ("clocks", "gpu_launches", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["dtype"] == "f64" and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["gpu_launches"] >= 3
    assert d["e2e"]["h2d_bytes_per_step"] == 8192 * 12 and d["e2e"]["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["value"] > 0 and c["cores"] >= 1 and "sample" in c
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


@pytest.mark.gpu
def test_dumped_outputs_repeat_from_run_to_run(tmp_path):
    """--dump-outputs: float32 / float64 .npy files within 64 MB (a seeded sample of the envs when all of them would not
    fit), the same on two runs with the same arguments, and equal to what the last timed step returns when the
    benchmark's env is stepped here directly (warm-up and timed steps)."""
    import bench
    import numpy as np
    import torch
    import marl_mass_b200 as mm
    from marl_mass_b200 import dist as mmd
    E, K, W = 65536, 4, 3
    runs = []
    for r in range(2):
        out = tmp_path / ("run%d" % r)
        d = run_bench("--envs", str(E), "--steps", str(K), "--warmup", str(W), "--skip-extra", "--skip-cpu",
                      "--dump-outputs", str(out))
        assert d["steps"] == K and d["warmup"] == W
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 * 10 ** 6
        runs.append({f.name[:-4]: np.load(str(f)) for f in sorted(out.iterdir())})
    a, b = runs
    assert set(a) == set(bench.DUMP_KEYS + ("env_index",))
    idx = a["env_index"]
    assert 30000 < len(idx) < E and (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < E
    assert a["obs"].shape == (len(idx), mm.MAXV, mm.NS)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    leg = bench.Leg(mm, mmd, "mass_td3", E, 0, 0)
    try:
        for t in list(range(W)) + list(range(K)):
            leg.step(t)
        torch.cuda.synchronize()
        sel = torch.from_numpy(idx.astype(np.int64)).cuda()
        v = leg.env.buffers()
        for k in bench.DUMP_KEYS:
            assert np.array_equal(v[k].index_select(0, sel).cpu().numpy().astype(np.float32), a[k]), k
        # and one step more gives other outputs: the dump is of exactly the last timed step
        leg.step(K)
        assert not np.array_equal(v["obs"].index_select(0, sel).cpu().numpy(), a["obs"])
    finally:
        leg.close()
    live = np.arange(mm.MAXV)[None, :] < a["n_agents"][:, None]
    assert live.any() and (np.abs(a["obs"][live]).sum(1) > 0).all() and (a["obs"][~live] == 0).all()

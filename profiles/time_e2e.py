"""Host-path timing: python profiles/time_e2e.py [envs] [steps]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
import marl_mass_b200 as mm
from bench import WORKLOADS
E = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
K = int(sys.argv[2]) if len(sys.argv) > 2 else 20
cfg = dict(mm.DEFAULT_CONFIG, **WORKLOADS["mass_td3"]["cfg"])
env = mm.MergeEnvBatched(E, cfg)
env.reset(seed=1)
acts = [torch.randint(0, 5, (E, mm.MAXV), dtype=torch.int8).pin_memory().numpy() for _ in range(4)]
dev_acts = [torch.from_numpy(a).cuda() for a in acts]
for t in range(30):
    env.step(dev_acts[t % 4], auto_reset=True)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for t in range(K):
    env.step(dev_acts[t % 4], auto_reset=True)
b.record(); torch.cuda.synchronize()
print("device-resident step at the same episode phase: %.3f ms/step" % (a.elapsed_time(b) / K))
for name, call, out in (("packed", env.step_host_packed, env.alloc_host_out(pinned=True, packed=True)),
                        ("ragged", env.step_host_ragged, env.alloc_host_out(pinned=True, ragged=True))):
    call(acts[0], auto_reset=True, out=out)
    env.stats(reset=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in range(K):
        call(acts[t % 4], auto_reset=True, out=out)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    s = env.stats(reset=True)
    print("%s: %.3f ms/step, %.3e agent-steps/s" % (name, dt / K * 1e3, s["agent_steps"] / dt))
    if name == "packed":
        t0 = time.perf_counter()
        rows, off = env.expand_obs_rows(out)
        t1 = time.perf_counter()
        env.expand_obs_rows(out, obs_rows=rows, row_offset=off)          # buffers of the first call reused: no page faults
        t2 = time.perf_counter()
        print("  expand_obs_rows on %d threads: %.1f ms for %d rows into fresh memory, %.1f ms into the same buffers again" % (
            len(os.sched_getaffinity(0)), (t1 - t0) * 1e3, rows.shape[0], (t2 - t1) * 1e3))

"""The evaluation protocol on the device (evaluation.evaluate_seeds) against the host one (evaluation.evaluation):
python profiles/time_eval_seeds.py [out.txt]

On the MASS td3 srew config of examples/mass_td3_srew.ini, with the MAPPO fused actor (a fixed ActorNetwork, seed fixed,
step = call count) as the action function:
  * mm_reset_seeded (seed copy + seeded spawn kernel + observation refresh) at 2^16 and 2^20 envs, CUDA events, median of
    10 after one warm-up call; and the spawn kernel alone from torch.profiler (a separate pass);
  * evaluate_seeds wall time (host clock around the call, which ends in a synchronise) at 2^16 and 2^20 seeds, after a
    warm-up evaluation at 2^16;
  * the record kernel's share of a policy step at 2^20 envs: T steps of (draw + mm_step) against T steps of (draw +
    mm_step + mm_eval_record), CUDA events, the two arms alternated three times;
  * evaluation() wall time at 1 024 and 4 096 seeds, and its linear extrapolation to 2^20 (labelled as such: it is not run
    there).
Writes the lines to out.txt (default profiles/r3_eval_seeds.txt) with the GPU name and power limit (nvidia-smi, read-only
query) read in the same run."""
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import marl_mass_b200 as mm  # noqa: E402
from marl_mass_b200 import _lib, evaluation as ev, rollout  # noqa: E402
from marl_mass_b200.train import load_ini  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_eval_seeds.txt")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()[0]
    return [x.strip() for x in out.split(",")]


class Actor(object):
    def __init__(self, net):
        self.net, self.calls = net, 0

    def __call__(self, obs, n_agents):
        self.calls += 1
        return rollout.actor_sample(self.net, obs, n_agents, seed=7919, step=self.calls)


def events_ms(fn, reps):
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return times


def main():
    name, power = gpu_info()
    lines = []

    def emit(rec):
        rec = dict(rec, gpu=name, power_limit=power)
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))

    env_cfg, _, _ = load_ini(os.path.join(ROOT, "examples", "mass_td3_srew.ini"))
    cfg = dict(mm.DEFAULT_CONFIG, **env_cfg)
    torch.manual_seed(0)
    net = rollout.ActorNetwork().cuda()
    td = cfg["traffic_density"]

    # seeded reset
    for E in (1 << 16, 1 << 20):
        env = mm.MergeEnvBatched(E, cfg)
        seeds = np.arange(E, dtype=np.int64)
        nc = ev.eval_num_cav(np.arange(E), td)
        env.reset_from_seeds_device(seeds, num_CAV=nc)
        torch.cuda.synchronize()
        t = events_ms(lambda: env.reset_from_seeds_device(seeds, num_CAV=nc), 10)
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                env.reset_from_seeds_device(seeds, num_CAV=nc)
            torch.cuda.synchronize()
        k = [e for e in prof.key_averages() if "seeded_reset_kernel" in e.key]
        kern = k[0].device_time_total / k[0].count / 1000.0 if k else float("nan")
        emit({"what": "mm_reset_seeded", "envs": E, "call_ms_median": statistics.median(t), "call_ms_min": min(t),
              "seeded_reset_kernel_ms": kern})
        env.close()

    # evaluate_seeds wall time
    ev.evaluate_seeds(Actor(net), cfg, np.arange(1 << 16))       # warm-up
    for N in (1 << 16, 1 << 20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = ev.evaluate_seeds(Actor(net), cfg, np.arange(N))
        wall = time.perf_counter() - t0
        lo, hi = r["crash_rate_ci95"]
        emit({"what": "evaluate_seeds", "seeds": N, "wall_s": wall, "crash_rate": r["crash_rate"], "crash_rate_ci95": [lo, hi],
              "mean_episode_reward": float(r["episode_reward"].mean()), "mean_steps": float(r["steps"].mean())})

    # the record kernel's share of a policy step at 2^20 envs
    E = 1 << 20
    env = mm.MergeEnvBatched(E, cfg)
    seeds = np.arange(E, dtype=np.int64)
    nc = ev.eval_num_cav(np.arange(E), td)
    dev = torch.device("cuda", 0)
    T = env.T

    def records():
        rec = {"active": torch.ones(E, dtype=torch.uint8, device=dev), "rewards": torch.zeros((E, T), device=dev),
               "steps": torch.zeros(E, dtype=torch.int32, device=dev),
               "avg_speed_sum": torch.zeros(E, dtype=torch.float64, device=dev),
               "traffic_speed_sum": torch.zeros(E, dtype=torch.float64, device=dev),
               "min_headway": torch.full((E,), float("inf"), device=dev), "merge_percent": torch.zeros(E, device=dev),
               "crashed": torch.zeros(E, dtype=torch.uint8, device=dev)}
        return rec

    def episode(with_record):
        env.reset_from_seeds_device(seeds, num_CAV=nc)
        n_agents = env.buffers()["n_agents"].clone()
        rec = records()
        st = _lib.MMEvalRecords(T=T, n_agents=n_agents.data_ptr(), **{k: v.data_ptr() for k, v in rec.items()})
        act = Actor(net)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for t in range(T):
            env.step(act(env.obs_view(), n_agents))
            if with_record:
                env.eval_record(st, t)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / T

    episode(True)
    arms = {False: [], True: []}
    for _ in range(3):
        for w in (False, True):
            arms[w].append(episode(w))
    base, withr = statistics.median(arms[False]), statistics.median(arms[True])
    emit({"what": "policy_step_2^20", "draw_plus_step_ms": base, "draw_plus_step_plus_record_ms": withr,
          "record_share": (withr - base) / withr, "runs_ms": {"without": arms[False], "with": arms[True]}})
    env.close()

    # the host protocol
    per_seed = []
    for N in (1024, 4096):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev.evaluation(Actor(net), cfg, list(range(N)))
        wall = time.perf_counter() - t0
        per_seed.append(wall / N)
        emit({"what": "evaluation", "seeds": N, "wall_s": wall})
    emit({"what": "evaluation_extrapolated_not_run", "seeds": 1 << 20, "wall_s_linear_from_4096": per_seed[-1] * (1 << 20)})
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

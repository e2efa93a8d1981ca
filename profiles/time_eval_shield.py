"""Cost of the evaluation's shield records (evaluate_seeds(shield_records=True), mm_eval_shield_record):
python profiles/time_eval_shield.py [out.txt]

On the MASS td3 srew config of examples/mass_td3_srew.ini, with the MAPPO fused actor (a fixed ActorNetwork, seed fixed,
step = call count) as the action function:
  * evaluate_seeds wall time (host clock around the call, which ends in a synchronise) at 2^16 and 2^20 seeds with
    shield_records off and on, the two arms alternated three times after one warm-up call of each;
  * eval_shield_record_kernel alone at 2^20 envs: CUDA events around 20 back-to-back launches on the record of one
    policy step (after a warm-up launch), median and minimum per launch, and the bytes it reads (8 of the 20 planes of
    the diagnostic record) over that time;
  * a policy step (draw + mm_step) at 2^20 envs on a handle with and without the diagnostic record, CUDA events over
    T steps, the two alternated three times: the price of record_diag itself.
Writes the lines to out.txt (default profiles/r3_eval_shield.txt) with the GPU name and power limit (nvidia-smi,
read-only query) read in the same run."""
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

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_eval_shield.txt")


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

    # evaluate_seeds wall time, records off / on
    for N in (1 << 16, 1 << 20):
        seeds = np.arange(N)
        for on in (False, True):
            ev.evaluate_seeds(Actor(net), cfg, seeds, shield_records=on)      # warm-up
        walls = {False: [], True: []}
        r = None
        for _ in range(3):
            for on in (False, True):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = ev.evaluate_seeds(Actor(net), cfg, seeds, shield_records=on) if on else \
                    ev.evaluate_seeds(Actor(net), cfg, seeds)
                walls[on].append(time.perf_counter() - t0)
        off, with_ = statistics.median(walls[False]), statistics.median(walls[True])
        emit({"what": "evaluate_seeds", "seeds": N, "wall_s_off": off, "wall_s_on": with_, "extra_share": (with_ - off) / off,
              "runs_s": {"off": walls[False], "on": walls[True]}, "crash_rate": r["crash_rate"],
              "intervention_rate": r["intervention_rate"], "mean_shield_solves": float(r["shield_solves"].mean()),
              "mean_lane_change_vetoes": float(r["lane_change_vetoes"].mean()),
              "min_agent_acc": float(r["min_agent_acc"].min()), "acc_correction_max": float(r["acc_correction_max"].max())})

    # the kernel alone at 2^20 envs
    E = 1 << 20
    dev = torch.device("cuda", 0)
    seeds = np.arange(E, dtype=np.int64)
    nc = ev.eval_num_cav(np.arange(E), td)
    env = mm.MergeEnvBatched(E, cfg, record_diag=True)
    T = env.T
    env.reset_from_seeds_device(seeds, num_CAV=nc)
    n_agents = env.buffers()["n_agents"].clone()
    act = Actor(net)
    env.step(act(env.obs_view(), n_agents))
    t = {k: torch.zeros(E, dtype=torch.int32, device=dev) for k in _lib.SHIELD_COUNTS}
    t.update({k: torch.zeros(E, dtype=torch.float64, device=dev) for k in _lib.SHIELD_F64})
    active = torch.ones(E, dtype=torch.uint8, device=dev)
    rec = _lib.MMEvalShieldRecords(T=T, n_agents=n_agents.data_ptr(), active=active.data_ptr(),
                                   **{k: v.data_ptr() for k, v in t.items()})
    env.eval_shield_record(rec, 0)
    torch.cuda.synchronize()
    per = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            env.eval_shield_record(rec, 0)
        b.record()
        torch.cuda.synchronize()
        per.append(a.elapsed_time(b) / 20)
    read_bytes = E * 3 * _lib.MAXV * (4 * 4 + 4 * 8) + E * (1 + 4 + 4 * 4 + 4 * 8)
    emit({"what": "eval_shield_record_kernel", "envs": E, "launch_ms_median": statistics.median(per),
          "launch_ms_min": min(per), "runs_ms": per, "bytes_read": read_bytes,
          "read_GBps_at_median": read_bytes / (statistics.median(per) * 1e-3) / 1e9})

    # the price of the diagnostic record itself: a policy step on handles with and without it
    plain = mm.MergeEnvBatched(E, cfg)

    def steps(h):
        h.reset_from_seeds_device(seeds, num_CAV=nc)
        na = h.buffers()["n_agents"].clone()
        ac = Actor(net)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(T):
            h.step(ac(h.obs_view(), na))
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / T

    steps(plain)
    steps(env)
    arms = {"plain": [], "record_diag": []}
    for _ in range(3):
        arms["plain"].append(steps(plain))
        arms["record_diag"].append(steps(env))
    emit({"what": "policy_step_2^20", "draw_plus_step_ms": statistics.median(arms["plain"]),
          "draw_plus_step_record_diag_ms": statistics.median(arms["record_diag"]), "runs_ms": arms})
    env.close()
    plain.close()
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

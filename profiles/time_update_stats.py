"""What update(stats=True) costs: python profiles/time_update_stats.py [out] [envs] [repeats]
(out defaults to profiles/r3_update_stats.txt).

Per example ini (mass_td3_srew, mass_td3_mixed_srew_shared): one 100-step collect() at 4096 envs, then four arms
alternately from the same saved networks / optimiser state (warm-up first, the device synchronised around every timed
call): update(impl) with stats off and on, for impl "torch" and "cuda", minibatch 2^18.  Also the statistics passes alone
(rollout.ppo_stats over every live row for the policy and the value network, what one update(impl="cuda", stats=True)
runs twice) with CUDA events.  Writes one JSON line per ini with the GPU name and power limit (nvidia-smi, read-only
query) read in the same run."""
import copy
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import marl_mass_b200 as mm  # noqa: E402
from marl_mass_b200 import rollout  # noqa: E402
from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout  # noqa: E402
from marl_mass_b200.train import load_ini  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_update_stats.txt")
E = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
REPEATS = int(sys.argv[3]) if len(sys.argv) > 3 else 10
MB = 1 << 18


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def run(ini):
    env_cfg, kw, tr = load_ini(os.path.join(ROOT, "examples", ini))
    env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, **env_cfg), device=0)
    obs0, _ = env.reset(seed=env_cfg["seed"])
    torch.manual_seed(0)
    shared = tr["shared_network"]
    pol = (BatchedMAPPOGIRollout if shared else BatchedMAPPORollout)(env, obs=obs0, **kw)
    pol.collect()
    torch.cuda.synchronize()
    opts = [pol.policy_opt] if shared else [pol.actor_opt, pol.critic_opt]
    sd_m = [copy.deepcopy(m.state_dict()) for m in pol.networks()]
    sd_o = [copy.deepcopy(o.state_dict()) for o in opts]
    arms = [(impl, stats) for impl in ("torch", "cuda") for stats in (False, True)]

    def timed_update(impl, stats):
        for m, sd in zip(pol.networks(), sd_m):
            m.load_state_dict(sd)
        for o, sd in zip(opts, sd_o):
            o.load_state_dict(copy.deepcopy(sd))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pol.update(minibatch=MB, impl=impl, stats=stats)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    times = {a: [] for a in arms}
    for a in arms:
        timed_update(*a)                          # warm-up
    for _ in range(REPEATS):
        for a in arms:
            times[a].append(timed_update(*a))

    idx, S, A8, G = pol._learner_batch()
    nets = [pol.policy] if shared else [pol.actor, pol.critic]
    old = rollout.ppo_targets(pol.policy_target if shared else pol.actor_target, S, A8, idx)

    def stats_pass():
        for net in nets:
            rollout.ppo_stats(net, S, A8, G, idx, None if net is getattr(pol, "critic", None) else old, pol.clip_param)

    for _ in range(3):
        stats_pass()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(20):
        stats_pass()
    e.record()
    torch.cuda.synchronize()
    name, power = gpu_info()
    med = {"%s_stats_%s" % (i, "on" if s else "off"): statistics.median(times[(i, s)]) for i, s in arms}
    rec = {"ini": ini, "gpu": name, "power_limit": power, "envs": E, "rollout_steps": pol.T, "samples": int(idx.numel()),
           "minibatch": MB, "repeats": REPEATS, "update_s_median": med,
           "update_s": {"%s_stats_%s" % (i, "on" if s else "off"): times[(i, s)] for i, s in arms},
           "stats_cost_s": {i: med[i + "_stats_on"] - med[i + "_stats_off"] for i in ("torch", "cuda")},
           "stats_pass_ms": a.elapsed_time(e) / 20}
    env.close()
    return rec


if __name__ == "__main__":
    lines = [json.dumps(run(ini)) for ini in ("mass_td3_srew.ini", "mass_td3_mixed_srew_shared.ini")]
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))

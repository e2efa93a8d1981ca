"""PPO update time, torch autograd against the learner kernels, on the workload of the recorded training logs:
python profiles/time_update.py [envs] [repeats]
python profiles/time_update.py [envs] launches

Per example ini (mass_td3_srew, mass_td3_mixed_srew_shared): one 100-step collect() at 4096 envs, then three arms
alternately from the same saved networks / optimiser state (warm-up first, the device synchronised around every timed
call): update(impl="torch"), update(impl="cuda") with the torch optimiser, and update(impl="cuda") with the device
optimiser (optimizer="cuda": clip_grad_norm_ + RMSprop in one launch per minibatch); and the gradient pass alone per
2^18-row minibatch with CUDA events.  Prints one JSON line per ini with the GPU name and power limit (nvidia-smi,
read-only query).  With "launches" instead of a repeat count: one update per arm under torch.profiler (a separate run:
tracing slows the host), and the device activities (kernels, memsets, copies) per update and per minibatch."""
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

E = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
LAUNCHES = len(sys.argv) > 2 and sys.argv[2] == "launches"
REPEATS = int(sys.argv[2]) if len(sys.argv) > 2 and not LAUNCHES else 10
MB = 1 << 18


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def run(ini):
    env_cfg, kw, tr = load_ini(os.path.join(ROOT, "examples", ini))
    env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, **env_cfg), device=0)
    obs0, _ = env.reset(seed=env_cfg["seed"])
    torch.manual_seed(0)
    shared = tr["shared_network"]
    cls = BatchedMAPPOGIRollout if shared else BatchedMAPPORollout
    pol = cls(env, obs=obs0, **kw)
    pol.collect()
    torch.cuda.synchronize()
    nets = {"policy": copy.deepcopy(pol.policy)} if shared else {"actor": copy.deepcopy(pol.actor),
                                                                  "critic": copy.deepcopy(pol.critic)}
    pol_dev = cls(env, obs=obs0, optimizer="cuda", **nets, **kw)     # the same networks, the device optimiser
    pol_dev.buf = pol.buf
    arms = {"torch": (pol, "torch"), "cuda": (pol, "cuda"), "cuda_devopt": (pol_dev, "cuda")}
    saved = {}
    for p in (pol, pol_dev):
        opts = [p.policy_opt] if shared else [p.actor_opt, p.critic_opt]
        saved[id(p)] = (p.networks(), opts, [copy.deepcopy(m.state_dict()) for m in pol.networks()],
                        [copy.deepcopy(o.state_dict()) for o in opts])

    def timed_update(arm):
        p, impl = arms[arm]
        mods, opts, sd_m, sd_o = saved[id(p)]
        for m, sd in zip(mods, sd_m):
            m.load_state_dict(sd)
        for o, sd in zip(opts, sd_o):
            o.load_state_dict(copy.deepcopy(sd))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st = p.update(minibatch=MB, impl=impl)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, st

    n_mb = -(-int(pol.buf["live"].sum()) // MB)
    if LAUNCHES:
        from torch.profiler import ProfilerActivity, profile
        counts = {}
        for arm in arms:
            timed_update(arm)                    # warm-up
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                timed_update(arm)
            n = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
            counts[arm] = {"device_activities": n, "per_minibatch": n / n_mb}
        name, power = gpu_info()
        print(json.dumps({"ini": ini, "gpu": name, "power_limit": power, "minibatches": n_mb, "launches": counts}), flush=True)
        env.close()
        return

    times = {arm: [] for arm in arms}
    for arm in arms:
        timed_update(arm)                        # warm-up
    for _ in range(REPEATS):
        for arm in arms:
            times[arm].append(timed_update(arm)[0])

    # the gradient pass alone, per 2^18-row minibatch
    b = pol.buf
    idx = b["live"].reshape(-1).nonzero().squeeze(1)
    S = b["states"].reshape(-1, mm.NS)
    A8 = b["actions"].reshape(-1).to(torch.int8)
    G = b["returns"].reshape(-1).contiguous()
    j = idx[torch.randperm(idx.numel(), device="cuda")[:MB]]
    if shared:
        old = rollout.ppo_targets(pol.policy_target, S, A8, idx)
        grad_pass = lambda: rollout.shared_network_gradients(pol.policy, S, A8, G, old, j, pol.clip_param)  # noqa: E731
        target_pass = lambda: rollout.ppo_targets(pol.policy_target, S, A8, idx, out=old)  # noqa: E731
    else:
        old = rollout.ppo_targets(pol.actor_target, S, A8, idx)
        q = rollout.ppo_targets(pol.critic_target, S, A8, idx)
        grad_pass = lambda: rollout.mappo_gradients(pol.actor, pol.critic, S, A8, G, old, q, j, pol.clip_param)  # noqa: E731
        target_pass = lambda: (rollout.ppo_targets(pol.actor_target, S, A8, idx, out=old),  # noqa: E731
                               rollout.ppo_targets(pol.critic_target, S, A8, idx, out=q))

    def events(fn, n=20):
        for _ in range(3):
            fn()
        a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(n):
            fn()
        e.record()
        torch.cuda.synchronize()
        return a.elapsed_time(e) / n

    name, power = gpu_info()
    rec = {"ini": ini, "gpu": name, "power_limit": power, "envs": E, "rollout_steps": pol.T, "samples": int(idx.numel()),
           "minibatch": MB, "minibatches": n_mb, "repeats": REPEATS,
           "update_torch_s_median": statistics.median(times["torch"]), "update_cuda_s_median": statistics.median(times["cuda"]),
           "update_cuda_devopt_s_median": statistics.median(times["cuda_devopt"]),
           "update_torch_s": times["torch"], "update_cuda_s": times["cuda"], "update_cuda_devopt_s": times["cuda_devopt"],
           "speedup": statistics.median(times["torch"]) / statistics.median(times["cuda"]),
           "speedup_devopt": statistics.median(times["torch"]) / statistics.median(times["cuda_devopt"]),
           "grad_pass_ms_per_minibatch": events(grad_pass), "target_pass_ms": events(target_pass, 5)}
    env.close()
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    for ini in ("mass_td3_srew.ini", "mass_td3_mixed_srew_shared.ini"):
        run(ini)

"""What GAE(lambda) returns cost: python profiles/time_lambda_returns.py [out] [repeats] [kernel]
(out defaults to profiles/r3_lambda_returns.txt).

- Kernel: mm_lambda_returns (lambda 0.95, with values) against mm_discounted_returns (the same kernel without values) on
  random rollouts of 4 096 and 65 536 envs x 100 steps x 12 slots, CUDA events over 50 launches after warm-up.  Bytes
  per element: rewards, values and the output in f32 plus a twelfth of a done byte (8.08 B without values).  At 4 096
  envs the working set (20-40 MB) stays in L2 between launches; at 65 536 (315-630 MB) it does not.
- Update: per example ini (mass_td3_srew: MAPPO, mass_td3_mixed_srew_shared: MAPPO_GI), one 100-step collect() at 4 096
  envs, then update(impl) with gae_lambda None and 0.95 for impl "torch" and "cuda" (torch optimiser, minibatch 2^18),
  the four arms alternated from the same saved networks and optimiser state, the device synchronised around every timed
  call, warm-up first; median of `repeats`.
With `kernel` only the kernel lines are measured.  One JSON line per measurement, with the GPU name and power limit (nvidia-smi, read-only query) read in the same run.

    python profiles/time_lambda_returns.py launches ROOT
counts the device activities (torch.profiler: kernels, memsets, copies) of one collect() and one update() per ini and
impl with gae_lambda unset, importing the package under ROOT: run it on two trees to compare their launches."""
import copy
import json
import os
import statistics
import subprocess
import sys
import time

LAUNCHES = len(sys.argv) > 1 and sys.argv[1] == "launches"
ROOT = sys.argv[2] if LAUNCHES else os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import marl_mass_b200 as mm  # noqa: E402
from marl_mass_b200 import rollout  # noqa: E402
from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout  # noqa: E402
from marl_mass_b200.train import load_ini  # noqa: E402

OUT = None if LAUNCHES else (sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_lambda_returns.txt"))
REPEATS = int(sys.argv[2]) if len(sys.argv) > 2 and not LAUNCHES else 10
E_UPDATE, MB, T = 4096, 1 << 18, 100
INIS = ("mass_td3_srew.ini", "mass_td3_mixed_srew_shared.ini")


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()[0]
    return [x.strip() for x in out.split(",")]


def kernel(E, launches=50):
    g = torch.Generator(device="cuda").manual_seed(E)
    R = torch.randn((T, E, 12), device="cuda", generator=g)
    V = torch.randn((T, E, 12), device="cuda", generator=g)
    D = (torch.rand((T, E), device="cuda", generator=g) < 0.01).float()
    fv = torch.randn((E, 12), device="cuda", generator=g)
    arms = {"discounted": lambda: rollout.discounted_returns(R, D, fv, 0.99),
            "lambda_0.95": lambda: rollout.lambda_returns(R, D, V, fv, 0.99, 0.95)}
    rec = {"envs": E, "steps": T, "elements": T * E * 12}
    for name, fn in arms.items():
        for _ in range(5):
            fn()
        # the python wrappers' own device work (dones -> u8, output allocation) is timed with the kernel
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(launches):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / launches
        per_elem = 12 + 1 / 12 if name != "discounted" else 8 + 1 / 12
        rec[name + "_ms"] = ms
        rec[name + "_GBps"] = T * E * 12 * per_elem / (ms * 1e-3) / 1e9
    # the kernel alone, from the profiler (the wrappers also convert dones and allocate)
    from torch.profiler import ProfilerActivity, profile
    for name, fn in arms.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                fn()
            torch.cuda.synchronize()
        ks = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "discounted_returns_kernel" in e.name]
        rec[name + "_kernel_us"] = sum(e.device_time for e in ks) / max(len(ks), 1)
    return rec


def learner(ini, E, **kw):
    env_cfg, rkw, tr = load_ini(os.path.join(ROOT, "examples", ini))
    env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, **env_cfg), device=0)
    obs0, _ = env.reset(seed=env_cfg["seed"])
    torch.manual_seed(0)
    pol = (BatchedMAPPOGIRollout if tr["shared_network"] else BatchedMAPPORollout)(env, obs=obs0, **rkw, **kw)
    return env, pol, tr["shared_network"]


def update_timing(ini):
    env, pol, shared = learner(ini, E_UPDATE)
    pol.collect()
    torch.cuda.synchronize()
    opts = [pol.policy_opt] if shared else [pol.actor_opt, pol.critic_opt]
    sd_m = [copy.deepcopy(m.state_dict()) for m in pol.networks()]
    sd_o = [copy.deepcopy(o.state_dict()) for o in opts]
    arms = [(impl, lam) for impl in ("torch", "cuda") for lam in (None, 0.95)]

    def timed(impl, lam):
        for m, sd in zip(pol.networks(), sd_m):
            m.load_state_dict(sd)
        for o, sd in zip(opts, sd_o):
            o.load_state_dict(copy.deepcopy(sd))
        pol.gae_lambda = lam
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pol.update(minibatch=MB, impl=impl)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    times = {a: [] for a in arms}
    for a in arms:
        timed(*a)
    for _ in range(REPEATS):
        for a in arms:
            times[a].append(timed(*a))
    name = lambda a: "%s_gae_%s" % (a[0], "none" if a[1] is None else a[1])  # noqa: E731
    samples = int(pol.buf["live"].sum())
    env.close()
    return {"ini": ini, "envs": E_UPDATE, "rollout_steps": T, "samples": samples, "minibatch": MB, "repeats": REPEATS,
            "update_s_median": {name(a): statistics.median(times[a]) for a in arms},
            "update_s": {name(a): times[a] for a in arms}}


def launches():
    from collections import Counter
    from torch.profiler import ProfilerActivity, profile
    out = {"root": ROOT}
    for ini in INIS:
        for impl in ("torch", "cuda"):
            env, pol, _ = learner(ini, 1024)
            pol.collect()
            pol.update(minibatch=1 << 16, impl=impl)      # one-time initialisation outside the count
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                pol.collect()
                torch.cuda.synchronize()
                torch.manual_seed(1)
                pol.update(minibatch=1 << 16, impl=impl)
                torch.cuda.synchronize()
            names = Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
            out["%s_%s" % (ini, impl)] = {"device_activities": sum(names.values()), "distinct": len(names),
                                           "returns_kernel": sum(v for k, v in names.items() if "discounted_returns" in k)}
            env.close()
    return out


if __name__ == "__main__":
    if LAUNCHES:
        print(json.dumps(launches()))
        sys.exit(0)
    gpu, power = gpu_info()
    kernels_only = len(sys.argv) > 3 and sys.argv[3] == "kernel"
    lines = [dict(kernel(E), what="kernel") for E in (4096, 65536)]
    lines += [] if kernels_only else [dict(update_timing(ini), what="update") for ini in INIS]
    lines = [json.dumps(dict(rec, gpu=gpu, power_limit=power)) for rec in lines]
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))

#!/usr/bin/env python
"""bench.py — shielded agent-steps/s of the batched merge env + CBF shield on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--envs E] [--impl reference] [--dump-outputs DIR]

A "step" is one policy step (3 physics sub-steps, 3 shield solves per CAV, observation, rewards) of every env of
the workload, with finished envs re-spawned on the device (auto-reset), under i.i.d. uniform meta-actions.
Prints ONE JSON line (rank 0).  Keys: see the task contract; in short
  value      whole-job agent-steps/s with actions already resident in HBM (CUDA events, max over ranks)
  e2e        same metric through the host-buffer C-ABI call mm_step_host (pinned host actions in, obs/reward/
             done/regional rewards out every step, copies inside the timed region)
  roofline   step kernel alone: algorithmic bytes/launch / mean launch time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle (C float64 port of the reference path) on this box's host cores, bounded sample
`--impl reference` times that CPU port as the reference arm (the Python reference cannot travel to the GPU box;
its in-container throughput is recorded in BASELINE.md / DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

MASS = dict(safety_guarantee="cbf-cav", HEADWAY_TIME=0.5, cbf_eta=0.03125)
WORKLOADS = {
    # BASELINE.json configs[4] scenario (the one the 1/2/4/8-GPU metric and the 1e8 target are quoted on):
    # MASS shield, hard density (td3), all-CAV (7-11 CAVs per env); one 2^20-env shard per GPU.
    "mass_td3": dict(cfg=dict(MASS, traffic_density=3, traffic_type="cav"), envs=1 << 20,
                     desc="MASS cbf-cav hard-density merge (BASELINE configs[4]: marl_cav-heading-t_headway-cbf-cav, "
                          "traffic_density=3, all-CAV 7-11 agents/env)"),
    # opt-in device-spawn variant: vehicle counts drawn per 128-env tile (include/marl_mass_b200.h couple_counts);
    # NOT the default workload - reported separately (profiles/README.md)
    "mass_td3_coupled": dict(cfg=dict(MASS, traffic_density=3, traffic_type="cav", couple_vehicle_counts=True), envs=1 << 20,
                             desc="MASS cbf-cav hard density, all-CAV, vehicle counts coupled per 128-env tile (opt-in spawn "
                                  "variant: every env keeps the reference's law, envs of a tile share n_CAV)"),
    "mass_td3_mixed": dict(cfg=dict(MASS, traffic_density=3, traffic_type="mixed"), envs=1 << 20,
                           desc="MASS cbf-cav-mixed hard density (4-6 CAV + 3-5 IDM/MOBIL HDV per env)"),
    "mass_td3_srew": dict(cfg=dict(MASS, traffic_density=3, traffic_type="cav", agent_reward="srew",
                                   HIGH_SPEED_REWARD=4, HEADWAY_COST=1, MERGING_LANE_COST=8), envs=65536,
                          desc="MASS td3 srew (BASELINE configs[3] env side), 65536 envs"),
    "mass_td1": dict(cfg=dict(MASS, traffic_density=1, traffic_type="cav"), envs=65536,
                     desc="MASS cbf-cav td1 (BASELINE configs[2]), 65536 envs"),
    "hss_td3": dict(cfg=dict(safety_guarantee="cbf-avs_cint", HEADWAY_TIME=0.5, cbf_eta=0.03125, traffic_density=3,
                             traffic_type="cav"), envs=4096,
                    desc="HSS cbf-avs_cint td3 (BASELINE configs[1]), 4096 envs"),
    "unsafe_td1": dict(cfg=dict(safety_guarantee="none", HEADWAY_TIME=1.2, traffic_density=1, traffic_type="cav"),
                       envs=65536, desc="no shield, td1 (BASELINE configs[0] LC-env sibling)"),
    "dmc_v0_td3": dict(cfg=dict(env_name="merge-multi-agent-v0", safety_guarantee="dmc", HEADWAY_TIME=1.2, traffic_density=3,
                                mixed_traffic=True), envs=65536,
                       desc="baseline supervisor dmc, env merge-multi-agent-v0, td3 mixed (marl_cav-heading-t_headway-dmc-mixed.ini)"),
    "priority_v0_td3": dict(cfg=dict(env_name="merge-multi-agent-v0", safety_guarantee="priority", HEADWAY_TIME=1.2, traffic_density=3,
                                     mixed_traffic=True), envs=65536,
                            desc="baseline supervisor priority, env merge-multi-agent-v0, td3 mixed (marl_cav-heading-t_headway-priority-mixed.ini)"),
    "unsafe_v0_td1": dict(cfg=dict(env_name="merge-multi-agent-v0", safety_guarantee="none", HEADWAY_TIME=1.2, traffic_density=1,
                                   mixed_traffic=True), envs=65536,
                          desc="no shield, env merge-multi-agent-v0, td1 mixed (BASELINE configs[0]: test-configs_marl-cav-unsafe.ini)"),
}

# DESIGN.md "Algorithmic bytes": per vehicle 84 B state read + 124 B state written, per agent 120 B obs + 8 B
# rewards + 1 B done + 1 B action, per env 33 B of scalars
BYTES_PER_VEHICLE = 84 + 124
BYTES_PER_AGENT = 120 + 8 + 1 + 1
BYTES_PER_ENV = 33


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for row in self.samples:
            if len(row) < 6:
                continue
            try:
                sm.append(float(row[0]))
                mx = float(row[1])
            except ValueError:
                continue
            for n, v in zip(names, row[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def static_config(wl, E, world, scaling="weak"):
    """The `config` object of the JSON line: the workload only, nothing measured - identical for the GPU arm and for
    `--impl reference` (the CPU arm times a bounded sample of exactly this workload; see cpu_baseline.sample)."""
    return {"workload": wl["desc"], "envs_per_gpu": E, "envs_total": E * world if scaling == "weak" else E * world,
            "actions": "i.i.d. uniform{0..4}", "auto_reset": True,
            "episode_phases": "staggered uniformly over the 100-step episode, per 128-env tile (untimed prologue)",
            "l2": "working set %.1f GB per GPU >> 126 MB L2 (no flush needed)" % (E * 3.0e-6)
                  if E >= 262144 else "inputs cycle through 8 action slabs; state working set %.0f MB" % (E * 3.0e-3)}


def cpu_port_throughput(cfg, budget_s, sample_envs, warmup_steps=1, fixed_steps=None, pool_scenes=1024):
    """Time the CPU port of the reference path (the C float64 restatement under oracle/) with all host threads on a
    bounded SAMPLE of the workload: `sample_envs` envs under the same action law, auto-reset, and - like the GPU arm -
    with the episode phases staggered uniformly per 128-env tile by an untimed prologue, so that every timed step is the
    average over all phases of an episode.  Scenes come from the host seed-exact spawn (a pool of `pool_scenes` scenes)."""
    import oracle
    import marl_mass_b200.spawn as spawn
    from marl_mass_b200 import DEFAULT_CONFIG
    full = dict(DEFAULT_CONFIG, **cfg)
    cores = host_cores()
    ocfg = oracle.make_config(full)
    E = sample_envs
    T = int(full["duration"] * full["policy_frequency"])
    from marl_mass_b200.env import traffic_type_of
    base = spawn.spawn_state(range(pool_scenes), full["traffic_density"], traffic_type_of(full))
    reps = E // pool_scenes + 1
    fresh = {k: np.ascontiguousarray(np.tile(v, (reps,) + (1,) * (v.ndim - 1))[:E]) for k, v in base.items()}
    st = {k: v.copy() for k, v in fresh.items()}
    rng = np.random.RandomState(0)
    out = oracle.empty_out(E)
    phase = (np.arange(E) // 128) % T

    def step(timed):
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        n_live = int(st["n_cav"].sum() if not full.get("env_name", "").endswith("hdv-v1") else st["n_veh"].sum())
        t0 = time.perf_counter()
        oracle.step(ocfg, st, a, out=out, n_threads=cores)
        dt = time.perf_counter() - t0
        return n_live, dt, out["done"] != 0

    def respawn(mask):   # host-side re-spawn (untimed, like the reference's env.reset between episodes)
        if mask.any():
            for k in st:
                st[k][mask] = fresh[k][mask]

    for j in range(T):                       # prologue: env tiles re-spawn at step (tile % T), as in the GPU arm
        _, _, done = step(False)
        respawn(done | (phase == j))
    agent_steps, t_total, n = 0, 0.0, 0
    per_step = []
    while True:
        n_live, dt, done = step(True)
        respawn(done)
        n += 1
        if n > warmup_steps:
            agent_steps += n_live
            t_total += dt
            per_step.append(dt)
        if fixed_steps is not None:
            if n >= warmup_steps + fixed_steps:
                break
        elif t_total >= budget_s:
            break
    return agent_steps / t_total, cores, len(per_step), E, float(np.mean(per_step)) * 1e3


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    sample = min(wl["envs"], 16384)
    v, cores, n_steps, E, ms = cpu_port_throughput(wl["cfg"], None, sample, warmup_steps=args.warmup,
                                                   fixed_steps=args.steps)
    line = {
        "impl": "reference", "metric": "shielded agent-steps/s", "value": v, "unit": "agent-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config(wl, wl["envs"], world),
        "cpu_baseline": {"value": v, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                         "sample": "%d of the workload's envs (same action law, auto-reset, episode phases staggered per "
                                   "128-env tile by an untimed %d-step prologue) x %d timed policy steps; ms_per_step is "
                                   "per sample step" % (E, 100, n_steps),
                         "note": "C float64 port of the reference env + shield (oracle/), all host threads; the Python "
                                 "reference cannot travel to the GPU box (BASELINE.md: ~94 agent-steps/s per core here)"},
        "e2e": {"value": v, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_JSON_FD = None


def claim_stdout():
    """Keep stdout to the ONE JSON line: everything any library prints to fd 1 from here on (NCCL's version banner,
    torchrun notices, ...) goes to stderr; `emit` writes the line to the real stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def load_traffic(workload, envs):
    """DRAM bytes per launch of the dominant kernel from THIS round's `ncu --set full` capture
    (profiles/r2_traffic.json, written by profiles/traffic_from_ncu.py), used only when it was taken on exactly this
    workload and batch - never scaled; otherwise null."""
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        for rec in tj["captures"]:
            if rec["workload"] == workload and int(rec["envs"]) == int(envs):
                return float(rec["dram_bytes"]), rec
    except Exception:
        pass
    return None, None


class Leg(object):
    """One batched env on this rank with its action pool, episode phases staggered (untimed prologue)."""

    def __init__(self, mm, mmd, name, E, dev, rank, policy=False):
        import torch
        self.torch, self.mm, self.mmd, self.rank = torch, mm, mmd, rank
        self.wl = dict(WORKLOADS[name])
        self.E = E
        self.cfg = dict(mm.DEFAULT_CONFIG, **self.wl["cfg"])
        self.env = mm.MergeEnvBatched(E, self.cfg, device=dev, record_diag=False)
        self.env.reset(seed=mmd.rank_seed(1, rank))
        gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
        # action pool resident in HBM (i.i.d. uniform{0..4}); cycled so every step reads a different slab
        self.pool = [torch.randint(0, 5, (E, mm.MAXV), generator=gen, device="cuda", dtype=torch.int8) for _ in range(8)]
        # Prologue (untimed): stagger the episode phases.  All envs are spawned together, so without this every env would
        # hit the 100-step horizon on the same step; re-spawning the envs of tile k at prologue step (k % T) spreads the
        # phases uniformly, which is the steady state of a long rollout (1/T of the envs re-spawn per timed step).  By
        # 128-env tile, not by env: in a real rollout the envs of a batch start together and only the rare crash
        # de-synchronises one, so neighbouring envs share their episode phase.
        T = int(self.cfg["duration"] * self.cfg["policy_frequency"])
        idx = (torch.arange(E, device="cuda", dtype=torch.int32) // 128) % T
        for j in range(T):
            self.env.step(self.pool[j % 8], auto_reset=True)
            self.env.reset(seed=mmd.rank_seed(3 + j, rank), mask=(idx == j).to(torch.uint8))
        self.policy = None
        if policy:
            from marl_mass_b200.rollout import BatchedMAPPORollout
            torch.manual_seed(rank)
            self.policy = BatchedMAPPORollout(self.env, roll_out_n_steps=1)
            self.vbuf = self.env.buffers()

    def step(self, t):
        if self.policy is None:
            self.env.step(self.pool[t % 8], auto_reset=True)
        else:
            self.env.step(self.policy._act(self.vbuf["obs"], self.vbuf["n_agents"])[0], auto_reset=True)

    def timed(self, K, W, barrier):
        """W untimed + K timed steps bracketed by barrier(); returns (ms_total, stats of the timed steps, launches)."""
        torch = self.torch
        for t in range(W):
            self.step(t)
        barrier()
        self.env.stats(reset=True)
        l0 = self.env.kernel_launches()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for t in range(K):
            self.step(t)
        ev1.record()
        barrier()
        return ev0.elapsed_time(ev1), self.env.stats(reset=True), self.env.kernel_launches() - l0

    def kernel_times(self, n):
        """Device time of the physics kernel + outputs kernel alone, one event pair per policy step (re-spawn outside)."""
        torch = self.torch
        v = self.env.buffers()
        ms, agents = [], 0.0
        for t in range(n):
            n_ag = float(v["n_agents"].sum())
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            self.env.step(self.pool[t % 8], auto_reset=False)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
            agents += n_ag
            self.env.reset(seed=self.mmd.rank_seed(2, self.rank), mask=v["done"])
        torch.cuda.synchronize()
        return float(np.mean(ms)), agents / max(n, 1)

    def algorithmic_bytes(self, mean_agents):
        cfg = self.cfg
        mean_hdv = 0.0 if cfg["traffic_type"] == "cav" else {1: 2.0, 2: 3.0, 3: 4.0}[int(cfg["traffic_density"])]
        return self.E * ((mean_agents + mean_hdv) * BYTES_PER_VEHICLE + mean_agents * BYTES_PER_AGENT + BYTES_PER_ENV)

    def close(self):
        self.env.close()


# What env.step hands its caller (obs, reward, done and the info views), minus the actions it was given.
DUMP_KEYS = ("obs", "reward", "done", "agents_rewards", "regional_rewards", "agents_dones", "average_speed", "traffic_speed",
             "min_headway", "merge_percent", "n_agents", "action_mask", "new_actions")
DUMP_BYTES = 64 * 10 ** 6      # all files of one dump together, .npy headers included
NPY_HEADER_BYTES = 128         # numpy writes a 128-byte header for arrays of these ranks


def dump_sample_size(env):
    """How many envs a dump keeps: all of them, or as many as fit in DUMP_BYTES at float32 per output value plus the
    float64 env index."""
    v = env.buffers()
    per_env = 8 + sum(4 * (v[k].numel() // env.n_envs) for k in DUMP_KEYS)
    return min(env.n_envs, (DUMP_BYTES - NPY_HEADER_BYTES * (len(DUMP_KEYS) + 1)) // per_env)


def dump_outputs(env, out_dir):
    """Write the outputs of env's last step as out_dir/<key>.npy (float32) for the envs listed in out_dir/env_index.npy
    (float64): every env when they fit in DUMP_BYTES, else a sample drawn with a fixed seed."""
    import torch
    E, n = env.n_envs, dump_sample_size(env)
    idx = np.arange(E) if n == E else np.sort(np.random.RandomState(0).choice(E, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    sel = torch.from_numpy(idx).to("cuda:%d" % env.device)
    v = env.buffers()
    for k in DUMP_KEYS:
        np.save(os.path.join(out_dir, k + ".npy"), v[k].index_select(0, sel).cpu().numpy().astype(np.float32))


BUILD_NAMES = {3: "generic, 3 CTAs/SM", 4: "generic, 4 CTAs/SM", 31: "all-CAV HSS specialised, 3 CTAs/SM",
               32: "all-CAV MASS specialised, 3 CTAs/SM", 41: "all-CAV HSS specialised, 4 CTAs/SM",
               42: "all-CAV MASS specialised, 4 CTAs/SM", 50: "warp-cooperative, no shield", 51: "warp-cooperative, HSS",
               52: "warp-cooperative, MASS"}


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mass_td3", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's envs on EVERY GPU (default); strong: the workload's envs split over the GPUs")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer pass (default min(steps, 20))")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-extra", action="store_true", help="only the headline leg: no strong-scaling / other-workload legs")
    ap.add_argument("--policy", action="store_true",
                    help="BASELINE configs[3]: sample the actions from the MAPPO actor (30-128-128-5) on the device "
                         "inside the timed region instead of reading pre-drawn uniform actions")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0's envs, a "
                         "seeded sample of them when all would exceed %d MB): the same arguments give the same inputs on "
                         "every run, so two builds can be compared output for output" % (DUMP_BYTES // 10 ** 6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    wl = dict(WORKLOADS[args.workload])
    if args.envs:
        wl["envs"] = args.envs
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    import torch
    import torch.distributed as dist
    import marl_mass_b200 as mm
    from marl_mass_b200 import dist as mmd

    rank, world, local_rank = mmd.rank_world()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if "MM_NCCL_DEBUG" in os.environ:
            os.environ["NCCL_DEBUG"] = os.environ["MM_NCCL_DEBUG"]
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    numa_cores = mmd.bind_to_gpu(dev) if world > 1 else 0   # host buffers on the GPU's own NUMA node
    K, W = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def fold(ms, stats):
        """max over ranks of the time, sum over ranks of the work"""
        tot = mmd.all_reduce_stats(stats)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms, tot

    E_total = wl["envs"]
    E = E_total if args.scaling == "weak" else max(128, (E_total // world) // 128 * 128)
    sampler = ClockSampler(dev)
    leg = Leg(mm, mmd, args.workload, E, dev, rank, policy=args.policy)
    env = leg.env
    sampler.start()
    ms_local, stats, launches = leg.timed(K, W, barrier)
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs)
    build = env.step_build()
    kms, _ = leg.kernel_times(min(K, 30))
    clocks = sampler.stop()
    ms_total, tot = fold(ms_local, stats)
    value = tot["agent_steps"] / (ms_total * 1e-3)
    mean_agents = stats["agent_steps"] / max(stats["env_steps"], 1.0)

    # CBF-QP alone (the metric's "CBF-QP solves/s"): 2^26 synthetic solves, ~10 % of rows active (SURVEY.md 8d)
    nq = 1 << 26
    g2 = torch.Generator(device="cuda").manual_seed(7)
    dtq = 1.0 / 15
    qa = dtq * torch.cos(torch.rand(nq, generator=g2, device="cuda", dtype=torch.float64) * 0.6 - 0.3)
    qcl = torch.randn(nq, generator=g2, device="cuda", dtype=torch.float64) * 3 + 2
    qca = torch.randn(nq, generator=g2, device="cuda", dtype=torch.float64) * 3 + 2
    qha = (torch.rand(nq, generator=g2, device="cuda") < 0.3).to(torch.uint8)
    qlo = torch.full((nq,), -12.5 * dtq, device="cuda", dtype=torch.float64) + 1e-3 * torch.rand(nq, generator=g2, device="cuda", dtype=torch.float64)
    qhi = qlo + 18.5 * dtq
    for _ in range(3):
        mm.shield_qp(qa, qcl, qca, qha, qlo, qhi)
    qp_runs = []
    for _ in range(4):   # best of 4 bursts of 10 launches (HBM-bound kernel timed alone -> burst peak applies)
        qe0, qe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        qe0.record()
        for _ in range(10):
            qu, qact = mm.shield_qp(qa, qcl, qca, qha, qlo, qhi)
        qe1.record()
        torch.cuda.synchronize()
        qp_runs.append(qe0.elapsed_time(qe1) / 10)
    qp_ms = min(qp_runs)
    qp_active = float((qact != 0).float().mean())
    del qa, qcl, qca, qha, qlo, qhi, qu, qact

    # e2e passes: host buffers through the C ABI, copies inside the timed region (wall clock around the calls)
    K2 = args.e2e_steps or min(K, 20)
    host_act = [torch.randint(0, 5, (E, mm.MAXV), dtype=torch.int8).pin_memory().numpy() for _ in range(4)]

    def e2e_pass(call, out):
        call(host_act[0], auto_reset=True, out=out)
        env.stats(reset=True)
        barrier()
        t0 = time.perf_counter()
        for t in range(K2):
            call(host_act[t % 4], auto_reset=True, out=out)
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        st_ = env.stats(reset=True)
        ms_, tot_ = fold(secs * 1e3, st_)
        return tot_["agent_steps"] / (ms_ * 1e-3)

    host_out = env.alloc_host_out(pinned=True)
    dense_value = e2e_pass(env.step_host, host_out)
    del host_out
    rag_out = env.alloc_host_out(pinned=True, ragged=True)
    ragged_value = e2e_pass(env.step_host_ragged, rag_out)
    rag_rows = float(rag_out["n_agents"].sum())
    del rag_out
    e2e = {"value": ragged_value, "unit": "agent-steps/s", "h2d_bytes_per_step": E * mm.MAXV,
           "d2h_bytes_per_step": int(rag_rows * mm.NS * 4 + E * (8 + 4 + 1 + mm.MAXV * 4 + 4)), "steps": K2,
           "api": "mm_step_host_ragged (pinned host buffers, half-wave chunks (28 416 envs) round-robin on 4 streams; observation rows "
                  "of the live agents only, as the reference returns them: packed on the device, exact-size copies)",
           "host_cores_bound": numa_cores,
           "dense": {"value": dense_value, "d2h_bytes_per_step": E * (mm.MAXV * mm.NS * 4 + 4 + 1 + mm.MAXV * 4 + 4),
                     "api": "mm_step_host (dense obs [E,12,30] by cudaMemcpyAsync)"}}
    if hasattr(env, "step_host_packed"):
        pk_out = env.alloc_host_out(pinned=True, packed=True)
        packed_value = e2e_pass(env.step_host_packed, pk_out)
        pk_bytes = env.packed_bytes(pk_out)
        e2e["ragged"] = {"value": ragged_value, "d2h_bytes_per_step": e2e["d2h_bytes_per_step"], "api": e2e["api"]}
        e2e.update({"value": packed_value, "d2h_bytes_per_step": int(pk_bytes),
                    "api": "mm_step_host_packed (pinned host buffers; per vehicle x, y, heading, speed as f32 + per agent "
                           "the slots of its 4 observed neighbours + ragged regional rewards: the observation rows are a "
                           "deterministic function of these, mm_expand_obs_rows builds them on the host)"})
        del pk_out

    peak, peak_src = load_peaks()
    bytes_per_launch = leg.algorithmic_bytes(mean_agents)
    achieved = bytes_per_launch / (kms * 1e-3) / 1e9
    traffic, traffic_rec = load_traffic(args.workload, E)
    cfg_out = static_config(wl, E, world, args.scaling)
    if args.policy:
        cfg_out["actions"] = ("sampled on device from the MAPPO actor 30-128-128-5 inside the timed region "
                              "(mm_actor_sample: fused TF32 forward + inverse-CDF draw, one launch per step)")
    line = {
        "metric": "shielded agent-steps/s", "value": value, "unit": "agent-steps/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg_out,
        "measured": {"mean_agents_per_env": round(mean_agents, 3),
                     "step_kernel_build": BUILD_NAMES.get(build, str(build)),
                     "shield_solves_per_s": tot["shield_solves"] / (ms_total * 1e-3),
                     "shield_active_frac": tot["shield_active"] / max(tot["shield_solves"], 1.0),
                     "lane_change_veto_frac": tot["lane_change_vetoes"] / max(tot["shield_solves"], 1.0),
                     "crashed_episode_frac": tot["crashed_episodes"] / max(tot["episodes"], 1.0)},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "step_kernel + outputs_kernel (one policy step)", "kernel_ms": kms,
                     "algorithmic_bytes_per_launch": bytes_per_launch, "peak_source": peak_src,
                     "traffic_source": (traffic_rec or {}).get("source"),
                     "note": "issue/latency-bound f64 kernels (SURVEY.md 8d): the HBM fraction is reported as asked; "
                             "see profiles/ for issue-slot and pipe utilisation"},
    }
    line["qp_microbench"] = {"solves_per_s": nq / (qp_ms * 1e-3), "n": nq, "ms": qp_ms, "active_frac": qp_active,
                             "ms_mean": float(np.mean(qp_runs)), "bytes_per_solve": 50, "achieved_GBps": nq * 50 / (qp_ms * 1e-3) / 1e9,
                             "hbm_frac": nq * 50 / (qp_ms * 1e-3) / 1e9 / peak, "dtype": "f64"}
    leg.close()
    del leg, env

    # ---- strong scaling of the same workload: its envs split over the GPUs (BASELINE configs[4] as stated)
    if not args.skip_extra and args.scaling == "weak":
        if world == 1:
            line["strong_scaling"] = {"envs_total": E_total, "envs_per_gpu": E_total, "value": value, "ms_per_step": ms_total / K,
                                      "note": "one GPU: same run as the headline"}
        else:
            Es = max(128, (E_total // world) // 128 * 128)
            sl = Leg(mm, mmd, args.workload, Es, dev, rank)
            ms_s, st_s, _ = sl.timed(K, W, barrier)
            ms_s, tot_s = fold(ms_s, st_s)
            line["strong_scaling"] = {"envs_total": Es * world, "envs_per_gpu": Es, "value": tot_s["agent_steps"] / (ms_s * 1e-3),
                                      "ms_per_step": ms_s / K, "step_kernel_build": BUILD_NAMES.get(sl.env.step_build(), "?")}
            sl.close()
            del sl

    # ---- the other BASELINE configs as short legs on one GPU (configs[0..3]; the headline is configs[4])
    if not args.skip_extra and world == 1 and args.workload == "mass_td3" and not args.envs:
        legs = {}
        for key, name, pol in (("configs[0] no shield (v0 env, td1 mixed)", "unsafe_v0_td1", False),
                               ("configs[1] HSS td3, 4096 envs", "hss_td3", False),
                               ("configs[2] MASS td1, 65536 envs", "mass_td1", False),
                               ("configs[3] MASS td3 srew, 65536 envs, uniform actions", "mass_td3_srew", False),
                               ("configs[3] MASS td3 srew, 65536 envs, actor in the loop", "mass_td3_srew", True),
                               ("MASS td3 mixed traffic, 262144 envs", "mass_td3_mixed", False)):
            En = WORKLOADS[name]["envs"] if name != "mass_td3_mixed" else 262144
            lg = Leg(mm, mmd, name, En, dev, rank, policy=pol)
            ms_l, st_l, _ = lg.timed(30, 20, barrier)    # 20 warm-up steps: every action slab has been seen twice (graph replay)
            kms_l, _ = lg.kernel_times(10)
            ag = st_l["agent_steps"] / max(st_l["env_steps"], 1.0)
            bpl = lg.algorithmic_bytes(ag)
            legs[key] = {"workload": WORKLOADS[name]["desc"], "envs": En, "value": st_l["agent_steps"] / (ms_l * 1e-3),
                         "ms_per_step": ms_l / 30, "step_kernel_build": BUILD_NAMES.get(lg.env.step_build(), "?"),
                         "roofline_frac": bpl / (kms_l * 1e-3) / 1e9 / peak, "kernel_ms": kms_l}
            lg.close()
            del lg
        line["workloads"] = legs

    if rank == 0 and world == 1 and not args.skip_cpu:
        v_cpu, cores, n_steps, e_cpu, _ = cpu_port_throughput(wl["cfg"], args.cpu_seconds, min(E, 16384))
        line["cpu_baseline"] = {"value": v_cpu, "unit": "agent-steps/s", "cores": cores, "kind": "port",
                                "sample": "%d envs of the workload, phases staggered, x %d policy steps (~%.0f s of CPU work)"
                                          % (e_cpu, n_steps, args.cpu_seconds)}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

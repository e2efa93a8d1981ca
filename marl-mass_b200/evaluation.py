"""Batched evaluation protocol (SURVEY.md §8f rank 3): `MAPPO.evaluation` (marl/mappo.py:255-361) with every
evaluation episode as one env of a single batch.

The reference runs `eval_episodes` episodes one after the other on `env_eval`, episode i from
`env.reset(is_training=False, testing_seeds=seeds[i], num_CAV=...)`, and returns
`(rewards, (vehicle_speed, vehicle_position), ext_info)`.  Here episode i is env i: the scenes are the reference's
own for those seeds (host replay of its MT19937 draws, `spawn.py`), all envs step together until the last one is
done, and each env's records stop at its own terminal step.  Same return structure, same keys.
"""
import operator
import time

import numpy as np

from ._lib import MAXV
from .env import MergeEnvBatched


def eval_num_cav(i, traffic_density):
    """The per-episode `num_CAV` argument of the training-time evaluation (mappo.py:280-286)."""
    return {1: (i + 1) % 3, 2: (i + 2) % 4, 3: (i + 4) % 6}[int(traffic_density)]


def evaluation(action_fn, config, test_seeds, eval_episodes=None, is_train=True, device=0, output_dir=None, tag="testing"):
    """action_fn(obs [E, 12, n_s] cuda f32, n_agents [E] cuda i32) -> actions [E, 12] (cuda, integer).

    Returns (rewards, (vehicle_speed, vehicle_position), ext_info) as `MAPPO.evaluation` does: rewards[i] is the list
    of global rewards of episode i; vehicle_speed[i] / vehicle_position[i] are arrays [steps_i, n_agents_i];
    ext_info has steps, avg_speeds, crash_count, step_time, min_headway, traffic_speeds, merge_percents.

    output_dir: where the reference records one video per episode (mappo.py:290-302, 321-327), this writes the same
    frames as PNG files `<tag>_episode_<i>/frame_<t>.png` (the first after reset, then one per policy step), rendered
    on the CPU from the device state (render.py); there is no video encoder in the image."""
    import torch
    seeds = [int(s) for s in (test_seeds.split(",") if isinstance(test_seeds, str) else test_seeds)]
    n_ep = len(seeds) if eval_episodes is None else int(eval_episodes)
    seeds = seeds[:n_ep]
    env = MergeEnvBatched(n_ep, config, device=device)
    td = env.config["traffic_density"]
    num_cav = [eval_num_cav(i, td) if is_train else 0 for i in range(n_ep)]
    env.reset_from_seeds(seeds, num_CAV=num_cav)
    v = env.buffers()
    n_agents = v["n_agents"].clone()
    n_host = n_agents.cpu().numpy()
    active = np.ones(n_ep, bool)
    rewards = [[] for _ in range(n_ep)]
    v_speed = [[] for _ in range(n_ep)]
    v_pos = [[] for _ in range(n_ep)]
    steps = np.zeros(n_ep, int)
    avg_speed = np.zeros(n_ep)
    traffic_speed = np.zeros(n_ep)
    merge_percent = np.full(n_ep, np.nan)
    crashed = np.zeros(n_ep, bool)
    min_headway = float("inf")
    t_total, n_steps = 0.0, 0

    def write_frames(st, which, t):
        import os
        from .render import render_scene, save_png
        for e in which:
            d = os.path.join(output_dir, "%s_episode_%d" % (tag, e))
            os.makedirs(d, exist_ok=True)
            save_png(os.path.join(d, "frame_%03d.png" % t), render_scene(st, int(e), env.config))
    if output_dir is not None:
        write_frames(env.get_state(), range(n_ep), 0)
    while active.any():
        t0 = time.process_time()
        a = action_fn(env.obs_view(), n_agents).to(torch.int8)
        env.step(a)
        torch.cuda.synchronize(device)
        t_total += time.process_time() - t0
        n_steps += 1
        st = env.get_state()
        out = {k: v[k].cpu().numpy() for k in ("reward", "done", "average_speed", "traffic_speed", "min_headway",
                                                "merge_percent")}
        if output_dir is not None:
            write_frames(st, np.nonzero(active)[0], n_steps)
        for e in np.nonzero(active)[0]:
            n = int(n_host[e])
            steps[e] += 1
            rewards[e].append(float(out["reward"][e]))
            avg_speed[e] += out["average_speed"][e]
            traffic_speed[e] += out["traffic_speed"][e]
            min_headway = min(min_headway, float(out["min_headway"][e]))
            v_speed[e].append(st["speed"][e, :n].copy())
            v_pos[e].append(st["x"][e, :n].copy())
            if out["done"][e]:
                active[e] = False
                merge_percent[e] = out["merge_percent"][e]
                crashed[e] = bool(st["crashed"][e, :n].any())
    env.close()
    ext_info = {"steps": [int(s) for s in steps], "avg_speeds": list(avg_speed / steps),
                "crash_count": [bool(c) for c in crashed], "step_time": [t_total / max(n_steps, 1)] * n_ep,
                "min_headway": min_headway, "traffic_speeds": list(traffic_speed / steps),
                "merge_percents": [float(m) for m in merge_percent]}
    return rewards, ([np.array(x) for x in v_speed], [np.array(x) for x in v_pos]), ext_info


def crash_rate_ci95(crashes, episodes):
    """Two-sided 95 % Clopper-Pearson interval of a binomial rate (crashes out of episodes)."""
    from scipy.stats import beta
    k, n = int(crashes), int(episodes)
    lo = float(beta.ppf(0.025, k, n - k + 1)) if k > 0 else 0.0
    hi = float(beta.ppf(0.975, k + 1, n - k)) if k < n else 1.0
    return lo, hi


def evaluate_seeds(action_fn, config, seeds, eval_episodes=None, is_train=True, device=0, vehicle_records=False,
                   batch=1 << 20, shield_records=False, control_profiles=None):
    """`evaluation` for many test seeds: the same episodes, bit for bit, for the same seeds and action function, with the
    scenes spawned on the device (`reset_from_seeds_device`) and the records kept there (mm_eval_record) - no host
    replay, no state copy and no synchronisation inside the step loop.

    action_fn and the num_CAV rule (`eval_num_cav` by episode index when is_train) are `evaluation`'s.  Every batch of at
    most `batch` envs (the last one, if shorter, on its own handle) runs exactly T = duration * policy_frequency policy
    steps - every episode has ended by then, which is checked once at the end.  Returns a dict of numpy arrays over the
    N episodes: rewards [N, T] f32 (0 after the episode's last step), steps [N], avg_speeds / traffic_speeds [N] (the
    float64 sums over the episode's steps / steps, as `evaluation` forms them), crashed [N] bool, merge_percents [N],
    min_headway [N] (per episode; `evaluation` reports the minimum over all of them), episode_reward [N] (float64 sum of
    the row of rewards), n_agents [N] (at reset); with vehicle_records also vehicle_speed / vehicle_position
    [N, T, 12] f64 (slots below n_agents, steps below steps; 0 elsewhere); and crash_rate with its 95 % Clopper-Pearson
    interval crash_rate_ci95.  An env's index inside its batch keys the draws of a row-keyed action function (the fused
    actor) and of the priority / dmc supervisors (Philox keyed by env): with those, results match `evaluation` and do not
    depend on `batch` as long as all seeds fit in one batch.

    shield_records / control_profiles (a sequence of K distinct episode indices into the seeds) run the batches on handles
    with the shield's diagnostic record (record_diag) and reduce it on the device after every step
    (mm_eval_shield_record).  shield_records adds, per episode: shield_solves, shield_active, shield_interventions,
    lane_change_vetoes [N] int64 and acc_correction_sum, acc_correction_max, steer_correction_max (|safe - nominal| of
    the shielded actions) and min_agent_acc (the hardest applied acceleration of a controlled vehicle, +inf if none
    moved) [N] f64, and intervention_rate (interventions over solves, 0 without solves).  control_profiles adds
    control_profile_episodes [K] and control_profiles, a dict of the per-sub-step fields of log_step
    (safe_controller.py:187-227) - moved, ran, active, is_lc_safe, hl_action, lane (int32) and x, y, heading, speed,
    min_headway, safe_acc, safe_steer, nom_acc, nom_steer (f64) - each [K, 3 T, 12] with row 3 t + s for sub-step s of
    policy step t, 0 after the episode."""
    import torch
    from . import _lib
    seeds = np.asarray([int(s) for s in seeds.split(",")] if isinstance(seeds, str) else seeds, np.int64).reshape(-1)
    n_ep = len(seeds) if eval_episodes is None else int(eval_episodes)
    seeds = seeds[:n_ep]
    batch = int(batch)
    if n_ep < 1 or batch < 1:
        raise ValueError("evaluate_seeds needs at least one seed and batch >= 1")
    profiles = None
    if control_profiles is not None:
        profiles = np.array([operator.index(i) for i in control_profiles], np.int64).reshape(-1)
        if len(np.unique(profiles)) != len(profiles):
            raise ValueError("evaluate_seeds: control_profiles holds an episode index more than once")
        if len(profiles) and (profiles.min() < 0 or profiles.max() >= n_ep):
            raise ValueError("evaluate_seeds: control_profiles must be episode indices in [0, %d)" % n_ep)
    diag = bool(shield_records) or profiles is not None
    dev = torch.device("cuda", device)
    env = None
    res = None
    for b0 in range(0, n_ep, batch):
        n = min(batch, n_ep - b0)
        if env is None or env.n_envs != n:
            if env is not None:
                env.close()
            env = MergeEnvBatched(n, config, device=device, record_diag=diag)
        T = env.T
        if res is None:
            td = env.config["traffic_density"]
            num_cav = eval_num_cav(np.arange(n_ep), td) if is_train else np.zeros(n_ep, np.int64)
            res = {"rewards": np.zeros((n_ep, T), np.float32), "steps": np.zeros(n_ep, np.int64),
                   "avg_speed_sum": np.zeros(n_ep), "traffic_speed_sum": np.zeros(n_ep),
                   "crashed": np.zeros(n_ep, bool), "merge_percents": np.zeros(n_ep), "min_headway": np.zeros(n_ep),
                   "n_agents": np.zeros(n_ep, np.int32)}
            if vehicle_records:
                res["vehicle_speed"] = np.zeros((n_ep, T, MAXV))
                res["vehicle_position"] = np.zeros((n_ep, T, MAXV))
            if diag:
                sh = {k: torch.zeros(n_ep, dtype=torch.int32, device=dev) for k in _lib.SHIELD_COUNTS}
                sh.update({k: torch.zeros(n_ep, dtype=torch.float64, device=dev) for k in _lib.SHIELD_F64})
                sh["min_agent_acc"].fill_(float("inf"))
            if profiles is not None:
                prof = {k: torch.zeros((len(profiles), 3 * T, MAXV), dtype=torch.int32, device=dev) for k in _lib.PROFILE_I}
                prof.update({k: torch.zeros((len(profiles), 3 * T, MAXV), dtype=torch.float64, device=dev)
                             for k in _lib.PROFILE_F})
        env.reset_from_seeds_device(seeds[b0:b0 + n], num_CAV=num_cav[b0:b0 + n])
        n_agents = env.buffers()["n_agents"].clone()
        rec = {"active": torch.ones(n, dtype=torch.uint8, device=dev), "rewards": torch.zeros((n, T), device=dev),
               "steps": torch.zeros(n, dtype=torch.int32, device=dev),
               "avg_speed_sum": torch.zeros(n, dtype=torch.float64, device=dev),
               "traffic_speed_sum": torch.zeros(n, dtype=torch.float64, device=dev),
               "min_headway": torch.full((n,), float("inf"), device=dev), "merge_percent": torch.zeros(n, device=dev),
               "crashed": torch.zeros(n, dtype=torch.uint8, device=dev)}
        if vehicle_records:
            rec["vehicle_speed"] = torch.zeros((n, T, MAXV), dtype=torch.float64, device=dev)
            rec["vehicle_position"] = torch.zeros((n, T, MAXV), dtype=torch.float64, device=dev)
        records = _lib.MMEvalRecords(T=T, n_agents=n_agents.data_ptr(), **{k: v.data_ptr() for k, v in rec.items()})
        if diag:
            ptrs = {k: v[b0:b0 + n].data_ptr() for k, v in sh.items()}
            if profiles is not None:
                slot = np.full(n, -1, np.int32)
                mine = (profiles >= b0) & (profiles < b0 + n)
                slot[profiles[mine] - b0] = np.nonzero(mine)[0]
                slot_dev = torch.from_numpy(slot).to(dev)
                ptrs["profile_slot"] = slot_dev.data_ptr()
                ptrs.update({"profile_" + k: v.data_ptr() for k, v in prof.items()})
            sh_records = _lib.MMEvalShieldRecords(T=T, n_agents=n_agents.data_ptr(), active=rec["active"].data_ptr(), **ptrs)
        for t in range(T):
            a = action_fn(env.obs_view(), n_agents).to(torch.int8)
            env.step(a)
            if diag:
                env.eval_shield_record(sh_records, t)
            env.eval_record(records, t)
        if rec["active"].any():     # the one synchronisation of the batch
            raise RuntimeError("evaluate_seeds: %d episodes of seeds[%d:%d] had not ended after T = %d policy steps"
                               % (int(rec["active"].sum()), b0, b0 + n, T))
        sl = slice(b0, b0 + n)
        res["rewards"][sl] = rec["rewards"].cpu().numpy()
        res["steps"][sl] = rec["steps"].cpu().numpy()
        res["avg_speed_sum"][sl] = rec["avg_speed_sum"].cpu().numpy()
        res["traffic_speed_sum"][sl] = rec["traffic_speed_sum"].cpu().numpy()
        res["crashed"][sl] = rec["crashed"].cpu().numpy() != 0
        res["merge_percents"][sl] = rec["merge_percent"].cpu().numpy()
        res["min_headway"][sl] = rec["min_headway"].cpu().numpy()
        res["n_agents"][sl] = n_agents.cpu().numpy()
        if vehicle_records:
            res["vehicle_speed"][sl] = rec["vehicle_speed"].cpu().numpy()
            res["vehicle_position"][sl] = rec["vehicle_position"].cpu().numpy()
    env.close()
    if shield_records:
        for k in _lib.SHIELD_COUNTS:
            res[k] = sh[k].cpu().numpy().astype(np.int64)
        for k in _lib.SHIELD_F64:
            res[k] = sh[k].cpu().numpy()
        solves = int(res["shield_solves"].sum())
        res["intervention_rate"] = int(res["shield_interventions"].sum()) / solves if solves else 0.0
    if profiles is not None:
        res["control_profiles"] = {k: v.cpu().numpy() for k, v in prof.items()}
        res["control_profile_episodes"] = profiles
    res["avg_speeds"] = res.pop("avg_speed_sum") / res["steps"]
    res["traffic_speeds"] = res.pop("traffic_speed_sum") / res["steps"]
    res["episode_reward"] = res["rewards"].astype(np.float64).sum(axis=1)
    k = int(res["crashed"].sum())
    res["crash_rate"] = k / n_ep
    res["crash_rate_ci95"] = crash_rate_ci95(k, n_ep)
    return res

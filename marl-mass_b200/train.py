"""Batched training driver: `run_mappo.py --option train --config <ini>` (run_mappo.py:86-340) with the per-env Python
loop replaced by E envs on the device.

    python -m marl_mass_b200.train --config examples/mass_td3_srew.ini --envs 4096 --iterations 30

Reads the reference's ini layout (sections MODEL_CONFIG / TRAIN_CONFIG / ENV_CONFIG, the keys run_mappo.py:113-171
reads), builds `MergeEnvBatched` + `BatchedMAPPORollout` (MAPPO.interact / train for the whole batch) and, every
`--eval-interval` iterations, runs the reference's evaluation protocol on `test_seeds` as one batch
(`evaluation.evaluation` = MAPPO.evaluation) and prints what the reference logs (run_mappo.py:295-332).
"""
import argparse
import configparser
import json
import time

import numpy as np


def load_ini(path):
    """-> (env_config dict for MergeEnvBatched, rollout kwargs, train dict).  Same keys and fallbacks as run_mappo.py."""
    c = configparser.ConfigParser()
    if not c.read(path):
        raise FileNotFoundError(path)
    E = "ENV_CONFIG"
    env_cfg = {
        "env_name": c.get(E, "env_name", fallback="merge-multi-agent-v0"),
        "seed": c.getint(E, "seed"), "simulation_frequency": c.getint(E, "simulation_frequency"),
        "duration": c.getint(E, "duration"), "policy_frequency": c.getint(E, "policy_frequency"),
        "COLLISION_REWARD": c.getint(E, "COLLISION_REWARD"), "HIGH_SPEED_REWARD": c.getint(E, "HIGH_SPEED_REWARD"),
        "HEADWAY_COST": c.getint(E, "HEADWAY_COST"), "HEADWAY_TIME": c.getfloat(E, "HEADWAY_TIME"),
        "MERGING_LANE_COST": c.getint(E, "MERGING_LANE_COST"), "traffic_density": c.getint(E, "traffic_density"),
        "action_masking": c.getboolean("MODEL_CONFIG", "action_masking", fallback=False),
        "safety_guarantee": c.get(E, "safety_guarantee"), "lateral_control": c.get(E, "lateral_control", fallback="steer"),
        "mixed_traffic": c.getboolean(E, "mixed_traffic", fallback=None),
        "traffic_type": c.get(E, "traffic_type", fallback="cav"), "agent_reward": c.get(E, "agent_reward", fallback="default"),
        "cbf_eta": c.getfloat(E, "cbf_eta", fallback=0.0),          # CBFType.GAMMA_B (run_mappo.py:138)
    }
    M, T = "MODEL_CONFIG", "TRAIN_CONFIG"
    rollout_kw = {
        "roll_out_n_steps": c.getint(M, "ROLL_OUT_N_STEPS"), "reward_gamma": c.getfloat(M, "reward_gamma"),
        "max_grad_norm": c.getfloat(M, "MAX_GRAD_NORM"), "reward_type": c.get(M, "reward_type"),
        "reward_scale": c.getfloat(T, "reward_scale"), "actor_lr": c.getfloat(T, "actor_lr"),
        "critic_lr": c.getfloat(T, "critic_lr"),
    }
    train = {"test_seeds": c.get(T, "test_seeds", fallback=",".join(str(i) for i in range(0, 600, 20))),
             "eval_episodes": c.getint(T, "EVAL_EPISODES", fallback=20), "torch_seed": c.getint(M, "torch_seed", fallback=0),
             # run_mappo.py:126,232: shared_network selects MAPPO_GI with its one ActorCriticNetwork
             "shared_network": c.getboolean(M, "shared_network", fallback=False),
             "critic_hidden_size": c.getint(M, "critic_hidden_size", fallback=128),
             # not a key of the reference: the GAE lambda of the returns (None: its Monte-Carlo returns), checked by train()
             "gae_lambda": c.get(M, "gae_lambda", fallback=None)}
    return env_cfg, rollout_kw, train


def train(config, n_envs=4096, iterations=30, device=0, eval_interval=10, minibatch=1 << 18, log=print, update_impl="torch",
          optimizer="torch", eval_seeds=0, eval_shield=False, update_stats=False, gae_lambda=None):
    """update_impl: "torch" (autograd, the default) or "cuda" (the on-device learner, `update(impl="cuda")`).
    optimizer: "torch" (clip_grad_norm_ + torch.optim.RMSprop, the default) or "cuda" (`rollout.DeviceRMSprop`: the same
    step in one launch per minibatch).
    eval_seeds: N > 0 also evaluates every eval point on the test seeds 0..N-1 (`evaluation.evaluate_seeds`, the
    reference's protocol with the scenes spawned and the records kept on the device) and logs the evalN_* keys: episodes,
    crash_rate with its 95 % Clopper-Pearson interval, mean episode reward, mean average speed, mean merge percent,
    minimum headway and the wall time in seconds.  Its draws come from a counter of their own, so the other keys are
    the same with and without it.
    eval_shield: with eval_seeds, also record the shield's activity on those episodes (`evaluate_seeds(shield_records=True)`)
    and log evalN_shield_intervention_rate (interventions over QP solves), evalN_lane_change_vetoes_per_episode,
    evalN_min_agent_acc (the hardest applied acceleration of any controlled vehicle) and evalN_acc_correction_max (the
    largest |safe - nominal| acceleration).
    update_stats: also measure every update (`update(stats=True)`, with either update_impl) and log the keys of
    `rollout.ppo_stats_keys` with an update_ prefix: update_approx_kl, update_clip_fraction, update_ratio_min /
    update_ratio_max, update_entropy_before / _after, update_explained_variance_before / _after, update_advantage_mean and
    update_advantage_std.  The update and every other key are the same with and without it.
    gae_lambda: a number in [0, 1] trains on GAE(lambda) returns (`BatchedMAPPORollout(gae_lambda=...)`, with either
    update_impl); None takes MODEL_CONFIG.gae_lambda from the ini, and without that key the returns are the reference's
    Monte-Carlo returns.  A non-number, NaN or a value outside [0, 1] is refused before anything is built."""
    if eval_shield and not eval_seeds > 0:
        raise ValueError("train: eval_shield records the shield on the eval_seeds episodes and needs eval_seeds > 0")
    import torch
    from . import evaluation as ev
    from .env import DEFAULT_CONFIG, MergeEnvBatched
    from .rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout, check_gae_lambda
    import torch.distributed as dist
    from . import dist as mmd
    env_cfg, rollout_kw, tr = load_ini(config) if isinstance(config, str) else config
    rank, world, local_rank = mmd.rank_world()
    if world > 1:                 # torchrun: one process per GPU, n_envs envs each, gradients averaged
        device = local_rank
        torch.cuda.set_device(device)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    torch.manual_seed(tr["torch_seed"])
    if env_cfg.get("env_name", "merge-multi-agent-v1") != "merge-multi-agent-v1":
        # env ids merge-multi-agent-v0 / -v05 observe 5 x 5 (no heading column, n_s = 25) and -hdv-v1 has no agents: the
        # networks of this driver and the fused actor kernels are the reference's 30-input ones (Model_common.py:11-23
        # with n_s = 30).  Rejected before anything is built (a 25-column state would otherwise be fed to 30 inputs).
        raise ValueError("train: env id %r is not covered by the batched learner (n_s = 30 env id merge-multi-agent-v1 only)"
                         % (env_cfg.get("env_name"),))
    if not isinstance(update_stats, bool):
        raise ValueError("train: update_stats must be True or False, got %r" % (update_stats,))
    if update_stats and update_impl not in ("torch", "cuda"):
        raise ValueError("train: update_stats measures the 'torch' or 'cuda' update, got update_impl %r" % (update_impl,))
    try:
        gae_lambda = check_gae_lambda(tr.get("gae_lambda") if gae_lambda is None else gae_lambda)
    except ValueError as e:
        raise ValueError("train: %s" % e) from None
    env = MergeEnvBatched(n_envs, dict(DEFAULT_CONFIG, **env_cfg), device=device)
    # rank-distinct spawn stream; its first observation goes to the rollout so that collect() does not re-spawn the
    # scenes with the (rank-independent) config seed
    obs0, _ = env.reset(seed=mmd.rank_seed(env_cfg["seed"], rank) if world > 1 else env_cfg["seed"])
    if tr.get("shared_network"):
        pol = BatchedMAPPOGIRollout(env, hidden_size=tr.get("critic_hidden_size", 128),
                                    seed=tr["torch_seed"] + 104729 * rank, obs=obs0, optimizer=optimizer, gae_lambda=gae_lambda,
                                    **rollout_kw)
    else:
        pol = BatchedMAPPORollout(env, seed=tr["torch_seed"] + 104729 * rank, obs=obs0, optimizer=optimizer,
                                  gae_lambda=gae_lambda, **rollout_kw)
    pol.sync_parameters()
    if rank != 0:
        log = lambda *_: None
    draws = {"n": 0}

    def act(obs, n_agents):      # MAPPO.action (mappo.py:231-236): a draw from the softmax, also at evaluation time
        draws["n"] += 1
        return pol.sample_actions(obs, n_agents, seed=tr["torch_seed"] + 7919, step=draws["n"])

    def act_seeds(obs, n_agents):
        draws["seeds"] += 1
        return pol.sample_actions(obs, n_agents, seed=tr["torch_seed"] + 7919, step=draws["seeds"])
    draws["seeds"] = 0

    history = []
    for it in range(iterations):
        t0 = time.perf_counter()
        env.stats(reset=True)
        pol.collect()
        torch.cuda.synchronize(device)
        t1 = time.perf_counter()
        up = pol.update(minibatch=minibatch, impl=update_impl, stats=update_stats)
        up = {(k if k in ("actor_loss", "critic_loss", "samples") else "update_" + k): v for k, v in up.items()}
        torch.cuda.synchronize(device)
        t2 = time.perf_counter()
        s = mmd.all_reduce_stats(env.stats())
        rec = {"iteration": it, "n_gpus": world, "agent_steps": s["agent_steps"], "collect_s": t1 - t0, "update_s": t2 - t1,
               "agent_steps_per_s": s["agent_steps"] / (t1 - t0), "mean_step_reward": s["reward_sum"] / max(s["env_steps"], 1),
               "crashed_episode_frac": s["crashed_episodes"] / max(s["episodes"], 1),
               "average_speed": s["speed_sum"] / max(s["env_steps"], 1), **up}
        if rank == 0 and eval_interval and (it % eval_interval == 0 or it == iterations - 1):
            rewards, _, info = ev.evaluation(act, env_cfg, tr["test_seeds"], eval_episodes=tr["eval_episodes"], device=device)
            rec.update({"eval_reward": float(np.mean([np.sum(r) for r in rewards])),       # run_mappo.py:303-306
                        "eval_avg_speed": float(np.mean(info["avg_speeds"])), "eval_crashes": int(np.sum(info["crash_count"])),
                        "eval_min_headway": info["min_headway"], "eval_merge_percent": float(np.mean(info["merge_percents"]))})
            if eval_seeds > 0:
                t3 = time.perf_counter()
                r = ev.evaluate_seeds(act_seeds, env_cfg, np.arange(int(eval_seeds)), device=device, shield_records=eval_shield)
                if eval_shield:
                    rec.update({"evalN_shield_intervention_rate": r["intervention_rate"],
                                "evalN_lane_change_vetoes_per_episode": float(np.mean(r["lane_change_vetoes"])),
                                "evalN_min_agent_acc": float(np.min(r["min_agent_acc"])),
                                "evalN_acc_correction_max": float(np.max(r["acc_correction_max"]))})
                rec.update({"evalN_episodes": int(eval_seeds), "evalN_crash_rate": r["crash_rate"],
                            "evalN_crash_rate_ci95": list(r["crash_rate_ci95"]),
                            "evalN_reward": float(np.mean(r["episode_reward"])), "evalN_avg_speed": float(np.mean(r["avg_speeds"])),
                            "evalN_merge_percent": float(np.mean(r["merge_percents"])),
                            "evalN_min_headway": float(np.min(r["min_headway"])), "evalN_s": time.perf_counter() - t3})
        if world > 1 and it == iterations - 1:      # the replicas must still hold identical networks
            flat = torch.cat([q.detach().reshape(-1) for m in pol.networks() for q in m.parameters()])
            hi, lo = flat.clone(), flat.clone()
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            rec["replica_param_max_diff"] = float((hi - lo).abs().max())
        history.append(rec)
        log(json.dumps(rec))
    env.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return history


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", required=True)
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--iterations", type=int, default=30)
    ap.add_argument("--eval-interval", type=int, default=10)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--update-impl", choices=("torch", "cuda"), default="torch",
                    help="PPO update: torch autograd or the on-device learner kernels")
    ap.add_argument("--optimizer", choices=("torch", "cuda"), default="torch",
                    help="gradient clipping + RMSprop step: torch ops or one device launch per minibatch")
    ap.add_argument("--eval-seeds", type=int, default=0,
                    help="N > 0: also evaluate on the test seeds 0..N-1 with the device-side protocol (evalN_* keys)")
    ap.add_argument("--eval-shield", action="store_true",
                    help="with --eval-seeds: also log the shield's interventions, vetoes and corrections (evalN_shield_* keys)")
    ap.add_argument("--update-stats", action="store_true",
                    help="also log what each update did: KL to the rollout policy, clip fraction, ratio range, entropy, "
                         "explained variance, advantage mean / std (update_* keys)")
    ap.add_argument("--gae-lambda", type=float, default=None,
                    help="train on GAE(lambda) returns with this lambda in [0, 1] (default: MODEL_CONFIG.gae_lambda of the "
                         "ini, else the Monte-Carlo returns)")
    a = ap.parse_args()
    train(a.config, a.envs, a.iterations, a.device, a.eval_interval, update_impl=a.update_impl, optimizer=a.optimizer,
          eval_seeds=a.eval_seeds, eval_shield=a.eval_shield, update_stats=a.update_stats, gae_lambda=a.gae_lambda)


if __name__ == "__main__":
    main()

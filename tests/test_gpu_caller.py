"""GPU suite, caller side (SURVEY.md 8f rank 1): the fused actor + exploration-draw kernel and the discounted-return
kernel, through the C ABI, against the reference vectors (tests/golden/mappo_caller.npz), the numpy restatements in
oracle/ and a plain torch fp32 evaluation of the same network.

Tolerances: the actor runs on tensor cores with fp16 operands (the mma.sync cross-check with TF32 ones: both have a
10-bit mantissa) and fp32 accumulation: log-probabilities within 2e-2 absolute of the fp32 network on O(1) inputs
(observed ~3e-3); returns are fp32 sums: 1e-5 relative.
"""
import os

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

LOGP_TOL = 2e-2


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()
    return m


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "mappo_caller.npz"))


def make_actor(g, torch, rollout):
    actor = rollout.ActorNetwork().cuda()
    sd = {k[2:].replace("_", ".", 1): torch.from_numpy(g[k]) for k in g.files if k.startswith("w_")}
    actor.load_state_dict(sd)
    return actor


def test_actor_log_probs_match_the_reference_network(mm, golden):
    import torch
    from marl_mass_b200 import rollout
    actor = make_actor(golden, torch, rollout)
    obs = torch.from_numpy(golden["obs"]).cuda()
    acts, logp = rollout.actor_sample(actor, obs, None, seed=3, step=1, want_logp=True)
    torch.cuda.synchronize()
    logp = logp.cpu().numpy()
    assert np.abs(logp - golden["logp"]).max() < LOGP_TOL           # reference ActorNetwork output (fp32, CPU)
    assert np.abs(np.exp(logp).sum(1) - 1).max() < 1e-5
    a = acts.cpu().numpy()
    assert a.shape == (obs.shape[0],) and a.min() >= 0 and a.max() <= 4


def test_actor_matches_torch_fp32_on_env_observations_and_masks_absent_agents(mm):
    import torch
    import oracle
    from marl_mass_b200 import rollout
    E = 2048
    env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3,
                                     HEADWAY_TIME=0.5, cbf_eta=0.03125), device=0)
    obs, _ = env.reset(seed=5)
    v = env.buffers()
    torch.manual_seed(0)
    actor = rollout.ActorNetwork().cuda()
    for p in actor.parameters():                    # larger weights than the default init: a sharper policy
        p.data.mul_(3.0)
    acts, logp = rollout.actor_sample(actor, obs, v["n_agents"], seed=9, step=4, want_logp=True)
    with torch.no_grad():
        want = actor(obs.view(-1, mm.NS)).view(E, mm.MAXV, mm.NA)
    torch.cuda.synchronize()
    assert float((logp - want).abs().max()) < LOGP_TOL
    # numpy float64 restatement of the reference network
    w = {k.replace(".", "_"): t.detach().cpu().numpy() for k, t in actor.state_dict().items()}
    ref = oracle.actor_log_probs(w, obs.view(-1, mm.NS).cpu().numpy()).reshape(E, mm.MAXV, mm.NA)
    assert np.abs(logp.cpu().numpy() - ref).max() < LOGP_TOL
    live = (torch.arange(mm.MAXV, device="cuda")[None, :] < v["n_agents"][:, None])
    assert bool((acts[~live] == 1).all())           # absent agents idle
    assert bool(((acts >= 0) & (acts <= 4)).all())
    # same (seed, step) -> same draw; another step -> another draw
    again = rollout.actor_sample(actor, obs, v["n_agents"], seed=9, step=4)
    other = rollout.actor_sample(actor, obs, v["n_agents"], seed=9, step=5)
    assert bool((again == acts).all()) and float((other != acts)[live].float().mean()) > 0.2
    env.close()


def test_tcgen05_and_mma_sync_actor_kernels_agree(mm):
    """The default tcgen05 kernel (fp16 operands, biases inside the MMAs, TMEM accumulators) against the independent
    mma.sync kernel (TF32 register fragments) and torch fp32, with the default weights and with 3x their scale (a sharper
    policy): fp16 and TF32 share the 10-bit mantissa and both accumulate in fp32 -> log-probabilities within 1e-2 of
    torch and of each other (observed at 3x scale: 5.7e-3 and 3.0e-3); the same uniform per row -> the same
    action except where the draw falls within that distance of a CDF step.  Neither row count is a multiple of the
    128-row tile."""
    import torch
    from marl_mass_b200 import rollout
    for torch_seed, scale, rows, span, seed in ((3, 3.0, 100003, 1.2, 5), (4, 1.0, 70001, 1.1, 9)):
        torch.manual_seed(torch_seed)
        actor = rollout.ActorNetwork().cuda()
        for p in actor.parameters():
            p.data.mul_(scale)
        obs = (torch.rand(rows, mm.NS, device="cuda") * 2 * span - span).contiguous()
        out = {}
        try:
            for name in ("mma", "tcgen05"):
                rollout.set_actor_impl(name)
                out[name] = rollout.actor_sample(actor, obs, None, seed=seed, step=2, want_logp=True)
                torch.cuda.synchronize()
        finally:
            rollout.set_actor_impl("tcgen05")
        with torch.no_grad():
            ref = torch.log_softmax(actor.fc3(torch.relu(actor.fc2(torch.relu(actor.fc1(obs))))), dim=1)
        (a_m, lp_m), (a_t, lp_t) = out["mma"], out["tcgen05"]
        for name, (_, lp) in out.items():
            assert float((lp - ref).abs().max()) < 1e-2, (name, scale)
        assert float((lp_m - lp_t).abs().max()) < 1e-2, scale
        assert float((a_m != a_t).float().mean()) < 5e-3, scale


def test_fused_shared_network_of_mappo_gi(mm):
    """mm_actor_sample_mlp with h1 = 160: the MAPPO_GI ActorCriticNetwork (state_split: three first-layer blocks over
    fixed column lists, scattered into one 30 -> 160 weight matrix) against the torch fp32 module - log-probabilities with
    and without invalid-action masking, the value head, draw frequencies following the softmax, absent agents -> IDLE."""
    import torch
    from marl_mass_b200 import rollout
    torch.manual_seed(11)
    pol = rollout.ActorCriticNetwork().cuda()
    for p in pol.parameters():
        p.data.mul_(2.0)
    n = 50000
    obs = (torch.rand(n, mm.NS, device="cuda") * 2.2 - 1.1).contiguous()
    mask = torch.randint(0, 32, (n,), device="cuda", dtype=torch.uint8) | 2           # IDLE always available
    a, lp, v = rollout.policy_sample(pol, obs, None, seed=3, step=1, want_logp=True, want_value=True)
    a_m, lp_m = rollout.policy_sample(pol, obs, None, seed=3, step=1, want_logp=True, action_mask=mask)
    torch.cuda.synchronize()
    with torch.no_grad():
        want = pol(obs)
        want_v = pol(obs, out_type="v").squeeze(1)
        bits = ((mask[:, None].int() >> torch.arange(5, device="cuda")[None, :]) & 1)
        want_m = pol(obs, action_mask=bits)
    assert float((lp - want).abs().max()) < 2e-2 and float((v - want_v).abs().max()) < 2e-2 * max(1.0, float(want_v.abs().max()))
    ok = bits.bool()
    assert float((lp_m - want_m)[ok].abs().max()) < 2e-2
    assert bool(ok.gather(1, a_m.long()[:, None]).all())                              # a masked action is never drawn
    # the weights change in place (an optimiser step): the cached dense first layer must follow
    with torch.no_grad():
        pol.fc12.weight.add_(0.05)
        lp2 = rollout.policy_sample(pol, obs, None, seed=3, step=1, want_logp=True)[1]
        assert float((lp2 - pol(obs)).abs().max()) < 2e-2
    # draw frequencies of one row replicated
    row = obs[:1].expand(200000, mm.NS).contiguous()
    acts = rollout.policy_sample(pol, row, None, seed=5, step=7)
    freq = torch.bincount(acts.long(), minlength=5).float() / acts.numel()
    p_row = pol(obs[:1]).exp()[0]
    assert float((freq - p_row).abs().max()) < 6 * float((p_row * (1 - p_row) / acts.numel()).sqrt().max()) + 2e-3
    # absent agents get IDLE
    env_obs = (torch.rand(64, 12, mm.NS, device="cuda") * 2 - 1).contiguous()
    n_ag = torch.randint(1, 12, (64,), device="cuda", dtype=torch.int32)
    acts = rollout.policy_sample(pol, env_obs, n_ag, seed=1, step=1)
    dead = torch.arange(12, device="cuda")[None, :] >= n_ag[:, None]
    assert bool((acts[dead] == 1).all())


def test_actor_kernel_appends_to_the_rollout_buffer(mm):
    """The draw kernels write slot t of the rollout buffer themselves (state the action was drawn from, action, live
    mask: MAPPO.interact's appends, mappo.py:117-131): same actions as the plain call, the rows copied bit for bit."""
    import torch
    from marl_mass_b200 import rollout
    torch.manual_seed(2)
    E = 3001
    obs = (torch.rand(E, 12, mm.NS, device="cuda") * 2 - 1).contiguous()
    n_ag = torch.randint(1, 12, (E,), device="cuda", dtype=torch.int32)
    for net, fn in ((rollout.ActorNetwork().cuda(), rollout.actor_sample), (rollout.ActorCriticNetwork().cuda(), rollout.policy_sample)):
        plain = fn(net, obs, n_ag, seed=4, step=9)
        S = torch.zeros(2, E, 12, mm.NS, device="cuda")
        A8 = torch.full((2, E, 12), -1, dtype=torch.int8, device="cuda")
        L8 = torch.full((2, E, 12), 7, dtype=torch.uint8, device="cuda")
        got = fn(net, obs, n_ag, seed=4, step=9, out_actions=A8[1], obs_copy=S[1], live_out=L8[1])
        torch.cuda.synchronize()
        assert got.data_ptr() == A8[1].data_ptr() and torch.equal(A8[1], plain)
        assert torch.equal(S[1], obs) and float(S[0].abs().max()) == 0.0 and int((A8[0] != -1).sum()) == 0
        assert torch.equal(L8[1].bool(), torch.arange(12, device="cuda")[None, :] < n_ag[:, None])


def test_rollouts_of_different_ranks_spawn_different_scenes(mm):
    """Data-parallel shards must not be replicas: a rollout that spawns its own scenes uses a spawn seed derived from its
    (rank-distinct) seed, never the env's config seed, so two ranks' first collect() see different scenes - and the same
    rank seed reproduces its scenes."""
    import torch
    from marl_mass_b200 import rollout
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5, cbf_eta=0.03125, seed=11)
    states = []
    for rank_seed in (0, 104729, 0):
        env = mm.MergeEnvBatched(256, cfg)
        pol = rollout.BatchedMAPPORollout(env, roll_out_n_steps=2, seed=rank_seed)
        pol.collect()
        torch.cuda.synchronize()
        states.append(env.get_state())
        env.close()
    assert not np.array_equal(states[0]["n_veh"], states[1]["n_veh"]) or not np.array_equal(states[0]["x"], states[1]["x"])
    assert np.array_equal(states[0]["n_veh"], states[2]["n_veh"])


def test_invalid_action_masking_of_the_gi_actor(mm):
    """Model_gi.ActorNetwork (marl/single_agent/Model_gi.py:63-66): logits[action_mask == 0] = -1e8, then log-softmax.
    The env's own action masks (action_masking = True) go straight into the kernel; masked actions are never drawn."""
    import torch
    from marl_mass_b200 import rollout
    E = 4096
    env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5,
                                     cbf_eta=0.03125, action_masking=True), device=0)
    obs, mask = env.reset(seed=8)                      # mask [E, 12, 5] int32 (unpacked)
    a0 = torch.randint(0, 5, (E, 12), device="cuda", dtype=torch.int8)
    for _ in range(30):                                # into the merge zone: lane changes become available for some
        obs, _, _, _ = env.step(a0, auto_reset=True)
    v = env.buffers()
    bits = v["action_mask"]
    mask = env.action_mask()
    torch.manual_seed(2)
    actor = rollout.ActorNetwork().cuda()
    for impl in ("tcgen05", "mma"):
        rollout.set_actor_impl(impl)
        acts, logp = rollout.actor_sample(actor, obs, v["n_agents"], seed=3, step=1, want_logp=True, action_mask=bits)
        with torch.no_grad():
            logits = actor.fc3(torch.relu(actor.fc2(torch.relu(actor.fc1(obs.view(-1, mm.NS)))))).view(E, mm.MAXV, mm.NA)
            logits = torch.where(mask == 0, torch.full_like(logits, -1e8), logits)
            want = torch.log_softmax(logits + 1e-8, dim=-1)
        live = torch.arange(mm.MAXV, device="cuda")[None, :] < v["n_agents"][:, None]
        avail = mask[live] != 0
        assert float((logp[live] - want[live]).abs()[avail].max()) < LOGP_TOL
        assert bool((logp[live][~avail] < -1e7).all())
        chosen = torch.gather(mask[live], 1, acts[live].long()[:, None])
        assert bool((chosen == 1).all())               # only available actions are drawn
        assert 0.0 < float((mask[live] == 0).float().mean()) < 0.9
    rollout.set_actor_impl("tcgen05")
    env.close()


def test_exploration_draw_follows_the_softmax(mm):
    """np.random.choice(p = softmax) (mappo.py:223-228): empirical action frequencies of many draws from a few fixed
    observation rows against the kernel's own probabilities."""
    import torch
    from marl_mass_b200 import rollout
    torch.manual_seed(1)
    actor = rollout.ActorNetwork().cuda()
    for p in actor.parameters():
        p.data.mul_(4.0)
    base = torch.rand(8, mm.NS, device="cuda") * 2 - 1
    reps = 1 << 16
    obs = base[:, None, :].expand(8, reps, mm.NS).contiguous()          # row r of `base` repeated `reps` times
    freq = torch.zeros(8, mm.NA, device="cuda")
    n_draws = 4
    for step in range(n_draws):
        a, logp = rollout.actor_sample(actor, obs, None, seed=21, step=step, want_logp=True)
        freq += torch.nn.functional.one_hot(a.long(), mm.NA).float().sum(1)
    p = logp[:, 0, :].exp()
    freq /= reps * n_draws
    # binomial standard error at n = 262144 is <= 1e-3; 6 sigma
    assert float((freq - p).abs().max()) < 6e-3, (freq, p)
    assert float(p.max()) > 0.4                                          # the test policy is not uniform


def test_discounted_returns_match_reference_vectors_and_restatement(mm, golden):
    import torch
    import oracle
    from marl_mass_b200 import rollout
    g = golden
    gamma = float(g["gamma"])
    # the reference's own outputs: one column per call of MAPPO._discount_reward, shorter columns end in a "done" pad
    for k, T in enumerate(g["lengths"]):
        r = torch.from_numpy(g["rewards"][:T, k].astype(np.float32)).cuda().view(T, 1, 1)
        d = torch.zeros(T, 1, device="cuda")
        fv = torch.tensor([[float(g["finals"][k])]], device="cuda")
        got = rollout.discounted_returns(r, d, fv, gamma).view(T).cpu().numpy()
        want = g["returns"][:T, k]
        assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max())
    # a full rollout with episode boundaries against the float64 restatement
    rng = np.random.RandomState(3)
    T, E, A = 100, 777, 12
    r = rng.uniform(-3, 1, size=(T, E, A)).astype(np.float32)
    d = (rng.uniform(size=(T, E)) < 0.02)
    fv = rng.uniform(-2, 2, size=(E, A)).astype(np.float32)
    got = rollout.discounted_returns(torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda(), torch.from_numpy(fv).cuda(),
                                     gamma).cpu().numpy()
    want = oracle.mappo_discount(r.reshape(T, E * A), d, fv.reshape(-1), gamma, cols_per_env=A).reshape(T, E, A)
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
    got0 = rollout.discounted_returns(torch.from_numpy(r).cuda(), torch.from_numpy(d).cuda(), None, gamma).cpu().numpy()
    want0 = oracle.mappo_discount(r.reshape(T, E * A), d, None, gamma, cols_per_env=A).reshape(T, E, A)
    assert np.abs(got0 - want0).max() <= 1e-5 * np.abs(want0).max()


def test_rollout_collect_and_update_run_on_the_fused_path(mm):
    """BatchedMAPPORollout end to end (fused actor draw, env step, CUDA returns, PPO update): shapes, masks, finite
    losses, and the fused and torch draws agree in distribution."""
    import torch
    from marl_mass_b200 import rollout
    E = 1024
    env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5,
                                     cbf_eta=0.03125, agent_reward="srew", HIGH_SPEED_REWARD=4, HEADWAY_COST=1,
                                     MERGING_LANE_COST=8), device=0)
    torch.manual_seed(0)
    pol = rollout.BatchedMAPPORollout(env, roll_out_n_steps=12, seed=4)
    l0 = env.kernel_launches()
    buf = pol.collect()
    assert buf["states"].shape == (12, E, mm.MAXV, mm.NS) and buf["returns"].shape == (12, E, mm.MAXV)
    assert bool(torch.isfinite(buf["returns"]).all())
    assert env.kernel_launches() > l0
    stats = pol.update(minibatch=1 << 15)
    assert np.isfinite(stats["actor_loss"]) and np.isfinite(stats["critic_loss"]) and stats["samples"] > 12 * E * 6
    v = env.buffers()
    fa, live = pol.act_fused(v["obs"], v["n_agents"])
    ta, _ = pol.act_torch(v["obs"], v["n_agents"])
    hf = torch.bincount(fa[live].long(), minlength=5).float() / live.sum()
    ht = torch.bincount(ta[live].long(), minlength=5).float() / live.sum()
    assert float((hf - ht).abs().max()) < 0.03
    env.close()


def test_batched_evaluation_equals_the_sequential_protocol(mm, tmp_path):
    """evaluation.evaluation (every evaluation episode as one env of a batch) == MAPPO.evaluation's loop
    (marl/mappo.py:255-361) driven through the single-env adapter, episode by episode, with the same action table."""
    import torch
    from marl_mass_b200 import evaluation as ev
    cfg = dict(safety_guarantee="cbf-cav", traffic_density=2, HEADWAY_TIME=0.5, cbf_eta=0.03125, traffic_type="mixed")
    seeds = [0, 25, 50, 75, 100, 125, 150]
    table = np.random.RandomState(0).randint(0, 5, size=(len(seeds), 100, 12))
    step = {"t": 0}

    def action_fn(obs, n_agents):
        a = torch.from_numpy(table[:, step["t"], :]).cuda()
        step["t"] += 1
        return a

    rewards, (vs, vp), info = ev.evaluation(action_fn, cfg, seeds, is_train=True, output_dir=str(tmp_path))
    # the frames the reference would record as a video (mappo.py:290-327): one after reset + one per policy step
    for i in range(len(seeds)):
        frames = sorted(os.listdir(os.path.join(str(tmp_path), "testing_episode_%d" % i)))
        assert len(frames) == info["steps"][i] + 1 and frames[0] == "frame_000.png"
    with open(os.path.join(str(tmp_path), "testing_episode_0", "frame_000.png"), "rb") as f:
        assert f.read(8) == b"\x89PNG\r\n\x1a\n"
    env = mm.make("merge-multi-agent-v1")
    env.config.update(cfg)
    assert env.render(mode="rgb_array") is not None and env.render(mode="rgb_array").shape == (120, 600, 3)
    min_hw = float("inf")
    for i, s in enumerate(seeds):
        obs, _ = env.reset(is_training=False, testing_seeds=s, num_CAV=ev.eval_num_cav(i, 2))
        n = len(env.controlled_vehicles)
        done, t, rs, sp, tsp = False, 0, [], 0.0, 0.0
        while not done:
            obs, r, done, inf = env.step(tuple(int(x) for x in table[i, t, :n]))
            t += 1
            rs.append(r)
            sp += inf["average_speed"]
            tsp += inf["traffic_speed"]
            min_hw = min(min_hw, inf["min_headway"])
        assert info["steps"][i] == t and np.allclose(rewards[i], rs, rtol=0, atol=0)
        assert abs(info["avg_speeds"][i] - sp / t) < 1e-5 and abs(info["traffic_speeds"][i] - tsp / t) < 1e-5
        assert info["crash_count"][i] == env.is_crashed()
        assert abs(info["merge_percents"][i] - inf["merge_percent"]) < 1e-6
        assert vs[i].shape == (t, n) and np.allclose(vs[i], inf["vehicle_speed"]) and np.allclose(vp[i], inf["vehicle_position"])
    assert abs(info["min_headway"] - min_hw) < 1e-6
    env.close()


def test_batched_evaluation_of_the_idm_baseline(mm):
    """eval_idm.py's protocol (the all-IDM env merge-multi-agent-hdv-v1 on the evaluation seeds) through the same batched
    `evaluation.evaluation`: equals the sequential loop over the adapter."""
    import torch
    from marl_mass_b200 import evaluation as ev
    cfg = dict(env_name="merge-multi-agent-hdv-v1", traffic_type="hdv", safety_guarantee="cbf-cav", traffic_density=3,
               HEADWAY_TIME=0.5, cbf_eta=0.03125)
    seeds = [132, 730, 103, 874, 343]
    idle = lambda obs, n_agents: torch.ones((obs.shape[0], 12), dtype=torch.int8, device="cuda")
    rewards, (vs, vp), info = ev.evaluation(idle, cfg, seeds, is_train=False)
    env = mm.make("merge-multi-agent-hdv-v1", config=cfg)
    for i, s in enumerate(seeds):
        obs, _ = env.reset(is_training=False, testing_seeds=s)
        n = len(env.road.vehicles)
        done, t, rs, sp = False, 0, [], 0.0
        while not done:
            obs, r, done, inf = env.step(())
            t += 1
            rs.append(r)
            sp += inf["average_speed"]
        assert info["steps"][i] == t and np.allclose(rewards[i], rs, rtol=0, atol=0)
        assert abs(info["avg_speeds"][i] - sp / t) < 1e-5 and info["merge_percents"][i] == inf["merge_percent"] == 100.0
        assert info["crash_count"][i] == env.is_crashed() and vs[i].shape == (t, n)
    env.close()


def test_shared_network_rollout_and_training_driver(mm):
    """MAPPO_GI with shared_network = True (the `*-shared*.ini` configs): one ActorCriticNetwork draws the actions and
    bootstraps the returns; one update changes it and re-syncs the target; the ini driver selects it."""
    import torch
    from marl_mass_b200.rollout import BatchedMAPPOGIRollout
    from marl_mass_b200.train import load_ini, train
    torch.manual_seed(0)
    E, T = 1024, 20
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, traffic_type="mixed", HEADWAY_TIME=0.5,
               cbf_eta=0.03125, agent_reward="srew", HIGH_SPEED_REWARD=4, HEADWAY_COST=1, MERGING_LANE_COST=8)
    env = mm.MergeEnvBatched(E, cfg)
    ro = BatchedMAPPOGIRollout(env, roll_out_n_steps=T)
    env.reset(seed=5)
    env.stats(reset=True)
    ro.obs = env.buffers()["obs"]
    b = ro.collect()
    assert b["states"].shape == (T, E, 12, 30) and torch.isfinite(b["returns"]).all()
    assert int(b["live"].sum()) == int(env.stats()["agent_steps"])
    # a rollout that did not end is bootstrapped with V(final state): gamma^k * V enters the last returns
    open_env = (b["dones"][-1] == 0).nonzero(as_tuple=True)[0][0]
    v_fin = ro.policy(ro.obs.view(-1, 30), out_type="v").view(E, 12)[open_env, 0]
    assert torch.allclose(b["returns"][-1, open_env, 0], b["rewards"][-1, open_env, 0] + 0.99 * v_fin, atol=1e-5)
    before = [p.detach().clone() for p in ro.policy.parameters()]
    st = ro.update(minibatch=1 << 15)
    assert st["samples"] == int(b["live"].sum()) and np.isfinite(st["actor_loss"]) and np.isfinite(st["critic_loss"])
    assert all(not torch.equal(a, p) for a, p in zip(before, ro.policy.parameters()))
    assert all(torch.equal(p, q) for p, q in zip(ro.policy.parameters(), ro.policy_target.parameters()))
    env.close()
    ini = os.path.join(ROOT, "examples", "mass_td3_mixed_srew_shared.ini")
    assert load_ini(ini)[2]["shared_network"] is True
    hist = train(ini, n_envs=512, iterations=2, eval_interval=1, log=lambda *_: None)
    assert len(hist) == 2 and np.isfinite(hist[-1]["eval_reward"]) and hist[-1]["agent_steps"] > 0

"""GPU suite: the evaluation protocol on the device - seed-exact scenes spawned by mm_reset_seeded and the episode records
of mm_eval_record - against the host path it replaces (`reset_from_seeds` + `evaluation.evaluation`), bit for bit."""
import os

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

INI = os.path.join(ROOT, "examples", "mass_td3_srew.ini")


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()
    return m


def _configs(mm):
    base = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", HEADWAY_TIME=0.5, cbf_eta=0.03125, traffic_density=3)
    return {
        "mass_td3_cav": dict(base),
        "mass_td3_mixed": dict(base, traffic_type="mixed", action_masking=True),
        "mass_td1": dict(base, traffic_density=1),
        "mass_td3_av": dict(base, traffic_type="av"),
        "hdv_td3": dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-hdv-v1", traffic_type="hdv", traffic_density=3),
        "v0_dmc_td3_mixed": dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-v0", safety_guarantee="dmc", mixed_traffic=True,
                                 traffic_density=3),
        "hss_td3_mixed": dict(base, safety_guarantee="cbf-avs", traffic_type="mixed"),
        "unsafe_td1": dict(mm.DEFAULT_CONFIG, traffic_density=1),
    }


def _test_seeds(n, salt):
    rng = np.random.RandomState(salt)
    edge = np.array([0, 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1], np.int64)
    return np.concatenate([edge, rng.randint(0, 2 ** 32, size=n - len(edge), dtype=np.int64)])


@pytest.mark.parametrize("name", ["mass_td3_cav", "mass_td3_mixed", "mass_td1", "mass_td3_av", "hdv_td3", "v0_dmc_td3_mixed"])
def test_seeded_reset_leaves_the_state_of_the_host_replay(mm, name):
    """reset_from_seeds_device vs reset_from_seeds on 65 536 seeds with the evaluation's num_CAV rule: every field of
    get_state, and the obs / n_agents / action_mask buffers, equal."""
    import torch
    from marl_mass_b200.evaluation import eval_num_cav
    cfg = _configs(mm)[name]
    E = 65536
    seeds = _test_seeds(E, 17)
    num_cav = eval_num_cav(np.arange(E), cfg["traffic_density"])
    host = mm.MergeEnvBatched(E, cfg)
    host.reset_from_seeds(seeds, num_CAV=num_cav)
    dev = mm.MergeEnvBatched(E, cfg)
    dev.reset(seed=99)          # a used handle: every field must be overwritten, the counters left as set_state leaves them
    dev.reset_from_seeds_device(seeds, num_CAV=num_cav)
    torch.cuda.synchronize()
    a, b = host.get_state(), dev.get_state()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    for k in ("obs", "n_agents", "action_mask"):
        assert torch.equal(host.buffers()[k], dev.buffers()[k]), k
    host.close()
    dev.close()


def test_seeded_reset_rejects_bad_seeds_on_a_handle(mm):
    from marl_mass_b200 import _lib
    env = mm.MergeEnvBatched(4, _configs(mm)["mass_td3_mixed"])
    with pytest.raises(_lib.MMError, match=r"\[0, 2\^32\)"):
        env.reset_from_seeds_device([0, 1, 2, 2 ** 32])
    with pytest.raises(_lib.MMError, match="num_CAV"):
        env.reset_from_seeds_device([0, 1, 2, 3], num_CAV=9)
    env.reset_from_seeds_device([0, 1, 2, 3], num_CAV=[1, 2, 3, 4])
    env.close()


class _Actor(object):
    """The fused actor kernel with a fixed network and seed, step = call count: a deterministic action function whose
    draws are keyed by the row, so both protocols see the same actions while they hold the same envs in the same order.
    The 5 x 5 observation of env id v0 is zero-padded to the network's 30 inputs."""

    def __init__(self):
        import torch
        from marl_mass_b200 import rollout
        torch.manual_seed(5)
        self.net, self.rollout, self.calls = rollout.ActorNetwork().cuda(), rollout, 0

    def __call__(self, obs, n_agents):
        import torch
        self.calls += 1
        if obs.shape[-1] != 30:
            obs = torch.nn.functional.pad(obs, (0, 30 - obs.shape[-1]))
        return self.rollout.actor_sample(self.net, obs.contiguous(), n_agents, seed=4242, step=self.calls)


def _assert_same_as_evaluation(mm, cfg, seeds, res, vehicle_records):
    from marl_mass_b200 import evaluation as ev
    rewards, (v_speed, v_pos), info = ev.evaluation(_Actor(), cfg, seeds)
    n = len(rewards)
    assert res["rewards"].shape[0] == n
    assert res["steps"].tolist() == info["steps"]
    for i in range(n):
        s = info["steps"][i]
        assert np.array_equal(res["rewards"][i, :s].astype(np.float64), np.array(rewards[i])), i
        assert not res["rewards"][i, s:].any()
    assert np.array_equal(res["avg_speeds"], np.array(info["avg_speeds"]))
    assert np.array_equal(res["traffic_speeds"], np.array(info["traffic_speeds"]))
    assert res["crashed"].tolist() == info["crash_count"]
    assert np.array_equal(res["merge_percents"], np.array(info["merge_percents"]))
    assert float(res["min_headway"].min()) == info["min_headway"]
    if vehicle_records:
        for i in range(n):
            s, k = info["steps"][i], int(res["n_agents"][i])
            assert np.array_equal(res["vehicle_speed"][i, :s, :k], v_speed[i]), i
            assert np.array_equal(res["vehicle_position"][i, :s, :k], v_pos[i]), i


@pytest.mark.parametrize("name", ["mass_td3_srew", "hss_td3_mixed", "unsafe_td1", "v0_dmc_td3_mixed"])
def test_evaluate_seeds_equals_evaluation(mm, name):
    """Every per-step reward, steps, average / traffic speeds, crash flags, merge percents and min headway equal to
    `evaluation` on the example ini's 20 test seeds (with the vehicle speed / position records) and on 1 024 seeds; the
    dmc config checks that the supervisor draws are keyed as after set_state."""
    from marl_mass_b200 import evaluation as ev
    from marl_mass_b200.train import load_ini
    env_cfg, _, tr = load_ini(INI)
    cfg = dict(mm.DEFAULT_CONFIG, **env_cfg) if name == "mass_td3_srew" else _configs(mm)[name]
    seeds20 = [int(s) for s in tr["test_seeds"].split(",")][:tr["eval_episodes"]]
    for seeds, vehicle_records in ((seeds20, True), (list(range(1024)), False)):
        res = ev.evaluate_seeds(_Actor(), cfg, seeds, vehicle_records=vehicle_records)
        _assert_same_as_evaluation(mm, cfg, seeds, res, vehicle_records)
        k = int(res["crashed"].sum())
        lo, hi = res["crash_rate_ci95"]
        assert res["crash_rate"] == k / len(seeds) and 0.0 <= lo <= res["crash_rate"] <= hi <= 1.0


def _obs_action(obs, n_agents):
    """A deterministic function of each observation row alone: the actions do not depend on where an env sits in a batch."""
    import torch
    key = torch.floor((obs[..., 1] * 997.0 + obs[..., 3] * 991.0 + obs[..., 8] * 983.0) * 1000.0)
    return torch.remainder(key, 5.0).to(torch.int8)


def test_evaluate_seeds_is_independent_of_the_batch_size(mm):
    from marl_mass_b200 import evaluation as ev
    cfg = _configs(mm)["mass_td3_mixed"]
    batch = 256
    N = 2 * batch + 77
    seeds = _test_seeds(N, 3)
    whole = ev.evaluate_seeds(_obs_action, cfg, seeds, vehicle_records=True)
    assert len(set(whole["steps"].tolist())) > 1        # episodes of different lengths: crashes end some early
    for b in (batch, 100, 1):
        part = ev.evaluate_seeds(_obs_action, cfg, seeds, vehicle_records=True, batch=b)
        for k, v in whole.items():
            if isinstance(v, np.ndarray):
                assert np.array_equal(v, part[k]), (b, k)
            else:
                assert v == part[k], (b, k)
    one = ev.evaluate_seeds(_obs_action, cfg, seeds[:1], vehicle_records=True)      # episode 0: the same num_CAV
    for k in ("rewards", "steps", "avg_speeds", "traffic_speeds", "crashed", "merge_percents", "min_headway", "vehicle_speed",
              "vehicle_position"):
        assert np.array_equal(one[k][0], whole[k][0]), k


def test_training_driver_logs_the_device_evaluation(mm):
    from marl_mass_b200.train import train
    base_keys = None
    for eval_seeds in (0, 256):
        hist = train(INI, n_envs=512, iterations=1, eval_interval=1, log=lambda *_: None, eval_seeds=eval_seeds)
        rec = hist[-1]
        if eval_seeds == 0:
            base_keys = set(rec)
            assert not any(k.startswith("evalN_") for k in rec)
            continue
        new = set(rec) - base_keys
        assert new == {"evalN_episodes", "evalN_crash_rate", "evalN_crash_rate_ci95", "evalN_reward", "evalN_avg_speed",
                       "evalN_merge_percent", "evalN_min_headway", "evalN_s"}
        assert rec["evalN_episodes"] == 256 and 0.0 <= rec["evalN_crash_rate"] <= 1.0
        lo, hi = rec["evalN_crash_rate_ci95"]
        assert lo <= rec["evalN_crash_rate"] <= hi and np.isfinite(rec["evalN_reward"]) and rec["evalN_s"] > 0

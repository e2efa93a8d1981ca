"""GPU suite: the evaluation's shield records and control profiles (mm_eval_shield_record, evaluate_seeds(shield_records,
control_profiles)) against a numpy reduction of the per-step diagnostic record on the host, against the single-env
adapter's state_hist / action_hist, and against evaluate_seeds without them."""
import os

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

INI = os.path.join(ROOT, "examples", "mass_td3_srew.ini")
COUNTS = ("shield_solves", "shield_active", "lane_change_vetoes", "shield_interventions")
F64 = ("acc_correction_sum", "acc_correction_max", "steer_correction_max", "min_agent_acc")


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
        "hss_td3_mixed": dict(base, safety_guarantee="cbf-avs", traffic_type="mixed"),
        "mass_td3_av": dict(base, traffic_type="av"),
        "mass_steervel_td2": dict(base, lateral_control="steer_vel", traffic_density=2),
        "v0_dmc_td3_mixed": dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-v0", safety_guarantee="dmc", mixed_traffic=True,
                                 traffic_density=3),
        "unsafe_td1": dict(mm.DEFAULT_CONFIG, traffic_density=1),
        "hdv_td3": dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-hdv-v1", traffic_type="hdv", traffic_density=3),
    }


UNSHIELDED = ("v0_dmc_td3_mixed", "unsafe_td1", "hdv_td3")


def _test_seeds(n, salt):
    rng = np.random.RandomState(salt)
    edge = np.array([0, 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1], np.int64)
    return np.concatenate([edge, rng.randint(0, 2 ** 32, size=n - len(edge), dtype=np.int64)])


class _Table(object):
    """Actions from a fixed table [N, T, 12] keyed by the global episode index: the k-th call is policy step k % T of the
    batch k // T, whose envs are the episodes batch * (k // T) + row.  Slots at or above n_agents get 1 (IDLE), as the
    single-env adapter fills them."""

    def __init__(self, n, T, batch, salt):
        import torch
        rng = np.random.RandomState(salt)
        self.table = torch.from_numpy(rng.randint(0, 5, size=(n, T, 12)).astype(np.int8)).cuda()
        self.T, self.batch, self.calls = T, batch, 0

    def __call__(self, obs, n_agents):
        import torch
        b, t = divmod(self.calls, self.T)
        self.calls += 1
        rows = self.batch * b + torch.arange(obs.shape[0], device=obs.device)
        a = self.table[rows, t].clone()
        a[torch.arange(12, device=obs.device)[None, :] >= n_agents[:, None]] = 1
        return a


def _T(mm, cfg):
    env = mm.MergeEnvBatched(1, cfg)
    T = env.T
    env.close()
    return T


def _host_reduction(mm, cfg, seeds, act, profiles, T):
    """The records from the diagnostic record copied to the host after every step (shield_diag), reduced in numpy in the
    documented order (sub-step, then slot), each env stopped after its first done."""
    import torch
    from marl_mass_b200.evaluation import eval_num_cav
    E = len(seeds)
    env = mm.MergeEnvBatched(E, cfg, record_diag=True)
    env.reset_from_seeds(seeds, num_CAV=eval_num_cav(np.arange(E), env.config["traffic_density"]))
    v = env.buffers()
    n_agents = v["n_agents"].clone()
    n_host = n_agents.cpu().numpy()
    active = np.ones(E, bool)
    r = {k: np.zeros(E, np.int64) for k in COUNTS}
    r.update({k: np.zeros(E) for k in F64})
    r["min_agent_acc"][:] = np.inf
    from marl_mass_b200._lib import PROFILE_F, PROFILE_I
    prof = {k: np.zeros((len(profiles), 3 * T, 12), np.int32) for k in PROFILE_I}
    prof.update({k: np.zeros((len(profiles), 3 * T, 12)) for k in PROFILE_F})
    for t in range(T):
        env.step(act(env.obs_view(), n_agents).to(torch.int8))
        torch.cuda.synchronize()
        d = env.shield_diag()
        done = v["done"].cpu().numpy().astype(bool)
        for s in range(3):
            for i in range(12):
                ran = active & (d["ran"][:, s, i] != 0)
                sa, na = d["safe_acc"][:, s, i], d["nom_acc"][:, s, i]
                ss, ns = d["safe_steer"][:, s, i], d["nom_steer"][:, s, i]
                r["shield_solves"] += ran
                r["shield_active"] += ran & (d["active"][:, s, i] != 0)
                r["lane_change_vetoes"] += ran & (d["is_lc_safe"][:, s, i] == 0)
                r["shield_interventions"] += ran & ((sa != na) | (ss != ns))
                da, ds = np.abs(sa - na), np.abs(ss - ns)
                r["acc_correction_sum"] = np.where(ran, r["acc_correction_sum"] + da, r["acc_correction_sum"])
                r["acc_correction_max"] = np.where(ran & (da > r["acc_correction_max"]), da, r["acc_correction_max"])
                r["steer_correction_max"] = np.where(ran & (ds > r["steer_correction_max"]), ds, r["steer_correction_max"])
                mv = active & (d["moved"][:, s, i] != 0) & (i < n_host)
                r["min_agent_acc"] = np.where(mv & (sa < r["min_agent_acc"]), sa, r["min_agent_acc"])
        for k, e in enumerate(profiles):
            if active[e]:
                for f in prof:
                    prof[f][k, 3 * t:3 * t + 3] = d[f][e]
        active &= ~done
    assert not active.any()
    env.close()
    return r, prof


@pytest.mark.parametrize("name", ["mass_td3_cav", "hss_td3_mixed", "mass_td3_av", "mass_steervel_td2", "v0_dmc_td3_mixed",
                                  "unsafe_td1", "hdv_td3"])
def test_shield_records_equal_the_host_reduction(mm, name):
    """4 096 seeds: every counter and f64 record bit for bit, and the control profiles of 64 episodes (every crashed
    episode first, up to 32) element for element, against the host reduction with the same action table."""
    from marl_mass_b200 import evaluation as ev
    cfg = _configs(mm)[name]
    N = 4096
    seeds = _test_seeds(N, 29)
    T = _T(mm, cfg)
    first = ev.evaluate_seeds(_Table(N, T, N, 7), cfg, seeds, shield_records=True)
    crashed = np.nonzero(first["crashed"])[0][:32]
    rest = np.setdiff1d(np.arange(N), crashed)
    profiles = np.concatenate([crashed, np.random.RandomState(3).choice(rest, 64 - len(crashed), replace=False)])
    res = ev.evaluate_seeds(_Table(N, T, N, 7), cfg, seeds, shield_records=True, control_profiles=profiles)
    for k in COUNTS + F64:
        assert np.array_equal(res[k], first[k]), k            # the profiles change nothing
    want, want_prof = _host_reduction(mm, cfg, seeds, _Table(N, T, N, 7), profiles, T)
    for k in COUNTS:
        assert res[k].dtype == np.int64 and np.array_equal(res[k], want[k]), k
    for k in F64:
        assert res[k].dtype == np.float64 and np.array_equal(res[k], want[k]), k
    assert np.array_equal(res["control_profile_episodes"], profiles)
    for f, v in want_prof.items():
        assert res["control_profiles"][f].shape == (64, 3 * T, 12) and np.array_equal(res["control_profiles"][f], v), f
    solves = int(res["shield_solves"].sum())
    assert res["intervention_rate"] == (int(res["shield_interventions"].sum()) / solves if solves else 0.0)
    if name in UNSHIELDED:
        for k in COUNTS:
            assert not res[k].any(), k
        assert res["intervention_rate"] == 0.0
    else:
        assert solves > 0 and res["shield_interventions"].sum() > 0
    has_agents = res["n_agents"] > 0
    assert np.isfinite(res["min_agent_acc"][has_agents]).all() and np.isinf(res["min_agent_acc"][~has_agents]).all()
    if name == "unsafe_td1":
        assert len(crashed) > 0


def _profile_rows(res, k, i):
    """Rows of profile k where vehicle slot i moved, in order: one state_hist / action_hist entry each."""
    p = res["control_profiles"]
    return [r for r in range(p["moved"].shape[1]) if p["moved"][k, r, i]]


@pytest.mark.parametrize("name", ["mass_td3_cav", "hss_td3_mixed"])
def test_profiles_equal_the_adapters_state_and_action_history(mm, name):
    """8 seeds replayed through make(..., store_profile=True) with the same action table: every vehicle's state_hist /
    action_hist entry equals its profile row bit for bit."""
    from marl_mass_b200 import evaluation as ev
    cfg = _configs(mm)[name]
    seeds = _test_seeds(8, 41)
    T = _T(mm, cfg)
    table = _Table(8, T, 8, 11)
    res = ev.evaluate_seeds(table, cfg, seeds, control_profiles=range(8))
    tab = table.table.cpu().numpy()
    p = res["control_profiles"]
    checked = 0
    for k, seed in enumerate(seeds):
        env = mm.make(cfg.get("env_name", "merge-multi-agent-v1"), config=dict(cfg, store_profile=True))
        env.reset(is_training=False, testing_seeds=int(seed), num_CAV=ev.eval_num_cav(k, cfg["traffic_density"]))
        n = len(env.controlled_vehicles)
        for t in range(T):
            _, _, done, _ = env.step(tuple(int(x) for x in tab[k, t, :n]))
            if done:
                break
        assert done and t + 1 == res["steps"][k]
        for v in env.road.vehicles:
            i = v._slot
            rows = _profile_rows(res, k, i)
            assert len(rows) == len(v.state_hist) == len(v.action_hist) > 0
            for row, st, ac in zip(rows, v.state_hist, v.action_hist):
                for f, key in (("x", "x"), ("y", "y"), ("heading", "heading"), ("speed", "speed"), ("headway", "min_headway"),
                               ("steering_angle", "nom_steer")):
                    assert st[f] == p[key][k, row, i], (k, i, row, f)
                for f, key in (("acceleration", "safe_acc"), ("steering", "safe_steer"), ("ull_acceleration", "nom_acc"),
                               ("ull_steering", "nom_steer")):
                    assert ac[f] == p[key][k, row, i], (k, i, row, f)
                hl = int(p["hl_action"][k, row, i])
                assert ac["lc_action"] == (hl if hl >= 0 else None)
                if p["ran"][k, row, i]:
                    assert ac["safe_diff"] == {"acceleration": p["safe_acc"][k, row, i] - p["nom_acc"][k, row, i],
                                               "steering": p["safe_steer"][k, row, i] - p["nom_steer"][k, row, i]}
                    assert st["safe_status"] == {"active_set": int(p["active"][k, row, i]),
                                                 "is_lc_safe": bool(p["is_lc_safe"][k, row, i])}
                    checked += 1
                else:
                    assert "safe_diff" not in ac and "safe_status" not in st
            assert not p["moved"][k, 3 * int(res["steps"][k]):, i].any()
        env.close()
    assert checked > 0


@pytest.mark.parametrize("name", ["mass_td3_cav", "mass_td3_mixed"])
def test_records_change_no_existing_key(mm, name):
    """65 536 seeds with the records on and off: every key evaluate_seeds returns without them is identical."""
    from marl_mass_b200 import evaluation as ev
    cfg = _configs(mm)[name]
    N = 65536
    seeds = _test_seeds(N, 5)
    T = _T(mm, cfg)
    off = ev.evaluate_seeds(_Table(N, T, N, 13), cfg, seeds, vehicle_records=True)
    on = ev.evaluate_seeds(_Table(N, T, N, 13), cfg, seeds, vehicle_records=True, shield_records=True,
                           control_profiles=[0, 7, N - 1])
    assert set(on) - set(off) == {"shield_solves", "shield_active", "shield_interventions", "lane_change_vetoes",
                                  "acc_correction_sum", "acc_correction_max", "steer_correction_max", "min_agent_acc",
                                  "intervention_rate", "control_profiles", "control_profile_episodes"}
    for k, v in off.items():
        if isinstance(v, np.ndarray):
            assert v.dtype == on[k].dtype and np.array_equal(v, on[k]), k
        else:
            assert v == on[k], k


def test_records_are_independent_of_the_batch_size(mm):
    from marl_mass_b200 import evaluation as ev
    cfg = _configs(mm)["mass_td3_mixed"]
    N = 4096
    seeds = _test_seeds(N, 8)
    T = _T(mm, cfg)
    profiles = [0, 1364, 1365, 2730, 4095, 17]
    whole = ev.evaluate_seeds(_Table(N, T, N, 19), cfg, seeds, shield_records=True, control_profiles=profiles)
    part = ev.evaluate_seeds(_Table(N, T, N // 3, 19), cfg, seeds, shield_records=True, control_profiles=profiles,
                             batch=N // 3)
    for k in COUNTS + F64 + ("steps", "crashed"):
        assert np.array_equal(whole[k], part[k]), k
    assert whole["intervention_rate"] == part["intervention_rate"]
    for f, v in whole["control_profiles"].items():
        assert np.array_equal(v, part["control_profiles"][f]), f


def test_a_handle_without_record_diag_is_refused(mm):
    import torch
    from marl_mass_b200 import _lib
    E = 64
    env = mm.MergeEnvBatched(E, _configs(mm)["mass_td3_cav"])
    env.reset_from_seeds_device(np.arange(E))
    t = {k: torch.zeros(E, dtype=torch.int32, device="cuda") for k in ("n_agents",) + COUNTS}
    t.update({k: torch.zeros(E, dtype=torch.float64, device="cuda") for k in F64})
    t["active"] = torch.ones(E, dtype=torch.uint8, device="cuda")
    rec = _lib.MMEvalShieldRecords(T=env.T, **{k: v.data_ptr() for k, v in t.items()})
    with pytest.raises(_lib.MMError, match=r"without record_diag \(status -3\)"):
        env.eval_shield_record(rec, 0)
    env.close()


def test_training_driver_logs_the_shield_records(mm):
    from marl_mass_b200.train import train
    base = train(INI, n_envs=512, iterations=2, eval_interval=1, log=lambda *_: None, eval_seeds=4096)
    hist = train(INI, n_envs=512, iterations=2, eval_interval=1, log=lambda *_: None, eval_seeds=4096, eval_shield=True)
    new = {"evalN_shield_intervention_rate", "evalN_lane_change_vetoes_per_episode", "evalN_min_agent_acc",
           "evalN_acc_correction_max"}
    for b, rec in zip(base, hist):
        assert set(rec) - set(b) == new and set(b) <= set(rec)
        assert not any(k.startswith("evalN_shield") for k in b)
        for k in new:
            assert np.isfinite(rec[k]), k
        assert 0.0 <= rec["evalN_shield_intervention_rate"] <= 1.0 and rec["evalN_acc_correction_max"] >= 0.0

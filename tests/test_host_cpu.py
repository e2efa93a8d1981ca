"""CPU suite, part 2: host logic and the C-ABI surface (no compute calls: there is no GPU here)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN_CASES, ROOT, V0_CASES
from helpers import load_golden

# a checkout of the reference project (hkbharath/MARL-MASS), for the tests that read its shipped configs
REFERENCE_ROOT = os.environ.get("MM_REFERENCE_ROOT", "")


def test_library_builds_loads_and_exports_every_declared_symbol():
    import marl_mass_b200 as mm
    from marl_mass_b200 import build
    build.build()
    L = mm.lib()
    header = open(os.path.join(ROOT, "include", "marl_mass_b200.h")).read()
    declared = set(re.findall(r"\b(mm_[a-z_]+)\s*\(", header))
    assert {"mm_create", "mm_step", "mm_step_host", "mm_reset", "mm_shield_qp", "mm_get_state"} <= declared
    for name in declared:
        assert hasattr(L, name), "declared in include/marl_mass_b200.h but not exported: " + name
    assert b"sm_100a" in L.mm_version()


def test_mm_config_layout_agrees_between_header_binding_and_integration_stub():
    """ABI drift guard: the mm_config struct of the header, the ctypes Structure of the product binding and the stub
    INTEGRATION.md shows a reference maintainer must list the same fields in the same order with the same types; the
    three copies of MM_ABI_VERSION agree; and the library refuses a config whose struct_size is not its own
    (validation happens before any CUDA call, so this runs without a GPU)."""
    import marl_mass_b200 as mm
    from marl_mass_b200 import _lib
    header = open(os.path.join(ROOT, "include", "marl_mass_b200.h")).read()
    body = re.search(r"typedef struct \{((?:(?!typedef struct).)*?)\} mm_config;", header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    ctype = {"int32_t": ctypes.c_int32, "double": ctypes.c_double}
    declared = []
    for typ, names in re.findall(r"\b(int32_t|double)\s+([^;]+);", body):
        declared += [(n.strip(), ctype[typ]) for n in names.split(",")]
    assert declared[0][0] == "struct_size" and declared[-1][0] == "supervisor" and len(declared) == 20
    assert [(n, t) for n, t in _lib.MMConfig._fields_] == declared
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    stub = re.search(r"class MMConfig\(C\.Structure\):.*?_fields_ = \[(.*?)\]\n", doc, re.S).group(1)
    stub_fields = [(n, getattr(ctypes, t)) for n, t in re.findall(r'\("(\w+)", C\.(c_\w+)\)', stub)]
    assert stub_fields == declared
    version = int(re.search(r"#define MM_ABI_VERSION (\d+)", header).group(1))
    L = mm.lib()
    assert L.mm_abi_version() == version == _lib.ABI_VERSION
    assert "mm_abi_version() == %d" % version in doc
    good = mm.make_mm_config(dict(mm.DEFAULT_CONFIG))
    assert good.struct_size == ctypes.sizeof(_lib.MMConfig)
    bad = mm.make_mm_config(dict(mm.DEFAULT_CONFIG))
    bad.struct_size -= 4          # e.g. a binding written before env_hdv was appended
    h = ctypes.c_void_p()
    assert L.mm_create(ctypes.byref(bad), 16, 0, 0, ctypes.byref(h)) == -1 and not h
    assert b"struct_size" in L.mm_last_error()


def test_shared_object_is_sm100a_only():
    from marl_mass_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out and "sm_90" not in out and "sm_80" not in out


def test_missing_library_fails_loudly(monkeypatch):
    from marl_mass_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libmarl_mass_b200.so")
    with pytest.raises(_lib.MMError, match="no CPU fallback"):
        _lib.lib()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "marl-mass_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), os.path.join(dirpath, f)


def test_config_mapping_and_error_behaviour():
    import marl_mass_b200 as mm
    c = mm.make_mm_config(dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", HEADWAY_TIME=0.5, cbf_eta=0.03125,
                               traffic_density=3, traffic_type="mixed", agent_reward="srew"))
    assert (c.shield, c.reward_kind, c.traffic_density, c.traffic_type) == (2, 1, 3, 1)
    assert c.duration_steps == 100 and c.substeps == 3 and c.dt == 1 / 15 and c.tau == 0.5 and c.eta == 0.03125
    for sg in ("cbf-avs_cint", "cbf-avs", "cbf-av", "cbf-hss"):
        assert mm.make_mm_config(dict(mm.DEFAULT_CONFIG, safety_guarantee=sg)).shield == 1
    with pytest.raises(ValueError, match="Undefined safety_type"):   # decentral_layer.py:817
        mm.make_mm_config(dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-foo"))
    with pytest.raises(AttributeError, match="Lateral control"):     # safe_controller.py:173-176
        mm.make_mm_config(dict(mm.DEFAULT_CONFIG, lateral_control="torque"))
    assert mm.make_mm_config(dict(mm.DEFAULT_CONFIG, lateral_control="steer_vel")).steer_vel == 1
    for sg, code in (("priority", 1), ("dmc", 2)):      # abstract.py:459-464: supervisors on the action tuple, vehicles un-shielded
        c = mm.make_mm_config(dict(mm.DEFAULT_CONFIG, safety_guarantee=sg, env_name="merge-multi-agent-v0"))
        assert (c.shield, c.supervisor, c.env_v0) == (0, code, 1)
    assert mm.make_mm_config(dict(mm.DEFAULT_CONFIG, safety_guarantee="priority")).supervisor == 1    # env v1 as well
    assert mm.make_mm_config(dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav")).supervisor == 0
    with pytest.raises(KeyError):
        mm.make("merge-v1")


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_seed_exact_spawn_matches_reference_reset(name):
    """Host replay of the reference's MT19937 draw order: reset(testing_seeds=s) builds the same scene."""
    import marl_mass_b200 as mm
    from marl_mass_b200 import _lib
    g, cfg = load_golden(name)
    st = mm.spawn.spawn_state(cfg["seeds"], cfg["traffic_density"], cfg["traffic_type"])
    rows = g["ep_start"][:-1]
    assert "steering_angle" in _lib.F64_FIELDS
    for k in _lib.F64_FIELDS + _lib.I32_FIELDS + _lib.ENV_FIELDS:
        assert np.array_equal(g["st_" + k][rows], st[k]), k


@pytest.mark.parametrize("name", V0_CASES)
def test_seed_exact_spawn_v0_env(name):
    import marl_mass_b200 as mm
    from marl_mass_b200.env import traffic_type_of
    g, cfg = load_golden(name)
    st = mm.spawn.spawn_state(cfg["seeds"], cfg["traffic_density"], traffic_type_of(cfg))
    rows = g["ep_start"][:-1]
    for k in ("x", "y", "speed", "target_speed", "timer", "lane", "target_lane", "n_veh", "n_cav", "n_merge"):
        assert np.array_equal(g["st_" + k][rows], st[k]), k
    assert np.array_equal(np.where(g["st_kind"][rows] == 3, 1, np.where(g["st_kind"][rows] == 4, 2, 0)), st["kind"])


def test_spawn_num_cav_override_and_ranges():
    import marl_mass_b200 as mm
    for seed in range(40):
        v, n_merge = mm.spawn.spawn_scene(seed, 3, "mixed", num_CAV=5)
        kinds = [k for k, *_ in v]
        assert kinds.count(1) == 5 and 3 <= kinds.count(2) <= 5 and kinds == sorted(kinds)
        assert n_merge == 5 - 5 // 2
        xs = [x for _, x, _, _ in v]
        assert len(set(np.round(xs, 9))) == len(xs) and all(1 <= x <= 264 for x in xs)
    with pytest.raises(ValueError):
        mm.spawn.spawn_scene(0, 1, "trucks")


def test_seed_exact_spawn_and_config_of_the_hdv_env():
    import marl_mass_b200 as mm
    g, cfg = load_golden("hdv_td3")
    st = mm.spawn.spawn_state(cfg["seeds"], cfg["traffic_density"], cfg["traffic_type"])
    rows = g["ep_start"][:-1]
    for k in ("x", "y", "speed", "target_speed", "timer", "kind", "lane", "target_lane", "n_veh", "n_cav", "n_merge"):
        assert np.array_equal(g["st_" + k][rows], st[k]), k
    assert (st["n_cav"] == 0).all() and (st["n_merge"] == 0).all() and (st["kind"][st["x"] != 0] == 2).all()
    c = mm.make_mm_config(dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-hdv-v1", traffic_type="hdv", traffic_density=3))
    assert c.env_hdv == 1 and c.traffic_type == 3
    for bad in (dict(env_name="merge-multi-agent-hdv-v1", traffic_type="mixed"), dict(env_name="merge-multi-agent-v1", traffic_type="hdv")):
        with pytest.raises(ValueError, match="go together"):
            mm.make_mm_config(dict(mm.DEFAULT_CONFIG, **bad))


def test_shard_ranges_cover_the_env_axis():
    from marl_mass_b200 import dist
    for total, world in ((1 << 20, 8), (65536, 4), (1000, 3), (5, 8)):
        spans = [dist.shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [e - b for b, e in spans]
        assert max(sizes) - min(sizes) <= 1
    assert len({dist.rank_seed(7, r) for r in range(8)}) == 8


_WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from marl_mass_b200 import dist as mmd
rank = int(os.environ["RANK"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=rank, world_size=2)
stats = {k: float(rank + 1) for k in mmd.SUM_KEYS}
stats["min_headway"] = 0.75 - 0.25 * rank
tot = mmd.all_reduce_stats(stats)
assert all(tot[k] == 3.0 for k in mmd.SUM_KEYS), tot
assert tot["min_headway"] == 0.5, tot
b, e = mmd.shard_range(65536 * 2, rank, 2)
assert e - b == 65536 and b == rank * 65536
s = mmd.summarize(tot)
assert s["crash_rate"] == 1.0 and s["shield_active_frac"] == 1.0
# the learner's data parallelism (rollout.py): parameters broadcast from rank 0, gradients averaged over the ranks
import torch
from marl_mass_b200.rollout import ActorCriticNetwork, BatchedMAPPOGIRollout
torch.manual_seed(100 + rank)
ro = BatchedMAPPOGIRollout.__new__(BatchedMAPPOGIRollout)
ro.policy, ro.policy_target = ActorCriticNetwork(), ActorCriticNetwork()
ro.sync_parameters()
flat = torch.cat([q.detach().reshape(-1) for m in ro.networks() for q in m.parameters()])
both = [torch.zeros_like(flat) for _ in range(2)]
dist.all_gather(both, flat)
assert torch.equal(both[0], both[1])
x = torch.randn(16, 30)
ro.policy(x).sum().backward()
params = [q for q in ro.policy.parameters() if q.grad is not None]
mine = torch.cat([q.grad.reshape(-1) for q in params]).clone()
grads = [torch.zeros_like(mine) for _ in range(2)]
dist.all_gather(grads, mine)
assert not torch.equal(grads[0], grads[1])
ro._allreduce_grads(params)
after = torch.cat([q.grad.reshape(-1) for q in params])
assert torch.allclose(after, (grads[0] + grads[1]) / 2, atol=1e-7)
dist.destroy_process_group()
print("ok", rank)
"""


def test_stats_all_reduce_world_size_2_gloo(tmp_path):
    """The only collective on the path (SURVEY.md §8e): SUM of the counters, MIN of min_headway; and the learner's
    parameter broadcast + gradient averaging over the ranks."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port],
                              env=dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1"),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and ("ok %d" % r) in o, o


def test_discounted_returns_match_reference_formula():
    """The episode-segment semantics of the rollout's returns (oracle.mappo_discount, the checker of the CUDA kernel in
    tests/test_gpu_caller.py) == MAPPO._discount_reward (marl/mappo.py:364-370) run per episode segment."""
    import torch
    import oracle
    from marl_mass_b200.rollout import ActorNetwork, CriticNetwork
    rng = np.random.RandomState(0)
    T, N, gamma = 37, 5, 0.99
    r = rng.randn(T, N)
    d = (rng.rand(T, N) < 0.1).astype(np.float64)
    fv = rng.randn(N)
    got = oracle.mappo_discount(r, d, fv, gamma)
    for n in range(N):
        start = 0
        ends = list(np.where(d[:, n] > 0)[0]) + ([T - 1] if d[T - 1, n] == 0 else [])
        for end in ends:
            seg = r[start:end + 1, n]
            running = 0.0 if d[end, n] > 0 else fv[n]
            want = np.zeros_like(seg)
            for t in reversed(range(len(seg))):        # the reference loop
                running = running * gamma + seg[t]
                want[t] = running
            assert np.allclose(got[start:end + 1, n], want, rtol=0, atol=1e-12)
            start = end + 1
    a, c = ActorNetwork(), CriticNetwork()
    x = torch.randn(7, 30)
    lp = a(x)
    assert lp.shape == (7, 5) and torch.allclose(lp.exp().sum(1), torch.ones(7), atol=1e-6)
    assert c(x, torch.nn.functional.one_hot(torch.arange(7) % 5, 5).float()).shape == (7, 1)
    assert sum(p.numel() for p in a.parameters()) == 30 * 128 + 128 + 128 * 128 + 128 + 128 * 5 + 5


def test_shipped_ini_files_map_onto_the_batched_path():
    """Every shipped marl/configs/*.ini resolves to an mm_config - the 8 look-ahead baseline configs (priority / dmc)
    included, as a supervisor on the action tuple.  Needs a checkout of the reference project, named by
    MM_REFERENCE_ROOT; skipped without one."""
    import configparser
    import glob
    import marl_mass_b200 as mm
    cfg_dir = os.path.join(REFERENCE_ROOT, "marl", "configs")
    if not REFERENCE_ROOT or not os.path.isdir(cfg_dir):
        pytest.skip("reference project not present (set MM_REFERENCE_ROOT)")
    ok, rejected = [], {}
    for f in sorted(glob.glob(os.path.join(cfg_dir, "*.ini"))):
        c = configparser.ConfigParser()
        c.read(f)
        e = c["ENV_CONFIG"]
        cfg = dict(mm.DEFAULT_CONFIG, env_name=e.get("env_name", "merge-multi-agent-v0"),      # run_mappo.py:142
                   safety_guarantee=e.get("safety_guarantee"), lateral_control=e.get("lateral_control", "steer"),
                   mixed_traffic=c.getboolean("ENV_CONFIG", "mixed_traffic", fallback=None),
                   traffic_type=e.get("traffic_type", "cav"), agent_reward=e.get("agent_reward", "default"),
                   traffic_density=int(e["traffic_density"]), HEADWAY_TIME=float(e["HEADWAY_TIME"]),
                   cbf_eta=float(e.get("cbf_eta", 0)),
                   action_masking=c.getboolean("MODEL_CONFIG", "action_masking", fallback=False))
        try:
            mm.make_mm_config(cfg)
            ok.append(os.path.basename(f))
        except (ValueError, KeyError, AttributeError) as ex:
            rejected[os.path.basename(f)] = str(ex)
    assert len(ok) == 37 and not rejected, rejected
    assert "test-idm-td3.ini" in ok
    for must in ("marl_cav-heading-t_headway-cbf-cav.ini", "marl_cav-heading-t_headway-cbf-avs_cint.ini",
                 "marl_cav-heading-t_headway-cbf-cav-td3-srew.ini", "marl_cav-heading-t_headway-cbf-cav-mixed.ini",
                 "test-configs_marl-cav-unsafe.ini", "marl_cav_heading-t_headway-cbf-av-steer_vel.ini"):
        assert must in ok


def test_training_driver_rejects_env_ids_it_does_not_cover():
    """The batched learner's networks take the 30-column KinematicLC state; the n_s = 25 env ids (v0, v05) and the all-HDV
    env are refused before anything is built (no GPU needed to find out)."""
    from marl_mass_b200 import train as tr
    for env_name in ("merge-multi-agent-v0", "merge-multi-agent-v05", "merge-multi-agent-hdv-v1"):
        cfg = ({"env_name": env_name, "seed": 0}, {}, {"torch_seed": 0})
        with pytest.raises(ValueError, match="not covered by the batched learner"):
            tr.train(cfg, n_envs=8, iterations=1)


def test_training_driver_reads_the_reference_ini_layout():
    """train.load_ini: the sections / keys / fallbacks of run_mappo.py:113-171, on the shipped example and (when the
    reference tree is present) on the reference's own MASS td3 srew ini - both must give the same configuration."""
    from marl_mass_b200 import train
    import marl_mass_b200 as mm
    env_cfg, kw, tr = train.load_ini(os.path.join(ROOT, "examples", "mass_td3_srew.ini"))
    assert env_cfg["safety_guarantee"] == "cbf-cav" and env_cfg["traffic_density"] == 3 and env_cfg["mixed_traffic"] is False
    assert env_cfg["agent_reward"] == "srew" and env_cfg["cbf_eta"] == 0.03125 and env_cfg["HEADWAY_TIME"] == 0.5
    assert kw == {"roll_out_n_steps": 100, "reward_gamma": 0.99, "max_grad_norm": 5.0, "reward_type": "regionalR",
                  "reward_scale": 20.0, "actor_lr": 5e-4, "critic_lr": 5e-4}
    assert len(tr["test_seeds"].split(",")) == 20 and tr["eval_episodes"] == 20
    c = mm.make_mm_config(dict(mm.DEFAULT_CONFIG, **env_cfg))
    assert (c.shield, c.reward_kind, c.traffic_type) == (2, 1, 0)
    ref = os.path.join(REFERENCE_ROOT, "marl", "configs", "marl_cav-heading-t_headway-cbf-cav-td3-srew.ini")
    if REFERENCE_ROOT and os.path.exists(ref):
        env_ref, kw_ref, tr_ref = train.load_ini(ref)
        assert env_ref == env_cfg and kw_ref == kw and tr_ref["test_seeds"] == tr["test_seeds"]


def test_render_scene_from_state():
    """CPU renderer that replaces the pygame viewer (abstract.py:512-556): frame shape of the reference's surface,
    vehicles drawn where the state puts them, in the reference's colours."""
    import marl_mass_b200 as mm
    from marl_mass_b200 import render
    st = mm.spawn.spawn_state([3], 3, "mixed")
    n = int(st["n_veh"][0])
    st["x"][0, :n] = np.linspace(260, 440, n)          # inside the window [250, 450] x [-16, 24]
    st["y"][0, :n] = np.where(st["kind"][0, :n] == 1, 0.0, 4.0)
    st["heading"][0, :n] = 0.0
    st["crashed"][0, 0] = 1
    img = render.render_scene(st, 0, dict(mm.DEFAULT_CONFIG))
    assert img.shape == (120, 600, 3) and img.dtype == np.uint8
    px = lambda x, y: img[int((y + 16) * 3), int((x - 250) * 3)]
    assert tuple(px(st["x"][0, 0], st["y"][0, 0])) == render.RED
    for i in range(1, n):
        want = render.GREEN if st["kind"][0, i] == 1 else render.BLUE
        assert tuple(px(st["x"][0, i], st["y"][0, i])) == want, i
    assert tuple(px(300.0, 14.0)) == render.GREY and tuple(px(420.0, 4.0)) == render.OBSTACLE
    assert (img == 255).all(axis=2).sum() > 600      # lane borders
    # a vehicle turned by 90 degrees covers 5 m in y
    st["heading"][0, 1] = np.pi / 2
    img2 = render.render_scene(st, 0, dict(mm.DEFAULT_CONFIG))
    x1, y1 = st["x"][0, 1], st["y"][0, 1]
    assert tuple(img2[int((y1 + 2.2 + 16) * 3), int((x1 - 250) * 3)]) != render.GREY
    assert tuple(img2[int((y1 + 16) * 3), int((x1 + 2.2 - 250) * 3)]) in (render.GREY, render.WHITE)


def _gi_net(g, prefix):
    import torch
    from marl_mass_b200.rollout import ActorCriticNetwork
    net = ActorCriticNetwork(30, 5, 128, 1, state_split=True)
    sd = {k: torch.from_numpy(g[prefix + k.replace(".", "_")]) for k in net.state_dict()}
    net.load_state_dict(sd)
    return net


def test_shared_actor_critic_network_matches_the_reference_vectors():
    """rollout.ActorCriticNetwork against outputs frozen from the reference's Model_gi.ActorCriticNetwork
    (oracle/refharness/gen_golden_mappo_gi.py): log-probabilities without / with action mask, state values."""
    import torch
    g = np.load(os.path.join(ROOT, "tests", "golden", "mappo_gi_caller.npz"))
    net = _gi_net(g, "w_")
    obs = torch.from_numpy(g["obs"])
    with torch.no_grad():
        assert np.abs(net(obs).numpy() - g["logp"]).max() < 1e-5
        masked = net(obs, action_mask=torch.from_numpy(g["mask"])).numpy()
        assert np.abs(net(obs, out_type="v").numpy() - g["value"]).max() < 1e-5
    keep = g["mask"] == 1
    assert np.abs(masked[keep] - g["logp_masked"][keep]).max() < 1e-5
    assert (masked[~keep] < -1e7).all() and (g["logp_masked"][~keep] < -1e7).all()


def test_shared_network_update_matches_one_reference_train_step():
    """shared_network_loss(pairwise=True) + RMSprop + grad clip = one MAPPO_GI.train update of the reference's own code
    (parameters after the step frozen in the fixture); the per-sample surrogate the batched learner uses differs from
    the reference's [N, N] table only through which (ratio, advantage) pairs enter the min / mean."""
    import torch
    from marl_mass_b200.rollout import shared_network_loss
    g = np.load(os.path.join(ROOT, "tests", "golden", "mappo_gi_caller.npz"))
    net, target = _gi_net(g, "w_"), _gi_net(g, "t_")
    opt = torch.optim.RMSprop(net.parameters(), lr=float(g["lr"]))
    s, a, r = (torch.from_numpy(g[k]) for k in ("train_states", "train_actions", "train_returns"))
    loss, a_loss, c_loss = shared_network_loss(net, target, s, a, r, float(g["clip_param"]), pairwise=True)
    opt.zero_grad()
    loss.backward()
    torch.nn.utils.clip_grad_norm_(net.parameters(), float(g["max_grad_norm"]))
    opt.step()
    moved = 0.0
    for k, v in net.state_dict().items():
        want = g["after_" + k.replace(".", "_")]
        assert np.abs(v.numpy() - want).max() < 2e-6, k
        moved = max(moved, float(np.abs(want - g["w_" + k.replace(".", "_")]).max()))
    assert moved > 1e-3
    # per-sample form: same critic term, a surrogate over the N diagonal pairs instead of all N x N
    net2 = _gi_net(g, "w_")
    l2, a2, c2 = shared_network_loss(net2, target, s, a, r, float(g["clip_param"]))
    assert abs(float(c2.detach()) - float(c_loss.detach())) < 1e-6 and np.isfinite(float(a2.detach()))
    with torch.no_grad():
        h = net2.trunk(s)
        ratio = torch.exp((net2.policy_head(h) * a).sum(1) - (target(s) * a).sum(1))
        adv = (r - net2.critic_linear(h)).squeeze(1)
        want = -torch.min(ratio * adv, torch.clamp(ratio, 0.8, 1.2) * adv).mean()
    assert abs(float(a2.detach()) - float(want)) < 1e-6


def test_mappo_update_matches_one_reference_train_step():
    """mappo_losses(pairwise=True) + RMSprop + grad clip on both networks = one MAPPO.train update of the reference's
    own code (oracle/refharness/gen_golden_mappo_train.py: parameters after the step frozen in the fixture)."""
    import torch
    from marl_mass_b200.rollout import ActorNetwork, CriticNetwork, mappo_losses
    g = np.load(os.path.join(ROOT, "tests", "golden", "mappo_train_step.npz"))

    def net(cls, prefix):
        n = cls()
        n.load_state_dict({k: torch.from_numpy(g[prefix + "_" + k.replace(".", "_")]) for k in n.state_dict()})
        return n
    actor, critic = net(ActorNetwork, "actor"), net(CriticNetwork, "critic")
    actor_t, critic_t = net(ActorNetwork, "actor_t"), net(CriticNetwork, "critic_t")
    s, a, r = (torch.from_numpy(g[k]) for k in ("train_states", "train_actions", "train_returns"))
    a_loss, c_loss = mappo_losses(actor, actor_t, critic, critic_t, s, a, r, float(g["clip_param"]), pairwise=True)
    for n, loss in ((actor, a_loss), (critic, c_loss)):
        opt = torch.optim.RMSprop(n.parameters(), lr=float(g["lr"]))
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(n.parameters(), float(g["max_grad_norm"]))
        opt.step()
    for name, n in (("actor", actor), ("critic", critic)):
        moved = 0.0
        for k, v in n.state_dict().items():
            want = g["%s_after_%s" % (name, k.replace(".", "_"))]
            assert np.abs(v.numpy() - want).max() < 2e-6, (name, k)
            moved = max(moved, float(np.abs(want - g["%s_%s" % (name, k.replace(".", "_"))]).max()))
        assert moved > 1e-3, name


@pytest.mark.parametrize("name", ["priority_v0_td3_mixed", "dmc_v0_td3_mixed"])
def test_supervisor_core_matches_reference_fixtures(name, tmp_path):
    """csrc/supervisor_core.h - the priority / dmc supervisors as host+device code, the source the supervisor kernels
    compile - built for the host and run on every step of the reference fixtures: the supervised tuple must be the one
    the reference handed to _simulate, and the number of draws it reports as consumed the number of np.random.rand()
    calls the reference made (the single-env adapter advances its MT19937 replay by that count)."""
    import oracle as orc
    g, cfg = load_golden(name)
    src = os.path.join(ROOT, "marl-mass_b200", "csrc", "supervisor_host.cpp")
    lib_path = str(tmp_path / "libsupervisor_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", src, "-o", lib_path])
    lib = ctypes.CDLL(lib_path)
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    lib.mm_supervisor_host.argtypes = [ctypes.c_int] * 3 + [dp] * 5 + [ip] * 5 + [dp, ctypes.c_double, ip]
    rows = g["row_of_step"]
    st = orc.state_from_golden(g, rows)
    kind = 0 if cfg["safety_guarantee"] == "priority" else 1
    replaced = 0
    for t in range(len(rows)):
        n, n_cav = int(st["n_veh"][t]), int(st["n_cav"][t])
        f = lambda k: np.ascontiguousarray(st[k][t, :n], np.float64)
        i = lambda k: np.ascontiguousarray(st[k][t, :n], np.int32)
        arrs = [f("x"), f("y"), f("heading"), f("speed"), f("target_speed"), i("lane"), i("target_lane"), i("speed_index"),
                i("crashed")]
        act = np.ascontiguousarray(g["act"][t, :n_cav], np.int32)
        draws = np.ascontiguousarray(np.nan_to_num(g["rand_draws"][t]), np.float64)
        used = ctypes.c_int(-1)
        rc = lib.mm_supervisor_host(kind, n, n_cav, *[a.ctypes.data_as(dp if a.dtype == np.float64 else ip) for a in arrs],
                                    act.ctypes.data_as(ip), draws.ctypes.data_as(dp), float(cfg["HEADWAY_TIME"]), ctypes.byref(used))
        assert rc == 0
        assert used.value == int(np.sum(~np.isnan(g["rand_draws"][t]))), (t, used.value)
        want = g["new_act"][t, :n_cav].astype(np.int32)
        assert np.array_equal(act, want), (t, g["act"][t, :n_cav].tolist(), act.tolist(), want.tolist())
        replaced += int(not np.array_equal(want, g["act"][t, :n_cav]))
    assert replaced >= 100


@pytest.mark.parametrize("name", ["priority_v0_td3_mixed", "dmc_v0_td3_mixed"])
def test_supervisor_draws_continue_the_spawn_stream(name):
    """Seed-exact supervisors in the single-env adapter: the reference takes the supervisors' np.random.rand() numbers from
    the process-global MT19937 stream that reset() seeded and the spawn consumed first; nothing else on the step path
    draws from it.  So the generator `spawn_scene` hands back, advanced step by step by the number of draws the
    supervisor consumed, reproduces every draw the reference logged for the episode."""
    from marl_mass_b200 import spawn
    from marl_mass_b200.env import traffic_type_of
    g, cfg = load_golden(name)
    ep, rows, rd = g["ep_start"], g["row_of_step"], g["rand_draws"]
    total = 0
    for k, seed in enumerate(cfg["seeds"]):
        rngs = []
        spawn.spawn_scene(seed, cfg["traffic_density"], traffic_type_of(cfg), 0, rng_out=rngs)
        rs = rngs[0]
        for t in np.where((rows >= ep[k]) & (rows < ep[k + 1] - 1))[0]:
            n = int(np.sum(~np.isnan(rd[t])))
            peek = np.random.RandomState()
            peek.set_state(rs.get_state())
            assert np.array_equal(peek.rand(32)[:n], rd[t, :n]), (seed, int(t))
            rs.rand(n)
            total += n
    assert total > 3000


def test_supervisor_core_compiles_for_sm100a(tmp_path):
    """The same header is device code: a thread-per-scene stub kernel around both supervisors compiles for sm_100a."""
    import shutil
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    stub = tmp_path / "supervisor_stub.cu"
    stub.write_text(r"""
#include "supervisor_core.h"
using namespace mmsup;
__global__ void supervisor_stub(int kind, int n_scenes, const Veh *scenes, const int *n_veh, const int *n_cav, int *actions,
                                const double *draws, double headway_time) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_scenes) return;
    Veh road[MAXV];
    const Veh *orig = scenes + (size_t)e * MAXV;
    for (int i = 0; i < n_veh[e]; ++i) road[i] = orig[i];
    if (kind == 0) priority_supervisor(road, orig, n_veh[e], n_cav[e], actions + e * MAXV, draws + e * 16, headway_time);
    else dmc_supervisor(road, orig, n_veh[e], n_cav[e], actions + e * MAXV, draws + e * 16, headway_time);
}
""")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-fmad=false", "-std=c++17",
                           "-I", os.path.join(ROOT, "marl-mass_b200", "csrc"), "-c", str(stub), "-o", str(tmp_path / "stub.o")])


@pytest.mark.parametrize("kind,td", [("priority", 1), ("priority", 3), ("dmc", 2), ("dmc", 3)])
def test_supervisor_core_agrees_with_the_python_restatement_on_fresh_scenes(kind, td, tmp_path):
    """Two independent restatements of the supervisors (csrc/supervisor_core.h built for the host, the pure-Python
    checker) on scenes the fixtures do not hold: other densities, random draws, scenes advanced by the un-shielded v0
    dynamics under random actions."""
    import marl_mass_b200 as mm
    import oracle as orc
    import supervisor as sup
    src = os.path.join(ROOT, "marl-mass_b200", "csrc", "supervisor_host.cpp")
    lib_path = str(tmp_path / "libsupervisor_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", src, "-o", lib_path])
    lib = ctypes.CDLL(lib_path)
    dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)
    lib.mm_supervisor_host.argtypes = [ctypes.c_int] * 3 + [dp] * 5 + [ip] * 5 + [dp, ctypes.c_double, ip]
    E = 24
    cfg = dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-v0", safety_guarantee="none", traffic_density=td,
               traffic_type="mixed", mixed_traffic=True, HEADWAY_TIME=1.2)
    st = mm.spawn.spawn_state(list(range(100, 100 + E)), td, "mixed")
    ocfg = orc.make_config(cfg)
    rng = np.random.RandomState(17 + td)
    fn = sup.priority_supervisor if kind == "priority" else sup.dmc_supervisor
    replaced = 0
    for t in range(30):
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        draws = rng.rand(E, 16)
        for e in range(E):
            n, n_cav = int(st["n_veh"][e]), int(st["n_cav"][e])
            want = fn(st, e, a[e], draws[e], 1.2)
            f = lambda k: np.ascontiguousarray(st[k][e, :n], np.float64)
            i = lambda k: np.ascontiguousarray(st[k][e, :n], np.int32)
            arrs = [f("x"), f("y"), f("heading"), f("speed"), f("target_speed"), i("lane"), i("target_lane"),
                    i("speed_index"), i("crashed")]
            act = np.ascontiguousarray(a[e, :n_cav], np.int32)
            d = np.ascontiguousarray(draws[e])
            assert lib.mm_supervisor_host(0 if kind == "priority" else 1, n, n_cav,
                                          *[x.ctypes.data_as(dp if x.dtype == np.float64 else ip) for x in arrs],
                                          act.ctypes.data_as(ip), d.ctypes.data_as(dp), 1.2, None) == 0
            assert act.tolist() == want, (t, e, a[e, :n_cav].tolist(), act.tolist(), want)
            replaced += int(want != a[e, :n_cav].tolist())
            a[e, :n_cav] = act           # the env then executes the supervised tuple
        orc.step(ocfg, st, a, n_threads=4)
    assert replaced > 0 or td == 1       # sparse traffic rarely needs the supervisor this early in an episode


def test_sub_step_ulp_tie_scene_is_recognised():
    """tests/golden/ulp_tie_scene.npz: the one scene of 37 M snapped soak env-steps whose shield record differed between the
    kernels and the oracle (profiles/soak_repro.py 302 1 snap).  Vehicle 4 steers by 4e-7 rad; its x after the first
    sub-step is one ulp apart on the two sides (cos(h + beta) by glibc vs the angle-sum form with libdevice tan) and
    vehicle 2 lands exactly there (373.5 + 17.5 / 15 == 374 + 10 / 15), so the second sub-step sees a tie on one side and
    an order on the other.  The soak reports such steps instead of failing; this pins the detector and the scene."""
    import oracle as orc
    from helpers import near_tie_inside_step
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    from soak_cases import CASES
    import importlib
    mm = importlib.import_module("marl_mass_b200")
    d = np.load(os.path.join(ROOT, "tests", "golden", "ulp_tie_scene.npz"))
    shield, traffic, td, reward, lateral = CASES[1]
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee=shield, lateral_control=lateral, traffic_type=traffic, traffic_density=td,
               agent_reward=reward, HEADWAY_TIME=0.5, cbf_eta=0.03125, HIGH_SPEED_REWARD=4, HEADWAY_COST=1, MERGING_LANE_COST=8)
    ocfg = orc.make_config(cfg)
    pre = {k[4:]: np.array(d[k])[None].copy() for k in d.files if k.startswith("pre_")}
    a = d["actions"][None].astype(np.int8)
    assert near_tie_inside_step(orc, ocfg, pre, 0, a) and ocfg.substeps == 3
    # the oracle's own records are the ones the soak expected
    st = {k: v.copy() for k, v in pre.items()}
    want = orc.step(ocfg, st, a, n_threads=1)
    for k in ("leader", "front_adj", "rear_adj"):
        assert np.array_equal(np.asarray(want["sh_" + k])[0], d["want_" + k])
    # and the scene without the coincidence (vehicle 2 a millimetre back) is not flagged
    pre["x"][0, 2] -= 1e-3
    pre["rec1_x"][0, 2] -= 1e-3
    assert not near_tie_inside_step(orc, ocfg, pre, 0, a)


def test_zero_numerator_division_identity():
    """csrc/mm_device.cuh div_nz: for a finite y != 0, x / y with x == +-0 is +-0 with the sign of the product - the value
    x * y has - so routing zero numerators around CUDA's division (whose slow path every zero quotient enters) cannot
    change a bit.  Checked here in IEEE double arithmetic on the host, signs of zero included."""
    rng = np.random.RandomState(5)
    y = np.concatenate([rng.uniform(-50, 50, 1000), [1e-2, -1e-2, 2.5, -2.5, 1e-300, -1e300]])
    y = y[y != 0]
    for zero in (0.0, -0.0):
        x = np.full_like(y, zero)
        q, p = x / y, x * y
        assert np.array_equal(q, p) and np.array_equal(np.signbit(q), np.signbit(p))
    x = rng.uniform(-5, 5, y.shape)
    stand_in = np.where(x == 0, 1.0, x)
    assert np.array_equal(np.where(x == 0, x * y, stand_in / y), x / y)

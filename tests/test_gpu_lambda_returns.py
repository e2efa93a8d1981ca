"""GPU suite, GAE(lambda) returns: the kernel (mm_lambda_returns through rollout.lambda_returns), the shared target
pass's value output, and gae_lambda of BatchedMAPPORollout / BatchedMAPPOGIRollout.

- The kernel against the float32 restatement bit for bit and the float64 one within 1e-5 (lambda_returns_ref.py), on
  random rollouts with terminal steps at random, at the last step and in runs, with and without final_value, column
  counts that are not multiples of 256 and one beyond the grid's stride; lambda = 1 is mm_discounted_returns bit for bit,
  lambda = 0 the one-step targets; values the recursion must not read (after a terminal step, at step 0) poisoned with NaN.
- gae_lambda=1.0 trains exactly as gae_lambda=None (3 collect + update iterations, both learners, both impls, both
  optimisers); the None path runs none of the new work.
- gae_lambda=0.95 on real rollouts: torch against CUDA update, the returns against the restatement fed with the values,
  advantage_mean of the statistics pass, and no live row's recursion reading a row without an agent.
- Two ranks under NCCL stay replicas (skipped with fewer than two GPUs).
"""
import copy
import os
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest

import lambda_returns_ref as ref
from conftest import ROOT

pytestmark = pytest.mark.gpu

GAMMA = 0.99
LOSS_TOL = 1e-3          # as test_gpu_learner.py's whole-update comparison


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()
    return m


def _cuda(a):
    import torch
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("lam", [0.0, 0.5, 0.95, 1.0])
def test_kernel_against_the_restatements(mm, lam):
    from marl_mass_b200 import rollout
    for T, E, seed in ((100, 37, 1), (100, 1000, 2), (7, 30001, 3)):      # 444, 12000 and 360012 columns
        r, d, v, fv = ref.random_rollout(T, E, 12, seed)
        for f in (fv, None):
            got = rollout.lambda_returns(_cuda(r), _cuda(d), _cuda(v), _cuda(f), GAMMA, lam).cpu().numpy()
            want32 = ref.lambda_returns_ref(r, d, v, f, GAMMA, lam)
            assert got.tobytes() == want32.tobytes(), (T, E, lam, f is None, np.abs(got - want32).max())
            want64 = ref.lambda_returns_ref(r, d, v, f, GAMMA, lam, dtype=np.float64)
            assert np.all(np.abs(got - want64) <= 1e-5 * np.maximum(np.abs(want64), 1.0)), (T, E, lam)
            if lam == 1.0:
                disc = rollout.discounted_returns(_cuda(r), _cuda(d), _cuda(f), GAMMA).cpu().numpy()
                assert got.tobytes() == disc.tobytes()
            if lam == 0.0:
                assert got.tobytes() == ref.one_step_targets_ref(r, d, v, f, GAMMA).tobytes()
            poisoned = v.copy()
            poisoned[0] = np.nan
            poisoned[1:][d[:-1] != 0] = np.nan
            again = rollout.lambda_returns(_cuda(r), _cuda(d), _cuda(poisoned), _cuda(f), GAMMA, lam).cpu().numpy()
            clean = ref.lambda_returns_ref(r, d, np.nan_to_num(poisoned, nan=0.0), f, GAMMA, lam)
            assert np.isfinite(again).all() and again.tobytes() == clean.tobytes()


def test_lambda_one_without_values_is_the_discounted_return(mm):
    import torch
    from marl_mass_b200 import _lib, rollout
    r, d, v, fv = ref.random_rollout(30, 50, 12, 9)
    rd, dd, fd = _cuda(r), _cuda(d), _cuda(fv)          # held until the kernel has read them
    out = torch.empty(r.shape, device="cuda")
    _lib.check(_lib.lib().mm_lambda_returns(rollout._ptr(rd), rollout._ptr(dd), rollout._ptr(None), rollout._ptr(fd), GAMMA,
                                            1.0, 30, 600, 12, rollout._ptr(out), rollout._stream()))
    assert out.cpu().numpy().tobytes() == ref.discounted_returns_ref(r, d, fv, GAMMA).tobytes()


# ---- the learners

def _config(shared, steps):
    from marl_mass_b200.train import load_ini
    ini = "mass_td3_mixed_srew_shared.ini" if shared else "mass_td3_srew.ini"
    env_cfg, kw, _ = load_ini(os.path.join(ROOT, "examples", ini))
    kw["roll_out_n_steps"] = steps
    return env_cfg, kw


def _learner(shared, envs=256, steps=20, **kw):
    import torch
    from marl_mass_b200.env import DEFAULT_CONFIG, MergeEnvBatched
    from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout
    env_cfg, rkw = _config(shared, steps)
    env = MergeEnvBatched(envs, dict(DEFAULT_CONFIG, **env_cfg), device=0)
    torch.manual_seed(11)
    pol = (BatchedMAPPOGIRollout if shared else BatchedMAPPORollout)(env, seed=5, **rkw, **kw)
    return env, pol


@pytest.mark.parametrize("optimizer", ["torch", "cuda"])
@pytest.mark.parametrize("impl", ["torch", "cuda"])
@pytest.mark.parametrize("shared", [False, True], ids=["mappo", "shared"])
def test_lambda_one_trains_exactly_as_no_lambda(mm, shared, impl, optimizer):
    import torch
    runs = {}
    for gae in (None, 1.0):
        env, pol = _learner(shared, optimizer=optimizer, gae_lambda=gae)
        recs = []
        torch.manual_seed(21)
        for _ in range(3):
            pol.collect()
            recs.append(pol.update(minibatch=1 << 12, impl=impl))
        if gae is not None:
            assert torch.equal(pol.buf["lambda_returns"], pol.buf["returns"])
        else:
            assert "lambda_returns" not in pol.buf
        runs[gae] = (recs, [[p.detach().clone() for p in m.parameters()] for m in pol.networks()])
        env.close()
    assert runs[None][0] == runs[1.0][0]
    for a, b in zip(runs[None][1], runs[1.0][1]):
        for p, q in zip(a, b):
            assert torch.equal(p, q), (shared, impl, optimizer)


def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return Counter(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


@pytest.mark.parametrize("impl", ["torch", "cuda"])
@pytest.mark.parametrize("shared", [False, True], ids=["mappo", "shared"])
def test_no_lambda_path_runs_none_of_the_new_work(mm, shared, impl):
    """collect() issues the same env launches with and without gae_lambda; the update without it runs no returns kernel,
    and every device activity of it also occurs in the update with gae_lambda (which adds the values, the kernel and
    the zero fill).  Both learners start from the same seeds, after a warm-up learner has run one iteration (one-time
    initialisation)."""
    import torch
    env, pol = _learner(shared)
    pol.collect()
    pol.update(minibatch=1 << 12, impl=impl)
    env.close()
    counts = {}
    for gae in (None, 0.95):
        env, pol = _learner(shared, gae_lambda=gae)
        l0 = env.kernel_launches()
        collect = _kernel_names(pol.collect)
        launches = env.kernel_launches() - l0
        torch.manual_seed(3)
        update = _kernel_names(lambda: pol.update(minibatch=1 << 12, impl=impl))
        counts[gae] = launches, collect, update
        env.close()
    assert counts[None][0] == counts[0.95][0] > 0
    assert counts[None][1] == counts[0.95][1]
    returns_kernel = [k for k in counts[0.95][2] if "discounted_returns_kernel" in k]
    assert len(returns_kernel) == 1 and counts[0.95][2][returns_kernel[0]] == 1
    assert not any("discounted_returns_kernel" in k for k in counts[None][2])
    assert not (counts[None][2] - counts[0.95][2]), counts[None][2] - counts[0.95][2]


@pytest.fixture(scope="module", params=[False, True], ids=["mappo", "shared"])
def collected(mm, request):
    env, pol = _learner(request.param, envs=512, steps=120, gae_lambda=0.95)     # episodes end at step 100
    pol.collect()
    yield request.param, pol
    env.close()


def _values_cuda(pol, shared):
    import torch
    from marl_mass_b200 import rollout
    idx, S, A8, _ = pol._learner_batch(with_returns=False)
    v = torch.zeros(S.shape[0], device="cuda")
    if shared:
        rollout.ppo_targets(pol.policy_target, S, A8, idx, value_out=v)
    else:
        rollout.ppo_targets(pol.critic_target, S, A8, idx, out=v)
    return v


def _restate(pol, values):
    b = pol.buf
    return ref.lambda_returns_ref(b["rewards"].cpu().numpy(), b["dones"].cpu().numpy(),
                                  values.view(b["rewards"].shape).cpu().numpy(), b["final_value"].cpu().numpy(),
                                  pol.gamma, pol.gae_lambda)


def _save(pol, shared):
    """the networks (targets included) and optimiser states, so that a test leaves the shared rollout as it found it"""
    opts = [pol.policy_opt] if shared else [pol.actor_opt, pol.critic_opt]
    return [copy.deepcopy(m.state_dict()) for m in pol.networks()], opts, [copy.deepcopy(o.state_dict()) for o in opts]


def _restore(pol, saved):
    for m, sd in zip(pol.networks(), saved[0]):
        m.load_state_dict(sd)
    for o, sd in zip(saved[1], saved[2]):
        o.load_state_dict(copy.deepcopy(sd))


def test_live_rows_never_read_rows_without_an_agent(collected):
    """within an episode n_agents is fixed, and a terminal step cuts the recursion: a live row at t that did not end its
    episode has a live row at t + 1 in the same slot.  Poisoning every value of a row without an agent with NaN changes
    no live row's lambda-return."""
    import torch
    from marl_mass_b200 import rollout
    shared, pol = collected
    b = pol.buf
    live, done = b["live"], b["dones"] != 0
    cont = live[:-1] & ~done[:-1, :, None]
    assert int(cont.sum()) > 0 and bool(done.any())
    assert bool(live[1:][cont].all())
    v = _values_cuda(pol, shared).view(live.shape)
    poisoned = torch.where(live, v, torch.full_like(v, float("nan")))
    a = rollout.lambda_returns(b["rewards"], b["dones"], v, b["final_value"], pol.gamma, 0.95)
    c = rollout.lambda_returns(b["rewards"], b["dones"], poisoned, b["final_value"], pol.gamma, 0.95)
    assert torch.equal(a[live], c[live]) and bool(torch.isfinite(c[live]).all())


def test_shared_target_pass_value_output(collected):
    """value_out leaves old_logp as it was and gives V_target(s) of the listed rows (fp16 operands: against the torch
    forward within 2e-3 of the values' scale); rows not listed keep what the buffer held"""
    import torch
    from marl_mass_b200 import rollout
    shared, pol = collected
    if not shared:
        pytest.skip("the value output belongs to the shared network")
    idx, S, A8, _ = pol._learner_batch(with_returns=False)
    plain = rollout.ppo_targets(pol.policy_target, S, A8, idx)
    v = torch.full((S.shape[0],), 7.0, device="cuda")
    with_v = rollout.ppo_targets(pol.policy_target, S, A8, idx, value_out=v)
    assert torch.equal(plain[idx], with_v[idx])
    with torch.no_grad():
        vt = pol.policy_target(S[idx], out_type="v")[:, 0]
    assert float((v[idx] - vt).abs().max()) <= 2e-3 * max(1.0, float(vt.abs().max()))
    dead = torch.ones(S.shape[0], dtype=torch.bool, device="cuda")
    dead[idx] = False
    assert bool((v[dead] == 7.0).all())


@pytest.mark.parametrize("impl", ["torch", "cuda"])
def test_lambda_returns_of_an_update_match_the_restatement(collected, impl):
    """the values each impl uses (torch: the target network's torch forward over the live rows; cuda: the target pass),
    taken before the update, through the float32 restatement: the update's buf["lambda_returns"] bit for bit"""
    import torch
    shared, pol = collected
    saved = _save(pol, shared)
    values = pol._rollout_values_torch() if impl == "torch" else _values_cuda(pol, shared)
    torch.manual_seed(5)
    pol.update(minibatch=1 << 22, impl=impl)
    got = pol.buf["lambda_returns"].cpu().numpy()
    assert got.tobytes() == _restate(pol, values).tobytes()
    assert not np.array_equal(got, pol.buf["returns"].cpu().numpy())
    _restore(pol, saved)


@pytest.mark.parametrize("impl", ["torch", "cuda"])
def test_advantage_mean_is_that_of_the_lambda_returns(collected, impl):
    import torch
    shared, pol = collected
    saved = _save(pol, shared)
    live = pol.buf["live"].reshape(-1)
    values = pol._rollout_values_torch() if impl == "torch" else _values_cuda(pol, shared)
    torch.manual_seed(5)
    rec = pol.update(minibatch=1 << 22, impl=impl, stats=True)
    G = pol.buf["lambda_returns"].reshape(-1)
    want = float((G[live].double() - values[live].double()).mean())
    scale = float(G[live].double().abs().mean())
    assert abs(rec["advantage_mean"] - want) <= 1e-6 * max(scale, 1.0), (rec["advantage_mean"], want)
    plain = float((pol.buf["returns"].reshape(-1)[live].double() - values[live].double()).mean())
    assert plain != want                                  # the key follows the returns the update trains on
    _restore(pol, saved)


def test_torch_and_cuda_updates_agree(collected):
    """one minibatch from identical networks and optimiser states: parameter deltas with cosine >= 0.99 per tensor and
    losses within 1e-3 relative (the tolerances of test_gpu_learner.py's whole-update test), the loss relative to the
    larger of itself and the mean |advantage|: the two impls' values differ by the fp16 operands of the target pass, so
    their lambda-returns differ too (checked within 1e-3 of their scale), and the actor loss, a mean of advantages that
    nearly cancel with lambda-returns, inherits that difference at the scale of the advantages"""
    import torch
    shared, pol = collected
    saved = _save(pol, shared)
    mods = pol.networks()[:1 if shared else 2]
    before = [p.detach().clone() for m in mods for p in m.parameters()]
    out = {}
    for impl in ("torch", "cuda"):
        _restore(pol, saved)
        torch.manual_seed(99)
        rec = pol.update(minibatch=1 << 22, impl=impl)
        out[impl] = rec, [p.detach().clone() for m in mods for p in m.parameters()], pol.buf["lambda_returns"].clone()
    (rt, at, gt), (rc, ac, gc) = out["torch"], out["cuda"]
    live = pol.buf["live"]
    _restore(pol, saved)
    adv = float((gt.reshape(-1) - pol._rollout_values_torch()).reshape(live.shape)[live].abs().mean())
    for k in ("actor_loss", "critic_loss"):
        assert abs(rc[k] - rt[k]) <= LOSS_TOL * max(abs(rt[k]), adv if k == "actor_loss" else 0.0, 1e-3), (k, rc[k], rt[k], adv)
    assert float((gc - gt)[live].abs().max()) <= 1e-3 * max(1.0, float(gt[live].abs().max()))
    for b, t, c in zip(before, at, ac):
        dt, dc = (t - b).reshape(-1), (c - b).reshape(-1)
        if float(dt.norm()) == 0.0:
            assert float(dc.norm()) == 0.0
            continue
        assert float(torch.dot(dt, dc) / (dt.norm() * dc.norm())) >= 0.99
    _restore(pol, saved)


@pytest.mark.parametrize("ini", ["mass_td3_srew.ini", "mass_td3_mixed_srew_shared.ini"])
def test_driver_option_and_ini_key(mm, ini, tmp_path):
    """train(gae_lambda=0.95) and the same value from MODEL_CONFIG.gae_lambda give the same run; the records carry the
    same keys as without it"""
    from marl_mass_b200.train import train
    path = os.path.join(ROOT, "examples", ini)
    timing = {"collect_s", "update_s", "agent_steps_per_s"}
    kw = dict(n_envs=128, iterations=2, eval_interval=0, update_impl="cuda", log=lambda *_: None)
    off = train(path, **kw)
    on = train(path, gae_lambda=0.95, **kw)
    keyed = tmp_path / ini
    keyed.write_text(open(path).read().replace("[MODEL_CONFIG]", "[MODEL_CONFIG]\ngae_lambda = 0.95"))
    from_ini = train(str(keyed), **kw)
    for a, b, c in zip(off, on, from_ini):
        assert set(a) == set(b) == set(c)
        assert {k: v for k, v in b.items() if k not in timing} == {k: v for k, v in c.items() if k not in timing}
    assert off[1]["critic_loss"] != on[1]["critic_loss"]


_DP = r"""
import sys
sys.path.insert(0, sys.argv[1])
from marl_mass_b200.train import train
h = train(sys.argv[2], n_envs=256, iterations=3, eval_interval=0, update_impl=sys.argv[3], gae_lambda=0.95)
print("REPLICA_DIFF", h[-1]["replica_param_max_diff"])
"""


@pytest.mark.parametrize("impl", ["torch", "cuda"])
def test_two_ranks_stay_replicas(mm, impl, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "dp.py"
    script.write_text(_DP)
    ini = os.path.join(ROOT, "examples", "mass_td3_srew.ini")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc_per_node", "2", str(script), ROOT, ini, impl],
                         cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    diffs = [float(line.split()[1]) for line in out.stdout.splitlines() if line.startswith("REPLICA_DIFF")]
    assert diffs and all(d == 0.0 for d in diffs), out.stdout[-2000:]

"""GPU suite, the learner's statistics pass (mm_ppo_stats through rollout.ppo_stats) and update(stats=True).

- A network against its own target pass: r == 1 exactly on every row (the passes share the forward), so K3 and CLIPPED
  are 0 and the ratio range is [1, 1], at the tile and grid edges of the device, with unsorted and duplicate indices.
- Exactly representable data (learner_ref.exact_*): N, CLIPPED and the value fields equal the fp16 restatement
  (ppo_stats_ref.py) bit for bit; the entropy and k3 sums, whose logf / expf differ from numpy's by ulps, within 1e-6.
- Rows of a real rollout after one update: every field within the tolerances stated in the test against the restatement.
- Determinism, the shared workspace, two halves combined, update(stats=True) against update(stats=False) and the driver.
"""
import copy
import math
import os

import numpy as np
import pytest

import learner_ref
import ppo_stats_ref
from conftest import ROOT

pytestmark = pytest.mark.gpu

K = ppo_stats_ref.K
CLIP = 0.2
VALUE = [K[k] for k in ("v", "v2", "g", "g2", "res2")]


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()
    return m


@pytest.fixture(scope="module")
def sms(mm):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _module(kind, seed):
    import torch
    from marl_mass_b200 import rollout
    torch.manual_seed(seed)
    return {"actor": rollout.ActorNetwork, "critic": rollout.CriticNetwork, "shared": rollout.ActorCriticNetwork}[kind]().cuda()


def _params(net):
    return {k: p.detach().cpu().numpy().copy() for k, p in net.named_parameters()}


def _rows(rows, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    S = torch.randn((rows, 30), device="cuda", generator=g)
    A8 = torch.randint(0, 5, (rows,), device="cuda", generator=g).to(torch.int8)
    G = 3 * torch.randn(rows, device="cuda", generator=g)
    return S, A8, G


def _idx(n, rows, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, rows, (n,), device="cuda", generator=g)          # unsorted, with duplicates


def _stats(net, S, A8, G, idx, old=None, clip=CLIP):
    from marl_mass_b200 import rollout
    return rollout.ppo_stats(net, S, A8, G, idx, old, clip).cpu().numpy()


@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
def test_network_equal_to_its_target_gives_ratio_one(mm, sms, kind):
    from marl_mass_b200 import rollout
    net = _module(kind, 1)
    rows = 120_000
    S, A8, G = _rows(rows, 2)
    for n in (1, 127, 128, 129, sms * 128 - 1, sms * 128 + 1, 100_003):
        idx = _idx(n, rows, n)
        old = None if kind == "critic" else rollout.ppo_targets(net, S, A8, idx)
        v = _stats(net, S, A8, G, idx, old)
        assert v[K["n"]] == n
        if kind == "critic":
            assert v[K["ratio_min"]] == math.inf and v[K["ratio_max"]] == -math.inf and not v[1:4].any()
            q = rollout.ppo_targets(net, S, A8, idx)[idx].double()
            assert abs(v[K["v"]] - float(q.sum())) <= 1e-12 * float(q.abs().sum())
        else:
            assert v[K["k3"]] == 0.0 and v[K["clipped"]] == 0.0, (n, v)
            assert v[K["ratio_min"]] == 1.0 and v[K["ratio_max"]] == 1.0, (n, v)
            assert 0 < v[K["entropy"]] / n <= math.log(5) * (1 + 1e-6)
        if kind == "actor":
            assert not v[VALUE].any()


def test_empty_index_list_gives_the_empty_value(mm):
    import torch
    S, A8, G = _rows(8, 3)
    j = torch.zeros(0, dtype=torch.int64, device="cuda")
    old = torch.zeros(8, device="cuda")
    for kind in ("actor", "critic", "shared"):
        v = _stats(_module(kind, 4), S, A8, G, j, old)
        assert v[K["ratio_min"]] == math.inf and v[K["ratio_max"]] == -math.inf
        assert not np.delete(v, [K["ratio_min"], K["ratio_max"]]).any(), (kind, v)


def _exact_case(kind, n, group, seed):
    """learner_ref's exactly representable rows and network; old_logp from the target pass, shifted by +-1 on the rows
    pushed outside the clip range"""
    rows = n + 40
    S, A8 = learner_ref.exact_rows(rows, seed)
    idx = learner_ref.exact_index(n, rows, seed + 1)
    learner_ref.exact_probe_actions(A8, idx, [0, n - 1])
    params = learner_ref.exact_params(kind, group, seed + 2)
    every = np.arange(rows)
    t = learner_ref.learner_pass(kind, params, S, A8, None, None, None, every, learner_ref.EXACT_CLIP, fp16=True, check=True)
    values = t["q"] if kind == "critic" else (t["v"] if kind == "shared" else np.zeros(rows, np.float32))
    G, shift = learner_ref.exact_offsets(values, idx, [0, n - 1], seed + 3)
    old = None if kind == "critic" else (t["logp"] - shift).astype(np.float32)
    return S, A8, G, idx, params, old


def _module_from(kind, params):
    import torch
    net = _module(kind, 0)
    with torch.no_grad():
        for name, p in net.named_parameters():
            p.copy_(torch.from_numpy(params[name]))
    return net


@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
def test_exact_data_bit_for_bit(mm, sms, kind):
    import torch
    clip = learner_ref.EXACT_CLIP
    for k, n in enumerate((129, sms * 128 + 1, 100_003)):
        S, A8, G, idx, params, old = _exact_case(kind, n, (1, 2, 4)[k], 500 + n)
        want = ppo_stats_ref.ppo_stats_ref(kind, params, S, A8, G, idx, old, clip, fp16=True)
        t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
        got = _stats(_module_from(kind, params), t(S), t(A8), t(G.astype(np.float32)), t(idx), t(old), clip)
        exact = [K["n"], K["clipped"]] + VALUE
        assert np.array_equal(got[exact], want[exact]), (kind, n, got, want)
        if kind != "critic":
            assert 0 < want[K["clipped"]] < n
            for f in ("entropy", "k3"):
                assert abs(got[K[f]] - want[K[f]]) <= 1e-6 * max(1.0, abs(want[K[f]])), (kind, n, f, got[K[f]], want[K[f]])
            for f in ("ratio_min", "ratio_max"):
                assert abs(got[K[f]] - want[K[f]]) <= 2e-7 * want[K[f]], (kind, n, f)


def _rollout(shared, envs=1024, steps=20, seed=11, **kw):
    import torch
    from marl_mass_b200.env import DEFAULT_CONFIG, MergeEnvBatched
    from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout
    from marl_mass_b200.train import load_ini
    ini = "mass_td3_mixed_srew_shared.ini" if shared else "mass_td3_srew.ini"
    env_cfg, rkw, _ = load_ini(os.path.join(ROOT, "examples", ini))
    rkw["roll_out_n_steps"] = steps
    env = MergeEnvBatched(envs, dict(DEFAULT_CONFIG, **env_cfg), device=0)
    torch.manual_seed(seed)
    pol = (BatchedMAPPOGIRollout if shared else BatchedMAPPORollout)(env, seed=5, **rkw, **kw)
    pol.collect()
    return env, pol


def _pairs(pol, shared):
    """(kind, updated network, target network) of a rollout object"""
    if shared:
        return [("shared", pol.policy, pol.policy_target)]
    return [("actor", pol.actor, pol.actor_target), ("critic", pol.critic, pol.critic_target)]


@pytest.fixture(scope="module", params=[False, True], ids=["mappo", "shared"])
def updated(mm, request):
    """a collected rollout at 1024 envs, its networks after one real update (impl cuda, 4 minibatches) and copies of the
    networks that collected it (the rollout policy and critic: the update ends by copying the networks to the targets)"""
    import torch
    env, pol = _rollout(request.param)
    saved = {kind: copy.deepcopy(net) for kind, net, _ in _pairs(pol, request.param)}
    batch = pol._learner_batch()
    torch.manual_seed(3)
    pol.update(minibatch=batch[0].numel() // 4 + 1, impl="cuda")
    yield request.param, pol, batch, saved
    env.close()


def test_collected_rows_after_an_update_match_the_restatement(updated):
    """fp16-operand restatement on the rows of a real rollout, the updated networks against the rollout policy.
    Tolerances: N exact; value sums 1e-5 relative (the f32 forward's summation order); entropy sum 1e-5 relative; k3
    sum 1e-5 relative + 1e-6 per row; the ratio range 1e-5 relative; CLIPPED exact once the rows within 1e-5 of the clip
    bound (either side) are left out of both counts."""
    import torch
    from marl_mass_b200 import rollout
    shared, pol, (idx, S, A8, G), saved = updated
    Sn, An, Gn, jn = S.cpu().numpy(), A8.cpu().numpy(), G.cpu().numpy(), idx.cpu().numpy()
    for kind, net, _ in _pairs(pol, shared):
        old = None if kind == "critic" else rollout.ppo_targets(saved[kind], S, A8, idx)
        got = _stats(net, S, A8, G, idx, old)
        on = None if old is None else old.cpu().numpy()
        want = ppo_stats_ref.ppo_stats_ref(kind, _params(net), Sn, An, Gn, jn, on, CLIP, fp16=True)
        n = len(jn)
        assert got[K["n"]] == want[K["n"]] == n
        for f in VALUE + [K["entropy"]]:
            assert abs(got[f] - want[f]) <= 1e-5 * max(abs(want[f]), 1.0), (kind, ppo_stats_ref.FIELDS[f], got[f], want[f])
        if kind == "critic":
            continue
        assert abs(got[K["k3"]] - want[K["k3"]]) <= 1e-5 * abs(want[K["k3"]]) + 1e-6 * n, (kind, got[K["k3"]], want[K["k3"]])
        for f in ("ratio_min", "ratio_max"):
            assert abs(got[K[f]] - want[K[f]]) <= 1e-5 * want[K[f]], (kind, f, got[K[f]], want[K[f]])
        # CLIPPED: the rows near the bound are the only ones the two may classify differently
        r = ppo_stats_ref.stat_rows(kind, _params(net), Sn, An, Gn, jn, on, CLIP, fp16=True)["ratio"].astype(np.float64)
        near = np.abs(np.abs(r - 1) - CLIP) <= 1e-5
        near_t = torch.from_numpy(jn[near]).cuda()
        got_near = _stats(net, S, A8, G, near_t, old)[K["clipped"]] if near.any() else 0.0
        want_near = float(((np.abs(r - 1) > CLIP) & near).sum())
        assert got[K["clipped"]] - got_near == want[K["clipped"]] - want_near, (kind, got[K["clipped"]], want[K["clipped"]])
        assert 0 < want[K["clipped"]]


def test_deterministic_halves_and_shared_workspace(updated):
    import torch
    from marl_mass_b200 import rollout
    shared, pol, (idx, S, A8, G), saved = updated
    for kind, net, _ in _pairs(pol, shared):
        old = None if kind == "critic" else rollout.ppo_targets(saved[kind], S, A8, idx)
        a, b = _stats(net, S, A8, G, idx, old), _stats(net, S, A8, G, idx, old)
        assert a.tobytes() == b.tobytes(), kind
        h = idx.numel() // 3
        x, y = _stats(net, S, A8, G, idx[:h], old), _stats(net, S, A8, G, idx[h:], old)
        for f in range(len(a)):
            if f == K["ratio_min"]:
                assert min(x[f], y[f]) == a[f]
            elif f == K["ratio_max"]:
                assert max(x[f], y[f]) == a[f]
            elif f in (K["n"], K["clipped"]):
                assert x[f] + y[f] == a[f]
            else:
                assert abs(x[f] + y[f] - a[f]) <= 1e-13 * max(abs(a[f]), abs(x[f]) + abs(y[f])), (kind, f)
    # the statistics partials share mm_ppo_grads' workspace: interleaved calls leave the gradients as they were
    kinds = _pairs(pol, shared)
    old = rollout.ppo_targets(saved[kinds[0][0]], S, A8, idx)
    j = idx[: 200_000]

    def grads():
        if shared:
            rollout.shared_network_gradients(pol.policy, S, A8, G, old, j, CLIP)
            return [p.grad.clone() for p in pol.policy.parameters()]
        q = rollout.ppo_targets(saved["critic"], S, A8, idx)
        rollout.mappo_gradients(pol.actor, pol.critic, S, A8, G, old, q, j, CLIP)
        return [p.grad.clone() for p in list(pol.actor.parameters()) + list(pol.critic.parameters())]

    g0 = grads()
    for kind, net, _ in kinds:
        _stats(net, S, A8, G, idx, None if kind == "critic" else old)
    g1 = grads()
    _stats(kinds[0][1], S, A8, G, idx[:77], None if kinds[0][0] == "critic" else old)
    g2 = grads()
    for x, y, z in zip(g0, g1, g2):
        assert torch.equal(x, y) and torch.equal(x, z)


def test_cuda_and_torch_statistics_agree(updated):
    """the kernel (fp16 operands) against ppo_stats_torch (fp32) on the same networks and rows.  Tolerances: N, exact;
    entropy and value sums 2e-3 relative; the ratio range 2e-3 relative; approx_kl and clip fraction within 0.25 of the
    torch values relative, + 1e-5 absolute (both are differences of nearby log-probabilities, where the fp16 roundings of
    the two networks do not cancel)"""
    from marl_mass_b200 import rollout
    shared, pol, (idx, S, A8, G), saved = updated
    for kind, net, _ in _pairs(pol, shared):
        old = None if kind == "critic" else rollout.ppo_targets(saved[kind], S, A8, idx)
        old_t = None if kind == "critic" else rollout._ppo_stats_torch(saved[kind], S, A8, G, idx, None, CLIP)[1]
        if old_t is not None:
            o = old.clone()
            o[idx] = old_t
            old_t = o
        c = _stats(net, S, A8, G, idx, old)
        t = rollout.ppo_stats_torch(net, S, A8, G, idx, old_t, CLIP).cpu().numpy()
        n = c[K["n"]]
        assert c[K["n"]] == t[K["n"]]
        for f in VALUE + [K["entropy"], K["ratio_min"], K["ratio_max"]]:
            if math.isinf(t[f]):
                assert c[f] == t[f]
            else:
                assert abs(c[f] - t[f]) <= 2e-3 * max(abs(t[f]), 1.0), (kind, ppo_stats_ref.FIELDS[f], c[f], t[f])
        for f in ("k3", "clipped"):
            assert abs(c[K[f]] - t[K[f]]) / n <= 0.25 * abs(t[K[f]]) / n + 1e-5, (kind, f, c[K[f]] / n, t[K[f]] / n)


@pytest.mark.parametrize("impl", ["torch", "cuda"])
@pytest.mark.parametrize("shared", [False, True], ids=["mappo", "shared"])
def test_update_with_stats_is_the_same_update(mm, shared, impl):
    """update(stats=True) against update(stats=False) from the same networks, optimiser state, rollout and torch seed,
    three minibatches: every parameter and loss bit for bit; the new keys in their ranges"""
    import torch
    env, pol_a = _rollout(shared, envs=512, steps=30)
    nets = {"policy": copy.deepcopy(pol_a.policy)} if shared else {"actor": copy.deepcopy(pol_a.actor),
                                                                    "critic": copy.deepcopy(pol_a.critic)}
    from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout
    from marl_mass_b200.train import load_ini
    ini = "mass_td3_mixed_srew_shared.ini" if shared else "mass_td3_srew.ini"
    _, rkw, _ = load_ini(os.path.join(ROOT, "examples", ini))
    rkw["roll_out_n_steps"] = 30
    pol_b = (BatchedMAPPOGIRollout if shared else BatchedMAPPORollout)(env, seed=5, **nets, **rkw)
    pol_b.buf = pol_a.buf
    mb = pol_a._learner_batch()[0].numel() // 3 + 1
    torch.manual_seed(21)
    ra = pol_a.update(minibatch=mb, impl=impl)
    torch.manual_seed(21)
    rb = pol_b.update(minibatch=mb, impl=impl, stats=True)
    for m_a, m_b in zip(pol_a.networks(), pol_b.networks()):
        for (name, p), q in zip(m_a.named_parameters(), m_b.parameters()):
            assert torch.equal(p, q), (shared, impl, name)
    assert {k: rb[k] for k in ra} == ra
    assert set(rb) - set(ra) == {"approx_kl", "clip_fraction", "ratio_min", "ratio_max", "entropy_before", "entropy_after",
                                 "explained_variance_before", "explained_variance_after", "advantage_mean", "advantage_std"}
    for k in ("entropy_before", "entropy_after"):
        assert 0 < rb[k] <= math.log(5) * (1 + 1e-6), (k, rb[k])
    assert 0 <= rb["clip_fraction"] <= 1 and rb["approx_kl"] >= 0
    assert 0 < rb["ratio_min"] <= 1 <= rb["ratio_max"]
    assert all(math.isfinite(rb[k]) for k in rb)
    env.close()


@pytest.mark.parametrize("impl", ["torch", "cuda"])
@pytest.mark.parametrize("ini", ["mass_td3_srew.ini", "mass_td3_mixed_srew_shared.ini"])
def test_driver_logs_update_stats_and_leaves_the_rest(mm, ini, impl):
    from marl_mass_b200.train import train
    path = os.path.join(ROOT, "examples", ini)
    timing = {"collect_s", "update_s", "agent_steps_per_s"}
    off = train(path, n_envs=256, iterations=2, eval_interval=0, update_impl=impl, log=lambda *_: None)
    on = train(path, n_envs=256, iterations=2, eval_interval=0, update_impl=impl, update_stats=True, log=lambda *_: None)
    for a, b in zip(off, on):
        new = set(b) - set(a)
        assert new == {"update_" + k for k in ("approx_kl", "clip_fraction", "ratio_min", "ratio_max", "entropy_before",
                                               "entropy_after", "explained_variance_before", "explained_variance_after",
                                               "advantage_mean", "advantage_std")}
        assert all(math.isfinite(b[k]) for k in new)
        assert {k: v for k, v in a.items() if k not in timing} == {k: b[k] for k in a if k not in timing}

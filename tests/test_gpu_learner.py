"""GPU suite, learner: the on-device PPO update (mm_ppo_targets / mm_ppo_grads through rollout.ppo_targets,
mappo_gradients, shared_network_gradients and update(impl="cuda")) against torch autograd in fp32 (TF32 off) on the
same rows.

Two references.  "fp32": the torch modules as they are.  "fp16 operands": the same autograd graph in fp32, with the
inputs, the weights and the hidden activations rounded to fp16 where the kernels round them (straight-through, so the
gradient is still taken with respect to the fp32 parameters).  Against the fp32 reference the kernels' forward differs by
fp16 rounding (~1e-4 of a pre-activation), which flips the ReLU mask of a few (row, unit) pairs and the clip decision
of rows next to a bound; on rows from collect() these flips average out, on a hundred synthetic N(0, 1) rows with
random networks (whose per-row contributions nearly cancel in the mean) they alone moved a bias gradient by 5e-2.  The
fp16-operand reference takes the same forward decisions, so it bounds what the gradient pass adds on top of its
forward: the fp16 rounding of the backward's dZ operands and the accumulation order.

Tolerances: per parameter tensor ||g_cuda - g_ref|| / ||g_ref|| <= 1e-2 against the fp16-operand reference on every
case and against the fp32 reference on rows from collect(); losses within 1e-3 relative; log-probabilities / Q values of
the target pass within 2e-2 absolute of the fp32 network.  Against fp32 on returns of reward_scale = 1 and in the later
minibatches of a real update, 3e-2 per tensor and 1e-2 on the losses: there the kernels stay within 3.4e-3 of the
fp16-operand reference while the fp32 gap reaches 1.3e-2, so the gap is the fp16 rounding of the forward, which that
reference models; which part of it is not isolated (leaving out the rows within 1e-2 of a clip bound did not shrink it).  test_gpu_learner_exact.py checks the kernels bit for bit on exactly representable data.
"""
import copy
import glob
import math
import os

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

GRAD_TOL = 1e-2
FP32_WIDE_TOL = 3e-2     # against fp32 after the first minibatch of an update and on large returns (module docstring)
LOSS_TOL = 1e-3
FWD_TOL = 2e-2
CLIP = 0.2


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return m


def _nets(kind, seed):
    import torch
    from marl_mass_b200 import rollout
    torch.manual_seed(seed)
    if kind == "mappo":
        return rollout.ActorNetwork().cuda(), rollout.CriticNetwork().cuda()
    return (rollout.ActorCriticNetwork().cuda(),)


def _rnd(t):
    """fp16 rounding in the forward, identity in the backward"""
    return t + (t.half().float() - t).detach()


def _fwd_fp16(kind, nets, s, onehot):
    """the networks' forward with fp16 operands where the kernels have them: -> (log-probabilities, values)"""
    import torch
    from torch.nn import functional as F
    lin = lambda x, m: F.linear(x, _rnd(m.weight), m.bias)  # noqa: E731
    s = _rnd(s)
    if kind == "mappo":
        actor, critic = nets
        h = _rnd(torch.relu(lin(_rnd(torch.relu(lin(s, actor.fc1))), actor.fc2)))
        logp = torch.log_softmax(lin(h, actor.fc3), -1)
        h = _rnd(torch.relu(lin(s, critic.fc1)))
        h = _rnd(torch.relu(lin(torch.cat([h, onehot], -1), critic.fc2)))
        return logp, lin(h, critic.fc3)
    (pol,) = nets
    h = torch.cat([torch.relu(lin(s[:, list(c)], m)) for c, m in ((pol.COLS1, pol.fc11), (pol.COLS2, pol.fc12),
                                                                 (pol.COLS3, pol.fc13))], 1)
    h = _rnd(torch.relu(lin(_rnd(h), pol.fc2)))
    return torch.log_softmax(lin(h, pol.actor_linear), 1), lin(h, pol.critic_linear)


def _torch_losses(kind, nets, S, A8, G, old_logp, q_target, j, operands="fp32"):
    """torch autograd on rows j with the given per-row constants (the losses of mappo_losses / shared_network_loss);
    operands "fp16": the forward with the kernels' fp16 roundings (module docstring)"""
    import torch
    from torch import nn
    s, a = S[j], A8[j].long()
    onehot = nn.functional.one_hot(a, 5).float()
    g = G[j]
    if operands == "fp16":
        logp_all, values = _fwd_fp16(kind, nets, s, onehot)
        logp = (logp_all * onehot).sum(1)
        ratio = torch.exp(logp - old_logp[j])
        adv = g - q_target[j] if kind == "mappo" else (g[:, None] - values.detach()).squeeze(1)
        a_loss = -torch.min(ratio * adv, torch.clamp(ratio, 1 - CLIP, 1 + CLIP) * adv).mean()
        return a_loss, nn.functional.mse_loss(values, g[:, None])
    if kind == "mappo":
        actor, critic = nets
        logp = (actor(s) * onehot).sum(1)
        ratio = torch.exp(logp - old_logp[j])
        adv = g - q_target[j]
        a_loss = -torch.min(ratio * adv, torch.clamp(ratio, 1 - CLIP, 1 + CLIP) * adv).mean()
        c_loss = nn.functional.mse_loss(critic(s, onehot), g[:, None])
        return a_loss, c_loss
    (pol,) = nets
    hidden = pol.trunk(s)
    logp = (pol.policy_head(hidden) * onehot).sum(1)
    values = pol.critic_linear(hidden)
    adv = (g[:, None] - values.detach()).squeeze(1)
    ratio = torch.exp(logp - old_logp[j])
    a_loss = -torch.min(ratio * adv, torch.clamp(ratio, 1 - CLIP, 1 + CLIP) * adv).mean()
    c_loss = nn.functional.mse_loss(values, g[:, None])
    return a_loss, c_loss


def _params(nets):
    return [(name, p) for k, m in enumerate(nets) for name, p in m.named_parameters(prefix="net%d" % k)]


def _torch_grads(kind, nets, S, A8, G, old_logp, q_target, j, operands="fp32"):
    for _, p in _params(nets):
        p.grad = None
    a_loss, c_loss = _torch_losses(kind, nets, S, A8, G, old_logp, q_target, j, operands)
    (a_loss + c_loss).backward()
    out = {n: p.grad.clone() for n, p in _params(nets)}
    for _, p in _params(nets):
        p.grad = None
    return out, float(a_loss.detach()), float(c_loss.detach())


def _cuda_grads(kind, nets, S, A8, G, old_logp, q_target, j):
    from marl_mass_b200 import rollout
    for _, p in _params(nets):
        p.grad = None
    if kind == "mappo":
        a, c = rollout.mappo_gradients(nets[0], nets[1], S, A8, G, old_logp, q_target, j, CLIP)
    else:
        _, a, c = rollout.shared_network_gradients(nets[0], S, A8, G, old_logp, j, CLIP)
    out = {n: p.grad.clone() for n, p in _params(nets)}
    for _, p in _params(nets):
        p.grad = None
    return out, float(a), float(c)


def _random_rows(rows, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    S = torch.randn((rows, 30), device="cuda", generator=g)
    A8 = torch.randint(0, 5, (rows,), device="cuda", generator=g).to(torch.int8)
    G = 3.0 * torch.randn(rows, device="cuda", generator=g)
    return S, A8, G


def _collected_rows(shared, envs=1024, steps=100, reward_scale=None):
    import torch
    from marl_mass_b200.env import DEFAULT_CONFIG, MergeEnvBatched
    from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout
    from marl_mass_b200.train import load_ini
    ini = "mass_td3_mixed_srew_shared.ini" if shared else "mass_td3_srew.ini"
    env_cfg, kw, _ = load_ini(os.path.join(ROOT, "examples", ini))
    kw["roll_out_n_steps"] = steps
    if reward_scale is not None:
        kw["reward_scale"] = reward_scale
    env = MergeEnvBatched(envs, dict(DEFAULT_CONFIG, **env_cfg), device=0)
    torch.manual_seed(11)
    pol = (BatchedMAPPOGIRollout if shared else BatchedMAPPORollout)(env, seed=5, **kw)
    b = pol.collect()
    torch.cuda.synchronize()
    S = b["states"].reshape(-1, 30)
    A8 = b["actions"].reshape(-1).to(torch.int8)
    G = b["returns"].reshape(-1).contiguous()
    live = b["live"].reshape(-1).nonzero().squeeze(1)
    env.close()
    return pol, S, A8, G, live


def _rel(a, b):
    return float((a - b).norm() / max(float(b.norm()), 1e-30))


def _check_grads(gc, gt, lc, lt, tag, tol=GRAD_TOL):
    worst = 0.0
    for n in gt:
        e = _rel(gc[n], gt[n])
        worst = max(worst, e)
        assert e <= tol, (tag, n, e)
    for x, y in zip(lc, lt):
        assert abs(x - y) <= LOSS_TOL * max(abs(y), 1e-3), (tag, x, y)
    return worst


def _constants(kind, nets, S, A8, live, seed):
    """old log-probabilities spread around the current policy's (ratios roughly in exp(+-0.3)) and a Q_target"""
    import torch
    from marl_mass_b200 import rollout
    g = torch.Generator(device="cuda").manual_seed(seed)
    noise = 0.15 * torch.randn(S.shape[0], device="cuda", generator=g)
    # ratios exp(-noise) within 2e-2 of a clip bound would flip between clipped and unclipped under the fp16 forward's
    # rounding: such rows get the current log-probability (r = 1) instead
    r = torch.exp(-noise)
    noise = torch.where(((r - (1 + CLIP)).abs() < 2e-2) | ((r - (1 - CLIP)).abs() < 2e-2), torch.zeros_like(noise), noise)
    old = rollout.ppo_targets(nets[0], S, A8, live) + noise
    q = rollout.ppo_targets(nets[1], S, A8, live) if kind == "mappo" else None
    return old, q


@pytest.mark.parametrize("kind", ["mappo", "shared"])
@pytest.mark.parametrize("source", ["random", "collected", "collected_unscaled"])
@pytest.mark.parametrize("n", [100003, 127, 1])
def test_gradients_match_torch_autograd(mm, kind, source, n):
    """All parameter tensors (MAPPO actor + critic; the shared network with fc11 / fc12 / fc13 folded back from the dense
    first layer and the value head critic_linear), rows in random order, n not a multiple of 128.
    Against the fp16-operand reference on every case, against the fp32 reference on rows from collect().
    "collected_unscaled": collect() with reward_scale = 1, returns up to a few hundred (2 (Q - G) and the advantages
    enter fp16 that large); there the fp32 comparison is held to FP32_WIDE_TOL (on a B200, 1.1e-2 on fc1.weight at
    n = 100 003), the fp16-operand one to GRAD_TOL."""
    import torch
    if source == "random":
        rows = 200000
        S, A8, G = _random_rows(rows, 1 + n)
        live = torch.arange(rows, device="cuda")
        nets = _nets(kind, 7)
    else:
        pol, S, A8, G, live = _collected_rows(kind == "shared", reward_scale=1.0 if source == "collected_unscaled" else None)
        nets = (pol.actor, pol.critic) if kind == "mappo" else (pol.policy,)
        if source == "collected_unscaled":
            assert float(G[live].abs().max()) > 100.0
    old, q = _constants(kind, nets, S, A8, live, 3)
    torch.manual_seed(n)
    j = live[torch.randperm(live.numel(), device="cuda")[:n]]
    gc, ac, cc = _cuda_grads(kind, nets, S, A8, G, old, q, j)
    if kind == "shared":     # the folded first layer: each block's gradient, and the value head, checked by name
        assert {"net0.fc11.weight", "net0.fc12.weight", "net0.fc13.weight", "net0.critic_linear.weight"} <= set(gc)
    gt, at, ct = _torch_grads(kind, nets, S, A8, G, old, q, j, "fp16")
    _check_grads(gc, gt, (ac, cc), (at, ct), (kind, source, n, "fp16 operands"))
    if source != "random":
        gt, at, ct = _torch_grads(kind, nets, S, A8, G, old, q, j)
        _check_grads(gc, gt, (ac, cc), (at, ct), (kind, source, n, "fp32"),
                     GRAD_TOL if source == "collected" else FP32_WIDE_TOL)


def test_shared_first_layer_gradient_lands_on_the_blocks_only(mm):
    """The kernel differentiates the dense 30 -> 160 layer; fc11 / fc12 / fc13 get their own blocks of it (shapes and
    values against autograd), and the value head critic_linear its gradient."""
    import torch
    from marl_mass_b200 import rollout
    S, A8, G = _random_rows(5000, 9)
    (pol,) = _nets("shared", 2)
    live = torch.arange(5000, device="cuda")
    old = rollout.ppo_targets(pol, S, A8, live)
    gc, _, _ = _cuda_grads("shared", (pol,), S, A8, G, old, None, live)
    gt, _, _ = _torch_grads("shared", (pol,), S, A8, G, old, None, live, "fp16")
    for name, shape in (("fc11", (32, 5)), ("fc12", (64, 10)), ("fc13", (64, 10))):
        assert tuple(gc["net0.%s.weight" % name].shape) == shape
        assert _rel(gc["net0.%s.weight" % name], gt["net0.%s.weight" % name]) <= GRAD_TOL
        assert _rel(gc["net0.%s.bias" % name], gt["net0.%s.bias" % name]) <= GRAD_TOL
    assert _rel(gc["net0.critic_linear.weight"], gt["net0.critic_linear.weight"]) <= GRAD_TOL
    assert _rel(gc["net0.critic_linear.bias"], gt["net0.critic_linear.bias"]) <= GRAD_TOL


def test_ratio_and_clip_regimes(mm):
    """Rows with r == 1 exactly, r above 1 + c and below 1 - c, advantages positive, negative and zero: clipped rows and
    zero-advantage rows contribute exactly nothing, the others what torch gives (ties included; against the fp16-operand
    reference, whose ratios are the kernels' up to accumulation order)."""
    import torch
    from marl_mass_b200 import rollout
    rows = 60000
    S, A8, _ = _random_rows(rows, 21)
    actor, critic = _nets("mappo", 4)
    live = torch.arange(rows, device="cuda")
    logp = rollout.ppo_targets(actor, S, A8, live)          # r == 1 exactly against these (same forward arithmetic)
    q = torch.zeros(rows, device="cuda")
    regime = torch.arange(rows, device="cuda") % 9           # (ratio kind, advantage sign) pairs
    rk, ak = regime // 3, regime % 3
    old = torch.where(rk == 0, logp, torch.where(rk == 1, logp - math.log(1.6), logp - math.log(0.5)))
    G = torch.where(ak == 0, torch.full_like(q, 2.0), torch.where(ak == 1, torch.full_like(q, -1.5), q))

    def grads(sel):
        j = live[sel]
        return _cuda_grads("mappo", (actor, critic), S, A8, G, old, q, j)[0]

    actor_names = [n for n in _params((actor,))]
    for sel in ((rk == 1) & (ak == 0), (rk == 2) & (ak == 1), ak == 2):      # clipped, clipped, zero advantage
        g = grads(sel)
        for n, _ in actor_names:
            assert float(g[n].abs().max()) == 0.0, n
    for sel in ((rk == 0) & (ak != 2), (rk == 1) & (ak == 1), (rk == 2) & (ak == 0), torch.ones(rows, dtype=torch.bool, device="cuda")):
        j = live[sel]
        gc, ac, _ = _cuda_grads("mappo", (actor, critic), S, A8, G, old, q, j)
        gt, at, _ = _torch_grads("mappo", (actor, critic), S, A8, G, old, q, j, "fp16")
        for n, _ in actor_names:
            assert _rel(gc[n], gt[n]) <= GRAD_TOL, n
        assert abs(ac - at) <= LOSS_TOL * max(abs(at), 1e-3)


@pytest.mark.parametrize("kind", ["mappo", "shared"])
def test_gradient_pass_is_deterministic(mm, kind):
    import torch
    from marl_mass_b200 import rollout
    rows = 150000
    S, A8, G = _random_rows(rows, 31)
    nets = _nets(kind, 8)
    live = torch.arange(rows, device="cuda")
    old, q = _constants(kind, nets, S, A8, live, 5)
    j = live[torch.randperm(rows, device="cuda")[:100003]]
    g1, a1, c1 = _cuda_grads(kind, nets, S, A8, G, old, q, j)
    g2, a2, c2 = _cuda_grads(kind, nets, S, A8, G, old, q, j)
    assert (a1, c1) == (a2, c2)
    for n in g1:
        assert torch.equal(g1[n], g2[n]), n


def test_target_pass_matches_the_target_networks_and_gives_ratio_one(mm):
    import torch
    from torch import nn
    from marl_mass_b200 import rollout
    rows = 70000
    S, A8, _ = _random_rows(rows, 41)
    actor, critic = _nets("mappo", 12)
    (pol,) = _nets("shared", 13)
    live = torch.randperm(rows, device="cuda")[:65536]
    onehot = nn.functional.one_hot(A8.long(), 5).float()
    with torch.no_grad():
        want_a = (actor(S) * onehot).sum(1)
        want_q = critic(S, onehot).squeeze(1)
        want_p = (pol(S) * onehot).sum(1)
    old = rollout.ppo_targets(actor, S, A8, live)
    qt = rollout.ppo_targets(critic, S, A8, live)
    oldp = rollout.ppo_targets(pol, S, A8, live)
    assert float((old[live] - want_a[live]).abs().max()) < FWD_TOL
    assert float((qt[live] - want_q[live]).abs().max()) < FWD_TOL * max(1.0, float(want_q.abs().max()))
    assert float((oldp[live] - want_p[live]).abs().max()) < FWD_TOL
    # actor == its target: every ratio is exactly 1, so with advantage 1 (returns 1, Q_target 0) the surrogate is exactly
    # -mean(1) = -1 over 2^16 rows (any r = 1 +- ulp would move the sum)
    G = torch.ones(rows, device="cuda")
    q0 = torch.zeros(rows, device="cuda")
    a_loss, _ = rollout.mappo_gradients(actor, critic, S, A8, G, old, q0, live, CLIP)
    assert float(a_loss) == -1.0
    _, a_loss, _ = rollout.shared_network_gradients(pol, S, A8, G, oldp, live, CLIP)
    # r == 1: the surrogate is -mean(G - V), V the value head; against the float64 restatement (fp16 rounding apart)
    import learner_ref
    params = {n: p.detach().double().cpu().numpy() for n, p in pol.named_parameters()}
    S64, A64, G64, live64 = S.cpu().numpy(), A8.cpu().numpy(), G.cpu().numpy(), live.cpu().numpy()
    t = learner_ref.learner_pass("shared", params, S64, A64, None, None, None, np.arange(rows), CLIP)
    want = learner_ref.learner_pass("shared", params, S64, A64, G64, t["logp"], None, live64, CLIP)["loss_a"]
    assert want == pytest.approx(-float(np.mean(G64[live64] - t["v"][live64])), rel=1e-12)
    assert abs(float(a_loss) - want) <= LOSS_TOL * max(abs(want), 1e-3), (float(a_loss), want)


@pytest.mark.parametrize("write", ["torch_op", "data_then_sync"])
def test_shared_first_layer_follows_parameter_writes(mm, write):
    """policy_sample, ppo_targets and shared_network_gradients run the shared network's first layer as it is at the
    call, although the dense 30 -> 160 layer is kept on the module between calls.  "torch_op": the parameters
    overwritten by an in-place torch op (as optimizer steps and load_state_dict write; torch bumps _version).
    "data_then_sync": overwritten through .data, which bumps no _version (sync_parameters' broadcast writes this way),
    then sync_parameters, which drops the kept layer."""
    import torch
    from torch import nn
    from marl_mass_b200 import rollout
    rows = 5000
    S, A8, G = _random_rows(rows, 51)
    live = torch.arange(rows, device="cuda")
    (pol,), (other,) = _nets("shared", 21), _nets("shared", 22)
    with torch.no_grad():
        for p in other.parameters():
            p.mul_(3.0)                     # log-probabilities far from pol's
    ro = rollout.BatchedMAPPOGIRollout.__new__(rollout.BatchedMAPPOGIRollout)     # only its networks are used
    ro.policy, ro.policy_target = pol, _nets("shared", 23)[0]
    old = rollout.ppo_targets(pol, S, A8, live)
    rollout.shared_network_gradients(pol, S, A8, G, old, live, CLIP)
    rollout.policy_sample(pol, S, want_logp=True)
    if write == "torch_op":
        with torch.no_grad():
            for p, q in zip(pol.parameters(), other.parameters()):
                p.copy_(q)
    else:
        versions = [p._version for p in pol.parameters()]
        for p, q in zip(pol.parameters(), other.parameters()):
            p.data.copy_(q.data)
        assert [p._version for p in pol.parameters()] == versions
        ro.sync_parameters()
    onehot = nn.functional.one_hot(A8.long(), 5).float()
    with torch.no_grad():
        want_all = other(S)
        want = (want_all * onehot).sum(1)
    assert float((want - old).abs().max()) > 10 * FWD_TOL      # a stale first layer would show
    got = rollout.ppo_targets(pol, S, A8, live)
    assert float((got - want).abs().max()) < FWD_TOL
    _, logp = rollout.policy_sample(pol, S, want_logp=True)
    assert float((logp - want_all).abs().max()) < FWD_TOL
    gc, _, _ = _cuda_grads("shared", (pol,), S, A8, G, got, None, live)
    gt, _, _ = _torch_grads("shared", (pol,), S, A8, G, got, None, live, "fp16")
    for n in gt:
        assert _rel(gc[n], gt[n]) <= GRAD_TOL, (n, _rel(gc[n], gt[n]))


@pytest.mark.parametrize("shared", [False, True])
def test_whole_update_cuda_against_torch(mm, shared):
    """update(impl="cuda") and update(impl="torch") from identical copies of the networks and optimisers on one rollout
    buffer, one minibatch: the same losses, parameter deltas with cosine >= 0.99 per tensor (RMSprop divides by the
    running RMS of the gradient, which amplifies fp16 noise in near-zero entries, so not elementwise), targets re-synced."""
    import torch
    pol, S, A8, G, live = _collected_rows(shared, envs=512, steps=60)
    mods = pol.networks()
    opts = [pol.policy_opt] if shared else [pol.actor_opt, pol.critic_opt]
    saved = [copy.deepcopy(m.state_dict()) for m in mods], [copy.deepcopy(o.state_dict()) for o in opts]
    before = [p.detach().clone() for m in mods[:1 if shared else 2] for p in m.parameters()]

    def run(impl):
        for m, sd in zip(mods, saved[0]):
            m.load_state_dict(sd)
        for o, sd in zip(opts, saved[1]):
            o.load_state_dict(sd)
        torch.manual_seed(99)
        stats = pol.update(minibatch=1 << 22, impl=impl)
        after = [p.detach().clone() for m in mods[:1 if shared else 2] for p in m.parameters()]
        for m, t in ((pol.policy, pol.policy_target),) if shared else ((pol.actor, pol.actor_target), (pol.critic, pol.critic_target)):
            for p, q in zip(m.parameters(), t.parameters()):
                assert torch.equal(p, q)
        return stats, after

    st_t, after_t = run("torch")
    st_c, after_c = run("cuda")
    assert st_t["samples"] == st_c["samples"] == live.numel()
    for k in ("actor_loss", "critic_loss"):
        assert abs(st_c[k] - st_t[k]) <= LOSS_TOL * max(abs(st_t[k]), 1e-3), (k, st_c[k], st_t[k])
    for b, t, c in zip(before, after_t, after_c):
        dt, dc = (t - b).reshape(-1), (c - b).reshape(-1)
        if float(dt.norm()) == 0.0:
            assert float(dc.norm()) == 0.0
            continue
        cos = float(torch.dot(dt, dc) / (dt.norm() * dc.norm()))
        assert cos >= 0.99, cos


@pytest.mark.parametrize("shared", [False, True])
def test_every_minibatch_of_a_real_update_matches_autograd(mm, monkeypatch, shared):
    """update(impl="cuda") on a collect() buffer of the shipped ini, 8 minibatches x 2 epochs: after every gradient pass
    the kernel's gradients and losses are held against torch autograd on the same rows with the networks as they are at
    that moment, old_logp / Q_target from the target networks as torch computes them.  From the second minibatch on the
    networks have left their targets, so ratios leave 1 and clipping acts.

    Against the fp16-operand reference every minibatch meets the collected-rows standard (GRAD_TOL, LOSS_TOL).  Against
    the fp32 reference, once the networks have left their targets, the fp16 rounding of the forward moves some
    minibatches past it: on a B200 the worst reached 1.3e-2 on a weight tensor and 5.6e-3 on a loss (not explained by
    clip decisions: leaving out the rows within 1e-2 of a bound did not shrink it), so that comparison is held to
    FP32_WIDE_TOL and 10 LOSS_TOL, and its worst values are printed."""
    import torch
    from torch import nn
    from marl_mass_b200 import rollout
    pol, S, A8, G, live = _collected_rows(shared)
    kind = "shared" if shared else "mappo"
    nets = (pol.policy,) if shared else (pol.actor, pol.critic)
    with torch.no_grad():
        onehot = nn.functional.one_hot(A8.long(), 5).float()
        tgt = pol.policy_target if shared else pol.actor_target
        old = (tgt(S) * onehot).sum(1)
        q = None if shared else pol.critic_target(S, onehot).squeeze(1)
    name = "shared_network_gradients" if shared else "mappo_gradients"
    kernel = getattr(rollout, name)
    seen = []

    def checked(*args, **kw):
        out = kernel(*args, **kw)
        j = args[5 if shared else 7]
        gc = {n: p.grad.clone() for n, p in _params(nets)}
        lc = (float(out[1]), float(out[2])) if shared else (float(out[0]), float(out[1]))
        gt, at, ct = _torch_grads(kind, nets, S, A8, G, old, q, j, "fp16")
        worst = _check_grads(gc, gt, lc, (at, ct), (kind, len(seen), "fp16"))
        gt, at, ct = _torch_grads(kind, nets, S, A8, G, old, q, j)
        worst32 = max(_rel(gc[n], gt[n]) for n in gt)
        loss32 = max(abs(x - y) / max(abs(y), 1e-3) for x, y in zip(lc, (at, ct)))
        assert worst32 <= FP32_WIDE_TOL and loss32 <= 10 * LOSS_TOL, (kind, len(seen), worst32, loss32)
        with torch.no_grad():
            s, a = S[j], A8[j].long()
            head = pol.policy(s) if shared else pol.actor(s)
            r = torch.exp(head.gather(1, a[:, None]).squeeze(1) - old[j])
            adv = G[j] - (pol.policy(s, out_type="v").squeeze(1) if shared else q[j])
            clipped = ((r > 1 + CLIP) & (adv > 0)) | ((r < 1 - CLIP) & (adv < 0))
            seen.append((worst, worst32, loss32, float(((r - 1).abs() > 1e-3).float().mean()), float(clipped.float().mean())))
        for n, p in _params(nets):
            p.grad = gc[n]
        return out

    monkeypatch.setattr(rollout, name, checked)
    minibatch = live.numel() // 8 + 1
    torch.manual_seed(17)
    pol.update(minibatch=minibatch, epochs=2, impl="cuda")
    assert len(seen) == 16
    for k, (worst, worst32, loss32, off_one, clipped) in enumerate(seen):
        print("%s minibatch %2d: worst rel err %.2e (fp16 operands) %.2e (fp32), loss %.1e (fp32); r != 1 on %.4f of rows, "
              "clipped %.4f" % (kind, k, worst, worst32, loss32, off_one, clipped))
    assert seen[0][3] == 0.0                                       # the first minibatch runs at the target networks
    assert all(s[3] > 0.0 for s in seen[1:])                       # afterwards the ratios really left 1
    assert max(s[4] for s in seen) > 0.0


@pytest.mark.parametrize("ini", sorted(glob.glob(os.path.join(ROOT, "examples", "*.ini"))))
def test_driver_with_cuda_learner(mm, ini):
    from marl_mass_b200.train import train
    hist = train(ini, n_envs=512, iterations=2, eval_interval=1, log=lambda *_: None, update_impl="cuda")
    assert len(hist) == 2
    for rec in hist:
        assert math.isfinite(rec["actor_loss"]) and math.isfinite(rec["critic_loss"]) and rec["samples"] > 0
        assert math.isfinite(rec["eval_reward"])

"""CPU test of the PPO update loop (`BatchedMAPPORollout.update` / `BatchedMAPPOGIRollout.update` with impl="torch",
optimizer="torch"): learners with CPU networks on a synthetic rollout buffer, several minibatches and two epochs, with and
without the statistics passes, held bit for bit against the torch update as each learner ran it in a loop of its own,
restated below.  The CUDA learner, the device optimiser and gae_lambda run CUDA kernels: the GPU suite covers them."""
import copy

import pytest
import torch
from torch import nn

T, E, MINIBATCH, EPOCHS, CLIP, MAX_GRAD_NORM = 7, 16, 200, 2, 0.2, 0.5


def _learner(shared):
    """a learner built as `__new__` + what update() reads, on the CPU, with a random rollout buffer"""
    from marl_mass_b200 import rollout as R
    cls = R.BatchedMAPPOGIRollout if shared else R.BatchedMAPPORollout
    ro = cls.__new__(cls)
    torch.manual_seed(1)
    ro.dev, ro.gae_lambda, ro.optimizer = torch.device("cpu"), None, "torch"
    ro.clip_param, ro.max_grad_norm = CLIP, MAX_GRAD_NORM
    if shared:
        ro.policy, ro.policy_target = R.ActorCriticNetwork(), R.ActorCriticNetwork()
        ro.policy_target.load_state_dict(ro.policy.state_dict())
        ro.policy_opt = torch.optim.RMSprop(ro.policy.parameters(), lr=5e-4)
    else:
        ro.actor, ro.critic = R.ActorNetwork(), R.CriticNetwork()
        ro.actor_target, ro.critic_target = R.ActorNetwork(), R.CriticNetwork()
        ro.actor_target.load_state_dict(ro.actor.state_dict())
        ro.critic_target.load_state_dict(ro.critic.state_dict())
        ro.actor_opt = torch.optim.RMSprop(ro.actor.parameters(), lr=5e-4)
        ro.critic_opt = torch.optim.RMSprop(ro.critic.parameters(), lr=1e-3)
    ro.buf = dict(states=torch.randn(T, E, 12, 30), actions=torch.randint(0, 5, (T, E, 12)), returns=torch.randn(T, E, 12),
                  live=torch.rand(T, E, 12) < 0.7)
    return ro


def _triples(ro, shared):
    """(network, target network, optimiser) of every trained network"""
    if shared:
        return [(ro.policy, ro.policy_target, ro.policy_opt)]
    return [(ro.actor, ro.actor_target, ro.actor_opt), (ro.critic, ro.critic_target, ro.critic_opt)]


def _stats_vector(nets, S, A8, G, idx, old_logp):
    """the statistics vector of (policy network, value network) with ppo_stats_torch"""
    from marl_mass_b200 import _lib
    from marl_mass_b200.rollout import ppo_stats_torch
    pol, val = nets
    v = ppo_stats_torch(pol, S, A8, G, idx, old_logp, CLIP)
    if val is not pol:
        vf = _lib.PPO_STAT["v"]
        v[vf:] = ppo_stats_torch(val, S, A8, G, idx, None, CLIP)[vf:]
    return v


def _reference_update(ro, shared, stats):
    """the torch update before MAPPO and MAPPO_GI shared one loop (one process, no gae_lambda): the whole buffer's one-hot
    actions, both losses read on the host after every minibatch, MAPPO's actor stepped before its critic is
    back-propagated"""
    from marl_mass_b200.rollout import NA, NS, mappo_losses, ppo_stats_keys, shared_network_loss
    b = ro.buf
    idx = b["live"].reshape(-1).nonzero(as_tuple=False).squeeze(1)
    S = b["states"].reshape(-1, NS)
    A = nn.functional.one_hot(b["actions"].reshape(-1), NA).float()
    G = b["returns"].reshape(-1, 1)
    if stats:
        A8, G1 = b["actions"].reshape(-1).to(torch.int8), G.reshape(-1)
        nets = (ro.policy_target,) * 2 if shared else (ro.actor_target, ro.critic_target)
        before = _stats_vector(nets, S, A8, G1, idx, None)
        with torch.no_grad():
            old_logp = torch.zeros(S.shape[0])
            old_logp[idx] = (nets[0](S[idx]) * A[idx]).sum(1)
    rec = {}
    for _ in range(EPOCHS):
        perm = idx[torch.randperm(idx.numel(), device=ro.dev)]
        for j in torch.tensor_split(perm, max(1, -(-idx.numel() // MINIBATCH))):
            if shared:
                loss, a_loss, c_loss = shared_network_loss(ro.policy, ro.policy_target, S[j], A[j], G[j], CLIP)
                steps = [(ro.policy, ro.policy_opt, loss)]
            else:
                a_loss, c_loss = mappo_losses(ro.actor, ro.actor_target, ro.critic, ro.critic_target, S[j], A[j], G[j], CLIP)
                steps = [(ro.actor, ro.actor_opt, a_loss), (ro.critic, ro.critic_opt, c_loss)]
            for net, opt, loss in steps:
                opt.zero_grad(set_to_none=True)
                loss.backward()
                nn.utils.clip_grad_norm_(list(net.parameters()), MAX_GRAD_NORM)
                opt.step()
            rec = {"actor_loss": float(a_loss.detach()), "critic_loss": float(c_loss.detach()), "samples": int(idx.numel())}
    if stats:
        nets = (ro.policy,) * 2 if shared else (ro.actor, ro.critic)
        rec.update(ppo_stats_keys(before.tolist(), _stats_vector(nets, S, A8, G1, idx, old_logp).tolist()))
    for net, target, _ in _triples(ro, shared):
        target.load_state_dict(net.state_dict())
    return rec


def _tensors(ro, shared):
    """every parameter of the networks and their targets, and every tensor of the optimiser states"""
    out = []
    for net, target, opt in _triples(ro, shared):
        out += list(net.parameters()) + list(target.parameters())
        for st in opt.state_dict()["state"].values():
            out += [st[k] for k in sorted(st)]
    return [t.detach() for t in out]


@pytest.mark.parametrize("stats", [False, True], ids=["plain", "stats"])
@pytest.mark.parametrize("shared", [False, True], ids=["mappo", "shared"])
def test_torch_update_matches_the_restated_loop(shared, stats):
    ro = _learner(shared)
    ref = copy.deepcopy(ro)
    assert int(ro.buf["live"].sum()) > 4 * MINIBATCH
    for it in range(2):        # the second update starts from stepped networks and optimiser state
        torch.manual_seed(10 + it)
        got = ro.update(minibatch=MINIBATCH, epochs=EPOCHS, impl="torch", stats=stats)
        torch.manual_seed(10 + it)
        want = _reference_update(ref, shared, stats)
        assert got == want
        assert len(got) == (13 if stats else 3)
        a, b = _tensors(ro, shared), _tensors(ref, shared)
        assert len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b))
    assert not torch.equal(_tensors(ro, shared)[0], _tensors(_learner(shared), shared)[0])      # the update moved them

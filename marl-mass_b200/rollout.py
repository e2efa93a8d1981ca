"""Batched MAPPO rollout on top of `MergeEnvBatched` (SURVEY.md §8f rank 1, BASELINE configs[3]).

The reference's `MAPPO.interact` (marl/mappo.py:102-158) steps ONE env, one agent at a time through a shared
actor; here the same data flow runs for E envs x up to 11 agents per step with no host synchronisation:

    obs [E,12,30] --actor--> log-probs --multinomial--> actions [E,12] int8 --env.step(auto_reset)--> ...

Kept from the reference: the networks (marl/single_agent/Model_common.py:5-40: actor 30-128-128-5 log-softmax,
critic on (state, one-hot action)), reward selection `regionalR | global_R` (mappo.py:122-125), reward scaling,
the discounted return (`_discount_reward`, mappo.py:364-370, final value 0 at episode end, critic bootstrap
otherwise) and the PPO-clip / critic losses of `MAPPO.train` (mappo.py:161-206) — batched over every live
(env, agent, t) sample instead of looped per agent.  The update runs as torch autograd (the default, and the numerics
reference) or, with `update(impl="cuda")`, through the learner kernels (mm_ppo_targets / mm_ppo_grads): one target
pass per update and one fused forward + backward per minibatch.
"""
import ctypes as C

import numpy as np
import torch
from torch import nn

from . import _lib
from . import dist as mmd
from ._lib import MAXV, NA, NS


class ActorNetwork(nn.Module):
    """marl/single_agent/Model_common.py:5-23 with output_act = log_softmax."""

    def __init__(self, state_dim=NS, hidden_size=128, output_size=NA):
        super().__init__()
        self.fc1 = nn.Linear(state_dim, hidden_size)
        self.fc2 = nn.Linear(hidden_size, hidden_size)
        self.fc3 = nn.Linear(hidden_size, output_size)

    def forward(self, state):
        out = torch.relu(self.fc1(state))
        out = torch.relu(self.fc2(out))
        return torch.log_softmax(self.fc3(out), dim=-1)


class CriticNetwork(nn.Module):
    """marl/single_agent/Model_common.py:26-41."""

    def __init__(self, state_dim=NS, action_dim=NA, hidden_size=128):
        super().__init__()
        self.fc1 = nn.Linear(state_dim, hidden_size)
        self.fc2 = nn.Linear(hidden_size + action_dim, hidden_size)
        self.fc3 = nn.Linear(hidden_size, 1)

    def forward(self, state, action_one_hot):
        out = torch.relu(self.fc1(state))
        out = torch.relu(self.fc2(torch.cat([out, action_one_hot], -1)))
        return self.fc3(out)


class ActorCriticNetwork(nn.Module):
    """marl/single_agent/Model_gi.py:137-220: the shared-trunk network of `MAPPO_GI` (mappo_gi.py:142-148 builds it
    with `state_split=True` and hidden size = critic_hidden_size).  The split reads the observation as five vehicles
    of FIVE features - presence | x, y | vx, vy - through fixed column lists that stop at column 24, also when the env
    delivers 5 x 6 = 30 columns (merge-multi-agent-v1): kept as the reference has it.  out_type "p": log-softmax over
    the actions, with `action_mask` the masked logits are -1e8 (Model_gi.py:207-213); "v": the state value."""
    COLS1 = (0, 5, 10, 15, 20)
    COLS2 = (1, 2, 6, 7, 11, 12, 16, 17, 21, 22)
    COLS3 = (3, 4, 8, 9, 13, 14, 18, 19, 23, 24)

    def __init__(self, state_dim=NS, action_dim=NA, hidden_size=128, critic_output_size=1, state_split=True):
        super().__init__()
        self.state_split = bool(state_split)
        if self.state_split:
            self.fc11 = nn.Linear(5, hidden_size // 4)
            self.fc12 = nn.Linear(10, hidden_size // 2)
            self.fc13 = nn.Linear(10, hidden_size // 2)
            self.fc2 = nn.Linear(hidden_size // 4 + hidden_size // 2 + hidden_size // 2, hidden_size)
        else:
            self.fc1 = nn.Linear(state_dim, hidden_size)
            self.fc2 = nn.Linear(hidden_size, hidden_size)
        self.actor_linear = nn.Linear(hidden_size, action_dim)
        self.critic_linear = nn.Linear(hidden_size, critic_output_size)

    def trunk(self, state):
        if self.state_split:
            out = torch.cat([torch.relu(self.fc11(state[:, self.COLS1])), torch.relu(self.fc12(state[:, self.COLS2])),
                             torch.relu(self.fc13(state[:, self.COLS3]))], 1)
        else:
            out = torch.relu(self.fc1(state))
        return torch.relu(self.fc2(out))

    def policy_head(self, hidden, action_mask=None):
        logits = self.actor_linear(hidden)
        if action_mask is not None:
            logits = torch.where(action_mask == 0, torch.full_like(logits, -1e8), logits)
            return torch.log_softmax(logits + 1e-8, dim=1)
        return torch.log_softmax(logits, dim=1)

    def forward(self, state, action_mask=None, out_type="p"):
        hidden = self.trunk(state)
        return self.policy_head(hidden, action_mask) if out_type == "p" else self.critic_linear(hidden)


def mappo_losses(actor, actor_target, critic, critic_target, states, actions_one_hot, returns, clip_param=0.2,
                 critic_loss="mse", pairwise=False):
    """The two losses of one `MAPPO.train` update (mappo.py:170-199): the PPO-clip surrogate with the advantage
    `return - Q_target(s, a)` for the actor, the regression of Q(s, a) on the return for the critic.  They share no
    parameters, so stepping the actor first (as the reference does) or both at once is the same update.
    `pairwise`: see `shared_network_loss`.  -> (actor_loss, critic_loss)"""
    with torch.no_grad():
        adv = returns - critic_target(states, actions_one_hot)
        old_logp = (actor_target(states) * actions_one_hot).sum(1)
    logp = (actor(states) * actions_one_hot).sum(1)
    ratio = torch.exp(logp - old_logp)
    if not pairwise:
        adv = adv.squeeze(1)
    actor_loss = -torch.min(ratio * adv, torch.clamp(ratio, 1.0 - clip_param, 1.0 + clip_param) * adv).mean()
    values = critic(states, actions_one_hot)
    if critic_loss == "huber":
        c_loss = nn.functional.smooth_l1_loss(values, returns)
    else:
        c_loss = nn.functional.mse_loss(values, returns)
    return actor_loss, c_loss


def shared_network_loss(policy, policy_target, states, actions_one_hot, returns, clip_param=0.2, critic_loss="mse",
                        pairwise=False):
    """The loss of one `MAPPO_GI.train` update with the shared network (mappo_gi.py:307-343): PPO-clip surrogate with
    the advantage `return - V(s)` (value detached) plus the value regression, summed.  -> (loss, actor_loss, critic_loss)

    `pairwise`: the reference multiplies `ratio` [N] by `advantages` [N, 1] (mappo_gi.py:313-326, mappo.py:173-183), which
    broadcasts to an [N, N] table of every ratio against every advantage before min / mean.  With its batches of 100
    samples that is what it trains on; with the 1e5..1e6-sample minibatches of the batched learner the table cannot
    exist, so the default is the per-sample PPO surrogate (ratio_i * adv_i) the formula stands for.  pairwise=True
    reproduces the reference's table (small batches; used to pin this function against the reference's arithmetic)."""
    hidden = policy.trunk(states)
    logp = (policy.policy_head(hidden) * actions_one_hot).sum(1)
    values = policy.critic_linear(hidden)
    adv = returns - values.detach()
    with torch.no_grad():
        old_logp = (policy_target(states) * actions_one_hot).sum(1)
    ratio = torch.exp(logp - old_logp)
    if not pairwise:
        adv = adv.squeeze(1)
    surr1 = ratio * adv
    surr2 = torch.clamp(ratio, 1.0 - clip_param, 1.0 + clip_param) * adv
    actor_loss = -torch.min(surr1, surr2).mean()
    if critic_loss == "huber":
        c_loss = nn.functional.smooth_l1_loss(values, returns)
    else:
        c_loss = nn.functional.mse_loss(values, returns)
    return actor_loss + c_loss, actor_loss, c_loss


def _ptr(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def discounted_returns(rewards, dones, final_value, gamma):
    """R_t = r_t + gamma * R_{t+1}, restarted after a terminal step (mappo.py:364-370 run per episode), one CUDA
    kernel for the whole rollout (mm_discounted_returns).

    rewards [T, E, A] f32 cuda, dones [T, E] (non-zero where step t ended the episode of env e), final_value [E, A]
    = bootstrap for the step after the last one (ignored where the last step was terminal) or None."""
    T, E, A = rewards.shape
    rewards = rewards.contiguous().float()
    d8 = (dones != 0).to(torch.uint8).contiguous()
    assert rewards.is_cuda and d8.shape == (T, E)
    fv = None if final_value is None else final_value.contiguous().float()
    out = torch.empty_like(rewards)
    _lib.check(_lib.lib().mm_discounted_returns(_ptr(rewards), _ptr(d8), _ptr(fv), C.c_float(gamma), T, C.c_int64(E * A),
                                                A, _ptr(out), _stream()))
    return out


def lambda_returns(rewards, dones, values, final_value, gamma, lam):
    """GAE(lambda) returns R_t = r_t + gamma * (lam * R_{t+1} + (1 - lam) * V_{t+1}), restarted after a terminal step, one
    CUDA kernel for the whole rollout (mm_lambda_returns, the kernel of `discounted_returns`).  lam = 1 gives
    `discounted_returns` bit for bit; lam = 0 the one-step targets r_t + gamma (1 - d_t) V_{t+1}.

    rewards, values [T, E, A] f32 cuda (values: V(s_t) of the networks that collected the rollout, finite wherever a
    recursion reads them - rows of an agent that does not exist are best zero), dones [T, E], final_value [E, A] or None
    (R and V after the last step)."""
    T, E, A = rewards.shape
    rewards = rewards.contiguous().float()
    values = values.contiguous().float()
    d8 = (dones != 0).to(torch.uint8).contiguous()
    assert rewards.is_cuda and d8.shape == (T, E) and values.shape == rewards.shape and values.device == rewards.device
    fv = None if final_value is None else final_value.contiguous().float()
    out = torch.empty_like(rewards)
    _lib.check(_lib.lib().mm_lambda_returns(_ptr(rewards), _ptr(d8), _ptr(values), _ptr(fv), C.c_float(gamma), C.c_float(lam),
                                            T, C.c_int64(E * A), A, _ptr(out), _stream()))
    return out


def check_gae_lambda(gae_lambda):
    """None, or the GAE lambda as a float in [0, 1]; anything else (a non-number, a bool, NaN, out of range) raises
    ValueError.  A string (an ini value) is parsed as a number."""
    if gae_lambda is None:
        return None
    x = gae_lambda
    if isinstance(x, str):
        try:
            x = float(x)
        except ValueError:
            x = None
    if isinstance(x, bool) or not isinstance(x, (int, float, np.integer, np.floating)) or not 0.0 <= float(x) <= 1.0:
        raise ValueError("gae_lambda must be None or a number in [0, 1], got %r" % (gae_lambda,))
    return float(x)


_ACTOR_IMPLS = {"tcgen05": 0, "mma": 1}


def set_actor_impl(name):
    """Kernel of mm_actor_sample (actor_sample without obs_copy / live_out), process-wide: 'tcgen05' (default: fp16
    operands, a warpgroup per 128-row tile, weights once per SM) or 'mma' (the warp-level mma.sync TF32 kernel, kept as
    an independent cross-check).  The appending actor_sample calls and policy_sample always run the tcgen05 kernel.
    Any other name raises ValueError."""
    if name not in _ACTOR_IMPLS:
        raise ValueError("actor impl must be one of %s, got %r" % (", ".join(map(repr, _ACTOR_IMPLS)), name))
    _lib.check(_lib.lib().mm_set_actor_impl(_ACTOR_IMPLS[name]))


def _first_layer_key(policy):
    return tuple((p.data_ptr(), p._version) for p in (policy.fc11.weight, policy.fc11.bias, policy.fc12.weight,
                                                      policy.fc12.bias, policy.fc13.weight, policy.fc13.bias))


def _split_first_layer(policy):
    """The three first-layer blocks of the state_split network (Model_gi.py:137-176: fc11 over the presence columns,
    fc12 over x / y, fc13 over vx / vy) as ONE 30 -> 160 layer: weight [160][30], zero outside the blocks, bias [160].

    Kept on the module itself (so it dies with it: a later module that reuses its id and memory starts empty) until a
    parameter is replaced or changed in place by a torch op (optimizer steps, load_state_dict: torch bumps `_version`).
    Writes through `.data` and collective writes (dist.broadcast) do not bump `_version`; after such writes call
    `first_layer_changed(policy)`, as `BatchedMAPPORollout.sync_parameters` does.  A `DeviceRMSprop` given the module
    as `shared_network` writes the layer it keeps along with the parameters, so it stays valid across device steps."""
    ps = (policy.fc11.weight, policy.fc11.bias, policy.fc12.weight, policy.fc12.bias, policy.fc13.weight, policy.fc13.bias)
    key = _first_layer_key(policy)
    hit = policy.__dict__.get("_mm_first_layer")
    if hit is not None and hit[0] == key:
        return hit[1], hit[2]
    h4, h2 = policy.fc11.out_features, policy.fc12.out_features
    w = torch.zeros((h4 + 2 * h2, NS), dtype=torch.float32, device=ps[0].device)
    w[:h4, list(policy.COLS1)] = ps[0].detach().float()
    w[h4:h4 + h2, list(policy.COLS2)] = ps[2].detach().float()
    w[h4 + h2:, list(policy.COLS3)] = ps[4].detach().float()
    b = torch.cat([ps[1].detach().float(), ps[3].detach().float(), ps[5].detach().float()]).contiguous()
    policy.__dict__["_mm_first_layer"] = (key, w, b)
    return w, b


def first_layer_changed(policy):
    """Drop the dense first layer `_split_first_layer` keeps on a shared network: required after its parameters were
    written in a way torch does not count (through `.data`, by a collective); any module is accepted."""
    policy.__dict__.pop("_mm_first_layer", None)


def policy_sample(policy, obs, n_agents=None, seed=0, step=0, want_logp=False, action_mask=None, want_value=False,
                  out_actions=None, obs_copy=None, live_out=None):
    """Fused forward + exploration draw of the MAPPO_GI shared network (mm_actor_sample_mlp with h1 = 160): `policy` is
    an ActorCriticNetwork with state_split and hidden size 128; -> actions int8 [...] (+ log-probabilities [..., 5] with
    want_logp, + V(s) [...] from critic_linear with want_value).  Other arguments as for `actor_sample`."""
    assert policy.state_split and policy.fc2.out_features == 128 and policy.fc2.in_features == 160, \
        "the fused kernel covers the reference's shared network (hidden size 128, state_split)"
    rows = obs.numel() // NS
    obs = obs.contiguous()
    assert obs.is_cuda and obs.dtype == torch.float32
    w1, b1 = _split_first_layer(policy)
    w = [policy.fc2.weight, policy.fc2.bias, policy.actor_linear.weight, policy.actor_linear.bias,
         policy.critic_linear.weight, policy.critic_linear.bias]
    w = [t.detach().contiguous().float() for t in w]
    actions = torch.empty(obs.shape[:-1], dtype=torch.int8, device=obs.device) if out_actions is None else out_actions
    assert actions.dtype == torch.int8 and actions.is_contiguous() and actions.numel() == rows
    _check_record_slots(rows, obs_copy, live_out)
    logp = torch.empty(obs.shape[:-1] + (NA,), dtype=torch.float32, device=obs.device) if want_logp else None
    values = torch.empty(obs.shape[:-1], dtype=torch.float32, device=obs.device) if want_value else None
    if n_agents is not None:
        assert n_agents.dtype == torch.int32 and n_agents.is_cuda and n_agents.numel() * MAXV == rows
    if action_mask is not None:
        assert action_mask.dtype == torch.uint8 and action_mask.is_cuda and action_mask.numel() == rows
        action_mask = action_mask.contiguous()
    _lib.check(_lib.lib().mm_actor_sample_mlp(_ptr(obs), _ptr(n_agents), C.c_int64(rows), 160, _ptr(w1), _ptr(b1), _ptr(w[0]),
                                              _ptr(w[1]), _ptr(w[2]), _ptr(w[3]), _ptr(w[4]), _ptr(w[5]), C.c_uint64(seed),
                                              C.c_uint64(step), _ptr(action_mask), _ptr(actions), _ptr(logp), _ptr(None),
                                              _ptr(values), _ptr(obs_copy), _ptr(live_out), _stream()))
    out = (actions,) + ((logp,) if want_logp else ()) + ((values,) if want_value else ())
    return out if len(out) > 1 else actions


def actor_sample(actor, obs, n_agents=None, seed=0, step=0, want_logp=False, action_mask=None, out_actions=None,
                 obs_copy=None, live_out=None):
    """Fused actor forward + exploration draw (mm_actor_sample): obs [..., 30] f32 cuda -> actions int8 [...].

    `actor` is an ActorNetwork (or any module with fc1/fc2/fc3 Linear layers 30-128-128-5); its parameters are read
    in place.  n_agents [E] int32 marks the live rows when obs is the env's [E, 12, 30] buffer.  With want_logp the
    log-probabilities of all five actions are returned too ([..., 5] f32).  action_mask: uint8 bit masks, one per row
    (`env.buffers()["action_mask"]`, bit k = action k available) for the MAPPO_GI actor's invalid-action masking.
    Rollout-buffer appends fused into the same launch (MAPPO.interact, mappo.py:117-131): out_actions (int8, slot t of
    the action buffer) receives the actions, obs_copy (f32, slot t of the state buffer) the rows they were drawn from,
    live_out (uint8) 1 where the row's agent exists."""
    rows = obs.numel() // NS
    obs = obs.contiguous()
    assert obs.is_cuda and obs.dtype == torch.float32
    w = [actor.fc1.weight, actor.fc1.bias, actor.fc2.weight, actor.fc2.bias, actor.fc3.weight, actor.fc3.bias]
    assert tuple(w[0].shape) == (128, NS) and tuple(w[2].shape) == (128, 128) and tuple(w[4].shape) == (NA, 128)
    w = [t.detach().contiguous().float() for t in w]
    actions = torch.empty(obs.shape[:-1], dtype=torch.int8, device=obs.device) if out_actions is None else out_actions
    assert actions.dtype == torch.int8 and actions.is_contiguous() and actions.numel() == rows
    logp = torch.empty(obs.shape[:-1] + (NA,), dtype=torch.float32, device=obs.device) if want_logp else None
    if n_agents is not None:
        assert n_agents.dtype == torch.int32 and n_agents.is_cuda and n_agents.numel() * MAXV == rows
    if action_mask is not None:
        assert action_mask.dtype == torch.uint8 and action_mask.is_cuda and action_mask.numel() == rows
        action_mask = action_mask.contiguous()
    if obs_copy is None and live_out is None:
        _lib.check(_lib.lib().mm_actor_sample(_ptr(obs), _ptr(n_agents), C.c_int64(rows), *[_ptr(t) for t in w],
                                              C.c_uint64(seed), C.c_uint64(step), _ptr(action_mask), _ptr(actions), _ptr(logp),
                                              _ptr(None), _stream()))
    else:
        _check_record_slots(rows, obs_copy, live_out)
        _lib.check(_lib.lib().mm_actor_sample_mlp(_ptr(obs), _ptr(n_agents), C.c_int64(rows), 128, *[_ptr(t) for t in w],
                                                  _ptr(None), _ptr(None), C.c_uint64(seed), C.c_uint64(step), _ptr(action_mask),
                                                  _ptr(actions), _ptr(logp), _ptr(None), _ptr(None), _ptr(obs_copy), _ptr(live_out),
                                                  _stream()))
    return (actions, logp) if want_logp else actions


# ---- on-device PPO learner (mm_ppo_targets / mm_ppo_grads): the update of `mappo_losses` / `shared_network_loss`
# (pairwise=False, critic_loss="mse") without autograd

def _ppo_kind(net):
    """-> (kind, parameters in mm_ppo_net order); asserts the reference's hidden sizes, which the kernels are built for."""
    if isinstance(net, ActorCriticNetwork):
        assert net.state_split and net.fc2.in_features == 160 and net.fc2.out_features == 128, \
            "the learner kernels cover the reference's shared network (hidden size 128, state_split)"
        w1, b1 = _split_first_layer(net)
        return _lib.PPO_SHARED, [w1, b1, net.fc2.weight, net.fc2.bias, net.actor_linear.weight, net.actor_linear.bias,
                                 net.critic_linear.weight, net.critic_linear.bias]
    shapes = [tuple(net.fc1.weight.shape), tuple(net.fc2.weight.shape), tuple(net.fc3.weight.shape)]
    if shapes == [(128, NS), (128, 128), (NA, 128)]:
        kind = _lib.PPO_ACTOR
    elif shapes == [(128, NS), (128, 128 + NA), (1, 128)]:
        kind = _lib.PPO_CRITIC
    else:
        raise AssertionError("the learner kernels cover the reference's ActorNetwork / CriticNetwork (hidden size 128)")
    return kind, [net.fc1.weight, net.fc1.bias, net.fc2.weight, net.fc2.bias, net.fc3.weight, net.fc3.bias]


def _ppo_net(params):
    for p in params:
        assert p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()
    ptrs = [p.data_ptr() for p in params] + [0] * (8 - len(params))
    return _lib.MMPpoNet(*ptrs)


def _check_rows(S, A8, idx, G=None):
    rows = S.shape[0]
    assert S.is_cuda and S.dtype == torch.float32 and S.is_contiguous() and S.dim() == 2 and S.shape[1] == NS
    assert A8.dtype == torch.int8 and A8.is_contiguous() and A8.numel() == rows
    assert idx.dtype == torch.int64 and idx.is_contiguous() and idx.dim() == 1 and idx.is_cuda
    if G is not None:
        assert G.dtype == torch.float32 and G.is_contiguous() and G.numel() == rows
    return rows


@torch.no_grad()
def ppo_targets(net, S, A8, idx, out=None, value_out=None):
    """Target pass of one update (mm_ppo_targets): for the rows listed in idx, the target log-probability of the taken
    action (`net` an ActorNetwork or the shared ActorCriticNetwork) or Q_target(s, one_hot(a)) (`net` a CriticNetwork).
    S [rows, 30] f32, A8 [rows] int8 (the rollout buffer as collected), idx int64 [n]; -> out [rows] f32, indexed like
    S (rows not listed are left as they are).  value_out [rows] f32 (shared network only): also V(s) from the same
    forward, indexed the same way."""
    rows = _check_rows(S, A8, idx)
    kind, params = _ppo_kind(net)
    out = torch.empty(rows, dtype=torch.float32, device=S.device) if out is None else out
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == rows
    if value_out is not None:
        assert kind == _lib.PPO_SHARED, "value_out is the shared network's V(s)"
        assert value_out.dtype == torch.float32 and value_out.is_contiguous() and value_out.numel() == rows
    if idx.numel() == 0:
        return out
    crit = kind == _lib.PPO_CRITIC
    _lib.check(_lib.lib().mm_ppo_targets(kind, _ptr(S), _ptr(A8), _ptr(idx), C.c_int64(idx.numel()), C.byref(_ppo_net(params)),
                                         _ptr(None if crit else out), _ptr(out if crit else value_out), _stream()))
    return out


def _grad_buffer(p):
    """p.grad, created if absent; the kernels overwrite it (as backward() after zero_grad(set_to_none=True) would)."""
    if p.grad is None:
        p.grad = torch.empty_like(p)
    return p.grad


def _ppo_grads(kind, params, grads, S, A8, G, old_logp, q_target, idx, clip, losses):
    if idx.numel() == 0:       # an empty shard of a data-parallel update: it contributes nothing to the all-reduce
        for g in grads:
            g.zero_()
        return
    out = _lib.MMPpoGrads(*([g.data_ptr() for g in grads] + [0] * (8 - len(grads))))
    _lib.check(_lib.lib().mm_ppo_grads(kind, _ptr(S), _ptr(A8), _ptr(G), _ptr(old_logp), _ptr(q_target), _ptr(idx),
                                       C.c_int64(idx.numel()), C.c_float(clip), C.byref(_ppo_net(params)), C.byref(out),
                                       _ptr(losses), _stream()))


def mappo_gradients(actor, critic, S, A8, G, old_logp, q_target, idx, clip=0.2, losses=None):
    """Gradient pass of one MAPPO minibatch (mm_ppo_grads, actor and critic): writes every parameter's .grad as
    `actor_loss.backward(); critic_loss.backward()` of `mappo_losses` (pairwise=False, critic_loss="mse") would after
    zero_grad(set_to_none=True), with old_logp / q_target from `ppo_targets` of actor_target / critic_target.  S [rows, 30],
    A8 [rows] int8, G [rows] f32 (the returns), idx int64 [n] the minibatch's rows in any order.  losses (optional) f32 [2]
    device buffer.  -> (actor_loss, critic_loss) device scalars, no host synchronisation."""
    _check_rows(S, A8, idx, G)
    ka, pa = _ppo_kind(actor)
    kc, pc = _ppo_kind(critic)
    assert ka == _lib.PPO_ACTOR and kc == _lib.PPO_CRITIC
    losses = torch.zeros(2, dtype=torch.float32, device=S.device) if losses is None else losses
    assert old_logp.numel() == S.shape[0] and q_target.numel() == S.shape[0]
    _ppo_grads(ka, pa, [_grad_buffer(p) for p in pa], S, A8, G, old_logp, q_target, idx, clip, losses)
    _ppo_grads(kc, pc, [_grad_buffer(p) for p in pc], S, A8, G, None, None, idx, clip, losses)
    return losses[0], losses[1]


def shared_network_gradients(policy, S, A8, G, old_logp, idx, clip=0.2, losses=None):
    """Gradient pass of one MAPPO_GI minibatch (mm_ppo_grads, shared network): writes every parameter's .grad as
    `loss.backward()` of `shared_network_loss` (pairwise=False, critic_loss="mse") would after zero_grad(set_to_none=True).
    The kernel differentiates the dense 30 -> 160 first layer; fc11 / fc12 / fc13 receive their own blocks of it.
    -> (loss, actor_loss, critic_loss) device scalars, no host synchronisation."""
    _check_rows(S, A8, idx, G)
    kind, params = _ppo_kind(policy)
    assert old_logp.numel() == S.shape[0]
    losses = torch.zeros(2, dtype=torch.float32, device=S.device) if losses is None else losses
    dev = S.device
    hit = policy.__dict__.get("_mm_fold")       # scratch for the dense first layer's gradient, kept on the module
    if hit is None or hit[0].device != dev:
        dense = (torch.empty((160, NS), device=dev), torch.empty(160, device=dev))
        cols = [torch.tensor(c, device=dev) for c in (policy.COLS1, policy.COLS2, policy.COLS3)]
        hit = policy.__dict__["_mm_fold"] = dense + (cols,)
    gw1, gb1, cols = hit
    grads = [gw1, gb1] + [_grad_buffer(p) for p in params[2:]]
    _ppo_grads(kind, params, grads, S, A8, G, old_logp, None, idx, clip, losses)
    o = 0
    for lin, c in zip((policy.fc11, policy.fc12, policy.fc13), cols):
        k = lin.out_features
        torch.index_select(gw1[o:o + k], 1, c, out=_grad_buffer(lin.weight))
        _grad_buffer(lin.bias).copy_(gb1[o:o + k])
        o += k
    return losses[0] + losses[1], losses[0], losses[1]


# ---- PPO diagnostics of one network over listed rows (mm_ppo_stats), and their torch reference

@torch.no_grad()
def ppo_stats(net, S, A8, G, idx, old_logp=None, clip=0.2):
    """Statistics pass of the learner (mm_ppo_stats) over the rows S[idx]: -> f64 device tensor [PPO_STATS_LEN] with the
    fields of `_lib.PPO_STAT_FIELDS` (row count; entropy of the policy; with old_logp [rows] the sums of k3 =
    (r - 1) - log r and of |r - 1| > clip and the range of r = exp(logp(a) - old_logp); sums of v, v^2, G, G^2 and
    (G - v)^2 for the value Q(s, a) of a CriticNetwork or V(s) of the shared network).  `net` as for `ppo_targets`; G [rows]
    the returns (may be None for an ActorNetwork).  Enqueued on the current stream, no synchronisation."""
    _check_rows(S, A8, idx, G)
    kind, params = _ppo_kind(net)
    if old_logp is not None:
        assert old_logp.dtype == torch.float32 and old_logp.is_contiguous() and old_logp.numel() == S.shape[0]
    out = torch.empty(_lib.PPO_STATS_LEN, dtype=torch.float64, device=S.device)
    _lib.check(_lib.lib().mm_ppo_stats(kind, _ptr(S), _ptr(A8), _ptr(G), _ptr(old_logp), _ptr(idx), C.c_int64(idx.numel()),
                                       C.c_float(clip), C.byref(_ppo_net(params)), _ptr(out), _stream()))
    return out


@torch.no_grad()
def _ppo_stats_torch(net, S, A8, G, idx, old_logp, clip):
    """-> (statistics vector, log p(a) per row of idx or None); rows in the module's dtype, sums in float64"""
    dt = next(net.parameters()).dtype
    s = S[idx].to(dt)
    onehot = torch.nn.functional.one_hot(A8[idx].long(), NA).to(dt)
    lp_all = v = logp = None
    if isinstance(net, ActorCriticNetwork):
        hidden = net.trunk(s)
        lp_all, v = net.policy_head(hidden), net.critic_linear(hidden)[:, 0]
    elif isinstance(net, CriticNetwork):
        v = net(s, onehot)[:, 0]
    else:
        lp_all = net(s)
    K = _lib.PPO_STAT
    out = torch.zeros(_lib.PPO_STATS_LEN, dtype=torch.float64, device=S.device)
    out[K["n"]] = idx.numel()
    out[K["ratio_min"]], out[K["ratio_max"]] = float("inf"), -float("inf")
    if lp_all is not None:
        logp = (lp_all * onehot).sum(1)            # as mappo_losses / shared_network_loss form it
        out[K["entropy"]] = (-(lp_all.exp() * lp_all).sum(1)).double().sum()
        if old_logp is not None and idx.numel():
            lr = logp - old_logp[idx].to(dt)
            r = torch.exp(lr)
            out[K["k3"]] = ((r - 1) - lr).double().sum()
            out[K["clipped"]] = ((r - 1).abs() > clip).double().sum()
            out[K["ratio_min"]], out[K["ratio_max"]] = r.min().double(), r.max().double()
    if v is not None:
        g = G[idx].to(dt)
        vd, gd, res = v.double(), g.double(), (g - v).double()
        out[K["v"]], out[K["v2"]] = vd.sum(), (vd * vd).sum()
        out[K["g"]], out[K["g2"]] = gd.sum(), (gd * gd).sum()
        out[K["res2"]] = (res * res).sum()
    return out, logp


def ppo_stats_torch(net, S, A8, G, idx, old_logp=None, clip=0.2):
    """`ppo_stats` from the torch modules: the per-row values in the module's dtype (float32: the numerics of the torch
    update path), the sums in float64.  Any device, any float dtype of `net`."""
    return _ppo_stats_torch(net, S, A8, G, idx, old_logp, clip)[0]


def ppo_stats_keys(before, after):
    """The diagnostics of one update from the statistics vectors (host sequences, all-reduced over ranks) of the pass over
    every live row with the rollout networks (`before`, no ratio) and with the updated ones against the rollout policy's
    log-probabilities (`after`).  Explained variance 1 - Var(G - v) / Var(G), advantage G - v of the rollout critic;
    variances and the advantage's std are population moments."""
    K = _lib.PPO_STAT
    n = before[K["n"]]
    if n <= 0:
        nan = float("nan")
        return dict.fromkeys(("approx_kl", "clip_fraction", "ratio_min", "ratio_max", "entropy_before", "entropy_after",
                              "explained_variance_before", "explained_variance_after", "advantage_mean", "advantage_std"), nan)

    def fit(v):
        mean_res = (v[K["g"]] - v[K["v"]]) / n
        var_res = v[K["res2"]] / n - mean_res * mean_res
        var_g = v[K["g2"]] / n - (v[K["g"]] / n) ** 2
        return mean_res, var_res, (1.0 - var_res / var_g) if var_g > 0 else float("nan")

    adv_mean, adv_var, ev_before = fit(before)
    return {"approx_kl": after[K["k3"]] / n, "clip_fraction": after[K["clipped"]] / n,
            "ratio_min": after[K["ratio_min"]], "ratio_max": after[K["ratio_max"]],
            "entropy_before": before[K["entropy"]] / n, "entropy_after": after[K["entropy"]] / n,
            "explained_variance_before": ev_before, "explained_variance_after": fit(after)[2],
            "advantage_mean": adv_mean, "advantage_std": max(adv_var, 0.0) ** 0.5}


# ---- the optimiser step on the device (mm_rmsprop_step): clip_grad_norm_ + RMSprop, one launch for whole networks

_MIRROR_COLS = {}


def _mirror_cols(cols):
    """host int32 column map of a mirror entry (kept alive here: the table points at it)"""
    if cols not in _MIRROR_COLS:
        _MIRROR_COLS[cols] = (C.c_int32 * len(cols))(*cols)
    return _MIRROR_COLS[cols]


class DeviceRMSprop(torch.optim.Optimizer):
    """`torch.nn.utils.clip_grad_norm_(params, max_grad_norm)` followed by `torch.optim.RMSprop(params, lr, alpha, eps)`
    (no momentum, not centred, no weight decay: the reference's optimiser, mappo.py:88-90, mappo_gi.py:150-156) in one
    kernel launch (mm_rmsprop_step); `rmsprop_step` steps several of them in one launch.  max_grad_norm None or <= 0:
    no clipping.  The parameters (one group, at most 16 float32 CUDA tensors on one device) are one network.

    - State: torch.optim.RMSprop's (`step`, `square_avg` per parameter), so the state_dict of either class loads into
      the other.
    - Gradients: every `.grad` is a view of one flat buffer, `flat_grad`.  `zero_grad()` zeros it in place and keeps the
      views (`set_to_none` is ignored); autograd accumulates into them and the learner kernels overwrite them.  A `.grad`
      replaced from outside is copied back into its view at the next step.
    - Unlike torch, every parameter is stepped on every call: a parameter whose `.grad` is None counts as a zero gradient
      (its square_avg decays) where torch would skip it.  Every learner parameter receives a gradient on every minibatch.
    - After a step, `.grad` holds the clipped gradients (as clip_grad_norm_ leaves them) and `total_norm` [1] the norm
      before clipping (what clip_grad_norm_ returns), on the device.
    - shared_network: the ActorCriticNetwork these parameters belong to, if any.  The kernel writes its fc11 / fc12 /
      fc13 updates into the dense first layer `_split_first_layer` keeps for it as well: device writes do not bump
      torch's `_version`, so without that the kept layer would go stale."""

    def __init__(self, params, lr, alpha=0.99, eps=1e-8, max_grad_norm=None, momentum=0, centered=False, weight_decay=0,
                 shared_network=None):
        if momentum != 0 or centered or weight_decay != 0:
            raise ValueError("DeviceRMSprop is the reference's RMSprop: momentum, centered and weight_decay are not supported")
        if not lr >= 0.0 or not eps >= 0.0 or not 0.0 <= alpha <= 1.0:
            raise ValueError("invalid lr, alpha or eps: %r, %r, %r" % (lr, alpha, eps))
        super().__init__(params, dict(lr=lr, alpha=alpha, eps=eps, momentum=0, centered=False, weight_decay=0))
        ps = self.param_groups[0]["params"]
        if not 1 <= len(ps) <= _lib.OPT_MAX_TENSORS:
            raise ValueError("DeviceRMSprop steps 1..%d parameter tensors, got %d" % (_lib.OPT_MAX_TENSORS, len(ps)))
        for p in ps:
            if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous() and p.device == ps[0].device):
                raise ValueError("DeviceRMSprop needs contiguous float32 CUDA parameters on one device")
        self.max_grad_norm = 0.0 if max_grad_norm is None else float(max_grad_norm)
        self.shared_network = shared_network
        self.flat_grad = torch.zeros(sum(p.numel() for p in ps), device=ps[0].device)
        self.total_norm = torch.zeros(1, device=ps[0].device)
        self._views, o = [], 0
        for p in ps:
            v = self.flat_grad[o:o + p.numel()].view_as(p)
            if p.grad is not None:
                v.copy_(p.grad)
            p.grad = v
            self._views.append(v)
            o += p.numel()

    def add_param_group(self, param_group):
        if self.param_groups:
            raise ValueError("DeviceRMSprop holds one parameter group (one network, clipped as a whole)")
        super().add_param_group(param_group)

    def zero_grad(self, set_to_none=True):
        """Zero the flat gradient buffer in place; the `.grad` views stay (set_to_none is ignored)."""
        self.flat_grad.zero_()
        for p, v in zip(self.param_groups[0]["params"], self._views):
            p.grad = v

    @torch.no_grad()
    def step(self, closure=None, grad_divisor=1):
        """One clip + RMSprop step; grad_divisor: divide the gradients first (the world size after an all-reduce sum of
        `flat_grad`), rounded as torch's `grad /= grad_divisor` on a CUDA tensor."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        rmsprop_step([self], grad_divisor)
        return loss

    def _mirrors(self):
        """{param index: (dest pointer, column map, row stride)} of the dense first layer kept for shared_network, when it
        is current (a stale one is rebuilt from the parameters at its next use)"""
        net = self.shared_network
        hit = None if net is None else net.__dict__.get("_mm_first_layer")
        if hit is None or hit[0] != _first_layer_key(net):
            return {}
        w, b = hit[1], hit[2]
        index = {id(p): k for k, p in enumerate(self.param_groups[0]["params"])}
        out, row = {}, 0
        for lin, cols in ((net.fc11, net.COLS1), (net.fc12, net.COLS2), (net.fc13, net.COLS3)):
            if id(lin.weight) in index:
                out[index[id(lin.weight)]] = (w.data_ptr() + 4 * row * NS, cols, NS)
            if id(lin.bias) in index:
                out[index[id(lin.bias)]] = (b.data_ptr() + 4 * row, (0,), 1)
            row += lin.out_features
        return out

    def _table(self, grad_scale):
        g = self.param_groups[0]
        if g.get("momentum", 0) != 0 or g.get("centered", False) or g.get("weight_decay", 0) != 0:
            raise ValueError("DeviceRMSprop is the reference's RMSprop: momentum, centered and weight_decay are not supported")
        ps = g["params"]
        mirrors = self._mirrors()
        tensors = (_lib.MMOptTensor * len(ps))()
        steps = []
        for k, (p, v) in enumerate(zip(ps, self._views)):
            if p.grad is not v:
                v.copy_(p.grad) if p.grad is not None else v.zero_()
                p.grad = v
            st = self.state[p]
            if "square_avg" not in st:
                st["step"] = torch.tensor(0.0)
                st["square_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            sq = st["square_avg"]
            assert sq.is_contiguous() and sq.device == p.device and sq.dtype == torch.float32
            steps.append(st["step"])
            t = tensors[k]
            t.param, t.grad, t.square_avg, t.numel = p.data_ptr(), v.data_ptr(), sq.data_ptr(), p.numel()
            if k in mirrors:
                dst, cols, ld = mirrors[k]
                t.mirror, t.mirror_cols, t.mirror_ncols, t.mirror_ld = dst, _mirror_cols(cols), len(cols), ld
        torch._foreach_add_(steps, 1)
        # alpha, 1 - alpha (in double, as torch forms it), eps, lr: rounded to float32 as torch rounds these scalars
        grp = _lib.MMOptGroup(tensors, len(ps), g["lr"], g["alpha"], 1.0 - g["alpha"], g["eps"], self.max_grad_norm,
                              grad_scale, self.total_norm.data_ptr())
        return grp, tensors


def rmsprop_step(optimizers, grad_divisor=1):
    """Step several DeviceRMSprop (one network each, on one device) in ONE launch of mm_rmsprop_step on the current
    stream.  grad_divisor > 1: the gradients are first multiplied by float32(1 / grad_divisor), which is what torch's
    `grad /= grad_divisor` computes on a CUDA tensor (a division by a CPU scalar runs as a product with its reciprocal)."""
    if not 1 <= len(optimizers) <= _lib.OPT_MAX_GROUPS:
        raise ValueError("rmsprop_step steps 1..%d optimisers in one launch" % _lib.OPT_MAX_GROUPS)
    scale = float(np.float32(1.0) / np.float32(grad_divisor))
    tables = [o._table(scale) for o in optimizers]
    groups = (_lib.MMOptGroup * len(tables))(*[t[0] for t in tables])
    _lib.check(_lib.lib().mm_rmsprop_step(groups, len(tables), _stream()))


def _check_record_slots(rows, obs_copy, live_out):
    if obs_copy is not None:
        assert obs_copy.is_cuda and obs_copy.dtype == torch.float32 and obs_copy.is_contiguous() and obs_copy.numel() == rows * NS
    if live_out is not None:
        assert live_out.is_cuda and live_out.dtype == torch.uint8 and live_out.is_contiguous() and live_out.numel() == rows


class BatchedMAPPORollout(object):
    """`MAPPO` (marl/mappo.py) on every env of a `MergeEnvBatched`: an actor and a critic network (Model_common.py), their
    target networks and one RMSprop optimiser each.  `collect`, `update` and the acting methods are written once for both
    learners; what MAPPO_GI does differently is in the small methods `BatchedMAPPOGIRollout` overrides (`_sampler`,
    `_learners`, `_kernel_targets`, `_kernel_gradients`, `_autograd_gradients` and the value / statistics networks)."""

    def __init__(self, env, actor=None, critic=None, actor_lr=5e-4, critic_lr=5e-4, **kw):
        """actor, critic: the networks to train (default: new ones); actor_lr, critic_lr: their RMSprop learning rates
        (mappo.py:88-90).  Every other argument is the rollout's, see `_setup`."""
        self._setup(env, **kw)
        self.actor = (actor or ActorNetwork()).to(self.dev)
        self.critic = (critic or CriticNetwork()).to(self.dev)
        self.actor_target = ActorNetwork().to(self.dev)
        self.critic_target = CriticNetwork().to(self.dev)
        self.actor_target.load_state_dict(self.actor.state_dict())
        self.critic_target.load_state_dict(self.critic.state_dict())
        self.actor_opt = self._make_optimizer(self.actor, actor_lr)
        self.critic_opt = self._make_optimizer(self.critic, critic_lr)

    def _setup(self, env, roll_out_n_steps=100, reward_gamma=0.99, reward_scale=20.0, reward_type="regionalR",
               clip_param=0.2, max_grad_norm=5.0, seed=0, fused=True, obs=None, reset_seed=None, optimizer="torch",
               gae_lambda=None):
        """What both learners share; the arguments are checked before anything touches the env or the GPU.

        obs: the observation of an env the caller has already reset (train.py resets with a rank-distinct spawn
        seed and hands its first observation over).  Without it the first collect() spawns the scenes itself with
        `reset_seed` (default: derived from `seed`, which the data-parallel driver makes rank-distinct) - never with the
        env's config seed, which is the same on every rank and would make the shards replicas of one another.
        optimizer: "torch" (torch.optim.RMSprop after clip_grad_norm_, the default) or "cuda" (`DeviceRMSprop`: the same
        step as one launch per minibatch, with either update impl).
        gae_lambda: None (the default: the Monte-Carlo returns of the reference) or a number in [0, 1]: update() trains on
        the lambda-returns (`lambda_returns`, stored as buf["lambda_returns"]) with the values of the networks that
        collected the rollout, the target networks at the start of the update.  1 gives the same returns bit for bit."""
        if optimizer not in ("torch", "cuda"):
            raise ValueError("optimizer must be 'torch' or 'cuda', got %r" % (optimizer,))
        self.gae_lambda = check_gae_lambda(gae_lambda)
        self.env = env
        self.dev = torch.device("cuda", env.device)
        self.T = int(roll_out_n_steps)
        self.gamma, self.reward_scale, self.reward_type = float(reward_gamma), float(reward_scale), reward_type
        self.clip_param, self.max_grad_norm = clip_param, max_grad_norm
        self.optimizer = optimizer
        self.obs = obs
        self.reset_seed = (0x5EED0000 + int(seed)) if reset_seed is None else int(reset_seed)
        self._slot = torch.arange(MAXV, device=self.dev)[None, :]
        self.buf = None
        self.E = env.n_envs
        self.seed, self._draws = int(seed), 0
        self.fused = bool(fused)

    def _sampler(self):
        """(the network that draws the actions, its fused draw: `actor_sample` or `policy_sample`)"""
        return self.actor, actor_sample

    @torch.no_grad()
    def act_fused(self, obs, n_agents):
        """The draw of `act_torch` through the fused CUDA kernel (TF32 actor + inverse-CDF sampling, one launch)."""
        net, sample = self._sampler()
        self._draws += 1
        a = sample(net, obs, n_agents, seed=self.seed, step=self._draws)
        return a, self._slot < n_agents[:, None]

    @torch.no_grad()
    def _record_act(self, obs, n_agents, a_slot, s_slot, l_slot):
        net, sample = self._sampler()
        self._draws += 1
        return sample(net, obs, n_agents, seed=self.seed, step=self._draws, out_actions=a_slot, obs_copy=s_slot,
                      live_out=l_slot)

    @torch.no_grad()
    def act_torch(self, obs, n_agents):
        """Plain torch fp32 policy + torch.multinomial (exploration_action, mappo.py:225-230, mappo_gi.py:368-373): the
        numerics reference of `act_fused`."""
        logp = self._sampler()[0](obs.reshape(-1, NS))                          # [E*12, 5]
        a = torch.multinomial(logp.exp(), 1).view(obs.shape[0], MAXV)
        live = self._slot < n_agents[:, None]
        return torch.where(live, a, torch.ones_like(a)).to(torch.int8), live

    def _act(self, obs, n_agents):
        return self.act_fused(obs, n_agents) if self.fused else self.act_torch(obs, n_agents)

    @torch.no_grad()
    def collect(self):
        """One rollout of T policy steps for every env; returns the batch dict (device tensors)."""
        env, E, T = self.env, self.E, self.T
        v = env.buffers()
        if self.obs is None:
            self.obs, _ = env.reset(seed=self.reset_seed)
        S = torch.empty((T, E, MAXV, NS), device=self.dev)
        A8 = torch.empty((T, E, MAXV), dtype=torch.int8, device=self.dev)
        L8 = torch.empty((T, E, MAXV), dtype=torch.uint8, device=self.dev)
        R = torch.empty((T, E, MAXV), device=self.dev)
        D = torch.empty((T, E), device=self.dev)
        for t in range(T):
            if self.fused:
                # the draw kernel appends to the rollout buffer itself: state S[t], action A8[t], live mask L8[t]
                a = self._record_act(self.obs, v["n_agents"], A8[t], S[t], L8[t])
            else:
                n_agents = v["n_agents"].clone()
                S[t].copy_(self.obs)
                a, live = self._act(self.obs, n_agents)
                A8[t].copy_(a)
                L8[t].copy_(live)
            self.obs, reward, done, info = env.step(a, auto_reset=True)
            if self.reward_type == "regionalR":
                R[t].copy_(info["regional_rewards"])
            else:
                R[t].copy_(reward[:, None].expand(E, MAXV))
            D[t].copy_(done)
        A, L = A8.long(), L8.bool()
        if self.reward_scale > 0:
            R /= self.reward_scale
        # bootstrap where the last step did not end the episode (mappo.py:148-150)
        final_value = self._final_value(self.obs, v["n_agents"])
        returns = discounted_returns(R, D, final_value, self.gamma)
        self.buf = dict(states=S, actions=A, returns=returns, live=L, dones=D, rewards=R, final_value=final_value)
        return self.buf

    def _final_value(self, obs, n_agents):
        a_fin, _ = self._act(obs, n_agents)
        onehot = torch.nn.functional.one_hot(a_fin.long(), NA).float()
        return self.critic(obs.reshape(-1, NS), onehot.view(-1, NA)).view(self.E, MAXV)

    def networks(self):
        """every module a replica must hold identically (sync_parameters, the replica check of train.py)"""
        return [self.actor, self.critic, self.actor_target, self.critic_target]

    def sample_actions(self, obs, n_agents, seed, step):
        """MAPPO.action (mappo.py:231-236): a draw from the softmax, also at evaluation time."""
        return actor_sample(self.actor, obs.contiguous(), n_agents, seed=seed, step=step)

    # ---- data parallelism over env shards (SURVEY.md 8e): one process per GPU, each with its own envs; the only
    # traffic is the gradient all-reduce of the two small networks (~42 k parameters each) per minibatch
    def _world(self):
        import torch.distributed as dist
        return dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1

    def sync_parameters(self, src=0):
        """Broadcast rank `src`'s networks (call once after construction under torchrun).  The broadcast writes the
        parameters behind torch's back, so the dense first layer kept on a shared network is dropped afterwards; call
        this also after writing the networks' parameters through `.data` yourself."""
        import torch.distributed as dist
        if self._world() > 1:
            for m in self.networks():
                for t in list(m.parameters()) + list(m.buffers()):
                    dist.broadcast(t.data, src)
        for m in self.networks():
            first_layer_changed(m)

    def _make_optimizer(self, net, lr, shared_network=None):
        if self.optimizer == "cuda":
            return DeviceRMSprop(net.parameters(), lr=lr, max_grad_norm=self.max_grad_norm, shared_network=shared_network)
        return torch.optim.RMSprop(net.parameters(), lr=lr)

    def _optimizer_step(self, opts, nets):
        """all-reduce (data parallel), clip_grad_norm_ and the RMSprop step of each optimiser in `opts` (nets: their
        networks): torch ops per network, or with optimizer="cuda" one in-place all-reduce of each flat gradient buffer
        and ONE mm_rmsprop_step launch for all of them (the division by the world size happens in the kernel)."""
        if self.optimizer == "cuda":
            w = self._world()
            if w > 1:
                import torch.distributed as dist
                for o in opts:
                    dist.all_reduce(o.flat_grad)
            rmsprop_step(opts, w)
            return
        for o, net in zip(opts, nets):
            params = list(net.parameters())
            self._allreduce_grads(params)
            nn.utils.clip_grad_norm_(params, self.max_grad_norm)
            o.step()

    def _allreduce_grads(self, params):
        import torch.distributed as dist
        w = self._world()
        if w == 1:
            return
        params = [q for q in params if q.grad is not None]
        flat = torch.cat([q.grad.reshape(-1) for q in params])
        dist.all_reduce(flat)
        flat /= w
        o = 0
        for q in params:
            q.grad.copy_(flat[o:o + q.numel()].view_as(q.grad))
            o += q.numel()

    def update(self, minibatch=1 << 18, epochs=1, impl="torch", stats=False):
        """One PPO update on the last rollout, all agents at once, with the per-sample surrogate (the reference's [N] x
        [N, 1] product is an N x N table): MAPPO's PPO-clip actor update and critic regression (mappo.py:161-206,
        `mappo_losses`), or MAPPO_GI's summed loss of the shared network (mappo_gi.py:307-349, `shared_network_loss`).
        `epochs` passes over the live rows in random minibatches (one torch.randperm per epoch, the only random draw of an
        update), an optimiser step after each; then the target networks take the updated parameters.  Under
        torch.distributed every rank runs the same number of minibatches and the gradients are averaged.
        impl: "torch" (autograd) or "cuda" (the learner kernels: one target pass over every live row - the target networks
        do not change within an update - then one gradient pass per minibatch).
        -> {"actor_loss", "critic_loss": the last minibatch's (0 with epochs=0), "samples"}; the losses stay on the device
        until one host read at the end.
        stats: also measure what the update did (the keys of `ppo_stats_keys`): a statistics pass over every live row with
        the rollout (target) networks before the first minibatch and one with the updated networks after the last, with
        `ppo_stats_torch` (impl "torch") or `ppo_stats` (impl "cuda"), all-reduced over ranks and read in one host read.
        The passes draw no random numbers and write no parameter: the update is the same with and without them.
        With gae_lambda set, the returns G of everything above (advantage, critic target, statistics) are the
        lambda-returns, from the rollout's values of every live row (MAPPO: Q_target(s, a), MAPPO_GI: V_target(s); one
        no-grad target forward with impl "torch", the target pass with impl "cuda") before the first minibatch."""
        assert impl in ("torch", "cuda"), impl
        gae = self.gae_lambda is not None
        batch = idx, S, A8, G = self._learner_batch(with_returns=not gae)
        n_mb = self._minibatch_count(idx, minibatch)
        targets = old_logp = None
        if impl == "cuda":
            targets, values = self._kernel_targets(batch, gae)
            old_logp = targets[0]
        elif gae:
            values = self._rollout_values_torch()
        if gae:
            batch = idx, S, A8, G = idx, S, A8, self._set_lambda_returns(values)
        before = self._stats_begin(impl, batch, old_logp) if stats else None
        nets, _, opts = zip(*self._learners())
        losses = torch.zeros(2, device=self.dev)       # written by the learner kernels
        last = losses.unbind()                        # (actor_loss, critic_loss) of the last minibatch; 0 with epochs=0
        codes = torch.arange(NA, dtype=torch.int8, device=self.dev)
        for _ in range(epochs):
            perm = idx[torch.randperm(idx.numel(), device=self.dev)]
            for j in torch.tensor_split(perm, n_mb):
                if impl == "cuda":
                    last = self._kernel_gradients(batch, j, targets, losses)
                else:       # one-hot actions as (a == k): 0 / 1 exactly, in fewer launches than one_hot(...).float()
                    last = self._autograd_gradients(S[j], (A8[j, None] == codes).float(), G[j, None])
                self._optimizer_step(opts, nets)
        a_loss, c_loss = torch.stack(last).tolist()
        rec = {"actor_loss": a_loss, "critic_loss": c_loss, "samples": int(idx.numel())}
        if stats:
            rec.update(self._stats_end(impl, batch, *before))
        for net, target, _ in self._learners():
            target.load_state_dict(net.state_dict())     # TARGET_TAU = 1.0 in every shipped ini
        return rec

    def _learners(self):
        """(network, its target network, its optimiser) of every network the update trains"""
        return [(self.actor, self.actor_target, self.actor_opt), (self.critic, self.critic_target, self.critic_opt)]

    def _kernel_targets(self, batch, gae):
        """Target pass of the CUDA update -> (the fixed arguments of `_kernel_gradients`, old_logp first; the rollout's
        values for the lambda-returns with gae, else None).  MAPPO: old_logp and q_target; with gae q_target is
        zero-filled first (the pass writes live rows only) and is also the values."""
        idx, S, A8, _ = batch
        old_logp = ppo_targets(self.actor_target, S, A8, idx)
        q_target = ppo_targets(self.critic_target, S, A8, idx, out=torch.zeros(S.shape[0], device=self.dev) if gae else None)
        return (old_logp, q_target), (q_target if gae else None)

    def _kernel_gradients(self, batch, j, targets, losses):
        """.grad of every trained parameter for the rows j by the learner kernels -> (actor_loss, critic_loss) device
        scalars, views of `losses`"""
        _, S, A8, G = batch
        return mappo_gradients(self.actor, self.critic, S, A8, G, *targets, j, self.clip_param, losses=losses)

    def _autograd_gradients(self, s, onehot, g):
        """.grad of every trained parameter for the rows s [n, 30], one-hot actions [n, 5], returns g [n, 1] by autograd
        -> (actor_loss, critic_loss) device scalars.  The two losses share no parameters, so the backward order does not
        matter."""
        actor_loss, critic_loss = mappo_losses(self.actor, self.actor_target, self.critic, self.critic_target, s, onehot, g,
                                               self.clip_param)
        self.actor_opt.zero_grad(set_to_none=True)
        self.critic_opt.zero_grad(set_to_none=True)
        actor_loss.backward()
        critic_loss.backward()
        return actor_loss.detach(), critic_loss.detach()

    def _learner_batch(self, with_returns=True):
        """(live row list, states [rows, 30], actions int8 [rows], returns [rows] or None) of the last rollout"""
        b = self.buf
        idx = b["live"].reshape(-1).nonzero(as_tuple=False).squeeze(1)
        S = b["states"].reshape(-1, NS)
        A8 = b["actions"].reshape(-1).to(torch.int8)
        G = self._returns().reshape(-1).contiguous() if with_returns else None
        return idx, S, A8, G

    def _returns(self):
        """the returns the update trains on: the lambda-returns with gae_lambda set, else the discounted returns"""
        return self.buf["returns"] if self.gae_lambda is None else self.buf["lambda_returns"]

    def _set_lambda_returns(self, values):
        """buf["lambda_returns"] from the rollout's values [rows] (zero on the rows of agents that do not exist);
        -> the lambda-returns as [rows]"""
        b = self.buf
        R = b["rewards"]
        b["lambda_returns"] = lambda_returns(R, b["dones"], values.view(R.shape), b["final_value"], self.gamma, self.gae_lambda)
        return b["lambda_returns"].view(-1)

    @torch.no_grad()
    def _rollout_values_torch(self):
        """the rollout's values of every live row from one no-grad forward of the target network(s), zero elsewhere:
        [rows] f32"""
        b = self.buf
        idx = b["live"].reshape(-1).nonzero(as_tuple=False).squeeze(1)
        v = torch.zeros(b["live"].numel(), device=self.dev)
        v[idx] = self._target_values(b["states"].reshape(-1, NS)[idx], b["actions"].reshape(-1)[idx])
        return v

    def _target_values(self, S, A):
        """Q_target(s, a) of the rows S [n, 30], A [n] (MAPPO's value of the rollout) -> [n]"""
        return self.critic_target(S, torch.nn.functional.one_hot(A, NA).float())[:, 0]

    def _minibatch_count(self, idx, minibatch):
        """minibatches per epoch, the same on every rank (those of the largest shard); one process needs no device copy"""
        n = idx.numel()
        if self._world() > 1:
            import torch.distributed as dist
            n_max = torch.tensor([n], device=self.dev)
            dist.all_reduce(n_max, op=dist.ReduceOp.MAX)
            n = int(n_max)
        return max(1, -(-n // int(minibatch)))

    def _stat_nets(self, target):
        """(policy network, value network) of the statistics passes: the rollout's (the targets) or the updated ones"""
        return (self.actor_target, self.critic_target) if target else (self.actor, self.critic)

    def _stats_pass(self, impl, target, batch, old_logp):
        """-> (statistics vector of the policy and value networks over every live row, the policy's log p(a) per row of
        idx from the torch pass or None)"""
        idx, S, A8, G = batch
        pol, val = self._stat_nets(target)
        if impl == "cuda":
            v, logp = ppo_stats(pol, S, A8, G, idx, old_logp, self.clip_param), None
        else:
            v, logp = _ppo_stats_torch(pol, S, A8, G, idx, old_logp, self.clip_param)
        if val is not pol:
            vf = _lib.PPO_STAT["v"]
            w = ppo_stats(val, S, A8, G, idx) if impl == "cuda" else _ppo_stats_torch(val, S, A8, G, idx, None, self.clip_param)[0]
            v[vf:] = w[vf:]
        return v, logp

    @torch.no_grad()
    def _stats_begin(self, impl, batch, old_logp=None):
        """statistics pass with the rollout networks; -> (its vector, the rollout policy's log p(a) indexed like the
        states: `old_logp` of the CUDA target pass, or from this pass)"""
        before, logp = self._stats_pass(impl, True, batch, None)
        if old_logp is None:
            idx, S = batch[0], batch[1]
            old_logp = torch.zeros(S.shape[0], dtype=logp.dtype, device=S.device)
            old_logp[idx] = logp
        return before, old_logp

    @torch.no_grad()
    def _stats_end(self, impl, batch, before, old_logp):
        """statistics pass with the updated networks against the rollout policy, all-reduce, one host read -> the keys"""
        after, _ = self._stats_pass(impl, False, batch, old_logp)
        b, a = mmd.all_reduce_ppo_stats(torch.stack([before, after])).tolist()
        return ppo_stats_keys(b, a)


class BatchedMAPPOGIRollout(BatchedMAPPORollout):
    """`MAPPO_GI` with `shared_network = True` (marl/mappo_gi.py; the 6 `*-shared*.ini` configs, run_mappo.py:232-277):
    ONE ActorCriticNetwork (Model_gi.py:137-220, state_split) gives the action distribution and the state value, one
    RMSprop optimiser at `actor_lr` (mappo_gi.py:150-156) steps the summed loss (`shared_network_loss`), the bootstrap
    value is V(final state) (mappo_gi.py:396-404).  Rollout, reward selection, scaling, returns and the update loop are
    the base class's; this class supplies the shared network to them.  It builds none of MAPPO's networks.
    As in the reference the policy is evaluated WITHOUT an action mask everywhere (`self.policy(state)`,
    mappo_gi.py:309,359): `action_masking` only changes what env.reset / step report.  With the reference's hidden size
    (128) the action draw and the bootstrap value come from the fused kernel (`policy_sample`: mm_actor_sample_mlp with
    the three first-layer blocks as one 30 -> 160 layer); other sizes run as torch layers."""

    def __init__(self, env, policy=None, hidden_size=128, actor_lr=5e-4, critic_lr=None, **kw):
        """policy: the shared network to train (default: a new one of `hidden_size`); actor_lr: its learning rate.
        critic_lr is accepted, as the ini files carry it, and unused: the reference's MAPPO_GI has no critic optimiser.
        Every other argument is the rollout's, see `BatchedMAPPORollout._setup`."""
        self._setup(env, **kw)
        net = policy or ActorCriticNetwork(NS, NA, hidden_size, 1, state_split=True)
        self.fused = self.fused and net.state_split and net.fc2.in_features == 160 and net.fc2.out_features == 128
        self.policy = net.to(self.dev)
        self.policy_target = ActorCriticNetwork(NS, NA, hidden_size, 1, state_split=self.policy.state_split).to(self.dev)
        self.policy_target.load_state_dict(self.policy.state_dict())
        self.policy_opt = self._make_optimizer(self.policy, actor_lr, shared_network=self.policy)

    def _sampler(self):
        return self.policy, policy_sample

    def _final_value(self, obs, n_agents):
        if self.fused:     # V(s) from the same kernel family: critic_linear as a sixth output column
            return policy_sample(self.policy, obs, n_agents, seed=self.seed, step=0, want_value=True)[1].view(self.E, MAXV)
        return self.policy(obs.reshape(-1, NS), out_type="v").view(self.E, MAXV)

    def networks(self):
        return [self.policy, self.policy_target]

    def _stat_nets(self, target):
        net = self.policy_target if target else self.policy
        return net, net

    def _target_values(self, S, A):
        """V_target(s) of the rows S [n, 30] (the value of the rollout of MAPPO_GI) -> [n]"""
        return self.policy_target(S, out_type="v")[:, 0]

    def sample_actions(self, obs, n_agents, seed, step):
        if self.fused:
            return policy_sample(self.policy, obs.contiguous(), n_agents, seed=seed, step=step)
        return self.act_torch(obs, n_agents)[0]

    def _learners(self):
        return [(self.policy, self.policy_target, self.policy_opt)]

    def _kernel_targets(self, batch, gae):
        """MAPPO_GI: old_logp of the shared target pass, which with gae also writes V_target(s) (into a zero-filled
        buffer), the values"""
        idx, S, A8, _ = batch
        values = torch.zeros(S.shape[0], device=self.dev) if gae else None
        return (ppo_targets(self.policy_target, S, A8, idx, value_out=values),), values

    def _kernel_gradients(self, batch, j, targets, losses):
        _, S, A8, G = batch
        return shared_network_gradients(self.policy, S, A8, G, *targets, j, self.clip_param, losses=losses)[1:]

    def _autograd_gradients(self, s, onehot, g):
        loss, actor_loss, critic_loss = shared_network_loss(self.policy, self.policy_target, s, onehot, g, self.clip_param)
        self.policy_opt.zero_grad(set_to_none=True)
        loss.backward()
        return actor_loss.detach(), critic_loss.detach()

"""GPU suite, optimiser: the device optimiser step (mm_rmsprop_step through rollout.DeviceRMSprop / rmsprop_step)
bit for bit against its numpy restatement (oracle/optim_ref.py), against torch's clip_grad_norm_ + RMSprop (foreach and
single-tensor), the dense first layer it keeps in step, determinism, state interchange with torch.optim.RMSprop, whole
updates of both rollout classes with optimizer="cuda" against optimizer="torch", and the training driver.

torch's CUDA kernels may contract a multiply and an add into one FMA; the library's kernels round every operation.  So
against torch: totals within 1e-6 relative, square_avg within 4 ulp per element per step, parameters within 4 ulp of
their tensor's largest magnitude per step (a parameter that passes near zero keeps the absolute rounding of the larger
values it was summed from).  The largest differences seen are printed."""
import copy
import glob
import math
import os

import numpy as np
import pytest

import optim_ref
from conftest import ROOT

pytestmark = pytest.mark.gpu

STEPS = 5
LR = 5e-4


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()
    return m


def _net(kind, seed):
    import torch
    from marl_mass_b200 import rollout
    torch.manual_seed(seed)
    return {"actor": rollout.ActorNetwork, "critic": rollout.CriticNetwork, "shared": rollout.ActorCriticNetwork}[kind]().cuda()


def _grads(net, seed, scale):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(p.shape, device="cuda", generator=g) * scale for p in net.parameters()]


def _ulps(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64))


def _param_ulps(a, b):
    return np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / np.spacing(np.float32(np.abs(b).max()))


def _np(ts):
    return [t.detach().cpu().numpy().copy() for t in ts]


@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
@pytest.mark.parametrize("scale,max_norm", [(100.0, 5.0), (1e-3, 5.0), (1.0, None)])
def test_device_step_matches_the_restatement_bit_for_bit(mm, kind, scale, max_norm):
    """parameters, square_avg, the clipped gradients and the norm after each of STEPS steps"""
    import torch
    from marl_mass_b200.rollout import DeviceRMSprop
    net = _net(kind, 3)
    opt = DeviceRMSprop(net.parameters(), lr=LR, max_grad_norm=max_norm)
    op, osq = _np(net.parameters()), [np.zeros(p.shape, np.float32) for p in net.parameters()]
    for s in range(STEPS):
        gs = _grads(net, 10 + s, scale)
        for p, g in zip(net.parameters(), gs):
            p.grad.copy_(g)
        opt.step()
        og = _np(gs)
        total = optim_ref.rmsprop_step(op, og, osq, LR, max_norm=max_norm)
        torch.cuda.synchronize()
        assert float(opt.total_norm) == float(total), (s, float(opt.total_norm), float(total))
        for a, b in zip(_np(p.grad for p in net.parameters()), og):
            np.testing.assert_array_equal(a, b)
        for a, b in zip(_np(net.parameters()), op):
            np.testing.assert_array_equal(a, b)
        for a, b in zip(_np(opt.state[p]["square_avg"] for p in net.parameters()), osq):
            np.testing.assert_array_equal(a, b)
    assert all(float(opt.state[p]["step"]) == STEPS for p in net.parameters())


def test_one_launch_steps_two_groups_with_different_lr(mm):
    """rmsprop_step([actor_opt, critic_opt]): each group as the restatement steps it on its own, divisor 3 included"""
    from marl_mass_b200.rollout import DeviceRMSprop, rmsprop_step
    nets = [_net("actor", 4), _net("critic", 5)]
    lrs = (5e-4, 2e-3)
    opts = [DeviceRMSprop(n.parameters(), lr=lr, max_grad_norm=5.0) for n, lr in zip(nets, lrs)]
    ref = [(_np(n.parameters()), [np.zeros(p.shape, np.float32) for p in n.parameters()]) for n in nets]
    scale = np.float32(1.0) / np.float32(3)
    for s in range(STEPS):
        want = []
        for k, (n, (op, osq)) in enumerate(zip(nets, ref)):
            gs = _grads(n, 100 * k + s, 30.0 if s % 2 else 1e-2)
            for p, g in zip(n.parameters(), gs):
                p.grad.copy_(g)
            want.append(optim_ref.rmsprop_step(op, _np(gs), osq, lrs[k], max_norm=5.0, grad_scale=scale))
        rmsprop_step(opts, grad_divisor=3)
        for k, (n, o, (op, osq)) in enumerate(zip(nets, opts, ref)):
            assert float(o.total_norm) == float(want[k])
            for a, b in zip(_np(n.parameters()) + _np(o.state[p]["square_avg"] for p in n.parameters()), op + osq):
                np.testing.assert_array_equal(a, b)


def test_grad_divisor_rounds_like_torch_division_on_the_device(mm):
    """`flat /= 3` of the torch all-reduce path and the kernel's scaling agree bit for bit (no clipping, lr 0)"""
    import torch
    from marl_mass_b200.rollout import DeviceRMSprop
    net = _net("critic", 6)
    opt = DeviceRMSprop(net.parameters(), lr=0.0, max_grad_norm=None)
    gs = _grads(net, 7, 1.0)
    flat = torch.cat([g.reshape(-1) for g in gs])
    opt.flat_grad.copy_(flat)
    opt.step(grad_divisor=3)
    flat /= 3
    assert torch.equal(opt.flat_grad, flat)


@pytest.mark.parametrize("foreach", [True, False])
@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
def test_device_step_against_torch(mm, kind, foreach):
    import torch
    from marl_mass_b200.rollout import DeviceRMSprop
    net_d, net_t = _net(kind, 8), _net(kind, 8)
    opt_d = DeviceRMSprop(net_d.parameters(), lr=LR, max_grad_norm=5.0)
    opt_t = torch.optim.RMSprop(net_t.parameters(), lr=LR, foreach=foreach)
    worst = [0.0, 0, 0.0]
    for s in range(STEPS):
        gs = _grads(net_d, 20 + s, 100.0 if s % 2 else 1e-3)
        for pd, pt, g in zip(net_d.parameters(), net_t.parameters(), gs):
            pd.grad.copy_(g)
            pt.grad = g.clone()
        opt_d.step()
        total_t = float(torch.nn.utils.clip_grad_norm_(list(net_t.parameters()), 5.0))
        opt_t.step()
        rel = abs(float(opt_d.total_norm) - total_t) / total_t
        u_sq = max(int(_ulps(a, b).max()) for a, b in zip(_np(opt_d.state[p]["square_avg"] for p in net_d.parameters()),
                                                           _np(opt_t.state[p]["square_avg"] for p in net_t.parameters())))
        u_p = max(float(_param_ulps(a, b).max()) for a, b in zip(_np(net_d.parameters()), _np(net_t.parameters())))
        worst = [max(worst[0], rel), max(worst[1], u_sq), max(worst[2], u_p)]
        assert rel <= 1e-6 and u_sq <= 4 * (s + 1) and u_p <= 4 * (s + 1), (s, rel, u_sq, u_p)
    print("%s foreach=%s: total %.1e rel, square_avg %d ulp, parameters %.1f ulp after %d steps" % (kind, foreach, *worst, STEPS))


def test_dense_first_layer_stays_in_step(mm):
    """After device steps of an ActorCriticNetwork, the dense layer kept by _split_first_layer (the same tensors, never
    rebuilt) equals a fresh rebuild bit for bit, and policy_sample draws the same actions with either."""
    import torch
    from marl_mass_b200 import rollout
    net = _net("shared", 9)
    opt = rollout.DeviceRMSprop(net.parameters(), lr=1e-2, max_grad_norm=5.0, shared_network=net)
    w0, b0 = rollout._split_first_layer(net)
    w_init = w0.clone()
    for s in range(STEPS):
        for p, g in zip(net.parameters(), _grads(net, 30 + s, 1.0)):
            p.grad.copy_(g)
        opt.step()
    w, b = rollout._split_first_layer(net)
    assert w is w0 and b is b0                      # the kept layer was written by the kernel, not rebuilt
    obs = torch.randn(4096, 12, 30, device="cuda")
    a_kept = rollout.policy_sample(net, obs, seed=3, step=1)
    rollout.first_layer_changed(net)
    w1, b1 = rollout._split_first_layer(net)
    assert w1 is not w0 and torch.equal(w1, w0) and torch.equal(b1, b0)
    assert not torch.equal(w0, w_init)
    a_fresh = rollout.policy_sample(net, obs, seed=3, step=1)
    assert torch.equal(a_kept, a_fresh)


def test_device_step_is_deterministic(mm):
    import torch
    from marl_mass_b200.rollout import DeviceRMSprop
    runs = []
    for _ in range(2):
        net = _net("shared", 11)
        opt = DeviceRMSprop(net.parameters(), lr=LR, max_grad_norm=5.0, shared_network=net)
        for s in range(STEPS):
            for p, g in zip(net.parameters(), _grads(net, 40 + s, 50.0)):
                p.grad.copy_(g)
            opt.step()
        runs.append([p.detach().clone() for p in net.parameters()] + [opt.total_norm.clone()])
    assert all(torch.equal(a, b) for a, b in zip(*runs))


@pytest.mark.parametrize("direction", ["device_to_torch", "torch_to_device"])
def test_state_dict_interchange_with_torch_rmsprop(mm, direction):
    """STEPS steps with one class, its state_dict loaded into the other, STEPS more: against continuing unchanged, within
    the tolerance of test_device_step_against_torch over 2 STEPS steps"""
    import torch
    from marl_mass_b200.rollout import DeviceRMSprop

    def make(cls, net):
        if cls == "device":
            return DeviceRMSprop(net.parameters(), lr=LR, max_grad_norm=5.0)
        return torch.optim.RMSprop(net.parameters(), lr=LR)

    def steps(net, opt, first):
        for s in range(first, first + STEPS):
            for p, g in zip(net.parameters(), _grads(net, 50 + s, 100.0 if s % 2 else 1e-3)):
                if isinstance(opt, DeviceRMSprop):
                    p.grad.copy_(g)
                else:
                    p.grad = g.clone()
            if not isinstance(opt, DeviceRMSprop):
                torch.nn.utils.clip_grad_norm_(list(net.parameters()), 5.0)
            opt.step()

    a, b = ("device", "torch") if direction == "device_to_torch" else ("torch", "device")
    net_x, net_y = _net("shared", 12), _net("shared", 12)
    opt_x, opt_y = make(a, net_x), make(a, net_y)
    steps(net_x, opt_x, 0)
    steps(net_y, opt_y, 0)
    opt_y2 = make(b, net_y)
    opt_y2.load_state_dict(copy.deepcopy(opt_y.state_dict()))
    assert all(float(opt_y2.state[p]["step"]) == STEPS for p in net_y.parameters())
    steps(net_x, opt_x, STEPS)
    steps(net_y, opt_y2, STEPS)
    assert all(float(opt_y2.state[p]["step"]) == 2 * STEPS for p in net_y.parameters())
    for p, q in zip(net_y.parameters(), net_x.parameters()):
        assert float(_param_ulps(p.detach().cpu().numpy(), q.detach().cpu().numpy()).max()) <= 4 * 2 * STEPS
    for p, q in zip(net_y.parameters(), net_x.parameters()):
        sy, sx = opt_y2.state[p]["square_avg"], opt_x.state[q]["square_avg"]
        assert int(_ulps(sy.cpu().numpy(), sx.cpu().numpy()).max()) <= 4 * 2 * STEPS


def _rollout_pair(shared, envs=512, steps=60):
    """one collect() of the shipped ini, and a second rollout object with copies of the same networks, optimizer="cuda",
    on the same buffer"""
    import torch
    from marl_mass_b200.env import DEFAULT_CONFIG, MergeEnvBatched
    from marl_mass_b200.rollout import BatchedMAPPOGIRollout, BatchedMAPPORollout
    from marl_mass_b200.train import load_ini
    ini = "mass_td3_mixed_srew_shared.ini" if shared else "mass_td3_srew.ini"
    env_cfg, kw, _ = load_ini(os.path.join(ROOT, "examples", ini))
    kw["roll_out_n_steps"] = steps
    env = MergeEnvBatched(envs, dict(DEFAULT_CONFIG, **env_cfg), device=0)
    torch.manual_seed(11)
    cls = BatchedMAPPOGIRollout if shared else BatchedMAPPORollout
    pol_t = cls(env, seed=5, **kw)
    pol_t.collect()
    nets = {"policy": copy.deepcopy(pol_t.policy)} if shared else {"actor": copy.deepcopy(pol_t.actor),
                                                                    "critic": copy.deepcopy(pol_t.critic)}
    pol_c = cls(env, seed=5, optimizer="cuda", **nets, **kw)
    pol_c.buf = pol_t.buf
    torch.cuda.synchronize()
    return env, pol_t, pol_c


@pytest.mark.parametrize("impl", ["torch", "cuda"])
@pytest.mark.parametrize("shared", [False, True])
def test_whole_update_with_device_optimizer(mm, monkeypatch, shared, impl):
    """update(impl, epochs=2) with optimizer="cuda" against optimizer="torch" from the same networks, data and
    torch.manual_seed (one minibatch per epoch): every parameter tensor within 1e-5 relative, the same stats keys, the
    first minibatch's losses identical (the networks have not been stepped yet).  Over more steps the two runs drift
    further apart: on a B200, 4 minibatches x 2 epochs left the MAPPO tensors up to 5.7e-4 apart (MAPPO_GI: 1.6e-5),
    which this test does not bound; where that growth comes from was not isolated."""
    import torch
    from marl_mass_b200 import rollout
    env, pol_t, pol_c = _rollout_pair(shared)
    name = {("torch", False): "mappo_losses", ("torch", True): "shared_network_loss",
            ("cuda", False): "mappo_gradients", ("cuda", True): "shared_network_gradients"}[(impl, shared)]
    fn = getattr(rollout, name)
    seen = []

    def recorded(*args, **kw):
        out = fn(*args, **kw)
        seen.append([float(x) for x in out])
        return out

    monkeypatch.setattr(rollout, name, recorded)
    live = int(pol_t.buf["live"].sum())
    stats = []
    for pol in (pol_t, pol_c):
        torch.manual_seed(99)
        stats.append(pol.update(minibatch=live, epochs=2, impl=impl))
    assert len(seen) == 4
    assert seen[0] == seen[2]
    assert set(stats[0]) == set(stats[1])
    worst = 0.0
    for m_t, m_c in zip(pol_t.networks(), pol_c.networks()):
        for p, q in zip(m_t.parameters(), m_c.parameters()):
            rel = float((p - q).norm() / p.norm())
            worst = max(worst, rel)
            assert rel <= 1e-5, rel
    print("shared=%s impl=%s: worst parameter tensor %.2e relative" % (shared, impl, worst))
    env.close()


@pytest.mark.parametrize("ini", sorted(glob.glob(os.path.join(ROOT, "examples", "*.ini"))))
def test_driver_with_device_optimizer(mm, ini):
    from marl_mass_b200.train import train
    hist = train(ini, n_envs=512, iterations=2, eval_interval=1, log=lambda *_: None, update_impl="cuda", optimizer="cuda")
    assert len(hist) == 2
    for rec in hist:
        assert math.isfinite(rec["actor_loss"]) and math.isfinite(rec["critic_loss"]) and rec["samples"] > 0
        assert math.isfinite(rec["eval_reward"])

"""CPU tests of the on-device PPO learner: the numpy restatement of its per-row loss derivative (oracle/learner_ref.py)
pinned against torch autograd on the CPU, ties and clip bounds included, and the argument checks of mm_ppo_targets /
mm_ppo_grads, which reject bad calls before any CUDA call (so they run without a GPU)."""
import ctypes as C

import numpy as np
import pytest
import torch

import learner_ref

CLIP = 0.2


def _torch_row_grads(ratio, adv, clip):
    """d(-mean(min(r adv, clamp(r) adv))) / d logp with r = exp(logp - old), via autograd, times N (per row)."""
    old = torch.zeros(len(ratio), dtype=torch.float32)
    logp = torch.log(torch.tensor(ratio, dtype=torch.float32)).requires_grad_(True)
    r = torch.exp(logp - old)
    a = torch.tensor(adv, dtype=torch.float32)
    loss = -torch.min(r * a, torch.clamp(r, 1.0 - clip, 1.0 + clip) * a).mean()
    loss.backward()
    return r.detach().numpy(), logp.grad.numpy() * len(ratio), float(loss.detach())


def test_ppo_row_derivative_matches_autograd_at_ties_and_clip_bounds():
    lo, hi = np.float32(1.0) - np.float32(CLIP), np.float32(1.0) + np.float32(CLIP)
    # ratios: exactly 1, both bounds, inside, above and below the clip range; advantages positive, negative and zero
    ratios = [1.0, float(lo), float(hi), 1.05, 0.95, 1.7, 0.3]
    advs = [2.5, -1.25, 0.0]
    R, A = np.meshgrid(np.array(ratios, np.float32), np.array(advs, np.float32))
    R, A = R.ravel(), A.ravel()
    r_t, g_t, loss_t = _torch_row_grads(R, A, CLIP)
    # the restatement takes the ratio torch actually formed (exp(log r) rounds)
    loss_o, g_o = learner_ref.ppo_row(r_t, A, CLIP)
    np.testing.assert_allclose(g_o, g_t, rtol=1e-6, atol=1e-7)
    assert abs(float(loss_o.mean()) - loss_t) <= 1e-6 * max(1.0, abs(loss_t))
    # clipped rows contribute nothing: r above 1 + c with adv > 0, below 1 - c with adv < 0
    clipped = ((r_t > hi) & (A > 0)) | ((r_t < lo) & (A < 0))
    assert clipped.any() and np.all(g_o[clipped] == 0.0)
    # a zero advantage gives a zero derivative; r == 1 (a tie of the two surrogates) gives adv * r, as unclipped rows do
    assert np.all(g_o[A == 0] == 0.0)
    one = (r_t == 1.0) & (A != 0)
    assert one.any()
    np.testing.assert_array_equal(g_o[one], -A[one])


def test_ppo_row_derivative_matches_autograd_on_random_rows():
    rng = np.random.default_rng(3)
    n = 4096
    ratio = np.exp(rng.normal(0, 0.3, n)).astype(np.float32)
    adv = rng.normal(0, 2.0, n).astype(np.float32)
    r_t, g_t, _ = _torch_row_grads(ratio, adv, CLIP)
    _, g_o = learner_ref.ppo_row(r_t, adv, CLIP)
    np.testing.assert_allclose(g_o, g_t, rtol=1e-5, atol=1e-6)


def test_logit_and_value_derivatives_match_autograd():
    rng = np.random.default_rng(4)
    n = 257
    z = torch.tensor(rng.normal(0, 1.5, (n, 5)), dtype=torch.float64, requires_grad=True)
    a = rng.integers(0, 5, n)
    g = rng.normal(0, 1, n)
    logp = torch.log_softmax(z, 1)[torch.arange(n), torch.from_numpy(a)]
    (logp * torch.from_numpy(g)).sum().backward()
    np.testing.assert_allclose(learner_ref.logit_grad(z.detach().numpy(), a, g), z.grad.numpy(), rtol=1e-10, atol=1e-12)
    v = torch.tensor(rng.normal(0, 1, (n, 1)), dtype=torch.float32, requires_grad=True)
    G = torch.tensor(rng.normal(0, 1, (n, 1)), dtype=torch.float32)
    loss = torch.nn.functional.mse_loss(v, G)
    loss.backward()
    l_o, d_o = learner_ref.value_row(v.detach().numpy(), G.numpy())
    np.testing.assert_allclose(d_o / n, v.grad.numpy(), rtol=1e-6)
    assert abs(float(l_o.mean()) - float(loss)) < 1e-6


@pytest.fixture(scope="module")
def L():
    import marl_mass_b200 as mm
    from marl_mass_b200 import build
    build.build()
    return mm.lib()


def _fake(n=8):
    """non-null host addresses: the checks must fail before anything is dereferenced or launched"""
    return [C.c_void_p(0x1000 * (k + 1)) for k in range(n)]


def _net(kind):
    from marl_mass_b200 import _lib
    p = [0x1000 * (k + 1) for k in range(8)]
    if kind != _lib.PPO_SHARED:
        p[6] = p[7] = 0
    return _lib.MMPpoNet(*p)


def _grads():
    from marl_mass_b200 import _lib
    return _lib.MMPpoGrads(*[0x2000 * (k + 1) for k in range(8)])


def _targets(L, kind, n=16, net="ok", old=True, q=True, states=True):
    from marl_mass_b200 import _lib
    f = _fake()
    nt = _net(kind if kind in (0, 1, 2) else 0) if net == "ok" else net
    return L.mm_ppo_targets(kind, f[0] if states else None, f[1], f[2], n, None if nt is None else C.byref(nt),
                            f[3] if old else None, f[4] if q else None, None)


def _grad_call(L, kind, n=16, clip=0.2, old=True, q=True, grads="ok", losses=True, net="ok"):
    f = _fake()
    nt = _net(kind if kind in (0, 1, 2) else 0) if net == "ok" else net
    g = _grads() if grads == "ok" else grads
    return L.mm_ppo_grads(kind, f[0], f[1], f[2], f[3] if old else None, f[4] if q else None, f[5], n, clip,
                          None if nt is None else C.byref(nt), None if g is None else C.byref(g), f[6] if losses else None, None)


def test_ppo_entry_points_reject_bad_arguments_before_any_cuda_call(L):
    from marl_mass_b200 import _lib

    def rejected(rc, what):
        assert rc == -1, (rc, what)
        assert what in L.mm_last_error().decode(), L.mm_last_error()

    rejected(_targets(L, 3), "kind")
    rejected(_targets(L, -1), "kind")
    rejected(_targets(L, 0, n=0), "n must be >= 1")
    rejected(_targets(L, 0, n=-5), "n must be >= 1")
    rejected(_targets(L, 0, net=None), "net")
    rejected(_targets(L, 2, net=_net(0)), "w4")                 # the shared network needs critic_linear
    rejected(_targets(L, 0, states=False), "states")
    rejected(_targets(L, 0, old=False), "old_logp")
    rejected(_targets(L, 1, q=False), "q_target")
    rejected(_grad_call(L, 7), "kind")
    rejected(_grad_call(L, 0, n=0), "n must be >= 1")
    for clip in (0.0, 1.0, -0.2, 1.5, float("nan")):
        rejected(_grad_call(L, 0, clip=clip), "clip")
    rejected(_grad_call(L, 0, old=False), "old_logp")
    rejected(_grad_call(L, 2, old=False), "old_logp")
    rejected(_grad_call(L, 0, q=False), "q_target")
    rejected(_grad_call(L, 0, grads=None), "grads")
    rejected(_grad_call(L, 0, losses=False), "losses")
    g = _grads()
    g.w4 = None
    rejected(_grad_call(L, 2, grads=g), "grads")
    rejected(_grad_call(L, 2, net=_net(1)), "w4")
    n = _net(0)
    n.b2 = None
    rejected(_grad_call(L, 0, net=n), "net")
    assert _lib.ABI_VERSION == 9 and L.mm_abi_version() == 9

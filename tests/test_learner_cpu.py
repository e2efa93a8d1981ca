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


# ---- the whole learner pass (learner_ref.learner_pass) against torch autograd in float64

def _torch_nets(kind, seed):
    from marl_mass_b200 import rollout
    torch.manual_seed(seed)
    net = {"actor": rollout.ActorNetwork, "critic": rollout.CriticNetwork, "shared": rollout.ActorCriticNetwork}[kind]()
    return net.double()


def _f64_rows(rows, seed):
    rng = np.random.default_rng(seed)
    return rng.normal(0, 1, (rows, 30)), rng.integers(0, 5, rows).astype(np.int8), rng.normal(0, 3, rows)


def _torch_pass(kind, net, S, A8, G, old, q, idx, clip=CLIP):
    """autograd of the batched losses on the rows S[idx]: -> ({name: grad}, actor loss, critic loss)"""
    j = torch.from_numpy(idx)
    s = torch.from_numpy(S)[j]
    onehot = torch.nn.functional.one_hot(torch.from_numpy(A8.astype(np.int64))[j], 5).double()
    g = torch.from_numpy(G)[j]
    net.zero_grad(set_to_none=True)
    a_loss = c_loss = torch.zeros((), dtype=torch.float64)
    if kind == "critic":
        c_loss = torch.nn.functional.mse_loss(net(s, onehot), g[:, None])
    else:
        hidden = net.trunk(s) if kind == "shared" else None
        logp = ((net.policy_head(hidden) if kind == "shared" else net(s)) * onehot).sum(1)
        if kind == "shared":
            values = net.critic_linear(hidden)
            adv = (g[:, None] - values.detach()).squeeze(1)
            c_loss = torch.nn.functional.mse_loss(values, g[:, None])
        else:
            adv = g - torch.from_numpy(q)[j]
        ratio = torch.exp(logp - torch.from_numpy(old)[j])
        a_loss = -torch.min(ratio * adv, torch.clamp(ratio, 1.0 - clip, 1.0 + clip) * adv).mean()
    (a_loss + c_loss).backward()
    return {n: p.grad.numpy().copy() for n, p in net.named_parameters()}, float(a_loss), float(c_loss)


def _params64(net):
    return {n: p.detach().numpy().copy() for n, p in net.named_parameters()}


def _assert_pass_matches(ref, grads, a_loss, c_loss, tol=1e-12):
    assert set(ref["grads"]) == set(grads)
    for n, g in grads.items():
        assert ref["grads"][n].shape == g.shape, n
        err = np.abs(ref["grads"][n] - g).max() / max(np.abs(g).max(), 1e-30)
        assert err <= tol, (n, err)
    assert abs(ref["loss_a"] - a_loss) <= tol * max(1.0, abs(a_loss))
    assert abs(ref["loss_c"] - c_loss) <= tol * max(1.0, abs(c_loss))


@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
def test_learner_pass_matches_torch_autograd_in_float64(kind):
    """Rows with r == 1 (old = the current log-probability: the tie of the two surrogates), ratios far outside the clip
    range on both sides and with both advantage signs (clipped and unclipped), unsorted and duplicate indices."""
    rows = 400
    S, A8, G = _f64_rows(rows, 7)
    net = _torch_nets(kind, 3)
    params = _params64(net)
    rng = np.random.default_rng(8)
    idx = rng.integers(0, rows, 333)                     # unsorted, with duplicates
    q = rng.normal(0, 1, rows)
    target = learner_ref.learner_pass(kind, params, S, A8, None, None, None, np.arange(rows), CLIP)
    if kind == "critic":
        old = None
        with torch.no_grad():
            want_q = net(torch.from_numpy(S), torch.nn.functional.one_hot(torch.from_numpy(A8.astype(np.int64)), 5).double())
        np.testing.assert_allclose(target["q"], want_q.numpy()[:, 0], rtol=1e-13, atol=1e-13)
    else:
        regime = np.arange(rows) % 4                      # r == 1, r ~ e^0.7, r ~ e^-0.7, r within the clip range
        old = target["logp"] - np.choose(regime, [0.0, 0.7, -0.7, 0.05])
        old[regime == 0] = target["logp"][regime == 0]
    ref = learner_ref.learner_pass(kind, params, S, A8, G, old, q, idx, CLIP)
    grads, a_loss, c_loss = _torch_pass(kind, net, S, A8, G, old, q, idx)
    _assert_pass_matches(ref, grads, a_loss, c_loss)
    if kind != "critic":
        r = ref["ratio"]
        clipped = ((r > 1 + CLIP) & (ref["adv"] > 0)) | ((r < 1 - CLIP) & (ref["adv"] < 0))
        assert clipped.any() and (~clipped & (np.abs(r - 1) > CLIP)).any() and np.all(ref["gl"][clipped] == 0)
        assert np.any(np.abs(r - 1) < 1e-15)


@pytest.mark.parametrize("shared", [False, True])
def test_learner_pass_matches_the_rollout_losses(shared):
    """The restatement against the losses the torch learner steps (rollout.mappo_losses / shared_network_loss) with the
    target networks equal to the networks: every ratio is 1, the tie of the two surrogates on every row."""
    import copy
    from marl_mass_b200 import rollout
    rows = 300
    S, A8, G = _f64_rows(rows, 11)
    idx = np.random.default_rng(12).permutation(rows)[:257]
    j = torch.from_numpy(idx)
    s, g = torch.from_numpy(S)[j], torch.from_numpy(G)[j][:, None]
    onehot = torch.nn.functional.one_hot(torch.from_numpy(A8.astype(np.int64))[j], 5).double()
    nets = [_torch_nets("shared", 5)] if shared else [_torch_nets("actor", 5), _torch_nets("critic", 6)]
    if shared:
        loss, a_loss, c_loss = rollout.shared_network_loss(nets[0], copy.deepcopy(nets[0]), s, onehot, g, CLIP)
        loss.backward()
    else:
        a_loss, c_loss = rollout.mappo_losses(nets[0], copy.deepcopy(nets[0]), nets[1], copy.deepcopy(nets[1]), s, onehot,
                                              g, CLIP)
        (a_loss + c_loss).backward()
    kinds = ["shared"] if shared else ["actor", "critic"]
    q = None
    if not shared:
        q = learner_ref.learner_pass("critic", _params64(nets[1]), S, A8, None, None, None, np.arange(rows), CLIP)["q"]
    for kind, net in zip(kinds, nets):
        params = _params64(net)
        old = None if kind == "critic" else learner_ref.learner_pass(kind, params, S, A8, None, None, None, np.arange(rows), CLIP)["logp"]
        ref = learner_ref.learner_pass(kind, params, S, A8, G, old, q, idx, CLIP)
        grads = {n: p.grad.numpy() for n, p in net.named_parameters()}
        _assert_pass_matches(ref, grads, float(a_loss) if kind != "critic" else 0.0, float(c_loss) if kind != "actor" else 0.0)


# ---- the exactly representable data of the bit-exact GPU tests: its premises, checked on the CPU

@pytest.mark.parametrize("n,group", [(1, 1), (17, 2), (129, 4), (129, 1), (100003, 2)])
def test_exact_data_premises_hold(n, group):
    """learner_ref.check_exact_case raises unless every fp16 / fp32 step of the kernel is exact on the data and the data
    is not degenerate; the float64 pass must then agree with it to the rounding of old_logp to fp32."""
    rows = n + 40
    S, A8 = learner_ref.exact_rows(rows, n)
    idx = learner_ref.exact_index(n, rows, n + 1)
    probes = [0, n - 1]
    all_rows = np.arange(rows)
    pa, pc = learner_ref.exact_params("actor", group, 3), learner_ref.exact_params("critic", group, 4)
    ps = learner_ref.exact_params("shared", group, 6)
    learner_ref.exact_probe_actions(A8, idx, probes)
    q = learner_ref.learner_pass("critic", pc, S, A8, None, None, None, all_rows, learner_ref.EXACT_CLIP, fp16=True, check=True)["q"]
    G, shift = learner_ref.exact_offsets(q, idx, probes, 5)
    logp = learner_ref.learner_pass("actor", pa, S, A8, None, None, None, all_rows, learner_ref.EXACT_CLIP, fp16=True, check=True)["logp"]
    cases = [("actor", pa, (logp - shift).astype(np.float32), q), ("critic", pc, None, None)]
    v = learner_ref.learner_pass("shared", ps, S, A8, None, None, None, all_rows, learner_ref.EXACT_CLIP, fp16=True, check=True)
    Gs, shift_s = learner_ref.exact_offsets(v["v"], idx, probes, 6)
    for kind, params, old, qt in cases + [("shared", ps, (v["logp"] - shift_s).astype(np.float32), None)]:
        g = Gs if kind == "shared" else G
        ref = learner_ref.check_exact_case(kind, params, S, A8, g, old, qt, idx)
        f64 = learner_ref.learner_pass(kind, params, S, A8, g, old, qt, idx, learner_ref.EXACT_CLIP)
        for name in ref["grads"]:
            # the float64 pass has p ~ e^-110 where the fp32 one has 0, and r = 1 only up to the fp32 rounding of old_logp
            scale = np.abs(ref["sums"][name]).max()
            np.testing.assert_allclose(ref["sums"][name], f64["sums"][name], rtol=0, atol=1e-5 * scale)
        for p in probes:                       # every probe row moves the sums: a lost or doubled row would show
            rest = np.delete(idx, p)
            without = learner_ref.learner_pass(kind, params, S, A8, g, old, qt, rest, learner_ref.EXACT_CLIP, fp16=True)
            assert any(not np.array_equal(ref["sums"][k], without["sums"][k]) for k in ref["sums"]), (kind, p)


def test_exact_data_premise_checks_fail_on_inexact_data():
    """the checks are live: a weight off the fp16 grid, an input off it, and sums too long for fp32 are each reported"""
    rows = 200
    S, A8 = learner_ref.exact_rows(rows, 1)
    idx = np.arange(rows)
    p = learner_ref.exact_params("critic", 1, 2)
    G = np.zeros(rows, np.float32)
    learner_ref.check_exact_case("critic", p, S, A8, G, None, None, idx)
    bad = dict(p, **{"fc2.weight": p["fc2.weight"] * np.float32(1 + 2 ** -12)})
    with pytest.raises(learner_ref.Exactness, match="W2"):
        learner_ref.check_exact_case("critic", bad, S, A8, G, None, None, idx)
    with pytest.raises(learner_ref.Exactness, match="input"):
        learner_ref.check_exact_case("critic", p, S + np.float32(2 ** -13), A8, G, None, None, idx)
    with pytest.raises(learner_ref.Exactness, match="2\\^24"):
        learner_ref.check_exact_case("critic", p, S, A8, G + np.float32(256), None, None, idx)

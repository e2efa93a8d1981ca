"""GPU suite, learner, bit for bit: mm_ppo_targets / mm_ppo_grads (through rollout.ppo_targets, mappo_gradients and
shared_network_gradients) on exactly representable data against learner_ref.learner_pass(fp16=True).

The networks and rows come from learner_ref.exact_params / exact_rows: small integers and quarter steps with sparse
weights, so every value the kernel rounds to fp16 is an fp16 value and every fp32 sum it forms is exact (fp16 products
are exact in fp32, and sums of multiples of one unit are exact while they stay below 2^24 units).  The policy head
gives p in {0, 1/c} exactly, old_logp comes from the target pass (r == 1 exactly, so the per-row derivative is -adv)
or is pushed outside the clip range to the side where PPO clips (derivative 0).  The kernel's result then does not
depend on summation order, and the only inexact step, the reduction's `sum * (1 / N)` in fp32, is the reference's too:
every gradient element and both losses must match bit for bit.  learner_ref.check_exact_case verifies these premises on
the data of every case and fails loudly if one does not hold.

A defect that touches a few rows or elements - a lost tail tile, a CTA partial counted twice, an entry scattered to the
wrong place - changes bits here, where the norm tolerances of test_gpu_learner.py could absorb it.  The probe rows
(the first row, the last row of a partial last tile, the first row of a CTA's second tile) are checked to move the
reference's sums, so losing or doubling any of them would show.
"""
import numpy as np
import pytest

import learner_ref

pytestmark = pytest.mark.gpu

CLIP = learner_ref.EXACT_CLIP
GROUPS = (1, 2, 4)


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


def _module(kind, params):
    import torch
    from marl_mass_b200 import rollout
    net = {"actor": rollout.ActorNetwork, "critic": rollout.CriticNetwork, "shared": rollout.ActorCriticNetwork}[kind]().cuda()
    with torch.no_grad():
        for name, p in net.named_parameters():
            p.copy_(torch.from_numpy(params[name]))
    return net


def _bits(v):
    return np.ascontiguousarray(np.asarray(v, np.float32)).view(np.int32)


def _assert_bitwise(got, want, what):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = _bits(got) != _bits(want)
    assert not bad.any(), (what, int(bad.sum()), float(np.abs(got.astype(np.float64) - want).max()))


class Case:
    """One exactly representable learner call: `which` "mappo" (actor + critic) or "shared", n rows of S through idx,
    the policy head's group size c.  S [rows, 30] has `rows` rows; `place` maps the compact rows to the rows of S the
    kernel reads (the rows beyond 2^31 floats)."""

    def __init__(self, which, n, sms, group, seed, rows=None, place=None):
        self.which, self.n, self.group = which, n, group
        rows_c = n + 40 if place is None else n
        S, A8 = learner_ref.exact_rows(rows_c, seed)
        idx = learner_ref.exact_index(n, rows_c, seed + 1) if place is None else np.arange(n, dtype=np.int64)
        tile2 = sms * 128
        self.probes = sorted({0} | ({n - 1} if n % 128 else set()) | ({tile2} if n > tile2 else set()))
        learner_ref.exact_probe_actions(A8, idx, self.probes)
        every = np.arange(rows_c)
        if which == "mappo":
            self.params = {"actor": learner_ref.exact_params("actor", group, seed + 2),
                           "critic": learner_ref.exact_params("critic", group, seed + 3)}
            q = learner_ref.learner_pass("critic", self.params["critic"], S, A8, None, None, None, every, CLIP,
                                         fp16=True, check=True)["q"]
            G, shift = learner_ref.exact_offsets(q, idx, self.probes, seed + 4)
            logp = learner_ref.learner_pass("actor", self.params["actor"], S, A8, None, None, None, every, CLIP,
                                            fp16=True, check=True)["logp"]
            self.kinds = {"actor": ((logp - shift).astype(np.float32), q), "critic": (None, None)}
            self.q_ref = q
        else:
            self.params = {"shared": learner_ref.exact_params("shared", group, seed + 5)}
            t = learner_ref.learner_pass("shared", self.params["shared"], S, A8, None, None, None, every, CLIP,
                                         fp16=True, check=True)
            G, shift = learner_ref.exact_offsets(t["v"], idx, self.probes, seed + 4)
            logp = t["logp"]
            self.kinds = {"shared": ((logp - shift).astype(np.float32), None)}
        self.S, self.A8, self.G, self.idx, self.shift, self.logp_ref = S, A8, G, idx, shift, logp
        self.ref = {k: learner_ref.check_exact_case(k, self.params[k], S, A8, G, old, q, idx)
                    for k, (old, q) in self.kinds.items()}
        self.rows, self.place = (rows_c if rows is None else rows), place

    def probes_visible(self):
        """the reference without each probe row differs from the full reference"""
        for k, (old, q) in self.kinds.items():
            for p in self.probes:
                rest = np.delete(self.idx, p)
                without = learner_ref.learner_pass(k, self.params[k], self.S, self.A8, self.G, old, q, rest, CLIP, fp16=True)
                assert any(not np.array_equal(self.ref[k]["sums"][m], without["sums"][m]) for m in without["sums"]), \
                    (self.which, self.n, k, p)

    def upload(self):
        import torch
        if self.place is None:
            self.St = torch.from_numpy(self.S).cuda()
            self.A8t = torch.from_numpy(self.A8).cuda()
            self.Gt = torch.from_numpy(self.G).cuda()
            self.idxt = torch.from_numpy(self.idx).cuda()
            self.shiftt = torch.from_numpy(self.shift).cuda()
            return
        # only the indexed rows of the large buffers are written; the kernels read no others
        dst = torch.from_numpy(self.place).cuda()
        self.St = torch.empty((self.rows, 30), device="cuda")
        self.A8t = torch.zeros(self.rows, dtype=torch.int8, device="cuda")
        self.Gt = torch.empty(self.rows, device="cuda")
        self.shiftt = torch.zeros(self.rows, device="cuda")
        self.St[dst] = torch.from_numpy(self.S).cuda()
        self.A8t[dst] = torch.from_numpy(self.A8).cuda()
        self.Gt[dst] = torch.from_numpy(self.G).cuda()
        self.shiftt[dst] = torch.from_numpy(self.shift).cuda()
        self.idxt = dst

    def run_and_check(self):
        """target passes and the gradient pass on the device, each output against the reference bit for bit"""
        import torch
        from marl_mass_b200 import rollout
        rows_of_idx = self.idx                 # the reference's rows in idx order (compact when `place` is set)
        j = self.idxt
        nets = {k: _module(k, p) for k, p in self.params.items()}
        for net in nets.values():
            for p in net.parameters():
                p.grad = torch.full_like(p, float("nan"))             # the kernels overwrite every element
        if self.which == "mappo":
            q = rollout.ppo_targets(nets["critic"], self.St, self.A8t, j)
            _assert_bitwise(q[j].cpu().numpy(), self.q_ref[rows_of_idx], "Q_target")
            logp = rollout.ppo_targets(nets["actor"], self.St, self.A8t, j)
            a, c = rollout.mappo_gradients(nets["actor"], nets["critic"], self.St, self.A8t, self.Gt, logp - self.shiftt, q, j, CLIP)
            losses = {"actor": (float(a), None), "critic": (None, float(c))}
        else:
            logp = rollout.ppo_targets(nets["shared"], self.St, self.A8t, j)
            _, a, c = rollout.shared_network_gradients(nets["shared"], self.St, self.A8t, self.Gt, logp - self.shiftt, j, CLIP)
            losses = {"shared": (float(a), float(c))}
        # logp: the reference's logf(c) is numpy's; at most 2 ulp apart
        d = np.abs(_bits(logp[j].cpu().numpy()).astype(np.int64) - _bits(self.logp_ref[rows_of_idx]).astype(np.int64))
        assert d.max() <= 2, ("logp ulp", int(d.max()))
        for k, net in nets.items():
            ref = self.ref[k]
            for name, p in net.named_parameters():
                _assert_bitwise(p.grad.cpu().numpy(), ref["grads"][name], (self.which, self.n, self.group, k, name))
            la, lc = losses[k]
            if la is not None:
                _assert_bitwise(la, ref["loss_a"], (self.which, self.n, k, "loss_a"))
            if lc is not None:
                _assert_bitwise(lc, ref["loss_c"], (self.which, self.n, k, "loss_c"))


def _sizes(sms):
    t = sms * 128
    return [1, 2, 15, 16, 17, 127, 128, 129, 255, 257, t - 1, t, t + 1, 2 * t + 77, 100003]


@pytest.mark.parametrize("which", ["mappo", "shared"])
def test_learner_bit_exact_at_every_tile_edge(mm, sms, which):
    """n at the tile, grid and second-tile edges of this device (S = its SM count) and 100 003; unsorted indices with
    duplicates and the last row of S; policy-head groups of 1, 2 and 4 actions in turn."""
    for k, n in enumerate(_sizes(sms)):
        case = Case(which, n, sms, GROUPS[k % 3], seed=1000 + n)
        case.probes_visible()
        case.upload()
        case.run_and_check()


def test_workspace_reuse_across_kinds_and_sizes(mm, sms):
    """calls that alternate kinds and shrink after a full grid: the partials workspace is shared, and a call must read
    only its own CTAs' partials"""
    t = sms * 128
    plan = [("shared", 2 * t + 77), ("mappo", 129), ("shared", 1), ("mappo", t + 1), ("shared", 17), ("mappo", 2)]
    cases = [Case(w, n, sms, GROUPS[k % 3], seed=2000 + k) for k, (w, n) in enumerate(plan)]
    for c in cases:
        c.upload()
    for c in cases + cases[::-1]:
        c.run_and_check()


def test_rows_beyond_2_31_floats(mm, sms):
    """72 M rows of S (8.6 GB; a 65 536-env, 100-step rollout has 78.6 M): rows whose first float lies beyond 2^31
    floats into S, and the last row, only those rows written"""
    rows = 72_000_000
    first = (1 << 31) // 30 + 1
    rng = np.random.default_rng(5)
    for k, which in enumerate(("mappo", "shared")):
        n = 2 * 128 + 77
        place = np.sort(rng.choice(np.arange(first, rows - 1), n - 1, replace=False))
        place = rng.permutation(np.append(place, rows - 1)).astype(np.int64)
        assert place.min() * 30 >= 1 << 31
        case = Case(which, n, sms, GROUPS[k], seed=3000 + k, rows=rows, place=place)
        case.upload()
        case.run_and_check()
        del case
        import torch
        torch.cuda.empty_cache()


def test_empty_index_list_gives_zero_gradients(mm):
    """an empty shard of a data-parallel update: every gradient is zero (not left as it was)"""
    import torch
    from marl_mass_b200 import rollout
    S = torch.zeros((4, 30), device="cuda")
    A8 = torch.zeros(4, dtype=torch.int8, device="cuda")
    G = torch.zeros(4, device="cuda")
    j = torch.zeros(0, dtype=torch.int64, device="cuda")
    actor = _module("actor", learner_ref.exact_params("actor", 1, 1))
    critic = _module("critic", learner_ref.exact_params("critic", 1, 2))
    pol = _module("shared", learner_ref.exact_params("shared", 1, 3))
    for net in (actor, critic, pol):
        for p in net.parameters():
            p.grad = torch.full_like(p, float("nan"))
    rollout.mappo_gradients(actor, critic, S, A8, G, G, G, j, CLIP)
    rollout.shared_network_gradients(pol, S, A8, G, G, j, CLIP)
    for net in (actor, critic, pol):
        for name, p in net.named_parameters():
            assert torch.equal(p.grad, torch.zeros_like(p)), name

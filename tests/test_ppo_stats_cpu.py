"""CPU tests of the learner's statistics pass (mm_ppo_stats): the C ABI declaration and export, the argument checks that
come before any CUDA call, the float64 restatement (ppo_stats_ref.py) against the torch statistics
(rollout.ppo_stats_torch) on float64 modules, the keys formed from the vectors, and the driver's refusals."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import ppo_stats_ref
from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "marl_mass_b200.h")
INI = os.path.join(ROOT, "examples", "mass_td3_srew.ini")
CLIP = 0.2


def test_header_declares_and_library_exports_the_entry_point():
    import marl_mass_b200 as mm
    from marl_mass_b200 import _lib
    src = open(HEADER).read()
    assert re.search(r"int mm_ppo_stats\(int kind, const float \*states, const int8_t \*actions, const float \*returns, "
                     r"const float \*old_logp,\s+const int64_t \*idx, int64_t n, float clip, const mm_ppo_net \*net, "
                     r"double \*stats, void \*stream\);", src)
    enum = re.search(r"enum \{ (MM_PPO_STAT_N,[^}]*)\};", src).group(1)
    names = [e.strip() for e in enum.split(",") if e.strip()]
    assert names[-1] == "MM_PPO_STATS_LEN" and len(names) - 1 == _lib.PPO_STATS_LEN
    assert [n[len("MM_PPO_STAT_"):].lower() for n in names[:-1]] == list(_lib.PPO_STAT_FIELDS)
    assert tuple(_lib.PPO_STAT_FIELDS) == ppo_stats_ref.FIELDS
    assert "mm_ppo_stats" in _lib.EXPORTS and mm.lib().mm_ppo_stats is not None
    assert re.search(r"#define MM_ABI_VERSION 9\b", src)


@pytest.fixture(scope="module")
def L():
    import marl_mass_b200 as mm
    from marl_mass_b200 import build
    build.build()
    return mm.lib()


def _net(kind):
    from marl_mass_b200 import _lib
    p = [0x1000 * (k + 1) for k in range(8)]
    if kind != _lib.PPO_SHARED:
        p[6] = p[7] = 0
    return _lib.MMPpoNet(*p)


def _call(L, kind, n=16, clip=CLIP, states=True, actions=True, returns=True, old=True, idx=True, net="ok", stats=True):
    """non-null fake host addresses: the checks must fail before anything is dereferenced or launched"""
    f = [C.c_void_p(0x1000 * (k + 1)) for k in range(6)]
    nt = _net(kind if kind in (0, 1, 2) else 0) if net == "ok" else net
    return L.mm_ppo_stats(kind, f[0] if states else None, f[1] if actions else None, f[2] if returns else None,
                          f[3] if old else None, f[4] if idx else None, n, clip, None if nt is None else C.byref(nt),
                          f[5] if stats else None, None)


def test_argument_checks_come_before_any_cuda_call(L):
    def rejected(rc, what):
        assert rc == -1, (rc, what)
        assert what in L.mm_last_error().decode(), (what, L.mm_last_error())

    rejected(_call(L, 3), "kind")
    rejected(_call(L, -1), "kind")
    rejected(_call(L, 0, n=-1), "n must be >= 0")
    rejected(_call(L, 0, net=None), "net")
    rejected(_call(L, 2, net=_net(0)), "w4")
    rejected(_call(L, 0, stats=False), "stats")
    rejected(_call(L, 0, n=0, stats=False), "stats")
    for k in (0, 1, 2):
        rejected(_call(L, k, states=False), "states")
        rejected(_call(L, k, actions=False), "idx")
        rejected(_call(L, k, idx=False), "idx")
    rejected(_call(L, 1, returns=False), "returns")
    rejected(_call(L, 2, returns=False), "returns")
    for clip in (0.0, 1.0, -0.2, 1.5, float("nan")):
        rejected(_call(L, 0, clip=clip), "clip")
        rejected(_call(L, 2, clip=clip), "clip")


# ---- the restatement against the torch statistics in float64

def _nets(kind, seed):
    from marl_mass_b200 import rollout
    torch.manual_seed(seed)
    return {"actor": rollout.ActorNetwork, "critic": rollout.CriticNetwork, "shared": rollout.ActorCriticNetwork}[kind]().double()


def _case(kind, seed=3, rows=500, n=777):
    rng = np.random.default_rng(seed)
    S = rng.normal(0, 1, (rows, 30))
    A8 = rng.integers(0, 5, rows).astype(np.int8)
    G = rng.normal(0, 3, rows)
    idx = rng.integers(0, rows, n)                       # unsorted, with duplicates
    net = _nets(kind, seed)
    params = {k: p.detach().numpy().copy() for k, p in net.named_parameters()}
    return net, params, S, A8, G, idx


def _torch(net, S, A8, G, idx, old, clip):
    from marl_mass_b200 import rollout
    t = lambda a: None if a is None else torch.from_numpy(np.asarray(a))  # noqa: E731
    return rollout.ppo_stats_torch(net, t(S), t(A8), t(G), t(idx), t(old), clip).numpy()


def _assert_close(got, want, tol=1e-12):
    for k, name in enumerate(ppo_stats_ref.FIELDS):
        if np.isinf(want[k]):
            assert got[k] == want[k], name
        else:
            assert abs(got[k] - want[k]) <= tol * max(1.0, abs(want[k])), (name, got[k], want[k])


@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
def test_restatement_matches_torch_statistics_in_float64(kind):
    """Rows with r == 1, ratios inside and outside the clip range on both sides, and rows exactly at |r - 1| = clip
    (clip is taken from such a row, where both computations form the same r, so it counts as not clipped)."""
    net, params, S, A8, G, idx = _case(kind)
    rows = len(S)
    for old in (None, "ratios"):
        if old is not None and kind != "critic":
            logp = ppo_stats_ref.stat_rows(kind, params, S, A8, G, np.arange(rows))["logp"]
            regime = np.arange(rows) % 4
            old = logp - np.choose(regime, [0.0, 0.5, -0.5, 0.1])
            old[regime == 0] = logp[regime == 0]
            # the clip bound: |r - 1| of a row with r ~ e^0.1 on which the restatement and torch agree bit for bit
            r_ref = ppo_stats_ref.stat_rows(kind, params, S, A8, G, np.arange(rows), old)["ratio"]
            from marl_mass_b200 import rollout
            _, lp_t = rollout._ppo_stats_torch(net, torch.from_numpy(S), torch.from_numpy(A8), torch.from_numpy(G),
                                               torch.arange(rows), None, CLIP)
            r_t = torch.exp(lp_t - torch.from_numpy(old)).numpy()
            at = np.flatnonzero((regime == 3) & (r_ref == r_t) & np.isin(np.arange(rows), idx))
            assert len(at)
            clip = float(abs(r_ref[at[0]] - 1.0))
            on_bound = np.abs(r_ref[idx] - 1.0) == clip
            assert on_bound.sum() >= 1
        else:
            old, clip = None, CLIP
        want = ppo_stats_ref.ppo_stats_ref(kind, params, S, A8, G, idx, old, clip)
        got = _torch(net, S, A8, G, idx, old, clip)
        _assert_close(got, want)
        if old is not None:
            r = ppo_stats_ref.stat_rows(kind, params, S, A8, G, idx, old, clip)["ratio"]
            assert 0 < want[ppo_stats_ref.K["clipped"]] < len(idx)
            assert np.any(r == 1.0) and np.any(r > 1 + clip) and np.any(r < 1 - clip)
        if kind == "critic" or old is None:
            assert got[ppo_stats_ref.K["ratio_min"]] == np.inf and got[ppo_stats_ref.K["ratio_max"]] == -np.inf
        if kind == "actor":
            assert np.all(got[ppo_stats_ref.K["v"]:] == 0)
        if kind == "critic":
            assert np.all(got[1:4] == 0)


def test_empty_index_list_gives_the_empty_vector():
    net, params, S, A8, G, _ = _case("shared")
    idx = np.zeros(0, np.int64)
    got = _torch(net, S, A8, G, idx, np.zeros(len(S)), CLIP)
    want = ppo_stats_ref.ppo_stats_ref("shared", params, S, A8, G, idx, np.zeros(len(S)), CLIP)
    assert np.array_equal(got, want)
    assert got[4] == np.inf and got[5] == -np.inf and not np.any(got[[0, 1, 2, 3, 6, 7, 8, 9, 10]])


def test_keys_from_the_vectors_match_direct_formulas():
    from marl_mass_b200 import rollout
    net, params, S, A8, G, idx = _case("shared", seed=9)
    St, At, Gt, jt = torch.from_numpy(S), torch.from_numpy(A8), torch.from_numpy(G), torch.from_numpy(idx)
    before, logp = rollout._ppo_stats_torch(net, St, At, Gt, jt, None, CLIP)
    old = torch.zeros(len(S), dtype=torch.float64)
    old[jt] = logp - 0.3 * torch.sin(torch.arange(len(idx), dtype=torch.float64))
    after = rollout.ppo_stats_torch(net, St, At, Gt, jt, old, CLIP)
    keys = rollout.ppo_stats_keys(before.tolist(), after.tolist())
    with torch.no_grad():
        h = net.trunk(St[jt])
        lp, v, g = net.policy_head(h), net.critic_linear(h)[:, 0], Gt[jt]
        lr = (lp * torch.nn.functional.one_hot(At[jt].long(), 5)).sum(1) - old[jt]
        r = lr.exp()
    adv = g - v
    want = {"approx_kl": float(((r - 1) - lr).mean()), "clip_fraction": float(((r - 1).abs() > CLIP).double().mean()),
            "ratio_min": float(r.min()), "ratio_max": float(r.max()),
            "entropy_before": float(-(lp.exp() * lp).sum(1).mean()), "entropy_after": float(-(lp.exp() * lp).sum(1).mean()),
            "explained_variance_before": float(1 - adv.var(unbiased=False) / g.var(unbiased=False)),
            "explained_variance_after": float(1 - adv.var(unbiased=False) / g.var(unbiased=False)),
            "advantage_mean": float(adv.mean()), "advantage_std": float(adv.std(unbiased=False))}
    assert set(keys) == set(want)
    for k, w in want.items():
        assert abs(keys[k] - w) <= 1e-10 * max(1.0, abs(w)), (k, keys[k], w)
    assert 0 < keys["clip_fraction"] < 1 and keys["approx_kl"] > 0
    assert all(np.isnan(v) for v in rollout.ppo_stats_keys([0.0] * 11, [0.0] * 11).values())


def test_train_refuses_bad_update_stats_after_the_existing_refusals(tmp_path):
    from marl_mass_b200.train import train
    for bad in ("yes", 1, None):
        with pytest.raises(ValueError, match="update_stats"):
            train(INI, n_envs=4, iterations=1, update_stats=bad)
    with pytest.raises(ValueError, match="update_stats"):
        train(INI, n_envs=4, iterations=1, update_stats=True, update_impl="jax")
    with pytest.raises(ValueError, match="eval_seeds"):         # the refusals that were there first still come first
        train(INI, n_envs=4, iterations=1, eval_seeds=0, eval_shield=True, update_stats="yes")
    v0 = tmp_path / "v0.ini"
    v0.write_text(re.sub(r"(?m)^env_name\s*=.*$", "env_name = merge-multi-agent-v0", open(INI).read())
                  if re.search(r"(?m)^env_name\s*=", open(INI).read())
                  else open(INI).read().replace("[ENV_CONFIG]", "[ENV_CONFIG]\nenv_name = merge-multi-agent-v0"))
    with pytest.raises(ValueError, match="env id"):
        train(str(v0), n_envs=4, iterations=1, update_stats="yes")

"""GPU suite: the CUDA path, called through the C ABI, against (a) the golden vectors frozen from the reference
and (b) the CPU oracle on seeded scenes.  Discrete outputs bit-exact; continuous state <= 1e-9 relative
(float64 core; the north-star tolerance is 1e-4), float32 outputs (obs, rewards) <= 2e-6.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN_CASES, HDV_TIE_CASES, SUPERVISED_CASES, TIE_CASES, V0_CASES, V0_TIE_CASES
from helpers import (ENV_FIELDS, F64_FIELDS, I32_FIELDS, LC_BOUNDARY_EPS, OUT_F, OUT_I, SH_F, SH_I, compare_states,
                     load_golden, obs25, rel_err, used_mask)

pytestmark = pytest.mark.gpu

STATE_TOL = 1e-9
F32_TOL = 2e-6


@pytest.fixture(scope="module")
def mm():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import marl_mass_b200 as m
    m.lib()  # raises if the sm_100a library was not built: there is no fallback to test
    return m


@pytest.fixture(scope="module")
def orc():
    import oracle
    oracle.lib()
    return oracle


def env_config(cfg):
    keys = ("simulation_frequency", "policy_frequency", "duration", "COLLISION_REWARD", "HIGH_SPEED_REWARD",
            "HEADWAY_COST", "HEADWAY_TIME", "MERGING_LANE_COST", "traffic_density", "safety_guarantee",
            "traffic_type", "agent_reward", "cbf_eta", "env_name", "mixed_traffic", "lateral_control")
    return {k: cfg[k] for k in keys}


def full_state(orc, g, rows):
    return orc.state_from_golden(g, rows)


def outputs_to_numpy(v, keys):
    import torch
    torch.cuda.synchronize()
    return {k: v[k].cpu().numpy() for k in keys}


def check_outputs(got, want, ncav):
    m = np.arange(12)[None, :] < ncav[:, None]
    for k in OUT_I:
        assert np.array_equal(got[k].astype(np.int32) * (m if got[k].ndim == 2 else 1),
                              np.asarray(want[k], np.int32)), k
    for k in OUT_F:
        assert rel_err(got[k], want[k]).max() <= F32_TOL, (k, rel_err(got[k], want[k]).max())


def check_shield(diag, want, lc_margin, tol=None):
    tol = STATE_TOL if tol is None else tol
    ran = want["sh_ran"] == 1
    assert np.array_equal(diag["ran"], want["sh_ran"])
    boundary = ran & (lc_margin < LC_BOUNDARY_EPS)
    for k in SH_I:
        bad = (diag[k] != want["sh_" + k]) & ran & ~boundary
        assert not bad.any(), (k, np.argwhere(bad)[:5].tolist())
    for k in SH_F:
        assert (rel_err(diag[k], want["sh_" + k]) * (ran & ~boundary)).max() <= tol, k
    return int(boundary.sum())


@pytest.mark.parametrize("name", GOLDEN_CASES + TIE_CASES)
def test_cuda_vs_golden_teacher_forced(mm, orc, name):
    """Reference pre-state + reference actions -> CUDA step -> reference post-state, outputs, shield record.
    The TIE_CASES hold exact ties in x / s / |ds| (positions and speeds snapped to integers): the x-ordered walks
    must detect them and reproduce the reference's stable-sort and "<=" tie rules through their exhaustive scans."""
    g, cfg = load_golden(name)
    rows = g["row_of_step"]
    T = len(rows)
    env = mm.MergeEnvBatched(T, env_config(cfg), record_diag=True)
    env.set_state(full_state(orc, g, rows))
    import torch
    act = torch.from_numpy(np.ascontiguousarray(g["act"])).cuda()
    _, _, _, v = env.step(act)
    got = outputs_to_numpy(v, OUT_F + OUT_I)
    if cfg["n_s"] == 25:
        got["obs"] = obs25(got["obs"])
    # per-agent action availability (abstract.py:219-240) against the reference's own _get_available_actions
    assert np.array_equal(v["action_mask"].cpu().numpy().astype(np.int32), g["avail_bits"])
    post = env.get_state()
    diag = env.shield_diag()
    # DESIGN.md "Veto tie rule": steps on which the reference's rounding noise put an exactly-zero veto test on the
    # other side leave the state / output comparison (their lane change is cancelled or not); next to none exist
    flipped = ((g["sh_ran"] == 1) & (diag["lc_margin"] < LC_BOUNDARY_EPS) &
               (diag["is_lc_safe"] != g["sh_is_lc_safe"])).any(axis=(1, 2))
    assert flipped.sum() <= 1, np.where(flipped)[0]
    keep = np.where(~flipped)[0]
    sub = lambda d: {k: d[k][keep] for k in d}
    compare_states(sub(post), sub(full_state(orc, g, rows + 1)), STATE_TOL, name)
    check_outputs(sub(got), {k: g[k][keep] for k in OUT_F + OUT_I}, g["st_n_cav"][rows][keep])
    nb = check_shield(diag, {k: g[k] for k in g.files if k.startswith("sh_")}, diag["lc_margin"])
    assert nb <= 0.01 * max(int((g["sh_ran"] == 1).sum()), 1) + 1
    env.close()


@pytest.mark.parametrize("name", ["hss_td3", "mass_td3_mixed", "unsafe_td2_mixed", "steervel_hss_td3_mixed"])
def test_cuda_free_running_episode(mm, orc, name):
    """Whole episodes on the GPU alone (state never re-synced) end on the reference's final state."""
    import torch
    g, cfg = load_golden(name)
    ep, rows = g["ep_start"], g["row_of_step"]
    n_ep = len(ep) - 1
    env = mm.MergeEnvBatched(n_ep, env_config(cfg))
    env.set_state(full_state(orc, g, ep[:-1]))
    lens = [int(((rows >= ep[j]) & (rows < ep[j + 1] - 1)).sum()) for j in range(n_ep)]
    first_step = [int(np.where(rows == ep[j])[0][0]) for j in range(n_ep)]
    finals = {}
    for t in range(max(lens)):
        a = np.ones((n_ep, 12), np.int8)
        for j in range(n_ep):
            if t < lens[j]:
                a[j] = g["act"][first_step[j] + t]
        _, _, done, v = env.step(torch.from_numpy(a).cuda())
        d = done.cpu().numpy()
        st = env.get_state()
        for j in range(n_ep):
            if t < lens[j]:
                assert int(d[j]) == int(g["done"][first_step[j] + t]), (name, j, t)
                if t == lens[j] - 1:
                    finals[j] = {k: st[k][j:j + 1].copy() for k in st}
    for j in range(n_ep):
        compare_states(finals[j], full_state(orc, g, [ep[j + 1] - 1]), 1e-6, "%s episode %d" % (name, j))
    env.close()


@pytest.mark.parametrize("shield,traffic,td,reward", [
    ("cbf-cav", "cav", 3, "default"), ("cbf-cav", "mixed", 3, "srew"), ("cbf-avs_cint", "cav", 3, "default"),
    ("cbf-avs_cint", "mixed", 2, "mrew"), ("none", "mixed", 1, "default"), ("cbf-cav", "cav", 1, "mrew"),
    ("cbf-cav+steer_vel", "mixed", 3, "default")])
def test_cuda_vs_oracle_seeded_rollout(mm, orc, shield, traffic, td, reward):
    """4096 device-spawned scenes, 40 policy steps of uniform random actions, CUDA and oracle advanced in lock
    step from the same start; state is re-synced from the oracle only when a discrete mismatch was excluded as
    a veto-boundary case (never observed so far)."""
    lockstep_rollout(mm, orc, shield, traffic, td, reward, 4096, 40, STATE_TOL)


@pytest.mark.parametrize("shield,traffic,td,reward", [
    ("cbf-cav", "cav", 3, "default"), ("cbf-cav", "mixed", 3, "srew"), ("cbf-avs_cint", "mixed", 2, "default")])
def test_cuda_vs_oracle_whole_episodes(mm, orc, shield, traffic, td, reward):
    """The same lock-step comparison over the WHOLE 100-step episode (queues behind the obstacle, everybody on cd0, the
    one-sub-step last policy step, terminal outputs): the late-episode states are where the x-sorted neighbour walks,
    the close-pair collision mask and the lane-change veto path do most of their work.  Neither side is re-synced, so
    the libm-level differences between the two float64 implementations compound over 300 sub-steps: continuous state
    within 1e-6 (as for the free-running golden episodes), every discrete field, output and shield record still exact.
    Envs drop out of the comparison when one of their vehicles comes (nearly) to a halt - see lockstep_rollout."""
    lockstep_rollout(mm, orc, shield, traffic, td, reward, 2048, 100, 1e-6)


@pytest.mark.parametrize("shield,traffic,td,reward", [("cbf-cav", "cav", 3, "default"), ("cbf-avs_cint", "mixed", 3, "srew")])
def test_four_ctas_per_sm_build_of_the_step_kernel(mm, orc, shield, traffic, td, reward):
    """The 4-CTAs-per-SM build (4 staged fields, 128 registers; chosen automatically for grids that then fit one wave)
    computes the same step: the strict lock-step comparison with that build forced."""
    try:
        mm.set_step_variant(4)
        lockstep_rollout(mm, orc, shield, traffic, td, reward, 4096, 40, STATE_TOL, expect_build=(4,))
    finally:
        mm.set_step_variant(0)


@pytest.mark.parametrize("shield,variant,build", [("cbf-cav", 3, 3), ("cbf-avs_cint", 3, 3), ("cbf-cav", 5, 3),
                                                  ("cbf-cav", 8, 32), ("cbf-avs_cint", 8, 31), ("cbf-cav", 6, 42),
                                                  ("cbf-avs_cint", 6, 41)])
def test_thread_per_env_builds_on_all_cav_scenes(mm, orc, shield, variant, build):
    """All-CAV scenes under MASS / HSS have five builds of the step kernel to choose from; at this batch size the
    automatic choice is the warp-cooperative one (asserted in lockstep_rollout).  The one-thread-per-env builds must
    compute the same step: the strict lock-step comparison with each forced - generic (3; 5: automatic among the generic
    builds), compile-time specialised for 3 CTAs per SM (8: automatic among the thread-per-env builds -> 31 HSS, 32 MASS)
    and for 4 CTAs per SM (6 -> 41, 42)."""
    try:
        mm.set_step_variant(variant)
        lockstep_rollout(mm, orc, shield, "cav", 3, "default", 4096, 40, STATE_TOL, expect_build=(build,))
    finally:
        mm.set_step_variant(0)


def test_automatic_build_choice_follows_the_batch_size(mm):
    """mm_step_build() after a step: warp-cooperative for a small all-CAV batch, specialised one-thread-per-env builds for
    larger ones (4 CTAs per SM where the wave structure favours it), generic when HDVs can be present."""
    import torch
    want = {(4096, "cav"): (52,), (65536, "cav"): (42,), (200000, "cav"): (32, 42), (4096, "mixed"): (3, 4)}
    for (E, traffic), builds in want.items():
        cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_type=traffic, traffic_density=3, HEADWAY_TIME=0.5,
                   cbf_eta=0.03125)
        env = mm.MergeEnvBatched(E, cfg)
        env.reset(seed=1)
        env.step(torch.ones((E, 12), dtype=torch.int8, device="cuda"))
        torch.cuda.synchronize()
        assert env.step_build() in builds, (E, traffic, env.step_build())
        env.close()


@pytest.mark.parametrize("shield,td,reward,T,resync", [
    ("cbf-cav", 3, "default", 40, False), ("cbf-avs_cint", 3, "srew", 40, False), ("none", 3, "default", 40, False),
    ("cbf-cav", 1, "mrew", 40, False), ("cbf-cav", 3, "srew", 100, True), ("cbf-avs_cint", 3, "default", 100, True)])
def test_warp_cooperative_build_of_the_step_kernel(mm, orc, shield, td, reward, T, resync):
    """The warp-cooperative build (merge_coop.cu: half a warp per env, one lane per vehicle, parallel neighbour
    classification over per-lane views, fixed-point rounds for the MASS acceleration chain, re-steer fix-ups) computes the
    same policy step as the one-thread-per-env kernel: the strict lock-step comparison with that build forced, free
    running for 40 steps and teacher-forced over the whole 100-step episode."""
    try:
        mm.set_step_variant(7)
        build = {"none": 50, "cbf-avs_cint": 51, "cbf-cav": 52}[shield]
        lockstep_rollout(mm, orc, shield, "cav", td, reward, 4096 if T == 40 else 2048, T, STATE_TOL, resync=resync,
                         expect_build=(build,))
    finally:
        mm.set_step_variant(0)


def test_exact_ties_with_the_warp_cooperative_build(mm, orc):
    try:
        mm.set_step_variant(7)
        tie_rollout(mm, orc, "cbf-cav", "cav", 3, False)
        tie_rollout(mm, orc, "cbf-avs_cint", "cav", 3, True)
    finally:
        mm.set_step_variant(0)


@pytest.mark.parametrize("shield,traffic,td,reward", [
    ("cbf-cav", "cav", 3, "default"), ("cbf-cav", "mixed", 3, "srew"), ("cbf-avs_cint", "mixed", 2, "default")])
def test_teacher_forced_whole_episodes(mm, orc, shield, traffic, td, reward):
    """Strict per-step parity over the WHOLE 100-step episode: after every policy step the device state is re-synced
    from the oracle (teacher forcing), so nothing compounds and nothing needs excluding - the queues behind the
    obstacle, (nearly) stopped vehicles and the terminal step are compared at the strict tolerance like every other
    state: every discrete field, output and shield record exact, continuous state within 1e-9."""
    lockstep_rollout(mm, orc, shield, traffic, td, reward, 2048, 100, STATE_TOL, resync=True)


@pytest.mark.parametrize("shield,traffic,td,snap_y", [("cbf-cav", "cav", 3, False), ("cbf-avs_cint", "mixed", 3, False),
                                                      ("cbf-cav", "mixed", 2, True), ("none", "cav", 3, True)])
def test_cuda_vs_oracle_scenes_with_exact_ties(mm, orc, shield, traffic, td, snap_y):
    """Tie handling at scale: before every policy step the x positions and speeds of 4096 scenes are snapped to
    integers (as in the TIE_CASES fixtures, where the oracle's tie rules are pinned on the reference), so vehicles share
    x / s and the closest-vehicle keys tie on both sides of an ego in most envs.  The x-ordered walks of the kernel must
    fall back to their exhaustive scans exactly there; CUDA and oracle are stepped from the same snapped state.
    snap_y: y on a 0.5 m grid as well (vehicles exactly between bc0 and bc1: the closest-lane argmin ties) and speeds
    on a 2.5 m/s grid (half-way between speed levels: np.round's half-to-even in speed_to_index)."""
    tie_rollout(mm, orc, shield, traffic, td, snap_y)


def test_exact_ties_with_the_four_cta_build(mm, orc):
    try:
        mm.set_step_variant(4)
        tie_rollout(mm, orc, "cbf-cav", "mixed", 3, True)
    finally:
        mm.set_step_variant(0)


@pytest.mark.parametrize("round_index", [0, 2])
def test_soak_round_with_snapped_scenes(round_index):
    """One round of profiles/soak_parity.py inside the suite: the 11 shield / traffic / density / reward / lateral-control
    variants x 1024 fresh scenes x the whole 100-step episode, every scene snapped to grid values before every policy
    step (exact ties in x, s and the closest-vehicle keys, vehicles on lane ends and after_end thresholds, speeds
    half-way between speed levels), compared per step against the oracle: every discrete state field, discrete output
    and non-boundary shield record identical.  Round 0 runs the automatic build choice (specialised builds on the
    all-CAV variants), round 2 forces the warp-cooperative build where it applies."""
    import subprocess
    import sys
    from conftest import ROOT
    p = subprocess.run([sys.executable, os.path.join(ROOT, "profiles", "soak_parity.py"), "1", str(round_index), "snap"],
                       env=dict(os.environ, MM_SOAK_ENVS="1024"), capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "SOAK OK" in p.stdout, (p.stdout[-1500:], p.stderr[-1500:])


def tie_rollout(mm, orc, shield, traffic, td, snap_y=False):
    import torch
    E, T = 4096, 30
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee=shield, traffic_type=traffic, traffic_density=td, HEADWAY_TIME=0.5,
               cbf_eta=0.03125)
    env = mm.MergeEnvBatched(E, cfg, record_diag=True)
    env.reset(seed=4321 + td)
    st = env.get_state()
    ocfg = orc.make_config(cfg)
    rng = np.random.RandomState(11)
    alive = np.ones(E, bool)
    same_x = 0
    for t in range(T):
        um = used_mask(st)
        st["x"] = np.where(um, np.round(st["x"]), st["x"])
        st["speed"] = np.where(um, np.round(st["speed"]), st["speed"])
        if snap_y:
            st["y"] = np.where(um, np.round(st["y"] * 2) / 2, st["y"])
            # 12.5, 17.5, ... m/s: half-way between two speed levels, FASTER / SLOWER round half to even
            st["speed"] = np.where(um, np.round(st["speed"] / 2.5) * 2.5, st["speed"])
        # the newest history record is the current state (log_step after every move): keep that invariant
        h1 = um & (st["hist_len"] >= 1)
        st["rec1_x"] = np.where(h1, st["x"], st["rec1_x"])
        st["rec1_vx"] = np.where(h1, st["speed"] * np.cos(st["heading"]), st["rec1_vx"])
        xs = np.where(um, st["x"], np.arange(12)[None, :] * 1e-3 - 1e6)      # unused slots: distinct dummies
        same_x += int((np.diff(np.sort(xs, axis=1), axis=1) == 0).sum())
        env.set_state(st)
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        want = orc.step(ocfg, st, a, n_threads=8)
        _, _, _, v = env.step(torch.from_numpy(a).cuda())
        got = outputs_to_numpy(v, OUT_F + OUT_I)
        post = env.get_state()
        diag = env.shield_diag()
        sel = np.where(alive)[0]
        sub = lambda d: {k: d[k][sel] for k in d}
        compare_states(sub(post), sub(st), STATE_TOL, "tie step %d" % t)
        check_outputs(sub(got), sub({k: want[k] for k in OUT_F + OUT_I}), st["n_cav"][sel])
        check_shield(sub(diag), sub({k: want[k] for k in want if k.startswith("sh_")}), diag["lc_margin"][sel])
        alive &= want["done"] == 0
    assert same_x > E      # on average more than one shared x per scene over the run
    env.close()


def lockstep_rollout(mm, orc, shield, traffic, td, reward, E, T, state_tol, resync=False, expect_build=None):
    import torch
    lateral = "steer_vel" if shield.endswith("+steer_vel") else "steer"
    shield = shield.split("+")[0]
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee=shield, lateral_control=lateral, traffic_type=traffic, traffic_density=td,
               agent_reward=reward, HEADWAY_TIME=0.5, cbf_eta=0.03125, HIGH_SPEED_REWARD=4, HEADWAY_COST=1,
               MERGING_LANE_COST=8)
    env = mm.MergeEnvBatched(E, cfg, record_diag=True)
    env.reset(seed=1234 + td)
    st = env.get_state()
    ocfg = orc.make_config(cfg)
    obs0 = outputs_to_numpy(env.buffers(), ("obs",))["obs"]
    assert rel_err(obs0, orc.observe(st, steer_vel=(lateral == "steer_vel"))).max() <= F32_TOL
    rng = np.random.RandomState(7)
    alive = np.ones(E, bool)
    clean = np.ones(E, bool)
    n_compared = 0
    worst = 0.0
    for t in range(T):
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        want = orc.step(ocfg, st, a, n_threads=8)
        _, _, _, v = env.step(torch.from_numpy(a).cuda())
        got = outputs_to_numpy(v, OUT_F + OUT_I)
        post = env.get_state()
        diag = env.shield_diag()
        if expect_build is not None:
            assert env.step_build() in expect_build, env.step_build()
        elif traffic == "cav" and lateral == "steer":
            # all-CAV scenes of the plain LC env at this batch size: the warp-cooperative build unless a test forces another
            assert env.step_build() in (50, 51, 52), env.step_build()
        # compare only envs that had not finished before this step (finished envs are not stepped by MAPPO) and, in the
        # whole-episode runs, that are still well conditioned (see below)
        sel = np.where(alive & clean)[0]
        sub = lambda d: {k: d[k][sel] for k in d}
        worst = max(worst, compare_states(sub(post), sub(st), state_tol, "step %d" % t))
        check_outputs(sub(got), sub({k: want[k] for k in OUT_F + OUT_I}), st["n_cav"][sel])
        check_shield(sub(diag), sub({k: want[k] for k in want if k.startswith("sh_")}), diag["lc_margin"][sel], state_tol)
        alive &= want["done"] == 0
        if resync:
            env.set_state(st)       # teacher forcing: the next step starts from the oracle's state on both sides
        if state_tol > STATE_TOL:
            # Free-running whole episodes: the steering law of a (nearly) stopped vehicle divides by not_zero(speed) =
            # +-0.01 twice, i.e. amplifies a 1e-16 difference in its lateral offset by ~1e5 and can flip the sign of the
            # command; harmless while it stands, but when it creeps forward again the two float64 implementations
            # leave on (physically meaningless) different headings.  An env is compared up to the step on which one
            # of its vehicles first drops below 3 m/s (it can then come to a halt within the next policy step);
            # per-step parity of the slow states is what the teacher-forced golden tests pin.
            clean &= ~((st["speed"] < 3.0) & used_mask(st)).any(axis=1)
            n_compared += len(sel)
    if state_tol > STATE_TOL:
        assert n_compared > 0.4 * E * T, n_compared     # a large part of the env-steps of the episode was compared
    if shield == "none":
        assert alive.sum() < E  # unshielded random driving does crash inside the window
    env.close()


def test_diag_off_equals_diag_on(mm):
    """The benchmarked instantiation (no shield record) computes the same step as the tested one."""
    import torch
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, traffic_type="mixed",
               HEADWAY_TIME=0.5, cbf_eta=0.03125)
    E = 2048
    a_env = mm.MergeEnvBatched(E, cfg, record_diag=True)
    b_env = mm.MergeEnvBatched(E, cfg, record_diag=False)
    a_env.reset(seed=5)
    b_env.set_state(a_env.get_state())
    rng = np.random.RandomState(3)
    for t in range(12):
        a = torch.from_numpy(rng.randint(0, 5, size=(E, 12)).astype(np.int8)).cuda()
        a_env.step(a)
        b_env.step(a)
    sa, sb = a_env.get_state(), b_env.get_state()
    for k in F64_FIELDS + I32_FIELDS + ENV_FIELDS:
        assert np.array_equal(sa[k], sb[k]), k
    va, vb = a_env.buffers(), b_env.buffers()
    torch.cuda.synchronize()
    for k in ("obs", "reward", "done", "regional_rewards", "min_headway"):
        assert torch.equal(va[k], vb[k]), k
    a_env.close()
    b_env.close()


def test_host_buffer_step_equals_device_step(mm):
    """mm_step_host (chunked over streams, pinned host buffers) == mm_step on device tensors."""
    import torch
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5, cbf_eta=0.03125)
    E = 40000  # not a multiple of the chunk size: exercises the ragged last chunk
    a_env = mm.MergeEnvBatched(E, cfg)
    b_env = mm.MergeEnvBatched(E, cfg)
    a_env.reset(seed=11)
    b_env.set_state(a_env.get_state())
    rng = np.random.RandomState(5)
    out = b_env.alloc_host_out()
    for t in range(5):
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        obs, rew, done, v = a_env.step(torch.from_numpy(a).cuda())
        b_env.step_host(a, out=out)
        torch.cuda.synchronize()
        assert np.array_equal(obs.cpu().numpy(), out["obs"])
        assert np.array_equal(rew.cpu().numpy(), out["reward"])
        assert np.array_equal(done.cpu().numpy(), out["done"])
        assert np.array_equal(v["regional_rewards"].cpu().numpy(), out["regional_rewards"])
        assert np.array_equal(v["n_agents"].cpu().numpy(), out["n_agents"])
    a_env.close()
    b_env.close()


def test_ragged_host_step_equals_device_step(mm):
    """mm_step_host_ragged: the live rows of every env, packed, == the dense device obs,
    over chunk boundaries (5 chunks of 28 416 envs on a 148-SM B200) with a short last chunk."""
    import torch
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5, cbf_eta=0.03125)
    E = 140001
    a_env = mm.MergeEnvBatched(E, cfg)
    b_env = mm.MergeEnvBatched(E, cfg)
    a_env.reset(seed=12)
    b_env.set_state(a_env.get_state())
    rng = np.random.RandomState(6)
    out = b_env.alloc_host_out(ragged=True)
    for t in range(4):
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        obs, rew, done, v = a_env.step(torch.from_numpy(a).cuda())
        out["obs_rows"][:] = np.nan
        b_env.step_host_ragged(a, out=out)
        torch.cuda.synchronize()
        n = v["n_agents"].cpu().numpy()
        assert np.array_equal(n, out["n_agents"])
        off = out["row_offset"]
        assert off[0] == 0 and off[E] == E * 12 and np.all(np.diff(off[:E]) >= n[:-1])
        dense = obs.cpu().numpy()
        live = np.arange(12)[None, :] < n[:, None]
        rows = (off[:E, None] + np.arange(12)[None, :])[live]
        assert np.array_equal(out["obs_rows"][rows], dense[live])
        assert np.isnan(out["obs_rows"]).all(axis=1).sum() == E * 12 - int(n.sum())   # nothing else was written
        assert np.array_equal(rew.cpu().numpy(), out["reward"])
        assert np.array_equal(done.cpu().numpy(), out["done"])
        assert np.array_equal(v["regional_rewards"].cpu().numpy(), out["regional_rewards"])
    a_env.close()
    b_env.close()


@pytest.mark.parametrize("traffic,lateral,E", [("cav", "steer", 70000), ("mixed", "steer_vel", 3000)])
def test_packed_host_step_expands_to_the_observation_rows(mm, traffic, lateral, E):
    """mm_step_host_packed hands over per-vehicle state + neighbour slots instead of observation rows;
    mm_expand_obs_rows rebuilds the rows on the host.  Two handles stepped with the same actions from the same spawn: the
    rebuilt rows equal the rows of mm_step_host_ragged to float32 rounding of the packed inputs (<= 1e-6 on the [-1, 1]
    scale), counts / reward / done / regional rewards are identical; several chunks (70 000 envs) and auto-reset."""
    import torch
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_type=traffic, traffic_density=3, HEADWAY_TIME=0.5,
               cbf_eta=0.03125, lateral_control=lateral, duration=2)
    a_env, b_env = mm.MergeEnvBatched(E, cfg), mm.MergeEnvBatched(E, cfg)
    a_env.reset(seed=77)
    b_env.reset(seed=77)
    rng = np.random.RandomState(3)
    pk, rg = a_env.alloc_host_out(pinned=True, packed=True), b_env.alloc_host_out(pinned=True, ragged=True)
    n_done = 0
    for t in range(14):
        act = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        a_env.step_host_packed(act, auto_reset=True, out=pk)
        b_env.step_host_ragged(act, auto_reset=True, out=rg)
        assert np.array_equal(pk["n_agents"].astype(np.int32), rg["n_agents"])
        assert np.array_equal(pk["done"], rg["done"]) and np.array_equal(pk["reward"], rg["reward"])
        assert np.array_equal(pk["regional_rewards"], rg["regional_rewards"])
        n_done += int(pk["done"].sum())
        rows, off = a_env.expand_obs_rows(pk, n_threads=4)
        assert off[-1] == rows.shape[0] == int(rg["n_agents"].sum())
        # the ragged path packs its rows per 64 Ki-env chunk; gather them env by env
        want = np.concatenate([rg["obs_rows"][rg["row_offset"][e]:rg["row_offset"][e] + rg["n_agents"][e]] for e in range(0, E, 997)])
        got = np.concatenate([rows[off[e]:off[e + 1]] for e in range(0, E, 997)])
        assert np.abs(got - want).max() <= 1e-6, np.abs(got - want).max()
        st = a_env.get_state()
        assert np.array_equal(pk["n_veh"].astype(np.int32), st["n_veh"])
        e = int(rng.randint(E))
        v0 = int(pk["n_veh"][:e].sum(dtype=np.int64))
        nv = int(st["n_veh"][e])
        assert np.allclose(pk["veh"][v0:v0 + nv, 0], st["x"][e, :nv].astype(np.float32), rtol=0, atol=0)
        assert np.allclose(pk["veh"][v0:v0 + nv, 2], st["heading"][e, :nv].astype(np.float32), rtol=0, atol=0)
        assert np.allclose(pk["veh"][v0:v0 + nv, 3], st["speed"][e, :nv].astype(np.float32), rtol=0, atol=0)
    assert n_done >= E    # every env finished a 10-step episode: re-spawned scenes went through the packed path
    # all-CAV: a fifth of the ragged path's bytes; with HDVs (state rows but no observation rows of their own) under half
    assert a_env.packed_bytes(pk) < (0.3 if traffic == "cav" else 0.5) * (int(rg["n_agents"].sum()) * 120 + E * 61)
    a_env.close()
    b_env.close()


@pytest.mark.parametrize("name", ["hss_td3", "mass_td3_srew", "mass_td1", "steervel_mass_td2", "ties_mass_td3"])
def test_stand_alone_shield_query_matches_the_reference_records(mm, orc, name):
    """mm_shield_query = safety_layer(...) for every CAV against the scene as it is.  The reference evaluates its shields
    front to back inside a sub-step, so its logged record of the FRONT-MOST vehicle in sub-step 0 (nobody has moved yet)
    is exactly such an evaluation (all-CAV fixtures: with HDVs the front-most vehicle is rarely a CAV): on every golden
    step whose front-most vehicle is a shielded CAV, the query - fed the
    nominal action the reference logged - must return the logged safe action, neighbour ids, active set and veto flag.
    The query writes nothing: the state is unchanged afterwards."""
    import torch
    g, cfg = load_golden(name)
    rows = g["row_of_step"]
    st = full_state(orc, g, rows)
    env = mm.MergeEnvBatched(len(rows), env_config(cfg))
    env.set_state(st)
    before = env.get_state()
    xs = np.where(used_mask(st), st["x"], -1e9)
    front = xs.argmax(axis=1)                                   # first maximum = lowest slot on ties, as the stable sort
    idx = np.arange(len(rows))
    ran0 = g["sh_ran"][:, 0, :]
    sel = ran0[idx, front] == 1
    assert sel.sum() > 50, sel.sum()
    nom_steer = np.where(ran0 == 1, g["sh_nom_steer"][:, 0, :], 0.0)
    nom_acc = np.where(ran0 == 1, g["sh_nom_acc"][:, 0, :], 0.0)
    out = env.shield_query(torch.from_numpy(nom_steer).cuda(), torch.from_numpy(nom_acc).cuda())
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in out.items()}
    r, f = idx[sel], front[sel]
    assert np.array_equal(out["ran"][r, f], np.ones(len(r), np.int32))
    for k in ("leader", "front_adj", "rear_adj", "constrain_adj", "active", "is_lc_safe"):
        assert np.array_equal(out[k][r, f], g["sh_" + k][r, 0, f]), k
    assert rel_err(out["safe_acc"][r, f], g["sh_safe_acc"][r, 0, f]).max() <= STATE_TOL
    # steering: a vetoed lane change re-steers towards the own lane only if a lane change is under way, i.e. it reads the
    # target lane - which the reference's act() has already updated for this sub-step when its shield runs, and the
    # fixture's pre-step state has not.  Compared wherever the shield did not veto.
    free = g["sh_is_lc_safe"][r, 0, f] == 1
    assert free.sum() > 30 and rel_err(out["safe_steer"][r, f][free], g["sh_safe_steer"][r, 0, f][free]).max() <= STATE_TOL
    compare_states(env.get_state(), before, 0.0, name + " (query left the state alone)")
    env.close()


def test_checkpoint_resume_continues_bit_identically(mm, tmp_path):
    """save() / load(): a rollout resumed from a checkpoint in a fresh handle continues exactly like the original."""
    import torch
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, traffic_type="mixed", HEADWAY_TIME=0.5,
               cbf_eta=0.03125, agent_reward="mrew")
    E = 3000
    a_env = mm.MergeEnvBatched(E, cfg)
    a_env.reset(seed=21)
    rng = np.random.RandomState(2)
    acts = [torch.from_numpy(rng.randint(0, 5, size=(E, 12)).astype(np.int8)).cuda() for _ in range(30)]
    for t in range(15):
        a_env.step(acts[t])
    path = str(tmp_path / "ckpt.npz")
    a_env.save(path)
    b_env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG))      # default config: load() must bring the stored one
    obs_b, _ = b_env.load(path)
    assert torch.equal(obs_b, a_env.buffers()["obs"])
    for t in range(15, 30):
        oa, ra, da, _ = a_env.step(acts[t])
        ob, rb, db, _ = b_env.step(acts[t])
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)
    sa, sb = a_env.get_state(), b_env.get_state()
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    a_env.close()
    b_env.close()


def test_qp_kernel_vs_golden_and_oracle(mm, orc):
    """mm_shield_qp: every QP the reference posed + 1e6 synthetic ones (oracle as the checker)."""
    import torch
    qs = []
    for name in GOLDEN_CASES:
        g, _ = load_golden(name)
        if len(g["qp_a"]):
            qs.append(np.stack([g["qp_" + k] for k in ("a", "c_lead", "c_adj", "has_adj", "lo", "hi", "u", "active")], 1))
    q = np.concatenate(qs)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    u, act = mm.shield_qp(dev(q[:, 0]), dev(q[:, 1]), dev(q[:, 2]), dev(q[:, 3].astype(np.uint8)), dev(q[:, 4]), dev(q[:, 5]))
    assert np.array_equal(u.cpu().numpy(), q[:, 6])
    assert np.array_equal(act.cpu().numpy(), q[:, 7].astype(np.uint8))
    rng = np.random.RandomState(0)
    n = 1 << 20
    dt = 1 / 15
    a = dt * np.cos(rng.uniform(-0.3, 0.3, n)) * rng.choice([1.0, 1.0, 1.0, -1.0, 0.0], n)
    c_lead, c_adj = rng.normal(0.1, 0.2, n), rng.normal(0.1, 0.2, n)
    has_adj = (rng.rand(n) < 0.3).astype(np.uint8)
    lo = -12.5 * dt + rng.uniform(-0.5, 0.5, n)
    hi = lo + rng.uniform(0, 1.5, n)
    u, act = mm.shield_qp(dev(a), dev(c_lead), dev(c_adj), dev(has_adj), dev(lo), dev(hi))
    u, act = u.cpu().numpy(), act.cpu().numpy()
    for i in rng.choice(n, 4000, replace=False):
        wu, wa = orc.qp(a[i], c_lead[i], c_adj[i], bool(has_adj[i]), lo[i], hi[i])
        assert u[i] == wu and act[i] == wa, i
    assert len(np.unique(act)) >= 8


def test_device_spawn_law(mm):
    """reset(): the device-side spawn follows merge_env_v1.py:180-211,265-364 (counts, slots, noise, speeds)."""
    for td, traffic, cav_rng, hdv_rng in ((1, "cav", (2, 6), (0, 0)), (3, "cav", (7, 11), (0, 0)),
                                          (3, "mixed", (4, 6), (3, 5)), (2, "mixed", (2, 4), (2, 4))):
        E = 20000
        env = mm.MergeEnvBatched(E, dict(mm.DEFAULT_CONFIG, traffic_density=td, traffic_type=traffic))
        env.reset(seed=td)
        st = env.get_state()
        ncav, nhdv = st["n_cav"], st["n_veh"] - st["n_cav"]
        assert ncav.min() == cav_rng[0] and ncav.max() == cav_rng[1]
        assert nhdv.min() == hdv_rng[0] and nhdv.max() == hdv_rng[1]
        m = used_mask(st)
        assert (st["kind"][m] > 0).all() and (st["kind"][~m] == 0).all()
        sp = st["speed"][m]
        assert sp.min() >= 25 and sp.max() < 27 and abs(sp.mean() - 26) < 0.02
        main = m & (st["y"] == 0.0)
        ramp = m & (st["y"] == 10.5)
        assert (main | ramp)[m].all()
        for sel, base in ((main, 10.0), (ramp, 5.0)):
            x = st["x"][sel]
            slot = np.round((x - base) / 50.0)
            noise = x - base - 50.0 * slot
            assert slot.min() == 0 and slot.max() == 5 and np.abs(noise).max() <= 4.0
            assert abs(noise.mean()) < 0.05 and abs(noise.std() - 8 / np.sqrt(12)) < 0.05
        # no slot is used twice within an env
        key = np.where(main, np.round((st["x"] - 10.0) / 50.0), np.where(ramp, 10 + np.round((st["x"] - 5.0) / 50.0), -1))
        for e in range(0, E, 97):
            k = key[e][m[e]]
            assert len(np.unique(k)) == len(k)
        # n_merge = CAVs spawned on the ramp; CAV split follows num_CAV // 2
        cav = np.arange(12)[None, :] < ncav[:, None]
        assert np.array_equal((cav & ramp).sum(1), st["n_merge"])
        assert np.array_equal((cav & main).sum(1)[ncav != 1], (ncav // 2)[ncav != 1])
        assert (st["target_speed"][cav] == 25.0).all() and (st["speed_index"][cav] == 3).all()
        assert (st["min_headway"][cav] == 4.5).all() and (st["hist_len"][m] == 0).all()
        hd = m & ~cav
        if hd.any():
            assert np.array_equal(st["target_speed"][hd], st["speed"][hd])
            assert np.allclose(st["timer"][hd], ((st["x"][hd] + st["y"][hd]) * np.pi) % 1.0, atol=1e-12)
        env.close()


def test_coupled_vehicle_counts_keep_the_law_and_share_counts_per_tile(mm):
    """couple_vehicle_counts (opt-in device spawn): the envs of a 128-env tile share (n_CAV, n_HDV); the counts are
    still uniform over the reference's ranges across tiles, everything else is drawn per env; the step path is the
    same kernel (parity is covered by the other tests: set_state does not care how a scene was drawn)."""
    import torch
    E = 128 * 600
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, traffic_type="mixed", HEADWAY_TIME=0.5,
               cbf_eta=0.03125, couple_vehicle_counts=True)
    env = mm.MergeEnvBatched(E, cfg)
    env.reset(seed=3)
    st = env.get_state()
    n_cav, n_veh = st["n_cav"].reshape(600, 128), st["n_veh"].reshape(600, 128)
    assert (n_cav == n_cav[:, :1]).all() and (n_veh == n_veh[:, :1]).all()
    assert set(np.unique(n_cav)) == {4, 5, 6} and set(np.unique(n_veh - n_cav)) == {3, 4, 5}
    for k in (4, 5, 6):
        assert abs((n_cav[:, 0] == k).mean() - 1 / 3) < 0.08
    x = st["x"].reshape(600, 128, 12)
    assert np.unique(np.round(x[:, :, 0], 6)).size > 0.9 * E          # positions are per env
    # a few steps with auto-reset run fine and the next episode draws new shared counts
    a = torch.ones((E, 12), dtype=torch.int8, device="cuda")
    for _ in range(101):
        env.step(a, auto_reset=True)
    st2 = env.get_state()
    n2 = st2["n_cav"].reshape(600, 128)
    same_tile = (n2 == n2[:, :1]).all(axis=1)
    assert same_tile.mean() > 0.95 and (n2[:, 0] != n_cav[:, 0]).mean() > 0.4
    env.close()


def test_full_size_properties(mm):
    """BASELINE size (65536 envs, MASS td3): size-independent invariants of a 100-step auto-reset rollout."""
    import torch
    E = 65536
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5, cbf_eta=0.03125,
               agent_reward="srew", HIGH_SPEED_REWARD=4, HEADWAY_COST=1, MERGING_LANE_COST=8)
    env = mm.MergeEnvBatched(E, cfg)
    obs, _ = env.reset(seed=99)
    gen = torch.Generator(device="cuda").manual_seed(0)
    episodes = 0
    for t in range(101):
        a = torch.randint(0, 5, (E, 12), generator=gen, device="cuda", dtype=torch.int8)
        obs, rew, done, v = env.step(a, auto_reset=True)
        assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
        n = v["n_agents"]
        assert int(n.min()) >= 7 and int(n.max()) <= 11
        present = obs[:, :, 0]
        idx = torch.arange(12, device="cuda")[None, :]
        assert torch.equal(present > 0, idx < n[:, None])          # ego rows present exactly for live agents
        assert torch.equal(v["agents_dones"].amax(1) > 0, done > 0)
        episodes += int(done.sum())
        if t < 99:
            assert int(done.sum()) <= E // 20                      # shielded: crashes are rare before the horizon
    s = env.stats()
    assert s["episodes"] == episodes and s["env_steps"] == 101 * E
    assert episodes >= E  # every env hit the 100-step horizon once
    # steps restarted at 0 for finished envs
    st = env.get_state()
    assert st["steps"].max() <= 100 and (st["steps"] <= 1).sum() >= E * 0.9
    env.close()


def test_batched_mappo_rollout(mm):
    """BASELINE configs[3] data flow on a small batch: policy + env on device, returns, one PPO update."""
    import torch
    from marl_mass_b200.rollout import BatchedMAPPORollout
    torch.manual_seed(0)
    E, T = 2048, 25
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav", traffic_density=3, HEADWAY_TIME=0.5, cbf_eta=0.03125,
               agent_reward="srew", HIGH_SPEED_REWARD=4, HEADWAY_COST=1, MERGING_LANE_COST=8)
    env = mm.MergeEnvBatched(E, cfg)
    ro = BatchedMAPPORollout(env, roll_out_n_steps=T)
    env.reset(seed=3)
    env.stats(reset=True)
    ro.obs = env.buffers()["obs"]
    b = ro.collect()
    assert b["states"].shape == (T, E, 12, 30) and b["returns"].shape == (T, E, 12)
    assert torch.isfinite(b["returns"]).all()
    s = env.stats()
    assert int(b["live"].sum()) == int(s["agent_steps"])          # every live (env, agent, t) sample is one agent-step
    assert set(torch.unique(b["actions"]).tolist()) <= {0, 1, 2, 3, 4}
    # terminal steps cut the return: R_t == r_t there
    term = b["dones"] > 0
    if term.any():
        t_idx, e_idx = term.nonzero(as_tuple=True)
        assert torch.allclose(b["returns"][t_idx, e_idx], b["rewards"][t_idx, e_idx])
    before = [p.detach().clone() for p in ro.actor.parameters()]
    st = ro.update(minibatch=1 << 16)
    assert st["samples"] == int(b["live"].sum()) and np.isfinite(st["actor_loss"]) and np.isfinite(st["critic_loss"])
    assert any(not torch.equal(a, p) for a, p in zip(before, ro.actor.parameters()))
    env.close()


@pytest.mark.parametrize("name", ["mass_td1", "hss_td3_mixed", "unsafe_td1", "steervel_mass_td2", "v05_steervel_unsafe_td1"])
def test_single_env_adapter_replays_reference_episodes(mm, name):
    """Drop-in surface: make(...).reset(is_training=False, testing_seeds=s) / step(tuple) reproduce what the
    reference returned for the same seeds and actions, for whole episodes (obs, reward, done, info)."""
    g, cfg = load_golden(name)
    ep, rows = g["ep_start"], g["row_of_step"]
    env = mm.make(cfg["env_name"], config=env_config(cfg))
    assert env.n_s == cfg["n_s"] and env.n_a == 5 and env.T == 100
    for j, seed in enumerate(cfg["seeds"]):
        obs, mask = env.reset(is_training=False, testing_seeds=seed)
        n = int(g["st_n_cav"][ep[j]])
        assert obs.shape == (n, cfg["n_s"]) and mask.shape == (n, 5) and mask.all()
        assert len(env.controlled_vehicles) == n
        steps = np.where((rows >= ep[j]) & (rows < ep[j + 1] - 1))[0]
        # reset observation == the reference's first observation (oracle-free: golden obs of step 0 is post-step,
        # so check the ego rows against the golden pre-state instead)
        assert np.allclose((obs[:, 1] + 1) * 150 - 150, g["st_x"][ep[j], :n], atol=1e-3)
        done = False
        for t in steps:
            assert not done
            a = tuple(int(x) for x in g["act"][t, :n])
            obs, reward, done, info = env.step(a)
            assert rel_err(obs, g["obs"][t, :n]).max() <= 1e-5
            assert abs(reward - g["reward"][t]) <= 1e-5 * max(1, abs(g["reward"][t]))
            assert done == bool(g["done"][t])
            assert rel_err(info["regional_rewards"], g["regional_rewards"][t, :n]).max() <= 1e-5
            assert rel_err(info["agents_rewards"], g["agents_rewards"][t, :n]).max() <= 1e-5
            assert list(info["agents_dones"]) == [bool(x) for x in g["agents_dones"][t, :n]]
            assert abs(info["average_speed"] - g["average_speed"][t]) <= 1e-4
            assert abs(info["traffic_speed"] - g["traffic_speed"][t]) <= 1e-4
            assert abs(info["min_headway"] - g["min_headway"][t]) <= 1e-4 * max(1, abs(g["min_headway"][t]))
            assert info["vehicle_speed"].shape == (t - steps[0] + 1, n)
        assert done and "merge_percent" in info
        assert abs(info["merge_percent"] - g["merge_percent"][steps[-1]]) <= 1e-3
        assert env.is_crashed() == bool(g["st_crashed"][ep[j + 1] - 1, :n].any())
    env.close()


def test_control_profiles_of_the_adapter(mm):
    """store_profile: env.road.vehicles[i].state_hist / action_hist (safe_controller.py:187-227) after a replayed
    reference episode - one record per vehicle and sub-step, the last record of a policy step equal to the golden
    post-step state, the shielded action equal to the golden shield record."""
    g, cfg = load_golden("mass_td3_mixed")
    ep, rows = g["ep_start"], g["row_of_step"]
    env = mm.make(cfg["env_name"], config=dict(env_config(cfg), store_profile=True))
    seed = cfg["seeds"][0]
    env.reset(is_training=False, testing_seeds=seed)
    n_veh = int(g["st_n_veh"][ep[0]])
    assert len(env.road.vehicles) == n_veh and [v.id for v in env.road.vehicles] == list(range(n_veh))
    steps = np.where((rows >= ep[0]) & (rows < ep[1] - 1))[0]
    n = len(env.controlled_vehicles)
    subs_total = 0
    for t in steps:
        env.step(tuple(int(x) for x in g["act"][t, :n]))
        post = rows[t] + 1
        n_sub = int(g["st_time"][post] - g["st_time"][rows[t]])          # 3, or fewer on a terminal step
        subs_total += n_sub
        for i, v in enumerate(env.road.vehicles):
            assert len(v.state_hist) == subs_total and len(v.action_hist) == subs_total
            last = v.state_hist[-1]
            # (free-running replay of a whole episode: the tolerance of the other adapter tests, not the teacher-forced one)
            assert abs(last["x"] - g["st_x"][post, i]) <= 1e-5 * max(1, abs(g["st_x"][post, i]))
            assert abs(last["y"] - g["st_y"][post, i]) <= 1e-5 and abs(last["heading"] - g["st_heading"][post, i]) <= 1e-5
            # the record is taken before the collision pass: a crash in this sub-step changes the speed afterwards
            if not g["st_crashed"][post, i]:
                assert abs(last["speed"] - g["st_speed"][post, i]) <= 1e-5 * max(1, g["st_speed"][post, i])
            assert abs(last["t_step"] - subs_total / 15) < 1e-9
            for sub in range(n_sub):
                a = v.action_hist[subs_total - n_sub + sub]
                if g["sh_ran"][t, sub, i]:
                    assert abs(a["acceleration"] - g["sh_safe_acc"][t, sub, i]) <= 1e-4 * max(1, abs(g["sh_safe_acc"][t, sub, i]))
                    assert abs(a["ull_acceleration"] - g["sh_nom_acc"][t, sub, i]) <= 1e-4 * max(1, abs(g["sh_nom_acc"][t, sub, i]))
                    assert "safe_diff" in a
                else:
                    assert a["acceleration"] == a["ull_acceleration"] and "safe_diff" not in a
    assert subs_total == int(g["st_time"][ep[1] - 1])
    env.close()


@pytest.mark.parametrize("name", ["hdv_td3"] + HDV_TIE_CASES)
def test_hdv_env_cuda_vs_golden_and_adapter(mm, orc, name):
    """merge-multi-agent-hdv-v1 (MergeEnvLCHDV, traffic_type = hdv): teacher-forced CUDA step vs the reference's states
    and outputs (one observation row / reward term per vehicle), then whole episodes through make(...)."""
    import torch
    g, cfg = load_golden(name)
    rows = g["row_of_step"]
    T = len(rows)
    env = mm.MergeEnvBatched(T, env_config(cfg), record_diag=True)
    st = full_state(orc, g, rows)
    env.set_state(st)
    nv = st["n_veh"]
    m = np.arange(12)[None, :] < nv[:, None]
    v = env.buffers()
    assert np.array_equal(v["n_agents"].cpu().numpy(), nv)                       # every vehicle is "observed"
    obs, rew, done, v = env.step(torch.from_numpy(np.ascontiguousarray(g["act"])).cuda())
    torch.cuda.synchronize()
    compare_states(env.get_state(), full_state(orc, g, rows + 1), STATE_TOL, "hdv teacher-forced")
    assert np.array_equal(done.cpu().numpy(), g["done"])
    assert rel_err(obs.cpu().numpy(), g["obs"]).max() <= F32_TOL and (obs.cpu().numpy()[~m] == 0).all()
    for k in ("reward", "average_speed", "traffic_speed", "min_headway", "merge_percent", "agents_rewards"):
        assert rel_err(v[k].cpu().numpy(), g[k]).max() <= F32_TOL, k
    assert (v["regional_rewards"] == 0).all() and (v["agents_dones"] == 0).all()
    assert (env.shield_diag()["ran"] == 0).all()
    env.close()
    if name in HDV_TIE_CASES:       # snapped before every step: no episode to replay
        return
    # adapter: whole episodes
    single = mm.make("merge-multi-agent-hdv-v1", config=env_config(cfg))
    ep = g["ep_start"]
    for j, seed in enumerate(cfg["seeds"]):
        obs, mask = single.reset(is_training=False, testing_seeds=seed)
        n = int(g["st_n_veh"][ep[j]])
        assert obs.shape == (n, 30) and len(single.controlled_vehicles) == 0 and len(single.road.vehicles) == n
        steps = np.where((rows >= ep[j]) & (rows < ep[j + 1] - 1))[0]
        for t in steps:
            obs, reward, done, info = single.step(())
            assert rel_err(obs, g["obs"][t, :n]).max() <= 1e-5
            assert abs(reward - g["reward"][t]) <= 1e-5 and done == bool(g["done"][t])
            assert abs(info["average_speed"] - g["average_speed"][t]) <= 1e-4
            assert abs(info["min_headway"] - g["min_headway"][t]) <= 1e-4 * max(1, abs(g["min_headway"][t]))
        assert done and info["merge_percent"] == 100.0 and not single.is_crashed()
    single.close()


def test_masked_reset_stats_and_errors(mm, orc):
    import torch
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-avs_cint", traffic_density=2, traffic_type="mixed",
               HEADWAY_TIME=0.5, cbf_eta=0.03125)
    E = 1000  # not a multiple of the 128-env tile
    env = mm.MergeEnvBatched(E, cfg, record_diag=True)
    env.reset(seed=1)
    before = env.get_state()
    mask = torch.zeros(E, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    env.reset(seed=2, mask=mask)
    after = env.get_state()
    m = mask.cpu().numpy().astype(bool)
    assert np.array_equal(before["x"][~m], after["x"][~m]) and not np.array_equal(before["x"][m], after["x"][m])
    # statistics == what the oracle counts on the same rollout
    env.stats(reset=True)
    st = env.get_state()
    ocfg = orc.make_config(cfg)
    rng = np.random.RandomState(1)
    agent_steps = solves = active = vetoes = 0
    for t in range(5):
        a = rng.randint(0, 5, size=(E, 12)).astype(np.int8)
        agent_steps += int(st["n_cav"].sum())
        want = orc.step(ocfg, st, a, n_threads=4)
        ran = want["sh_ran"] == 1
        solves += int(ran.sum()); active += int((want["sh_active"][ran] != 0).sum())
        vetoes += int((want["sh_is_lc_safe"][ran] == 0).sum())
        env.step(torch.from_numpy(a).cuda())
    s = env.stats()
    assert (s["agent_steps"], s["env_steps"], s["shield_solves"], s["shield_active"], s["lane_change_vetoes"]) == \
           (agent_steps, 5 * E, solves, active, vetoes)
    # error behaviour of the C ABI: status + message, never a crash
    with pytest.raises(mm.MMError, match="num_cav"):
        env.reset(num_CAV=12)
    bad = env.get_state()
    bad["kind"][0, 0] = 2
    with pytest.raises(mm.MMError, match="CAVs"):
        env.set_state(bad)
    bad = env.get_state()
    bad["n_veh"][5] = 12
    with pytest.raises(mm.MMError, match="n_veh"):
        env.set_state(bad)
    env.close()
    plain = mm.MergeEnvBatched(8, cfg)
    with pytest.raises(mm.MMError, match="record_diag"):
        plain.shield_diag()
    plain.close()
    with pytest.raises(mm.MMError):
        mm.MergeEnvBatched(0, cfg)


def test_action_masking_surface(mm):
    """action_masking=True: batched view = per-agent bits; the single-env adapter reproduces the reference's
    aliased-rows mask (`[[0] * n_a] * n`, abstract.py:475-479), i.e. the union over agents in every row."""
    import torch
    g, cfg = load_golden("mass_td3_srew")
    c = dict(env_config(cfg), action_masking=True)
    env = mm.make("merge-multi-agent-v1", config=c)
    obs, mask = env.reset(is_training=False, testing_seeds=cfg["seeds"][0])
    n = len(env.controlled_vehicles)
    assert mask.shape == (n, 5) and (mask == mask[0]).all() and mask[0, 1] == 1
    rows = g["row_of_step"]
    for t in range(30):
        obs, r, d, info = env.step(tuple(int(x) for x in g["act"][t, :n]))
        bits = g["avail_bits"][t, :n]
        union = int(np.bitwise_or.reduce(bits))
        want = np.array([[(union >> a) & 1 for a in range(5)]] * n)
        assert np.array_equal(info["action_mask"], want)
    env.close()
    b = mm.MergeEnvBatched(64, dict(c, traffic_density=3))
    _, m = b.reset(seed=0)
    assert m.shape == (64, 12, 5) and m.dtype == torch.int32
    n_ag = b.buffers()["n_agents"]
    live = torch.arange(12, device="cuda")[None, :] < n_ag[:, None]
    assert bool((m[..., 1] == live.int()).all())          # IDLE exactly for live agents
    assert bool((m[..., 2] == 0).all())                   # LANE_RIGHT is never available on this network
    assert bool((m[live][:, 3] == 1).all() and (m[live][:, 4] == 1).all())   # spawn speed index is 3
    b.close()


@pytest.mark.parametrize("name", V0_CASES + V0_TIE_CASES)
def test_v0_env_cuda_vs_golden_and_adapter(mm, orc, name):
    """BASELINE configs[0]: env merge-multi-agent-v0 (no shield, MDPVehicle, 5x5 observation) teacher-forced against
    the reference, then whole episodes through make('merge-multi-agent-v0')."""
    import torch
    g, cfg = load_golden(name)
    rows = g["row_of_step"]
    env = mm.MergeEnvBatched(len(rows), env_config(cfg))
    assert env.n_s == 25
    env.set_state(full_state(orc, g, rows))
    _, _, _, v = env.step(torch.from_numpy(np.ascontiguousarray(g["act"])).cuda())
    got = outputs_to_numpy(v, OUT_F + OUT_I)
    got["obs"] = obs25(got["obs"])
    assert np.array_equal(env.obs_view().cpu().numpy(), got["obs"])
    compare_states(env.get_state(), full_state(orc, g, rows + 1), STATE_TOL, name, v0=True)
    check_outputs(got, {k: g[k] for k in OUT_F + OUT_I}, g["st_n_cav"][rows])
    assert np.array_equal(v["action_mask"].cpu().numpy().astype(np.int32), g["avail_bits"])
    env.close()
    if name in V0_TIE_CASES:        # snapped before every step: no episode to replay
        return
    single = mm.make("merge-multi-agent-v0", config=env_config(cfg))
    ep = g["ep_start"]
    for j, seed in enumerate(cfg["seeds"]):
        obs, mask = single.reset(is_training=False, testing_seeds=seed)
        n = int(g["st_n_cav"][ep[j]])
        assert obs.shape == (n, 25) and single.n_s == 25
        done = False
        for t in np.where((rows >= ep[j]) & (rows < ep[j + 1] - 1))[0]:
            obs, reward, done, info = single.step(tuple(int(x) for x in g["act"][t, :n]))
            assert rel_err(obs, g["obs"][t, :n]).max() <= 1e-5
            assert abs(reward - g["reward"][t]) <= 1e-5 * max(1, abs(g["reward"][t]))
            assert done == bool(g["done"][t])
        assert done
    single.close()


@pytest.mark.parametrize("name", SUPERVISED_CASES)
def test_supervised_step_reproduces_the_reference(mm, orc, name):
    """safety_guarantee = priority | dmc: the supervisor replaces the meta-actions before _simulate (abstract.py:459-467).
    Teacher-forced on every step of the reference fixtures: from the reference's pre-state, with the policy's tuple and
    the np.random.rand() draws the reference consumed, one mm_step (supervisor + physics + outputs) must produce the
    supervised tuple the reference executed (info["new_action"]), its post-state and its outputs, and report the number
    of draws the reference made."""
    import torch
    g, cfg = load_golden(name)
    rows = g["row_of_step"]
    T = len(rows)
    env = mm.MergeEnvBatched(T, env_config(cfg))
    assert env.n_s == 25 and mm.make_mm_config(env.config).supervisor == {"priority": 1, "dmc": 2}[cfg["safety_guarantee"]]
    env.set_state(full_state(orc, g, rows))
    draws = np.zeros((T, 32))
    draws[:, :16] = np.nan_to_num(g["rand_draws"])
    env.set_supervisor_draws(torch.from_numpy(draws).cuda())
    _, _, _, v = env.step(torch.from_numpy(np.ascontiguousarray(g["act"])).cuda())
    got = outputs_to_numpy(v, OUT_F + OUT_I + ("new_actions",))
    live = np.arange(12)[None, :] < g["st_n_cav"][rows][:, None]
    assert np.array_equal(got["new_actions"][live], g["new_act"][live])
    assert int((g["new_act"][live] != g["act"][live]).sum()) > 100          # the supervisors did replace actions
    assert np.array_equal(env.supervisor_draws_used(), np.sum(~np.isnan(g["rand_draws"]), axis=1))
    got["obs"] = obs25(got["obs"])
    compare_states(env.get_state(), full_state(orc, g, rows + 1), STATE_TOL, name, v0=True)
    check_outputs(got, {k: g[k] for k in OUT_F + OUT_I}, g["st_n_cav"][rows])
    env.close()


@pytest.mark.parametrize("name", SUPERVISED_CASES)
def test_single_env_adapter_replays_supervised_episodes(mm, name):
    """make("merge-multi-agent-v0") with safety_guarantee = priority | dmc is seed-exact: reset(testing_seeds = s) builds
    the reference's scene and leaves its MT19937 stream where the reference's is, every step hands the supervisor the
    next draws of that stream and advances it by what was consumed - the whole episode reproduces the reference's
    supervised tuples, rewards and observations."""
    g, cfg = load_golden(name)
    ep, rows = g["ep_start"], g["row_of_step"]
    env = mm.make("merge-multi-agent-v0", config={k: cfg[k] for k in cfg if k not in ("seeds", "env_name")})
    for k, seed in enumerate(cfg["seeds"][:3]):
        obs, _ = env.reset(is_training=False, testing_seeds=seed)
        steps = np.where((rows >= ep[k]) & (rows < ep[k + 1] - 1))[0]
        n = len(env.controlled_vehicles)
        for t in steps:
            obs, reward, done, info = env.step(tuple(int(a) for a in g["act"][t, :n]))
            assert tuple(info["new_action"]) == tuple(int(a) for a in g["new_act"][t, :n]), (seed, int(t))
            assert abs(reward - float(g["reward"][t])) <= 1e-4 * max(1.0, abs(float(g["reward"][t])))
            assert np.abs(obs - g["obs"][t, :n]).max() <= 1e-5, (seed, int(t))
            assert done == bool(g["done"][t])
    env.close()


def test_batched_supervisors_draw_from_philox_and_only_touch_the_actions(mm):
    """Batched mode: the supervisors take their uniform numbers from Philox keyed (seed, env, episode, policy step).
    Two handles with the same seed agree bit for bit, the executed tuples differ from the policy's on some steps, and an
    env whose tuple was not changed moves exactly as without a supervisor."""
    import torch
    E = 2048
    cfg = dict(mm.DEFAULT_CONFIG, env_name="merge-multi-agent-v0", safety_guarantee="dmc", traffic_density=3, mixed_traffic=True)
    a_env, b_env = mm.MergeEnvBatched(E, cfg), mm.MergeEnvBatched(E, cfg)
    c_env = mm.MergeEnvBatched(E, dict(cfg, safety_guarantee="none"))
    for env in (a_env, b_env, c_env):
        env.reset(seed=5)
    gen = torch.Generator(device="cuda").manual_seed(1)
    changed_total = 0
    for t in range(12):
        act = torch.randint(0, 5, (E, 12), generator=gen, device="cuda", dtype=torch.int8)
        pre = c_env.get_state()
        _, _, _, va = a_env.step(act)
        _, _, _, vb = b_env.step(act)
        torch.cuda.synchronize()
        na = va["new_actions"].cpu().numpy()
        assert np.array_equal(na, vb["new_actions"].cpu().numpy())
        sa, sb = a_env.get_state(), b_env.get_state()
        assert all(np.array_equal(sa[k], sb[k]) for k in sa)
        live = np.arange(12)[None, :] < pre["n_cav"][:, None]
        changed = ((na != act.cpu().numpy()) & live).any(axis=1)
        changed_total += int(changed.sum())
        # the un-supervised handle executes the supervised tuples: same dynamics
        c_env.step(torch.from_numpy(np.where(live, na, act.cpu().numpy())).cuda())
        sc = c_env.get_state()
        assert all(np.array_equal(sa[k], sc[k]) for k in ("x", "y", "speed", "lane", "crashed"))
    assert changed_total > 0
    for env in (a_env, b_env, c_env):
        env.close()



"""CPU tests of the GAE(lambda) returns (mm_lambda_returns, rollout.lambda_returns, gae_lambda of the learners and the
driver): the C ABI declaration, export and ctypes signature, the argument checks that come before any CUDA call, the
refusals of the learners and of train(), and the numpy restatements of the recursion (lambda_returns_ref.py)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import lambda_returns_ref as ref
from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "marl_mass_b200.h")
INI = os.path.join(ROOT, "examples", "mass_td3_srew.ini")


def test_header_declares_and_library_exports_the_entry_point():
    import marl_mass_b200 as mm
    from marl_mass_b200 import _lib
    src = open(HEADER).read()
    assert re.search(r"int mm_lambda_returns\(const float \*rewards, const uint8_t \*dones, const float \*values, "
                     r"const float \*final_value, float gamma,\s+float lambda, int T, int64_t n_cols, int cols_per_env, "
                     r"float \*out, void \*stream\);", src)
    # mm_discounted_returns keeps its signature, and the ABI version stays
    assert re.search(r"int mm_discounted_returns\(const float \*rewards, const uint8_t \*dones, const float \*final_value, "
                     r"float gamma, int T,\s+int64_t n_cols, int cols_per_env, float \*out, void \*stream\);", src)
    assert re.search(r"#define MM_ABI_VERSION 9\b", src)
    assert "mm_lambda_returns" in _lib.EXPORTS
    f = mm.lib().mm_lambda_returns
    assert f.argtypes == [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int, C.c_int64, C.c_int,
                          C.c_void_p, C.c_void_p]
    assert f.restype == C.c_int


@pytest.fixture(scope="module")
def L():
    import marl_mass_b200 as mm
    from marl_mass_b200 import build
    build.build()
    return mm.lib()


def _call(L, rewards=True, dones=True, values=True, fv=True, gamma=0.99, lam=0.95, T=10, n_cols=24, cpe=12, out=True):
    """non-null fake host addresses: the checks must fail before anything is dereferenced or launched"""
    p = [C.c_void_p(0x1000 * (k + 1)) for k in range(5)]
    return L.mm_lambda_returns(p[0] if rewards else None, p[1] if dones else None, p[2] if values else None,
                               p[3] if fv else None, gamma, lam, T, n_cols, cpe, p[4] if out else None, None)


def test_argument_checks_come_before_any_cuda_call(L):
    def rejected(rc, what):
        assert rc == -1, (rc, what)
        assert what in L.mm_last_error().decode(), (what, L.mm_last_error())

    for k in ("rewards", "dones", "out"):
        rejected(_call(L, **{k: False}), "rewards, dones and out are required")
    for lam in (-0.01, 1.01, -np.inf, np.inf, np.nan):
        rejected(_call(L, lam=lam), "lambda must be in [0, 1]")
        rejected(_call(L, lam=lam, values=False), "lambda must be in [0, 1]")
    for gamma in (np.nan, np.inf, -np.inf):
        rejected(_call(L, gamma=gamma), "gamma must be finite")
        rejected(_call(L, gamma=gamma, lam=1.0, values=False), "gamma must be finite")
    for lam in (0.0, 0.5, 0.95, float(np.nextafter(np.float32(1), np.float32(0)))):
        rejected(_call(L, lam=lam, values=False), "values are required for lambda < 1")
    rejected(_call(L, T=-1), "bad rollout shape")
    rejected(_call(L, n_cols=25), "bad rollout shape")
    rejected(_call(L, cpe=0), "bad rollout shape")
    rejected(_call(L, n_cols=-12), "bad rollout shape")


def test_learners_refuse_a_bad_gae_lambda_before_touching_the_env():
    from marl_mass_b200 import rollout
    for bad in ("x", "nan", float("nan"), -0.1, 1.5, True, [0.9], float("inf")):
        for cls in (rollout.BatchedMAPPORollout, rollout.BatchedMAPPOGIRollout):
            with pytest.raises(ValueError, match="gae_lambda"):
                cls(None, gae_lambda=bad)
    assert rollout.check_gae_lambda(None) is None
    for ok, want in ((0, 0.0), (1, 1.0), (0.95, 0.95), ("0.9", 0.9), (np.float32(0.5), 0.5)):
        assert rollout.check_gae_lambda(ok) == want


def test_train_refuses_bad_gae_lambda_after_the_existing_refusals(tmp_path):
    from marl_mass_b200.train import load_ini, train
    for bad in ("abc", float("nan"), -0.5, 1.0001, True):
        with pytest.raises(ValueError, match="gae_lambda"):
            train(INI, n_envs=4, iterations=1, gae_lambda=bad)
    with pytest.raises(ValueError, match="eval_seeds"):         # the refusals that were there first still come first
        train(INI, n_envs=4, iterations=1, eval_seeds=0, eval_shield=True, gae_lambda="abc")
    with pytest.raises(ValueError, match="update_stats"):
        train(INI, n_envs=4, iterations=1, update_stats="yes", gae_lambda="abc")
    text = open(INI).read()
    assert "gae_lambda" not in text and load_ini(INI)[2]["gae_lambda"] is None     # the shipped inis: the reference's returns
    for value in ("abc", "nan", "2"):
        bad = tmp_path / ("bad_%s.ini" % value)
        bad.write_text(text.replace("[MODEL_CONFIG]", "[MODEL_CONFIG]\ngae_lambda = %s" % value))
        with pytest.raises(ValueError, match="gae_lambda"):
            train(str(bad), n_envs=4, iterations=1)
    good = tmp_path / "good.ini"
    good.write_text(text.replace("[MODEL_CONFIG]", "[MODEL_CONFIG]\ngae_lambda = 0.95"))
    env_cfg, kw, tr = load_ini(str(good))
    assert tr["gae_lambda"] == "0.95" and kw == load_ini(INI)[1]
    v0 = tmp_path / "v0.ini"
    v0.write_text(re.sub(r"(?m)^env_name\s*=.*$", "env_name = merge-multi-agent-v0", text)
                  if re.search(r"(?m)^env_name\s*=", text) else text.replace("[ENV_CONFIG]", "[ENV_CONFIG]\nenv_name = merge-multi-agent-v0"))
    with pytest.raises(ValueError, match="env id"):
        train(str(v0), n_envs=4, iterations=1, gae_lambda="abc")


def test_cli_has_the_option():
    import subprocess
    import sys
    out = subprocess.run([sys.executable, "-m", "marl_mass_b200.train", "--help"], cwd=ROOT, capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 0 and "--gae-lambda" in out.stdout


# ---- the restatements

@pytest.mark.parametrize("lam", [0.0, 0.5, 0.95, 1.0])
def test_float32_and_float64_recursions_agree_with_the_td_residual_form(lam):
    r, d, v, fv = ref.random_rollout(100, 37, 12, seed=int(lam * 100) + 1)
    for f in (fv, None):
        r32 = ref.lambda_returns_ref(r, d, v, f, 0.99, lam)
        r64 = ref.lambda_returns_ref(r, d, v, f, 0.99, lam, dtype=np.float64)
        gae = ref.gae_returns_ref(r, d, v, f, 0.99, lam)
        assert r32.dtype == np.float32 and r64.dtype == np.float64
        assert np.abs(r64 - gae).max() <= 1e-12 * max(1.0, np.abs(gae).max())
        assert np.all(np.abs(r32 - r64) <= 1e-5 * np.maximum(np.abs(r64), 1.0))


def test_lambda_one_is_the_discounted_return_and_lambda_zero_the_one_step_target():
    r, d, v, fv = ref.random_rollout(60, 41, 12, seed=7)
    for f in (fv, None):
        disc = ref.discounted_returns_ref(r, d, f, 0.99)
        assert ref.lambda_returns_ref(r, d, v, f, 0.99, 1.0).tobytes() == disc.tobytes()
        assert ref.lambda_returns_ref(r, d, v, f, 0.99, 0.0).tobytes() == ref.one_step_targets_ref(r, d, v, f, 0.99).tobytes()
    # the discounted return itself, from its definition in float64
    disc = ref.discounted_returns_ref(r, d, fv, 0.99)
    want = np.zeros_like(r, dtype=np.float64)
    run = fv.astype(np.float64)
    for t in range(59, -1, -1):
        run = np.where((d[t] != 0)[:, None], 0.0, run) * 0.99 + r[t]
        want[t] = run
    assert np.abs(disc - want).max() <= 1e-5 * np.abs(want).max()


def test_values_after_a_terminal_step_and_at_step_zero_are_never_read():
    r, d, v, fv = ref.random_rollout(50, 29, 12, seed=3)
    poisoned = v.copy()
    poisoned[0] = np.nan
    poisoned[1:][d[:-1] != 0] = np.nan
    for lam in (0.0, 0.5, 0.95, 1.0):
        a = ref.lambda_returns_ref(r, d, v * np.where(np.isnan(poisoned), 0, 1).astype(np.float32), fv, 0.99, lam)
        b = ref.lambda_returns_ref(r, d, np.nan_to_num(poisoned, nan=0.0), fv, 0.99, lam)
        c = ref.lambda_returns_ref(r, d, poisoned, fv, 0.99, lam)
        assert np.isfinite(c).all() and a.tobytes() == b.tobytes() == c.tobytes()

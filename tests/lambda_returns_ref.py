"""numpy restatements of mm_lambda_returns (rollout.lambda_returns) for the tests.

`lambda_returns_ref` runs the kernel's recursion column by column over [T, E, A] arrays:
  float32: every product and sum rounded to float32 in the kernel's order (the library is built with -fmad=false and
           the lambda mix uses __fmul_rn / __fadd_rn, so nothing is fused), which the kernel must match bit for bit;
  float64: the same recursion in float64, the accuracy reference.
`gae_returns_ref` is the textbook form in float64, from the TD residuals: A_t = delta_t + gamma lambda (1 - d_t) A_{t+1},
delta_t = r_t + gamma (1 - d_t) V_{t+1} - V_t, R_t = A_t + V_t, with V_T = final_value: an independent check of the
recursion in the two forms above."""
import numpy as np


def lambda_returns_ref(rewards, dones, values, final_value, gamma, lam, dtype=np.float32):
    """rewards [T, E, A], dones [T, E], values [T, E, A] or None (lambda = 1 only), final_value [E, A] or None"""
    f = np.dtype(dtype).type
    r = np.asarray(rewards).astype(f)
    T = r.shape[0]
    g, lm = f(gamma), f(lam)
    oml = f(1) - lm
    run = np.zeros(r.shape[1:], f) if final_value is None else np.asarray(final_value).astype(f).copy()
    v_next = run.copy()
    out = np.empty_like(r)
    for t in range(T - 1, -1, -1):
        done = (np.asarray(dones[t]) != 0)[:, None]
        run = np.where(done, f(0), run)
        v_next = np.where(done, f(0), v_next)
        if values is not None:
            run = lm * run + oml * v_next
            v_next = np.asarray(values[t]).astype(f)
        run = run * g + r[t]
        out[t] = run
    return out


def discounted_returns_ref(rewards, dones, final_value, gamma):
    """mm_discounted_returns in float32: run = run * gamma + r, restarted after a terminal step"""
    return lambda_returns_ref(rewards, dones, None, final_value, gamma, 1.0)


def one_step_targets_ref(rewards, dones, values, final_value, gamma):
    """lambda = 0: r_t + gamma (1 - d_t) V_{t+1} in float32 (V_T = final_value, 0 when None)"""
    r = np.asarray(rewards, np.float32)
    v = np.asarray(values, np.float32)
    nxt = np.concatenate([v[1:], (np.zeros_like(v[:1]) if final_value is None else
                                  np.asarray(final_value, np.float32)[None])], 0)
    nxt = np.where((np.asarray(dones) != 0)[:, :, None], np.float32(0), nxt)
    return nxt * np.float32(gamma) + r


def gae_returns_ref(rewards, dones, values, final_value, gamma, lam):
    """float64 GAE(lambda) advantages from the TD residuals, plus the values"""
    r = np.asarray(rewards, np.float64)
    v = np.asarray(values, np.float64)
    T = r.shape[0]
    v_next = np.zeros_like(v[0]) if final_value is None else np.asarray(final_value, np.float64)
    adv = np.zeros_like(v[0])
    out = np.empty_like(r)
    for t in range(T - 1, -1, -1):
        keep = (np.asarray(dones[t]) == 0)[:, None]
        delta = r[t] + gamma * keep * v_next - v[t]
        adv = delta + gamma * lam * keep * adv
        out[t] = adv + v[t]
        v_next = v[t]
    return out


def random_rollout(T, E, A, seed, done_rate=0.08):
    """rewards / values N(0, 1) f32, dones u8 at random steps with the last step and runs of consecutive steps forced
    in some envs, final_value f32"""
    rng = np.random.default_rng(seed)
    r = rng.normal(0, 1, (T, E, A)).astype(np.float32)
    v = rng.normal(0, 2, (T, E, A)).astype(np.float32)
    d = (rng.random((T, E)) < done_rate).astype(np.uint8)
    d[T - 1, ::3] = 1                         # the last step terminal
    d[T // 2: T // 2 + 3, 1::5] = 1           # three terminal steps in a row
    d[T - 2:, 2::7] = 1                       # the last two
    fv = rng.normal(0, 2, (E, A)).astype(np.float32)
    return r, d, v, fv

"""Numpy restatement of the per-row loss derivatives of the on-device PPO learner (learner.cu, `ppo_row` and the
value term), as torch autograd computes them for `rollout.mappo_losses` / `shared_network_loss` (pairwise=False,
critic_loss="mse").

For one row with ratio r = exp(logp_a - old_logp), advantage adv and clip c, the PPO-clip term is
    l = -min(s1, s2),  s1 = r adv,  s2 = clamp(r, 1 - c, 1 + c) adv
and autograd's rules give
    d l / d r    = -(w1 adv + w2 adv [1 - c <= r <= 1 + c])
                   w1, w2 = (1, 0) if s1 < s2, (0, 1) if s1 > s2, (1/2, 1/2) at a tie (torch.min splits the gradient;
                   clamp passes it at its bounds, inclusive)
    d l / d logp_a = (d l / d r) r                       (exp backward)
    d l / d z_k  = (d l / d logp_a) (delta_ka - softmax(z)_k)      (log-softmax backward, z = logits)
The value term (V - G)^2 gives d / d V = 2 (V - G).  The mean over N rows multiplies all of these by 1 / N.
"""
import numpy as np


def ppo_row(ratio, adv, clip):
    """-> (loss, d loss / d logp_a) per row, float32 arithmetic as the kernel does it (before the 1/N)."""
    r = np.asarray(ratio, np.float32)
    adv = np.asarray(adv, np.float32)
    lo, hi = np.float32(1.0) - np.float32(clip), np.float32(1.0) + np.float32(clip)
    s1 = r * adv
    s2 = np.minimum(np.maximum(r, lo), hi) * adv
    loss = -np.minimum(s1, s2)
    w1 = np.where(s1 < s2, np.float32(1.0), np.where(s1 == s2, np.float32(0.5), np.float32(0.0))).astype(np.float32)
    w2 = np.float32(1.0) - w1
    inside = ((r >= lo) & (r <= hi)).astype(np.float32)
    d_r = -(w1 * adv + w2 * (adv * inside))
    return loss, d_r * r


def logit_grad(logits, action, g_logp):
    """d loss / d z for log-softmax logits z [N, 5], the taken action [N] and d loss / d logp_a [N]."""
    z = np.asarray(logits, np.float64)
    p = np.exp(z - z.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    onehot = np.eye(z.shape[1])[np.asarray(action)]
    return np.asarray(g_logp, np.float64)[:, None] * (onehot - p)


def value_row(values, returns):
    """-> (loss, d loss / d V) per row of the MSE value term (before the 1/N)."""
    d = np.asarray(values, np.float32) - np.asarray(returns, np.float32)
    return d * d, np.float32(2.0) * d

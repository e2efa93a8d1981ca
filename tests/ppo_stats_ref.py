"""Float64 restatement of the learner's statistics pass (mm_ppo_stats: learner.cu's ppo_kernel<KIND, false, true>), built
on the forward of learner_ref.learner_pass.

With fp16=False everything runs in float64: the reference the torch statistics (rollout.ppo_stats_torch) on float64
modules must match.  With fp16=True the forward is learner_pass's fp16 mode (the kernel's roundings) and the per-row values
are formed in float32 in the kernel's order: p_k = e_k / s and log p_k = (z_k - m) - log s from the pass, the entropy
-sum_k p_k log p_k accumulated over k = 0..4, r = exp(logp(a) - old_logp), k3 = (r - 1) - (logp(a) - old_logp), clipped
|r - 1| > clip, the residual G - v; squares and sums in float64.
"""
import numpy as np

import learner_ref

FIELDS = ("n", "entropy", "k3", "clipped", "ratio_min", "ratio_max", "v", "v2", "g", "g2", "res2")
K = {k: i for i, k in enumerate(FIELDS)}


def stat_rows(kind, params, S, A8, G, idx, old_logp=None, clip=0.2, fp16=False):
    """-> dict of per-row arrays over idx: entropy, logp, ratio, k3, clipped (actor, shared; ratio terms with old_logp),
    v, g, res (critic, shared)"""
    dt = np.float32 if fp16 else np.float64
    idx = np.asarray(idx, np.int64)
    A8 = np.asarray(A8)
    out = {}
    base = learner_ref.learner_pass(kind, params, S, A8, None, None, None, idx, clip, fp16=fp16)
    if kind != "critic":
        # log p_k of every action: the pass's log p(a) with each action in turn (the policy forward ignores the action)
        lp = [learner_ref.learner_pass(kind, params, S, np.full_like(A8, k), None, None, None, idx, clip, fp16=fp16)["logp"]
              for k in range(learner_ref.NA)]
        p = base["p"].astype(dt)
        pl = np.zeros(len(idx), dt)
        for k in range(learner_ref.NA):
            pl = (pl + p[:, k] * np.asarray(lp[k], dt)).astype(dt)
        out["entropy"] = (-pl).astype(dt)
        logp = np.asarray(base["logp"], dt)
        out["logp"] = logp
        if old_logp is not None:
            lr = (logp - np.asarray(old_logp)[idx].astype(dt)).astype(dt)
            r = np.exp(lr).astype(dt)
            out["ratio"] = r
            out["k3"] = ((r - dt(1)) - lr).astype(dt)
            out["clipped"] = np.abs(r - dt(1)) > dt(clip)
    if kind != "actor":
        v = np.asarray(base["q" if kind == "critic" else "v"], dt)
        g = np.asarray(G)[idx].astype(dt)
        out["v"], out["g"], out["res"] = v, g, (g - v).astype(dt)
    return out


def ppo_stats_ref(kind, params, S, A8, G, idx, old_logp=None, clip=0.2, fp16=False):
    """-> float64 [11], the fields of FIELDS, as mm_ppo_stats defines them"""
    rows = stat_rows(kind, params, S, A8, G, idx, old_logp, clip, fp16)
    s = np.zeros(len(FIELDS))
    s[K["n"]] = len(np.asarray(idx))
    s[K["ratio_min"]], s[K["ratio_max"]] = np.inf, -np.inf
    d = lambda k: rows[k].astype(np.float64)  # noqa: E731
    if "entropy" in rows:
        s[K["entropy"]] = d("entropy").sum()
    if "ratio" in rows and len(rows["ratio"]):
        s[K["k3"]] = d("k3").sum()
        s[K["clipped"]] = float(rows["clipped"].sum())
        s[K["ratio_min"]], s[K["ratio_max"]] = d("ratio").min(), d("ratio").max()
    if "v" in rows:
        v, g, res = d("v"), d("g"), d("res")
        s[K["v"]], s[K["v2"]], s[K["g"]], s[K["g2"]], s[K["res2"]] = v.sum(), (v * v).sum(), g.sum(), (g * g).sum(), (res * res).sum()
    return s

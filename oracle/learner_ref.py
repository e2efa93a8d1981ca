"""Numpy restatement of the on-device PPO learner (learner.cu): the per-row loss derivatives, as torch autograd computes
them for `rollout.mappo_losses` / `shared_network_loss` (pairwise=False, critic_loss="mse"), and the whole target and
gradient pass of the three network kinds (`learner_pass`).

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

# ActorCriticNetwork (state_split): the observation columns of fc11 / fc12 / fc13 (Model_gi.py:137-176)
COLS1 = (0, 5, 10, 15, 20)
COLS2 = (1, 2, 6, 7, 11, 12, 16, 17, 21, 22)
COLS3 = (3, 4, 8, 9, 13, 14, 18, 19, 23, 24)
KINDS = ("actor", "critic", "shared")
NA = 5


def ppo_row(ratio, adv, clip, dtype=np.float32):
    """-> (loss, d loss / d logp_a) per row in `dtype` arithmetic (float32: as the kernel does it), before the 1/N."""
    r = np.asarray(ratio, dtype)
    adv = np.asarray(adv, dtype)
    one = dtype(1.0)
    lo, hi = one - dtype(clip), one + dtype(clip)
    s1 = r * adv
    s2 = np.minimum(np.maximum(r, lo), hi) * adv
    loss = -np.minimum(s1, s2)
    w1 = np.where(s1 < s2, one, np.where(s1 == s2, dtype(0.5), dtype(0.0))).astype(dtype)
    w2 = one - w1
    inside = ((r >= lo) & (r <= hi)).astype(dtype)
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


def _layers(kind, params):
    """The three layers as the kernel holds them: (W1 [H1][30], b1, W2 [128][IN2], b2, W3 [OUT3][128], b3).  The shared
    network's first-layer blocks become one dense 30 -> 160 layer (zero outside the blocks), its value head output 5."""
    p = {k: np.asarray(v, np.float64) for k, v in params.items()}
    if kind != "shared":
        return p["fc1.weight"], p["fc1.bias"], p["fc2.weight"], p["fc2.bias"], p["fc3.weight"], p["fc3.bias"]
    h4, h2 = p["fc11.weight"].shape[0], p["fc12.weight"].shape[0]
    w1 = np.zeros((h4 + 2 * h2, 30))
    w1[:h4, COLS1] = p["fc11.weight"]
    w1[h4:h4 + h2, COLS2] = p["fc12.weight"]
    w1[h4 + h2:, COLS3] = p["fc13.weight"]
    b1 = np.concatenate([p["fc11.bias"], p["fc12.bias"], p["fc13.bias"]])
    w3 = np.concatenate([p["actor_linear.weight"], p["critic_linear.weight"]])
    b3 = np.concatenate([p["actor_linear.bias"], p["critic_linear.bias"]])
    return w1, b1, p["fc2.weight"], p["fc2.bias"], w3, b3


def _unit(v):
    """the largest power of two of which every element of v is an integer multiple (1 for an all-zero array)"""
    v = np.asarray(v, np.float64)
    nz = np.abs(v[v != 0])
    if nz.size == 0:
        return 1.0
    m, e = np.frexp(nz)                                   # nz = m 2^e, m in [1/2, 1): m 2^53 is an integer
    mi = (m * 2.0 ** 53).astype(np.int64)
    return float(np.ldexp((mi & -mi).astype(np.float64), e - 53).min())


class Exactness(AssertionError):
    """a premise of exact fp16 / fp32 arithmetic does not hold for the data given to learner_pass(check=True)"""


def learner_pass(kind, params, S, A8, G, old_logp, q_target, idx, clip, fp16=False, check=False):
    """The target pass and the gradient pass of learner.cu on the rows S[idx] (duplicate and unsorted entries are rows
    like any other), in numpy float64.

    kind: "actor" (ActorNetwork), "critic" (CriticNetwork) or "shared" (ActorCriticNetwork, state_split); params:
    {torch parameter name: array} in torch layout.  S [rows, 30], A8 [rows], G [rows] the returns, old_logp [rows] (actor,
    shared), q_target [rows] (actor; the advantage is G - q_target), indexed like S.  G None: the target pass alone.

    fp16=True rounds to fp16 exactly where the kernel does: the inputs, W1, W2, W3, h1 and h2 after ReLU, dZ3 and the
    masked dZ2 and dZ1; the ReLU masks of the backward are taken from the fp16 activations.  Biases, the log-softmax and
    the per-row loss run in float32 in the kernel's order, the row sums are exact (float64) and the final 1/N is the
    reduction's float32 `sum * (1 / N)`.  With check=True (needs fp16=True) it raises `Exactness` unless every value the
    kernel rounds to fp16 is an fp16 value, every float32 intermediate is exact and every sum the kernel accumulates in
    float32 stays below 2^24 of its unit: then the kernel's result does not depend on its summation order and this
    function predicts it bit for bit.

    -> dict: grads {name: array, torch layout}, sums (the same before the 1/N), loss_a, loss_c (0 for the kind that
    has none), logp (actor, shared) / q (critic) / v (shared) per row of idx, and the per-row ratio, gl (d loss / d logp_a
    before the 1/N) and adv."""
    assert kind in KINDS, kind
    assert not check or fp16, "the exactness checks describe the fp16 pass"
    f32 = np.float32
    idx = np.asarray(idx, np.int64)
    n = len(idx)
    S, A8 = np.asarray(S), np.asarray(A8)
    w1, b1, w2, b2, w3, b3 = _layers(kind, params)
    H1, out3 = w1.shape[0], w3.shape[0]

    def r16(v, what):
        if not fp16:
            return v
        h = np.asarray(v, np.float64).astype(np.float16).astype(np.float64)
        if check and not np.array_equal(h, v):
            raise Exactness("%s is not exact in fp16" % what)
        return h

    def exact32(v, what):
        if check and not np.array_equal(np.asarray(v, np.float64).astype(f32).astype(np.float64), v):
            raise Exactness("%s is not exact in fp32" % what)

    def mm(a, b, what):
        """a @ b, which the kernel accumulates in fp32"""
        if check and a.size and b.size:
            bound = np.abs(a) @ np.abs(b)
            if bound.max() >= 2.0 ** 24 * _unit(a) * _unit(b):
                raise Exactness("the sums of %s reach 2^24 units" % what)
        return a @ b

    def lin(x, w, b, what):
        acc = mm(x, w.T, what)
        if not fp16:
            return acc + b
        exact32(acc, what)
        out = acc.astype(f32) + b.astype(f32)
        exact32(acc + b, what + " + bias")
        return out.astype(np.float64)

    x = r16(S[idx].astype(np.float64), "the input rows")
    a = A8[idx].astype(np.int64)
    onehot = np.eye(NA)[a]
    w1, w2, w3 = r16(w1, "W1"), r16(w2, "W2"), r16(w3, "W3")
    h1 = r16(np.maximum(lin(x, w1, b1, "x W1^T"), 0.0), "h1")
    h1in = np.concatenate([h1, onehot], 1) if kind == "critic" else h1
    h2 = r16(np.maximum(lin(h1in, w2, b2, "h1 W2^T"), 0.0), "h2")
    z = lin(h2, w3, b3, "h2 W3^T")
    out = {"active": (float((h1 > 0).mean()) if n else 0.0, float((h2 > 0).mean()) if n else 0.0)}
    dz = np.zeros((n, out3))
    loss_a = np.zeros(n)
    loss_c = np.zeros(n)
    g = None if G is None else np.asarray(G)[idx].astype(np.float64)
    if kind != "critic":
        zl = z[:, :NA]
        if fp16:     # learner.cu: m = max, e_k = expf(z_k - m), s = e_0 + ... + e_4, logp = (z_a - m) - logf(s)
            zl = zl.astype(f32)
            m = zl.max(1)
            e = np.exp(zl - m[:, None])
            s = f32(0)
            for k in range(NA):
                s = s + e[:, k]
            logp = (zl[np.arange(n), a] - m) - np.log(s)
            p = (e / s[:, None]).astype(np.float64)
        else:
            m = zl.max(1)
            e = np.exp(zl - m[:, None])
            s = e.sum(1)
            logp = zl[np.arange(n), a] - m - np.log(s)
            p = e / s[:, None]
        out["logp"], out["p"] = logp, p
        if g is not None:
            dt = f32 if fp16 else np.float64
            adv = (g - np.asarray(q_target, np.float64)[idx]) if kind == "actor" else g - z[:, 5]
            exact32(adv, "the advantage")
            adv = adv.astype(dt)
            ratio = np.exp(logp.astype(dt) - np.asarray(old_logp)[idx].astype(dt))
            la, gl = ppo_row(ratio, adv, clip, dt)
            if check:
                la64, gl64 = ppo_row(ratio.astype(np.float64), adv.astype(np.float64), clip, np.float64)
                if not (np.array_equal(la64, la) and np.array_equal(gl64, gl)):
                    raise Exactness("the per-row PPO term is not exact in fp32")
            loss_a = la.astype(np.float64)
            gl = gl.astype(np.float64)
            d = gl[:, None] * (onehot - p)
            exact32(d, "d loss / d z")
            dz[:, :NA] = d
            out.update(ratio=ratio, gl=gl, adv=adv)
    if kind != "actor":
        kv = 0 if kind == "critic" else 5
        out["q" if kind == "critic" else "v"] = z[:, kv].astype(f32) if fp16 else z[:, kv]
    if g is None:
        return out
    if kind != "actor":
        dv = z[:, kv] - g
        exact32(dv, "V - G")
        loss_c = dv * dv
        exact32(loss_c, "(V - G)^2")
        dz[:, kv] = 2.0 * dv
    dz = r16(dz, "dZ3")
    dz2 = r16(np.where(h2 > 0, mm(dz, w3, "dZ3 W3"), 0.0), "dZ2")
    dz1 = r16(np.where(h1 > 0, mm(dz2, w2[:, :H1], "dZ2 W2"), 0.0), "dZ1")
    ones = np.ones((n, 1))
    sums = {}
    sums["w3"] = mm(dz.T, np.concatenate([h2, ones], 1), "dZ3^T [h2 | 1]")
    sums["w2"] = mm(dz2.T, np.concatenate([h1in, ones], 1), "dZ2^T [h1 | 1]")
    sums["w1"] = mm(dz1.T, np.concatenate([x, ones], 1), "dZ1^T [x | 1]")
    ls = mm(np.stack([loss_a, loss_c]), ones, "the loss sums")[:, 0] if n else np.zeros(2)
    if fp16:
        inv = f32(1) / f32(max(n, 1))
        scale = lambda v: (np.asarray(v, np.float64).astype(f32) * inv).astype(np.float64) + 0.0  # noqa: E731
    else:
        scale = lambda v: np.asarray(v, np.float64) / max(n, 1)  # noqa: E731
    raw = {}
    if kind == "shared":
        h4, h2w = params["fc11.weight"].shape[0], params["fc12.weight"].shape[0]
        blocks = (("fc11", 0, h4, COLS1), ("fc12", h4, h4 + h2w, COLS2), ("fc13", h4 + h2w, H1, COLS3))
        for name, lo, hi, cols in blocks:
            raw[name + ".weight"] = sums["w1"][lo:hi][:, list(cols)]
            raw[name + ".bias"] = sums["w1"][lo:hi, -1]
        raw["fc2.weight"], raw["fc2.bias"] = sums["w2"][:, :-1], sums["w2"][:, -1]
        raw["actor_linear.weight"], raw["actor_linear.bias"] = sums["w3"][:NA, :-1], sums["w3"][:NA, -1]
        raw["critic_linear.weight"], raw["critic_linear.bias"] = sums["w3"][5:6, :-1], sums["w3"][5:6, -1]
    else:
        for k in (1, 2, 3):
            raw["fc%d.weight" % k], raw["fc%d.bias" % k] = sums["w%d" % k][:, :-1], sums["w%d" % k][:, -1]
    out["sums"] = raw
    out["grads"] = {k: scale(v) for k, v in raw.items()}
    out["loss_a"], out["loss_c"] = (float(scale(ls[0])), float(scale(ls[1])))
    return out


# ---- exactly representable learner data: networks and rows on coarse dyadic grids with sparse weights, so that every
# value learner.cu rounds to fp16 is an fp16 value and every fp32 sum it forms is exact; its result then does not depend
# on summation order and learner_pass(fp16=True) predicts it bit for bit (the only inexact step left is the reduction's
# sum * (1 / N), which numpy reproduces)

EXACT_CLIP = 0.25      # 1 - c and 1 + c exact, so a clipped row's loss -(1 +- c) adv is exact too
PUSH = 1.0             # log-ratio of the rows pushed outside the clip range: r = e^(+-1), far from 1 +- c
PARAM_NAMES = {"actor": ("fc1", "fc2", "fc3"), "critic": ("fc1", "fc2", "fc3"),
               "shared": ("fc11", "fc12", "fc13", "fc2", "actor_linear", "critic_linear")}


def _sparse(rng, shape, k, values):
    w = np.zeros(shape)
    for o in range(shape[0]):
        w[o, rng.choice(shape[1], k, replace=False)] = rng.choice(values, k)
    return w


def exact_params(kind, group, seed):
    """Parameters {torch name: float32 array} of a network whose activations stay small integers (x, W1, W2, b1, b2
    integer, two or three non-zeros per row) and whose policy head gives p in {0, 1/group} exactly: the first `group`
    actions share one W3 row and bias 0, the others have bias -128 and small rows, so their logits lie more than 104
    below the group's and expf of their difference is exactly 0 in fp32."""
    assert group in (1, 2, 4)
    rng = np.random.default_rng(seed)
    ints = (-1.0, 1.0)
    p = {}

    def layer(name, out, inp, k):
        p[name + ".weight"] = _sparse(rng, (out, inp), k, ints)
        p[name + ".bias"] = rng.choice((-1.0, 0.0, 0.0, 1.0), out)

    if kind == "shared":
        layer("fc11", 32, 5, 2)
        layer("fc12", 64, 10, 2)
        layer("fc13", 64, 10, 2)
        layer("fc2", 128, 160, 3)
    else:
        layer("fc1", 128, 30, 2)
        layer("fc2", 128, 128 + (NA if kind == "critic" else 0), 3)
        if kind == "critic":
            p["fc2.weight"][:, 128:] = rng.choice((-1.0, 0.0, 1.0), (128, NA))
    quarter = (-0.5, -0.25, 0.25, 0.5)
    value = (_sparse(rng, (1, 128), 4, quarter), rng.choice(quarter, 1))
    if kind == "critic":
        p["fc3.weight"], p["fc3.bias"] = value
    else:
        w3 = _sparse(rng, (NA, 128), 2, (-0.25, 0.25))
        w3[:group] = _sparse(rng, (1, 128), 3, quarter)
        b3 = np.where(np.arange(NA) < group, 0.0, -128.0)
        head = "fc3" if kind == "actor" else "actor_linear"
        p[head + ".weight"], p[head + ".bias"] = w3, b3
        if kind == "shared":
            p["critic_linear.weight"], p["critic_linear.bias"] = value
    return {k: v.astype(np.float32) for k, v in p.items()}


def exact_rows(rows, seed):
    """S [rows, 30] with entries in {-1, 0, 1} and A8 [rows] int8 uniform over the five actions"""
    rng = np.random.default_rng(seed)
    S = rng.choice((-1.0, 0.0, 0.0, 1.0), (rows, 30)).astype(np.float32)
    A8 = rng.integers(0, NA, rows).astype(np.int8)
    return S, A8


def exact_index(n, rows, seed):
    """n row indices into [0, rows): unsorted, with duplicate entries and the last row of S (from n >= 3 on)"""
    rng = np.random.default_rng(seed)
    idx = rng.permutation(rows)[:n].astype(np.int64)
    if n >= 3:
        idx[rng.integers(0, n)] = rows - 1
        k = max(1, n // 50)
        idx[rng.choice(n, k, replace=False)] = idx[rng.choice(n, k, replace=False)]
    return idx


def exact_probe_actions(A8, idx, probes):
    """the rows at the positions `probes` of idx take action 4, outside every policy head's group (A8 changed in place)"""
    A8[np.asarray(idx, np.int64)[list(probes)]] = NA - 1


def exact_offsets(values, idx, probes, seed):
    """Per row of S: G = values (Q_ref or V_ref, float32) + an integer offset in {-2, -1, 1, 2} (0 on some rows) and
    the log-ratio shift of the rows pushed outside the clip range (to the side where PPO clips them: r = e > 1 + c with
    a positive advantage, r = 1/e < 1 - c with a negative one).  The rows at the positions `probes` of idx keep r == 1,
    a non-zero offset, so that each contributes to every kind's gradient (with `exact_probe_actions`).
    -> (G [rows] f32, shift [rows] f32: old_logp = target logp - shift)"""
    rng = np.random.default_rng(seed)
    rows = len(values)
    off = rng.choice((-2.0, -1.0, 0.0, 1.0, 2.0), rows)
    push = rng.random(rows) < 0.2
    probe_rows = np.asarray(idx, np.int64)[list(probes)]
    off[probe_rows] = np.where(rng.random(len(probe_rows)) < 0.5, -1.0, 2.0)
    push[probe_rows] = False
    push &= off != 0
    shift = np.where(push, np.sign(off) * PUSH, 0.0).astype(np.float32)
    G = (np.asarray(values, np.float64) + off).astype(np.float32)
    assert np.array_equal(G.astype(np.float64), np.asarray(values, np.float64) + off)
    return G, shift


def check_exact_case(kind, params, S, A8, G, old_logp, q_target, idx, clip=EXACT_CLIP):
    """learner_pass(fp16=True, check=True) plus the checks that the data exercises the kernel: ReLU masks mixed, all
    five actions among the rows, every policy row's p in {0, 1/group} and derivative -adv (r == 1) or 0 (clipped), and
    non-zero sums in every bias column (and the critic's one-hot columns).  -> the reference's result

    The exactness (learner_pass check=True) assumes a dyadic clip; 1 +- 0.2 differ between float32 and float64."""
    ref = learner_pass(kind, params, S, A8, G, old_logp, q_target, idx, clip, fp16=True, check=True)
    idx = np.asarray(idx, np.int64)
    a = np.asarray(A8)[idx]
    if len(idx) >= 128 and len(set(a.tolist())) != NA:
        raise Exactness("not all five actions occur")
    if len(idx) >= 16 and not all(0.1 < f < 0.9 for f in ref["active"]):
        raise Exactness("the ReLU masks are not mixed: active shares %s" % (ref["active"],))
    if kind != "critic":
        group = int(np.sum(np.asarray(params["fc3.bias" if kind == "actor" else "actor_linear.bias"]) == 0))
        if not np.all((ref["p"] == 0) | (ref["p"] == 1.0 / group)):
            raise Exactness("a policy row's probabilities are not in {0, 1/%d}" % group)
        gl, adv, ratio = ref["gl"], ref["adv"], ref["ratio"]
        one = ratio == 1
        if not (np.array_equal(gl[one], -adv[one].astype(np.float64)) and np.all(gl[~one] == 0)):
            raise Exactness("a policy row's derivative is neither -adv at r == 1 nor 0 when clipped")
    for name, s in ref["sums"].items():
        if name.endswith(".bias") and len(idx) >= 128 and not np.any(s != 0):
            raise Exactness("no contribution reaches %s" % name)
    if kind == "critic" and len(idx) >= 128 and not np.all(np.any(ref["sums"]["fc2.weight"][:, 128:] != 0, axis=0)):
        raise Exactness("a one-hot column of the critic receives no contribution")
    return ref

"""CPU tests of the device optimiser step (mm_rmsprop_step, rollout.DeviceRMSprop): the numpy float32 restatement of the
kernel (oracle/optim_ref.py) against torch's clip_grad_norm_ + torch.optim.RMSprop on the CPU, the argument checks of
the entry point, which reject bad calls before any CUDA call, and the hyperparameters DeviceRMSprop refuses."""
import ctypes as C

import numpy as np
import pytest
import torch

import optim_ref

STEPS = 6


def _net_params(kind, seed):
    from marl_mass_b200 import rollout
    torch.manual_seed(seed)
    net = {"actor": rollout.ActorNetwork, "critic": rollout.CriticNetwork, "shared": rollout.ActorCriticNetwork}[kind]()
    return [p.detach().clone() for p in net.parameters()]


def _ulps(a, b):
    """elementwise distance in float32 units in the last place (same-sign values)"""
    ia, ib = np.asarray(a, np.float32).view(np.int32).astype(np.int64), np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(ia - ib)


def _param_ulps(a, b):
    """distance in float32 ulp of the tensor's largest magnitude: a parameter that passes near zero inherits the
    rounding of the larger values it was summed from, which an elementwise ulp count would blow up"""
    return np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / np.spacing(np.float32(np.abs(b).max()))


def _run_both(params0, grad_fn, lr, max_norm, divisor=1):
    """STEPS steps of torch (grad / divisor as a float32 product, clip_grad_norm_, RMSprop single-tensor) and of the
    restatement from the same parameters and gradients -> per step (torch totals, oracle totals) and both final states"""
    scale = np.float32(1.0) / np.float32(divisor)
    tp = [torch.nn.Parameter(p.clone()) for p in params0]
    opt = torch.optim.RMSprop(tp, lr=lr, foreach=False)
    op = [p.numpy().copy() for p in params0]
    osq = [np.zeros_like(p) for p in op]
    totals = []
    for s in range(STEPS):
        gs = grad_fn(s)
        for p, g in zip(tp, gs):
            p.grad = g.clone().mul_(torch.tensor(scale))
        t_total = float(torch.nn.utils.clip_grad_norm_(tp, max_norm)) if max_norm else None
        t_grads = [p.grad.numpy().copy() for p in tp]
        opt.step()
        og = [g.numpy().copy() for g in gs]
        o_total = optim_ref.rmsprop_step(op, og, osq, lr, max_norm=max_norm, grad_scale=scale)
        totals.append((t_total, float(o_total), t_grads, og))
    tsq = [opt.state[p]["square_avg"].numpy() for p in tp]
    return totals, [p.detach().numpy() for p in tp], tsq, op, osq


@pytest.mark.parametrize("kind", ["actor", "critic", "shared"])
@pytest.mark.parametrize("case", ["clip_active", "clip_inactive", "no_clip", "zero_grads", "divisor_3"])
def test_restatement_matches_torch_clip_and_rmsprop(kind, case):
    """torch's CPU kernels fuse square_avg + (1 - alpha) * g * g into one FMA, the kernel and its restatement round each
    operation, so square_avg and parameters may differ by an ulp per step even with the clip coefficient 1; with clipping
    active the norm's summation order differs from torch's (per-tensor norms, then the norm of those), which moves the
    coefficient by a few ulp.  Totals within 1e-6 relative, clipped gradients within 4 ulp (bit for bit when the
    coefficient is 1), square_avg within 4 ulp per element per step, parameters within 4 ulp of their tensor's largest
    magnitude per step (`_param_ulps`)."""
    params0 = _net_params(kind, 1)
    gen = torch.Generator().manual_seed(2)
    scale = {"clip_active": 100.0, "zero_grads": 0.0}.get(case, 1e-3)
    max_norm = None if case == "no_clip" else 5.0
    divisor = 3 if case == "divisor_3" else 1
    grads = [[torch.randn(p.shape, generator=gen) * scale for p in params0] for _ in range(STEPS)]
    totals, tp, tsq, op, osq = _run_both(params0, lambda s: grads[s], 5e-4, max_norm, divisor)
    for t_total, o_total, t_grads, o_grads in totals:
        if t_total is not None:
            assert abs(o_total - t_total) <= 1e-6 * max(t_total, 1e-30), (t_total, o_total)
        if case == "clip_active":
            assert t_total > 5.0
        elif case != "no_clip":
            assert t_total < 5.0
        worst_g = max(int(_ulps(a, b).max()) for a, b in zip(t_grads, o_grads))
        assert worst_g <= (0 if case != "clip_active" else 4), worst_g
    u_sq = max(int(_ulps(a, b).max()) for a, b in zip(tsq, osq))
    u_p = max(float(_param_ulps(a, b).max()) for a, b in zip(tp, op))
    print("%s %s: square_avg %d ulp, parameters %.1f ulp after %d steps" % (kind, case, u_sq, u_p, STEPS))
    assert u_sq <= 4 * STEPS and u_p <= 4 * STEPS, (u_sq, u_p)
    if case == "zero_grads":      # the coefficient clamps to 1 and the parameters stay where they are
        for a, p0 in zip(op, params0):
            np.testing.assert_array_equal(a, p0.numpy())


def test_restatement_norm_order_and_mirror():
    """The restated norm is the documented order: per-thread sequential sums over a strided walk across the tensors,
    then two shfl_down trees; and the mirror writes every updated element at its dense position."""
    rng = np.random.default_rng(0)
    gs = [rng.normal(0, 1, n).astype(np.float32) for n in (700, 5, 1300)]
    acc = np.zeros(optim_ref.THREADS, np.float32)
    for g in gs:
        for i, x in enumerate(g):
            acc[i % optim_ref.THREADS] = np.float32(acc[i % optim_ref.THREADS] + np.float32(x * x))
    warps = []
    for w in range(optim_ref.THREADS // 32):
        v = acc[32 * w:32 * w + 32].copy()
        for off in (16, 8, 4, 2, 1):
            for lane in range(off):
                v[lane] = np.float32(v[lane] + v[lane + off])
        warps.append(v[0])
    v = np.array(warps + [0.0] * (32 - len(warps)), np.float32)
    for off in (16, 8, 4, 2, 1):
        for lane in range(off):
            v[lane] = np.float32(v[lane] + v[lane + off])
    assert optim_ref.group_norm(gs) == np.sqrt(v[0])
    # mirror: fc12's weight [64][10] at rows 32.. of a [160][30] layer, columns COLS2
    from marl_mass_b200.rollout import ActorCriticNetwork
    p = rng.normal(0, 1, (64, 10)).astype(np.float32)
    dense = np.zeros((160, 30), np.float32)
    optim_ref.rmsprop_step([p], [np.ones_like(p)], [np.zeros_like(p)], 1e-2, mirrors=[(0, dense, 32, ActorCriticNetwork.COLS2)])
    np.testing.assert_array_equal(dense[32:96][:, list(ActorCriticNetwork.COLS2)], p)
    assert np.count_nonzero(dense) == p.size


@pytest.fixture(scope="module")
def L():
    import marl_mass_b200 as mm
    from marl_mass_b200 import build
    build.build()
    return mm.lib()


def test_rmsprop_entry_point_rejects_bad_arguments_before_any_cuda_call(L):
    from marl_mass_b200 import _lib
    cols = (C.c_int32 * 5)(0, 5, 10, 15, 20)

    def table(n=2, **kw):
        ts = (_lib.MMOptTensor * max(n, 1))()
        for k in range(max(n, 1)):
            ts[k].param, ts[k].grad, ts[k].square_avg, ts[k].numel = 0x1000 * (k + 1), 0x2000 * (k + 1), 0x3000 * (k + 1), 160
        for f, v in kw.items():
            setattr(ts[0], f, v)
        return ts

    def group(ts, n=2, **kw):
        g = _lib.MMOptGroup(ts, n, 5e-4, 0.99, 0.01, 1e-8, 5.0, 1.0, None)
        for f, v in kw.items():
            setattr(g, f, v)
        return g

    def call(groups, n=None):
        arr = (_lib.MMOptGroup * max(len(groups), 1))(*groups)
        return L.mm_rmsprop_step(None if groups is None else arr, len(groups) if n is None else n, None)

    def rejected(rc, what):
        assert rc == -1, (rc, what)
        assert what in L.mm_last_error().decode(), L.mm_last_error()

    rejected(L.mm_rmsprop_step(None, 1, None), "groups is null")
    rejected(call([group(table())], n=0), "n_groups")
    rejected(call([group(table())], n=-1), "n_groups")
    rejected(call([group(table())] * 9), "n_groups")
    rejected(call([group(None)]), "tensors is null")
    rejected(call([group(table(), n=0)]), "n_tensors")
    rejected(call([group(table(17), n=17)]), "n_tensors")
    rejected(call([group(table(), n=-3)]), "n_tensors")
    for f in ("param", "grad", "square_avg"):
        rejected(call([group(table(**{f: None}))]), "param, grad and square_avg are required")
    rejected(call([group(table(), n=2), group(table(grad=None))]), "are required")      # a bad second group
    rejected(call([group(table(numel=-1))]), "numel must be >= 0")
    rejected(call([group(table(mirror=0x9000))]), "column map")                        # a mirror without a map
    rejected(call([group(table(mirror=0x9000, mirror_cols=cols, mirror_ncols=0, mirror_ld=30))]), "column map")
    rejected(call([group(table(mirror=0x9000, mirror_cols=cols, mirror_ncols=17, mirror_ld=30))]), "column map")
    rejected(call([group(table(mirror=0x9000, mirror_cols=cols, mirror_ncols=5, mirror_ld=0))]), "mirror_ld")
    rejected(call([group(table(mirror=0x9000, mirror_cols=cols, mirror_ncols=5, mirror_ld=-30))]), "mirror_ld")
    rejected(call([group(table(mirror=0x9000, mirror_cols=cols, mirror_ncols=5, mirror_ld=30, numel=162))]), "multiple")
    rejected(call([group(table(mirror=0x9000, mirror_cols=cols, mirror_ncols=5, mirror_ld=20))]), "mirror_cols must lie")
    bad = (C.c_int32 * 5)(0, 5, -1, 15, 20)
    rejected(call([group(table(mirror=0x9000, mirror_cols=bad, mirror_ncols=5, mirror_ld=30))]), "mirror_cols must lie")
    assert _lib.ABI_VERSION == 9 and L.mm_abi_version() == 9


def test_device_rmsprop_rejects_unsupported_hyperparameters():
    from marl_mass_b200.rollout import DeviceRMSprop
    p = [torch.nn.Parameter(torch.zeros(3))]
    for kw in ({"momentum": 0.9}, {"centered": True}, {"weight_decay": 1e-4}):
        with pytest.raises(ValueError, match="momentum, centered and weight_decay"):
            DeviceRMSprop(p, lr=1e-3, **kw)
    for kw in ({"lr": -1.0}, {"lr": 1e-3, "alpha": 1.5}, {"lr": 1e-3, "eps": -1.0}):
        with pytest.raises(ValueError, match="invalid"):
            DeviceRMSprop(p, **kw)
    with pytest.raises(ValueError, match="CUDA"):        # CPU parameters: no kernel to step them with
        DeviceRMSprop(p, lr=1e-3)

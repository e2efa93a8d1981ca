"""numpy float32 restatement of the device optimiser step (mm_rmsprop_step, marl-mass_b200/csrc/optim.cu):
torch.nn.utils.clip_grad_norm_ followed by torch.optim.RMSprop (no momentum, not centred, no weight decay) for one group
of parameter tensors, with the kernel's summation order for the norm and its order of operations, every operation
rounded to float32.

Norm order: thread t of THREADS walks the tensors in order and, within a tensor, the elements t, t + THREADS, ...,
adding g * g to one float32 accumulator; lane sums of a warp: shfl_down at offsets 16, 8, 4, 2, 1 (lane 0 keeps the
sum); the THREADS / 32 warp sums, padded with zeros to 32, the same way.  total = sqrt(sum)."""
import numpy as np

THREADS = 512
f32 = np.float32


def _warp_tree(v):
    """v [..., 32] -> lane 0 after v[i] += v[i + off] for off = 16, 8, 4, 2, 1"""
    v = v.copy()
    for off in (16, 8, 4, 2, 1):
        v[..., :off] = v[..., :off] + v[..., off:2 * off]
    return v[..., 0]


def group_norm(grads):
    """the kernel's float32 2-norm of the concatenated (already scaled) gradients"""
    acc = np.zeros(THREADS, f32)
    for g in grads:
        g = np.asarray(g, f32).ravel()
        pad = np.zeros(-(-g.size // THREADS) * THREADS, f32)
        pad[:g.size] = g
        for row in pad.reshape(-1, THREADS):       # zeros past the end add nothing: acc + 0 * 0 == acc
            acc = acc + row * row
    warps = _warp_tree(acc.reshape(THREADS // 32, 32))
    return np.sqrt(_warp_tree(np.concatenate([warps, np.zeros(32 - warps.size, f32)])))


def clip_coef(total, max_norm):
    """clip_grad_norm_'s coefficient as torch evaluates it: reciprocal(total + 1e-6) * max_norm, clamped to 1"""
    if not max_norm or max_norm <= 0:
        return f32(1.0)
    c = (f32(1.0) / (f32(total) + f32(1e-6))) * f32(max_norm)
    return f32(1.0) if c > 1 else c


def rmsprop_step(params, grads, square_avgs, lr, alpha=0.99, eps=1e-8, max_norm=None, grad_scale=1.0, mirrors=()):
    """One step of the group, in place on float32 arrays: grads become the scaled, clipped gradients, params and
    square_avgs their RMSprop update.  lr, alpha, eps, max_norm as the Python floats torch is given (rounded to float32
    as torch rounds scalars; 1 - alpha in double first); grad_scale a float32 factor (1 / world for a data-parallel
    average).  mirrors: (tensor index, dest array [rows, ld], row offset, column map) - the dense first layer the kernel
    keeps in step.  -> total (float32, before clipping)"""
    scale = f32(grad_scale)
    for g in grads:
        g *= scale
    total = group_norm(grads)
    coef = clip_coef(total, max_norm)
    a, oma, e, neg_lr = f32(alpha), f32(1.0 - alpha), f32(eps), -f32(lr)
    for p, g, sq in zip(params, grads, square_avgs):
        g *= coef
        sq *= a
        sq += (oma * g) * g
        avg = np.sqrt(sq) + e
        p += neg_lr * (g / avg)
    for k, dst, row0, cols in mirrors:
        p = params[k].reshape(-1, len(cols))
        dst[row0:row0 + p.shape[0], list(cols)] = p
    return f32(total)

// optim.cu — the learner's optimiser step on the device: clip_grad_norm_ + torch.optim.RMSprop (alpha, eps, no momentum,
// not centred, no weight decay) for whole networks, one CTA per network ("group").
//
// Order of the gradient norm (the numpy restatement the tests use repeats it): thread t of the group's OPT_THREADS threads walks the
// group's tensors in table order and, within tensor k, the elements i = t, t + OPT_THREADS, ...; it adds each g * g to one
// float accumulator (each product and sum rounded: the library builds with -fmad=false).  The 32 lanes of a warp then add
// with shfl_down at offsets 16, 8, 4, 2, 1 (lane 0 keeps the warp sum); warp 0 does the same over the OPT_THREADS / 32 warp
// sums, padded with zeros to 32.  total = sqrtf(sum).  Fixed order, no atomics: the step is deterministic.
#include <cuda_runtime.h>

#include "mm_internal.h"

namespace mm {
namespace {

constexpr int OPT_THREADS = 512;

struct OptTensorK {
    float *p, *g, *sq, *mirror;
    int64_t numel, ld;
    int ncols;
    uint8_t cols[MM_OPT_MAX_MIRROR_COLS];
};

struct OptGroupK {
    OptTensorK t[MM_OPT_MAX_TENSORS];
    int n;
    float lr, alpha, one_minus_alpha, eps, max_norm, grad_scale;
    float *total;
};

struct OptLaunchK {
    OptGroupK g[MM_OPT_MAX_GROUPS];
};

__device__ __forceinline__ float warp_sum_down(float v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v = v + __shfl_down_sync(0xffffffffu, v, off);
    return v;
}

__global__ void __launch_bounds__(OPT_THREADS) rmsprop_kernel(const __grid_constant__ OptLaunchK L) {
    const OptGroupK &G = L.g[blockIdx.x];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    __shared__ float part[OPT_THREADS / 32];
    __shared__ float coef_s;

    // 1. scale and norm: torch.nn.utils.clip_grad_norm_ sees the gradients after the data-parallel average
    float acc = 0.f;
    for (int k = 0; k < G.n; ++k) {
        const OptTensorK &e = G.t[k];
        for (int64_t i = t; i < e.numel; i += OPT_THREADS) {
            const float g = e.g[i] * G.grad_scale;
            acc = acc + g * g;
        }
    }
    acc = warp_sum_down(acc);
    if (lane == 0) part[warp] = acc;
    __syncthreads();
    if (warp == 0) {
        float v = lane < OPT_THREADS / 32 ? part[lane] : 0.f;
        v = warp_sum_down(v);
        if (lane == 0) {
            const float total = sqrtf(v);
            // clip_grad_norm_: clip_coef = max_norm / (total + 1e-6), a python float over a tensor, which torch evaluates as
            // reciprocal(total + 1e-6) * max_norm; clamp(max=1) keeps a NaN
            float c = 1.f;
            if (G.max_norm > 0.f) {
                c = (1.f / (total + 1e-6f)) * G.max_norm;
                c = c > 1.f ? 1.f : c;
            }
            coef_s = c;
            if (G.total) *G.total = total;
        }
    }
    __syncthreads();
    const float coef = coef_s, neg_lr = -G.lr;

    // 2. clip (always multiplied, as torch does), then RMSprop with torch's order of operations
    for (int k = 0; k < G.n; ++k) {
        const OptTensorK &e = G.t[k];
        for (int64_t i = t; i < e.numel; i += OPT_THREADS) {
            const float g = (e.g[i] * G.grad_scale) * coef;
            e.g[i] = g;
            float sq = e.sq[i] * G.alpha;                   // square_avg.mul_(alpha)
            sq = sq + (G.one_minus_alpha * g) * g;          // .addcmul_(grad, grad, value=1 - alpha)
            e.sq[i] = sq;
            const float avg = sqrtf(sq) + G.eps;            // square_avg.sqrt().add_(eps)
            const float p = e.p[i] + neg_lr * (g / avg);    // param.addcdiv_(grad, avg, value=-lr)
            e.p[i] = p;
            if (e.mirror) {
                const int64_t r = i / e.ncols, c = i - r * e.ncols;
                e.mirror[r * e.ld + e.cols[c]] = p;
            }
        }
    }
}

}  // namespace

int launch_rmsprop_step(const mm_opt_group *groups, int n_groups, void *stream) {
    OptLaunchK L;
    for (int gi = 0; gi < n_groups; ++gi) {
        const mm_opt_group &src = groups[gi];
        OptGroupK &G = L.g[gi];
        G.n = src.n_tensors;
        G.lr = src.lr;
        G.alpha = src.alpha;
        G.one_minus_alpha = src.one_minus_alpha;
        G.eps = src.eps;
        G.max_norm = src.max_norm;
        G.grad_scale = src.grad_scale;
        G.total = src.total_norm;
        for (int k = 0; k < src.n_tensors; ++k) {
            const mm_opt_tensor &s = src.tensors[k];
            OptTensorK &e = G.t[k];
            e.p = s.param;
            e.g = s.grad;
            e.sq = s.square_avg;
            e.numel = s.numel;
            e.mirror = s.mirror;
            e.ld = s.mirror ? s.mirror_ld : 0;
            e.ncols = s.mirror ? s.mirror_ncols : 1;
            for (int c = 0; c < MM_OPT_MAX_MIRROR_COLS; ++c) e.cols[c] = (s.mirror && c < s.mirror_ncols) ? (uint8_t)s.mirror_cols[c] : 0;
        }
    }
    rmsprop_kernel<<<(unsigned)n_groups, OPT_THREADS, 0, (cudaStream_t)stream>>>(L);
    return cudaGetLastError() != cudaSuccess;
}

}  // namespace mm

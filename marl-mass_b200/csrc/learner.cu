// learner.cu — the PPO update of MAPPO / MAPPO_GI on the device: forward, per-row loss and backward of the reference's
// networks fused per 128-row tile, weight gradients summed per CTA and reduced in a fixed order.
//
// Reference: marl/mappo.py:161-206 (MAPPO.train), marl/mappo_gi.py:307-349 (MAPPO_GI.train, shared branch), batched as
// rollout.mappo_losses / rollout.shared_network_loss with the per-sample surrogate and the MSE critic loss.  The torch
// learner runs every minibatch through dozens of launches and recomputes the target networks each time; here
//   * ppo_kernel<KIND, false> (the target pass, once per update) writes the per-row constants of the update: the target
//     log-probability of the taken action (actor, shared network) or Q_target(s, a) (critic);
//   * ppo_kernel<KIND, true> (the gradient pass, once per minibatch) gathers its rows through the index list, runs the
//     forward with the same code as the target pass (so r == 1 exactly where the network equals its target), the per-row
//     loss derivative and the backward, and accumulates the weight gradients of its tiles in registers;
//   * ppo_reduce_kernel sums the CTA partials in CTA order and applies 1/N: no float atomics anywhere, two calls with
//     the same inputs give bit-identical gradients;
//   * ppo_kernel<KIND, false, true> (the statistics pass, mm_ppo_stats) runs the same forward over listed rows and sums
//     per-row diagnostics (entropy, ratio to old_logp, value against the return) in f64 per CTA, and
//     ppo_stats_reduce_kernel adds the CTA partials in CTA order.
//
// Network kinds (torch Linear layout: weight [out][in], bias [out]):
//   ACTOR   ActorNetwork   30 -> 128 -> 128 -> 5, log-softmax
//   CRITIC  CriticNetwork  30 -> 128, [h1, one_hot(a)] 133 -> 128, 128 -> 1
//   SHARED  ActorCriticNetwork (state_split): the three first-layer blocks as one dense 30 -> 160 layer (zero outside the
//           blocks, as rollout._split_first_layer builds it for the draw), 160 -> 128, actor_linear 5 + critic_linear 1
//
// Math: warp-level mma.sync m16n8k16, fp16 operands, fp32 accumulation; biases, log-softmax and the loss in fp32.  A
// warp owns 16 rows of the tile for the forward and for the backward down to dZ (row-local), the CTA's 8 warps share the
// weight-gradient products dW^T = dZ^T . [act | 1] (K = the tile's 128 rows), whose operands are the row-major tiles
// already in shared memory, read transposed by ldmatrix.trans.  Bias gradients ride in the same products through a
// column of ones appended to each activation tile (and the critic's one-hot action through extra columns of h1).
// Per-row values entering fp16 (g * (e_a - p), 2 (Q - G)) are O(1..100); the 1/N stays out of them (it would push them
// below fp16's normal range at N = 2^18) and is applied by the reduction in fp32.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <mutex>
#include "mm_internal.h"

namespace mm {

namespace {

constexpr int LT = 256;               // threads per CTA (8 warps x 16 rows)
constexpr int LROWS = 128;            // rows per tile
constexpr int SX = 40;                // stride (halves) of the input tile [row][32 + pad]: 30 features, a ones column at 30
constexpr int NA = MM_NA;

template <int KIND> struct LK;
template <> struct LK<MM_PPO_ACTOR> { static constexpr int H1 = 128, IN2 = 128, OUT3 = 5; };
template <> struct LK<MM_PPO_CRITIC> { static constexpr int H1 = 128, IN2 = 133, OUT3 = 1; };
template <> struct LK<MM_PPO_SHARED> { static constexpr int H1 = 160, IN2 = 160, OUT3 = 6; };

template <int KIND> struct LG {
    static constexpr int H1 = LK<KIND>::H1, IN2 = LK<KIND>::IN2, OUT3 = LK<KIND>::OUT3;
    static constexpr int K2 = (IN2 + 15) / 16 * 16;          // forward K of layer 2 (h1 plus the critic's one-hot)
    static constexpr int N2G = (IN2 + 1 + 7) / 8 * 8;        // columns of the layer-2 weight gradient (ones column at IN2)
    static constexpr int SB0 = (K2 > N2G ? K2 : N2G) + 8;
    static constexpr int SB = ((SB0 / 8) % 2) ? SB0 : SB0 + 8;   // activation stride (halves): 8 x odd = conflict-free ldmatrix
    static constexpr int S3 = 136;                            // W3 [16][136]; h2 columns 0..127, ones at 128
    // partials per CTA (floats): dW1aug [H1][32], dW2aug [128][N2G], dW3aug [16][136], 2 loss sums
    static constexpr int P1 = 0, P2 = P1 + H1 * 32, P3 = P2 + 128 * N2G, PL = P3 + 16 * S3, P = (PL + 2 + 31) / 32 * 32;
    // shared memory (bytes)
    static constexpr uint32_t W1S = 0;                                   // [H1][SX] f16
    static constexpr uint32_t W2S = W1S + H1 * SX * 2;                   // [128][SB] f16
    static constexpr uint32_t W3S = W2S + 128 * SB * 2;                  // [16][S3] f16
    static constexpr uint32_t XS = W3S + 16 * S3 * 2;                    // [128][SX] f16
    static constexpr uint32_t H1S = XS + LROWS * SX * 2;                 // [128][SB] f16: h1 | one-hot | 1
    static constexpr uint32_t H2S = H1S + LROWS * SB * 2;                // [128][SB] f16: h2 | 1; later dZ1
    static constexpr uint32_t DZ2S = H2S + LROWS * SB * 2;               // [128][SB] f16
    static constexpr uint32_t DZ3S = DZ2S + LROWS * SB * 2;              // [128][24] f16
    static constexpr uint32_t B1S = DZ3S + LROWS * 24 * 2;               // f32 [H1]
    static constexpr uint32_t B2S = B1S + H1 * 4;                        // f32 [128]
    static constexpr uint32_t B3S = B2S + 128 * 4;                       // f32 [8]
    static constexpr uint32_t RG = B3S + 8 * 4;                          // i64 [128] source row (-1: padding)
    static constexpr uint32_t RA = RG + LROWS * 8;                       // i32 [128] action
    static constexpr uint32_t RF = RA + LROWS * 4;                       // f32 [3][128] return, old logp, q target
    static constexpr uint32_t RED = RF + 3 * LROWS * 4;                  // f32 [8][2] loss sums per warp
    static constexpr uint32_t SMEM = RED + 16 * 4;
};
static_assert(LG<MM_PPO_SHARED>::SMEM <= 227 * 1024, "learner shared memory");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], uint32_t a) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
}
__device__ __forceinline__ void ldsm4t(uint32_t (&r)[4], uint32_t a) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a) : "memory");
}
__device__ __forceinline__ void ldsm2(uint32_t (&r)[2], uint32_t a) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a) : "memory");
}
__device__ __forceinline__ void ldsm2t(uint32_t (&r)[2], uint32_t a) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(a) : "memory");
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t h2u(__half2 h) { return *reinterpret_cast<uint32_t *>(&h); }

// Row-local product of one warp: acc[NT] (+)= A[16 rows][16 KS] . B, A row-major at a (stride sa halves), columns n0..
// B_T = false: B given as W [n][k] (stride sb) - the forward x . W^T;  B_T = true: B given as W [k][n] - the backward dZ . W.
template <int NT, int KS, bool B_T>
__device__ __forceinline__ void row_gemm(float (&acc)[NT][4], uint32_t a, int sa, uint32_t b, int sb, int n0, int lane) {
    const uint32_t a_l = a + (uint32_t)((((lane & 7) + ((lane >> 3) & 1) * 8) * sa + ((lane >> 4) & 1) * 8) * 2);
    uint32_t b_l;
    if (B_T) b_l = b + (uint32_t)((((lane & 7) + ((lane >> 3) & 1) * 8) * sb + n0 + ((lane >> 4) & 1) * 8) * 2);
    else b_l = b + (uint32_t)(((n0 + (lane & 7) + ((lane >> 4) & 1) * 8) * sb + ((lane >> 3) & 1) * 8) * 2);
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
        uint32_t af[4];
        ldsm4(af, a_l + ks * 32);
#pragma unroll
        for (int j = 0; j + 1 < NT; j += 2) {
            uint32_t bf[4];
            if (B_T) ldsm4t(bf, b_l + (uint32_t)((ks * 16 * sb + j * 8) * 2));
            else ldsm4(bf, b_l + (uint32_t)((j * 8 * sb + ks * 16) * 2));
            mma16816(acc[j], af, bf[0], bf[1]);
            mma16816(acc[j + 1], af, bf[2], bf[3]);
        }
        if (NT & 1) {
            uint32_t bf[2];
            if (B_T) ldsm2t(bf, b_l + (uint32_t)((ks * 16 * sb + (NT - 1) * 8) * 2));
            else ldsm2(bf, b_l + (uint32_t)(((NT - 1) * 8 * sb + ks * 16) * 2));
            mma16816(acc[NT - 1], af, bf[0], bf[1]);
        }
    }
}

// Weight-gradient product over the tile's 128 rows: acc[NT] += A^T . B with A stored [row][m] (columns m0..m0+15) and
// B stored [row][n] (columns n0..n0+8 NT), both read transposed.
template <int NT>
__device__ __forceinline__ void wgrad_gemm(float (&acc)[NT][4], uint32_t a, int sa, int m0, uint32_t b, int sb, int n0, int lane) {
    const uint32_t a_l = a + (uint32_t)((((lane & 7) + ((lane >> 4) & 1) * 8) * sa + m0 + ((lane >> 3) & 1) * 8) * 2);
    const uint32_t b_l = b + (uint32_t)((((lane & 7) + ((lane >> 3) & 1) * 8) * sb + n0 + ((lane >> 4) & 1) * 8) * 2);
#pragma unroll 2
    for (int ks = 0; ks < LROWS / 16; ++ks) {
        uint32_t af[4];
        ldsm4t(af, a_l + (uint32_t)(ks * 16 * sa * 2));
#pragma unroll
        for (int j = 0; j + 1 < NT; j += 2) {
            uint32_t bf[4];
            ldsm4t(bf, b_l + (uint32_t)((ks * 16 * sb + j * 8) * 2));
            mma16816(acc[j], af, bf[0], bf[1]);
            mma16816(acc[j + 1], af, bf[2], bf[3]);
        }
        if (NT & 1) {
            uint32_t bf[2];
            ldsm2t(bf, b_l + (uint32_t)((ks * 16 * sb + (NT - 1) * 8) * 2));
            mma16816(acc[NT - 1], af, bf[0], bf[1]);
        }
    }
}

template <int NT> __device__ __forceinline__ void zero(float (&acc)[NT][4]) {
#pragma unroll
    for (int j = 0; j < NT; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
}

// accumulator (rows g, g+8 of the warp's 16; columns n0 + 8j + 2t, +1) -> relu(acc + bias) as f16 at dst[row][col]
template <int NT>
__device__ __forceinline__ void store_relu(const float (&acc)[NT][4], const float *bias, __half *dst, int sd, int row0, int n0, int g,
                                           int t) {
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        const int c = n0 + 8 * j + 2 * t;
        const float b0 = bias[c], b1 = bias[c + 1];
        *reinterpret_cast<__half2 *>(dst + (row0 + g) * sd + c) = __floats2half2_rn(fmaxf(acc[j][0] + b0, 0.f), fmaxf(acc[j][1] + b1, 0.f));
        *reinterpret_cast<__half2 *>(dst + (row0 + g + 8) * sd + c) = __floats2half2_rn(fmaxf(acc[j][2] + b0, 0.f), fmaxf(acc[j][3] + b1, 0.f));
    }
}

// accumulator dH -> dZ = dH where the layer's ReLU output (act) is positive, as f16 at dst
template <int NT>
__device__ __forceinline__ void store_masked(const float (&acc)[NT][4], const __half *act, int sact, __half *dst, int sd, int row0, int n0,
                                             int g, int t) {
#pragma unroll
    for (int j = 0; j < NT; ++j) {
        const int c = n0 + 8 * j + 2 * t;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int r = row0 + g + 8 * h;
            const float2 m = __half22float2(*reinterpret_cast<const __half2 *>(act + r * sact + c));
            *reinterpret_cast<__half2 *>(dst + r * sd + c) =
                __floats2half2_rn(m.x > 0.f ? acc[j][2 * h] : 0.f, m.y > 0.f ? acc[j][2 * h + 1] : 0.f);
        }
    }
}

// The per-row derivative of the PPO-clip term -min(r adv, clamp(r, 1 - c, 1 + c) adv) with respect to log p(a), with
// torch autograd's rules: min splits the gradient half / half at a tie, clamp passes it at its bounds (inclusive), and
// d r / d logp = r.  The numpy restatement next to the other reference restatements pins this against torch autograd.
__device__ __forceinline__ float ppo_row(float r, float adv, float clip, float &loss) {
    const float lo = 1.0f - clip, hi = 1.0f + clip;
    const float s1 = r * adv, s2 = fminf(fmaxf(r, lo), hi) * adv;
    loss = -fminf(s1, s2);
    const float w1 = s1 < s2 ? 1.0f : (s1 == s2 ? 0.5f : 0.0f), w2 = 1.0f - w1;
    const float inside = (r >= lo && r <= hi) ? 1.0f : 0.0f;
    const float d_r = -(w1 * adv + w2 * (adv * inside));
    return d_r * r;
}

// statistics partials per CTA: the MM_PPO_STAT_* fields as f64, RATIO_MIN / RATIO_MAX included
constexpr int NSTAT = MM_PPO_STATS_LEN;

// The three passes over listed rows are one kernel, so that they run the same forward arithmetic:
//   <KIND, false>        the target pass: writes the per-row constants (old_logp_out / q_target_out; the shared network
//                        writes V(s) to q_target_out when it is non-null)
//   <KIND, true>         the gradient pass: adds the loss and the backward, weight-gradient partials per CTA
//   <KIND, false, true>  the statistics pass: reduces per-row diagnostics (entropy, ratio, value fit) into NSTAT f64
//                        partials per CTA, written through `partials` (old_logp_in nullable: no ratio)
// STATS is a trailing defaulted parameter so that the target and gradient passes compile exactly as they did without it.
template <int KIND, bool GRAD, bool STATS = false>
__global__ void __launch_bounds__(LT, 1)
ppo_kernel(const float *__restrict__ states, const int8_t *__restrict__ actions, const float *__restrict__ returns,
           const float *__restrict__ old_logp_in, const float *__restrict__ q_target_in, const int64_t *__restrict__ idx, int64_t n,
           float clip, mm_ppo_net net, float *__restrict__ old_logp_out, float *__restrict__ q_target_out, float *__restrict__ partials) {
    static_assert(!(GRAD && STATS), "one pass at a time");
    using L = LG<KIND>;
    constexpr int H1 = L::H1, IN2 = L::IN2, OUT3 = L::OUT3, SB = L::SB, S3 = L::S3, N2T = L::N2G / 8;
    extern __shared__ __align__(16) unsigned char lsm[];
    __half *w1s = reinterpret_cast<__half *>(lsm + L::W1S), *w2s = reinterpret_cast<__half *>(lsm + L::W2S);
    __half *w3s = reinterpret_cast<__half *>(lsm + L::W3S), *xs = reinterpret_cast<__half *>(lsm + L::XS);
    __half *h1s = reinterpret_cast<__half *>(lsm + L::H1S), *h2s = reinterpret_cast<__half *>(lsm + L::H2S);
    __half *dz2s = reinterpret_cast<__half *>(lsm + L::DZ2S), *dz3s = reinterpret_cast<__half *>(lsm + L::DZ3S);
    float *b1s = reinterpret_cast<float *>(lsm + L::B1S), *b2s = reinterpret_cast<float *>(lsm + L::B2S);
    float *b3s = reinterpret_cast<float *>(lsm + L::B3S);
    int64_t *rg = reinterpret_cast<int64_t *>(lsm + L::RG);
    int32_t *ra = reinterpret_cast<int32_t *>(lsm + L::RA);
    float *rf = reinterpret_cast<float *>(lsm + L::RF);
    float *red = reinterpret_cast<float *>(lsm + L::RED);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3, row0 = warp * 16;

    // weights as fp16 in the layouts the products read, zero padding; constant columns of the activation tiles
    for (int e = tid; e < H1 * SX; e += LT) {
        const int o = e / SX, i = e % SX;
        w1s[e] = __float2half_rn(i < NS ? net.w1[o * NS + i] : 0.f);
    }
    for (int e = tid; e < 128 * SB; e += LT) {
        const int o = e / SB, i = e % SB;
        w2s[e] = __float2half_rn(i < IN2 ? net.w2[o * IN2 + i] : 0.f);
    }
    for (int e = tid; e < 16 * S3; e += LT) {
        const int o = e / S3, i = e % S3;
        float v = 0.f;
        if (i < 128 && o < OUT3) v = (KIND == MM_PPO_SHARED && o == 5) ? net.w4[i] : net.w3[o * 128 + i];
        w3s[e] = __float2half_rn(v);
    }
    for (int e = tid; e < H1; e += LT) b1s[e] = net.b1[e];
    if (tid < 128) b2s[tid] = net.b2[tid];
    if (tid < 8) b3s[tid] = tid < OUT3 ? ((KIND == MM_PPO_SHARED && tid == 5) ? net.b4[0] : net.b3[tid]) : 0.f;
    for (int e = tid; e < LROWS * (SX - NS); e += LT) {
        const int r = e / (SX - NS), i = NS + e % (SX - NS);
        xs[r * SX + i] = __float2half_rn(i == NS ? 1.f : 0.f);
    }
    for (int e = tid; e < LROWS * (SB - H1); e += LT) {
        const int r = e / (SB - H1), i = H1 + e % (SB - H1);
        h1s[r * SB + i] = __float2half_rn(i == IN2 ? 1.f : 0.f);
    }
    for (int e = tid; e < LROWS * 24; e += LT) dz3s[e] = __float2half_rn(0.f);
    __syncthreads();

    const uint32_t w1a = smem_u32(w1s), w2a = smem_u32(w2s), w3a = smem_u32(w3s), xa = smem_u32(xs), h1a = smem_u32(h1s);
    const uint32_t h2a = smem_u32(h2s), dz2a = smem_u32(dz2s), dz3a = smem_u32(dz3s);

    // per-CTA weight-gradient accumulators: dW2 rows 16 warp.. (all N2T column tiles); dW3 column tiles warp, warp + 8,
    // warp + 16; dW1 rows 16 warp.. (4 column tiles) and, for H1 = 160, one tile of rows 128..159
    float g2[N2T][4], g3[3][1][4], g1[4][4], g1x[1][4];
    zero(g2); zero(g3[0]); zero(g3[1]); zero(g3[2]); zero(g1); zero(g1x);
    float loss_a = 0.f, loss_c = 0.f;
    // statistics pass: this thread's rows, in tile order (f64 sums, f32 ratio range)
    double st[NSTAT];
#pragma unroll
    for (int f = 0; f < NSTAT; ++f) st[f] = 0.0;
    float r_min = __int_as_float(0x7f800000), r_max = -__int_as_float(0x7f800000);
    const bool with_ratio = STATS && KIND != MM_PPO_CRITIC && old_logp_in != nullptr;

    const int64_t n_tiles = (n + LROWS - 1) / LROWS;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // ---- gather of the warp's 16 rows (two lanes per row, 15 features each) and their per-row constants
        {
            const int r = row0 + (lane >> 1), half = lane & 1;
            const int64_t i = tile * LROWS + r;
            const int64_t src = i < n ? idx[i] : -1;
            const float *s = states + (src < 0 ? 0 : src) * NS + 15 * half;
#pragma unroll
            for (int k = 0; k < 15; ++k) xs[r * SX + 15 * half + k] = __float2half_rn(src < 0 ? 0.f : s[k]);
            if (!half) {
                const int a = src < 0 ? 0 : (int)actions[src];
                rg[r] = src;
                ra[r] = a;
                if (GRAD) {
                    rf[r] = src < 0 ? 0.f : returns[src];
                    rf[LROWS + r] = (src < 0 || KIND == MM_PPO_CRITIC) ? 0.f : old_logp_in[src];
                    rf[2 * LROWS + r] = (src < 0 || KIND != MM_PPO_ACTOR) ? 0.f : q_target_in[src];
                }
                if (STATS) {
                    rf[r] = (src < 0 || KIND == MM_PPO_ACTOR) ? 0.f : returns[src];
                    rf[LROWS + r] = (src < 0 || !with_ratio) ? 0.f : old_logp_in[src];
                }
                if (KIND == MM_PPO_CRITIC) {
#pragma unroll
                    for (int k = 0; k < NA; ++k) h1s[r * SB + 128 + k] = __float2half_rn(k == a ? 1.f : 0.f);
                }
            } else if (GRAD) {
#pragma unroll
                for (int k = 0; k < 8; ++k) h2s[r * SB + 128 + k] = __float2half_rn(k == 0 ? 1.f : 0.f);
            }
        }
        __syncwarp();

        // ---- forward, row-local: h1 = relu(x W1^T + b1), h2 = relu([h1 | a] W2^T + b2), z3 = h2 W3^T + b3
#pragma unroll
        for (int n0 = 0; n0 + 64 <= H1; n0 += 64) {
            float acc[8][4];
            zero(acc);
            row_gemm<8, 2, false>(acc, xa + row0 * SX * 2, SX, w1a, SX, n0, lane);
            store_relu(acc, b1s, h1s, SB, row0, n0, g, t);
        }
        if constexpr (H1 % 64 != 0) {
            float acc[(H1 % 64) / 8][4];
            zero(acc);
            row_gemm<(H1 % 64) / 8, 2, false>(acc, xa + row0 * SX * 2, SX, w1a, SX, H1 - H1 % 64, lane);
            store_relu(acc, b1s, h1s, SB, row0, H1 - H1 % 64, g, t);
        }
        __syncwarp();
#pragma unroll
        for (int n0 = 0; n0 < 128; n0 += 64) {
            float acc[8][4];
            zero(acc);
            row_gemm<8, L::K2 / 16, false>(acc, h1a + row0 * SB * 2, SB, w2a, SB, n0, lane);
            store_relu(acc, b2s, h2s, SB, row0, n0, g, t);
        }
        __syncwarp();
        float z3[1][4];
        zero(z3);
        row_gemm<1, 8, false>(z3, h2a + row0 * SB * 2, SB, w3a, S3, 0, lane);

        // ---- per row: thread t = 0 finishes row g, t = 1 row g + 8 (the quad's other threads idle here)
        {
            const unsigned full = 0xffffffffu;
            const int q0 = lane & ~3;
            float zl[8], zh[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int src = q0 + (k >> 1);
                const float lo_e = __shfl_sync(full, z3[0][0], src), lo_o = __shfl_sync(full, z3[0][1], src);
                const float hi_e = __shfl_sync(full, z3[0][2], src), hi_o = __shfl_sync(full, z3[0][3], src);
                zl[k] = (k & 1) ? lo_o : lo_e;
                zh[k] = (k & 1) ? hi_o : hi_e;
            }
            if (t < 2) {
                const int r = row0 + g + 8 * t;
                const int64_t src = rg[r];
                const int a = ra[r];
                float z[8], dz[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { z[k] = (t ? zh[k] : zl[k]) + b3s[k]; dz[k] = 0.f; }
                if (KIND != MM_PPO_CRITIC) {
                    // log-softmax over the five action logits, log p(a)
                    float m = z[0];
#pragma unroll
                    for (int k = 1; k < NA; ++k) m = fmaxf(m, z[k]);
                    float e[NA], s = 0.f;
#pragma unroll
                    for (int k = 0; k < NA; ++k) { e[k] = expf(z[k] - m); s += e[k]; }
                    float za = z[0];
#pragma unroll
                    for (int k = 1; k < NA; ++k) za = k == a ? z[k] : za;
                    const float logp = (za - m) - logf(s);
                    if (!GRAD && !STATS) {
                        if (src >= 0) old_logp_out[src] = logp;
                    } else if (STATS && src >= 0) {
                        // entropy -sum p_k log p_k of the full log-softmax; ratio, k3 and clipping against old_logp
                        const float lse = logf(s);
                        float pl = 0.f;
#pragma unroll
                        for (int k = 0; k < NA; ++k) pl += (e[k] / s) * ((z[k] - m) - lse);
                        st[MM_PPO_STAT_ENTROPY] += (double)(-pl);
                        if (with_ratio) {
                            const float lr = logp - rf[LROWS + r];
                            const float ratio = expf(lr);
                            st[MM_PPO_STAT_K3] += (double)((ratio - 1.f) - lr);
                            st[MM_PPO_STAT_CLIPPED] += fabsf(ratio - 1.f) > clip ? 1.0 : 0.0;
                            r_min = fminf(r_min, ratio);
                            r_max = fmaxf(r_max, ratio);
                        }
                    } else if (GRAD && src >= 0) {
                        const float adv = KIND == MM_PPO_ACTOR ? rf[r] - rf[2 * LROWS + r] : rf[r] - z[5];
                        const float ratio = expf(logp - rf[LROWS + r]);
                        float l;
                        const float gl = ppo_row(ratio, adv, clip, l);
                        loss_a += l;
#pragma unroll
                        for (int k = 0; k < NA; ++k) dz[k] = gl * ((k == a ? 1.f : 0.f) - e[k] / s);
                    }
                }
                if (KIND != MM_PPO_ACTOR) {
                    constexpr int kv = KIND == MM_PPO_CRITIC ? 0 : 5;
                    if (!GRAD && !STATS) {
                        if ((KIND == MM_PPO_CRITIC || q_target_out != nullptr) && src >= 0) q_target_out[src] = z[kv];
                    } else if (STATS && src >= 0) {
                        // the value's fit to the return: v = Q(s, a) or V(s), G, and the residual G - v, in f32
                        const float v = z[kv], gr = rf[r], res = gr - v;
                        st[MM_PPO_STAT_V] += (double)v;
                        st[MM_PPO_STAT_V2] += (double)v * (double)v;
                        st[MM_PPO_STAT_G] += (double)gr;
                        st[MM_PPO_STAT_G2] += (double)gr * (double)gr;
                        st[MM_PPO_STAT_RES2] += (double)res * (double)res;
                    } else if (GRAD && src >= 0) {
                        const float d = z[kv] - rf[r];
                        loss_c += d * d;
                        dz[kv] = 2.f * d;
                    }
                }
                if (STATS && src >= 0) st[MM_PPO_STAT_N] += 1.0;
                if (GRAD) {
                    uint4 v;
                    v.x = h2u(__floats2half2_rn(dz[0], dz[1]));
                    v.y = h2u(__floats2half2_rn(dz[2], dz[3]));
                    v.z = h2u(__floats2half2_rn(dz[4], dz[5]));
                    v.w = h2u(__floats2half2_rn(dz[6], dz[7]));
                    *reinterpret_cast<uint4 *>(dz3s + r * 24) = v;
                }
            }
        }
        if (!GRAD) {
            __syncwarp();
            continue;
        }
        __syncwarp();

        // ---- backward, row-local: dZ2 = (dZ3 W3) * [h2 > 0]
#pragma unroll
        for (int n0 = 0; n0 < 128; n0 += 64) {
            float acc[8][4];
            zero(acc);
            row_gemm<8, 1, true>(acc, dz3a + row0 * 24 * 2, 24, w3a, S3, n0, lane);
            store_masked(acc, h2s, SB, dz2s, SB, row0, n0, g, t);
        }
        __syncthreads();

        // ---- weight gradients of layers 2 and 3 over the whole tile
        wgrad_gemm<N2T>(g2, dz2a, SB, warp * 16, h1a, SB, 0, lane);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            const int nt = warp + 8 * q;
            if (nt < 17) wgrad_gemm<1>(g3[q], dz3a, 24, 0, h2a, SB, nt * 8, lane);
        }
        __syncthreads();

        // ---- dZ1 = (dZ2 W2) * [h1 > 0], row-local, into the h2 tile (no longer read)
#pragma unroll
        for (int n0 = 0; n0 + 64 <= H1; n0 += 64) {
            float acc[8][4];
            zero(acc);
            row_gemm<8, 8, true>(acc, dz2a + row0 * SB * 2, SB, w2a, SB, n0, lane);
            store_masked(acc, h1s, SB, h2s, SB, row0, n0, g, t);
        }
        if constexpr (H1 % 64 != 0) {
            float acc[(H1 % 64) / 8][4];
            zero(acc);
            row_gemm<(H1 % 64) / 8, 8, true>(acc, dz2a + row0 * SB * 2, SB, w2a, SB, H1 - H1 % 64, lane);
            store_masked(acc, h1s, SB, h2s, SB, row0, H1 - H1 % 64, g, t);
        }
        __syncthreads();

        // ---- weight gradient of layer 1
        wgrad_gemm<4>(g1, h2a, SB, warp * 16, xa, SX, 0, lane);
        if (H1 > 128) wgrad_gemm<1>(g1x, h2a, SB, 128 + (warp >> 2) * 16, xa, SX, (warp & 3) * 8, lane);
        __syncthreads();
    }
    if (STATS) {
        // warp butterfly, then the 8 warps in order by one thread per field (the dZ3 tile, unused here, holds the warps'
        // sums): the CTA's partial has a fixed summation order
        st[MM_PPO_STAT_RATIO_MIN] = (double)r_min;
        st[MM_PPO_STAT_RATIO_MAX] = (double)r_max;
#pragma unroll
        for (int f = 0; f < NSTAT; ++f)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double x = __shfl_xor_sync(0xffffffffu, st[f], o);
                st[f] = f == MM_PPO_STAT_RATIO_MIN ? fmin(st[f], x) : f == MM_PPO_STAT_RATIO_MAX ? fmax(st[f], x) : st[f] + x;
            }
        double *wsum = reinterpret_cast<double *>(dz3s);
        if (lane == 0)
#pragma unroll
            for (int f = 0; f < NSTAT; ++f) wsum[warp * NSTAT + f] = st[f];
        __syncthreads();
        if (tid < NSTAT) {
            double acc = wsum[tid];
            for (int w = 1; w < LT / 32; ++w) {
                const double x = wsum[w * NSTAT + tid];
                acc = tid == MM_PPO_STAT_RATIO_MIN ? fmin(acc, x) : tid == MM_PPO_STAT_RATIO_MAX ? fmax(acc, x) : acc + x;
            }
            reinterpret_cast<double *>(partials)[(int64_t)blockIdx.x * NSTAT + tid] = acc;
        }
        return;
    }
    if (!GRAD) return;

    // ---- this CTA's partial sums, each element written by exactly one thread
    float *part = partials + (int64_t)blockIdx.x * L::P;
    auto put = [&](const float (&acc)[4], int base, int ld, int m0, int n0) {
        float *p = part + base;
        *reinterpret_cast<float2 *>(p + (m0 + g) * ld + n0 + 2 * t) = make_float2(acc[0], acc[1]);
        *reinterpret_cast<float2 *>(p + (m0 + g + 8) * ld + n0 + 2 * t) = make_float2(acc[2], acc[3]);
    };
#pragma unroll
    for (int j = 0; j < N2T; ++j) put(g2[j], L::P2, L::N2G, warp * 16, 8 * j);
#pragma unroll
    for (int q = 0; q < 3; ++q)
        if (warp + 8 * q < 17) put(g3[q][0], L::P3, S3, 0, (warp + 8 * q) * 8);
#pragma unroll
    for (int j = 0; j < 4; ++j) put(g1[j], L::P1, 32, warp * 16, 8 * j);
    if (H1 > 128) put(g1x[0], L::P1, 32, 128 + (warp >> 2) * 16, (warp & 3) * 8);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        loss_a += __shfl_xor_sync(0xffffffffu, loss_a, o);
        loss_c += __shfl_xor_sync(0xffffffffu, loss_c, o);
    }
    if (lane == 0) { red[2 * warp] = loss_a; red[2 * warp + 1] = loss_c; }
    __syncthreads();
    if (tid == 0) {
        float sa = 0.f, sc = 0.f;
        for (int w = 0; w < LT / 32; ++w) { sa += red[2 * w]; sc += red[2 * w + 1]; }
        part[L::PL] = sa;
        part[L::PL + 1] = sc;
    }
}

// The statistics partials of n_parts CTAs combined in CTA order (sums; min / max for the ratio range) into stats.
// n_parts = 0 writes the empty value: zeros, RATIO_MIN = +inf, RATIO_MAX = -inf.
__global__ void ppo_stats_reduce_kernel(const double *__restrict__ partials, int n_parts, double *__restrict__ stats) {
    const int f = threadIdx.x;
    if (f >= NSTAT) return;
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    double acc = f == MM_PPO_STAT_RATIO_MIN ? inf : f == MM_PPO_STAT_RATIO_MAX ? -inf : 0.0;
    for (int c = 0; c < n_parts; ++c) {
        const double x = partials[(int64_t)c * NSTAT + f];
        acc = f == MM_PPO_STAT_RATIO_MIN ? fmin(acc, x) : f == MM_PPO_STAT_RATIO_MAX ? fmax(acc, x) : acc + x;
    }
    stats[f] = acc;
}

// Sum of the CTA partials in CTA order, times 1/N, scattered into the torch parameters' layout.
template <int KIND>
__global__ void __launch_bounds__(256) ppo_reduce_kernel(const float *__restrict__ partials, int n_parts, float inv_n,
                                                         mm_ppo_grads_out gr, float *__restrict__ losses) {
    using L = LG<KIND>;
    constexpr int H1 = L::H1, IN2 = L::IN2, NA3 = KIND == MM_PPO_CRITIC ? 1 : NA;
    constexpr int E1 = H1 * NS, E2 = E1 + H1, E3 = E2 + 128 * IN2, E4 = E3 + 128, E5 = E4 + NA3 * 128, E6 = E5 + NA3;
    constexpr int E7 = E6 + (KIND == MM_PPO_SHARED ? 128 : 0), E8 = E7 + (KIND == MM_PPO_SHARED ? 1 : 0), ET = E8 + 2;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < ET; e += gridDim.x * blockDim.x) {
        int loc;
        float *dst;
        if (e < E1) { loc = L::P1 + (e / NS) * 32 + e % NS; dst = gr.w1 + e; }
        else if (e < E2) { loc = L::P1 + (e - E1) * 32 + NS; dst = gr.b1 + (e - E1); }
        else if (e < E3) { const int k = e - E2; loc = L::P2 + (k / IN2) * L::N2G + k % IN2; dst = gr.w2 + k; }
        else if (e < E4) { loc = L::P2 + (e - E3) * L::N2G + IN2; dst = gr.b2 + (e - E3); }
        else if (e < E5) { const int k = e - E4; loc = L::P3 + (k / 128) * L::S3 + k % 128; dst = gr.w3 + k; }
        else if (e < E6) { loc = L::P3 + (e - E5) * L::S3 + 128; dst = gr.b3 + (e - E5); }
        else if (e < E7) { loc = L::P3 + 5 * L::S3 + (e - E6); dst = gr.w4 + (e - E6); }
        else if (e < E8) { loc = L::P3 + 5 * L::S3 + 128; dst = gr.b4; }
        else {
            const int s = e - E8;                      // loss slot: 0 = PPO surrogate, 1 = value regression
            if ((s == 0 && KIND == MM_PPO_CRITIC) || (s == 1 && KIND == MM_PPO_ACTOR)) continue;
            loc = L::PL + s;
            dst = losses + s;
        }
        float acc = 0.f;
        for (int c = 0; c < n_parts; ++c) acc += partials[(int64_t)c * L::P + loc];
        *dst = acc * inv_n;
    }
}

struct Workspace {
    float *ptr = nullptr;
    size_t floats = 0;
};
Workspace g_ws[MM_MAX_DEVICES];
std::mutex g_ws_mutex;

int device_sms(int &dev, int &sms) {
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MM_MAX_DEVICES) return 1;
    return cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess;
}

template <int KIND, bool GRAD, bool STATS = false>
int prepare(int dev) {
    static bool ready[MM_MAX_DEVICES] = {};
    if (ready[dev]) return 0;
    if (cudaFuncSetAttribute(ppo_kernel<KIND, GRAD, STATS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LG<KIND>::SMEM) !=
        cudaSuccess)
        return 1;
    ready[dev] = true;
    return 0;
}

// The partials workspace: sized once per device for the largest kind's gradient partials at one CTA per SM (the
// statistics partials are far smaller), reused by every call; calls on one device are ordered on the caller's stream, as
// the update loop issues them.  -> null when the allocation fails.
float *workspace(int dev, int sms) {
    std::lock_guard<std::mutex> lock(g_ws_mutex);
    const size_t need = (size_t)sms * LG<MM_PPO_SHARED>::P;
    static_assert(LG<MM_PPO_ACTOR>::P * sizeof(float) >= NSTAT * sizeof(double), "statistics partials fit the workspace");
    if (g_ws[dev].floats < need) {
        if (g_ws[dev].ptr) cudaFree(g_ws[dev].ptr);
        g_ws[dev].ptr = nullptr;
        g_ws[dev].floats = 0;
        if (cudaMalloc(&g_ws[dev].ptr, need * sizeof(float)) != cudaSuccess) return nullptr;
        g_ws[dev].floats = need;
    }
    return g_ws[dev].ptr;
}

template <int KIND>
int launch_targets_t(const float *states, const int8_t *actions, const int64_t *idx, int64_t n, const mm_ppo_net &net, float *old_logp,
                     float *q_target, cudaStream_t s) {
    int dev = 0, sms = 0;
    if (device_sms(dev, sms) || prepare<KIND, false>(dev)) return 1;
    const int64_t tiles = (n + LROWS - 1) / LROWS, grid = tiles < sms ? tiles : sms;
    ppo_kernel<KIND, false><<<(unsigned)grid, LT, LG<KIND>::SMEM, s>>>(states, actions, nullptr, nullptr, nullptr, idx, n, 0.f, net,
                                                                        old_logp, q_target, nullptr);
    return cudaGetLastError() != cudaSuccess;
}

template <int KIND>
int launch_grads_t(const float *states, const int8_t *actions, const float *returns, const float *old_logp, const float *q_target,
                   const int64_t *idx, int64_t n, float clip, const mm_ppo_net &net, const mm_ppo_grads_out &gr, float *losses,
                   cudaStream_t s) {
    int dev = 0, sms = 0;
    if (device_sms(dev, sms) || prepare<KIND, true>(dev)) return 1;
    const int64_t tiles = (n + LROWS - 1) / LROWS, grid = tiles < sms ? tiles : sms;
    float *ws = workspace(dev, sms);
    if (!ws) return 1;
    ppo_kernel<KIND, true><<<(unsigned)grid, LT, LG<KIND>::SMEM, s>>>(states, actions, returns, old_logp, q_target, idx, n, clip, net,
                                                                       nullptr, nullptr, ws);
    ppo_reduce_kernel<KIND><<<(unsigned)((LG<KIND>::P + 255) / 256), 256, 0, s>>>(ws, (int)grid, 1.0f / (float)n, gr, losses);
    return cudaGetLastError() != cudaSuccess;
}

template <int KIND>
int launch_stats_t(const float *states, const int8_t *actions, const float *returns, const float *old_logp, const int64_t *idx,
                   int64_t n, float clip, const mm_ppo_net &net, double *stats, cudaStream_t s) {
    int dev = 0, sms = 0;
    if (device_sms(dev, sms) || prepare<KIND, false, true>(dev)) return 1;
    const int64_t tiles = (n + LROWS - 1) / LROWS, grid = tiles < sms ? tiles : sms;
    float *ws = workspace(dev, sms);
    if (!ws) return 1;
    if (grid > 0)
        ppo_kernel<KIND, false, true><<<(unsigned)grid, LT, LG<KIND>::SMEM, s>>>(states, actions, returns, old_logp, nullptr, idx, n,
                                                                              clip, net, nullptr, nullptr, ws);
    ppo_stats_reduce_kernel<<<1, 32, 0, s>>>(reinterpret_cast<const double *>(ws), (int)grid, stats);
    return cudaGetLastError() != cudaSuccess;
}

}  // namespace

int launch_ppo_stats(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                     const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net, double *stats, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (kind == MM_PPO_ACTOR) return launch_stats_t<MM_PPO_ACTOR>(states, actions, returns, old_logp, idx, n, clip, *net, stats, s);
    if (kind == MM_PPO_CRITIC) return launch_stats_t<MM_PPO_CRITIC>(states, actions, returns, old_logp, idx, n, clip, *net, stats, s);
    return launch_stats_t<MM_PPO_SHARED>(states, actions, returns, old_logp, idx, n, clip, *net, stats, s);
}

int launch_ppo_targets(int kind, const float *states, const int8_t *actions, const int64_t *idx, int64_t n, const mm_ppo_net *net,
                       float *old_logp, float *q_target, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (kind == MM_PPO_ACTOR) return launch_targets_t<MM_PPO_ACTOR>(states, actions, idx, n, *net, old_logp, q_target, s);
    if (kind == MM_PPO_CRITIC) return launch_targets_t<MM_PPO_CRITIC>(states, actions, idx, n, *net, old_logp, q_target, s);
    return launch_targets_t<MM_PPO_SHARED>(states, actions, idx, n, *net, old_logp, q_target, s);
}

int launch_ppo_grads(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                     const float *q_target, const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net,
                     const mm_ppo_grads_out *grads, float *losses, void *stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (kind == MM_PPO_ACTOR)
        return launch_grads_t<MM_PPO_ACTOR>(states, actions, returns, old_logp, q_target, idx, n, clip, *net, *grads, losses, s);
    if (kind == MM_PPO_CRITIC)
        return launch_grads_t<MM_PPO_CRITIC>(states, actions, returns, old_logp, q_target, idx, n, clip, *net, *grads, losses, s);
    return launch_grads_t<MM_PPO_SHARED>(states, actions, returns, old_logp, q_target, idx, n, clip, *net, *grads, losses, s);
}

}  // namespace mm

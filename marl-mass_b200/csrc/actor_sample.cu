// actor_sample.cu — the MAPPO actor (30-128-128-5, ReLU, log-softmax) and its exploration draw, fused in one kernel.
//
// Reference: marl/single_agent/Model_common.py:5-23 (ActorNetwork), marl/mappo.py:209-228 (_softmax_action +
// exploration_action: np.random.choice(p=softmax) = inverse CDF of one uniform).  The reference evaluates the shared
// actor once per agent per step on the CPU; the batched rollout (BASELINE configs[3]) evaluates it for every
// (env, agent) row of the observation buffer the step kernel has just written, 786 432 rows at 65 536 envs.  As three
// torch Linear layers that is 1.7 ms per step against 0.9 ms for the env step itself (profiles/README.md): the hidden
// activations (2 x 400 MB) go through HBM four times.  Here all three layers stay on chip and only the observations
// (120 B / row) and the actions (1 B / row) touch HBM.
//
// Two implementations of the same network and draw:
//   * actor_mlp_wg_kernel<H1> (default; the only kernel of mm_actor_sample_mlp): all three layers as tcgen05.mma with
//     fp16 operands and the accumulators in TMEM, one warpgroup per 128-row tile - see the section further down;
//   * actor_sample_kernel (mm_set_actor_impl(1)): TF32 mma.sync.m16n8k8 per warp, kept as the independent cross-check.
//     The accumulator fragment of layer L (thread holds rows g, g+8 and columns 2t, 2t+1 of each 8-wide tile) is reused
//     directly as the A fragment of layer L+1 (rows g, g+8, columns t, t+4) by permuting the K index of that layer:
//     A column t <-> hidden unit 8kk+2t, A column t+4 <-> 8kk+2t+1, and the weights are laid out in shared memory in
//     fragment order with the same permutation, so no shuffle or shared-memory round trip separates the layers.
// Measured at 786 432 rows on a B200: torch layers 1.89 ms, mma.sync 0.204 ms, tcgen05 warpgroup kernel 0.067 ms
// (profiles/README.md); this op is ~33 GFLOP per step, so both are bound by their epilogues and staging, not by the
// tensor pipe.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "mm_internal.h"

namespace mm {

constexpr int AC_IN = 30, AC_HID = 128, AC_OUT = 5;
constexpr int AC_KT1 = 4;              // k-tiles of layer 1 (30 inputs padded to 32)
constexpr int AC_NT = AC_HID / 8;      // 16 n-tiles of the hidden layers = k-tiles of the next layer
constexpr int AC_THREADS = 256;
constexpr int AC_GRP = 8;              // layer-2 n-tiles accumulated together (independent MMA chains per warp)
// shared memory (32-bit words): fragment-ordered TF32 weights, then the fp32 biases
constexpr int AC_W1F = 0;
constexpr int AC_W2F = AC_W1F + AC_KT1 * AC_NT * 64;
constexpr int AC_W3F = AC_W2F + AC_NT * AC_NT * 64;
constexpr int AC_B1 = AC_W3F + AC_NT * 64;
constexpr int AC_B2 = AC_B1 + AC_HID;
constexpr int AC_B3 = AC_B2 + AC_HID;
constexpr int AC_SMEM_WORDS = AC_B3 + 8;

__device__ __forceinline__ uint32_t to_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Philox4x32-10, one counter block per row: (seed, step) is the key, the row index the counter
__device__ __forceinline__ uint32_t philox_row(uint64_t seed, uint64_t step, uint64_t row) {
    uint32_t k0 = (uint32_t)seed ^ (uint32_t)(step * 0x9E3779B97F4A7C15ull), k1 = (uint32_t)(seed >> 32) ^ (uint32_t)(step >> 7);
    uint32_t c0 = (uint32_t)row, c1 = (uint32_t)(row >> 32), c2 = (uint32_t)step, c3 = 0x6d6d6173u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

// Invalid-action masking of the MAPPO_GI actor (marl/single_agent/Model_gi.py:63-66: logits[action_mask == 0] = -1e8
// before the log-softmax): bit k of mask_bits[row] set = action k available (the env kernel's action_mask buffer).
__device__ __forceinline__ void apply_action_mask(float (&l)[AC_OUT], const uint8_t *mask_bits, int64_t row) {
    if (!mask_bits) return;
    const uint32_t bits = mask_bits[row];
#pragma unroll
    for (int k = 0; k < AC_OUT; ++k)
        if (!((bits >> k) & 1u)) l[k] = -1e8f;
}

__global__ void __launch_bounds__(AC_THREADS, 1)
actor_sample_kernel(const float *__restrict__ obs, const int32_t *__restrict__ n_agents, int64_t n_rows,
                    const float *__restrict__ w1, const float *__restrict__ b1, const float *__restrict__ w2,
                    const float *__restrict__ b2, const float *__restrict__ w3, const float *__restrict__ b3,
                    uint64_t seed, uint64_t step, const uint8_t *__restrict__ mask_bits, int8_t *__restrict__ actions,
                    float *__restrict__ logp_all, float *__restrict__ logp_sel) {
    extern __shared__ __align__(16) uint32_t ac_sm[];
    float *sm_f = reinterpret_cast<float *>(ac_sm);
    const int tid = threadIdx.x, lane = tid & 31, g = lane >> 2, t = lane & 3;

    // weights into fragment order (torch Linear weight is [out][in]; B(k, n) = weight[n][k])
    for (int idx = tid; idx < AC_KT1 * AC_NT * 64; idx += AC_THREADS) {
        int r = idx & 1, ln = (idx >> 1) & 31, tile = idx >> 6, j = tile % AC_NT, kk = tile / AC_NT;
        int k = 8 * kk + (ln & 3) + 4 * r, n = 8 * j + (ln >> 2);
        ac_sm[AC_W1F + idx] = to_tf32(k < AC_IN ? w1[n * AC_IN + k] : 0.f);
    }
    for (int idx = tid; idx < AC_NT * AC_NT * 64; idx += AC_THREADS) {
        int r = idx & 1, ln = (idx >> 1) & 31, tile = idx >> 6, j = tile % AC_NT, kk = tile / AC_NT;
        int k = 8 * kk + 2 * (ln & 3) + r, n = 8 * j + (ln >> 2);
        ac_sm[AC_W2F + idx] = to_tf32(w2[n * AC_HID + k]);
    }
    for (int idx = tid; idx < AC_NT * 64; idx += AC_THREADS) {
        int r = idx & 1, ln = (idx >> 1) & 31, kk = idx >> 6;
        int k = 8 * kk + 2 * (ln & 3) + r, n = ln >> 2;
        ac_sm[AC_W3F + idx] = to_tf32(n < AC_OUT ? w3[n * AC_HID + k] : 0.f);
    }
    for (int idx = tid; idx < AC_HID; idx += AC_THREADS) {
        sm_f[AC_B1 + idx] = b1[idx];
        sm_f[AC_B2 + idx] = b2[idx];
    }
    if (tid < 8) sm_f[AC_B3 + tid] = tid < AC_OUT ? b3[tid] : 0.f;
    __syncthreads();

    const int64_t n_tiles = (n_rows + 15) / 16;
    const int64_t warp0 = (int64_t)blockIdx.x * (AC_THREADS / 32) + (tid >> 5);
    const int64_t warp_stride = (int64_t)gridDim.x * (AC_THREADS / 32);
    const uint2 *w1f = reinterpret_cast<const uint2 *>(ac_sm + AC_W1F) + lane;
    const uint2 *w2f = reinterpret_cast<const uint2 *>(ac_sm + AC_W2F) + lane;
    const uint2 *w3f = reinterpret_cast<const uint2 *>(ac_sm + AC_W3F) + lane;

    for (int64_t tile = warp0; tile < n_tiles; tile += warp_stride) {
        const int64_t r_lo = tile * 16 + g, r_hi = r_lo + 8;
        const bool ok_lo = r_lo < n_rows, ok_hi = r_hi < n_rows;
        const float *o_lo = obs + r_lo * AC_IN, *o_hi = obs + r_hi * AC_IN;

        // layer 1: [16 x 32] x [32 x 128]
        uint32_t a1[AC_KT1][4];
#pragma unroll
        for (int kk = 0; kk < AC_KT1; ++kk) {
            const int c0 = 8 * kk + t, c1 = c0 + 4;
            a1[kk][0] = to_tf32(ok_lo && c0 < AC_IN ? o_lo[c0] : 0.f);
            a1[kk][1] = to_tf32(ok_hi && c0 < AC_IN ? o_hi[c0] : 0.f);
            a1[kk][2] = to_tf32(ok_lo && c1 < AC_IN ? o_lo[c1] : 0.f);
            a1[kk][3] = to_tf32(ok_hi && c1 < AC_IN ? o_hi[c1] : 0.f);
        }
        uint32_t h1[AC_NT][4];   // relu(layer 1) as the A fragments of layer 2
#pragma unroll
        for (int j = 0; j < AC_NT; ++j) {
            float acc[4];
            acc[0] = acc[2] = sm_f[AC_B1 + 8 * j + 2 * t];
            acc[1] = acc[3] = sm_f[AC_B1 + 8 * j + 2 * t + 1];
#pragma unroll
            for (int kk = 0; kk < AC_KT1; ++kk) {
                uint2 b = w1f[(kk * AC_NT + j) * 32];
                mma_tf32(acc, a1[kk], b.x, b.y);
            }
            // accumulator (rows g, g+8; cols 2t, 2t+1) -> A fragment (rows g, g+8; k-columns t, t+4) of k-tile j
            h1[j][0] = to_tf32(fmaxf(acc[0], 0.f));
            h1[j][1] = to_tf32(fmaxf(acc[2], 0.f));
            h1[j][2] = to_tf32(fmaxf(acc[1], 0.f));
            h1[j][3] = to_tf32(fmaxf(acc[3], 0.f));
        }
        // layers 2 and 3: each group of 8 hidden n-tiles of layer 2 is consumed by layer 3 as soon as it is complete
        float lg[4];
        lg[0] = lg[2] = sm_f[AC_B3 + 2 * t];
        lg[1] = lg[3] = sm_f[AC_B3 + 2 * t + 1];
#pragma unroll
        for (int jb = 0; jb < AC_NT; jb += AC_GRP) {
            float acc[AC_GRP][4];
#pragma unroll
            for (int q = 0; q < AC_GRP; ++q) {
                acc[q][0] = acc[q][2] = sm_f[AC_B2 + 8 * (jb + q) + 2 * t];
                acc[q][1] = acc[q][3] = sm_f[AC_B2 + 8 * (jb + q) + 2 * t + 1];
            }
#pragma unroll
            for (int kk = 0; kk < AC_NT; ++kk) {
#pragma unroll
                for (int q = 0; q < AC_GRP; ++q) {
                    uint2 b = w2f[(kk * AC_NT + jb + q) * 32];
                    mma_tf32(acc[q], h1[kk], b.x, b.y);
                }
            }
#pragma unroll
            for (int q = 0; q < AC_GRP; ++q) {
                uint32_t h2[4] = {to_tf32(fmaxf(acc[q][0], 0.f)), to_tf32(fmaxf(acc[q][2], 0.f)),
                                  to_tf32(fmaxf(acc[q][1], 0.f)), to_tf32(fmaxf(acc[q][3], 0.f))};
                uint2 b = w3f[(jb + q) * 32];
                mma_tf32(lg, h2, b.x, b.y);
            }
        }

        // logits of row g: columns (2t, 2t+1) in lg[0..1] of the quad's threads; row g+8 in lg[2..3]
        const unsigned full = 0xffffffffu;
        const int q0 = lane & ~3;
        float l_lo[AC_OUT], l_hi[AC_OUT];
#pragma unroll
        for (int k = 0; k < AC_OUT; ++k) {
            const int src = q0 + (k >> 1);
            float lo_e = __shfl_sync(full, lg[0], src), lo_o = __shfl_sync(full, lg[1], src);
            float hi_e = __shfl_sync(full, lg[2], src), hi_o = __shfl_sync(full, lg[3], src);
            l_lo[k] = (k & 1) ? lo_o : lo_e;
            l_hi[k] = (k & 1) ? hi_o : hi_e;
        }
        // thread t = 0 finishes row g, t = 1 row g+8 (the other two threads of the quad idle here)
        if (t < 2) {
            const int64_t row = t == 0 ? r_lo : r_hi;
            if (row < n_rows) {
                float l[AC_OUT];
#pragma unroll
                for (int k = 0; k < AC_OUT; ++k) l[k] = t == 0 ? l_lo[k] : l_hi[k];
                apply_action_mask(l, mask_bits, row);
                float m = l[0];
#pragma unroll
                for (int k = 1; k < AC_OUT; ++k) m = fmaxf(m, l[k]);
                float e[AC_OUT], S = 0.f;
#pragma unroll
                for (int k = 0; k < AC_OUT; ++k) { e[k] = __expf(l[k] - m); S += e[k]; }
                const float logS = __logf(S);
                // np.random.choice(p): first k whose cumulative probability exceeds one uniform draw
                const float u = (float)(philox_row(seed, step, (uint64_t)row) >> 8) * (1.0f / 16777216.0f);
                const float target = u * S;
                int a = AC_OUT - 1;
                float c = 0.f;
                bool found = false;
#pragma unroll
                for (int k = 0; k < AC_OUT; ++k) {
                    c += e[k];
                    if (!found && target < c) { a = k; found = true; }
                }
                bool live = true;
                if (n_agents) live = (int)(row % MAXV) < n_agents[row / MAXV];
                actions[row] = (int8_t)(live ? a : 1);   // absent agents idle (their rows are ignored by the env)
                if (logp_sel) logp_sel[row] = l[a] - m - logS;
                if (logp_all) {
#pragma unroll
                    for (int k = 0; k < AC_OUT; ++k) logp_all[row * AC_OUT + k] = l[k] - m - logS;
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// tcgen05 helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t tc_smem(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, "
                 "%23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
                   "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
                   "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
    // K-major, SWIZZLE_NONE: start address, LBO (between the two 16-byte k-chunks of an MMA), SBO (between 8-row groups)
    return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(128u >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
                 ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));    // low half = a, high half = b
    return r;
}

// ------------------------------------------------------------------------------------------------
// tcgen05 kernel: fp16 operands, one warpgroup per tile, four (H1 = 128) or three (H1 = 160) tiles in flight per SM
// ------------------------------------------------------------------------------------------------
//   H1 = 128: MAPPO ActorNetwork 30-128-128-5 (Model_common.py:5-23).
//   H1 = 160: MAPPO_GI ActorCriticNetwork with state_split (Model_gi.py:137-220): its three first-layer blocks
//             (5 -> 32, 10 -> 64, 10 -> 64 over fixed column lists) are ONE 30 -> 160 layer whose weight matrix is zero
//             outside the blocks; the host scatters fc11 / fc12 / fc13 into it (rollout.py).  The optional sixth output
//             column is critic_linear (the state value V(s), mappo_gi.py:396-404).
// Per 128-row tile (= the 128 TMEM lanes):
//   layer 1   D1[128 x H1]  = A1[128 x 32] * W1^T    tcgen05.mma kind::f16, K = 16
//   layer 2   D2[128 x 128] = h1[128 x H1] * W2^T
//   layer 3   D3[128 x 16]  = h2[128 x 128] * W3^T   5 logits, the value, 10 zero columns: as per-thread FMAs this
//             output layer was ~55 % of the instructions of an earlier kernel
//   then log-softmax and the inverse-CDF draw in the thread that owns the row.
// fp16 operands (kind::f16): fp16 has TF32's 10-bit mantissa, observations live in [-1, 1] and the hidden activations of
// these networks stay far below 65 504, so half of TF32's shared memory per operand.  Operands are K-major, no swizzle,
// laid out [k-chunk][row] in 16-byte pieces of 8 halves: core matrices of 8 rows, SBO = 128 B between 8-row groups,
// LBO = one chunk between the two k-chunks of an MMA.  Design:
//   * the weights sit in shared memory ONCE per SM and every warpgroup (128 threads = the 128 rows of a tile) runs its
//     own tile pipeline on its own operand buffers, TMEM columns, named barrier and mbarrier: while one warpgroup runs
//     an epilogue, the others' MMAs and loads proceed, with no CTA-wide barrier;
//   * warp w reads TMEM lane quarter w % 4 (hardware rule), i.e. the rows of its own quarter of the tile;
//   * biases ride in the MMAs: an extra K-step multiplies a constant block (1, 1, 0, ...) by (hi, lo) fp16 halves of the
//     bias (layer 1 uses its two padding columns k = 30, 31), so the accumulator already holds D + b to ~2^-22;
//   * the epilogue of a hidden layer is cvt.rn.relu.f16x2.f32 - one instruction per two activations - and a 16-byte
//     shared store per eight;
//   * D2 reuses D1's columns and h2 h1's shared memory; D3 reuses the first 16 columns of the tile's TMEM region (D2 is
//     dead once epilogue 2 has synchronised).
template <int H1>
struct WgLayout {
    static constexpr int NWG = H1 == 128 ? 4 : 3;            // tiles in flight: shared memory (H1 = 160) or TMEM (128) bound
    static constexpr int THREADS = 128 * NWG;
    static constexpr int ROWS = 128;
    static constexpr int CH1 = H1 / 8;
    static constexpr uint32_t A_CHUNK = ROWS * 16;
    static constexpr uint32_t W1_CHUNK = H1 * 16;
    static constexpr uint32_t W3_CHUNK = 16 * 16;
    static constexpr uint32_t W1 = 0;                             // [4 chunks][H1]: k = 30, 31 carry b1 (hi, lo)
    static constexpr uint32_t W2 = W1 + 4 * W1_CHUNK;             // [CH1 + 2][128]: the last two chunks carry b2
    static constexpr uint32_t W3 = W2 + (CH1 + 2) * A_CHUNK;      // [16 + 2][16]: the last two carry b3 and the value bias
    static constexpr uint32_t ONES = W3 + 18 * W3_CHUNK;          // [2 chunks][128]: (1, 1, 0, ..., 0) per row
    static constexpr uint32_t TILE0 = ONES + 2 * A_CHUNK;         // per warpgroup: A1 [4][128], A2 [CH1][128]
    static constexpr uint32_t TILE_BYTES = (4 + CH1) * A_CHUNK;
    static constexpr uint32_t BAR = TILE0 + NWG * TILE_BYTES;     // NWG mbarriers + the TMEM base address
    static constexpr uint32_t SMEM = BAR + 8 * NWG + 16;
    static constexpr uint32_t TMEM_COLS = 512;
    static constexpr uint32_t REGION = H1;                        // TMEM columns per warpgroup
    static constexpr uint32_t IDESC1 = (1u << 4) | ((uint32_t)(H1 >> 3) << 17) | ((128u >> 4) << 24);
    static constexpr uint32_t IDESC2 = (1u << 4) | ((uint32_t)(AC_HID >> 3) << 17) | ((128u >> 4) << 24);
    static constexpr uint32_t IDESC3 = (1u << 4) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
};
static_assert(WgLayout<128>::SMEM <= 227 * 1024 && WgLayout<160>::SMEM <= 227 * 1024, "actor kernel shared memory");
static_assert(WgLayout<128>::NWG * WgLayout<128>::REGION <= 512 && WgLayout<160>::NWG * WgLayout<160>::REGION <= 512, "actor kernel TMEM columns");

__device__ __forceinline__ uint32_t pack_relu_h2(uint32_t a_bits, uint32_t b_bits) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(__uint_as_float(b_bits)), "f"(__uint_as_float(a_bits)));
    return r;
}
__device__ __forceinline__ uint32_t hi_lo_h2(float b) {          // fp16 halves whose sum is b to ~2^-22
    const __half hi = __float2half_rn(b), lo = __float2half_rn(b - __half2float(hi));
    return (uint32_t)__half_as_ushort(hi) | ((uint32_t)__half_as_ushort(lo) << 16);
}
__device__ __forceinline__ void wg_sync(int wg) { asm volatile("bar.sync %0, 128;" ::"r"(wg + 1) : "memory"); }

template <int H1>
__global__ void __launch_bounds__(WgLayout<H1>::THREADS, 1)
actor_mlp_wg_kernel(const float *__restrict__ obs, const int32_t *__restrict__ n_agents, int64_t n_rows,
                    const float *__restrict__ w1, const float *__restrict__ b1, const float *__restrict__ w2,
                    const float *__restrict__ b2, const float *__restrict__ w3, const float *__restrict__ b3,
                    const float *__restrict__ wv, const float *__restrict__ bv, uint64_t seed, uint64_t step,
                    const uint8_t *__restrict__ mask_bits, int8_t *__restrict__ actions, float *__restrict__ logp_all,
                    float *__restrict__ logp_sel, float *__restrict__ values, float *__restrict__ obs_copy,
                    uint8_t *__restrict__ live_out) {
    using L = WgLayout<H1>;
    extern __shared__ __align__(128) uint8_t wg_sm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wg = warp >> 2;
    uint4 *w1f = reinterpret_cast<uint4 *>(wg_sm + L::W1), *w2f = reinterpret_cast<uint4 *>(wg_sm + L::W2);
    uint4 *w3f = reinterpret_cast<uint4 *>(wg_sm + L::W3), *ones = reinterpret_cast<uint4 *>(wg_sm + L::ONES);
    uint4 *a1 = reinterpret_cast<uint4 *>(wg_sm + L::TILE0 + wg * L::TILE_BYTES), *a2 = a1 + 4 * L::ROWS;
    uint64_t *bars = reinterpret_cast<uint64_t *>(wg_sm + L::BAR);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(wg_sm + L::BAR + 8 * L::NWG);
    const uint32_t bar = tc_smem(bars + wg);

    // ---- one-time setup: weights and biases in operand layout (fp16), the constant block, barriers, TMEM ----
    for (int idx = tid; idx < 4 * H1; idx += L::THREADS) {
        const int c = idx / H1, n = idx % H1, k = 8 * c;
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = k + q < AC_IN ? w1[n * AC_IN + k + q] : 0.f;
        uint4 o = make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
        if (c == 3) o.w = hi_lo_h2(b1[n]);                            // k = 30, 31
        w1f[idx] = o;
    }
    for (int idx = tid; idx < (L::CH1 + 2) * L::ROWS; idx += L::THREADS) {
        const int c = idx / L::ROWS, n = idx % L::ROWS;
        if (c < L::CH1) {
            const float4 lo = *reinterpret_cast<const float4 *>(w2 + n * H1 + 8 * c), hi = *reinterpret_cast<const float4 *>(w2 + n * H1 + 8 * c + 4);
            w2f[idx] = make_uint4(pack_h2(lo.x, lo.y), pack_h2(lo.z, lo.w), pack_h2(hi.x, hi.y), pack_h2(hi.z, hi.w));
        } else {
            w2f[idx] = make_uint4(c == L::CH1 ? hi_lo_h2(b2[n]) : 0u, 0u, 0u, 0u);
        }
    }
    for (int idx = tid; idx < 18 * 16; idx += L::THREADS) {          // rows 0..4 logits, 5 the value head, rest zero
        const int c = idx / 16, n = idx % 16;
        if (c < 16) {
            float v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = n < AC_OUT ? w3[n * AC_HID + 8 * c + q] : (n == AC_OUT && wv ? wv[8 * c + q] : 0.f);
            w3f[idx] = make_uint4(pack_h2(v[0], v[1]), pack_h2(v[2], v[3]), pack_h2(v[4], v[5]), pack_h2(v[6], v[7]));
        } else {
            const float b = n < AC_OUT ? b3[n] : (n == AC_OUT && bv ? bv[0] : 0.f);
            w3f[idx] = make_uint4(c == 16 ? hi_lo_h2(b) : 0u, 0u, 0u, 0u);
        }
    }
    for (int idx = tid; idx < 2 * L::ROWS; idx += L::THREADS) ones[idx] = make_uint4(idx < L::ROWS ? 0x3C003C00u : 0u, 0u, 0u, 0u);
    if (tid < L::NWG) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(bars + tid)));
    if (tid == 0) asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(tc_smem(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot + (uint32_t)wg * L::REGION;          // this warpgroup's columns
    const uint32_t a1_addr = tc_smem(a1), a2_addr = tc_smem(a2), w1_addr = tc_smem(w1f), w2_addr = tc_smem(w2f);
    const uint32_t w3_addr = tc_smem(w3f), ones_addr = tc_smem(ones);

    const int r = tid & 127;                                              // row of the tile = TMEM lane
    const uint32_t t_lane = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
    const int64_t n_tiles = (n_rows + L::ROWS - 1) / L::ROWS;
    const int64_t stride = (int64_t)gridDim.x * L::NWG;
    // observation rows: a tile is 128 x 30 floats = 960 contiguous float4 (row-per-thread loads touched 30 cache lines per
    // request: 5.3 x the minimal sector count, L1 request stage 55 % busy - profiles/r2_x_*); thread r takes float4
    // r, r + 128, ...: coalesced, and each float4 is two in-row pairs (30 and the flat index are even) -> two half2 stores
    constexpr int TILE_F4 = L::ROWS * AC_IN / 4, PRE = (TILE_F4 + 127) / 128;
    const int64_t total_f = n_rows * AC_IN;
    float4 pre[PRE];
    auto fetch = [&](int64_t tile) {
#pragma unroll
        for (int q = 0; q < PRE; ++q) {
            const int i = r + 128 * q;
            const int64_t g = tile * (L::ROWS * AC_IN) + 4 * i;                    // flat float index
            pre[q] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < TILE_F4 && tile < n_tiles) {
                if (g + 4 <= total_f) pre[q] = __ldg(reinterpret_cast<const float4 *>(obs + g));
                else if (g + 2 <= total_f) { const float2 h = __ldg(reinterpret_cast<const float2 *>(obs + g)); pre[q].x = h.x; pre[q].y = h.y; }
            }
        }
    };
    uint32_t *a1w = reinterpret_cast<uint32_t *>(a1);
    a1[3 * L::ROWS + r].w = 0x3C003C00u;                       // k = 30, 31: the constant 1 that multiplies b1 (never overwritten)
    auto a1_word = [&](int f) {                                // 32-bit word of A1 that holds elements (f, f + 1) of the flat tile
        const int row = f / AC_IN, col = f - AC_IN * row;
        return ((col >> 3) * L::ROWS + row) * 4 + ((col & 7) >> 1);
    };
    // tile t belongs to warpgroup (t / gridDim.x) % NWG of CTA t % gridDim.x: a short batch spreads over the SMs first
    int64_t tile = (int64_t)wg * gridDim.x + blockIdx.x;
    fetch(tile);
    uint32_t parity = 0;
    for (; tile < n_tiles; tile += stride) {
        // ---- stage the observation rows as fp16; rollout buffer (MAPPO.interact appends the state it acted on,
        // mappo.py:117-131): the rows pass through here anyway - stored now, not behind the loads, so that the prefetch
        // stays asynchronous ----
#pragma unroll
        for (int q = 0; q < PRE; ++q) {
            const int i = r + 128 * q;
            if (i < TILE_F4) {
                a1w[a1_word(4 * i)] = pack_h2(pre[q].x, pre[q].y);
                a1w[a1_word(4 * i + 2)] = pack_h2(pre[q].z, pre[q].w);
                if (obs_copy) {
                    const int64_t g = tile * (L::ROWS * AC_IN) + 4 * i;
                    if (g + 4 <= total_f) __stcs(reinterpret_cast<float4 *>(obs_copy + g), pre[q]);
                    else if (g + 2 <= total_f) __stcs(reinterpret_cast<float2 *>(obs_copy + g), make_float2(pre[q].x, pre[q].y));
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        wg_sync(wg);
        if (r == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 2; ++j)
                tc_mma(tmem, tc_desc(a1_addr + j * 2 * L::A_CHUNK, L::A_CHUNK), tc_desc(w1_addr + j * 2 * L::W1_CHUNK, L::W1_CHUNK),
                       L::IDESC1, j > 0);
            tc_commit(bar);
        }
        fetch(tile + stride);                                  // next tile's rows: in flight during this tile's MMAs and epilogues
        tc_wait(bar, parity); parity ^= 1;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- epilogue 1: h1 = relu(D1) -> A2 ----
#pragma unroll 1
        for (int col = 0; col < H1; col += 32) {
            uint32_t v[32];
            tc_ld32(t_lane + (uint32_t)col, v);
#pragma unroll
            for (int g = 0; g < 4; ++g)
                a2[(col / 8 + g) * L::ROWS + r] = make_uint4(pack_relu_h2(v[8 * g], v[8 * g + 1]), pack_relu_h2(v[8 * g + 2], v[8 * g + 3]),
                                                            pack_relu_h2(v[8 * g + 4], v[8 * g + 5]), pack_relu_h2(v[8 * g + 6], v[8 * g + 7]));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        wg_sync(wg);
        if (r == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int j = 0; j < H1 / 16; ++j)
                tc_mma(tmem, tc_desc(a2_addr + j * 2 * L::A_CHUNK, L::A_CHUNK), tc_desc(w2_addr + j * 2 * L::A_CHUNK, L::A_CHUNK),
                       L::IDESC2, j > 0);
            tc_mma(tmem, tc_desc(ones_addr, L::A_CHUNK), tc_desc(w2_addr + (H1 / 16) * 2 * L::A_CHUNK, L::A_CHUNK), L::IDESC2, 1);
            tc_commit(bar);
        }
        tc_wait(bar, parity); parity ^= 1;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // ---- epilogue 2: h2 = relu(D2) -> the first 16 chunks of A2 (MMA2 has finished reading h1) ----
#pragma unroll 1
        for (int col = 0; col < AC_HID; col += 32) {
            uint32_t v[32];
            tc_ld32(t_lane + (uint32_t)col, v);
#pragma unroll
            for (int g = 0; g < 4; ++g)
                a2[(col / 8 + g) * L::ROWS + r] = make_uint4(pack_relu_h2(v[8 * g], v[8 * g + 1]), pack_relu_h2(v[8 * g + 2], v[8 * g + 3]),
                                                            pack_relu_h2(v[8 * g + 4], v[8 * g + 5]), pack_relu_h2(v[8 * g + 6], v[8 * g + 7]));
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        wg_sync(wg);
        // ---- output layer 128 -> 5 (+ value), N = 16, into the first columns of the region ----
        if (r == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int j = 0; j < AC_HID / 16; ++j)
                tc_mma(tmem, tc_desc(a2_addr + j * 2 * L::A_CHUNK, L::A_CHUNK), tc_desc(w3_addr + j * 2 * L::W3_CHUNK, L::W3_CHUNK),
                       L::IDESC3, j > 0);
            tc_mma(tmem, tc_desc(ones_addr, L::A_CHUNK), tc_desc(w3_addr + 16 * L::W3_CHUNK, L::W3_CHUNK), L::IDESC3, 1);
            tc_commit(bar);
        }
        tc_wait(bar, parity); parity ^= 1;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        {
            const int64_t row = tile * L::ROWS + r;
            uint32_t v[16];
            tc_ld16(t_lane, v);
            if (row < n_rows) {
                float l[AC_OUT];
#pragma unroll
                for (int k = 0; k < AC_OUT; ++k) l[k] = __uint_as_float(v[k]);
                if (values) values[row] = __uint_as_float(v[AC_OUT]);
                apply_action_mask(l, mask_bits, row);
                float m = l[0];
#pragma unroll
                for (int k = 1; k < AC_OUT; ++k) m = fmaxf(m, l[k]);
                float e[AC_OUT], S = 0.f;
#pragma unroll
                for (int k = 0; k < AC_OUT; ++k) { e[k] = __expf(l[k] - m); S += e[k]; }
                const float logS = __logf(S);
                const float u = (float)(philox_row(seed, step, (uint64_t)row) >> 8) * (1.0f / 16777216.0f);
                const float target = u * S;
                int a = AC_OUT - 1;
                float c = 0.f;
                bool found = false;
#pragma unroll
                for (int k = 0; k < AC_OUT; ++k) {
                    c += e[k];
                    if (!found && target < c) { a = k; found = true; }
                }
                bool live = true;
                if (n_agents) live = (int)(row % MAXV) < n_agents[row / MAXV];
                actions[row] = (int8_t)(live ? a : 1);
                if (live_out) live_out[row] = live ? 1 : 0;
                if (logp_sel) logp_sel[row] = l[a] - m - logS;
                if (logp_all) {
#pragma unroll
                    for (int k = 0; k < AC_OUT; ++k) logp_all[row * AC_OUT + k] = l[k] - m - logS;
                }
            }
        }
        // no barrier here: the next tile's first wg_sync orders these TMEM reads before its first MMA
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(*tmem_slot) : "memory");
}

// Implementation of mm_actor_sample, chosen by mm_set_actor_impl: the tcgen05 kernel (default) or, when set, the
// mma.sync kernel as the independent cross-check.  mm_actor_sample_mlp always runs the tcgen05 kernel.
static bool g_actor_mma = false;
void set_actor_impl(int impl) { g_actor_mma = impl == 1; }

template <int H1>
static int launch_actor_mlp_t(const float *obs, const int32_t *n_agents, int64_t n_rows, const float *w1, const float *b1,
                              const float *w2, const float *b2, const float *w3, const float *b3, const float *wv, const float *bv,
                              uint64_t seed, uint64_t step, const uint8_t *mask_bits, int8_t *actions, float *logp_all,
                              float *logp_sel, float *values, float *obs_copy, uint8_t *live_out, void *stream) {
    static bool ready[MM_MAX_DEVICES] = {};
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MM_MAX_DEVICES) return 1;
    if (!ready[dev]) {
        if (cudaFuncSetAttribute(actor_mlp_wg_kernel<H1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WgLayout<H1>::SMEM) != cudaSuccess)
            return 1;
        ready[dev] = true;
    }
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t n_tiles = (n_rows + 127) / 128, grid = n_tiles < sms ? n_tiles : sms;   // persistent: one CTA per SM
    actor_mlp_wg_kernel<H1><<<(unsigned)grid, WgLayout<H1>::THREADS, WgLayout<H1>::SMEM, (cudaStream_t)stream>>>(
        obs, n_agents, n_rows, w1, b1, w2, b2, w3, b3, wv, bv, seed, step, mask_bits, actions, logp_all, logp_sel, values, obs_copy,
        live_out);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int launch_actor_mlp(const float *obs, const int32_t *n_agents, int64_t n_rows, int h1, const float *w1, const float *b1,
                     const float *w2, const float *b2, const float *w3, const float *b3, const float *wv, const float *bv,
                     uint64_t seed, uint64_t step, const uint8_t *mask_bits, int8_t *actions, float *logp_all, float *logp_sel,
                     float *values, float *obs_copy, uint8_t *live_out, void *stream) {
    if (n_rows <= 0) return 0;
    if (h1 == 128)
        return launch_actor_mlp_t<128>(obs, n_agents, n_rows, w1, b1, w2, b2, w3, b3, wv, bv, seed, step, mask_bits, actions, logp_all,
                                       logp_sel, values, obs_copy, live_out, stream);
    if (h1 == 160)
        return launch_actor_mlp_t<160>(obs, n_agents, n_rows, w1, b1, w2, b2, w3, b3, wv, bv, seed, step, mask_bits, actions, logp_all,
                                       logp_sel, values, obs_copy, live_out, stream);
    return 2;
}

// The lambda-return R_t = r_t + gamma * (lambda R_{t+1} + (1 - lambda) V_{t+1}), restarted after a terminal step, for every
// (env, agent) column of a rollout at once.  rewards / values / out [T][n_cols], dones [T][n_cols / cols_per_env] (1 where
// step t ended the episode of that env), final_value [n_cols] (R and V after the last step; ignored where the last step was
// terminal).  values == nullptr is lambda = 1, the discounted return of MAPPO._discount_reward (marl/mappo.py:364-370):
// run = run * gamma + r, the expression mm_discounted_returns has always computed.  With values the mix is rounded
// product by product (__fmul_rn / __fadd_rn, never contracted whatever -fmad says), so lambda = 1 gives
// 1 * run + 0 * v == run and the same bits as without values (up to the sign of a zero run); values[t][c] is read only
// when step t - 1 did not end the episode, and a non-finite value there would turn 0 * v into NaN.
__global__ void __launch_bounds__(256) discounted_returns_kernel(const float *__restrict__ rewards,
                                                                 const uint8_t *__restrict__ dones,
                                                                 const float *__restrict__ values,
                                                                 const float *__restrict__ final_value, float gamma, float lambda,
                                                                 int T, int64_t n_cols, int cols_per_env, float *__restrict__ out) {
    const int64_t n_env = n_cols / cols_per_env;
    const float one_minus_lambda = __fsub_rn(1.f, lambda);
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_cols; c += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = c / cols_per_env;
        float run = final_value ? final_value[c] : 0.f, v_next = run;
        for (int t = T - 1; t >= 0; --t) {
            if (dones[(int64_t)t * n_env + e]) run = v_next = 0.f;
            if (values) {
                run = __fadd_rn(__fmul_rn(lambda, run), __fmul_rn(one_minus_lambda, v_next));
                v_next = values[(int64_t)t * n_cols + c];
            }
            run = run * gamma + rewards[(int64_t)t * n_cols + c];
            out[(int64_t)t * n_cols + c] = run;
        }
    }
}

int launch_discounted_returns(const float *rewards, const uint8_t *dones, const float *values, const float *final_value,
                              float gamma, float lambda, int T, int64_t n_cols, int cols_per_env, float *out, void *stream) {
    if (n_cols <= 0 || T <= 0) return 0;
    int64_t blocks = (n_cols + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    discounted_returns_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(rewards, dones, values, final_value, gamma,
                                                                               lambda, T, n_cols, cols_per_env, out);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int launch_actor_sample(const float *obs, const int32_t *n_agents, int64_t n_rows, const float *w1, const float *b1,
                        const float *w2, const float *b2, const float *w3, const float *b3, uint64_t seed, uint64_t step,
                        const uint8_t *mask_bits, int8_t *actions, float *logp_all, float *logp_sel, void *stream) {
    if (n_rows <= 0) return 0;
    if (!g_actor_mma)
        return launch_actor_mlp(obs, n_agents, n_rows, 128, w1, b1, w2, b2, w3, b3, nullptr, nullptr, seed, step, mask_bits, actions,
                                logp_all, logp_sel, nullptr, nullptr, nullptr, stream);
    static bool ready[MM_MAX_DEVICES] = {};
    const int smem = AC_SMEM_WORDS * (int)sizeof(uint32_t);
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MM_MAX_DEVICES) return 1;
    if (!ready[dev]) {
        if (cudaFuncSetAttribute(actor_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return 1;
        ready[dev] = true;
    }
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int64_t tiles = (n_rows + 15) / 16, ctas = (tiles + AC_THREADS / 32 - 1) / (AC_THREADS / 32);
    if (ctas > sms) ctas = sms;   // persistent: one CTA per SM, warps stride over the 16-row tiles
    actor_sample_kernel<<<(unsigned)ctas, AC_THREADS, smem, (cudaStream_t)stream>>>(obs, n_agents, n_rows, w1, b1, w2, b2, w3,
                                                                                     b3, seed, step, mask_bits, actions, logp_all, logp_sel);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace mm

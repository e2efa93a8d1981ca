// merge_step.cu — sm_100a kernels of the batched merge environment and its HSS / MASS CBF shields.
//
// One thread advances one environment by one whole policy step (3 physics sub-steps, each = ordered
// act() pass + ordered step() pass with the shield inside + pairwise collision pass), then builds the
// KinematicLC observations, local/regional rewards, terminal flags and info scalars.  Within an env the
// reference semantics are strictly sequential (front-to-back by x: a follower's shield reads its leader's
// already-updated position, shielded action and pre-step record), so the parallel axis is the env axis.
//
// Memory plan per thread: the four fields every neighbour scan touches (x, y, heading, speed) and the packed
// discrete state live in shared memory as [slot][thread] planes (bank-conflict free for any per-thread slot
// index); the colder fields stay in HBM/L2 as [field][slot][env] planes and are touched O(1) times per
// vehicle per sub-step.  Arithmetic is IEEE double, compiled with -fmad=false, so that every threshold
// decision (lane argmin, neighbour order, crash test, veto, active set) reproduces the float64 reference.
//
// Reference map (paths relative to the reference tree):
//   sub-step driver ............ highway_env/envs/common/abstract.py:512-532, road/road.py:269-292
//   CAV controllers ............ vehicle/controller.py:90-197, 293-337
//   HDV IDM + MOBIL ............ vehicle/behavior.py:74-266, road/road.py:352-381
//   bicycle model, collisions .. vehicle/kinematics.py:122-209, vehicle/safe_controller.py:100-185, utils.py:55-121
//   lane algebra ............... road/lane.py:61-210, road/road.py:51-109
//   shields .................... vehicle/safety/decentral_layer.py:15-817, vehicle/safety/cbf.py:110-430
//   observation / rewards ...... envs/common/observation.py:181-273, envs/merge_env_v1.py:64-178,373-474
#include <cuda_runtime.h>
#include <math_constants.h>
#include <cstdlib>
#include "mm_internal.h"
#include "spawn_core.h"

// Other builds of the step kernel: a small translation unit defines one of the macros below and includes this file; the
// kernel then lives in its own namespace and only its launcher is exported.
//   MM_VARIANT4 (merge_step_occ4.cu): built for FOUR CTAs per SM - x, y, heading, speed staged (cos / sin of the heading
//     stay in the L2-resident tile), 128 registers.  A grid that fits one wave of 4 CTAs / SM but not one of 3 (e.g.
//     65 536 envs = 512 CTAs on 148 SMs) otherwise runs a second, almost empty wave: 2 x the CTA latency instead of 1.3 x.
//   MM_SPEC_SHIELD = MM_SHIELD_MASS | MM_SHIELD_HSS (merge_step_spec_mass.cu / _hss.cu): specialised at compile time for
//     the benchmark configurations - every vehicle a CAV (no IDM / MOBIL code, no second act pass), env id
//     merge-multi-agent-v1 with lateral_control = "steer", the shield kind a constant.  Same source, same arithmetic;
//     launch_step picks it when the handle's config matches and no env can hold an HDV.
#if defined(MM_VARIANT4) && defined(MM_SPEC_SHIELD)      // both: merge_step_spec_mass4.cu / _hss4.cu
#define MM_SPEC 1
#define MM_NHOT 4
#ifndef MM_MIN_BLOCKS
#define MM_MIN_BLOCKS 4
#endif
#if MM_SPEC_SHIELD == 2
#define MM_KNS mms_mass4
#define MM_VARIANT_LAUNCH launch_step_spec_mass4
#else
#define MM_KNS mms_hss4
#define MM_VARIANT_LAUNCH launch_step_spec_hss4
#endif
#elif defined(MM_VARIANT4)
#define MM_KNS mm4
#define MM_NHOT 4
#ifndef MM_MIN_BLOCKS
#define MM_MIN_BLOCKS 4
#endif
#define MM_VARIANT_LAUNCH launch_step_occ4
#elif defined(MM_SPEC_SHIELD)
#define MM_SPEC 1
#define MM_NHOT 6
#if MM_SPEC_SHIELD == 2
#define MM_KNS mms_mass
#define MM_VARIANT_LAUNCH launch_step_spec_mass
#else
#define MM_KNS mms_hss
#define MM_VARIANT_LAUNCH launch_step_spec_hss
#endif
#else
#define MM_KNS mm
#define MM_NHOT 6
#endif
#ifdef MM_VARIANT_LAUNCH
#define MM_VARIANT_TU 1
#endif
#ifndef MM_PW
#define MM_PW MM_TILE
#endif
#define MM_TPE 1
// one call site per kernel: inline, the shield reads the env's order words and counts from the caller's registers (as an
// out-of-line function it took them through the stack: 152 -> 140 registers, 144 -> 48 bytes of stack in the MASS build)
#ifndef MM_SHIELD_FN
#define MM_SHIELD_FN __forceinline__
#endif
// likewise the steering law and the libdevice trigonometry (same code, same bits: only the call, its argument moves
// and the convergence barriers around it go): 8.02 -> 7.75 ms per 2^20-env step; tan / atan / asin stay calls in the
// generic builds, which measured 2 % faster that way with HDVs present (profiles/r2_z_ab_inline*.txt)
#ifndef MM_STEER_FN
#define MM_STEER_FN __forceinline__
#endif
#ifndef MM_HDV_FN            // IDM / MOBIL helpers (they took `Env &`): mixed traffic 0.905 -> 0.783 ms at 65 536 envs
#define MM_HDV_FN __forceinline__
#endif
#ifndef MM_TRIG_FN
#define MM_TRIG_FN __forceinline__
#endif
#if !defined(MM_TRIG1_FN) && defined(MM_SPEC_SHIELD)
#define MM_TRIG1_FN __forceinline__
#endif
#include "mm_device.cuh"
#include "mm_philox.cuh"

namespace MM_KNS {

// ------------------------------------------------------------------------------------------------
// the policy-step kernel
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// TMA bulk copies (cp.async.bulk, 1-D): the hot planes of a tile - x, y, heading, speed = the first four fields,
// 48 KB contiguous, and the 6 KB flags plane - move between HBM and shared memory as two bulk transactions issued
// by one thread, completion signalled on an mbarrier (load) / a bulk async-group (store).
// ------------------------------------------------------------------------------------------------
constexpr uint32_t HOT_FIELD_BYTES = (uint32_t)SMV * TILE * sizeof(double);       // 11 of the 12 slots of one field
constexpr uint32_t HOT_FLAG_BYTES = (uint32_t)MAXV * TILE * sizeof(uint32_t);

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// issue: called by every thread of the CTA; thread 0 arms the barrier and starts the copies.  wait: every thread spins on
// the barrier's phase.  Between the two the caller issues its own global loads (env scalars, the action tuple) so that
// their latency overlaps the tile transfer instead of following it.
__device__ __forceinline__ void tile_bulk_load_issue(const DevState &st, size_t tile, uint64_t *mbar) {
    const uint32_t bar = smem_u32(mbar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double *g64 = st.f64 + tile * (size_t)F_COUNT * MAXV * TILE;
        const uint32_t *gfl = st.flags + tile * (size_t)MAXV * TILE;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(N_HOT * HOT_FIELD_BYTES + HOT_FLAG_BYTES) : "memory");
#pragma unroll
        for (int f = 0; f < N_HOT; ++f)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(sm_planes + f * SMV * BLOCK)), "l"(g64 + (size_t)f * MAXV * TILE), "r"(HOT_FIELD_BYTES), "r"(bar) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(sm_planes + N_HOT * SMV * BLOCK)), "l"(gfl), "r"(HOT_FLAG_BYTES), "r"(bar) : "memory");
    }
}
__device__ __forceinline__ void tile_bulk_load_wait(uint64_t *mbar) {
    const uint32_t bar = smem_u32(mbar);
    uint32_t done = 0;
    while (!done) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar) : "memory");
    }
}

__device__ __forceinline__ void tile_bulk_store(const DevState &st, size_t tile) {
    // every thread: make its shared-memory writes visible to the async proxy, then one thread issues the copies
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
        double *g64 = st.f64 + tile * (size_t)F_COUNT * MAXV * TILE;
        uint32_t *gfl = st.flags + tile * (size_t)MAXV * TILE;
#pragma unroll
        for (int f = 0; f < N_HOT; ++f)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                         ::"l"(g64 + (size_t)f * MAXV * TILE), "r"(smem_u32(sm_planes + f * SMV * BLOCK)), "r"(HOT_FIELD_BYTES) : "memory");
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                     ::"l"(gfl), "r"(smem_u32(sm_planes + N_HOT * SMV * BLOCK)), "r"(HOT_FLAG_BYTES) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // shared memory may be released after this
    }
}

__device__ __forceinline__ void load_env(Env &ev, const DevState &st, size_t e) {
    const uint32_t *fl = st.flags + flags_index(e, 0);
    for (int i = 0; i < ev.n_veh; ++i) {
#pragma unroll
        for (int f = 0; f < N_HOT; ++f) SMF(f, i) = GF(f, i);
        FL(i) = fl[i * TILE];
    }
}
__device__ __forceinline__ void store_env(const Env &ev, const DevState &st, size_t e) {
    uint32_t *fl = st.flags + flags_index(e, 0);
    for (int i = 0; i < ev.n_veh; ++i) {
#pragma unroll
        for (int f = 0; f < N_HOT; ++f) GF(f, i) = SMF(f, i);
        fl[i * TILE] = FL(i);
    }
}

// Shield counters of one policy step (solves, active QPs, lane-change vetoes), summed over the 32 envs of a warp and added
// to that warp's row of partial sums: no atomics on the step path; mm_stats() folds the rows.  (The other statistics are
// accumulated by the outputs kernel into the same rows.)
__device__ __forceinline__ void flush_shield_counts(uint32_t shield_counts, double *stats, size_t first_env_of_warp) {
    const unsigned full = 0xffffffffu;
    // three 10-bit counters, each <= 33 per env: summed over 32 lanes they stay below 2^11 - widen before adding
    uint32_t a = shield_counts & 1023u, b = (shield_counts >> 10) & 1023u, c = (shield_counts >> 20) & 1023u;
    a = __reduce_add_sync(full, a);
    b = __reduce_add_sync(full, b);
    c = __reduce_add_sync(full, c);
    if ((threadIdx.x & 31) == 0) {
        double *row = stats + (first_env_of_warp >> 5) * N_STATS;
        row[ST_SOLVES] += (double)a;
        row[ST_ACTIVE] += (double)b;
        row[ST_VETOES] += (double)c;
    }
}

// MM_PHASE_SYNC: CTA-wide barriers that keep the four warps of a CTA in the same phase of the step, so that they
// share instruction-cache lines (the kernel is ~130 KB of SASS; instruction fetch was a top stall without them).
//   0: none   1: one barrier per sub-step   2: additionally one per vehicle rank inside the act / step passes
//   3: additionally one between a rank's control law and its shield + move (experiment)
#ifndef MM_PHASE_SYNC
#define MM_PHASE_SYNC 2
#endif
#ifndef MM_SORT_LANES
#define MM_SORT_LANES 0   // measured: < 1 % (profiles/README.md); kept as an experiment knob
#endif
#ifndef MM_RANK_BARRIER_STRIDE
#define MM_RANK_BARRIER_STRIDE 1   // experiment knob: a barrier every n-th rank of the step loop
#endif
#define PHASE_BARRIER(level) do { if (MM_PHASE_SYNC >= (level)) __syncthreads(); } while (0)

// The 12 action bytes of an env as 12 nibbles (out-of-range bytes read as IDLE).  Packed right behind the loads, before
// the sub-step loop: the loop then reads a register that is known to have arrived.  (Selecting from the three loaded
// words inside the loop made ptxas wait there, every rank, on a scoreboard it shares with the two cold-field prefetches
// issued just above - their L2 round trip, meant to overlap the steering law, was exposed: 3.4 % of the stall samples.)
__device__ __forceinline__ uint64_t pack_actions(uint32_t lo, uint32_t mid, uint32_t hi) {
    uint64_t acts = 0;
#pragma unroll
    for (int k = 0; k < MAXV; ++k) {
        const uint32_t w = k < 4 ? lo : (k < 8 ? mid : hi);
        const uint32_t b = (w >> (8 * (k & 3))) & 0xffu;
        acts |= (uint64_t)(b <= 4u ? b : (uint32_t)A_IDLE) << (4 * k);
    }
    return acts;
}
__device__ __forceinline__ int meta_action(uint64_t acts, int i) { return (int)((acts >> (4 * i)) & 7u); }

// DYN_RANKS: the rank loops run to the largest vehicle count of the CTA's envs instead of MAXV - 1.  Only worth a
// second instantiation when the envs of a tile share their counts (mm_config.couple_counts); with independent counts
// some env of 128 almost always has 11 vehicles, and the constant trip count compiles to the faster loop.
template <bool DIAG, bool DYN_RANKS>
__global__ void __launch_bounds__(BLOCK, MM_MIN_BLOCKS) step_kernel(const __grid_constant__ StepParams p) {
    const int tid = threadIdx.x;
#if MM_SORT_LANES
    // Lane <-> env assignment inside the CTA is free: give each warp envs with (nearly) the same vehicle count, so
    // that the per-rank loops do not idle lanes (counts are 7..11 at hard density).  Stable counting sort of the
    // CTA's 128 envs by n_veh with warp ballots; deterministic.
    __shared__ int s_wcnt[BLOCK / 32][16];
    __shared__ unsigned char s_perm[BLOCK];
    {
        const int l0 = blockIdx.x * BLOCK + tid;
        int key = 15;
        if (l0 < p.env_count) key = (int)((p.st.einfo[(size_t)p.env_offset + l0] >> EI_NVEH_SHIFT) & EI_4BIT);
        const int warp = tid >> 5, lane = tid & 31;
        int rank_in_warp = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            unsigned m = __ballot_sync(0xffffffffu, key == k);
            if (lane == 0) s_wcnt[warp][k] = __popc(m);
            if (key == k) rank_in_warp = __popc(m & ((1u << lane) - 1u));
        }
        __syncthreads();
        int pos = rank_in_warp;
        for (int k = 0; k < 16; ++k)
            for (int w = 0; w < BLOCK / 32; ++w)
                if (k < key || (k == key && w < warp)) pos += s_wcnt[w][k];
        s_perm[pos] = (unsigned char)tid;
        __syncthreads();
    }
    const int local = blockIdx.x * BLOCK + (int)s_perm[tid];
#else
    const int local = blockIdx.x * BLOCK + tid;
#endif
    const bool valid = local < p.env_count;
    const size_t e = (size_t)p.env_offset + (valid ? local : 0);

    Env ev;
    ev.tid = tid;
    ev.g = p.st.f64 + f64_index(e, 0, 0);
    ev.n_veh = 0;
    ev.n_cav = 0;
    ev.live = 0;
    ev.pos = 0;
    uint32_t ei = 0, act_lo = 0, act_mid = 0, act_hi = 0;
    int steps = 0, time = 0;
    __shared__ uint64_t s_mbar;
    const size_t tile = ((size_t)p.env_offset + (size_t)blockIdx.x * BLOCK) / TILE;   // launches are tile-aligned
    if (tid == 0) {
        s_tile_g = p.st.f64 + tile * (size_t)F_COUNT * MAXV * TILE;
        s_cfgd[0] = p.cfg.dt; s_cfgd[1] = p.cfg.eta; s_cfgd[2] = p.cfg.tau;
    }
    if (MM_TMA) tile_bulk_load_issue(p.st, tile, &s_mbar);   // (contains the CTA barrier that publishes the two above)
    else __syncthreads();
    if (valid) {
        // env scalars and the 12 action bytes: requested while the tile is in flight
        ei = p.st.einfo[e];
        const uint32_t *a32 = reinterpret_cast<const uint32_t *>(p.actions + e * MAXV);
        act_lo = a32[0]; act_mid = a32[1]; act_hi = a32[2];
    }
    if (MM_TMA) tile_bulk_load_wait(&s_mbar);
    const uint64_t acts = pack_actions(act_lo, act_mid, act_hi);
    if (valid) {
        ev.n_veh = (ei >> EI_NVEH_SHIFT) & EI_4BIT;
        ev.n_cav = (ei >> EI_NCAV_SHIFT) & EI_4BIT;
        steps = (ei >> EI_STEPS_SHIFT) & EI_STEPS_MASK;
        time = (ei >> EI_TIME_SHIFT) & EI_TIME_MASK;
        if (!MM_TMA) load_env(ev, p.st, e);
        if (DIAG) {
            size_t plane = (size_t)p.n_envs * 3 * MAXV;
            for (int k = 0; k < 3 * MAXV; ++k) {
                size_t idx = e * 3 * MAXV + k;
                p.out.sh_i[idx] = 0;
                p.out.sh_i[plane + idx] = MM_NB_NONE; p.out.sh_i[2 * plane + idx] = MM_NB_NONE;
                p.out.sh_i[3 * plane + idx] = MM_NB_NONE;
                p.out.sh_i[4 * plane + idx] = 0; p.out.sh_i[5 * plane + idx] = 0; p.out.sh_i[6 * plane + idx] = 0;
                p.out.sh_i[7 * plane + idx] = 0; p.out.sh_i[8 * plane + idx] = -1; p.out.sh_i[9 * plane + idx] = 0;
                for (int q = 0; q < 10; ++q) p.out.sh_f[q * plane + idx] = 0.0;
            }
        }
        steps = min(steps + 1, (int)EI_STEPS_MASK);  // abstract.py:457
    }
    bool running = valid;
    uint32_t shield_counts = 0;
    const bool sv = CFG_STEER_VEL(p.cfg) && !CFG_V0(p.cfg);
    // All-CAV envs: a CAV's act() reads and writes only its own state (controller.py:90-134), so it can run right
    // before that vehicle's step() instead of in a separate pass; the result is identical and the action never
    // leaves registers.  With HDVs present the two ordered passes are kept (MOBIL reads the others' target lanes).
    // The choice is made per CTA so that the barriers below stay uniform.
    const bool merged = MM_SPEC ? true : __syncthreads_and(!valid || ev.n_cav == ev.n_veh) != 0;
    // uniform trip count when ranks are barrier-separated: the largest vehicle count of the CTA's envs
    int n_rank = MM_PHASE_SYNC >= 2 ? MAXV - 1 : 0;
    if (DYN_RANKS && MM_PHASE_SYNC >= 2)
        while (n_rank > 0 && !__syncthreads_or(ev.n_veh >= n_rank)) --n_rank;
#pragma unroll 1
    for (int sub = 0; sub < p.cfg.substeps; ++sub) {  // abstract.py:514-531
        PHASE_BARRIER(1);
        uint64_t ord = 0;
        const bool apply_meta = running && (time % p.cfg.substeps == 0);   // abstract.py:516-519
        if (running) {
            if (apply_meta && !merged) {
                for (int i = 0; i < ev.n_cav; ++i) {
                    double st_, ac_;
                    cav_act(ev, i, meta_action(acts, i), sv, st_, ac_);
                }
            }
            // road.py:277,286: stable sort by x, descending.  After the first sub-step the live order of the previous
            // one is that order unless two vehicles share an x (stability then decides by slot id: sort again).
            bool resort = sub == 0;
            if (!resort) {
                double prev = X(nib(ev.live, 0));
                for (int q = 1; q < ev.n_veh; ++q) {
                    double xq = X(nib(ev.live, q));
                    resort |= xq == prev;
                    prev = xq;
                }
            }
            if (resort) {
                ev.live = order_by_x_desc(ev);
                ev.pos = invert_order(ev.live, ev.n_veh);
            }
            ord = ev.live;
        }
        const int n_live = running ? ev.n_veh : 0;
        if (!merged) {
#pragma unroll 1
            for (int q = 0; q < (MM_PHASE_SYNC >= 2 ? n_rank : n_live); ++q) {  // road.act()
                PHASE_BARRIER(2);
                if (q < n_live) {
                    int i = (int)((ord >> (4 * q)) & 15u);
                    if (is_cav(FL(i))) {
                        double st_, ac_;
                        cav_act(ev, i, A_NONE, sv, st_, ac_);
                        GF(F_ACT_STEER, i) = st_;
                        GF(F_ACT_ACC, i) = ac_;
                    } else {
                        hdv_act(ev, i);
                    }
                }
            }
        }
#pragma unroll 1
        for (int q = 0; q < (MM_PHASE_SYNC >= 2 ? n_rank : n_live); ++q) {  // road.step(dt): same order
            if (MM_RANK_BARRIER_STRIDE == 1 || q % MM_RANK_BARRIER_STRIDE == 0) PHASE_BARRIER(2);
            int i = 0;
            double rec1vx = 0, ge = 0, st_ = 0, ac_ = 0;
            if (q < n_live) {
                i = (int)((ord >> (4 * q)) & 15u);
                // the two cold fields of the ego the step needs, requested before the steering law so that their L2
                // round trip overlaps it
                rec1vx = GF(F_REC1VX, i);
                ge = GF(F_GVX, i);
                if (merged) {
                    // sub-step 0 calls act(meta) and then act(None); the second call recomputes the same controls
                    cav_act(ev, i, apply_meta ? meta_action(acts, i) : A_NONE, sv, st_, ac_);
                } else {
                    st_ = GF(F_ACT_STEER, i);
                    ac_ = GF(F_ACT_ACC, i);
                }
            }
            PHASE_BARRIER(3);
            if (q < n_live) vehicle_step<DIAG>(ev, p, i, sub < 3 ? sub : 2, e, shield_counts, st_, ac_, rec1vx, ge);
        }
        PHASE_BARRIER(2);
        if (running) {
            if (uint32_t close = close_pair_mask(ev)) collision_pass(ev, close);
            time = min(time + 1, (int)EI_TIME_MASK);
            if (is_terminal(ev, steps, p.cfg)) running = false;  // abstract.py:530
        }
    }
    PHASE_BARRIER(1);
    if (valid) {
        if (!MM_TMA) store_env(ev, p.st, e);
        p.st.einfo[e] = (ei & 0xfffu) | ((uint32_t)steps << EI_STEPS_SHIFT) | ((uint32_t)time << EI_TIME_SHIFT);
    }
    if (MM_TMA) tile_bulk_store(p.st, tile);
    flush_shield_counts(shield_counts, p.out.stats, (size_t)p.env_offset + (size_t)((blockIdx.x * BLOCK + tid) & ~31));
}

#ifndef MM_VARIANT_TU
// ------------------------------------------------------------------------------------------------
// device-side spawn (merge_env_v1.py:180-211, 265-364; abstract.py:176-199) with Philox4x32-10
// ------------------------------------------------------------------------------------------------
// The constructor writes of slot i of the env whose field base is g (Vehicle / ControlledVehicle / MDPLCVehicle /
// IDMVehicle.__init__ at heading 0): every f64 field cleared, then position, speed, target speed, the IDM timer,
// min_headway and cos(heading) = 1; returns the flags word.  kind MM_KIND_NONE leaves the slot empty with flags
// `empty_flags`.  The two spawns differ only in what they leave where the reference has no value: reset_kernel writes
// min_headway 4.5 into every slot and flags 0 into empty ones, mm_set_state of a spawn.py scene 0 for the HDVs and empty
// slots and hl_action None (-1 on the host) into empty ones.
__device__ __forceinline__ uint32_t construct_vehicle(double *g, int i, int kind, double x, double y, double speed,
                                                      double min_headway, uint32_t empty_flags) {
    uint32_t f = empty_flags;
    double tspeed = 0, timer = 0;
    if (kind != MM_KIND_NONE) {
        const bool cav = kind == MM_KIND_CAV;
        int lane = closest_lane(x, y, 0.0);
        int sidx = 0;
        if (cav) {
            sidx = speed_to_index(speed);
            tspeed = 10.0 + sidx * (30.0 - 10.0) / 4;
        } else {
            tspeed = speed;
            timer = pymod_pos((x + y) * PI, 1.0);  // behavior.py:54
        }
        f = (uint32_t)kind | ((uint32_t)lane << FL_LANE_SHIFT) | ((uint32_t)lane << FL_TLANE_SHIFT) |
            ((uint32_t)sidx << FL_SIDX_SHIFT) | ((uint32_t)A_NONE << FL_HL_SHIFT);
    }
    for (int fld = 0; fld < F_COUNT; ++fld) g[(fld * MAXV + i) * TILE] = 0.0;
    g[(F_X * MAXV + i) * TILE] = x;
    g[(F_Y * MAXV + i) * TILE] = y;
    g[(F_V * MAXV + i) * TILE] = speed;
    g[(F_TSPEED * MAXV + i) * TILE] = tspeed;
    g[(F_TIMER * MAXV + i) * TILE] = timer;
    g[(F_MINHW * MAXV + i) * TILE] = min_headway;
    g[(F_COSH * MAXV + i) * TILE] = 1.0;            // heading 0
    return f;
}

__global__ void __launch_bounds__(BLOCK) reset_kernel(const __grid_constant__ ResetParams p) {
    const int local = blockIdx.x * BLOCK + threadIdx.x;
    if (local >= p.env_count) return;
    const size_t e = (size_t)p.env_offset + local;
    if (p.use_done) { if (!p.out.done[e]) return; }
    else if (p.mask && !p.mask[e]) return;

    uint32_t episode = p.st.episode[e];
    p.st.episode[e] = episode + 1;
    Philox rng(p.seed, (uint64_t)e, episode);

    // _num_vehicles (merge_env_v1.py:180-211, 476-495)
    int lo_c, lo_h;
    switch (p.cfg.traffic_density) {
        case 1: lo_c = 1; lo_h = 1; break;
        case 2: lo_c = 2; lo_h = 2; break;
        default: lo_c = 4; lo_h = 3; break;
    }
    // couple_counts: the two count draws come from a stream keyed by the TILE (and the env's episode number), so the
    // envs of a tile that re-spawn together share (n_CAV, n_HDV); the env's own stream still makes the two draws, so
    // everything after them is the same whichever way the counts were drawn
    int d_cav = p.num_cav > 0 ? 0 : rng.below(3);
    int d_hdv = rng.below(3);
    if (p.cfg.couple_counts) {
        Philox tile_rng(p.seed ^ 0x7469'6c65'636e'7473ull, (uint64_t)(e / TILE), episode);
        d_cav = tile_rng.below(3);
        d_hdv = tile_rng.below(3);
    }
    int n_cav = p.num_cav > 0 ? p.num_cav : lo_c + d_cav;
    int n_hdv = lo_h + d_hdv;
    if (p.cfg.traffic_type == MM_TRAFFIC_CAV) { n_cav += n_hdv; n_hdv = 0; }
    else if (p.cfg.traffic_type == MM_TRAFFIC_AV) { n_hdv = n_cav + n_hdv - 1; n_cav = 1; }   // merge_env_v1.py:485-489
    else if (p.cfg.traffic_type == MM_TRAFFIC_HDV) { n_hdv = n_cav + n_hdv; n_cav = 0; }      // merge_env_v1.py:490-494
    if (n_cav + n_hdv > 11) n_cav = 11 - n_hdv;

    // spawn slots without replacement: main [10,60,...,260], ramp [5,55,...,255] (merge_env_v1.py:284-319)
    int main_slots[6] = {0, 1, 2, 3, 4, 5}, ramp_slots[6] = {0, 1, 2, 3, 4, 5};
    for (int k = 0; k < 5; ++k) {  // Fisher-Yates: a uniformly random order of the six slots of each road
        int j = k + rng.below(6 - k);
        int t = main_slots[k]; main_slots[k] = main_slots[j]; main_slots[j] = t;
        j = k + rng.below(6 - k);
        t = ramp_slots[k]; ramp_slots[k] = ramp_slots[j]; ramp_slots[j] = t;
    }
    int n_s_c = n_cav != 1 ? n_cav / 2 : rng.below(2);
    int n_m_c = n_cav - n_s_c;
    int n_s_h = n_hdv != 1 ? n_hdv / 2 : rng.below(2);
    int n_m_h = n_hdv - n_s_h;
    if (n_s_c + n_s_h > 6) n_s_h = 6 - n_s_c;
    if (n_m_c + n_m_h > 6) n_m_h = 6 - n_m_c;
    int n_veh = n_s_c + n_m_c + n_s_h + n_m_h;
    n_hdv = n_s_h + n_m_h;

    int mi = 0, ri = 0;
    double *g = p.st.f64 + f64_index(e, 0, 0);
    for (int i = 0; i < MAXV; ++i) {
        int kind = MM_KIND_NONE;
        double x = 0, y = 0, speed = 0;
        if (i < n_veh) {
            bool cav = i < n_cav;
            bool on_main = cav ? (i < n_s_c) : (i - n_cav < n_s_h);
            double noise = rng.uniform() * 8 - 4;
            speed = rng.uniform() * 2 + 25;
            if (on_main) { x = 10.0 + 50.0 * main_slots[mi++] + noise; y = 0.0; }
            else { x = 5.0 + 50.0 * ramp_slots[ri++] + noise; y = 10.5; }
            kind = cav ? MM_KIND_CAV : MM_KIND_HDV;
        }
        p.st.flags[flags_index(e, i)] = construct_vehicle(g, i, kind, x, y, speed, 180.0 / 40.0 /* safe_controller.py:56 */, 0u);
    }
    p.st.einfo[e] = (uint32_t)n_veh | ((uint32_t)n_cav << EI_NCAV_SHIFT) | ((uint32_t)n_m_c << EI_NMERGE_SHIFT);
}

// The reference's own scene for each env's test seed (spawn_core.h: its MT19937 draws), written as mm_set_state leaves
// the state spawn.spawn_state builds for it: the same f64 fields (cold ones cleared), flags and einfo; the episode
// counters are not touched (mm_set_state leaves them too).  Arguments checked by mm_reset_seeded: every scene fits.
__global__ void __launch_bounds__(BLOCK) seeded_reset_kernel(const __grid_constant__ SeededResetParams p) {
    const int e = blockIdx.x * BLOCK + threadIdx.x;
    if (e >= p.n_envs) return;
    mmspawn::MT19937 mt;
    mmspawn::Scene sc;
    mmspawn::spawn_scene((uint32_t)p.seeds[e], p.cfg.traffic_density, p.cfg.traffic_type, p.num_cav ? p.num_cav[e] : 0,
                         sc, mt);
    double *g = p.st.f64 + f64_index(e, 0, 0);
    for (int i = 0; i < MAXV; ++i) {
        const bool live = i < sc.n_veh;
        const int kind = live ? sc.kind[i] : MM_KIND_NONE;
        p.st.flags[flags_index(e, i)] = construct_vehicle(g, i, kind, live ? sc.x[i] : 0.0, live ? sc.y[i] : 0.0,
                                                          live ? sc.speed[i] : 0.0, kind == MM_KIND_CAV ? 180.0 / 40.0 : 0.0,
                                                          (uint32_t)A_NONE << FL_HL_SHIFT);
    }
    p.st.einfo[e] = (uint32_t)sc.n_veh | ((uint32_t)sc.n_cav << EI_NCAV_SHIFT) | ((uint32_t)sc.n_merge << EI_NMERGE_SHIFT);
}

// ------------------------------------------------------------------------------------------------
// state (un)packing between the env-major host mirror and the SoA planes
// ------------------------------------------------------------------------------------------------
// host mirror field order (mm_state_host): f64: x y heading speed target_speed gvx rec1_x rec1_vx rec2_x rec2_vx
// act_steer act_acc safe_steer safe_acc timer min_headway steering_angle; i32: kind lane target_lane speed_index crashed
// hl_action hist_len fg_set is_collaborating is_lc_safe collaborate_adj; env: n_veh n_cav n_merge steps time
__constant__ int c_host_f64_to_field[17] = {F_X, F_Y, F_H, F_V, F_TSPEED, F_GVX, -1, F_REC1VX, F_REC2X, F_REC2VX,
                                            F_ACT_STEER, F_ACT_ACC, F_SAFE_STEER, F_SAFE_ACC, F_TIMER, F_MINHW, F_STEERANG};

__global__ void pack_state_kernel(DevState st, int n_envs, const double *f64_em, const int32_t *i32_em,
                                  const int32_t *env_em) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t E = (size_t)n_envs;
    if (idx >= E * MAXV) return;
    size_t e = idx / MAXV;
    int i = (int)(idx % MAXV);
    for (int k = 0; k < 17; ++k) {
        int fld = c_host_f64_to_field[k];
        if (fld >= 0) st.f64[f64_index(e, fld, i)] = f64_em[(size_t)k * E * MAXV + idx];
    }
    {
        double2 sc = m_sincos(f64_em[(size_t)2 * E * MAXV + idx]);   // host field 2 = heading
        st.f64[f64_index(e, F_COSH, i)] = sc.y;
        st.f64[f64_index(e, F_SINH, i)] = sc.x;
    }
    const size_t P = E * MAXV;
    int hl = i32_em[5 * P + idx];
    int hist = i32_em[6 * P + idx];
    uint32_t f = ((uint32_t)i32_em[0 * P + idx] & 3u) | (((uint32_t)i32_em[1 * P + idx] & 7u) << FL_LANE_SHIFT) |
                 (((uint32_t)i32_em[2 * P + idx] & 7u) << FL_TLANE_SHIFT) |
                 (((uint32_t)max(i32_em[3 * P + idx], 0) & 7u) << FL_SIDX_SHIFT) |
                 (i32_em[4 * P + idx] ? FL_CRASHED : 0u) | ((uint32_t)((hl >= 0 && hl <= 4) ? hl : A_NONE) << FL_HL_SHIFT) |
                 ((uint32_t)min(max(hist, 0), 2) << FL_HIST_SHIFT) | (i32_em[7 * P + idx] ? FL_FG : 0u) |
                 (i32_em[8 * P + idx] ? FL_COLLAB : 0u) | (i32_em[9 * P + idx] ? FL_LCSAFE : 0u) |
                 (i32_em[10 * P + idx] ? FL_CADJ : 0u);
    st.flags[flags_index(e, i)] = f;
    if (i == 0) {
        st.einfo[e] = ((uint32_t)env_em[e] & 15u) | (((uint32_t)env_em[E + e] & 15u) << EI_NCAV_SHIFT) |
                      (((uint32_t)env_em[2 * E + e] & 15u) << EI_NMERGE_SHIFT) |
                      (((uint32_t)min(env_em[3 * E + e], 255) & EI_STEPS_MASK) << EI_STEPS_SHIFT) |
                      (((uint32_t)min(env_em[4 * E + e], 4095) & EI_TIME_MASK) << EI_TIME_SHIFT);
    }
}

__global__ void unpack_state_kernel(DevState st, int n_envs, double *f64_em, int32_t *i32_em, int32_t *env_em) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t E = (size_t)n_envs;
    if (idx >= E * MAXV) return;
    size_t e = idx / MAXV;
    int i = (int)(idx % MAXV);
    for (int k = 0; k < 17; ++k) {
        int fld = c_host_f64_to_field[k];
        if (fld < 0) fld = F_X;  // rec1_x == x (the record is taken right after the move)
        f64_em[(size_t)k * E * MAXV + idx] = st.f64[f64_index(e, fld, i)];
    }
    const size_t P = E * MAXV;
    uint32_t f = st.flags[flags_index(e, i)];
    int hl = fl_hl(f);
    i32_em[0 * P + idx] = fl_kind(f);
    i32_em[1 * P + idx] = fl_lane(f);
    i32_em[2 * P + idx] = fl_tlane(f);
    i32_em[3 * P + idx] = fl_kind(f) == MM_KIND_CAV ? (int)((f >> FL_SIDX_SHIFT) & 7u) : (fl_kind(f) ? -1 : 0);
    i32_em[4 * P + idx] = (f & FL_CRASHED) ? 1 : 0;
    i32_em[5 * P + idx] = hl == A_NONE ? -1 : hl;
    i32_em[6 * P + idx] = fl_hist(f);
    i32_em[7 * P + idx] = (f & FL_FG) ? 1 : 0;
    i32_em[8 * P + idx] = (f & FL_COLLAB) ? 1 : 0;
    i32_em[9 * P + idx] = (f & FL_LCSAFE) ? 1 : 0;
    i32_em[10 * P + idx] = (f & FL_CADJ) ? 1 : 0;
    if (i == 0) {
        uint32_t ei = st.einfo[e];
        env_em[e] = (ei >> EI_NVEH_SHIFT) & EI_4BIT;
        env_em[E + e] = (ei >> EI_NCAV_SHIFT) & EI_4BIT;
        env_em[2 * E + e] = (ei >> EI_NMERGE_SHIFT) & EI_4BIT;
        env_em[3 * E + e] = (ei >> EI_STEPS_SHIFT) & EI_STEPS_MASK;
        env_em[4 * E + e] = (ei >> EI_TIME_SHIFT) & EI_TIME_MASK;
    }
}

// ------------------------------------------------------------------------------------------------
// ragged observation rows for the host path (mm_step_host_ragged)
// ------------------------------------------------------------------------------------------------
// The reference returns obs as an [A, n_s] array per env (merge_env_v1.py:164): only the agents that exist.  The
// dense device buffer [E][12][30] keeps zero rows for the absent ones; over PCIe those rows are a quarter of the
// bytes at hard density.  Pass 1: exclusive scan of n_agents over the chunk -> first row of every env and the chunk's
// row count.  Pass 2: each warp moves one env's live rows (the leading rows of its block) to their packed place in a
// device staging buffer, from where the copy engine takes exactly the packed bytes.  (Storing the rows straight into
// mapped pinned memory from the kernel was measured too: 31 GB/s against 49 GB/s for the copy engine.)
__global__ void __launch_bounds__(1024) ragged_offsets_kernel(const int32_t *__restrict__ n_agents, int count,
                                                              int64_t base_row, int64_t *__restrict__ row_offset,
                                                              int64_t *__restrict__ chunk_rows) {
    // one CTA, 32 warps, each walking a contiguous segment 32 envs at a time: coalesced loads, warp scans (see
    // packed_offsets_kernel in merge_outputs.cu; a private run of envs per thread cost 52 us per chunk)
    __shared__ int warp_sum[32];
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int seg = ((count + 31) / 32 + 31) / 32 * 32;
    const int lo = min(warp * seg, count), hi = min(lo + seg, count);
    int sum = 0;
    for (int e = lo + lane; e < hi; e += 32) sum += n_agents[e];
    sum = __reduce_add_sync(full, sum);
    if (lane == 0) warp_sum[warp] = sum;
    __syncthreads();
    if (warp == 0) {
        const int w = warp_sum[lane];
        int wi = w;
        for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_up_sync(full, wi, off);
            if (lane >= off) wi += v;
        }
        warp_sum[lane] = wi - w;   // exclusive
        if (lane == 31) *chunk_rows = wi;
    }
    __syncthreads();
    int64_t run = base_row + warp_sum[warp];
    for (int e0 = lo; e0 < hi; e0 += 32) {
        const int e = e0 + lane;
        const int n = e < hi ? n_agents[e] : 0;
        int incl = n;
        for (int off = 1; off < 32; off <<= 1) {
            const int v = __shfl_up_sync(full, incl, off);
            if (lane >= off) incl += v;
        }
        if (e < hi) row_offset[e] = run + incl - n;
        run += __shfl_sync(full, incl, 31);
    }
}

__global__ void __launch_bounds__(256) ragged_copy_kernel(const float *__restrict__ obs, const int32_t *__restrict__ n_agents,
                                                          const int64_t *__restrict__ row_offset, int count,
                                                          float *__restrict__ rows_out) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; e < count; e += warps) {
        const int n2 = n_agents[e] * (NS / 2);                                 // float2 elements of the live rows
        const float2 *src = reinterpret_cast<const float2 *>(obs + (size_t)e * MAXV * NS);
        float2 *dst = reinterpret_cast<float2 *>(rows_out + row_offset[e] * NS);
        for (int k = lane; k < n2; k += 32) dst[k] = __ldcs(src + k);
    }
}

void launch_ragged_pack(const float *obs, const int32_t *n_agents, int count, int64_t base_row, int64_t *row_offset_dev,
                        int64_t *chunk_rows_dev, float *rows_stage, void *stream) {
    if (count <= 0) return;
    ragged_offsets_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(n_agents, count, base_row, row_offset_dev, chunk_rows_dev);
    ragged_copy_kernel<<<(count + 7) / 8, 256, 0, (cudaStream_t)stream>>>(obs, n_agents, row_offset_dev, count, rows_stage);
}

// ------------------------------------------------------------------------------------------------
// stand-alone shield query (mm_shield_query): safety_layer(...) for every CAV of the current scenes, nothing stepped
// ------------------------------------------------------------------------------------------------
// decentral_layer.py:767-817 as the reference calls it from MDPLCVehicle.step: (nominal action, vehicle, road) -> (safe
// action, status).  One thread per env; the scene is copied to shared memory, every CAV is evaluated against the scene AS
// IT IS (no vehicle has moved: the view the front-most vehicle of a sub-step has), and nothing is written back.
struct ShieldQueryParams {
    DevState st;
    mm_config cfg;
    int n_envs;
    const double *nom_steer, *nom_acc;                 // [E][MAXV] clipped low-level action per CAV
    double *safe_steer, *safe_acc, *min_headway;       // [E][MAXV]
    int32_t *ran, *leader, *front_adj, *rear_adj, *constrain_adj, *active, *is_lc_safe;   // [E][MAXV]
};

__global__ void __launch_bounds__(BLOCK) shield_query_kernel(const __grid_constant__ ShieldQueryParams p) {
    const int tid = threadIdx.x;
    const int local = blockIdx.x * BLOCK + tid;
    if (tid == 0) {                                   // MM_TPE: one CTA = one tile (BLOCK == TILE, env 0 starts a tile)
        s_tile_g = p.st.f64 + (size_t)blockIdx.x * F_COUNT * MAXV * TILE;
        s_cfgd[0] = p.cfg.dt; s_cfgd[1] = p.cfg.eta; s_cfgd[2] = p.cfg.tau;
    }
    __syncthreads();
    if (local >= p.n_envs) return;
    const size_t e = (size_t)local;
    Env ev;
    ev.tid = tid;
    ev.g = p.st.f64 + f64_index(e, 0, 0);
    const uint32_t ei = p.st.einfo[e];
    ev.n_veh = (ei >> EI_NVEH_SHIFT) & EI_4BIT;
    ev.n_cav = (ei >> EI_NCAV_SHIFT) & EI_4BIT;
    load_env(ev, p.st, e);
    ev.live = order_by_x_desc(ev);
    ev.pos = invert_order(ev.live, ev.n_veh);
    for (int i = 0; i < MAXV; ++i) {
        const size_t k = e * MAXV + i;
        int ran = 0;
        ShieldRec rec{MM_NB_NONE, MM_NB_NONE, MM_NB_NONE, 0, 0, 1, 0.0, 0.0};
        double steer = 0.0, acc = 0.0;
        if (i < ev.n_cav) {
            const uint32_t f = FL(i);
            steer = p.nom_steer[k];
            acc = p.nom_acc[k];
            // get_safe_action gate (safe_controller.py:229-239)
            if (CFG_SHIELD(p.cfg) != MM_SHIELD_NONE && !CFG_V0(p.cfg) && (f & FL_FG) && fl_hist(f) >= 2) {
                const double nom_steer = steer, nom_acc = acc;
                shield<false, true>(ev, p.cfg, i, nom_steer, nom_acc, GF(F_REC1VX, i), GF(F_GVX, i), steer, acc, rec);
                FL(i) = f;          // the evaluation of one vehicle leaves no trace for the next one
                ran = 1;
            }
        }
        p.ran[k] = ran; p.leader[k] = rec.leader; p.front_adj[k] = rec.front_adj; p.rear_adj[k] = rec.rear_adj;
        p.constrain_adj[k] = rec.constrain_adj; p.active[k] = rec.active; p.is_lc_safe[k] = rec.is_lc_safe;
        p.safe_steer[k] = steer; p.safe_acc[k] = acc; p.min_headway[k] = ran ? rec.min_headway : 0.0;
    }
}

// ------------------------------------------------------------------------------------------------
// stand-alone QP kernel (solves/s microbenchmark, known-answer tests)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) qp_kernel(const double *__restrict__ a, const double *__restrict__ c_lead,
                                                 const double *__restrict__ c_adj, const uint8_t *__restrict__ has_adj,
                                                 const double *__restrict__ lo, const double *__restrict__ hi, int64_t n,
                                                 double *__restrict__ u, uint8_t *__restrict__ active) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int act;
        u[i] = solve_cbf_qp(a[i], c_lead[i], c_adj[i], has_adj[i] != 0, lo[i], hi[i], act);
        active[i] = (uint8_t)act;
    }
}
#endif  // MM_VARIANT_TU

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
constexpr size_t STEP_SMEM = (size_t)PLANES_F64 * sizeof(double);

// Function attributes belong to a device (context): set them once per device the process launches on, and report a
// failure through the launch error the caller checks (cudaGetLastError in capi.cu).
static bool step_attrs_ready(size_t smem) {
    static bool ready[MM_MAX_DEVICES] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MM_MAX_DEVICES) return false;
    if (ready[dev]) return true;
    cudaError_t ce = cudaFuncSetAttribute(step_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(step_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(step_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return false;   // the error stays pending for cudaGetLastError
    ready[dev] = true;
    return true;
}

void launch_step_impl(const StepParams &p, bool diag, void *stream) {
    if (!step_attrs_ready(STEP_SMEM)) return;
    int grid = (p.env_count + BLOCK - 1) / BLOCK;
    if (grid <= 0) return;
    if (diag) step_kernel<true, false><<<grid, BLOCK, STEP_SMEM, (cudaStream_t)stream>>>(p);
    else if (p.cfg.couple_counts) step_kernel<false, true><<<grid, BLOCK, STEP_SMEM, (cudaStream_t)stream>>>(p);
    else step_kernel<false, false><<<grid, BLOCK, STEP_SMEM, (cudaStream_t)stream>>>(p);
}

#ifndef MM_VARIANT_TU
static int g_step_variant = 0;
static unsigned long long g_variant_epoch = 0;     // bumped by every change of the variant: cached step graphs are keyed on it
void set_step_variant(int v) { g_step_variant = (v >= 3 && v <= 8) ? v : 0; ++g_variant_epoch; }
unsigned long long step_variant_epoch() { return g_variant_epoch; }

// Picks the build of the step kernel: 4 CTAs / SM when the wave structure of the grid favours it (e.g. 512 CTAs on 148
// SMs: one wave instead of a full and an almost empty one), else the default 3 CTAs / SM build.
int launch_step(const StepParams &p, bool diag, void *stream) {
    const mm_config &c = p.cfg;
    const int grid = (p.env_count + BLOCK - 1) / BLOCK;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // CTA latency (arbitrary units) with c CTAs resident per SM, measured (profiles/README.md, occupancy sweep and
    // time_variants.py): the grid costs its full waves plus one partial wave at the occupancy of the remainder
    auto estimate = [&](int per_sm, const double *lat) {
        const int slots = per_sm * sms, full = grid / slots, rem = grid - full * slots;
        return full * lat[per_sm] + lat[(rem + sms - 1) / sms];
    };
    static const double lat3[4] = {0.0, 9.55, 11.42, 12.27}, lat4[5] = {0.0, 10.5, 12.6, 13.5, 16.2};
    const bool small_grid = grid <= 8 * sms;      // measured: still ahead at 1024 CTAs, behind at 1536 (time_variants.py)
    const bool automatic = g_step_variant == 0 || g_step_variant == 5 || g_step_variant == 8;
    const bool four = g_step_variant == 4 || g_step_variant == 6 || (automatic && !diag && !p.cfg.couple_counts && small_grid &&
                                              estimate(4, lat4) < 0.97 * estimate(3, lat3));
    // the specialised builds: all-CAV envs of the plain LC env (v1, lateral_control "steer") under MASS or HSS
    const bool plain_all_cav = p.all_cav && !c.couple_counts && !c.env_v0 && !c.steer_vel && !c.env_hdv && c.traffic_type == MM_TRAFFIC_CAV;
    // the warp-cooperative build (merge_coop.cu): half a warp per env, for grids too small to fill the machine with
    // one thread per env
    // Measured crossover (profiles/r2_e_ab_coop_sizes.txt): at 8 192 envs the cooperative build is 1.4-1.6 x faster
    // (0.22 / 0.27 ms per step against 0.36 / 0.38 for HSS / MASS), at 16 384 envs the thread-per-env builds are ahead
    // again (0.37 / 0.40 against 0.39 / 0.49); at 2^20 envs it costs 3 x more issue slots per env.
    const bool coop_pays = p.env_count <= 12288;
    if (plain_all_cav && (g_step_variant == 7 || (g_step_variant == 0 && coop_pays))) {
        launch_step_coop(p, diag, stream);
        return MM_BUILD_COOP + c.shield;
    }
    const bool spec_ok = (g_step_variant == 0 || g_step_variant == 6 || g_step_variant == 8) && p.all_cav && !c.couple_counts && !c.env_v0 && !c.steer_vel &&
                         !c.env_hdv && c.traffic_type == MM_TRAFFIC_CAV;
    if (spec_ok && four && c.shield == MM_SHIELD_MASS) { launch_step_spec_mass4(p, diag, stream); return MM_BUILD_SPEC_MASS4; }
    if (spec_ok && four && c.shield == MM_SHIELD_HSS) { launch_step_spec_hss4(p, diag, stream); return MM_BUILD_SPEC_HSS4; }
    if (spec_ok && !four && c.shield == MM_SHIELD_MASS) { launch_step_spec_mass(p, diag, stream); return MM_BUILD_SPEC_MASS; }
    if (spec_ok && !four && c.shield == MM_SHIELD_HSS) { launch_step_spec_hss(p, diag, stream); return MM_BUILD_SPEC_HSS; }
    if (four) { launch_step_occ4(p, diag, stream); return MM_BUILD_GENERIC4; }
    launch_step_impl(p, diag, stream);
    return MM_BUILD_GENERIC3;
}

void launch_reset(const ResetParams &p, void *stream) {
    int grid = (p.env_count + BLOCK - 1) / BLOCK;
    if (grid <= 0) return;
    reset_kernel<<<grid, BLOCK, 0, (cudaStream_t)stream>>>(p);
}

void launch_seeded_reset(const SeededResetParams &p, void *stream) {
    int grid = (p.n_envs + BLOCK - 1) / BLOCK;
    if (grid <= 0) return;
    seeded_reset_kernel<<<grid, BLOCK, 0, (cudaStream_t)stream>>>(p);
}

void launch_pack_state(const DevState &st, int n_envs, const double *f64_em, const int32_t *i32_em,
                       const int32_t *env_em, void *stream) {
    size_t n = (size_t)n_envs * MAXV;
    pack_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(st, n_envs, f64_em, i32_em, env_em);
}

void launch_unpack_state(const DevState &st, int n_envs, double *f64_em, int32_t *i32_em, int32_t *env_em,
                         void *stream) {
    size_t n = (size_t)n_envs * MAXV;
    unpack_state_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(st, n_envs, f64_em, i32_em, env_em);
}

void launch_shield_query(const DevState &st, const mm_config &cfg, int n_envs, const double *nom_steer, const double *nom_acc,
                         double *safe_steer, double *safe_acc, double *min_headway, int32_t *const *out_i, void *stream) {
    static bool ready[MM_MAX_DEVICES] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MM_MAX_DEVICES) return;
    if (!ready[dev]) {
        if (cudaFuncSetAttribute(shield_query_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)STEP_SMEM) != cudaSuccess) return;
        ready[dev] = true;
    }
    ShieldQueryParams p{st, cfg, n_envs, nom_steer, nom_acc, safe_steer, safe_acc, min_headway,
                        out_i[0], out_i[1], out_i[2], out_i[3], out_i[4], out_i[5], out_i[6]};
    const int grid = (n_envs + BLOCK - 1) / BLOCK;
    if (grid <= 0) return;
    shield_query_kernel<<<grid, BLOCK, STEP_SMEM, (cudaStream_t)stream>>>(p);
}

void launch_qp(const double *a, const double *c_lead, const double *c_adj, const uint8_t *has_adj, const double *lo,
               const double *hi, int64_t n, double *u, uint8_t *active, void *stream) {
    if (n <= 0) return;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    qp_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, c_lead, c_adj, has_adj, lo, hi, n, u, active);
}
#endif  // MM_VARIANT_TU

}  // namespace MM_KNS

#ifdef MM_VARIANT_TU
namespace mm {
void MM_VARIANT_LAUNCH(const StepParams &p, bool diag, void *stream) { MM_KNS::launch_step_impl(p, diag, stream); }
}  // namespace mm
#endif

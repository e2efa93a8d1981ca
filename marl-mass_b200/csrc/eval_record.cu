// eval_record.cu — per-step episode records of the evaluation protocol (mm_eval_record), kept on the device.
//
// MAPPO.evaluation (marl/mappo.py:255-361, evaluation.evaluation) reads after every policy step the global reward, the info
// scalars and, per controlled vehicle, crashed / speed / x.  The vehicle fields live in the tiled state (mm_internal.h),
// which only the library addresses, so this kernel takes the records where the state is instead of the host pulling the
// whole state every step.  One thread per env; an env's records stop at its first done, as the reference's loop does.
#include <cuda_runtime.h>
#include "mm_internal.h"

namespace mm {

__global__ void __launch_bounds__(256) eval_record_kernel(const DevState st, const DevOut out, int n_envs,
                                                          const mm_eval_records r, int t) {
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= n_envs || !r.active[e]) return;
    const size_t row = (size_t)e * r.T + t;
    r.rewards[row] = out.reward[e];
    r.avg_speed_sum[e] += (double)out.average_speed[e];
    r.traffic_speed_sum[e] += (double)out.traffic_speed[e];
    const float hw = out.min_headway[e];
    if (hw < r.min_headway[e]) r.min_headway[e] = hw;       // min(min_headway, v) of the reference's loop
    r.steps[e] += 1;
    const int n = r.n_agents[e];
    if (r.vehicle_speed)
        for (int i = 0; i < n; ++i) r.vehicle_speed[row * MAXV + i] = st.f64[f64_index(e, F_V, i)];
    if (r.vehicle_position)
        for (int i = 0; i < n; ++i) r.vehicle_position[row * MAXV + i] = st.f64[f64_index(e, F_X, i)];
    if (out.done[e]) {
        bool crashed = false;
        for (int i = 0; i < n; ++i) crashed = crashed || (st.flags[flags_index(e, i)] & FL_CRASHED) != 0;
        r.crashed[e] = crashed ? 1 : 0;
        r.merge_percent[e] = out.merge_percent[e];
        r.active[e] = 0;
    }
}

void launch_eval_record(const DevState &st, const DevOut &out, int n_envs, const mm_eval_records &r, int t, void *stream) {
    const int grid = (n_envs + 255) / 256;
    if (grid <= 0) return;
    eval_record_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(st, out, n_envs, r, t);
}

// Shield records (mm_eval_shield_record) from the diagnostic record DevOut.sh_i / sh_f ([E][3][MAXV] planes).  One thread
// per env accumulates its episode's sums in one fixed order (sub-step, then slot), so they are exact and independent of
// the launch.  An env's record is 36 consecutive values per plane: read by its own thread, every load of a warp would
// touch 32 sectors 144 / 288 B apart.  Instead each warp stages the sub-step s slice of its 32 envs (12 values per env
// and plane) through shared memory with lanes walking the slice in order, and stores per element only what the sums need.
constexpr int SR_WARPS = 4, SR_PAD = MAXV + 1;   // row stride 13 spreads the lanes' rows over the banks

__global__ void __launch_bounds__(SR_WARPS * 32) eval_shield_record_kernel(const DevOut out, int n_envs,
                                                                         const mm_eval_shield_records r, int t) {
    __shared__ double s_da[SR_WARPS][32 * SR_PAD], s_ds[SR_WARPS][32 * SR_PAD], s_acc[SR_WARPS][32 * SR_PAD];
    __shared__ uint8_t s_fl[SR_WARPS][32 * SR_PAD];
    enum { RAN = 1, ACTIVE = 2, VETO = 4, INTERVENED = 8, MOVED = 16 };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e0 = (blockIdx.x * SR_WARPS + warp) * 32, e = e0 + lane;
    const bool mine = e < n_envs && r.active[e];
    if (!__ballot_sync(0xffffffffu, mine)) return;      // warp-uniform: no env of this warp is still running
    const size_t plane = (size_t)n_envs * 3 * MAXV;
    const int nk = min(32, n_envs - e0) * MAXV;
    int solves = 0, act = 0, vetoes = 0, interv = 0, n_agents = 0;
    double acc_sum = 0.0, acc_max = 0.0, steer_max = 0.0, min_acc = 0.0;
    if (mine) {
        solves = r.shield_solves[e]; act = r.shield_active[e]; vetoes = r.lane_change_vetoes[e];
        interv = r.shield_interventions[e]; acc_sum = r.acc_correction_sum[e]; acc_max = r.acc_correction_max[e];
        steer_max = r.steer_correction_max[e]; min_acc = r.min_agent_acc[e]; n_agents = r.n_agents[e];
    }
    double *da = s_da[warp], *ds = s_ds[warp], *sacc = s_acc[warp];
    uint8_t *fl = s_fl[warp];
    for (int s = 0; s < 3; ++s) {
        for (int k = lane; k < nk; k += 32) {
            const int j = k / MAXV, i = k - j * MAXV;
            const size_t idx = ((size_t)(e0 + j) * 3 + s) * MAXV + i;
            const int32_t ran = out.sh_i[idx], active = out.sh_i[5 * plane + idx], lc_safe = out.sh_i[6 * plane + idx],
                          moved = out.sh_i[7 * plane + idx];
            const double sa = out.sh_f[idx], ss = out.sh_f[plane + idx], na = out.sh_f[2 * plane + idx],
                         ns = out.sh_f[3 * plane + idx];
            const int o = j * SR_PAD + i;
            da[o] = fabs(sa - na);
            ds[o] = fabs(ss - ns);
            sacc[o] = sa;
            fl[o] = (ran ? RAN : 0) | (active ? ACTIVE : 0) | (lc_safe == 0 ? VETO : 0) |
                    (sa != na || ss != ns ? INTERVENED : 0) | (moved ? MOVED : 0);
        }
        __syncwarp();
        if (mine) {
            for (int i = 0; i < MAXV; ++i) {
                const int o = lane * SR_PAD + i;
                const int f = fl[o];
                if (f & RAN) {
                    solves += 1;
                    act += (f & ACTIVE) ? 1 : 0;
                    vetoes += (f & VETO) ? 1 : 0;
                    interv += (f & INTERVENED) ? 1 : 0;
                    const double a = da[o], st = ds[o];
                    acc_sum += a;
                    if (a > acc_max) acc_max = a;
                    if (st > steer_max) steer_max = st;
                }
                if ((f & MOVED) && i < n_agents && sacc[o] < min_acc) min_acc = sacc[o];
            }
        }
        __syncwarp();
    }
    if (mine) {
        r.shield_solves[e] = solves; r.shield_active[e] = act; r.lane_change_vetoes[e] = vetoes;
        r.shield_interventions[e] = interv; r.acc_correction_sum[e] = acc_sum; r.acc_correction_max[e] = acc_max;
        r.steer_correction_max[e] = steer_max; r.min_agent_acc[e] = min_acc;
    }
    if (!r.profile_slot) return;
    // control profiles: the warp copies the 36 values of each plane of every selected env of its 32, one after the other
    const int slot = mine ? r.profile_slot[e] : -1;
    int32_t *const pi[6] = {r.profile_moved, r.profile_ran, r.profile_active, r.profile_is_lc_safe, r.profile_hl_action,
                            r.profile_lane};
    const int qi[6] = {7, 0, 5, 6, 8, 9};
    double *const pf[9] = {r.profile_x, r.profile_y, r.profile_heading, r.profile_speed, r.profile_min_headway,
                           r.profile_safe_acc, r.profile_safe_steer, r.profile_nom_acc, r.profile_nom_steer};
    const int qf[9] = {5, 6, 7, 8, 9, 0, 1, 2, 3};
    for (unsigned sel = __ballot_sync(0xffffffffu, slot >= 0); sel; sel &= sel - 1) {
        const int j = __ffs(sel) - 1;
        const int k = __shfl_sync(0xffffffffu, slot, j);
        const size_t src = (size_t)(e0 + j) * 3 * MAXV, dst = ((size_t)k * 3 * r.T + 3 * (size_t)t) * MAXV;
        for (int q = lane; q < 3 * MAXV; q += 32) {
#pragma unroll
            for (int c = 0; c < 6; ++c)
                if (pi[c]) pi[c][dst + q] = out.sh_i[qi[c] * plane + src + q];
#pragma unroll
            for (int c = 0; c < 9; ++c)
                if (pf[c]) pf[c][dst + q] = out.sh_f[qf[c] * plane + src + q];
        }
    }
}

void launch_eval_shield_record(const DevOut &out, int n_envs, const mm_eval_shield_records &r, int t, void *stream) {
    const int per_cta = SR_WARPS * 32;
    const int grid = (n_envs + per_cta - 1) / per_cta;
    if (grid <= 0) return;
    eval_shield_record_kernel<<<grid, per_cta, 0, (cudaStream_t)stream>>>(out, n_envs, r, t);
}

}  // namespace mm

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

}  // namespace mm

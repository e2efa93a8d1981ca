// capi.cu — host side of the C ABI declared in include/marl_mass_b200.h.
// Owns device memory, launches the kernels of merge_step.cu, and implements the host-buffer step
// (chunked over streams so that PCIe copies overlap compute).  No torch types anywhere.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <thread>
#include <vector>

#include "mm_internal.h"
#include "spawn_core.h"

using namespace mm;

static_assert(mmspawn::TRAFFIC_CAV == MM_TRAFFIC_CAV && mmspawn::TRAFFIC_MIXED == MM_TRAFFIC_MIXED &&
              mmspawn::TRAFFIC_AV == MM_TRAFFIC_AV && mmspawn::TRAFFIC_HDV == MM_TRAFFIC_HDV &&
              mmspawn::KIND_CAV == MM_KIND_CAV && mmspawn::KIND_HDV == MM_KIND_HDV, "spawn_core.h codes");

namespace {

thread_local std::string g_last_error;

int fail(mm_status code, const char *what, cudaError_t ce = cudaSuccess) {
    char buf[512];
    if (ce != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(ce));
    else snprintf(buf, sizeof buf, "%s", what);
    g_last_error = buf;
    return (int)code;
}

#define CUDA_OK(expr)                                                        \
    do {                                                                     \
        cudaError_t _ce = (expr);                                            \
        if (_ce != cudaSuccess) return fail(MM_ERR_CUDA, #expr, _ce);        \
    } while (0)

constexpr int HOST_STREAMS = 4;      // compute streams of the *_host entry points (DESIGN.md §6: four beat two and eight)
constexpr int N_STREAMS = 2 * HOST_STREAMS;   // mm_step_host_packed adds one copy stream per compute stream
constexpr int GRAPH_MAX_ENVS = 131072;   // mm_step replays a CUDA graph up to this batch size (above, launch overhead is noise)
constexpr int MM_SUP_TASKS_PER_ENV = 2;   // predicted collisions per env and step the dmc task list holds (more: evaluated in place)
constexpr int MAX_HOST_CHUNKS = 64;   // chunks of one mm_step_host_ragged / _packed call
constexpr int HOST_F64 = 17, HOST_I32 = 11, HOST_ENV = 5;

}  // namespace

struct mm_env {
    int n_envs = 0, device = 0, record_diag = 0;
    mm_config cfg{};
    DevState st{};
    DevOut out{};
    int8_t *actions = nullptr;
    // baseline supervisors (mm_config.supervisor): the tuples _simulate executes (info["new_action"]), the draws a caller
    // supplied for the next steps (null: Philox), the draws each env consumed in the last step
    int8_t *new_actions = nullptr;
    const double *sup_draws = nullptr;
    int32_t *sup_used = nullptr;
    char *sup_tasks = nullptr;          // dmc pass 2: MM_SUP_TASKS_PER_ENV task records per env (allocated with the first dmc use)
    int *sup_task_count = nullptr;      // one counter per call (calls start on distinct tiles)
    // mm_step_host_ragged, allocated on first use: first packed row of every env, packed-row staging, per-chunk counts
    int64_t *row_offset = nullptr;
    float *rows_stage = nullptr;
    int64_t *chunk_rows_dev = nullptr, *chunk_rows_host = nullptr;
    cudaEvent_t chunk_done[MAX_HOST_CHUNKS]{};
    // mm_step_host_packed, allocated on first use: packed vehicle rows / neighbour words, per-env offsets inside a chunk,
    // count bytes, running totals chained chunk to chunk (device + pinned host mirror), one event per chunk's scan
    float *veh_packed = nullptr;
    uint16_t *nbr_packed = nullptr;
    int32_t *voff = nullptr, *aoff = nullptr;
    uint8_t *n_veh_u8 = nullptr, *n_agents_u8 = nullptr;
    int64_t *chunk_base_dev = nullptr, *chunk_base_host = nullptr, *chunk_base_host_dev = nullptr;
    cudaEvent_t scan_done[MAX_HOST_CHUNKS]{};
    // mm_reset_seeded, allocated on first use: the test seeds and num_CAV values of the envs
    int64_t *seeds = nullptr;
    int32_t *seed_num_cav = nullptr;
    size_t stats_rows = 0;
    uint64_t seed = 0;
    int64_t launches = 0;
    // true while some env may hold an HDV (spawned under a traffic_type other than cav, or put there by mm_set_state):
    // the step kernel's all-CAV builds are used only when this is false
    bool hdv_possible = true;
    int last_build = 0;       // MM_BUILD_* of the step kernel the last step launched
    // the stream the caller last enqueued work of this handle on, and an event to order the internal streams of the
    // *_host entry points after that work
    cudaStream_t last_stream = nullptr;
    cudaEvent_t caller_done = nullptr;
    // Small batches are launch-bound (a policy step of 4 096 envs is four kernels of 3-100 us): mm_step replays the
    // sequence as a CUDA graph.  One instantiated graph per (action buffer, auto_reset); `epoch` advances with everything
    // a captured launch bakes in (config, seed, HDV knowledge, supervisor draws, the process-wide step variant).
    struct StepGraph {
        const int8_t *actions; int auto_reset; uint64_t epoch; unsigned long long variant_epoch;
        cudaGraphExec_t exec; int build; int launches;
    };
    std::vector<StepGraph> graphs;
    uint64_t epoch = 0;
    cudaStream_t streams[N_STREAMS]{};
    std::vector<void *> allocs;
};

namespace {

// The allocation helpers do nothing when *ptr is already set, so lazily allocated buffers are requested piece by piece on
// every call: a failure half-way leaves a handle that retries the missing pieces instead of using null pointers.
template <typename T>
int dev_alloc(mm_env *env, T **ptr, size_t count, bool zero = true) {
    if (*ptr) return 0;
    void *p = nullptr;
    CUDA_OK(cudaMalloc(&p, count * sizeof(T)));
    env->allocs.push_back(p);
    if (zero) CUDA_OK(cudaMemset(p, 0, count * sizeof(T)));
    *ptr = static_cast<T *>(p);
    return 0;
}

// Pinned host memory, freed by mm_destroy.  With `dev` the block is mapped and *dev receives its device address.
template <typename T>
int host_alloc(T **ptr, size_t count, bool zero, T **dev = nullptr) {
    if (!*ptr) {
        void *p = nullptr;
        CUDA_OK(cudaHostAlloc(&p, count * sizeof(T), dev ? cudaHostAllocMapped : cudaHostAllocDefault));
        if (zero) memset(p, 0, count * sizeof(T));
        *ptr = static_cast<T *>(p);
    }
    if (dev && !*dev) CUDA_OK(cudaHostGetDevicePointer((void **)dev, *ptr, 0));
    return 0;
}

int event_alloc(cudaEvent_t *events, int n) {
    for (int i = 0; i < n; ++i)
        if (!events[i]) CUDA_OK(cudaEventCreateWithFlags(&events[i], cudaEventDisableTiming));
    return 0;
}

int validate(const mm_config *c) {
    if (!c) return fail(MM_ERR_ARG, "config is null");
    if (c->struct_size != (int32_t)sizeof(mm_config))
        return fail(MM_ERR_ARG, "mm_config.struct_size does not match this library's sizeof(mm_config): the binding was "
                                "built against another revision of marl_mass_b200.h (see mm_abi_version)");
    if (c->shield < MM_SHIELD_NONE || c->shield > MM_SHIELD_MASS) return fail(MM_ERR_ARG, "Undefined safety_type");
    if (c->reward_kind < MM_REW_DEFAULT || c->reward_kind > MM_REW_MREW) return fail(MM_ERR_ARG, "unknown agent_reward");
    if (c->traffic_density < 1 || c->traffic_density > 3) return fail(MM_ERR_ARG, "traffic_density must be 1, 2 or 3");
    if (c->traffic_type < MM_TRAFFIC_CAV || c->traffic_type > MM_TRAFFIC_HDV) return fail(MM_ERR_ARG, "unknown traffic_type");
    if ((c->traffic_type == MM_TRAFFIC_HDV) != (c->env_hdv != 0))
        return fail(MM_ERR_ARG, "traffic_type hdv and the env id merge-multi-agent-hdv-v1 go together");
    if (c->substeps < 1 || c->substeps > 3) return fail(MM_ERR_ARG, "substeps must be in 1..3");
    if (c->duration_steps < 1 || c->duration_steps > 255) return fail(MM_ERR_ARG, "duration_steps must be in 1..255");
    if (!(c->dt > 0)) return fail(MM_ERR_ARG, "dt must be positive");
    if (c->supervisor < MM_SUPERVISOR_NONE || c->supervisor > MM_SUPERVISOR_DMC) return fail(MM_ERR_ARG, "unknown supervisor");
    if (c->supervisor != MM_SUPERVISOR_NONE && c->shield != MM_SHIELD_NONE)
        return fail(MM_ERR_ARG, "safety_guarantee is either a CBF shield or a baseline supervisor, not both");
    return 0;
}

StepParams step_params(mm_env *env, const int8_t *actions, int off, int count) {
    StepParams p{};
    p.st = env->st;
    p.out = env->out;
    p.actions = actions;
    p.cfg = env->cfg;
    p.n_envs = env->n_envs;
    p.env_offset = off;
    p.env_count = count;
    p.obs_mask = nullptr;
    p.all_cav = env->hdv_possible ? 0 : 1;
    return p;
}

int reset_stats(mm_env *env) {
    std::vector<double> h(env->stats_rows * N_STATS, 0.0);
    for (size_t r = 0; r < env->stats_rows; ++r) h[r * N_STATS + ST_MINHW] = std::numeric_limits<double>::infinity();
    CUDA_OK(cudaMemcpy(env->out.stats, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice));
    return 0;
}

// Envs per chunk of the host paths.  Large batches: HALF A WAVE of the step kernel's default build - 3 CTAs of 128 envs
// per SM make 56 832 envs a wave on a 148-SM B200 - rounded to the 768-env granule every tile size divides; two chunks
// on different streams fill the machine, and the copy of the last chunk that trails the compute is half as long.
// Measured on the packed path at 2^20 envs: mid-round kernels (profiles/r2_k_e2e_chunks.txt) 56 832 -> 11.0 ms per step,
// 65 536 (1.15 waves) 11.4, 75 264 (one wave of the 4-CTA build) 11.8, 113 664 -> 12.8, 150 528 -> 14.0; final kernels
// (profiles/r2_final_e2e_chunks.txt) 56 832 -> 8.87, 37 888 -> 8.73, 28 416 -> 8.68, 18 944 -> 9.44 against 7.5 ms for the
// un-chunked device-resident step.  A mid-size batch is still cut in 4 chunks (>= 16 Ki envs), one per stream, so that
// its device-to-host copies overlap the compute of the following chunks instead of trailing a single launch.
int host_chunk_target(int n_envs) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int half_wave = sms * 3 * TILE / 2 / 768 * 768;
    int t = (n_envs + 3) / 4;     // one chunk per stream
    if (t < 16384) t = 16384;
    if (t > half_wave) t = half_wave;
    return t;
}

// The chunks of one host-path call: `used` <= `max_chunks` chunks of `chunk` envs each, the last one shorter.  `chunk` is
// a multiple of 768 envs, which every supported tile size (32..384) divides; this also keeps the per-warp statistics
// rows of different chunks disjoint.
struct ChunkPlan {
    int n_envs, chunk, used;
    int off(int c) const { return c * chunk; }
    int count(int c) const { return n_envs - c * chunk < chunk ? n_envs - c * chunk : chunk; }
};

ChunkPlan plan_chunks(int n_envs, int max_chunks) {
    const int target = host_chunk_target(n_envs);
    int n_chunks = (n_envs + target - 1) / target;
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > max_chunks) n_chunks = max_chunks;
    const int chunk = ((n_envs + n_chunks - 1) / n_chunks + 767) / 768 * 768;
    return {n_envs, chunk, (n_envs + chunk - 1) / chunk};
}

// The *_host entry points run on the handle's own non-blocking streams.  Work the caller enqueued earlier (mm_reset,
// mm_step, a masked reset on its own stream) must be complete before they touch the state: order every internal stream
// after the last caller stream this handle saw.
int order_after_caller(mm_env *env, int n_str) {
    CUDA_OK(cudaEventRecord(env->caller_done, env->last_stream));
    for (int c = 0; c < n_str; ++c) CUDA_OK(cudaStreamWaitEvent(env->streams[c], env->caller_done, 0));
    return 0;
}

// enqueue one policy step (+ optional re-spawn of finished envs) for envs [off, off+count) on `stream`
void enqueue_step(mm_env *env, const int8_t *actions_dev, int auto_reset, int off, int count, cudaStream_t stream) {
    if (auto_reset && env->cfg.traffic_type != MM_TRAFFIC_CAV && !env->hdv_possible) { env->hdv_possible = true; ++env->epoch; }
    if (env->cfg.supervisor != MM_SUPERVISOR_NONE) {
        // abstract.py:459-464: new_action = safety_supervisor / safety_layer_dmc (env, action); _simulate(new_action)
        int8_t *na = env->new_actions + (size_t)off * MAXV;
        cudaMemcpyAsync(na, actions_dev + (size_t)off * MAXV, (size_t)count * MAXV, cudaMemcpyDeviceToDevice, stream);
        const bool dmc = env->cfg.supervisor != MM_SUPERVISOR_PRIORITY;
        launch_supervisor(env->st, off, count, dmc ? 1 : 0, env->new_actions, env->sup_draws, MM_SUPERVISOR_DRAWS,
                          env->cfg.headway_time, env->seed, env->sup_used,
                          env->sup_tasks + (size_t)off * MM_SUP_TASKS_PER_ENV * supervisor_task_bytes(),
                          env->sup_task_count + off / TILE, count * MM_SUP_TASKS_PER_ENV, stream);
        env->launches += dmc ? 2 : 1;
        actions_dev = env->new_actions;
    }
    StepParams p = step_params(env, actions_dev, off, count);
    env->last_build = launch_step(p, env->record_diag != 0, stream);      // physics of the policy step (state -> state)
    launch_outputs(p, true, stream);                    // observations, rewards, flags, info, statistics
    env->launches += 2;
    if (auto_reset) {
        ResetParams r{};
        r.st = env->st; r.out = env->out; r.mask = nullptr; r.cfg = env->cfg; r.seed = env->seed;
        r.n_envs = env->n_envs; r.env_offset = off; r.env_count = count; r.num_cav = 0; r.use_done = 1;
        launch_reset(r, stream);
        StepParams o = step_params(env, nullptr, off, count);
        o.obs_mask = env->out.done;
        launch_observe(o, stream);
        env->launches += 2;
    }
}

// host-buffer step of envs [off, off+count) on `stream`: their actions from the caller's host buffer, then the step
int enqueue_host_step(mm_env *env, const int8_t *actions, int auto_reset, int off, int count, cudaStream_t stream) {
    CUDA_OK(cudaMemcpyAsync(env->actions + (size_t)off * MAXV, actions + (size_t)off * MAXV, (size_t)count * MAXV,
                            cudaMemcpyHostToDevice, stream));
    enqueue_step(env, env->actions, auto_reset, off, count, stream);
    return 0;
}

// the per-env outputs of envs [off, off+count) to the caller's host buffers; a null buffer is not copied
int copy_env_outputs(mm_env *env, int off, int count, cudaStream_t stream, float *reward, uint8_t *done,
                     float *regional_rewards, int32_t *n_agents_i32) {
    if (reward)
        CUDA_OK(cudaMemcpyAsync(reward + off, env->out.reward + off, (size_t)count * sizeof(float), cudaMemcpyDeviceToHost, stream));
    if (done)
        CUDA_OK(cudaMemcpyAsync(done + off, env->out.done + off, (size_t)count, cudaMemcpyDeviceToHost, stream));
    if (regional_rewards)
        CUDA_OK(cudaMemcpyAsync(regional_rewards + (size_t)off * MAXV, env->out.regional_rewards + (size_t)off * MAXV,
                                (size_t)count * MAXV * sizeof(float), cudaMemcpyDeviceToHost, stream));
    if (n_agents_i32)
        CUDA_OK(cudaMemcpyAsync(n_agents_i32 + off, env->out.n_agents + off, (size_t)count * sizeof(int32_t),
                                cudaMemcpyDeviceToHost, stream));
    return 0;
}

int ensure_supervisor_stack(mm_env *env) {
    // the supervisors keep 2 x 12 vehicles x 18-point trajectories per thread: a 17 KB frame
    CUDA_OK(cudaSetDevice(env->device));
    size_t stack = 0;
    CUDA_OK(cudaDeviceGetLimit(&stack, cudaLimitStackSize));
    if (stack < 32768) CUDA_OK(cudaDeviceSetLimit(cudaLimitStackSize, 32768));
    const size_t E_pad = ((size_t)env->n_envs + TILE - 1) / TILE * TILE;
    int rc = dev_alloc(env, &env->sup_tasks, E_pad * MM_SUP_TASKS_PER_ENV * supervisor_task_bytes(), false);
    rc |= dev_alloc(env, &env->sup_task_count, E_pad / TILE + 1, false);
    return rc;
}

}  // namespace

extern "C" {

const char *mm_last_error(void) { return g_last_error.c_str(); }
const char *mm_version(void) { return "marl-mass_b200 0.2 (sm_100a, f64 core)"; }
int mm_abi_version(void) { return MM_ABI_VERSION; }

int mm_create(const mm_config *cfg, int n_envs, int device, int record_diag, mm_env **out) {
    if (!out) return fail(MM_ERR_ARG, "out is null");
    *out = nullptr;
    if (int rc = validate(cfg)) return rc;
    if (n_envs < 1) return fail(MM_ERR_ARG, "n_envs must be >= 1");
    CUDA_OK(cudaSetDevice(device));
    mm_env *env = new mm_env();
    env->n_envs = n_envs; env->device = device; env->record_diag = record_diag; env->cfg = *cfg;
    const size_t E = (size_t)n_envs;
    const size_t E_pad = (E + TILE - 1) / TILE * TILE;   // state is tiled: [n_tiles][field][slot][TILE]
    int rc = 0;
    rc |= dev_alloc(env, &env->st.f64, (size_t)F_COUNT * MAXV * E_pad);
    rc |= dev_alloc(env, &env->st.flags, (size_t)MAXV * E_pad);
    rc |= dev_alloc(env, &env->st.einfo, E_pad);
    rc |= dev_alloc(env, &env->st.episode, E_pad);
    rc |= dev_alloc(env, &env->out.obs, E * MAXV * NS);
    rc |= dev_alloc(env, &env->out.reward, E);
    rc |= dev_alloc(env, &env->out.agents_rewards, E * MAXV);
    rc |= dev_alloc(env, &env->out.regional_rewards, E * MAXV);
    rc |= dev_alloc(env, &env->out.average_speed, E);
    rc |= dev_alloc(env, &env->out.traffic_speed, E);
    rc |= dev_alloc(env, &env->out.min_headway, E);
    rc |= dev_alloc(env, &env->out.merge_percent, E);
    rc |= dev_alloc(env, &env->out.done, E);
    rc |= dev_alloc(env, &env->out.agents_dones, E * MAXV);
    rc |= dev_alloc(env, &env->out.n_agents, E);
    rc |= dev_alloc(env, &env->out.action_mask, E * MAXV);
    rc |= dev_alloc(env, &env->actions, E * MAXV);
    rc |= dev_alloc(env, &env->new_actions, E * MAXV);
    rc |= dev_alloc(env, &env->sup_used, E);
    env->stats_rows = (E + 31) / 32;
    rc |= dev_alloc(env, &env->out.stats, env->stats_rows * N_STATS);
    if (record_diag) {
        rc |= dev_alloc(env, &env->out.sh_i, (size_t)10 * E * 3 * MAXV);
        rc |= dev_alloc(env, &env->out.sh_f, (size_t)10 * E * 3 * MAXV);
    }
    if (rc) { mm_destroy(env); return rc; }
    if ((rc = reset_stats(env))) { mm_destroy(env); return rc; }
    for (int i = 0; i < N_STREAMS; ++i) {
        cudaError_t ce = cudaStreamCreateWithFlags(&env->streams[i], cudaStreamNonBlocking);
        if (ce != cudaSuccess) { mm_destroy(env); return fail(MM_ERR_CUDA, "cudaStreamCreate", ce); }
    }
    {
        cudaError_t ce = cudaEventCreateWithFlags(&env->caller_done, cudaEventDisableTiming);
        if (ce != cudaSuccess) { mm_destroy(env); return fail(MM_ERR_CUDA, "cudaEventCreate", ce); }
    }
    if (cfg->supervisor != MM_SUPERVISOR_NONE)
        if (int rc2 = ensure_supervisor_stack(env)) { mm_destroy(env); return rc2; }
    *out = env;
    return 0;
}

int mm_destroy(mm_env *env) {
    if (!env) return 0;
    cudaSetDevice(env->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < N_STREAMS; ++i)
        if (env->streams[i]) cudaStreamDestroy(env->streams[i]);
    for (int i = 0; i < MAX_HOST_CHUNKS; ++i)
        if (env->chunk_done[i]) cudaEventDestroy(env->chunk_done[i]);
    for (auto &g : env->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    if (env->caller_done) cudaEventDestroy(env->caller_done);
    for (int i = 0; i < MAX_HOST_CHUNKS; ++i)
        if (env->scan_done[i]) cudaEventDestroy(env->scan_done[i]);
    if (env->chunk_base_host) cudaFreeHost(env->chunk_base_host);
    if (env->chunk_rows_host) cudaFreeHost(env->chunk_rows_host);
    for (void *p : env->allocs) cudaFree(p);
    delete env;
    return 0;
}

int mm_set_config(mm_env *env, const mm_config *cfg) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (int rc = validate(cfg)) return rc;
    env->cfg = *cfg;
    ++env->epoch;
    if (cfg->supervisor != MM_SUPERVISOR_NONE) return ensure_supervisor_stack(env);
    return 0;
}

int mm_set_supervisor_draws(mm_env *env, const double *draws_dev) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    env->sup_draws = draws_dev;
    ++env->epoch;
    return 0;
}

int mm_supervisor_draws_used(mm_env *env, int32_t *n_used_host) {
    if (!env || !n_used_host) return fail(MM_ERR_ARG, "null argument");
    CUDA_OK(cudaSetDevice(env->device));
    CUDA_OK(cudaDeviceSynchronize());
    CUDA_OK(cudaMemcpy(n_used_host, env->sup_used, (size_t)env->n_envs * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return 0;
}

int mm_num_envs(const mm_env *env) { return env ? env->n_envs : 0; }
int mm_step_build(const mm_env *env) { return env ? env->last_build : 0; }
int64_t mm_kernel_launches(const mm_env *env) { return env ? env->launches : 0; }

int mm_reset(mm_env *env, uint64_t seed, const uint8_t *mask_dev, int num_cav, void *stream) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (num_cav < 0 || num_cav > 11) return fail(MM_ERR_ARG, "num_cav must be in 0..11");
    CUDA_OK(cudaSetDevice(env->device));
    if (seed != env->seed) ++env->epoch;      // the auto-reset of a captured step carries the seed
    env->seed = seed;
    env->last_stream = (cudaStream_t)stream;
    const bool hdv_before = env->hdv_possible;
    if (env->cfg.traffic_type != MM_TRAFFIC_CAV) env->hdv_possible = true;
    else if (!mask_dev) env->hdv_possible = false;      // every env re-spawned all-CAV
    if (hdv_before != env->hdv_possible) ++env->epoch;
    ResetParams r{};
    r.st = env->st; r.out = env->out; r.mask = mask_dev; r.cfg = env->cfg; r.seed = seed;
    r.n_envs = env->n_envs; r.env_offset = 0; r.env_count = env->n_envs; r.num_cav = num_cav; r.use_done = 0;
    launch_reset(r, stream);
    StepParams o = step_params(env, nullptr, 0, env->n_envs);
    o.obs_mask = mask_dev;
    launch_observe(o, stream);
    env->launches += 2;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_check_seeds(const mm_config *cfg, int n_envs, const int64_t *seeds, const int32_t *num_cav) {
    if (int rc = validate(cfg)) return rc;
    if (n_envs < 1) return fail(MM_ERR_ARG, "n_envs must be >= 1");
    if (!seeds) return fail(MM_ERR_ARG, "seeds is null");
    mmspawn::MT19937 mt;
    for (int e = 0; e < n_envs; ++e) {
        char buf[200];
        if (seeds[e] < 0 || seeds[e] > (int64_t)0xffffffffLL) {
            snprintf(buf, sizeof buf, "seed %lld of env %d: a test seed must lie in [0, 2^32)", (long long)seeds[e], e);
            return fail(MM_ERR_ARG, buf);
        }
        const int c = num_cav ? num_cav[e] : 0;
        if (c < 0 || c > 11) {
            snprintf(buf, sizeof buf, "num_CAV %d of env %d must be in 0..11", c, e);
            return fail(MM_ERR_ARG, buf);
        }
        if (!mmspawn::spawn_fits((uint32_t)seeds[e], cfg->traffic_density, c, mt)) {
            snprintf(buf, sizeof buf, "num_CAV %d of env %d (seed %lld): the reference's spawn raises or builds more than 11 "
                                      "vehicles at traffic_density %d", c, e, (long long)seeds[e], cfg->traffic_density);
            return fail(MM_ERR_ARG, buf);
        }
    }
    return 0;
}

int mm_reset_seeded(mm_env *env, const int64_t *seeds, const int32_t *num_cav, void *stream) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (int rc = mm_check_seeds(&env->cfg, env->n_envs, seeds, num_cav)) return rc;
    CUDA_OK(cudaSetDevice(env->device));
    const size_t E = (size_t)env->n_envs;
    int err = dev_alloc(env, &env->seeds, E, false);
    if (num_cav) err |= dev_alloc(env, &env->seed_num_cav, E, false);
    if (err) return err;
    // what mm_set_state concludes from the scenes: every traffic_type but cav puts at least one HDV into every env
    const bool any_hdv = env->cfg.traffic_type != MM_TRAFFIC_CAV;
    if (env->hdv_possible != any_hdv) ++env->epoch;
    env->hdv_possible = any_hdv;
    env->last_stream = (cudaStream_t)stream;
    CUDA_OK(cudaMemcpyAsync(env->seeds, seeds, E * sizeof(int64_t), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    if (num_cav)
        CUDA_OK(cudaMemcpyAsync(env->seed_num_cav, num_cav, E * sizeof(int32_t), cudaMemcpyHostToDevice, (cudaStream_t)stream));
    SeededResetParams r{env->st, env->cfg, env->seeds, num_cav ? env->seed_num_cav : nullptr, env->n_envs};
    launch_seeded_reset(r, stream);
    StepParams o = step_params(env, nullptr, 0, env->n_envs);
    launch_observe(o, stream);
    env->launches += 2;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_eval_record(mm_env *env, const mm_eval_records *rec, int t, void *stream) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (!rec) return fail(MM_ERR_ARG, "records are null");
    if (!rec->n_agents || !rec->active || !rec->rewards || !rec->steps || !rec->avg_speed_sum || !rec->traffic_speed_sum ||
        !rec->min_headway || !rec->merge_percent || !rec->crashed)
        return fail(MM_ERR_ARG, "mm_eval_record: every record array but vehicle_speed / vehicle_position is required");
    if (rec->T < 1) return fail(MM_ERR_ARG, "mm_eval_record: T must be >= 1");
    if (t < 0 || t >= rec->T) return fail(MM_ERR_ARG, "mm_eval_record: t must be in [0, T)");
    CUDA_OK(cudaSetDevice(env->device));
    env->last_stream = (cudaStream_t)stream;
    launch_eval_record(env->st, env->out, env->n_envs, *rec, t, stream);
    env->launches += 1;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_eval_shield_record(mm_env *env, const mm_eval_shield_records *rec, int t, void *stream) {
    // the records first, so that a null handle can stand in for one in a test without a device
    if (!rec) return fail(MM_ERR_ARG, "records are null");
    if (!rec->n_agents || !rec->active || !rec->shield_solves || !rec->shield_active || !rec->lane_change_vetoes ||
        !rec->shield_interventions || !rec->acc_correction_sum || !rec->acc_correction_max || !rec->steer_correction_max ||
        !rec->min_agent_acc)
        return fail(MM_ERR_ARG, "mm_eval_shield_record: every record array but profile_slot / profile_* is required");
    if (rec->T < 1) return fail(MM_ERR_ARG, "mm_eval_shield_record: T must be >= 1");
    if (t < 0 || t >= rec->T) return fail(MM_ERR_ARG, "mm_eval_shield_record: t must be in [0, T)");
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (!env->record_diag) return fail(MM_ERR_STATE, "handle was created without record_diag");
    CUDA_OK(cudaSetDevice(env->device));
    env->last_stream = (cudaStream_t)stream;
    launch_eval_shield_record(env->out, env->n_envs, *rec, t, stream);
    env->launches += 1;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_step(mm_env *env, const int8_t *actions_dev, int auto_reset, void *stream) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    CUDA_OK(cudaSetDevice(env->device));
    env->last_stream = (cudaStream_t)stream;
    const int8_t *actions = actions_dev ? actions_dev : env->actions;
    if (env->n_envs > GRAPH_MAX_ENVS) {
        enqueue_step(env, actions, auto_reset, 0, env->n_envs, (cudaStream_t)stream);
        CUDA_OK(cudaGetLastError());
        return 0;
    }
    // graph replay: first sight of a key runs eagerly (one-time function-attribute setup stays out of a capture), the
    // second captures the sequence on an internal stream, later ones replay it on the caller's stream
    const unsigned long long vep = step_variant_epoch();
    for (auto &g : env->graphs) {
        if (g.actions != actions || g.auto_reset != auto_reset) continue;
        if (g.epoch != env->epoch || g.variant_epoch != vep) {      // stale: drop and start over
            if (g.exec) cudaGraphExecDestroy(g.exec);
            g = env->graphs.back();
            env->graphs.pop_back();
            break;
        }
        if (!g.exec) {
            cudaStream_t cs = env->streams[0];
            cudaGraph_t graph = nullptr;
            CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            const int64_t l0 = env->launches;
            enqueue_step(env, actions, auto_reset, 0, env->n_envs, cs);
            g.launches = (int)(env->launches - l0);
            env->launches = l0;
            g.build = env->last_build;
            cudaError_t ce = cudaStreamEndCapture(cs, &graph);
            if (ce != cudaSuccess || !graph) return fail(MM_ERR_CUDA, "cudaStreamEndCapture", ce);
            ce = cudaGraphInstantiate(&g.exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ce != cudaSuccess) { g.exec = nullptr; return fail(MM_ERR_CUDA, "cudaGraphInstantiate", ce); }
        }
        CUDA_OK(cudaGraphLaunch(g.exec, (cudaStream_t)stream));
        env->launches += g.launches;
        env->last_build = g.build;
        return 0;
    }
    if (env->graphs.size() >= 16) {      // bounded cache: forget the oldest key
        if (env->graphs.front().exec) cudaGraphExecDestroy(env->graphs.front().exec);
        env->graphs.erase(env->graphs.begin());
    }
    env->graphs.push_back({actions, auto_reset, env->epoch, vep, nullptr, 0, 0});
    enqueue_step(env, actions, auto_reset, 0, env->n_envs, (cudaStream_t)stream);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_step_host(mm_env *env, const int8_t *actions, int auto_reset, float *obs, float *reward, uint8_t *done,
                 float *regional_rewards, int32_t *n_agents) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (!actions) return fail(MM_ERR_ARG, "actions is null");
    CUDA_OK(cudaSetDevice(env->device));
    // Chunks issued round-robin on the compute streams: chunk k's device-to-host copies run while chunks k+1.. compute.
    const ChunkPlan plan = plan_chunks(env->n_envs, std::numeric_limits<int>::max());
    if (int rc = order_after_caller(env, HOST_STREAMS)) return rc;
    for (int c = 0; c < plan.used; ++c) {
        const int off = plan.off(c), count = plan.count(c);
        cudaStream_t s = env->streams[c % HOST_STREAMS];
        if (int rc = enqueue_host_step(env, actions, auto_reset, off, count, s)) return rc;
        if (obs)
            CUDA_OK(cudaMemcpyAsync(obs + (size_t)off * MAXV * NS, env->out.obs + (size_t)off * MAXV * NS,
                                    (size_t)count * MAXV * NS * sizeof(float), cudaMemcpyDeviceToHost, s));
        if (int rc = copy_env_outputs(env, off, count, s, reward, done, regional_rewards, n_agents)) return rc;
    }
    for (int c = 0; c < HOST_STREAMS; ++c) CUDA_OK(cudaStreamSynchronize(env->streams[c]));
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_step_host_ragged(mm_env *env, const int8_t *actions, int auto_reset, float *obs_rows, int64_t *row_offset,
                        float *reward, uint8_t *done, float *regional_rewards, int32_t *n_agents) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (!actions || !obs_rows || !row_offset) return fail(MM_ERR_ARG, "actions, obs_rows and row_offset are required");
    CUDA_OK(cudaSetDevice(env->device));
    const int E = env->n_envs;
    // staging for the packed rows, offsets, per-chunk counts, events: allocated on first use
    int err = dev_alloc(env, &env->row_offset, (size_t)E + 1, false);
    err |= dev_alloc(env, &env->rows_stage, (size_t)E * MAXV * NS, false);
    err |= dev_alloc(env, &env->chunk_rows_dev, MAX_HOST_CHUNKS, false);
    err |= host_alloc(&env->chunk_rows_host, MAX_HOST_CHUNKS, false);
    err |= event_alloc(env->chunk_done, MAX_HOST_CHUNKS);
    if (err) return err;
    const ChunkPlan plan = plan_chunks(E, MAX_HOST_CHUNKS);
    // Software pipeline over the chunks, HOST_STREAMS deep: a chunk's compute + packing is enqueued on its stream; when
    // its row count has arrived (one event wait on the host) its packed rows follow on the same stream - exactly that many
    // bytes - and only then the stream's next chunk.  The copies of chunk c overlap the compute of chunks c+1..c+3.
    auto enqueue_compute = [&](int c) -> int {
        const int off = plan.off(c), count = plan.count(c);
        cudaStream_t s = env->streams[c % HOST_STREAMS];
        if (int rc = enqueue_host_step(env, actions, auto_reset, off, count, s)) return rc;
        // chunk c packs its rows from row off * MAXV on: offsets are absolute and increasing, dense inside a chunk
        launch_ragged_pack(env->out.obs + (size_t)off * MAXV * NS, env->out.n_agents + off, count, (int64_t)off * MAXV,
                           env->row_offset + off, env->chunk_rows_dev + c, env->rows_stage, s);
        env->launches += 2;
        CUDA_OK(cudaMemcpyAsync(env->chunk_rows_host + c, env->chunk_rows_dev + c, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaEventRecord(env->chunk_done[c], s));
        return 0;
    };
    auto enqueue_copies = [&](int c) -> int {
        const int off = plan.off(c), count = plan.count(c);
        cudaStream_t s = env->streams[c % HOST_STREAMS];
        CUDA_OK(cudaEventSynchronize(env->chunk_done[c]));
        const int64_t rows = env->chunk_rows_host[c];
        const size_t first = (size_t)off * MAXV * NS;
        if (rows > 0)
            CUDA_OK(cudaMemcpyAsync(obs_rows + first, env->rows_stage + first, (size_t)rows * NS * sizeof(float),
                                    cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaMemcpyAsync(row_offset + off, env->row_offset + off, (size_t)count * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        return copy_env_outputs(env, off, count, s, reward, done, regional_rewards, n_agents);
    };
    if (int rc = order_after_caller(env, HOST_STREAMS)) return rc;
    for (int c = 0; c < plan.used && c < HOST_STREAMS; ++c)
        if (int rc = enqueue_compute(c)) return rc;
    for (int c = 0; c < plan.used; ++c) {
        if (int rc = enqueue_copies(c)) return rc;
        if (c + HOST_STREAMS < plan.used)
            if (int rc = enqueue_compute(c + HOST_STREAMS)) return rc;
    }
    for (int c = 0; c < HOST_STREAMS; ++c) CUDA_OK(cudaStreamSynchronize(env->streams[c]));
    row_offset[E] = (int64_t)E * MAXV;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_step_host_packed(mm_env *env, const int8_t *actions, int auto_reset, const mm_packed_host *out) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (!actions || !out || !out->veh || !out->nbr || !out->n_veh || !out->n_agents)
        return fail(MM_ERR_ARG, "actions, out->veh, out->nbr, out->n_veh and out->n_agents are required");
    CUDA_OK(cudaSetDevice(env->device));
    const int E = env->n_envs;
    // allocated on first use, zero-filled
    int err = dev_alloc(env, &env->out.veh, (size_t)E * MAXV * MM_VEH_F32);
    err |= dev_alloc(env, &env->out.nbr, (size_t)E * MAXV);
    err |= dev_alloc(env, &env->veh_packed, (size_t)E * MAXV * MM_VEH_F32);
    err |= dev_alloc(env, &env->nbr_packed, (size_t)E * MAXV);
    err |= dev_alloc(env, &env->voff, (size_t)E);
    err |= dev_alloc(env, &env->aoff, (size_t)E);
    err |= dev_alloc(env, &env->n_veh_u8, (size_t)E);
    err |= dev_alloc(env, &env->n_agents_u8, (size_t)E);
    err |= dev_alloc(env, &env->chunk_base_dev, (size_t)(MAX_HOST_CHUNKS + 1) * 2);
    // mapped: the scan kernel writes a chunk's totals here itself.  (A small device-to-host memcpy per chunk on the
    // compute streams sits in the copy engine's queue until its chunk has run - and every data copy issued later queues
    // behind it: measured, the packed rows then left only after ALL compute had finished.)  Zero-filled: the chain of
    // totals starts from chunk_base_host[0..1] = 0.
    err |= host_alloc(&env->chunk_base_host, (size_t)(MAX_HOST_CHUNKS + 1) * 2, true, &env->chunk_base_host_dev);
    err |= event_alloc(env->chunk_done, MAX_HOST_CHUNKS);
    err |= event_alloc(env->scan_done, MAX_HOST_CHUNKS);
    if (err) return err;
    const ChunkPlan plan = plan_chunks(E, MAX_HOST_CHUNKS);
    // Chunks round-robin on the compute streams; ALL of a step's compute is enqueued up front (a chunk touches only its
    // own envs and its own range of the packed buffers), so the GPU never waits for the host.  The packed rows of the
    // batch are dense from the first env to the last: a chunk's scan starts from the totals of the chunk before it (a
    // device-side chain base[c] -> base[c+1], one event wait between neighbouring chunks' scans).  The host learns a
    // chunk's totals with the chunk's event and then issues exactly-sized copies on a copy stream, in chunk order, while
    // later chunks compute.
    auto enqueue_compute = [&](int c) -> int {
        const int off = plan.off(c), count = plan.count(c);
        cudaStream_t s = env->streams[c % HOST_STREAMS];
        if (int rc = enqueue_host_step(env, actions, auto_reset, off, count, s)) return rc;
        if (c > 0) CUDA_OK(cudaStreamWaitEvent(s, env->scan_done[c - 1], 0));
        launch_packed_pack(env->st.einfo + off, env->out.n_agents + off, env->out.veh + (size_t)off * MAXV * MM_VEH_F32,
                           env->out.nbr + (size_t)off * MAXV, count, env->chunk_base_dev + 2 * c, env->chunk_base_dev + 2 * (c + 1),
                           env->chunk_base_host_dev + 2 * (c + 1), env->voff + off, env->aoff + off, env->veh_packed, env->nbr_packed, env->n_veh_u8 + off,
                           env->n_agents_u8 + off, s);
        env->launches += 2;
        CUDA_OK(cudaEventRecord(env->scan_done[c], s));
        CUDA_OK(cudaEventRecord(env->chunk_done[c], s));
        return 0;
    };
    auto enqueue_copies = [&](int c) -> int {
        const int off = plan.off(c), count = plan.count(c);
        cudaStream_t s = env->streams[HOST_STREAMS + c % HOST_STREAMS];      // copy streams: the compute streams stay busy
        CUDA_OK(cudaEventSynchronize(env->chunk_done[c]));
        const int64_t v0 = env->chunk_base_host[2 * c], v1 = env->chunk_base_host[2 * (c + 1)];
        const int64_t a0 = env->chunk_base_host[2 * c + 1], a1 = env->chunk_base_host[2 * (c + 1) + 1];
        if (v1 > v0)
            CUDA_OK(cudaMemcpyAsync(out->veh + v0 * MM_VEH_F32, env->veh_packed + v0 * MM_VEH_F32, (size_t)(v1 - v0) * MM_VEH_F32 * sizeof(float),
                                    cudaMemcpyDeviceToHost, s));
        if (a1 > a0)
            CUDA_OK(cudaMemcpyAsync(out->nbr + a0, env->nbr_packed + a0, (size_t)(a1 - a0) * sizeof(uint16_t), cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaMemcpyAsync(out->n_veh + off, env->n_veh_u8 + off, (size_t)count, cudaMemcpyDeviceToHost, s));
        CUDA_OK(cudaMemcpyAsync(out->n_agents + off, env->n_agents_u8 + off, (size_t)count, cudaMemcpyDeviceToHost, s));
        return copy_env_outputs(env, off, count, s, out->reward, out->done, out->regional_rewards, nullptr);
    };
    if (int rc = order_after_caller(env, N_STREAMS)) return rc;
    for (int c = 0; c < plan.used; ++c)
        if (int rc = enqueue_compute(c)) return rc;
    for (int c = 0; c < plan.used; ++c)
        if (int rc = enqueue_copies(c)) return rc;
    for (int c = 0; c < N_STREAMS; ++c) CUDA_OK(cudaStreamSynchronize(env->streams[c]));
    CUDA_OK(cudaGetLastError());
    return 0;
}

// Host side of the packed path: the observation rows the reference returns (envs/common/observation.py:241-273 with
// normalize_obs 181-193), rebuilt from the packed state.  Plain CPU code, no device involved.
int mm_expand_obs_rows(const mm_packed_host *in, int n_envs, int steer_vel, float *obs_rows, int64_t *row_offset, int n_threads) {
    if (!in || !in->veh || !in->nbr || !in->n_veh || !in->n_agents || !obs_rows || !row_offset)
        return fail(MM_ERR_ARG, "mm_expand_obs_rows: null argument");
    if (n_envs < 0) return fail(MM_ERR_ARG, "n_envs must be >= 0");
    std::vector<int64_t> vbase((size_t)n_envs + 1);
    int64_t rv = 0, ra = 0;
    for (int e = 0; e < n_envs; ++e) {
        vbase[e] = rv; row_offset[e] = ra;
        rv += in->n_veh[e]; ra += in->n_agents[e];
    }
    vbase[n_envs] = rv; row_offset[n_envs] = ra;
    const double KX = 2.0 / 300.0, KY = 2.0 / 24.0, KV = 2.0 / 90.0, KH = 2.0 / 3.141592653589793, HPI = 3.141592653589793 / 2;
    auto work = [&](int e0, int e1) {
        for (int e = e0; e < e1; ++e) {
            const float *veh = in->veh + vbase[e] * MM_VEH_F32;
            const int n_cav = in->n_agents[e], n_veh = in->n_veh[e];
            double vx[MM_MAXV], vy[MM_MAXV];                      // Vehicle.velocity = speed * [cos, sin](heading)
            for (int j = 0; j < n_veh && j < MM_MAXV; ++j) {
                const double h = veh[j * MM_VEH_F32 + 2], sp = veh[j * MM_VEH_F32 + 3];
                if (h == 0.0) { vx[j] = sp; vy[j] = sp * h; continue; }   // most vehicles drive straight: cos = 1, sin = +-0
                vx[j] = sp * std::cos(h);
                vy[j] = sp * std::sin(h);
            }
            for (int i = 0; i < n_cav && i < n_veh; ++i) {
                float *row = obs_rows + (row_offset[e] + i) * MM_NS;
                const double ex = veh[i * MM_VEH_F32], ey = veh[i * MM_VEH_F32 + 1], eh = veh[i * MM_VEH_F32 + 2];
                const double evx = vx[i], evy = vy[i];
                row[0] = 1.0f; row[1] = (float)((ex + 150.0) * KX - 1.0); row[2] = (float)((ey + 12.0) * KY - 1.0);
                row[3] = (float)((evx + 45.0) * KV - 1.0); row[4] = (float)((evy + 45.0) * KV - 1.0);
                row[5] = (float)((eh + HPI) * KH - 1.0);
                const unsigned w = in->nbr[row_offset[e] + i];
                for (int k = 0; k < 4; ++k) {
                    float *r = row + 6 * (k + 1);
                    const int o = (int)((w >> (4 * k)) & 15u);
                    if (o >= n_veh) { r[0] = r[1] = r[2] = r[3] = r[4] = r[5] = 0.f; continue; }
                    const float *ov = veh + o * MM_VEH_F32;
                    double oh = ov[2];
                    if (steer_vel && o < n_cav) oh = oh - eh;
                    r[0] = 1.0f; r[1] = (float)(((double)ov[0] - ex + 150.0) * KX - 1.0);
                    r[2] = (float)(((double)ov[1] - ey + 12.0) * KY - 1.0); r[3] = (float)((vx[o] - evx + 45.0) * KV - 1.0);
                    r[4] = (float)((vy[o] - evy + 45.0) * KV - 1.0); r[5] = (float)((oh + HPI) * KH - 1.0);
                }
            }
        }
    };
    if (n_threads < 1) n_threads = 1;
    if (n_threads == 1 || n_envs < 4096) { work(0, n_envs); return 0; }
    std::vector<std::thread> pool;
    const int per = (n_envs + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; ++t) {
        const int e0 = t * per, e1 = e0 + per < n_envs ? e0 + per : n_envs;
        if (e0 < e1) pool.emplace_back(work, e0, e1);
    }
    for (auto &th : pool) th.join();
    return 0;
}

int mm_buffers_get(mm_env *env, mm_buffers *b) {
    if (!env || !b) return fail(MM_ERR_ARG, "null argument");
    b->obs = env->out.obs; b->reward = env->out.reward; b->done = env->out.done;
    b->agents_rewards = env->out.agents_rewards; b->regional_rewards = env->out.regional_rewards;
    b->agents_dones = env->out.agents_dones; b->average_speed = env->out.average_speed;
    b->traffic_speed = env->out.traffic_speed; b->min_headway = env->out.min_headway;
    b->merge_percent = env->out.merge_percent; b->n_agents = env->out.n_agents; b->actions = env->actions; b->action_mask = env->out.action_mask;
    b->new_actions = env->new_actions;
    return 0;
}

int mm_get_state(mm_env *env, mm_state_host *dst) {
    if (!env || !dst) return fail(MM_ERR_ARG, "null argument");
    CUDA_OK(cudaSetDevice(env->device));
    const size_t E = (size_t)env->n_envs, P = E * MAXV;
    double *f64 = nullptr; int32_t *i32 = nullptr, *envv = nullptr;
    CUDA_OK(cudaMalloc(&f64, HOST_F64 * P * sizeof(double)));
    CUDA_OK(cudaMalloc(&i32, HOST_I32 * P * sizeof(int32_t)));
    CUDA_OK(cudaMalloc(&envv, HOST_ENV * E * sizeof(int32_t)));
    CUDA_OK(cudaDeviceSynchronize());
    launch_unpack_state(env->st, env->n_envs, f64, i32, envv, nullptr);
    CUDA_OK(cudaDeviceSynchronize());
    double *fd[HOST_F64] = {dst->x, dst->y, dst->heading, dst->speed, dst->target_speed, dst->gvx, dst->rec1_x, dst->rec1_vx,
                            dst->rec2_x, dst->rec2_vx, dst->act_steer, dst->act_acc, dst->safe_steer, dst->safe_acc,
                            dst->timer, dst->min_headway, dst->steering_angle};
    int32_t *id[HOST_I32] = {dst->kind, dst->lane, dst->target_lane, dst->speed_index, dst->crashed, dst->hl_action,
                             dst->hist_len, dst->fg_set, dst->is_collaborating, dst->is_lc_safe, dst->collaborate_adj};
    int32_t *ed[HOST_ENV] = {dst->n_veh, dst->n_cav, dst->n_merge, dst->steps, dst->time};
    for (int k = 0; k < HOST_F64; ++k)
        if (fd[k]) CUDA_OK(cudaMemcpy(fd[k], f64 + k * P, P * sizeof(double), cudaMemcpyDeviceToHost));
    for (int k = 0; k < HOST_I32; ++k)
        if (id[k]) CUDA_OK(cudaMemcpy(id[k], i32 + k * P, P * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (int k = 0; k < HOST_ENV; ++k)
        if (ed[k]) CUDA_OK(cudaMemcpy(ed[k], envv + k * E, E * sizeof(int32_t), cudaMemcpyDeviceToHost));
    cudaFree(f64); cudaFree(i32); cudaFree(envv);
    return 0;
}

int mm_set_state(mm_env *env, const mm_state_host *src) {
    if (!env || !src) return fail(MM_ERR_ARG, "null argument");
    CUDA_OK(cudaSetDevice(env->device));
    const size_t E = (size_t)env->n_envs, P = E * MAXV;
    const double *fd[HOST_F64] = {src->x, src->y, src->heading, src->speed, src->target_speed, src->gvx, src->rec1_x,
                                  src->rec1_vx, src->rec2_x, src->rec2_vx, src->act_steer, src->act_acc, src->safe_steer,
                                  src->safe_acc, src->timer, src->min_headway, src->steering_angle};
    const int32_t *id[HOST_I32] = {src->kind, src->lane, src->target_lane, src->speed_index, src->crashed, src->hl_action,
                                   src->hist_len, src->fg_set, src->is_collaborating, src->is_lc_safe, src->collaborate_adj};
    const int32_t *ed[HOST_ENV] = {src->n_veh, src->n_cav, src->n_merge, src->steps, src->time};
    for (int k = 0; k < HOST_F64; ++k) if (!fd[k]) return fail(MM_ERR_ARG, "mm_set_state: every f64 field is required");
    for (int k = 0; k < HOST_I32; ++k) if (!id[k]) return fail(MM_ERR_ARG, "mm_set_state: every i32 field is required");
    for (int k = 0; k < HOST_ENV; ++k) if (!ed[k]) return fail(MM_ERR_ARG, "mm_set_state: every env field is required");
    for (size_t e = 0; e < E; ++e) {
        const int min_cav = env->cfg.env_hdv ? 0 : 1;      // the all-HDV env has no controlled vehicle
        if (ed[0][e] < 1 || ed[0][e] > 11 || ed[1][e] < min_cav || ed[1][e] > ed[0][e])
            return fail(MM_ERR_STATE, "mm_set_state: need 1 <= n_cav <= n_veh <= 11 (n_cav = 0 only in the all-HDV env)");
        for (int i = 0; i < ed[0][e]; ++i) {
            int kind = id[0][e * MAXV + i];
            if (kind != (i < ed[1][e] ? MM_KIND_CAV : MM_KIND_HDV))
                return fail(MM_ERR_STATE, "mm_set_state: slots [0,n_cav) must be CAVs and [n_cav,n_veh) HDVs");
        }
    }
    bool any_hdv = false;
    for (size_t e = 0; e < E; ++e) any_hdv = any_hdv || ed[1][e] < ed[0][e];
    if (env->hdv_possible != any_hdv) ++env->epoch;
    env->hdv_possible = any_hdv;
    env->last_stream = nullptr;
    double *f64 = nullptr; int32_t *i32 = nullptr, *envv = nullptr;
    CUDA_OK(cudaMalloc(&f64, HOST_F64 * P * sizeof(double)));
    CUDA_OK(cudaMalloc(&i32, HOST_I32 * P * sizeof(int32_t)));
    CUDA_OK(cudaMalloc(&envv, HOST_ENV * E * sizeof(int32_t)));
    for (int k = 0; k < HOST_F64; ++k) CUDA_OK(cudaMemcpy(f64 + k * P, fd[k], P * sizeof(double), cudaMemcpyHostToDevice));
    for (int k = 0; k < HOST_I32; ++k) CUDA_OK(cudaMemcpy(i32 + k * P, id[k], P * sizeof(int32_t), cudaMemcpyHostToDevice));
    for (int k = 0; k < HOST_ENV; ++k) CUDA_OK(cudaMemcpy(envv + k * E, ed[k], E * sizeof(int32_t), cudaMemcpyHostToDevice));
    CUDA_OK(cudaDeviceSynchronize());
    launch_pack_state(env->st, env->n_envs, f64, i32, envv, nullptr);
    StepParams o = step_params(env, nullptr, 0, env->n_envs);
    launch_observe(o, nullptr);
    env->launches += 2;
    CUDA_OK(cudaDeviceSynchronize());
    cudaFree(f64); cudaFree(i32); cudaFree(envv);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_get_shield_diag(mm_env *env, mm_shield_diag_host *dst) {
    if (!env || !dst) return fail(MM_ERR_ARG, "null argument");
    if (!env->record_diag) return fail(MM_ERR_STATE, "handle was created without record_diag");
    CUDA_OK(cudaSetDevice(env->device));
    CUDA_OK(cudaDeviceSynchronize());
    const size_t P = (size_t)env->n_envs * 3 * MAXV;
    int32_t *id[10] = {dst->ran, dst->leader, dst->front_adj, dst->rear_adj, dst->constrain_adj, dst->active, dst->is_lc_safe,
                       dst->moved, dst->hl_action, dst->lane};
    double *fd[10] = {dst->safe_acc, dst->safe_steer, dst->nom_acc, dst->nom_steer, dst->lc_margin,
                      dst->x, dst->y, dst->heading, dst->speed, dst->min_headway};
    for (int k = 0; k < 10; ++k)
        if (id[k]) CUDA_OK(cudaMemcpy(id[k], env->out.sh_i + k * P, P * sizeof(int32_t), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 10; ++k)
        if (fd[k]) CUDA_OK(cudaMemcpy(fd[k], env->out.sh_f + k * P, P * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}

int mm_stats(mm_env *env, mm_stats_t *out, int reset) {
    if (!env || !out) return fail(MM_ERR_ARG, "null argument");
    CUDA_OK(cudaSetDevice(env->device));
    CUDA_OK(cudaDeviceSynchronize());
    std::vector<double> h(env->stats_rows * N_STATS);
    CUDA_OK(cudaMemcpy(h.data(), env->out.stats, h.size() * sizeof(double), cudaMemcpyDeviceToHost));
    double acc[N_STATS] = {0};
    acc[ST_MINHW] = std::numeric_limits<double>::infinity();
    for (size_t r = 0; r < env->stats_rows; ++r)
        for (int k = 0; k < N_STATS; ++k) {
            double v = h[r * N_STATS + k];
            acc[k] = k == ST_MINHW ? std::fmin(acc[k], v) : acc[k] + v;
        }
    out->agent_steps = acc[ST_AGENT_STEPS]; out->env_steps = acc[ST_ENV_STEPS]; out->episodes = acc[ST_EPISODES];
    out->crashed_episodes = acc[ST_CRASHED]; out->reward_sum = acc[ST_REWARD]; out->speed_sum = acc[ST_SPEED];
    out->merge_percent_sum = acc[ST_MERGE]; out->shield_solves = acc[ST_SOLVES]; out->shield_active = acc[ST_ACTIVE];
    out->lane_change_vetoes = acc[ST_VETOES]; out->min_headway = acc[ST_MINHW];
    if (reset) return reset_stats(env);
    return 0;
}

int mm_shield_query(mm_env *env, const double *nom_steer, const double *nom_acc, const mm_shield_query_out *out, void *stream) {
    if (!env || !nom_steer || !nom_acc || !out) return fail(MM_ERR_ARG, "null argument");
    int32_t *oi[7] = {out->ran, out->leader, out->front_adj, out->rear_adj, out->constrain_adj, out->active, out->is_lc_safe};
    for (int k = 0; k < 7; ++k)
        if (!oi[k]) return fail(MM_ERR_ARG, "mm_shield_query: every output array is required");
    if (!out->safe_steer || !out->safe_acc || !out->min_headway) return fail(MM_ERR_ARG, "mm_shield_query: every output array is required");
    CUDA_OK(cudaSetDevice(env->device));
    env->last_stream = (cudaStream_t)stream;
    launch_shield_query(env->st, env->cfg, env->n_envs, nom_steer, nom_acc, out->safe_steer, out->safe_acc, out->min_headway, oi, stream);
    env->launches += 1;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_shield_qp(const double *a, const double *c_lead, const double *c_adj, const uint8_t *has_adj, const double *lo,
                 const double *hi, int64_t n, double *u, uint8_t *active, void *stream) {
    if (!a || !c_lead || !c_adj || !has_adj || !lo || !hi || !u || !active) return fail(MM_ERR_ARG, "null argument");
    if (n < 0) return fail(MM_ERR_ARG, "n must be >= 0");
    launch_qp(a, c_lead, c_adj, has_adj, lo, hi, n, u, active, stream);
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_actor_sample(const float *obs, const int32_t *n_agents, int64_t n_rows, const float *w1, const float *b1,
                    const float *w2, const float *b2, const float *w3, const float *b3, uint64_t seed, uint64_t step,
                    const uint8_t *action_mask, int8_t *actions, float *logp_all, float *logp_sel, void *stream) {
    if (!obs || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !actions) return fail(MM_ERR_ARG, "null argument");
    if (n_rows < 0) return fail(MM_ERR_ARG, "n_rows must be >= 0");
    if (n_agents && n_rows % MAXV != 0) return fail(MM_ERR_ARG, "n_rows must be a multiple of MM_MAXV when n_agents is given");
    if (launch_actor_sample(obs, n_agents, n_rows, w1, b1, w2, b2, w3, b3, seed, step, action_mask, actions, logp_all, logp_sel,
                            stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int mm_actor_sample_mlp(const float *obs, const int32_t *n_agents, int64_t n_rows, int h1, const float *w1, const float *b1,
                        const float *w2, const float *b2, const float *w3, const float *b3, const float *value_w,
                        const float *value_b, uint64_t seed, uint64_t step, const uint8_t *action_mask, int8_t *actions,
                        float *logp_all, float *logp_sel, float *values, float *obs_copy, uint8_t *live_out, void *stream) {
    if (!obs || !w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !actions) return fail(MM_ERR_ARG, "null argument");
    if (h1 != 128 && h1 != 160) return fail(MM_ERR_ARG, "h1 must be 128 (ActorNetwork) or 160 (ActorCriticNetwork, state_split)");
    if (n_rows < 0) return fail(MM_ERR_ARG, "n_rows must be >= 0");
    if (n_agents && n_rows % MAXV != 0) return fail(MM_ERR_ARG, "n_rows must be a multiple of MM_MAXV when n_agents is given");
    if (values && (!value_w || !value_b)) return fail(MM_ERR_ARG, "values needs value_w and value_b");
    if (launch_actor_mlp(obs, n_agents, n_rows, h1, w1, b1, w2, b2, w3, b3, value_w, value_b, seed, step, action_mask, actions,
                         logp_all, logp_sel, values, obs_copy, live_out, stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int mm_set_actor_impl(int impl) {
    if (impl != 0 && impl != 1) return fail(MM_ERR_ARG, "impl must be 0 (tcgen05 fp16, default) or 1 (mma.sync TF32 cross-check)");
    set_actor_impl(impl);
    return 0;
}

int mm_supervise(mm_env *env, int kind, int8_t *actions_dev, const double *draws_dev, int32_t *n_used_dev, void *stream) {
    if (!env) return fail(MM_ERR_ARG, "env is null");
    if (kind != 0 && kind != 1) return fail(MM_ERR_ARG, "kind must be 0 (priority) or 1 (dmc)");
    if (!actions_dev) return fail(MM_ERR_ARG, "actions are required");
    if (int rc = ensure_supervisor_stack(env)) return rc;
    env->last_stream = (cudaStream_t)stream;
    launch_supervisor(env->st, 0, env->n_envs, kind, actions_dev, draws_dev, MM_SUPERVISOR_DRAWS, env->cfg.headway_time, env->seed,
                      n_used_dev, env->sup_tasks, env->sup_task_count, env->n_envs * MM_SUP_TASKS_PER_ENV, stream);
    env->launches += kind == 1 ? 2 : 1;
    CUDA_OK(cudaGetLastError());
    return 0;
}

int mm_set_step_variant(int variant) {
    if (variant != 0 && (variant < 3 || variant > 8))
        return fail(MM_ERR_ARG, "variant must be 0 (automatic), 3, 4 (a generic build forced), 5 (automatic, generic builds only) "
                                "6 (4 CTAs per SM forced, specialised builds allowed), 7 (warp-cooperative build forced) or 8 (automatic among the "
                                "one-thread-per-env builds)");
    set_step_variant(variant);
    return 0;
}

int mm_discounted_returns(const float *rewards, const uint8_t *dones, const float *final_value, float gamma, int T,
                          int64_t n_cols, int cols_per_env, float *out, void *stream) {
    if (!rewards || !dones || !out) return fail(MM_ERR_ARG, "null argument");
    if (T < 0 || n_cols < 0 || cols_per_env <= 0 || n_cols % cols_per_env != 0)
        return fail(MM_ERR_ARG, "bad rollout shape");
    if (launch_discounted_returns(rewards, dones, nullptr, final_value, gamma, 1.f, T, n_cols, cols_per_env, out, stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int mm_lambda_returns(const float *rewards, const uint8_t *dones, const float *values, const float *final_value, float gamma,
                      float lambda, int T, int64_t n_cols, int cols_per_env, float *out, void *stream) {
    if (!rewards || !dones || !out) return fail(MM_ERR_ARG, "rewards, dones and out are required");
    if (T < 0 || n_cols < 0 || cols_per_env <= 0 || n_cols % cols_per_env != 0)
        return fail(MM_ERR_ARG, "bad rollout shape");
    if (!(lambda >= 0.f && lambda <= 1.f)) return fail(MM_ERR_ARG, "lambda must be in [0, 1]");
    if (!std::isfinite(gamma)) return fail(MM_ERR_ARG, "gamma must be finite");
    if (lambda < 1.f && !values) return fail(MM_ERR_ARG, "values are required for lambda < 1");
    if (launch_discounted_returns(rewards, dones, values, final_value, gamma, lambda, T, n_cols, cols_per_env, out, stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

static int check_ppo_net(int kind, const mm_ppo_net *net) {
    if (kind != MM_PPO_ACTOR && kind != MM_PPO_CRITIC && kind != MM_PPO_SHARED)
        return fail(MM_ERR_ARG, "kind must be 0 (MAPPO actor), 1 (MAPPO critic) or 2 (MAPPO_GI shared network)");
    if (!net || !net->w1 || !net->b1 || !net->w2 || !net->b2 || !net->w3 || !net->b3)
        return fail(MM_ERR_ARG, "net: w1, b1, w2, b2, w3 and b3 are required");
    if (kind == MM_PPO_SHARED && (!net->w4 || !net->b4)) return fail(MM_ERR_ARG, "net: the shared network needs w4 and b4 (critic_linear)");
    return 0;
}

int mm_ppo_targets(int kind, const float *states, const int8_t *actions, const int64_t *idx, int64_t n, const mm_ppo_net *net,
                   float *old_logp, float *q_target, void *stream) {
    if (int rc = check_ppo_net(kind, net)) return rc;
    if (!states || !actions || !idx) return fail(MM_ERR_ARG, "states, actions and idx are required");
    if (kind == MM_PPO_CRITIC ? !q_target : !old_logp)
        return fail(MM_ERR_ARG, kind == MM_PPO_CRITIC ? "the critic's target pass writes q_target" : "the target pass writes old_logp");
    if (n < 1) return fail(MM_ERR_ARG, "n must be >= 1");
    if (launch_ppo_targets(kind, states, actions, idx, n, net, old_logp, q_target, stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int mm_ppo_grads(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                 const float *q_target, const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net,
                 const mm_ppo_grads_out *grads, float *losses, void *stream) {
    if (int rc = check_ppo_net(kind, net)) return rc;
    if (!states || !actions || !returns || !idx || !grads || !losses) return fail(MM_ERR_ARG, "states, actions, returns, idx, grads and losses are required");
    if (!grads->w1 || !grads->b1 || !grads->w2 || !grads->b2 || !grads->w3 || !grads->b3 ||
        (kind == MM_PPO_SHARED && (!grads->w4 || !grads->b4)))
        return fail(MM_ERR_ARG, "grads: one output buffer per parameter is required");
    if (kind != MM_PPO_CRITIC && !old_logp) return fail(MM_ERR_ARG, "old_logp (from the target pass) is required");
    if (kind == MM_PPO_ACTOR && !q_target) return fail(MM_ERR_ARG, "q_target (from the critic's target pass) is required");
    if (n < 1) return fail(MM_ERR_ARG, "n must be >= 1");
    if (!(clip > 0.f && clip < 1.f)) return fail(MM_ERR_ARG, "clip must be in (0, 1)");
    if (launch_ppo_grads(kind, states, actions, returns, old_logp, q_target, idx, n, clip, net, grads, losses, stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int mm_ppo_stats(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                 const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net, double *stats, void *stream) {
    if (int rc = check_ppo_net(kind, net)) return rc;
    if (n < 0) return fail(MM_ERR_ARG, "n must be >= 0");
    if (!stats) return fail(MM_ERR_ARG, "stats is required");
    if (n > 0 && (!states || !actions || !idx)) return fail(MM_ERR_ARG, "states, actions and idx are required");
    if (n > 0 && kind != MM_PPO_ACTOR && !returns) return fail(MM_ERR_ARG, "returns are required for the value statistics");
    if (old_logp && !(clip > 0.f && clip < 1.f)) return fail(MM_ERR_ARG, "clip must be in (0, 1)");
    if (launch_ppo_stats(kind, states, actions, returns, old_logp, idx, n, clip, net, stats, stream))
        return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

int mm_rmsprop_step(const mm_opt_group *groups, int n_groups, void *stream) {
    if (!groups) return fail(MM_ERR_ARG, "groups is null");
    if (n_groups < 1 || n_groups > MM_OPT_MAX_GROUPS) return fail(MM_ERR_ARG, "n_groups must be in 1..MM_OPT_MAX_GROUPS (8)");
    for (int gi = 0; gi < n_groups; ++gi) {
        const mm_opt_group &g = groups[gi];
        if (!g.tensors) return fail(MM_ERR_ARG, "group tensors is null");
        if (g.n_tensors < 1 || g.n_tensors > MM_OPT_MAX_TENSORS)
            return fail(MM_ERR_ARG, "n_tensors must be in 1..MM_OPT_MAX_TENSORS (16)");
        for (int k = 0; k < g.n_tensors; ++k) {
            const mm_opt_tensor &t = g.tensors[k];
            if (!t.param || !t.grad || !t.square_avg) return fail(MM_ERR_ARG, "param, grad and square_avg are required");
            if (t.numel < 0) return fail(MM_ERR_ARG, "numel must be >= 0");
            if (!t.mirror) continue;
            if (!t.mirror_cols || t.mirror_ncols < 1 || t.mirror_ncols > MM_OPT_MAX_MIRROR_COLS)
                return fail(MM_ERR_ARG, "a mirror needs a column map (mirror_cols, 1..16 entries)");
            if (t.mirror_ld < 1) return fail(MM_ERR_ARG, "mirror_ld must be >= 1");
            if (t.numel % t.mirror_ncols != 0) return fail(MM_ERR_ARG, "numel must be a multiple of mirror_ncols");
            for (int c = 0; c < t.mirror_ncols; ++c)
                if (t.mirror_cols[c] < 0 || t.mirror_cols[c] >= t.mirror_ld || t.mirror_cols[c] > 255)
                    return fail(MM_ERR_ARG, "mirror_cols must lie in [0, min(mirror_ld, 256))");
        }
    }
    if (launch_rmsprop_step(groups, n_groups, stream)) return fail(MM_ERR_CUDA, cudaGetErrorString(cudaGetLastError()));
    return 0;
}

}  // extern "C"

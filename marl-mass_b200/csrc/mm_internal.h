// mm_internal.h — layout shared by the kernels (merge_step.cu) and the host side of the C ABI (capi.cu).
//
// HBM layout: array of tiles of structure-of-arrays.  A tile is TILE = 128 consecutive envs (= one CTA);
// inside a tile every (field, slot) is a contiguous run of 128 values, so a warp's access is one or two
// fully used 128-byte lines, and the whole state of a CTA is one contiguous ~190 KB span (one TLB entry —
// a plain [field][slot][E] layout put the 180 planes of an env 8 MB apart at E = 2^20 and thrashed the
// 128-entry TLB: 80 ms/step instead of 22, profiles/r1_v1_*).
//   f64   [n_tiles][F_COUNT][MM_MAXV][TILE]   vehicle state (15 reference fields + cached cos/sin of the heading)
//   flags [n_tiles][MM_MAXV][TILE] u32        packed discrete vehicle state (bit layout below)
//   einfo [E_pad] u32                         packed env scalars: n_veh, n_cav, n_merge, steps, time
//   episode [E_pad] u32                       episode counter (RNG stream id for device-side spawn)
// Outputs are env-major (what the caller consumes): obs [E][MM_MAXV][MM_NS] f32, etc.
#pragma once
#include <stdint.h>
#include <stddef.h>
#include "marl_mass_b200.h"

namespace mm {

constexpr int MAXV = MM_MAXV;
constexpr int NS = MM_NS;
#ifndef MM_TILE
#define MM_TILE 128
#endif
constexpr int TILE = MM_TILE;   // envs per tile == threads per CTA of the step kernel
#define MM_MAX_DEVICES 64        // per-device one-time setup tables (function attributes)

enum F64Field {
    F_X = 0, F_Y, F_H, F_V,          // position, heading, speed            (staged in shared memory)
    F_COSH, F_SINH,                  // cos / sin of the heading (derived; refreshed by every move; staged as well)
    F_TSPEED,                        // target_speed
    F_GVX,                           // fg_params["g"]["vx"] of the last integration
    F_REC1VX,                        // state_hist[-1]["vx"] (x of that record == current x)
    F_REC2X, F_REC2VX,               // state_hist[-2]["x"], ["vx"]
    F_ACT_STEER, F_ACT_ACC,          // low-level action of the current sub-step
    F_SAFE_STEER, F_SAFE_ACC,        // shielded action of the last step()
    F_TIMER,                         // IDMVehicle.timer
    F_MINHW,                         // MDPLCVehicle.min_headway
    F_STEERANG,                      // MDPLCVehicle.steering_angle (lateral_control = steer_vel only)
    F_COUNT
};

// flags word
constexpr uint32_t FL_KIND_SHIFT = 0, FL_KIND_MASK = 3u;
constexpr uint32_t FL_LANE_SHIFT = 2, FL_TLANE_SHIFT = 5, FL_SIDX_SHIFT = 8, FL_3BIT = 7u;
constexpr uint32_t FL_CRASHED = 1u << 11;
constexpr uint32_t FL_HL_SHIFT = 12;         // 3 bits, 7 = None
constexpr uint32_t FL_HIST_SHIFT = 15;       // 2 bits, saturating len(state_hist)
constexpr uint32_t FL_FG = 1u << 17;
constexpr uint32_t FL_COLLAB = 1u << 18;     // is_collaborating
constexpr uint32_t FL_LCSAFE = 1u << 19;     // is_lc_safe
constexpr uint32_t FL_CADJ = 1u << 20;       // collaborate_adj

// einfo word
constexpr uint32_t EI_NVEH_SHIFT = 0, EI_NCAV_SHIFT = 4, EI_NMERGE_SHIFT = 8, EI_4BIT = 15u;
constexpr uint32_t EI_STEPS_SHIFT = 12, EI_STEPS_MASK = 255u;
constexpr uint32_t EI_TIME_SHIFT = 20, EI_TIME_MASK = 4095u;

struct DevState {
    double *f64;        // [n_tiles][F_COUNT][MAXV][TILE]
    uint32_t *flags;    // [n_tiles][MAXV][TILE]
    uint32_t *einfo;    // [E_pad]
    uint32_t *episode;  // [E_pad]
};

struct DevOut {
    float *obs, *reward, *agents_rewards, *regional_rewards, *average_speed, *traffic_speed, *min_headway,
          *merge_percent;
    uint8_t *done, *agents_dones, *action_mask;
    int32_t *n_agents;
    // packed-state outputs (mm_step_host_packed; null until that path is first used): per vehicle x, y, heading, speed
    // as float32 [E][MAXV][MM_VEH_F32], and per agent the slots of its (up to) 4 observed neighbours, 4 bits each in observation
    // order, 0xF = none [E][MAXV]
    float *veh;
    uint16_t *nbr;
    // per-sub-step shield record [E][3][MAXV] (record_diag only, else null)
    int32_t *sh_i;      // 10 planes: ran, leader, front_adj, rear_adj, constrain_adj, active, is_lc_safe, moved, hl_action, lane
    double *sh_f;       // 10 planes: safe_acc, safe_steer, nom_acc, nom_steer, lc_margin, x, y, heading, speed, min_headway
    double *stats;      // [N_STATS] accumulators
};

enum StatSlot { ST_AGENT_STEPS = 0, ST_ENV_STEPS, ST_EPISODES, ST_CRASHED, ST_REWARD, ST_SPEED, ST_MERGE,
                ST_SOLVES, ST_ACTIVE, ST_VETOES, ST_MINHW, N_STATS };

struct StepParams {
    DevState st;
    DevOut out;
    const int8_t *actions;   // [E][MAXV]
    mm_config cfg;
    int n_envs;
    int env_offset;          // first env of this launch (chunked host path)
    int env_count;           // envs in this launch
    const uint8_t *obs_mask; // outputs kernel without rewards: refresh only envs whose mask byte is set (null: all)
    int all_cav;             // host-side knowledge: no env of the handle can hold an HDV (enables the specialised builds)
};

struct ResetParams {
    DevState st;
    DevOut out;
    const uint8_t *mask;     // [E] or null; when use_done != 0 the done flags are the mask
    mm_config cfg;
    uint64_t seed;
    int n_envs, env_offset, env_count, num_cav, use_done;
};

struct SeededResetParams {
    DevState st;
    mm_config cfg;
    const int64_t *seeds;    // [n_envs] in [0, 2^32), checked by mm_reset_seeded
    const int32_t *num_cav;  // [n_envs] or null (0: drawn)
    int n_envs;
};

// launchers (merge_step.cu)
int launch_step(const StepParams &p, bool diag, void *stream);   // returns the MM_BUILD_* it launched
// the same kernel compiled for 4 CTAs per SM (merge_step_occ4.cu): picked when that makes the grid a single wave
void launch_step_occ4(const StepParams &p, bool diag, void *stream);
// the same kernel specialised at compile time for all-CAV envs of the plain LC env (merge_step_spec_mass.cu / _hss.cu)
void launch_step_spec_mass(const StepParams &p, bool diag, void *stream);
void launch_step_spec_hss(const StepParams &p, bool diag, void *stream);
void launch_step_spec_mass4(const StepParams &p, bool diag, void *stream);   // ... and for 4 CTAs per SM
void launch_step_spec_hss4(const StepParams &p, bool diag, void *stream);
// the warp-cooperative build: half a warp per env, one lane per vehicle (merge_coop.cu); all-CAV plain LC envs only
void launch_step_coop(const StepParams &p, bool diag, void *stream);
unsigned long long step_variant_epoch();   // changes whenever set_step_variant was called
void set_step_variant(int v);   // 0: automatic, 3 / 4: force the generic 3- or 4-CTAs-per-SM build, 5: automatic without the specialised builds
void launch_reset(const ResetParams &p, void *stream);
void launch_seeded_reset(const SeededResetParams &p, void *stream);   // the scenes of spawn.py (spawn_core.h)
// evaluation records of policy step t (eval_record.cu); arguments already checked by mm_eval_record
void launch_eval_record(const DevState &st, const DevOut &out, int n_envs, const mm_eval_records &r, int t, void *stream);
// shield records and control profiles of policy step t from the diagnostic record (eval_record.cu); checked by
// mm_eval_shield_record
void launch_eval_shield_record(const DevOut &out, int n_envs, const mm_eval_shield_records &r, int t, void *stream);
// outputs kernel (merge_outputs.cu): observations, rewards, terminal flags, info scalars and statistics of the policy step
// the physics kernel has just advanced (with_rewards), or the first observation after a (re)spawn / set_state (!with_rewards,
// optionally only for envs whose p.obs_mask byte is set)
void launch_outputs(const StepParams &p, bool with_rewards, void *stream);
inline void launch_observe(const StepParams &p, void *stream) { launch_outputs(p, false, stream); }
void launch_pack_state(const DevState &st, int n_envs, const double *f64_em /*[17][E][MAXV]*/,
                       const int32_t *i32_em /*[11][E][MAXV]*/, const int32_t *env_em /*[5][E]*/, void *stream);
void launch_unpack_state(const DevState &st, int n_envs, double *f64_em, int32_t *i32_em, int32_t *env_em,
                         void *stream);
// out_i: ran, leader, front_adj, rear_adj, constrain_adj, active, is_lc_safe (device arrays [n_envs][MAXV])
void launch_shield_query(const DevState &st, const mm_config &cfg, int n_envs, const double *nom_steer, const double *nom_acc,
                         double *safe_steer, double *safe_acc, double *min_headway, int32_t *const *out_i, void *stream);
void launch_qp(const double *a, const double *c_lead, const double *c_adj, const uint8_t *has_adj,
               const double *lo, const double *hi, int64_t n, double *u, uint8_t *active, void *stream);

// obs / n_agents / row_offset_dev are passed already offset to the chunk; rows_stage is the base of the device staging
// buffer [E * MAXV][NS] (row offsets are absolute); chunk_rows_dev receives the chunk's packed row count
void launch_ragged_pack(const float *obs, const int32_t *n_agents, int count, int64_t base_row, int64_t *row_offset_dev,
                        int64_t *chunk_rows_dev, float *rows_stage, void *stream);

// mm_step_host_packed: exclusive scans of n_veh / n_agents over a chunk of envs (chained to the previous chunk's totals
// through base_in -> base_out, two int64 each: vehicles, agents; base_out_host = the same totals written to mapped pinned
// host memory, so that no device-to-host copy of them queues in front of the data copies) and the ragged copy of the chunk's vehicle rows and
// neighbour words to their packed place
void launch_packed_pack(const uint32_t *einfo, const int32_t *n_agents, const float *veh, const uint16_t *nbr, int count,
                        const int64_t *base_in, int64_t *base_out, int64_t *base_out_host, int32_t *voff, int32_t *aoff,
                        float *veh_packed, uint16_t *nbr_packed, uint8_t *n_veh_u8, uint8_t *n_agents_u8, void *stream);

// caller-side kernels (actor_sample.cu)
int launch_actor_sample(const float *obs, const int32_t *n_agents, int64_t n_rows, const float *w1, const float *b1,
                        const float *w2, const float *b2, const float *w3, const float *b3, uint64_t seed, uint64_t step,
                        const uint8_t *mask_bits, int8_t *actions, float *logp_all, float *logp_sel, void *stream);
void set_actor_impl(int impl);   // 0: the fp16 tcgen05 kernel (default), 1: the mma.sync cross-check (checked by the C ABI)
// the fp16 tcgen05 kernel for a 30 - h1 - 128 - 5 network (h1 = 128 or 160), optional value head (wv [128], bv [1] -> values)
int launch_actor_mlp(const float *obs, const int32_t *n_agents, int64_t n_rows, int h1, const float *w1, const float *b1,
                     const float *w2, const float *b2, const float *w3, const float *b3, const float *wv, const float *bv,
                     uint64_t seed, uint64_t step, const uint8_t *mask_bits, int8_t *actions, float *logp_all, float *logp_sel,
                     float *values, float *obs_copy, uint8_t *live_out, void *stream);
int launch_discounted_returns(const float *rewards, const uint8_t *dones, const float *values, const float *final_value,
                              float gamma, float lambda, int T, int64_t n_cols, int cols_per_env, float *out, void *stream);

// on-device PPO learner (learner.cu); arguments already checked by the C ABI
int launch_ppo_targets(int kind, const float *states, const int8_t *actions, const int64_t *idx, int64_t n, const mm_ppo_net *net,
                       float *old_logp, float *q_target, void *stream);
int launch_ppo_grads(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                     const float *q_target, const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net,
                     const mm_ppo_grads_out *grads, float *losses, void *stream);
int launch_ppo_stats(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                     const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net, double *stats, void *stream);
// clip_grad_norm_ + RMSprop, one CTA per group (optim.cu); arguments already checked by the C ABI
int launch_rmsprop_step(const mm_opt_group *groups, int n_groups, void *stream);

// envs [env_offset, env_offset + env_count); draws null: Philox draws keyed (seed, env, episode, step); n_used_out
// (nullable) [n_envs]: how many draws each env's supervisor consumed
void launch_supervisor(const DevState &st, int env_offset, int env_count, int kind, int8_t *actions, const double *draws,
                       int draws_per_env, double headway_time, uint64_t seed, int32_t *n_used_out, void *tasks,
                       int *task_count, int task_capacity, void *stream);
size_t supervisor_task_bytes();

// element (field f, slot i) of env e
__host__ __device__ inline size_t f64_index(size_t e, int f, int i) {
    return (((e / TILE) * F_COUNT + (size_t)f) * MAXV + (size_t)i) * TILE + (e % TILE);
}
__host__ __device__ inline size_t flags_index(size_t e, int i) {
    return ((e / TILE) * MAXV + (size_t)i) * TILE + (e % TILE);
}

}  // namespace mm

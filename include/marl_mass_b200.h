/* marl_mass_b200.h — C ABI of the B200-native batched merge environment + HSS/MASS CBF shields.
 *
 * The reference (hkbharath/MARL-MASS) is pure Python and has no FFI; its boundary for this path is two
 * Python call surfaces (SURVEY.md §8b).  Each entry point below names the reference interface it replaces
 * (paths relative to the reference tree).  The Python host (marl-mass_b200/env.py) binds these with ctypes;
 * INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions: every function returns 0 on success and a negative mm_status on failure, never throws;
 * mm_last_error() gives the text.  A handle owns all of its device memory.  Kernels are enqueued on the
 * caller's stream (a cudaStream_t passed as void*; NULL = default stream) with no implicit synchronisation,
 * except the *_host entry points, which return after the results are in the host buffers.
 * One host thread per handle.
 *
 * Host-side state/diagnostic arrays are env-major, [n_envs][MM_MAXV] per vehicle field, slot = index in the
 * reference's road.vehicles (CAVs first, which is also controlled_vehicles order and the vehicle id).
 */
#ifndef MARL_MASS_B200_H
#define MARL_MASS_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MM_MAXV 12          /* vehicle slots per env (reference max is 11: td3 = 6 CAV + 5 HDV) */
#define MM_OBS_ROWS 5       /* KinematicLCObservation vehicles_count (observation.py:132) */
#define MM_OBS_FEATS 6      /* presence,x,y,vx,vy,heading (observation.py:232) */
#define MM_NS 30            /* MergeEnvLCMARL.n_s (merge_env_v1.py:413) */
#define MM_NA 5             /* n_a: LANE_LEFT, IDLE, LANE_RIGHT, FASTER, SLOWER (action.py:141-147) */
#define MM_VEH_F32 4        /* floats per vehicle of the packed host path: x, y, heading, speed */

typedef enum { MM_OK = 0, MM_ERR_ARG = -1, MM_ERR_CUDA = -2, MM_ERR_STATE = -3 } mm_status;

enum { MM_KIND_NONE = 0, MM_KIND_CAV = 1, MM_KIND_HDV = 2 };
enum { MM_SHIELD_NONE = 0, MM_SHIELD_HSS = 1, MM_SHIELD_MASS = 2 };
enum { MM_REW_DEFAULT = 0, MM_REW_SREW = 1, MM_REW_MREW = 2 };
enum { MM_TRAFFIC_CAV = 0, MM_TRAFFIC_MIXED = 1, MM_TRAFFIC_AV = 2 /* one CAV, the rest HDVs (merge_env_v1.py:485-489) */,
       MM_TRAFFIC_HDV = 3 /* HDVs only (490-494); with env_hdv */ };
enum { MM_SUPERVISOR_NONE = 0, MM_SUPERVISOR_PRIORITY = 1, MM_SUPERVISOR_DMC = 2 };
enum { MM_NB_NONE = -1, MM_NB_OBSTACLE = -2 };
/* QP active-set code reported per shield solve */
enum { MM_ACT_LEAD = 1, MM_ACT_UPPER = 2, MM_ACT_LOWER = 4, MM_ACT_ADJ = 8, MM_ACT_SLACK = 16 };

/* Replaces: env.config[...] keys set by run_mappo.py:145-171 and the class globals CBFType.GAMMA_B / TAU
 * (run_mappo.py:137-139).  As in the reference, a changed config is picked up by the next reset. */
/* ABI guard: MM_ABI_VERSION changes whenever a struct of this header changes layout or an entry point changes its
 * signature; mm_abi_version() returns the value the library was built with, and mm_create / mm_set_config reject a
 * config whose struct_size field is not sizeof(mm_config) (a binding built against another revision of the header
 * fails loudly instead of handing the library garbage). */
#define MM_ABI_VERSION 9
int mm_abi_version(void);

typedef struct {
    int32_t struct_size;     /* = sizeof(mm_config), set by the caller (ABI guard) */
    int32_t shield;          /* safety_guarantee: none -> NONE; cbf-avs_cint|hss|av|avs -> HSS; cbf-cav|mass -> MASS */
    int32_t reward_kind;     /* agent_reward: default | srew | mrew */
    int32_t traffic_density; /* 1..3 (merge_env_v1.py:180-211) */
    int32_t traffic_type;    /* cav (all vehicles are CAVs) | mixed (HDVs are IDMVehicleHist) */
    int32_t duration_steps;  /* duration * policy_frequency (100) */
    int32_t substeps;        /* simulation_frequency // policy_frequency (3) */
    double dt;               /* 1 / simulation_frequency */
    double eta;              /* cbf_eta -> CBFType.GAMMA_B */
    double tau;              /* HEADWAY_TIME -> CBFType.TAU */
    double collision_reward, high_speed_reward, headway_cost, headway_time, merging_lane_cost;
    int32_t env_v0;          /* 1: env id merge-multi-agent-v0 (MergeEnvMARL, merge_env_v1.py:389-408): MDPVehicle CAVs
                                (no [-12.5, 6] acceleration clip, never shielded); obs columns 0..4 of each row */
    int32_t steer_vel;       /* 1: lateral_control = steer_vel (safe_controller.py:84-98,124-150): steering angle is a
                                state driven by a steering-velocity command; neighbour CAV headings are observed
                                relative to the ego */
    int32_t couple_counts;   /* device spawn only (no reference counterpart; default 0).  1: the vehicle COUNTS of an
                                episode (merge_env_v1.py:180-211) are drawn once per 128-env tile instead of once per
                                env; every env still follows the reference's law, but the envs of a tile share
                                (n_CAV, n_HDV), which lets a CTA skip the vehicle ranks none of its envs has */
    int32_t env_hdv;         /* 1: env id merge-multi-agent-hdv-v1 (MergeEnvLCHDV, merge_env_v1.py:552-674; traffic_type
                                hdv): no controlled vehicles - every vehicle is observed and rewarded (its row in obs /
                                agents_rewards), any crash ends the episode, no regional rewards / per-agent dones */
    int32_t supervisor;      /* safety_guarantee: priority -> PRIORITY, dmc -> DMC, else NONE.  The look-ahead baselines
                                (vehicle/safety/central_layer.py:16-178, decentralised_dmc.py:70-198) that AbstractEnv.step
                                runs on the action tuple before _simulate (abstract.py:459-464); shield must be NONE */
} mm_config;

typedef struct mm_env mm_env;

/* Host mirror of the full per-env state, for teacher forcing (SURVEY.md §8c) and checkpointing.
 * Replaces: nothing in the reference (it never checkpoints env state); fields follow
 * Vehicle / ControlledVehicle / MDPLCVehicle / IDMVehicleHist attributes.
 * rec1_* / rec2_* are state_hist[-1] / state_hist[-2] (x and vx of the record).  The reference logs a record right
 * after every move (safe_controller.py:187-205, behavior.py:509-519), so between policy steps rec1_x == x always:
 * mm_set_state does not store rec1_x (it is not read back from the caller's buffer), mm_get_state returns x for it. */
typedef struct {
    double *x, *y, *heading, *speed, *target_speed, *gvx, *rec1_x, *rec1_vx, *rec2_x, *rec2_vx,
           *act_steer, *act_acc, *safe_steer, *safe_acc, *timer, *min_headway,
           *steering_angle;                                                        /* [n_envs][MM_MAXV] */
    int32_t *kind, *lane, *target_lane, *speed_index, *crashed, *hl_action, *hist_len, *fg_set,
            *is_collaborating, *is_lc_safe, *collaborate_adj;                        /* [n_envs][MM_MAXV] */
    int32_t *n_veh, *n_cav, *n_merge, *steps, *time;                                 /* [n_envs] */
} mm_state_host;

/* Device pointers of the step outputs (valid until mm_destroy; contents valid after the step's stream work).
 * Replaces the return values of MergeEnv.step (merge_env_v1.py:126-166) and AbstractEnv.step's info dict
 * (abstract.py:489-498). */
typedef struct {
    float *obs;               /* [n_envs][MM_MAXV][MM_NS]; rows >= n_agents are zero */
    float *reward;            /* [n_envs] mean of local rewards (merge_env_v1.py:517-524) */
    uint8_t *done;            /* [n_envs] _is_terminal (merge_env_v1.py:168-172) */
    float *agents_rewards;    /* [n_envs][MM_MAXV] info["agents_rewards"] */
    float *regional_rewards;  /* [n_envs][MM_MAXV] info["regional_rewards"] */
    uint8_t *agents_dones;    /* [n_envs][MM_MAXV] info["agents_dones"] */
    float *average_speed;     /* [n_envs] info["average_speed"] */
    float *traffic_speed;     /* [n_envs] info["traffic_speed"] */
    float *min_headway;       /* [n_envs] info["min_headway"] */
    float *merge_percent;     /* [n_envs] info["merge_percent"] at done, else -1 */
    int32_t *n_agents;        /* [n_envs] len(env.controlled_vehicles) */
    int8_t *actions;          /* [n_envs][MM_MAXV] device-side action buffer read by mm_step(actions=NULL) */
    uint8_t *action_mask;     /* [n_envs][MM_MAXV] bit a = meta-action a available (_get_available_actions,
                                 abstract.py:219-240), per agent; info["action_mask"] when action_masking is on */
    int8_t *new_actions;      /* [n_envs][MM_MAXV] info["new_action"]: the tuple _simulate executed when a baseline
                                 supervisor is configured (abstract.py:458-467); not written otherwise */
} mm_buffers;

/* Host arrays receiving the per-sub-step shield record of the last mm_step, [n_envs][3][MM_MAXV].
 * Replaces: safe_status/safe_diff/safe_action logged by MDPLCVehicle.log_step (safe_controller.py:187-227). */
typedef struct {
    int32_t *ran, *leader, *front_adj, *rear_adj, *constrain_adj, *active, *is_lc_safe;
    /* control profile (safe_controller.py:187-227 log_step), every vehicle that moved in the sub-step: */
    int32_t *moved, *hl_action /* -1 none */, *lane;
    double *safe_acc, *safe_steer, *nom_acc, *nom_steer, *lc_margin;   /* applied and nominal action (all vehicles) */
    double *x, *y, *heading, *speed, *min_headway;                     /* state after the sub-step's move */
} mm_shield_diag_host;

/* Episode statistics accumulated on the device since the last mm_stats(reset=1).
 * Sums are what ranks all-reduce(SUM); min_headway all-reduces with MIN. */
typedef struct {
    double agent_steps, env_steps, episodes, crashed_episodes, reward_sum, speed_sum, merge_percent_sum,
           shield_solves, shield_active, lane_change_vetoes;
    double min_headway;
} mm_stats_t;

/* gym.make(env_id) + config mutation (run_mappo.py:143-171).  record_diag != 0 keeps the per-sub-step shield
 * record (test / control-profile use; costs extra stores). */
int mm_create(const mm_config *cfg, int n_envs, int device, int record_diag, mm_env **out);
int mm_destroy(mm_env *env);
int mm_set_config(mm_env *env, const mm_config *cfg);
int mm_num_envs(const mm_env *env);

/* AbstractEnv.reset (abstract.py:176-209) for every env whose mask byte is non-zero (mask == NULL: all).
 * Spawn follows merge_env_v1.py:180-211,265-364 with a counter-based RNG keyed by (seed, env index, episode
 * counter): the same law as the reference, not the same MT19937 stream (use mm_set_state for exact scenes).
 * num_cav > 0 pins the CAV count (reset(num_CAV=...)).  mask is a DEVICE pointer.  Writes the first obs. */
int mm_reset(mm_env *env, uint64_t seed, const uint8_t *mask_dev, int num_cav, void *stream);

/* AbstractEnv.reset(is_training=False, testing_seeds=seeds[e], num_CAV=num_cav[e]) for every env at once: exactly the
 * reference's scene for each seed, built on the device from its MT19937 draws (numpy's legacy RandomState(seed), as
 * spawn.py replays it on the host).  The state is what mm_set_state leaves for that scene - every field, einfo, the
 * episode counters and the spawn seed untouched - and obs / n_agents / action_mask are refreshed as mm_set_state does.
 * seeds [n_envs] int64 and num_cav [n_envs] int32 (NULL: 0, the count is drawn) are HOST arrays, copied before the call
 * returns; the work is enqueued on `stream` without synchronisation.  Arguments are checked before any CUDA call
 * (MM_ERR_ARG): a seed outside [0, 2^32) (where numpy raises ValueError), a num_cav outside 0..11, and a num_cav for
 * which the reference's spawn would raise or build more than 11 vehicles (that depends on the seed's HDV-count draw). */
int mm_reset_seeded(mm_env *env, const int64_t *seeds, const int32_t *num_cav, void *stream);
/* The checks of mm_reset_seeded for n_envs envs of a handle with config cfg, alone: pure host code, no device. */
int mm_check_seeds(const mm_config *cfg, int n_envs, const int64_t *seeds, const int32_t *num_cav);

/* Episode records of the reference's evaluation protocol (MAPPO.evaluation, marl/mappo.py:255-361; evaluation.evaluation)
 * kept on the device.  mm_eval_record(env, rec, t) runs after the t-th mm_step(auto_reset = 0) of an evaluation and, for
 * every env whose active byte is still set: stores the global reward at rewards[e][t]; adds info["average_speed"] and
 * info["traffic_speed"] (as float64, in step order) to avg_speed_sum / traffic_speed_sum; keeps the minimum of
 * info["min_headway"] in min_headway (a value replaces it only when smaller); counts steps; with vehicle_speed /
 * vehicle_position set, stores speed and x of slots 0..n_agents[e]-1 at [e][t][slot] (float64); and when done is set,
 * records merge_percent and crashed (any of the first n_agents[e] vehicles crashed) and clears active.  n_agents is the
 * agent count at reset (the caller copies mm_buffers.n_agents after the reset).  The caller initialises the records:
 * active 1, sums and steps 0, min_headway +inf.  All pointers are DEVICE pointers, enqueued on `stream`.  Checked before
 * any CUDA call (MM_ERR_ARG): null env / records / required pointers, T >= 1, 0 <= t < T. */
typedef struct {
    int32_t T;                          /* step capacity of rewards / vehicle_speed / vehicle_position */
    const int32_t *n_agents;            /* [n_envs] agents at reset */
    uint8_t *active;                    /* [n_envs] 1 until the episode's first done */
    float *rewards;                     /* [n_envs][T] */
    int32_t *steps;                     /* [n_envs] */
    double *avg_speed_sum, *traffic_speed_sum;   /* [n_envs] */
    float *min_headway;                 /* [n_envs] */
    float *merge_percent;               /* [n_envs] written at done */
    uint8_t *crashed;                   /* [n_envs] written at done */
    double *vehicle_speed, *vehicle_position;    /* nullable, [n_envs][T][MM_MAXV] */
} mm_eval_records;
int mm_eval_record(mm_env *env, const mm_eval_records *rec, int t, void *stream);

/* Shield activity and control profiles of the evaluation's episodes (MDPLCVehicle.log_step, safe_controller.py:187-227:
 * state_hist / action_hist with safe_diff and safe_status), reduced on the device from the per-sub-step shield record of
 * a handle created with record_diag.  mm_eval_shield_record(env, rec, t) runs after the t-th mm_step(auto_reset = 0) and
 * BEFORE mm_eval_record(t) (which clears active at done, so the terminal step is still counted), on every env whose
 * active byte is set (`active` / `n_agents` are those of the mm_eval_records).  It visits sub-step s = 0, 1, 2 and, in
 * each, vehicle slot i = 0..MM_MAXV-1, and where the shield ran (ran[e][s][i]) adds 1 to shield_solves, to shield_active
 * when active != 0, to lane_change_vetoes when is_lc_safe == 0 (the counting rules of mm_stats), to shield_interventions
 * when safe_acc != nom_acc or safe_steer != nom_steer; adds |safe_acc - nom_acc| (the float64 difference, then its
 * absolute value: safe_diff["acceleration"]) to acc_correction_sum in that order; and keeps the running maxima of
 * |safe_acc - nom_acc| and |safe_steer - nom_steer|.  Where a vehicle moved (moved[e][s][i]) and i < n_agents[e], it keeps
 * the minimum applied acceleration (safe_acc) in min_agent_acc.  The caller initialises the records: counters, sum and
 * maxima 0, min_agent_acc +inf.
 * Control profiles: profile_slot (nullable, [n_envs]) maps an env to a profile row k >= 0, or -1 for none; a selected
 * env copies its three sub-step rows of each non-null profile_* array, [K][3 T][MM_MAXV] at row 3 t + s, verbatim from
 * the shield record while it is active (rows after its episode keep what the caller wrote).  k is not checked: the
 * caller builds the map.  All pointers are DEVICE pointers, enqueued on `stream`.  Checked before any CUDA call:
 * MM_ERR_ARG for null records / env / required pointers, T < 1 or t outside [0, T); MM_ERR_STATE for a handle created
 * without record_diag. */
typedef struct {
    int32_t T;                          /* row capacity of the profiles: 3 T rows per profile */
    const int32_t *n_agents;            /* [n_envs] agents at reset */
    const uint8_t *active;              /* [n_envs] the active bytes of the mm_eval_records */
    int32_t *shield_solves, *shield_active, *lane_change_vetoes, *shield_interventions;     /* [n_envs] */
    double *acc_correction_sum, *acc_correction_max, *steer_correction_max, *min_agent_acc;  /* [n_envs] */
    const int32_t *profile_slot;        /* nullable, [n_envs]: -1 or the profile row k */
    /* nullable, [K][3 T][MM_MAXV] each: the planes of mm_shield_diag_host of the same names */
    int32_t *profile_moved, *profile_ran, *profile_active, *profile_is_lc_safe, *profile_hl_action, *profile_lane;
    double *profile_x, *profile_y, *profile_heading, *profile_speed, *profile_min_headway, *profile_safe_acc,
           *profile_safe_steer, *profile_nom_acc, *profile_nom_steer;
} mm_eval_shield_records;
int mm_eval_shield_record(mm_env *env, const mm_eval_shield_records *rec, int t, void *stream);

/* MergeEnv.step (merge_env_v1.py:126-166): actions_dev is [n_envs][MM_MAXV] int8 on the device
 * (NULL: use mm_buffers.actions).  auto_reset != 0 re-spawns finished envs after their outputs are written
 * (the obs of a finished env is then the first obs of its next episode, as MAPPO.interact does, mappo.py:133-135). */
int mm_step(mm_env *env, const int8_t *actions_dev, int auto_reset, void *stream);

/* Same step through HOST buffers (pinned or pageable): copies actions in, steps, copies obs/reward/done out,
 * chunked over internal streams so copies overlap compute.  Any output pointer may be NULL. */
int mm_step_host(mm_env *env, const int8_t *actions, int auto_reset, float *obs, float *reward, uint8_t *done,
                 float *regional_rewards, int32_t *n_agents);

/* mm_step_host with the observations as the reference returns them (obs ndarray [A, n_s] per env,
 * merge_env_v1.py:126-166): only the rows of the agents that exist.  Env e's rows are
 * obs_rows[row_offset[e] * 30 .. (row_offset[e] + n_agents[e]) * 30); offsets are absolute, increasing, and dense inside
 * every chunk of the call (half a wave of the step kernel, 28 416 envs on a 148-SM part; chunk c starts at row chunk_first_env * MM_MAXV; row_offset[n_envs] = n_envs * MM_MAXV).
 * obs_rows has room for n_envs * MM_MAXV rows of 30 f32 (pinned memory for full PCIe speed); only the packed rows are
 * transferred: a quarter fewer bytes at hard density.  row_offset [n_envs + 1] int64 host; the other outputs as in
 * mm_step_host (nullable). */
int mm_step_host_ragged(mm_env *env, const int8_t *actions, int auto_reset, float *obs_rows, int64_t *row_offset,
                        float *reward, uint8_t *done, float *regional_rewards, int32_t *n_agents);
/* The same step with the observation in PACKED form: instead of the [A, 30] rows, what they are a function of.
 *   veh     [sum n_veh][MM_VEH_F32] f32   x, y, heading, speed of every vehicle, envs in order, slots in order (CAVs first)
 *   nbr     [sum n_agents] u16   per agent: the slots of the (up to) 4 other vehicles its observation shows, 4 bits each in
 *                                row order (close_vehicles_to(count = 4), road.py:257-267), 0xF = that row is empty
 *   n_veh, n_agents [n_envs] u8  the counts; all offsets are their running sums (dense from the first env to the last)
 *   reward [n_envs] f32, done [n_envs] u8, regional_rewards [n_envs][MM_MAXV] f32 as in mm_step_host (nullable)
 * About 215 bytes per env-step at hard density against 1.1 KB for the packed rows of mm_step_host_ragged: the host path
 * is bound by PCIe and host memory, not by the kernels.  Row i of env e is rebuilt by mm_expand_obs_rows:
 * ego columns from veh[i] (vx, vy = speed * cos / sin(heading), kinematics.py:215-217), row k + 1 from veh[slot k of nbr]
 * - veh[i] (observation.py:241-273, 181-193); inputs are float32, so the rebuilt rows agree with mm_step_host's to ~2e-7 (float32 rounding of positions up to 450 m mapped onto
 * [-1, 1]), inside the 1e-4 tolerance of the path.  With auto_reset the packed state of a finished env is that of its next
 * episode (like obs), reward / done / regional_rewards describe the finished step.  veh needs room for n_envs * 11 rows,
 * nbr for n_envs * MM_MAXV entries (pinned memory for full PCIe speed). */
typedef struct {
    float *veh;
    uint16_t *nbr;
    uint8_t *n_veh, *n_agents;
    float *reward;
    uint8_t *done;
    float *regional_rewards;
} mm_packed_host;
int mm_step_host_packed(mm_env *env, const int8_t *actions, int auto_reset, const mm_packed_host *out);
/* Pure host function (no device): obs_rows [sum n_agents][30] f32 and row_offset [n_envs + 1] from a packed step, on
 * n_threads host threads.  steer_vel: the config's lateral_control == "steer_vel" (neighbour CAV headings relative). */
int mm_expand_obs_rows(const mm_packed_host *in, int n_envs, int steer_vel, float *obs_rows, int64_t *row_offset, int n_threads);
int mm_buffers_get(mm_env *env, mm_buffers *out);
int mm_get_state(mm_env *env, mm_state_host *dst);        /* synchronous */
int mm_set_state(mm_env *env, const mm_state_host *src);  /* synchronous; also refreshes obs / n_agents */
int mm_get_shield_diag(mm_env *env, mm_shield_diag_host *dst);   /* requires record_diag */
int mm_stats(mm_env *env, mm_stats_t *out, int reset);    /* synchronous */

/* The shield alone: safety_layer(safety_type, action, vehicle, dt, ...) (highway_env/vehicle/safety/decentral_layer.py:
 * 767-817, as MDPLCVehicle.step calls it through get_safe_action, safe_controller.py:229-250) for every CAV of the current
 * scenes, against the scenes as they are - the view the front-most vehicle of a sub-step has; nothing is stepped and no
 * state is written (the reference's side effects on the vehicle - is_collaborating, is_lc_safe, target_lane_index,
 * min_headway, the on-ramp HDV record shift - are returned / kept local instead).  Inputs: the clipped low-level action
 * per CAV, nom_steer / nom_acc [n_envs][MM_MAXV] f64 DEVICE.  Outputs [n_envs][MM_MAXV], DEVICE: the shielded action,
 * the time headway the shield computed, and the status the reference logs: whether the shield ran (its gate: fg_params
 * set and two history records), the neighbour classification of multi_agent_state (slot ids, MM_NB_NONE, MM_NB_OBSTACLE),
 * constrain_adj, the QP active set (MM_ACT_*), is_lc_safe. */
typedef struct {
    double *safe_steer, *safe_acc, *min_headway;
    int32_t *ran, *leader, *front_adj, *rear_adj, *constrain_adj, *active, *is_lc_safe;
} mm_shield_query_out;
int mm_shield_query(mm_env *env, const double *nom_steer, const double *nom_acc, const mm_shield_query_out *out, void *stream);

/* The CBF-QP alone (cbf.py:110-161 through cvxopt.solvers.qp): n independent solves on DEVICE arrays;
 * u and active may alias nothing else.  Used for the solves/s microbenchmark and the QP known-answer tests. */
int mm_shield_qp(const double *a, const double *c_lead, const double *c_adj, const uint8_t *has_adj,
                 const double *lo, const double *hi, int64_t n, double *u, uint8_t *active, void *stream);

/* Caller side of the path (SURVEY.md 8f rank 1, BASELINE configs[3]: policy + env on the device).
 *
 * mm_actor_sample: the shared MAPPO actor (marl/single_agent/Model_common.py:5-23: Linear 30-128, ReLU, Linear 128-128,
 * ReLU, Linear 128-5, log-softmax) evaluated on n_rows observation rows [n_rows][30] f32 and, fused with it, the
 * exploration draw of marl/mappo.py:209-228 (np.random.choice(p = softmax): inverse CDF of one uniform per row;
 * here Philox4x32-10 keyed by (seed, step, row)).  Weights are torch.nn.Linear parameters as they lie in memory
 * (weight [out][in], bias [out]), TF32 tensor-core math with fp32 accumulation: the two 128-wide layers run as
 * tcgen05.mma kind::tf32 with the accumulators in TMEM (one persistent CTA per SM, 128 rows per tile), the 128 -> 5
 * output layer, the log-softmax and the draw in the thread that owns the row.  n_agents (nullable) [n_rows / 12]:
 * rows whose slot index (row % 12) is >= n_agents[row / 12] get action 1 (IDLE).  action_mask (nullable) [n_rows] u8,
 * bit k = action k available (the env's action_mask buffer): the invalid-action masking of the MAPPO_GI actor
 * (marl/single_agent/Model_gi.py:63-66, logits of unavailable actions = -1e8 before the log-softmax).  logp_all [n_rows][5] and
 * logp_sel [n_rows] are optional outputs (log-probabilities of all actions / of the drawn one).  All pointers are
 * DEVICE pointers; enqueued on `stream`, no synchronisation. */
int mm_actor_sample(const float *obs, const int32_t *n_agents, int64_t n_rows, const float *w1, const float *b1,
                    const float *w2, const float *b2, const float *w3, const float *b3, uint64_t seed, uint64_t step,
                    const uint8_t *action_mask, int8_t *actions, float *logp_all, float *logp_sel, void *stream);

/* The same fused forward + draw for a 30 - h1 - 128 - 5 network, fp16 tensor-core operands with fp32 accumulation:
 * h1 = 128 is the MAPPO actor above; h1 = 160 is the shared-trunk network of MAPPO_GI with state_split
 * (marl/single_agent/Model_gi.py:137-220): its three first-layer blocks fc11 / fc12 / fc13 over fixed column lists are
 * one 30 -> 160 layer whose weight w1 [160][30] is zero outside the blocks (the caller scatters them; b1 = the three
 * biases concatenated), w2 = fc2.weight [128][160], w3 / b3 = actor_linear.  value_w [128] / value_b [1] (nullable) =
 * critic_linear: values [n_rows] receives V(s) from the same hidden activations (the bootstrap value of
 * mappo_gi.py:396-404).  Rollout-buffer appends of MAPPO.interact (mappo.py:117-131), fused: obs_copy (nullable)
 * [n_rows][30] receives the rows the actions were drawn from (point it at slot t of the state buffer), live_out (nullable)
 * [n_rows] u8 = 1 where the row belongs to an agent that exists (needs n_agents), and `actions` can be slot t of the
 * action buffer.  Everything else as in mm_actor_sample. */
int mm_actor_sample_mlp(const float *obs, const int32_t *n_agents, int64_t n_rows, int h1, const float *w1, const float *b1,
                        const float *w2, const float *b2, const float *w3, const float *b3, const float *value_w,
                        const float *value_b, uint64_t seed, uint64_t step, const uint8_t *action_mask, int8_t *actions,
                        float *logp_all, float *logp_sel, float *values, float *obs_copy, uint8_t *live_out, void *stream);

/* Implementation switch of mm_actor_sample (process-wide): 0 = tcgen05 with fp16 operands, one warpgroup per 128-row
 * tile and the weights once per SM (default, the kernel of mm_actor_sample_mlp); 1 = the warp-level mma.sync TF32 kernel
 * kept as an independent cross-check.  Any other value: MM_ERR_ARG, the switch unchanged. */
int mm_set_actor_impl(int impl);

/* mm_discounted_returns: MAPPO._discount_reward (marl/mappo.py:364-370) for every (env, agent) column of a rollout at
 * once: out[t][c] = rewards[t][c] + gamma * out[t+1][c], restarted after a step with dones[t][c / cols_per_env] != 0,
 * seeded after the last step with final_value[c] (nullable: 0).  rewards / out [T][n_cols] f32, dones
 * [T][n_cols / cols_per_env] u8, DEVICE pointers. */
int mm_discounted_returns(const float *rewards, const uint8_t *dones, const float *final_value, float gamma, int T,
                          int64_t n_cols, int cols_per_env, float *out, void *stream);

/* mm_lambda_returns: the lambda-return (GAE(lambda) return) of every (env, agent) column of a rollout, in the same kernel as
 * mm_discounted_returns.  Per column, from t = T - 1 down to 0, with run = v_next = final_value[c] (nullable: 0):
 *   if dones[t][c / cols_per_env]: run = v_next = 0
 *   run = (lambda * run + (1 - lambda) * v_next) * gamma + rewards[t][c];  out[t][c] = run;  v_next = values[t][c]
 * each product and sum rounded to float32 separately (never fused).  values [T][n_cols] f32 = V(s_t) of the networks that
 * collected the rollout; nullable when lambda == 1, which gives mm_discounted_returns' output bit for bit (with values as
 * well, as long as they are finite where they are read; up to the sign of a zero).  values[t][c] is read only where step
 * t - 1 did not end the episode.  lambda = 0 gives the one-step targets r_t + gamma (1 - d_t) V(s_{t+1}).  DEVICE
 * pointers; arguments are checked before any CUDA call (MM_ERR_ARG): rewards, dones and out required, 0 <= lambda <= 1,
 * finite gamma, values required when lambda < 1, the rollout shape as for mm_discounted_returns. */
int mm_lambda_returns(const float *rewards, const uint8_t *dones, const float *values, const float *final_value, float gamma,
                      float lambda, int T, int64_t n_cols, int cols_per_env, float *out, void *stream);

/* On-device PPO learner: the networks of one MAPPO / MAPPO_GI update with the per-sample PPO-clip surrogate and the MSE
 * value loss (marl/mappo.py:161-206, marl/mappo_gi.py:307-349; rollout.mappo_losses / shared_network_loss with
 * pairwise=False, critic_loss="mse").  Network kinds, parameters as torch.nn.Linear lays them out (weight [out][in]):
 *   MM_PPO_ACTOR   ActorNetwork 30-128-128-5, log-softmax: w1..b3 = fc1..fc3
 *   MM_PPO_CRITIC  CriticNetwork: w1 / b1 = fc1 (30 -> 128), w2 / b2 = fc2 ([h1, one_hot(a)] 133 -> 128), w3 / b3 = fc3 (-> 1)
 *   MM_PPO_SHARED  ActorCriticNetwork with state_split, hidden 128: w1 [160][30] / b1 [160] = fc11 / fc12 / fc13 as one dense
 *                  layer, zero outside the blocks (as for mm_actor_sample_mlp), w2 / b2 = fc2, w3 / b3 = actor_linear,
 *                  w4 [128] / b4 [1] = critic_linear
 * w4 / b4 are used by MM_PPO_SHARED only.  Rows: states [rows][30] f32, actions [rows] int8 (0..4) and returns [rows] f32
 * are the rollout buffer as collected; idx [n] int64 lists the rows of the pass in any order.  DEVICE pointers, enqueued on
 * `stream`, no allocation after the first call on a device and no synchronisation.  Arguments are checked before any
 * CUDA call (MM_ERR_ARG): kind, required pointers, n >= 1, 0 < clip < 1. */
enum { MM_PPO_ACTOR = 0, MM_PPO_CRITIC = 1, MM_PPO_SHARED = 2 };
typedef struct { const float *w1, *b1, *w2, *b2, *w3, *b3, *w4, *b4; } mm_ppo_net;
typedef struct { float *w1, *b1, *w2, *b2, *w3, *b3, *w4, *b4; } mm_ppo_grads_out;

/* Target pass (forward only), once per update with the TARGET networks: for every listed row, old_logp[row] = log p(a)
 * (MM_PPO_ACTOR, MM_PPO_SHARED) or q_target[row] = Q(s, one_hot(a)) (MM_PPO_CRITIC); outputs are indexed like states.
 * MM_PPO_SHARED with a non-null q_target also writes q_target[row] = V(s) from the same forward (the values of the
 * rollout for mm_lambda_returns); MM_PPO_ACTOR ignores q_target.  Rows not listed are not written.  Replaces the no-grad half of MAPPO.train (mappo.py:170-183) and MAPPO_GI.train (mappo_gi.py:307-320), which torch
 * recomputes for every minibatch. */
int mm_ppo_targets(int kind, const float *states, const int8_t *actions, const int64_t *idx, int64_t n, const mm_ppo_net *net,
                   float *old_logp, float *q_target, void *stream);

/* Gradient pass, once per minibatch: the gradients of the mean loss over the n listed rows, written (not accumulated) into
 * `grads` in the parameters' layout (MM_PPO_SHARED: w1 in the dense [160][30] layout), and the mean losses into losses[0]
 * (PPO surrogate: MM_PPO_ACTOR, MM_PPO_SHARED) / losses[1] (value MSE: MM_PPO_CRITIC, MM_PPO_SHARED); the other slot is
 * left as it is.  Advantage: returns - q_target (MM_PPO_ACTOR, q_target from the critic's target pass) or returns - V(s)
 * (MM_PPO_SHARED, V detached).  old_logp from the target pass; ratio r = exp(log p(a) - old_logp), and since both passes
 * run the same forward arithmetic r == 1 exactly while a network equals its target.  The per-row derivative follows
 * torch autograd: min splits the gradient half / half at a tie, clamp passes it at its bounds.  Deterministic: each CTA
 * sums its tiles, a second kernel adds the CTA partials in a fixed order (two calls with equal inputs give bit-identical
 * gradients); the partials workspace is allocated once per device and shared by the calls on that device, which must
 * therefore be ordered (one stream).  Replaces actor_loss.backward() / critic_loss.backward() of MAPPO.train and
 * loss.backward() of MAPPO_GI.train. */
int mm_ppo_grads(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                 const float *q_target, const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net,
                 const mm_ppo_grads_out *grads, float *losses, void *stream);

/* Statistics pass (forward only, the same forward arithmetic as the target and gradient passes): the standard PPO
 * diagnostics of one network over the n listed rows, reduced into stats[MM_PPO_STATS_LEN] (f64, DEVICE pointer), written
 * (not accumulated).  Per row, in f32 as the passes compute it:
 *   ACTOR, SHARED  the entropy -sum_k p_k log p_k of the log-softmax (ENTROPY); with old_logp (nullable) the ratio
 *                  r = exp(logp(a) - old_logp), k3 = (r - 1) - (logp(a) - old_logp) (K3), |r - 1| > clip (CLIPPED) and the
 *                  range of r (RATIO_MIN, RATIO_MAX)
 *   CRITIC, SHARED the value v = Q(s, one_hot(a)) (CRITIC) or V(s) (SHARED) against the return G: v, v^2, G, G^2 and
 *                  (G - v)^2 (V, V2, G, G2, RES2; v^2, G^2 and (G - v)^2 squared in f64)
 * N counts the rows.  Sums and counts combine across data-parallel shards with SUM, RATIO_MIN with MIN and RATIO_MAX with
 * MAX.  Fields a kind has no term for are 0; where no ratio is formed (CRITIC, old_logp null, n = 0) RATIO_MIN = +inf and
 * RATIO_MAX = -inf.  n = 0 (an empty shard) writes that empty value.  Deterministic: each thread sums its rows in f64 in a
 * fixed order, each CTA writes one partial per field, a second kernel adds them in CTA order; no float atomics.  The
 * partials share mm_ppo_grads' workspace, so calls on one device must be ordered with it (one stream).  Arguments are
 * checked before any CUDA call (MM_ERR_ARG): kind, net, n >= 0, stats, and for n > 0 states, actions, idx and returns
 * (CRITIC, SHARED); 0 < clip < 1 when old_logp is given. */
enum { MM_PPO_STAT_N, MM_PPO_STAT_ENTROPY, MM_PPO_STAT_K3, MM_PPO_STAT_CLIPPED, MM_PPO_STAT_RATIO_MIN,
       MM_PPO_STAT_RATIO_MAX, MM_PPO_STAT_V, MM_PPO_STAT_V2, MM_PPO_STAT_G, MM_PPO_STAT_G2, MM_PPO_STAT_RES2,
       MM_PPO_STATS_LEN };
int mm_ppo_stats(int kind, const float *states, const int8_t *actions, const float *returns, const float *old_logp,
                 const int64_t *idx, int64_t n, float clip, const mm_ppo_net *net, double *stats, void *stream);

/* Optimiser step of the learner on the device: for each group (one network), torch.nn.utils.clip_grad_norm_(params,
 * max_norm) followed by torch.optim.RMSprop(lr, alpha, eps).step() without momentum, centring or weight decay
 * (marl/mappo.py:88-90, marl/mappo_gi.py:150-156), in one launch with one CTA per group.  Per group:
 *   g = grad * grad_scale                      (the data-parallel average: grad_scale = 1.0f / world, the float reciprocal
 *                                               that torch multiplies by for `grad /= world` on a CUDA tensor)
 *   total = ||g||_2 over every tensor of the group, summed in a fixed order (optim.cu; deterministic)
 *   coef = min(1, (1 / (total + 1e-6)) * max_norm), or 1 when max_norm <= 0 (no clipping); g *= coef, written to grad
 *   square_avg = square_avg * alpha; square_avg = square_avg + (one_minus_alpha * g) * g
 *   param = param + (-lr) * (g / (sqrt(square_avg) + eps))
 * each operation rounded on its own, as torch's single-tensor and foreach RMSprop order them.  total (before clipping,
 * what clip_grad_norm_ returns) goes to total_norm when it is not null.  param, grad, square_avg [numel] f32 and
 * total_norm, mirror are DEVICE pointers; the tables and mirror_cols are HOST memory, read before the call returns.
 * Mirror (nullable): the kernel also stores every updated param element i, as (r, c) = (i / mirror_ncols,
 * i % mirror_ncols), at mirror[r * mirror_ld + mirror_cols[c]]: the dense 30 -> 160 first layer of the shared network
 * (fc11 / fc12 / fc13 at their rows and columns) stays equal to its blocks without a rebuild.  Arguments are checked
 * before any CUDA call (MM_ERR_ARG): null pointers, 1 <= n_groups <= MM_OPT_MAX_GROUPS, 1 <= n_tensors <=
 * MM_OPT_MAX_TENSORS, numel >= 0, and a mirror needs mirror_cols with 1..MM_OPT_MAX_MIRROR_COLS entries in
 * [0, min(mirror_ld, 256)) and a numel that is a multiple of mirror_ncols. */
#define MM_OPT_MAX_GROUPS 8
#define MM_OPT_MAX_TENSORS 16
#define MM_OPT_MAX_MIRROR_COLS 16
typedef struct {
    float *param, *grad, *square_avg;
    int64_t numel;
    float *mirror;
    const int32_t *mirror_cols;
    int32_t mirror_ncols;
    int64_t mirror_ld;
} mm_opt_tensor;
typedef struct {
    const mm_opt_tensor *tensors;
    int32_t n_tensors;
    float lr, alpha, one_minus_alpha, eps, max_norm, grad_scale;
    float *total_norm;
} mm_opt_group;
int mm_rmsprop_step(const mm_opt_group *groups, int n_groups, void *stream);

/* The step kernel (the physics of a policy step) exists in several builds of one source: generic for 3 CTAs per SM
 * (6 staged fields, 168 registers; the faster one per unit of work), generic for 4 CTAs per SM (4 staged fields, 128
 * registers), and two builds specialised at compile time for all-CAV envs of env id merge-multi-agent-v1 with
 * lateral_control "steer" under the MASS / the HSS shield (no IDM / MOBIL code, configuration reads folded to constants).
 * A fifth build maps half a warp to an env and a lane to a vehicle (the warp-cooperative build, merge_coop.cu) for
 * batches too small to fill the machine with one thread per env.
 * 0 (default): automatic - for all-CAV envs of the plain LC env the warp-cooperative build up to 12 288 envs and a
 * specialised build above (when none of the handle's envs can hold an HDV: spawned under traffic_type cav, or checked by
 * mm_set_state); the 4-CTA build for small grids whose wave structure
 * favours it (e.g. 65 536 envs = 512 CTAs on 148 SMs: one wave instead of a full and an almost empty one, -27 % step
 * time).  3 / 4: force a generic build; 5: automatic among the generic builds only; 6: 4 CTAs per SM forced, specialised
 * builds allowed; 7: the warp-cooperative build forced where it applies; 8: automatic among the one-thread-per-env builds
 * (process-wide; tests and A/B timing). */
int mm_set_step_variant(int variant);
enum { MM_BUILD_GENERIC3 = 3, MM_BUILD_GENERIC4 = 4, MM_BUILD_SPEC_HSS = 31, MM_BUILD_SPEC_MASS = 32,
       MM_BUILD_SPEC_HSS4 = 41, MM_BUILD_SPEC_MASS4 = 42 /* specialised and built for 4 CTAs per SM */,
       MM_BUILD_COOP = 50 /* + shield kind: the warp-cooperative build (half a warp per env) */ };
/* which build the handle's last mm_step / mm_step_host* launched (0 before the first step) */
int mm_step_build(const mm_env *env);

/* The baseline supervisors of safety_guarantee = priority | dmc (highway_env/vehicle/safety/central_layer.py:16-178,
 * decentralised_dmc.py:70-198; called from AbstractEnv.step before _simulate, abstract.py:459-467).  With
 * mm_config.supervisor set, mm_step / mm_step_host* run them on every policy step: the supervised tuples land in
 * mm_buffers.new_actions and are what the step executes.  The reference draws np.random.rand() numbers for them (one per
 * CAV for the priority tie-break, then two per IDM decision of the look-ahead); the batched path draws from
 * Philox4x32-10 keyed (seed, env, episode, policy step).  For teacher forcing and for the seed-exact single-env adapter
 * the caller can supply the draws: mm_set_supervisor_draws(draws_dev [n_envs][MM_SUPERVISOR_DRAWS] f64 DEVICE, consumed in
 * order; NULL returns to Philox) applies to every following step until changed, and mm_supervisor_draws_used copies to
 * the host how many draws each env consumed in the last step (the adapter advances its MT19937 replay by that).
 *
 * mm_supervise is the supervisor alone: rewrites actions [n_envs][MM_MAXV] int8 DEVICE in place for the current scenes;
 * kind 0 = priority, 1 = dmc; draws_dev as above (NULL: Philox); n_used_dev (nullable) [n_envs] int32 DEVICE.  It returns
 * the reference's tuples on every step of the reference fixtures (tests/test_zz_supervisor_gpu.py). */
#define MM_SUPERVISOR_DRAWS 32
int mm_supervise(mm_env *env, int kind, int8_t *actions_dev, const double *draws_dev, int32_t *n_used_dev, void *stream);
int mm_set_supervisor_draws(mm_env *env, const double *draws_dev);
int mm_supervisor_draws_used(mm_env *env, int32_t *n_used_host);

/* Launch bookkeeping for bench.py ("gpu_launches") */
int64_t mm_kernel_launches(const mm_env *env);
const char *mm_last_error(void);
const char *mm_version(void);

#ifdef __cplusplus
}
#endif
#endif

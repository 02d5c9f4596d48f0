/*
 * kin_b200.h -- C ABI of the B200-native kinematic env rollout (libkin_b200.so).
 *
 * Drop-in boundary for the hot path of jerry102102102/RL_brain_trainer's kinematic
 * Approach -> Finisher stack.  The reference has no FFI: its boundary is the Gymnasium-style
 * Python class `ArmKinematicEnv` (hrl_ws/src/hrl_trainer/hrl_trainer/kinematic_phase1/envs/
 * arm_kinematic_env.py:69-365, below "AKE") plus the eval orchestrators that loop over it.
 * Each entry point here states which reference call it replaces.  The Python host side
 * (rl_brain_trainer_b200/env.py) binds these with ctypes and mirrors the reference's class API.
 *
 * Conventions
 *  - plain C, no torch types; every pointer is a DEVICE pointer unless named host_*.
 *  - the caller owns every buffer; no hidden allocation, no hidden synchronisation.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *  - return value: 0 = KIN_OK, otherwise a KIN_ERR_* code; kin_last_error_string() explains
 *    (thread-local).  Functions are thread-compatible, not thread-safe per handle.
 *  - all arithmetic is fp32 on the device (the reference is fp64 on the CPU and casts the
 *    observation to fp32); counters are integers, flags are bits.
 *
 * The python binding parses the structs in this header (one field per line:
 * `float name;`, `float name[N];`, `int name;`), so the header is the single source of truth.
 */
#ifndef KIN_B200_H
#define KIN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KIN_ABI_VERSION 4
#define KIN_NJ 7
#define KIN_OBS_DIM 56
#define KIN_ROUTE_OBS_DIM 80
#define KIN_MAX_MILESTONES 4
#define KIN_MAX_STAGES 16
#define KIN_MAX_COMPONENTS 64

#define KIN_OK 0
#define KIN_ERR_INVALID_ARG 1
#define KIN_ERR_CUDA 2
#define KIN_ERR_NO_DEVICE 3
#define KIN_ERR_UNSUPPORTED 4

/* policy mode == index of the one-hot in obs["mode_flag"] (AKE:544-551) */
#define KIN_MODE_APPROACH 0
#define KIN_MODE_DOCK 1
/* kernel specialisation hint: every env in the batch is in this mode, or per-env (read from flags) */
#define KIN_MODE_PER_ENV (-1)

/* ---- per-env state: struct-of-arrays, one 32-bit word per row, env index fastest -----------
 * state[row * stride + env]; stride >= n, stride % 32 == 0.  Rows (== private fields of AKE:80-100):   */
#define KIN_ROW_Q 0            /* 7  joint positions                                              */
#define KIN_ROW_DQ 7           /* 7  last executed joint delta                                    */
#define KIN_ROW_PREV_ACTION 14 /* 7  last (clipped) action                                        */
#define KIN_ROW_GOAL_POSE 21   /* 6  goal [x y z roll pitch yaw]                                  */
#define KIN_ROW_EE_POSE 27     /* 6  cached FK(q)                                                 */
#define KIN_ROW_MIN_POS 33     /* 1  running min position error                                   */
#define KIN_ROW_CNT0 34        /* 1  u32: episode_step | dwell_count << 16                        */
#define KIN_ROW_CNT1 35        /* 1  u32: near_goal_entry_count | near_goal_drift_count << 16     */
#define KIN_ROW_FLAGS 36       /* 1  u32: KIN_FLAG_* bits                                         */
#define KIN_ROW_ENTRY 37       /* 4  entry pos err, ori err, action l2, dq norm (dock reward)     */
#define KIN_ROW_GOAL_Q 41      /* 7  goal joint vector (info only; the step never reads it)       */
#define KIN_ROW_EPISODE 48     /* 1  u32: episodes completed by this slot (auto-reset RNG counter)*/
#define KIN_ROW_ROUTE 49       /* 1  u32: route_index | ready_streak << 16 (route wrappers)       */
#define KIN_ROW_ROUTE2 50      /* 1  u32: last_route_index | completed_waypoints << 16 (sequence) */
#define KIN_STATE_ROWS 64

#define KIN_FLAG_PRE_NEAR_HIT 0x1u
#define KIN_FLAG_NEAR_HIT 0x2u
#define KIN_FLAG_MODE_SHIFT 4 /* 2 bits */
#define KIN_FLAG_STAGE_SHIFT 8 /* 4 bits: curriculum stage the episode was sampled from */

/* ---- per-step result byte (done[env]) ------------------------------------------------------ */
#define KIN_DONE_TERMINATED 0x1u
#define KIN_DONE_TRUNCATED 0x2u
#define KIN_DONE_SUCCESS 0x4u
#define KIN_DONE_PRE_NEAR 0x8u      /* info["curr_in_pre_near_goal"] */
#define KIN_DONE_NEAR 0x10u         /* info["curr_in_near_goal"]     */
#define KIN_DONE_REASON_SHIFT 5     /* 2 bits: 0 running, 1 success, 2 max_steps, 3 invalid_state */
#define KIN_DONE_AUTORESET 0x80u    /* slot was re-seeded in this call (obs is the new episode's) */

/* ---- optional per-step scalars: aux[row * stride + env] (AKE:353-364 info keys) ------------- */
#define KIN_AUX_POS_ERR 0         /* position_error_norm    */
#define KIN_AUX_ORI_ERR 1         /* orientation_error_norm */
#define KIN_AUX_ACTION_L2 2       /* action_l2              */
#define KIN_AUX_DQ_L2 3           /* executed_delta_q_l2    */
#define KIN_AUX_DQ_CHANGE_L2 4    /* delta_q_change_l2      */
#define KIN_AUX_DOCK_LIMIT 5      /* dock_action_limit      */
#define KIN_AUX_DQC_SCALE 6       /* dock_delta_q_change_limit_scale */
#define KIN_AUX_MARGIN_MIN 7      /* joint_limit_margin_min */
#define KIN_AUX_ROWS 8

/* Flattened Phase1EnvConfig (AKE:32-66) + the precomputed FK chain.  Field names follow the
 * reference's config keys: ar_* = ApproachRewardConfig (reward_approach.py:13-72),
 * dr_* = DockRewardConfig (reward_dock.py:13-102), term_* = TerminationConfig
 * (termination.py:11-17), obs_* = ObservationBuilderConfig (observation_builder.py:18-21),
 * rr_* = RouteRewardConfig (route/reward_route.py:14-33).                                     */
typedef struct KinEnvParams {
    /* joint specs (kinematics/joint_limits.py:37-47) */
    float joint_lower[7];
    float joint_upper[7];
    float joint_delta_limit[7];
    /* FK chain of v5_1/ee_fk.py:98-134 with the constant transforms pre-multiplied on the host in
     * fp64 (rl_brain_trainer_b200/kinematics.py): p = fk_pbase + fk_pq0*q0; R = fk_C[0]*Rz(q1);
     * for j=2..6: p += R*fk_t[j-2]; R = R*fk_C[j-1]*Rz(qj);  R_ee = R*fk_AT                     */
    float fk_pbase[3];
    float fk_pq0[3];
    float fk_C[54];
    float fk_t[15];
    float fk_AT[9];
    /* derived on the host in fp64 (params.py) so the kernels multiply instead of divide:
     * 1/max(span,1e-9), 1/max(delta_limit,1e-9), 1/pos_err_scale, 1/ori_err_scale, 1/max(episode_length,1),
     * 1/max(dwell_steps_target,1)                                                                */
    float k_inv_span[7];
    float k_inv_delta_limit[7];
    float k_inv_pos_err_scale;
    float k_inv_ori_err_scale;
    float k_inv_episode_length;
    float k_inv_dwell_steps_target;
    /* env */
    float action_delta_scale;
    int dynamic_action_delta_scale_enabled;
    float dynamic_action_delta_scale_near_pos_threshold_m;
    float dynamic_action_delta_scale_far_pos_threshold_m;
    float dynamic_action_delta_scale_near_multiplier;
    float dynamic_action_delta_scale_far_multiplier;
    float dock_action_delta_scale;
    float dock_residual_action_limit;
    float dock_delta_q_change_limit_scale;
    float dock_dynamic_action_limit_near_pos_threshold_m;
    float dock_dynamic_action_limit_far_pos_threshold_m;
    float dock_dynamic_residual_action_limit_near;
    float dock_dynamic_residual_action_limit_far;
    float dock_dynamic_delta_q_change_limit_scale_near;
    float dock_dynamic_delta_q_change_limit_scale_far;
    int episode_length;
    int dwell_steps_target;
    /* termination */
    int term_max_episode_steps;
    float term_success_pos_threshold_m;
    float term_success_ori_threshold_rad;
    int term_success_dwell_steps;
    int term_require_orientation;
    int term_terminate_on_success;
    /* observation */
    float obs_pos_err_scale_m;
    float obs_ori_err_scale_rad;
    /* approach reward */
    float ar_position_progress_weight;
    float ar_orientation_progress_weight;
    float ar_near_field_orientation_progress_weight;
    float ar_pre_near_goal_pos_threshold_m;
    float ar_near_goal_pos_threshold_m;
    float ar_near_goal_ori_threshold_rad;
    float ar_coarse_orientation_bonus_threshold_rad;
    int ar_n_milestones;
    float ar_orientation_milestone_thresholds_rad[4];
    float ar_orientation_milestone_bonuses[4];
    float ar_near_field_orientation_center_weight;
    int ar_use_orientation_gate;
    float ar_pre_near_goal_bonus;
    float ar_near_goal_bonus;
    float ar_near_goal_bonus_decay;
    float ar_pre_near_to_near_progress_weight;
    float ar_coarse_orientation_bonus;
    float ar_handover_pos_threshold_m;
    float ar_handover_ori_threshold_rad;
    float ar_handover_bonus;
    float ar_handover_retention_bonus;
    float ar_handover_dwell_bonus;
    float ar_handover_leave_penalty;
    float ar_handover_regression_weight;
    float ar_handover_smoothness_multiplier;
    float ar_dock_coarse_ready_pos_threshold_m;
    float ar_dock_coarse_ready_ori_threshold_rad;
    float ar_dock_coarse_ready_action_threshold;
    float ar_dock_coarse_ready_dq_threshold;
    float ar_dock_coarse_ready_bonus;
    float ar_dock_coarse_ready_retention_bonus;
    float ar_dock_coarse_ready_dwell_bonus;
    float ar_dock_coarse_ready_leave_penalty;
    float ar_dock_coarse_ready_regression_weight;
    float ar_finisher_ready_pos_threshold_m;
    float ar_finisher_ready_ori_threshold_rad;
    float ar_finisher_ready_action_threshold;
    float ar_finisher_ready_dq_threshold;
    float ar_finisher_ready_bonus;
    float ar_finisher_ready_retention_bonus;
    float ar_finisher_ready_dwell_bonus;
    float ar_finisher_ready_leave_penalty;
    float ar_finisher_ready_regression_weight;
    float ar_near_handoff_pos_threshold_m;
    float ar_near_handoff_ori_threshold_rad;
    float ar_near_handoff_action_weight;
    float ar_near_handoff_dq_weight;
    float ar_near_handoff_motion_bonus_weight;
    float ar_near_handoff_settle_bonus_weight;
    float ar_same_step_alignment_bonus;
    float ar_dwell_bonus;
    float ar_drift_penalty_weight;
    int ar_drift_penalty_escalation_start;
    float ar_drift_penalty_escalation_per_count;
    float ar_near_goal_leave_penalty;
    float ar_action_magnitude_weight;
    float ar_action_delta_weight;
    float ar_joint_limit_penalty_weight;
    float ar_success_bonus;
    /* dock (Finisher) reward */
    float dr_position_progress_weight;
    float dr_orientation_progress_weight;
    float dr_stay_in_zone_bonus;
    float dr_dwell_bonus;
    float dr_leave_zone_penalty;
    float dr_working_range_bonus;
    float dr_working_range_dwell_bonus;
    int dr_working_range_dwell_start;
    float dr_working_range_exit_penalty;
    float dr_drift_penalty_position_weight;
    float dr_drift_penalty_orientation_weight;
    float dr_action_magnitude_weight;
    float dr_action_delta_weight;
    float dr_joint_limit_penalty_weight;
    float dr_success_bonus;
    float dr_tight_pose_pos_threshold_m;
    float dr_tight_pose_ori_threshold_rad;
    float dr_tight_pose_bonus;
    float dr_tight_pose_dwell_bonus;
    float dr_strict_pose_leave_penalty;
    float dr_strict_center_reward_weight;
    float dr_strict_center_position_weight;
    float dr_strict_center_orientation_weight;
    float dr_strict_center_small_action_bonus_weight;
    float dr_strict_center_small_action_pos_radius_m;
    float dr_strict_center_small_action_ori_radius_rad;
    float dr_strict_center_small_action_scale;
    float dr_strict_center_small_action_power;
    float dr_strict_center_dwell_bonus_weight;
    int dr_strict_center_dwell_start;
    int dr_strict_center_dwell_escalation_start;
    float dr_strict_center_dwell_escalation_per_step;
    float dr_strict_zone_drift_penalty_multiplier;
    float dr_strict_zone_action_penalty_multiplier;
    float dr_tight_position_shaping_radius_m;
    float dr_tight_position_shaping_weight;
    float dr_tight_orientation_shaping_radius_rad;
    float dr_tight_orientation_shaping_weight;
    float dr_convergence_position_radius_m;
    float dr_convergence_position_progress_weight;
    float dr_convergence_orientation_radius_rad;
    float dr_convergence_orientation_progress_weight;
    float dr_position_first_orientation_pos_threshold_m;
    float dr_position_first_orientation_pre_scale;
    float dr_action_delta_violation_threshold;
    float dr_action_delta_violation_weight;
    float dr_delta_q_change_penalty_threshold;
    float dr_delta_q_change_penalty_weight;
    float dr_entry_action_penalty_near_pos_threshold_m;
    float dr_entry_action_penalty_far_pos_threshold_m;
    float dr_entry_action_penalty_near_multiplier;
    float dr_entry_action_penalty_far_multiplier;
    float dr_basin_outer_radius_m;
    float dr_basin_inner_radius_m;
    float dr_basin_dwell_radius_m;
    float dr_basin_outer_bonus;
    float dr_basin_inner_bonus;
    float dr_basin_dwell_bonus;
    float dr_basin_outer_exit_penalty;
    float dr_basin_inner_exit_penalty;
    float dr_basin_dwell_break_penalty;
    float dr_basin_drift_penalty_weight;
    float dr_near_strict_pos_threshold_m;
    float dr_near_strict_ori_threshold_rad;
    float dr_preserve_state_bonus;
    float dr_preserve_position_tolerance_m;
    float dr_preserve_orientation_tolerance_rad;
    float dr_strict_hold_bonus;
    float dr_low_motion_bonus;
    float dr_low_motion_action_threshold;
    float dr_low_motion_dq_threshold;
    float dr_tiny_correction_bonus;
    float dr_tiny_correction_action_threshold;
    float dr_worse_than_entry_position_weight;
    float dr_worse_than_entry_orientation_weight;
    float dr_worse_than_entry_position_tolerance_m;
    float dr_worse_than_entry_orientation_tolerance_rad;
    float dr_near_strict_regression_multiplier;
    float dr_aggressive_action_weight;
    float dr_aggressive_action_threshold;
    float dr_dq_penalty_weight;
    float dr_dq_penalty_threshold;
    float dr_near_strict_action_penalty_multiplier;
    float dr_near_strict_dq_penalty_multiplier;
    /* route reward (route wrappers only) */
    float rr_q_goal_progress_weight;
    float rr_ee_position_progress_weight;
    float rr_ee_orientation_progress_weight;
    float rr_route_tangent_progress_weight;
    float rr_same_step_route_ready_bonus;
    float rr_route_ready_dwell_bonus;
    float rr_low_motion_near_waypoint_bonus;
    float rr_orientation_regression_penalty_weight;
    float rr_q_route_regression_penalty_weight;
    float rr_off_route_penalty_weight;
    float rr_action_magnitude_weight;
    float rr_action_delta_weight;
    float rr_dq_penalty_weight;
    float rr_no_progress_penalty;
    float rr_route_ready_pos_threshold_m;
    float rr_route_ready_ori_threshold_rad;
    float rr_route_ready_q_threshold;
    float rr_route_ready_action_threshold;
    float rr_route_ready_dq_threshold;
} KinEnvParams;

/* Device-side reset sampler: the Stage 0-11 curriculum shells and the random-start pair sampler
 * (envs/curriculum.py:90-101, envs/reset_samplers.py:168-420).  Counter-based Philox4x32-10,
 * key = (seed, env), counter = (episode, draw); validated distributionally against the
 * reference's numpy PCG64 samplers (bit-identical streams are a host-side feature, samplers.py). */
typedef struct KinSamplerParams {
    int n_stages;
    int current_stage;
    int curriculum_enabled;
    int stage_mix_enabled;
    float start_q[112];
    float start_noise[112];
    float goal_q[112];
    float goal_noise[112];
    float start_sample_margin_fraction;
    float goal_sample_margin_fraction;
    /* workspace_stage_sampling (reset_samplers.py:344-389) */
    float current_stage_ratio;
    float previous_stage_ratio;
    float old_workspace_replay_ratio;
    float failure_replay_ratio;
    int previous_stage_min_index;
    int old_workspace_max_stage_index;
    /* random_start_pair_sampling (reset_samplers.py:213-309) */
    int random_start_enabled;
    float source_ratio[6];
    int home_stage_index;
    int known_target_max_stage_index;
    int mixed_target_max_stage_index;
    int frontier_min_stage_index;
    int frontier_max_stage_index;
    int frontier_target_min_stage_index;
    int frontier_target_max_stage_index;
    int stress_target_min_stage_index;
    int stress_target_max_stage_index;
    int old_success_max_stage_index;
    float random_valid_start_margin_fraction;
    float stress_start_margin_fraction;
    float failure_recovery_q_noise[7];
    float initial_dq_noise[7];
    float initial_prev_action_noise[7];
    float min_pair_joint_l2;
    /* dock resets (reset_samplers.py:426-471): goal shell + init noise around the goal */
    int dock_use_stage_goal;
    float dock_goal_q[7];
    float dock_goal_noise[7];
    float dock_init_q_noise[7];
    /* close-bucket branch (reset_samplers.py:452-515): rejection-sample a start whose pose error lies in the bucket */
    float dock_close_bucket_probability;
    float dock_close_init_q_noise[7];
    float dock_close_bucket_min_pos_error_m;
    float dock_close_bucket_max_pos_error_m;
    float dock_close_bucket_min_ori_error_rad;
    float dock_close_bucket_max_ori_error_rad;
    int dock_close_bucket_max_attempts;
    /* handoff-state replay (reset_samplers.py:434-446): with this probability a reset copies one state of the buffer
     * (built by the Approach rollouts, training/build_finisher_handoff_state_buffer.py).  dock_handoff_states is a DEVICE
     * pointer to [count][KIN_HANDOFF_STATE_FLOATS] floats owned by the caller:
     * initial_q 7 | initial_dq 7 | initial_prev_action 7 | goal_q 7 | goal_pose6 6.                                       */
    float dock_handoff_state_probability;
    int dock_handoff_state_count;
    const float *dock_handoff_states;
    /* adaptive frontier targets (this project's extension, coverage.FrontierCurriculum): DEVICE pointers owned by the caller.
     * The reference stops at per-bucket sampling priorities (workspace/adaptive_frontier_sampler.py); the rule that turns them into
     * goals is this project's own.  Armed when frontier_probability > 0, frontier_bucket_count > 0 and every pointer is non-null,
     * and only reached by the random-start pair sampler (approach mode, random_start_enabled).  Draw order of one armed reset:
     *   1. u < frontier_probability                          (the coin; an UNARMED sampler draws nothing here: today's stream)
     *   2. the start source mix, as without the table
     *   3. coin taken:  k = integers(0, B - 1), u = uniform(), bucket b = u < alias_prob[k] ? k : alias_index[k];
     *                   target j = integers(offset[b], offset[b + 1] - 1); goal_q = targets[j][0:7];
     *                   stage = targets[j][7], or current_stage when it is -1 (a uniform-valid target)
     *      otherwise:   the stage-shell target of the source (sample_target_stage + goal shell)
     *   4. the start of the source (failure_recovery jitters the goal of step 3), dq and prev-action noise
     *   5. min_pair_joint_l2 retries (at most 12) redraw step 3 the same way: from the table when the coin was taken.
     * The goal pose is FK(goal_q), computed on the device as for every sampled reset.                                           */
    float frontier_probability;
    int frontier_bucket_count;
    int frontier_target_count;
    const int *frontier_bucket_offset;   /* [bucket_count + 1], CSR into frontier_targets */
    const float *frontier_alias_prob;    /* [bucket_count] */
    const int *frontier_alias_index;     /* [bucket_count] */
    const float *frontier_targets;       /* [target_count][KIN_FRONTIER_TARGET_FLOATS]: goal_q 7 | stage (-1: uniform-valid) */
} KinSamplerParams;
#define KIN_HANDOFF_STATE_FLOATS 34
#define KIN_FRONTIER_TARGET_FLOATS 8

/* SB3 MultiInputPolicy weights, fp32, row-major [out][in] exactly as in policy.pth (SURVEY F4):
 * x[in_dim] -> tanh(W0 x + b0)[64] -> tanh(W1 h + b1)[64] -> Wa h + ba [7]; value head likewise -> [1]. */
typedef struct KinPolicyWeights {
    int in_dim;
    int has_value;
    const float *pi_w0;
    const float *pi_b0;
    const float *pi_w1;
    const float *pi_b1;
    const float *act_w;
    const float *act_b;
    const float *vf_w0;
    const float *vf_b0;
    const float *vf_w1;
    const float *vf_b1;
    const float *val_w;
    const float *val_b;
    const float *log_std;
} KinPolicyWeights;

/* per-episode rows of the fused Approach -> Finisher evaluation: result[row * stride + episode] */
#define KIN_RES_SUCCESS 0             /* u32 pipeline success (last finisher step, else approach) */
#define KIN_RES_FLAGS 1               /* u32 bit0 approach_success, bit1 ready_hit, bit2 ready_dwell, bit3 final_ready, bits 4-5 handoff_kind */
#define KIN_RES_HANDOFF_STEP 2        /* i32, -1 if none */
#define KIN_RES_FIRST_READY_STEP 3    /* i32, -1 if none */
#define KIN_RES_MAX_READY_STREAK 4    /* i32 */
#define KIN_RES_STEPS 5               /* u32 approach_steps | finisher_steps << 16 */
#define KIN_RES_FINAL_POS 6           /* f32 final_position_error (pipeline) */
#define KIN_RES_FINAL_ORI 7
#define KIN_RES_APPROACH_POS 8        /* f32 approach_final_position_error */
#define KIN_RES_APPROACH_ORI 9
#define KIN_RES_MIN_POS 10
#define KIN_RES_MIN_ORI 11
#define KIN_RES_FINAL_ACTION 12       /* f32 final_action_magnitude */
#define KIN_RES_FINAL_DQ 13           /* f32 final_dq_norm */
#define KIN_RES_FINAL_Q 14            /* 7 x f32 */
#define KIN_RES_APPROACH_ACTION 21    /* f32 action magnitude / dq norm at the END OF THE APPROACH phase (what _failure_reason reads) */
#define KIN_RES_APPROACH_DQ 22
#define KIN_RES_ROWS 24

/* Dense q-goal route (route/route_dataset.py:16-99): device arrays, one row per waypoint. */
typedef struct KinRouteTable {
    int n_waypoints;
    int pad0;
    const float *q_goal;
    const float *pose6;
    const float *next_q_delta;
    const float *progress_m;
    /* Optional pruning table for the nearest-waypoint scan of the route reward (route_env.py:135 scans the whole route every step):
     * nearest_lb[i * nearest_lb_k + k] <= min over waypoints j with |j - i| >= k of |q_goal[j] - q_goal[i]| (k = 0 .. nearest_lb_k - 1,
     * +inf where no such j exists).  With it the step kernels visit waypoints outward from the env's current target and stop as soon
     * as the triangle inequality rules the rest out -- the SAME minimum, a handful of candidates instead of all of them.
     * NULL / 0: every waypoint is visited. */
    const float *nearest_lb;
    int nearest_lb_k;
    int pad1;
} KinRouteTable;

/* per-step scalars of the route wrappers: raux[row * stride + env] (route/route_env.py:175-190 info keys) */
#define KIN_RAUX_Q_ERR 0        /* route_q_error_norm        */
#define KIN_RAUX_NEAREST 1      /* nearest_route_q_distance  */
#define KIN_RAUX_POS_ERR 2      /* position_error_norm       */
#define KIN_RAUX_ORI_ERR 3      /* orientation_error_norm    */
#define KIN_RAUX_FLAGS 4        /* u32: bit0 route_ready, bit1 route_regression, bit2 route_orientation_hit, bit3 waypoint_success */
#define KIN_RAUX_ROUTE_INDEX 5  /* u32 route_index after the step (advanced in sequence mode) */
#define KIN_RAUX_STREAK 6       /* u32 route_ready_streak    */
#define KIN_RAUX_COMPLETED 7    /* u32 route_completed_waypoints (sequence mode) */
#define KIN_RAUX_ROWS 8

/* ---------------------------------------------------------------------------------------------
 * library
 * ------------------------------------------------------------------------------------------- */
int kin_abi_version(void);
/* sha256 (hex) of the sources this library was compiled from (rl_brain_trainer_b200/build.py::source_hash: every csrc .cu / .cuh / .h and
 * this header), "unstamped" for a build outside build.py.  The Python loader refuses (after one rebuild attempt) a library whose hash
 * differs from the tree it sits in.  No reference counterpart: the reference is interpreted Python.                                  */
const char *kin_source_hash(void);
const char *kin_last_error_string(void);
/* number of SMs / device name of the current device (for grid sizing and bench metadata) */
int kin_device_info(int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len);

/* Replaces: ArmKinematicEnv.__init__(config) -- validates and stores a host copy of the params.   */
int kin_params_create(const KinEnvParams *host_params, void **handle);
int kin_params_set_sampler(void *handle, const KinSamplerParams *host_sampler);
int kin_params_destroy(void *handle);

/* Replaces: compute_ee_pose6 / ee_pose6_from_q (kinematics/fk_interface.py:21, v5_1/ee_fk.py:120).
 * q [n,7] row-major -> pose6 [n,6] row-major.                                                    */
int kin_fk_pose6(void *handle, const float *q, float *pose6, int n, void *stream);

/* Replaces: ArmKinematicEnv.reset(options={initial_q, initial_dq, initial_prev_action, goal_q,
 * goal_pose6, policy_mode}) (AKE:102-211, explicit-options branch) for a batch.
 * env_ids: NULL = envs [0, n_reset) else int32 [n_reset] slots; option arrays are [n_reset,7|6]
 * row-major; initial_dq / initial_prev_action / goal_pose6 may be NULL (zeros / FK(clip(goal_q))).
 * goal_q may be NULL only if goal_pose6 is given.  obs (nullable) is [n_reset,56].               */
int kin_env_reset(void *handle, float *state, int stride, int n_envs, const int *env_ids, int n_reset,
                  int mode, const float *initial_q, const float *initial_dq, const float *initial_prev_action,
                  const float *goal_q, const float *goal_pose6, float *obs, void *stream);

/* Replaces: sample_approach_reset / sample_dock_reset + reset (AKE:157-176) on the device, for the
 * slots whose mask byte is non-zero (mask NULL = all).  Requires kin_params_set_sampler.          */
int kin_env_reset_sampled(void *handle, float *state, int stride, int n_envs, const uint8_t *mask, int mode,
                          uint64_t seed, float *obs, void *stream);

/* Replaces: ArmKinematicEnv.step(action) (AKE:213-365) for n envs -- the fused env-step kernel.
 * action [n,7] row-major; obs [n,56] row-major; reward [n]; done [n] (KIN_DONE_* bits);
 * aux (nullable) [KIN_AUX_ROWS][stride]; components (nullable) [KIN_MAX_COMPONENTS][stride] =
 * info["reward_components"] in the reference's dict order.  mode_hint: KIN_MODE_APPROACH /
 * KIN_MODE_DOCK when the whole batch is in one mode (specialised kernel), else KIN_MODE_PER_ENV.
 * auto_reset != 0: finished slots are re-seeded in the same kernel by the device sampler
 * (VecEnv semantics: obs is the first observation of the next episode, KIN_DONE_AUTORESET set,
 * terminal_obs (nullable, [n,56]) receives the last observation of the finished episode).        */
int kin_env_step(void *handle, float *state, int stride, int n_envs, int mode_hint, const float *action,
                 float *obs, float *reward, uint8_t *done, float *aux, float *components, int auto_reset,
                 uint64_t seed, float *terminal_obs, void *stream);

/* Replaces: ArmKinematicEnv.current_observation() (AKE:381) -> obs [n,56].                        */
int kin_env_observe(void *handle, const float *state, int stride, int n_envs, float *obs, void *stream);

/* rows of the handoff-state output of kin_rollout_handoff_states: [KIN_HO_ROWS][stride] floats */
#define KIN_HO_FINAL_Q 0              /* approach end state: q, dq, prev_action (7 each) */
#define KIN_HO_FINAL_DQ 7
#define KIN_HO_FINAL_PA 14
#define KIN_HO_SNAP_Q 21              /* first-confirmed snapshot (zeros when there was none) */
#define KIN_HO_SNAP_DQ 28
#define KIN_HO_SNAP_PA 35
#define KIN_HO_GOAL_Q 42
#define KIN_HO_GOAL_POSE 49           /* 6 */
#define KIN_HO_FINAL_METRICS 55       /* position error, orientation error, action magnitude, dq norm */
#define KIN_HO_SNAP_METRICS 59
#define KIN_HO_FINAL_STEP 63          /* step counts as floats; KIN_HO_SNAP_STEP = -1 when no snapshot */
#define KIN_HO_SNAP_STEP 64
#define KIN_HO_ROWS 65

/* Replaces: `model.predict(obs, deterministic=True)` of the SB3 MultiInputPolicy
 * (eval/eval_three_stage.py:25-27) for a batch: obs [n,in_dim] -> action [n,7] (clipped to +-1),
 * value [n] (nullable).                                                                           */
int kin_policy_forward(const KinPolicyWeights *host_weights, const float *obs, float *action, float *value,
                       int n, void *stream);

/* Replaces: the per-episode loop of evaluate_workspace_expansion_checkpoint / _run_pairs
 * (eval/eval_workspace_expansion.py:126-147, eval/eval_full_workspace_coverage.py:120-164):
 * _run_approach_with_handoff + _finisher_ready + _run_policy(dock), fused into ONE persistent
 * kernel with the policy in the loop, one thread per episode, state in registers.
 * episode inputs are [n,7|6] row-major (initial_dq / initial_prev_action nullable);
 * result is [KIN_RES_ROWS][stride] words; env_steps (nullable, device u64) += steps executed.     */
int kin_rollout_approach_finisher(void *approach_handle, void *finisher_handle,
                                  const KinPolicyWeights *host_approach, const KinPolicyWeights *host_finisher,
                                  const float *initial_q, const float *initial_dq, const float *initial_prev_action,
                                  const float *goal_q, const float *goal_pose6, int n, int stride,
                                  int handoff_confirm_steps, int variant, uint32_t *result,
                                  unsigned long long *env_steps, void *stream);

/* Replaces: training/build_finisher_handoff_state_buffer.py:73-112 -- the Approach policy alone over n episodes with the handoff
 * bookkeeping of _run_approach_with_handoff; besides the usual result rows it writes, per episode, the approach end state and the
 * first-confirmed snapshot (q, dq, prev_action, their error / action / dq metrics and step), the goal pose and goal_q
 * (KIN_HO_* rows) from which the three handoff modes (final_settled, first_confirmed, final_always) are assembled.  Strict fp32. */
int kin_rollout_handoff_states(void *approach_handle, const KinPolicyWeights *host_approach, const float *initial_q, const float *initial_dq,
                               const float *initial_prev_action, const float *goal_q, const float *goal_pose6, int n, int stride,
                               int handoff_confirm_steps, uint32_t *result, float *handoff_out, unsigned long long *env_steps, void *stream);

/* Replaces: RouteKinematicEnv.reset(options={route_index, start_route_index}) / RouteSequenceKinematicEnv.reset and
 * the evaluator's state override (route/route_env.py:49-97, route/route_sequence_env.py:96-137,
 * eval/eval_route_curriculum.py:67-87).  route_index [n_reset] int32; last_route_index (nullable, sequence mode);
 * initial_q (nullable -> waypoint(start_route_index[i]) with start_route_index nullable -> route_index-1);
 * obs [n_reset,80] nullable.  route_index[i] < 0 skips entry i (masked reset: pass every slot, -1 for the ones that keep
 * running -- no host-side compaction of the finished slots).                                                        */
int kin_route_reset(void *handle, const KinRouteTable *host_route, float *state, int stride, int n_envs, const int *env_ids,
                    int n_reset, const int *route_index, const int *start_route_index, const int *last_route_index,
                    const float *initial_q, const float *initial_dq, const float *initial_prev_action, float *obs, void *stream);

/* sample_route_reset (route/route_reset_samplers.py:43-117) as a table: reset-mode probabilities in the reference's order
 * (prefix_start, random_prefix, segment, replay, recovery), the inclusive target-waypoint range of every mode, the three noise
 * scales; forced_mode >= 0 pins the mode (config.mode = "<name>_reset").  sequence_length > 0: RouteSequenceKinematicEnv.reset
 * (route/route_sequence_env.py:120-124) clamps the target to [1, max_route_index] and sets last = min(target + length - 1, max). */
typedef struct KinRouteResetParams {
    float mode_cdf[5];
    int forced_mode;
    int index_lo[5];
    int index_hi[5];
    float q_noise_std;
    float dq_noise_std;
    float prev_action_noise_std;
    int sequence_length;
    int max_route_index;
} KinRouteResetParams;

/* Replaces: RouteKinematicEnv.reset() without options (route/route_env.py:60-73 -> sample_route_reset) for every slot whose
 * done byte has KIN_DONE_TERMINATED or KIN_DONE_TRUNCATED set (done == NULL: every slot) -- the route env's auto-reset, one
 * launch, no host round trip.  Draws are Philox4x32(seed, env, counter): distributionally, not bitwise, the reference's numpy
 * stream.  obs [n_envs,80] (nullable): the rows of the reset slots are rewritten, the others untouched.                        */
int kin_route_reset_sampled(void *handle, const KinRouteTable *host_route, const KinRouteResetParams *host_reset, float *state, int stride,
                            int n_envs, const uint8_t *done, uint64_t seed, uint32_t counter, float *obs, void *stream);

/* Replaces: RouteKinematicEnv.step (route/route_env.py:124-192; sequence_mode = 0) and RouteSequenceKinematicEnv.step
 * with the in-episode waypoint advance (route/route_sequence_env.py:139-257; sequence_mode = 1).
 * obs [n,80]; reward = route reward (route/reward_route.py:54-143); done = KIN_DONE_* with route semantics;
 * raux (nullable) [KIN_RAUX_ROWS][stride]; rcomp (nullable) [17][stride] = route reward components.            */
int kin_route_step(void *handle, const KinRouteTable *host_route, float *state, int stride, int n_envs, const float *action,
                   float *obs, float *reward, uint8_t *done, float *raux, float *rcomp, int sequence_mode,
                   int reset_ready_streak_on_advance, void *stream);

/* Replaces: a VecEnv of RouteKinematicEnv / RouteSequenceKinematicEnv (kinematic_phase1/train_route_curriculum.py) stepping and
 * auto-resetting -- kin_route_step followed, in the same launch, by the sampled reset of every slot the step finished
 * (KIN_DONE_TERMINATED or KIN_DONE_TRUNCATED).  reward / done / raux / rcomp describe the step just taken; the finished slots'
 * done bytes also get KIN_DONE_AUTORESET and their obs rows hold the first observation of the next episode.
 * Counter convention: state row KIN_ROW_EPISODE counts the episodes a slot has finished.  A finished slot draws
 * episode = row + 1, resets exactly as kin_route_reset_sampled(host_reset, seed, counter = episode) would, and stores episode back
 * into the row; so the counter lives on the device and a CUDA graph can replay the call unchanged.  A sampled reset of the whole
 * batch with counter 0 plus a zeroed KIN_ROW_EPISODE row starts the sequence: later resets of a slot use counters 1, 2, ...
 * terminal_obs (nullable, [n,80], 16-byte aligned): the rows of the finished slots receive the finished episode's last
 * observation; rows of other slots are either untouched or, when a slot within the same group of 32 finished, set to that
 * slot's obs row.  host_reset: as for kin_route_reset_sampled, every mode's waypoint range inside the route.                    */
int kin_route_step_autoreset(void *handle, const KinRouteTable *host_route, const KinRouteResetParams *host_reset, float *state,
                             int stride, int n_envs, const float *action, float *obs, float *reward, uint8_t *done, float *raux,
                             float *rcomp, int sequence_mode, int reset_ready_streak_on_advance, uint64_t seed, float *terminal_obs,
                             void *stream);

/* Replaces: evaluate_sequential_route / _roll_one (eval/eval_route_curriculum.py:55-125,188-218) for n independent
 * replicas, fused with the 80-input route policy: replica r starts at start_q[r] (nullable -> waypoint(start_index-1))
 * and chains waypoints start_index..end_index, each from the actual final state of the previous one.
 * prefix [n] int32 = longest_success_prefix; success_bits (nullable) [n][ceil((end-start+1)/32)] u32 bitmask.     */
int kin_route_probe(void *handle, const KinRouteTable *host_route, const KinPolicyWeights *host_policy, const float *start_q,
                    int start_index, int end_index, int n, int *prefix, uint32_t *success_bits, unsigned long long *env_steps,
                    void *stream);

/* kin_route_probe that also writes, for the first detail_replicas replicas, the per-waypoint row of _roll_one
 * (eval/eval_route_curriculum.py:111-131) from which _summarize_rows / _failure_reason / _chunk_metrics (:127-186) are computed:
 * rows [detail_replicas][end_index - start_index + 1][KIN_ROUTE_ROW_FIELDS] floats.                                            */
#define KIN_ROUTE_ROW_SUCCESS 0
#define KIN_ROUTE_ROW_READY_HIT 1
#define KIN_ROUTE_ROW_READY_DWELL 2
#define KIN_ROUTE_ROW_FIRST_READY_STEP 3 /* -1: never ready */
#define KIN_ROUTE_ROW_MAX_READY_STREAK 4
#define KIN_ROUTE_ROW_STEPS 5
#define KIN_ROUTE_ROW_FINAL_POS 6
#define KIN_ROUTE_ROW_FINAL_ORI 7
#define KIN_ROUTE_ROW_FINAL_Q_ERR 8
#define KIN_ROUTE_ROW_MIN_POS 9
#define KIN_ROUTE_ROW_MIN_ORI 10
#define KIN_ROUTE_ROW_MIN_Q_ERR 11
#define KIN_ROUTE_ROW_FINAL_ACTION_L2 12
#define KIN_ROUTE_ROW_FINAL_DQ_L2 13
#define KIN_ROUTE_ROW_FIELDS 14
int kin_route_probe_rows(void *handle, const KinRouteTable *host_route, const KinPolicyWeights *host_policy, const float *start_q,
                         int start_index, int end_index, int n, int *prefix, uint32_t *success_bits, unsigned long long *env_steps,
                         float *rows, int detail_replicas, void *stream);

/* The same probe with the 80-input actor on tcgen05 (kind::tf32 operands, fp32 accumulation; csrc/kin_route_tc.cu): actions move by
 * O(1e-3) against the strict-fp32 probe, which stays the parity path.  Same arguments and outputs.                              */
int kin_route_probe_tc(void *handle, const KinRouteTable *host_route, const KinPolicyWeights *host_policy, const float *start_q,
                    int start_index, int end_index, int n, int *prefix, uint32_t *success_bits, unsigned long long *env_steps,
                    void *stream);

/* ---------------------------------------------------------------------------------------------
 * PPO agent update (third-party arithmetic: stable-baselines3 2.8.0 PPO, call sites
 * kinematic_phase1/train_workspace_expansion.py:189-232; restated in DESIGN.md section 3 "K3").
 * All parameters live in ONE flat fp32 buffer in this order (sizes for in_dim = 56):
 *   pi_w0[64*in] pi_b0[64] pi_w1[64*64] pi_b1[64] act_w[7*64] act_b[7]
 *   vf_w0[64*in] vf_b0[64] vf_w1[64*64] vf_b1[64] val_w[64] val_b[1] log_std[7]          = 16150 floats
 * ------------------------------------------------------------------------------------------- */
#define KIN_PPO_TILE 64          /* samples per tile; minibatches are unions of tiles */
#define KIN_PPO_STATS 8          /* per-minibatch statistics, see KIN_PPO_STAT_* */
#define KIN_PPO_STAT_POLICY_LOSS 0
#define KIN_PPO_STAT_VALUE_LOSS 1
#define KIN_PPO_STAT_ENTROPY 2
#define KIN_PPO_STAT_APPROX_KL 3
#define KIN_PPO_STAT_CLIP_FRACTION 4
#define KIN_PPO_STAT_GRAD_NORM 5
#define KIN_PPO_STAT_SAMPLES 6
#define KIN_PPO_STAT_SKIP 7         /* set by kin_peer_grad_gather after a peer timed out: kin_ppo_adam then leaves the parameters untouched */

typedef struct KinPpoHyper {
    float gamma;
    float gae_lambda;
    float clip_range;
    float ent_coef;
    float vf_coef;
    float max_grad_norm;
    float learning_rate;
    float adam_beta1;
    float adam_beta2;
    float adam_eps;
    int normalize_advantage;
    int pad0;
} KinPpoHyper;

int kin_ppo_param_count(int in_dim);

/* Replaces: policy.forward(obs) during collect_rollouts (SB3 on_policy_algorithm.py): a = mean + exp(log_std) * eps,
 * value, log_prob.  obs [n,56]; action [n,7] (unclipped sample, what SB3 stores); the env clips it itself.
 * eps is Philox4x32(seed, env, step).  deterministic != 0 -> action = mean.                                       */
int kin_policy_act(const KinPolicyWeights *host_weights, const float *obs, float *action, float *logp, float *value, int n,
                   uint64_t seed, uint32_t step, int deterministic, void *stream);

/* Replaces: the TimeLimit bootstrap of collect_rollouts: reward += gamma * V(terminal_obs) where the episode was
 * truncated (not terminated).  terminal_obs [n,56], done [n] KIN_DONE_* bytes.                                    */
int kin_ppo_bootstrap(const KinPolicyWeights *host_weights, const float *terminal_obs, const uint8_t *done, float *reward, float gamma,
                      int n, void *stream);

/* Replaces: RolloutBuffer.compute_returns_and_advantage (GAE).  reward/value/episode_start are [T][n] (episode_start u8),
 * last_value [n], last_done [n] u8 (KIN_DONE_* bytes of the last step) -> advantage, returns [T][n];
 * tile_sums (nullable) [T*n/64][2] doubles = (sum adv, sum adv^2) per 64-sample tile.                            */
int kin_ppo_gae(const float *reward, const float *value, const uint8_t *episode_start, const float *last_value, const uint8_t *last_done,
                float gamma, float gae_lambda, int T, int n, float *advantage, float *returns, double *tile_sums, void *stream);

/* One PPO minibatch gradient (SB3 ppo.py train(): clipped surrogate + vf_coef * MSE + ent_coef * entropy term, advantages
 * normalised per minibatch).  The minibatch is the union of the 64-sample tiles tile_ids[0..n_tiles); sample s of tile j is
 * row tile_ids[j]*64 + s of obs [S,56] / action [S,7] / old_logp / advantage / returns.  global_batch = samples in the
 * whole (all-rank) minibatch.  grad [P] receives the SUM over local samples of d(loss*global_batch)/dparam / global_batch,
 * i.e. ranks all-reduce (sum) grad and stats afterwards.  partials: scratch [grid][P + KIN_PPO_STATS + 8] floats.
 * grad == NULL (both variants): the per-CTA rows stay unreduced in partials[0 .. min(grid, tiles)) for kin_peer_grad_push.
 * adv_stats (nullable): this minibatch's (mean, 1/(std+eps)) from kin_ppo_adv_stats; NULL -> computed from tile_sums.     */
int kin_ppo_grad(const float *params, int in_dim, const KinPpoHyper *host_hyper, const float *obs, const float *action, const float *old_logp,
                 const float *advantage, const float *returns, const double *tile_sums, const int *tile_ids, int n_tiles,
                 long long global_batch, float *partials, int grid, float *grad, float *stats, const float *adv_stats, void *stream);

/* Replaces: RolloutBuffer.get (SB3 buffers.py): `indices = np.random.permutation(buffer_size * n_envs)`, minibatches = consecutive
 * slices of the permuted samples.  Physically permutes one rollout: destination sample d = source sample perm[d] (perm: a permutation of
 * 0 .. n_samples - 1, n_samples a multiple of 128) for obs (obs_is_image: the 16 KB-per-128-samples bf16 operand images of
 * kin_ppo_collect / kin_route_obs_images, rows moved between swizzle phases; else fp32 [n_samples][in_dim]), action [n][7], old_logp,
 * advantage, returns; tile_sums_out [n_samples / 64][2] = (sum adv, sum adv^2) per 64-sample tile of the NEW order.  Minibatch m of the
 * epoch is then tiles [m * k, (m + 1) * k) of the permuted buffers for the gradient kernels below -- SB3's per-sample minibatches
 * instead of unions of 64-sample tiles of the rollout order.  Not in place.                                                        */
int kin_ppo_shuffle(const void *obs, int obs_is_image, int in_dim, const float *action, const float *old_logp, const float *advantage,
                    const float *returns, const int *perm, long long n_samples, void *obs_out, float *action_out, float *old_logp_out,
                    float *advantage_out, float *returns_out, double *tile_sums_out, void *stream);

/* (mean, 1 / (std + 1e-8)) of the advantages of n_minibatches minibatches at once (minibatch m = tile_ids[m * n .. (m + 1) * n),
 * n = n_tiles_per_minibatch), torch semantics (unbiased std); normalize == 0 writes (0, 1).  adv_stats [n_minibatches][2]; pass
 * adv_stats + 2 * m to the gradient kernels so they skip their own (serial) pass over the tile sums.                          */
int kin_ppo_adv_stats(const double *tile_sums, const int *tile_ids, int n_tiles_per_minibatch, int n_minibatches, int normalize,
                      float *adv_stats, void *stream);

/* Tensor-core variant of kin_ppo_grad: the same minibatch gradient with every GEMM (forward, data gradients and the
 * sample-reduction weight-gradient GEMMs) on tcgen05.mma kind::f16 (bf16 operands, fp32 accumulation in TMEM).
 * n_tiles must be even (two 64-sample tiles form one 128-row GEMM tile).  partials: scratch [grid][P + 16] floats.
 * logp_out / value_out (nullable, [S]) receive this variant's own log-prob / value of every visited sample; with
 * forward_only != 0 nothing else is computed (used to refresh old_logp with the same arithmetic the update uses).
 * obs_is_image != 0: obs is the rollout buffer kin_ppo_collect wrote -- one 16 KB bf16 operand image per 128 consecutive
 * samples -- and every pair (tile_ids[2j], tile_ids[2j+1]) must be (2m, 2m+1), i.e. one whole image.
 * weight_image (nullable): the bf16 operand image of params (kin_ppo_pack_weights / kin_ppo_adam keep it current); each CTA then
 * fetches its weights with bulk copies instead of converting them from fp32.
 * in_dim: 56 (Approach / Finisher policies) or 80 (the route policy of train_route_curriculum.py).  The route policy runs layer 1 on
 * its 60 live observation columns -- the 20 constant columns are folded into the bias (csrc/kin_ppo_layout.cuh), gradients come back
 * in the full 80-column layout -- so obs must be the folded images of kin_route_obs_images (obs_is_image = 1) and weight_image, when
 * given, the folded image kin_ppo_pack_weights(in_dim = 80) builds.                                                               */
int kin_ppo_grad_tc(const float *params, int in_dim, const KinPpoHyper *host_hyper, const void *obs, const float *action, const float *old_logp,
                    const float *advantage, const float *returns, const double *tile_sums, const int *tile_ids, int n_tiles,
                    long long global_batch, float *partials, int grid, float *grad, float *stats, float *logp_out, float *value_out,
                    int forward_only, int obs_is_image, const float *adv_stats, const void *weight_image, void *stream);

/* kin_ppo_grad_tc with the gradient exchange over NVLink peer memory (kin_peer_* buffers) fused into the kernel's tail: after a grid
 * barrier every CTA reduces a column slice of the partial rows, stores it into every rank's receive buffer, waits for the same slice
 * from every rank and writes grad / stats = the sum over ranks in RANK ORDER (bitwise identical on all ranks; with world == 1 bitwise
 * the plain reduction).  Replaces the kin_peer_grad_push + kin_peer_grad_gather launches between the gradient kernel and kin_ppo_adam.
 * epoch counts exchanges from 1 and must advance by one per call on every rank; *timed_out is the sticky device flag of
 * kin_peer_grad_gather (a dead peer marks stats[KIN_PPO_STAT_SKIP], kin_ppo_adam then leaves the parameters untouched).            */
int kin_ppo_grad_tc_exchange(const float *params, int in_dim, const KinPpoHyper *host_hyper, const void *obs, const float *action,
                             const float *old_logp, const float *advantage, const float *returns, const double *tile_sums, const int *tile_ids,
                             int n_tiles, long long global_batch, float *partials, int grid, float *grad, float *stats, int obs_is_image,
                             const float *adv_stats, const void *weight_image, void *const *peer_buffers, int rank, int world, unsigned epoch,
                             int *timed_out, void *stream);

/* kin_ppo_grad_tc_exchange + kin_ppo_adam in ONE launch: after the rank-ordered sum every CTA also applies clip_grad_norm_ + Adam
 * (SB3 ppo.py train(): th.nn.utils.clip_grad_norm_ + optimizer.step, kin_ppo_adam's arithmetic) to the slice of the summed gradient it
 * owns -- per-CTA sums of squares, a second grid barrier, the same clip coefficient in every CTA and on every rank -- and keeps the bf16
 * weight image (56-input policies) in step.  params_rw must be params (updated in place; the kernel reads the weights only in its
 * prologue), step counts optimiser steps from 1, norm_scratch holds 2 * grid floats, stats_accum (nullable) receives the running sums of
 * kin_ppo_adam.  A minibatch whose exchange timed out leaves the parameters untouched.  With world == 1 the peer buffer is the rank's own
 * (kin_peer_buffer_create(n_params, 1, ..)): single-GPU training runs one launch per minibatch too.                                  */
int kin_ppo_grad_tc_update(const float *params, int in_dim, const KinPpoHyper *host_hyper, const void *obs, const float *action, const float *old_logp,
                           const float *advantage, const float *returns, const double *tile_sums, const int *tile_ids, int n_tiles,
                           long long global_batch, float *partials, int grid, float *grad, float *stats, int obs_is_image, const float *adv_stats,
                           void *weight_image, void *const *peer_buffers, int rank, int world, unsigned epoch, int *timed_out, float *params_rw,
                           float *adam_m, float *adam_v, int step, float *stats_accum, float *norm_scratch, void *stream);

/* Experimental variant switch of kin_ppo_grad_tc / kin_ppo_grad_tc_exchange.  When enabled, 56-input policies on operand images with
 * minibatches of at least one 128-sample tile per CTA (n_tiles / 2 >= grid, 2 <= grid <= SM count) run the gradient pass on the
 * three-tile-streams-per-SM kernel (csrc/kin_ppo_tc3.cu: one CTA per SM, grid split between actor and critic CTAs); everything else, and
 * everything by default, runs the two-CTAs-per-SM kernel (the three-stream kernel measured 4 % slower: both are bound by the
 * shared-memory data pipe, DESIGN.md).  enabled: 0 / 1, negative = leave; actor_pct: share of the CTAs that work on the actor (10..90),
 * else leave.  Defaults: off, 52 %, or the environment (KIN_PPO_TC3=1, KIN_PPO_TC3_ACTOR_PCT).  Returns enabled | actor_pct << 8 after
 * the change.  Same reference call replaced as kin_ppo_grad_tc (SB3 ppo.py train(), one minibatch).                                 */
int kin_ppo_tc3_config(int enabled, int actor_pct);

/* Replaces: OnPolicyAlgorithm.collect_rollouts (SB3 on_policy_algorithm.py) over a VecEnv of ArmKinematicEnv, fused into ONE
 * launch: n_steps x (actor + critic forward on tcgen05, a = mean + exp(log_std) * eps, log-prob, env step with reward and
 * termination, in-register auto-reset from the device sampler).  n_envs must be a multiple of 128.  Outputs, time-major:
 * obs_tiles [n_steps][n_envs/128][16 KB] bf16 operand images ([obs | 1 | 0] rows, SWIZZLE_128B) consumed by
 * kin_ppo_grad_tc(obs_is_image = 1); action [T][n][7]; logp / value / reward [T][n]; done / episode_start [T][n] u8;
 * start_io [n] u8 (in: "previous step finished an episode" of step 0, out: the same for the next rollout); last_value [n].
 * Episodes that hit the time limit append (t * n + env, terminal observation) to boot_index / boot_obs (capacity boot_cap,
 * count in *boot_count, reset by this call); kin_ppo_bootstrap_list then adds gamma * V(terminal_obs) to their rewards.
 * eps is Philox4x32(noise_seed, env, first_step + t) -- the draws of kin_policy_act; resets use Philox(reset_seed, env, episode).
 * params: the flat PARAM_ORDER buffer; weight_image (nullable): its bf16 operand image.  tiles_per_cta: 0 (auto), 1, 2 or 4. */
int kin_ppo_collect(void *handle, float *state, int stride, int n_envs, int mode, const float *params, const void *weight_image, int in_dim, int n_steps,
                    uint64_t noise_seed, uint32_t first_step, uint64_t reset_seed, void *obs_tiles, float *action, float *logp, float *value,
                    float *reward, uint8_t *done, uint8_t *episode_start, uint8_t *start_io, float *last_value, int *boot_count,
                    int *boot_index, float *boot_obs, int boot_cap, int tiles_per_cta, void *stream);

/* Route observations [n_rows][80] fp32 -> folded bf16 operand images [n_rows / 128][16 KB]: rows of [60 live columns | 1 | 0 0 0]
 * (20 of the 80 columns are constants of the path and are folded into the layer-1 bias, see csrc/kin_ppo_layout.cuh), SWIZZLE_128B.
 * kin_ppo_grad_tc(in_dim = 80, obs_is_image = 1) consumes them; n_rows must be a multiple of 128.                               */
int kin_route_obs_images(const float *obs, long long n_rows, void *images, void *stream);

/* Replaces: collect_rollouts over a VecEnv of RouteKinematicEnv / RouteSequenceKinematicEnv (kinematic_phase1/train_route_curriculum.py:
 * 113-145; route/route_env.py:49-212, route/route_sequence_env.py:96-278, route/route_reset_samplers.py:43-117), fused into ONE launch:
 * n_steps x (80-input actor + critic forward on tcgen05, Gaussian sample + log-prob, kin_route_step semantics with the in-episode
 * waypoint advance when sequence_mode != 0, sampled route reset of finished slots as kin_route_reset_sampled draws it with
 * Philox(reset_seed, env, first_step + t)).  n_envs must be a multiple of 128.  Outputs, time-major: obs [n_steps + 1][n_envs][80] fp32
 * (row t = the observation the policy saw at step t, row n_steps = the observation after the last step), action [T][n][7],
 * logp / value / reward [T][n], done / episode_start [T][n] u8, route_flags [T][n] (the KIN_RAUX_FLAGS word of the step: bit0
 * route_ready, bit1 regression, bit2 orientation hit, bit3 waypoint success), start_io / last_value [n].  Time-limit episodes append
 * (t * n + env, terminal observation [80]) to boot_index / boot_obs for kin_ppo_bootstrap_list(in_dim = 80).                     */
int kin_route_collect(void *handle, const KinRouteTable *host_route, const KinRouteResetParams *host_reset, float *state, int stride, int n_envs,
                      const float *params, int n_steps, uint64_t noise_seed, uint32_t first_step, uint64_t reset_seed, int sequence_mode,
                      int reset_ready_streak_on_advance, float *obs, float *action, float *logp, float *value, float *reward, uint8_t *done,
                      uint8_t *episode_start, int *route_flags, uint8_t *start_io, float *last_value, int *boot_count, int *boot_index,
                      float *boot_obs, int boot_cap, int tiles_per_cta, void *stream);

/* reward[boot_index[i]] += gamma * V(boot_obs[i]) for i < min(*boot_count, boot_cap) (strict-fp32 critic of the flat params);
 * in_dim 56 or 80 (boot_obs rows of in_dim floats). */
int kin_ppo_bootstrap_list(const float *params, int in_dim, const float *boot_obs, const int *boot_index, const int *boot_count, int boot_cap,
                           float *reward, float gamma, void *stream);

/* clip_grad_norm_(max_grad_norm) + Adam step on the flat parameter buffer (torch.optim.Adam semantics, eps = 1e-5 in SB3).
 * max_grad_norm <= 0 skips the clip (torch's clip_grad_norm_(0) would zero the gradient instead).
 * adam_m / adam_v [P]; step = 1-based update count.  stats[5] receives the gradient norm; stats_accum (nullable, [8]) gets
 * stats[0..5] added and slot 7 incremented: running sums over the minibatches of one update without host round trips.
 * weight_image (nullable, in_dim 56): the bf16 operand image is rewritten in step with the parameters.                   */
int kin_ppo_adam(float *params, const float *grad, float *adam_m, float *adam_v, int n_params, const KinPpoHyper *host_hyper, int step,
                 float *stats, float *stats_accum, void *weight_image, int in_dim, void *stream);

/* Build the 36 KB bf16 operand image of the flat parameters (the B operands of the tensor-core kernels: W0 | W1 | WO of both
 * nets as SWIZZLE_128B tiles, layer-1 bias folded in as column 56).  kin_ppo_adam(weight_image != NULL) keeps it current.   */
int kin_ppo_pack_weights(const float *params, int in_dim, void *weight_image, void *stream);

/* ---- populations: K independent PPO runs through the same launches ---------------------------------------------------------------
 * A population member is one complete single-rank 56-input trainer (kin_ppo_collect + kin_ppo_grad_tc in image mode + kin_ppo_adam):
 * its own parameters, Adam state, env state, rollout buffers, seeds and hyper-parameters.  The kin_pop_* launches below run one phase
 * of ALL members at once, the member index on a grid dimension; each member's CTAs run the standalone kernel's body on that member's
 * descriptor, so member k's results are bitwise those of the standalone calls on the same buffers.  Members share the env params
 * (KinEnvParams bytes and policy mode), n_envs, n_steps and the minibatch shape.
 * The caller owns a DEVICE array of n_members descriptors and re-uploads it when a pointer, seed, step or hyper-parameter changes.
 * KIN_POP_MAX bounds n_members for two reasons.  kin_pop_adam passes every member's Adam bias corrections as a by-value kernel
 * argument (2 x 64 floats, 512 B).  kin_pop_collect resets the members' bootstrap counts from one block of KIN_POP_MAX threads.
 * 64 is also well past the sweep sizes the population serves (8 to 32 seeds / settings); larger sweeps run as several populations.
 * New entry points only: no existing struct, signature or behaviour changed, so KIN_ABI_VERSION stays 4.                        */
#define KIN_POP_MAX 64

typedef struct KinPopMember {
    const KinSamplerParams *sampler;   /* the member's device sampler (kin_params_device_sampler): its curriculum stage */
    float *state;                      /* SoA env state of the member's env handle */
    int stride;
    int boot_cap;
    uint64_t noise_seed;               /* kin_ppo_collect's noise_seed / first_step / reset_seed */
    uint64_t reset_seed;
    uint32_t first_step;
    int pad0;
    float *params;                     /* flat PARAM_ORDER parameters (read by every phase, written by kin_pop_adam) */
    void *weight_image;                /* their bf16 operand image (kin_ppo_pack_weights; kept current by kin_pop_adam) */
    void *obs_tiles;                   /* rollout buffers, as kin_ppo_collect / kin_ppo_gae take them */
    float *action;
    float *logp;
    float *value;
    float *reward;
    uint8_t *done;
    uint8_t *episode_start;
    uint8_t *start_io;
    float *last_value;
    int *boot_count;
    int *boot_index;
    float *boot_obs;
    float *advantage;
    float *returns;
    double *tile_sums;
    const int *tile_ids;               /* this epoch's tile permutation: minibatch m = tile_ids[m * n .. (m + 1) * n) */
    float *adv_stats;                  /* [minibatches per epoch][2], kin_ppo_adv_stats' output */
    float *partials;                   /* kin_ppo_grad_tc scratch, [grid][P + 16] */
    float *grad;
    float *stats;
    float *stats_accum;
    float *adam_m;
    float *adam_v;
    KinPpoHyper hyper;                 /* gamma, gae_lambda, clip_range, ent_coef, vf_coef, max_grad_norm, Adam, normalize_advantage */
} KinPopMember;

/* The device copy of the handle's sampler (NULL until kin_params_set_sampler) and a byte comparison of two handles' env params. */
int kin_params_device_sampler(void *handle, const void **sampler);
int kin_params_same_env(void *handle_a, void *handle_b, int *same);

/* Replaces: collect_rollouts (SB3 on_policy_algorithm.py), once per member: kin_ppo_collect(handle, member.state, member.stride, n_envs,
 * mode, member.params, member.weight_image, 56, n_steps, member.noise_seed, member.first_step, member.reset_seed, member's buffers,
 * tiles_per_cta = 1) for every member, with member.sampler in place of the handle's.  handle supplies the shared env params.        */
int kin_pop_collect(void *handle, const KinPopMember *members, int n_members, int n_envs, int mode, int n_steps, void *stream);

/* kin_ppo_bootstrap_list(member.params, 56, member's list, member.boot_cap, member.reward, member.hyper.gamma) for every member;
 * max_boot_cap >= every member's boot_cap sizes the grid.                                                                        */
int kin_pop_bootstrap_list(const KinPopMember *members, int n_members, int max_boot_cap, void *stream);

/* Replaces: RolloutBuffer.compute_returns_and_advantage, once per member: kin_ppo_gae on the member's buffers (last_done = the done
 * bytes of step n_steps - 1) with its gamma / gae_lambda, tile sums included.                                                      */
int kin_pop_gae(const KinPopMember *members, int n_members, int n_envs, int n_steps, void *stream);

/* kin_ppo_adv_stats(member.tile_sums, member.tile_ids, n_tiles_per_minibatch, n_minibatches, member.hyper.normalize_advantage,
 * member.adv_stats) for every member.                                                                                             */
int kin_pop_adv_stats(const KinPopMember *members, int n_members, int n_tiles_per_minibatch, int n_minibatches, void *stream);

/* Replaces: one minibatch of SB3 ppo.py train() (loss and backward), once per member: kin_ppo_grad_tc(member.params, 56, &member.hyper,
 * member.obs_tiles, .., member.tile_sums, member.tile_ids + minibatch * n_tiles_per_minibatch, n_tiles_per_minibatch, global_batch,
 * member.partials, grid, member.grad, member.stats, NULL, NULL, 0, 1, member.adv_stats + 2 * minibatch, member.weight_image) --
 * gradient kernel and reduction, min(grid, n_tiles_per_minibatch / 2) CTAs per net and member.                                      */
int kin_pop_grad_tc(const KinPopMember *members, int n_members, int minibatch, int n_tiles_per_minibatch, long long global_batch, int grid,
                    void *stream);

/* Replaces: clip_grad_norm_ + optimizer.step, once per member: kin_ppo_adam(member.params, member.grad, member.adam_m, member.adam_v, P,
 * &member.hyper, host_steps[k], member.stats, member.stats_accum, member.weight_image, 56).  host_hypers / host_steps are HOST arrays
 * [n_members]: the bias corrections 1 - beta^step are computed on the host from host_hypers[k].adam_beta1 / adam_beta2, as
 * kin_ppo_adam computes them, so host_hypers[k] must equal member k's descriptor hyper.                                            */
int kin_pop_adam(const KinPopMember *members, int n_members, const KinPpoHyper *host_hypers, const int *host_steps, void *stream);

/* ---- gradient exchange over NVLink peer memory (the training path's one collective; SURVEY 8e(ii)) ------------------------------
 * Replaces: the per-minibatch all-reduce (sum) of the flat gradient + 5 loss statistics between the gradient kernel and Adam.
 * Every rank (one per GPU of ONE node, world <= 8) owns a receive buffer; peers open it through CUDA IPC.  Per exchange:
 * kin_peer_grad_push reduces this rank's per-CTA partial rows and stores the result into slot[epoch & 1][rank] of EVERY rank's
 * buffer (posted NVLink stores) followed by a release-store of `epoch` into the peer's arrival counter; kin_peer_grad_gather
 * waits (on the device) until all `world` counters reached `epoch` and writes grad / stats = the sum of the slots in rank
 * order, bitwise identical on every rank.  epoch = 1, 2, 3, ... must advance by one per exchange on all ranks.  A dead peer is
 * reported through *timed_out (device int, zero it once) after ~10 s instead of hanging the GPU.                              */
#define KIN_PEER_HANDLE_BYTES 64
int kin_peer_buffer_bytes(int n_params, int world);
int kin_peer_buffer_create(int n_params, int world, void **buffer, unsigned char *ipc_handle /* [KIN_PEER_HANDLE_BYTES] */);
int kin_peer_buffer_open(const unsigned char *ipc_handle, void **buffer);
int kin_peer_buffer_close(void *buffer);
int kin_peer_buffer_destroy(void *buffer);
/* peer_buffers: HOST array of `world` device pointers (own buffer at index rank, the others from kin_peer_buffer_open). */
int kin_peer_grad_push(const float *partials, int n_cta, int n_params, long long global_batch, void *const *peer_buffers, int rank, int world,
                       unsigned epoch, void *stream);
int kin_peer_grad_gather(const void *local_buffer, int n_params, int world, unsigned epoch, float *grad, float *stats, int *timed_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* KIN_B200_H */

/*
 * usv_b200.h -- C ABI of the B200-native ASV (USV) hot path.
 *
 * One shared library (libusv_b200.so), plain pointers and sizes only.  Every
 * entry point replaces a chain of eager torch ops behind one of the reference's
 * Python method surfaces; the reference location each one stands in for is
 * cited as  [ref: path:line]  relative to the reference repo root, with
 *   OIGE = omniisaacgymenvs/,  SNAP = 811_3.5*(classic snapshot)/,  RLG = rl_games/rl_games/.
 *
 * Conventions
 *   - all pointers are DEVICE pointers owned by the caller (torch tensors); the
 *     library never allocates, frees or synchronises; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*), so calls are asynchronous and re-entrant.
 *   - return value: 0 = ok, <0 = argument error (USV_E_*), >0 = cudaError_t of the
 *     launch.  usv_b200_error_string() decodes both.
 *   - float data is fp32; reset/done flags are int64 (torch.long) as in
 *     [ref: OIGE/tasks/base/rl_task.py:129-130]; rollout dones are uint8 as in
 *     [ref: RLG/common/a2c_common.py:454].
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     returns a cudaError_t.
 */
#ifndef USV_B200_H_
#define USV_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define USV_B200_ABI_VERSION 1

enum {
  USV_OK = 0,
  USV_E_NULL = -1,      /* required pointer is NULL            */
  USV_E_SIZE = -2,      /* negative / inconsistent size        */
  USV_E_PARAM = -3,     /* parameter outside supported range   */
  USV_E_ALIGN = -4,     /* pointer not aligned as documented   */
  USV_E_UNSUPPORTED = -5
};

int usv_b200_abi_version(void);
const char* usv_b200_error_string(int code);
/* number of kernels this library has launched since load (bench.py "gpu_launches") */
int64_t usv_b200_launch_count(void);
/* sizeof() of a struct of this header by name (-1 if unknown): lets FFI mirrors verify their layout */
int64_t usv_b200_sizeof(const char* struct_name);

/* ------------------------------------------------------------------------- */
/* A1  HydrostaticsObject.compute_archimedes_metacentric_local                */
/*     [ref: OIGE/envs/USV/Hydrostatics.py:63-133]                            */
/* out6[n,6] = [R^T (0,0,-rho*g*V) , (-w*sin(roll)*F, -l*sin(pitch)*F, 0)*amp] */
typedef struct {
  float water_density;
  float gravity;                          /* signed, e.g. -9.81 */
  float metacentric_width;
  float metacentric_length;
  float average_hydrostatics_force_value; /* 275 */
  float amplify_torque;
} UsvHydrostaticsParams;

int usv_hydrostatics_f32(const float* submerged_volume /*[n]*/, const float* rpy /*[n,3]*/,
                         const float* quat /*[n,4] w,x,y,z*/, float* out6 /*[n,6]*/,
                         float* force_global /*[n,3] or NULL*/, float* torque_global /*[n,3] or NULL*/,
                         int64_t n, const UsvHydrostaticsParams* p, void* stream);

/* ------------------------------------------------------------------------- */
/* A2  HydrodynamicsObject.ComputeHydrodynamicsEffects + ComputeDampingMatrix */
/*     [ref: OIGE/envs/USV/Hydrodynamics.py:176-245]                          */
typedef struct {
  float linear_damping_forward_speed[6];
  float offset_linear_damping;
  float offset_lin_forward_damping_speed;
  float offset_nonlin_damping;
  float scaling_damping;
  int32_t use_drag_scale;    /* _use_drag_scale_randomization */
  int32_t use_water_current;
  float flow_vel[3];
} UsvHydrodynamicsParams;

int usv_hydrodynamics_f32(const float* quat /*[n,4]*/, const float* world_vel6 /*[n,6]*/,
                          const float* linear_damping /*[n,6]*/, const float* quadratic_damping /*[n,6]*/,
                          const float* drag_scale /*[n] (the (n,1) tensor)*/,
                          float* drag6 /*[n,6]*/, float* local_vel6 /*[n,6] or NULL*/,
                          float* damping6 /*[n,6] or NULL: the diagonal of ComputeDampingMatrix*/,
                          int64_t n, const UsvHydrodynamicsParams* p, void* stream);

/* ------------------------------------------------------------------------- */
/* A4  DynamicsFirstOrder.get_cmd_interpolated / set_target_force             */
/*     [ref: OIGE/envs/USV/ThrusterDynamics.py:179-219]                       */
/* idx = clamp(round_half_even(((cmd+1)/2)*(n_lut-1)), 0, n_lut-1)            */
int usv_thruster_target_f32(const float* cmd2 /*[n,2]*/, const float* lut_left /*[n_lut]*/,
                            const float* lut_right /*[n_lut]*/, int32_t n_lut,
                            const float* mult_left /*[n] or NULL (=1)*/,
                            const float* mult_right /*[n] or NULL (=1)*/,
                            float* before_dynamics2 /*[n,2]*/, float* after_randomization2 /*[n,2] or NULL*/,
                            int64_t n, void* stream);

/* A5  DynamicsFirstOrder.update / update_forces                              */
/*     [ref: OIGE/envs/USV/ThrusterDynamics.py:129-141,221-234]               */
/* cur = cur*alpha + (1-alpha)*target ; thrusters[:,0]=cur[:,0], [:,3]=cur[:,1] */
int usv_thruster_lag_f32(float* current_forces2 /*[n,2] in/out*/, const float* target2 /*[n,2]*/,
                         float alpha, float* thrusters6 /*[n,6]: only cols 0,3 written*/,
                         int64_t n, void* stream);

/* LUT builder: F.interpolate(points, size=n_out, mode="linear", align_corners=True) */
/*     [ref: OIGE/envs/USV/ThrusterDynamics.py:152-177]                       */
int usv_thruster_build_lut_f32(const float* points /*[n_pts]*/, int32_t n_pts,
                               float* lut /*[n_out]*/, int32_t n_out, void* stream);

/* A3/A6/A10  per-episode uniform re-draws of rows of an (N, ld) tensor:       */
/*   dst[env_ids[j], c] = base[c] + (lo[c] + u*(hi[c]-lo[c]))                  */
/* u from Philox4x32-10 keyed (seed; env_id, counter, stream_id+c/4).          */
/*     [ref: OIGE/envs/USV/Hydrodynamics.py:136-174, ThrusterDynamics.py:112-127, */
/*           OIGE/tasks/USV/USV_disturbances.py:127-151]                      */
int usv_randomize_rows_f32(float* dst, int64_t ld, const int64_t* env_ids, int64_t n_ids,
                           int32_t ncols, const float* base /*[ncols]*/, const float* lo /*[ncols]*/,
                           const float* hi /*[ncols]*/, int32_t log_space,
                           uint64_t seed, uint64_t counter, uint32_t stream_id, void* stream);

/* ------------------------------------------------------------------------- */
/* Fused env step (Variant A, classic CaptureXY) == VecEnvRLGames.step         */
/*     [ref: OIGE/envs/vec_env_rlgames.py:120-217; SNAP/USV_Virtual.py:571-866; */
/*           SNAP/USV_capture_xy.py:80-275; SNAP/USV_task_rewards.py:40-76,380-540; */
/*           OIGE/tasks/USV/USV_disturbances.py; OIGE/tasks/base/rl_task.py:283-303] */
/* State is structure-of-arrays, tiled by warp (AoSoA): envs are grouped in tiles of 32 and inside a tile the
 * fields are consecutive 128-byte lines:  field f of env i lives at
 *     base[((i >> 5) * COUNT + f) * 32 + (i & 31)]          (COUNT = USV_S_COUNT / USV_C_COUNT / USV_ST_COUNT).
 * `*_stride` is the capacity in envs (a multiple of 32, >= n); buffers hold stride*COUNT floats, 128 B aligned. */

/* dynamic fields (read+written every step) */
enum {
  USV_S_X = 0, USV_S_Y, USV_S_PSI, USV_S_VX, USV_S_VY, USV_S_R,
  USV_S_THR_L, USV_S_THR_R,      /* DynamicsFirstOrder.current_forces            */
  USV_S_PREV_D,                  /* prev_position_dist / prev_position_error     */
  USV_S_PREV_W,                  /* Penalties.prev_state["angular_velocity"]     */
  USV_S_PREV_ASUM,               /* sum(Penalties.prev_actions)                  */
  USV_S_GOAL_CNT,                /* int32 bit pattern: CaptureXYTask._goal_reached */
  USV_S_PROGRESS,                /* int32 bit pattern: RLTask.progress_buf       */
  USV_S_COUNT
};
/* per-episode constants (read every step, rewritten on reset) */
enum {
  USV_C_TX = 0, USV_C_TY,        /* task._target_positions                       */
  USV_C_MASS,                    /* MDD.platforms_mass                           */
  USV_C_LIN_U, USV_C_LIN_V, USV_C_LIN_R,    /* hydrodynamics.linear_damping[:, (0,1,5)]    */
  USV_C_QUAD_U, USV_C_QUAD_V, USV_C_QUAD_R, /* hydrodynamics.quadratic_damping[:, (0,1,5)] */
  USV_C_KDRAG,                   /* hydrodynamics.drag_scale                     */
  USV_C_THR_ML, USV_C_THR_MR,    /* effective left/right thruster multipliers    */
  USV_C_KIZ,                     /* yaw-inertia scale                            */
  USV_C_FCX, USV_C_FCY,          /* UF.disturbance_forces_const                  */
  USV_C_FXF, USV_C_FYF, USV_C_FXS, USV_C_FYS, USV_C_FAMP,
  USV_C_TC, USV_C_TF, USV_C_TS, USV_C_TAMP, /* TD.*                              */
  USV_C_COUNT
};
/* optional per-episode statistics accumulators (episode_sums), SoA as well */
enum {
  USV_ST_DISTANCE_REWARD = 0, USV_ST_ALIGNMENT_REWARD, USV_ST_VELOCITY_REWARD,
  USV_ST_POSITION_ERROR, USV_ST_VELOCITY_NORM, USV_ST_BOUNDARY_PENALTY, USV_ST_BOUNDARY_DIST,
  USV_ST_LINEAR_VEL_PENALTY, USV_ST_ANGULAR_VEL_PENALTY, USV_ST_ANGULAR_VEL_VARIATION_PENALTY,
  USV_ST_ENERGY_PENALTY, USV_ST_ACTION_VARIATION_PENALTY,
  USV_ST_NORMED_LINEAR_VEL, USV_ST_NORMED_ANGULAR_VEL, USV_ST_ACTIONS_SUM,
  USV_ST_COUNT
};

enum { USV_REWARD_LINEAR = 0, USV_REWARD_SQUARE = 1, USV_REWARD_EXPONENTIAL = 2 };

/* closed set of penalty lambda forms that appear in cfg/task/USV (SURVEY A9)  */
enum {
  USV_PEN_OFF = 0,
  USV_PEN_NEG_SUM = 1,          /* -sum(x)*c1 + c2                               */
  USV_PEN_EXP_NEG_SUMSQ = 2,    /* (exp(-sum(x^2)) - 1)*c1                       */
  USV_PEN_NEG_ABS = 3,          /* -abs(x)*c1 + c2        (norm for vectors)     */
  USV_PEN_NEG_DEADZONE = 4,     /* -clamp(abs(x)-d, min=0)*c1                    */
  USV_PEN_EXP_NEG_ABS = 5       /* (exp(-k*abs(x)) - 1)*c1                       */
};
typedef struct { int32_t form; float c1; float c2; float k; } UsvPenaltyTerm;

typedef struct {
  uint64_t seed;               /* Philox key                                    */
  uint64_t step_counter;       /* global control-step index (Philox counter)    */
  int64_t  env_id_offset;      /* global id of local env 0 (rank sharding)      */
  /* simulation */
  float dt;                    /* sim.dt                                        */
  int32_t n_substeps;          /* env.controlFrequencyInv                       */
  int32_t max_episode_length;
  float clip_actions;          /* env.clipActions                               */
  float clip_obs;              /* env.clipObservations.state                    */
  /* planar rigid body standing in for PhysX (DESIGN.md "integrator")          */
  float izz;                   /* base yaw inertia [kg m^2] (config constant)   */
  float thr_y_left, thr_y_right; /* thruster mount y  (heron.urdf:167,242)      */
  float lag_alpha;             /* fp32 exp(-dt/timeConstant)                    */
  /* env origins (world frame; only the sinusoidal disturbances read world positions):
   * origin(i) = (grid_row_offset - (i / envs_per_row)*env_spacing, (i % envs_per_row)*env_spacing - grid_col_offset)
   * envs_per_row == 0 -> all origins 0 */
  float env_spacing, grid_row_offset, grid_col_offset;
  int32_t envs_per_row;
  /* hydrodynamics (planar components u,v,r of the 6-vectors) */
  float lin_fwd[3];
  float offset_linear_damping, offset_lin_forward_damping_speed, offset_nonlin_damping, scaling_damping;
  int32_t use_drag_scale;
  /* thruster LUT */
  int32_t n_lut;
  /* action path  [ref: SNAP/USV_Virtual.py:571-617 ; OIGE/tasks/USV_Virtual.py:1042-1101] */
  int32_t action_affine;       /* 0 classic (raw +-1 to LUT) ; 1 live u=0.5(a+1) */
  int32_t action_noise;  float action_noise_min, action_noise_max;
  float action_bias;           /* live: initial_action_bias while the host-side call counter is below its limit */
  int32_t penalties_use_u;     /* live: penalties see u in [0,1] instead of the raw action */
  int32_t first_call;          /* 1 on the very first step: Penalties.prev_state is None -> deltas are 0 */
  /* observation noise [ref: OIGE/tasks/USV/USV_disturbances.py:533-601] */
  int32_t noise_pos;     float pos_noise_min, pos_noise_max;
  int32_t noise_vel;     float vel_noise_min, vel_noise_max;
  int32_t noise_heading; float heading_noise_min, heading_noise_max;
  /* disturbances evaluated every sub-step */
  int32_t use_const_force, use_sin_force, use_const_torque, use_sin_torque;
  /* CaptureXY task [ref: SNAP/USV_capture_xy.py ; USV_task_parameters.py:17-57] */
  float position_tolerance; int32_t kill_after_n_steps_in_tolerance;
  float kill_dist, boundary_cost, goal_reward, time_reward;
  float goal_speed_gate;       /* 0.05 in the classic task                      */
  int32_t reward_mode; float position_scale, exponential_reward_coeff;
  float align_la1, align_la2, align_la3;
  /* penalties [ref: SNAP/USV_task_rewards.py:380-540] */
  UsvPenaltyTerm pen_linear_vel, pen_angular_vel, pen_angular_vel_variation, pen_energy, pen_action_variation;
  /* ---- reset-time randomisation (A3, A6, A10, A11, A14, A19) ---- */
  float goal_random_position; int32_t retarget_on_reset;
  float spawn_min_dist, spawn_max_dist;    /* after curriculum, set by host     */
  int32_t spawn_about_origin;              /* live task: the spawn annulus is centred on the env origin, not the target */
  int32_t retarget_after_spawn;            /* live reset_idx order: get_spawns (around the OLD target) first, set_targets last
                                              (OIGE/tasks/USV_Virtual.py:1542,1622); classic: target first */
  int32_t reset_pose_external;             /* scene replay (OIGE/tasks/USV_Virtual.py:1395-1458): pose, velocity and target of a
                                              resetting env were written by the host; the kernel only re-draws the dynamics
                                              randomisation and clears the episode bookkeeping */
  float spawn_vel_range;                   /* 1.5: vx,vy ~ U(-1.5,1.5)          */
  int32_t mass_rand; float mass_min, mass_max, mass_base;
  int32_t drag_rand; float lin_base[3], quad_base[3], lin_rand[3], quad_rand[3];
  int32_t kdrag_rand; float kdrag_min, kdrag_max; int32_t kdrag_log;
  int32_t thr_rand, thr_separate; float thr_rand_frac, thr_left_frac, thr_right_frac;
  int32_t mass_coupling; float couple_mass_max, couple_thr_a, couple_kiz_min, couple_kiz_max;
  int32_t couple_targets;                  /* which scalars the mass-driven coupling overrides: bit 0 drag_scale, bit 1 thruster,
                                              bit 2 yaw_inertia (7 = the shipped target list)  [ref: OIGE/tasks/USV_Virtual.py:393-411] */
  int32_t kiz_rand, kiz_log;               /* independent episode-wise k_Iz ~ U / log-U [couple_kiz_min, couple_kiz_max] when yaw_inertia is
                                              not a coupling target  [ref: OIGE/tasks/USV_Virtual.py:153-170,193-214,1532-1533] */
  int32_t use_water_current; float flow_vel_xy[2];   /* env.water_current: drag acts on the velocity relative to a uniform world-frame
                                              flow  [ref: OIGE/envs/USV/Hydrodynamics.py:224-237 ; OIGE/tasks/USV_Virtual.py:444-445,1111-1116] */
  float force_const_min, force_const_max, force_sin_min, force_sin_max;
  float force_min_freq, force_max_freq, force_min_shift, force_max_shift;
  float torque_const_min, torque_const_max, torque_sin_min, torque_sin_max;
  float torque_min_freq, torque_max_freq, torque_min_shift, torque_max_shift;
  int32_t use_force_disturbance, use_torque_disturbance;
} UsvStepParams;

typedef struct {
  float*   state;   int64_t state_stride;   /* [stride/32][USV_S_COUNT][32]                    */
  float*   consts;  int64_t consts_stride;  /* [stride/32][USV_C_COUNT][32]                    */
  float*   stats;   int64_t stats_stride;   /* [stride/32][USV_ST_COUNT][32] or NULL (stats off) */
  int64_t* reset_buf;                        /* [n] RLTask.reset_buf (in: reset now; out: done) */
  const float* lut_left;                     /* [n_lut]                                        */
  const float* lut_right;                    /* [n_lut]                                        */
  uint32_t* nonfinite_flag;                  /* device word, OR-ed with 1 on NaN/Inf obs/rew, or NULL */
  /* optional device-side addend to UsvStepParams.step_counter (NULL = 0): lets a captured CUDA graph of control steps advance
   * its Philox step index between replays.  Honoured by usv_step_fused_f32 / usv_rollout_fused_f32 (classic task). */
  const uint64_t* step_offset;
} UsvEnvBuffers;

/* one control step for n envs: reset-if-flagged, action -> thrust target, n_substeps of
 * {lag, forces, integrate}, obs (clamped), reward + penalties, kills, progress/done.      */
int usv_step_fused_f32(const UsvEnvBuffers* b, const float* actions /*[n,2]*/,
                       float* obs /*[n,13]*/, float* rew /*[n]*/,
                       int64_t n, const UsvStepParams* p, void* stream);

/* A7 stand-alone: the planar rigid body behind the simulator surface USVVirtual expects (HeronView.get_world_poses / get_velocities /
 * set_*, <body>.apply_forces_and_torques_at_pos, world.step())  [ref: OIGE/tasks/USV_Virtual.py:772-774,1119-1133,1567-1572].
 * wrench[n,3] accumulates (Fx, Fy, Tz) in the body frame over the apply_* calls of one physics step (forces / torques are the
 * reference's [n,3] tensors, only their planar components enter; a force applied at the body-frame offset (offset_x, offset_y)
 * -- a thruster mount -- adds r x F; is_global: rotate world-frame forces by R(psi)^T, pose[n,3] = (x, y, psi) then required);
 * usv_planar_rigid_step_f32 integrates one sim dt with the fused step's semi-implicit Euler and clears the wrench.            */
int usv_planar_wrench_accumulate_f32(float* wrench /*[n,3]*/, const float* forces /*[n,3] or NULL*/, const float* torques /*[n,3] or NULL*/,
                                     const float* pose /*[n,3] or NULL*/, float offset_x, float offset_y, int32_t is_global, int64_t n,
                                     void* stream);
int usv_planar_rigid_step_f32(float* pose /*[n,3]*/, float* vel /*[n,3]: vx, vy (world), r*/, float* wrench /*[n,3]*/,
                              const float* mass /*[n]*/, const float* izz /*[n]*/, float dt, int64_t n, void* stream);

/* A9/A16-A18 stand-alone: the classic CaptureXYTask's get_state_observations / compute_reward / update_kills and
 * Penalties.compute_penalty on the CALLER's state tensors -- the same device code as the task part of usv_step_fused_f32, so the
 * reference's task classes can be fed identical state tensors and compared output by output.
 *   [ref: SNAP/USV_capture_xy.py:80-97 (obs), :101-227 (reward), :231-275 (kills) ; SNAP/USV_task_rewards.py:40-76,422-506 ;
 *         SNAP/USV_core.py:31-54 (observation tensor, "local" frame)]
 * `what` selects the calls; like the reference, compute_reward advances the goal counter and prev_position_dist, compute_penalty
 * advances prev_state / prev_actions, the other two are pure.  All tensors row-major fp32 unless noted; optional ones may be NULL. */
enum { USV_CXY_OBS = 1, USV_CXY_REWARD = 2, USV_CXY_PENALTY = 4, USV_CXY_KILLS = 8, USV_CXY_ALL = 15 };
typedef struct {
  const float* position;          /* [n,2] current_state["position"]                                              */
  const float* heading;           /* [n,2] current_state["orientation"] = (cos, sin) of the yaw                   */
  const float* linear_velocity;   /* [n,2] world frame                                                            */
  const float* angular_velocity;  /* [n]                                                                          */
  const float* actions;           /* [n,2] what Penalties sees (PENALTY only)                                     */
  const float* target;            /* [n,2] _target_positions                                                      */
  const uint8_t* just_reset;      /* [n] 1 = env in just_had_been_reset (distance reward zeroed) or NULL          */
  float* prev_position_dist;      /* [n] in/out (REWARD)                                                          */
  float* prev_angular_velocity;   /* [n] in/out (PENALTY): prev_state["angular_velocity"]                         */
  float* prev_action_sum;         /* [n] in/out (PENALTY): sum(prev_actions, -1)                                  */
  int32_t* goal_reached;          /* [n] in/out (REWARD updates, KILLS reads): _goal_reached                      */
  float* obs;                     /* [n,13] out, clamped to +-clip_obs like VecEnvRLGames._process_data           */
  float* reward;                  /* [n] out: compute_reward's return value (task reward, penalties NOT included) */
  float* reward_terms;            /* [n,3] out or NULL: distance, alignment, speed reward                         */
  float* penalty;                 /* [n] out: compute_penalty's return value                                      */
  float* penalty_terms;           /* [n,5] out or NULL: linear vel, angular vel, its variation, energy, action variation */
  int64_t* die;                   /* [n] out: update_kills                                                        */
  float kill_dist;                /* curriculum-resolved kill distance of this step (update_kills(step))          */
  uint32_t what;                  /* USV_CXY_* bits                                                               */
  int32_t first_reward;           /* prev_position_dist is None: the progress term starts from the current distance */
  int32_t first_penalty;          /* prev_state / prev_actions are None: both variations are zero                 */
} UsvCaptureXYIO;
int usv_capturexy_obs_reward_done_f32(const UsvCaptureXYIO* io, int64_t n, const UsvStepParams* p, void* stream);

/* T control steps in ONE launch with the state held in registers between steps;
 * actions[T,n,2] are given up-front (open loop), outputs are [T,n,...]; obs/rew/done may be NULL
 * (then only the final state is written).  step_counter advances by 1 per step.           */
int usv_rollout_fused_f32(const UsvEnvBuffers* b, const float* actions /*[T,n,2]*/,
                          float* obs /*[T,n,13] or NULL*/, float* rew /*[T,n] or NULL*/,
                          int64_t* done /*[T,n] or NULL*/, int32_t T,
                          int64_t n, const UsvStepParams* p, void* stream);

/* force/torque probe of the fused kernel's planar model (parity hook): for given planar states
 * returns the body-frame drag (u,v,r), thrust wrench and world accelerations of ONE sub-step.  */
int usv_planar_forces_f32(const UsvEnvBuffers* b, float* out /*[n,8]: du,dv,dr,Fx,Fy,Tz,ax,ay*/,
                          int64_t n, const UsvStepParams* p, void* stream);

/* ------------------------------------------------------------------------- */
/* Variant B: live CaptureXY with 16 static obstacles and a per-env potential field (SURVEY rows B1-B6)            */
/*     [ref: OIGE/tasks/USV/USV_capture_xy_static_obs.py ; OIGE/tasks/USV/d_multi_gemini.py ;                      */
/*           OIGE/tasks/USV_Virtual.py:771-1101,1223-1240,1502-1662 ; OIGE/tasks/USV/USV_core.py:55-125]           */
#define USV_B_OBS 33          /* 3 + 20 (5 task scalars + 5 nearest obstacles x 3) + prev_action 2 + priv 8        */
#define USV_B_OBSTACLES 16    /* CaptureXYTask.big                                                                 */
#define USV_B_CLOSEST 5
#define USV_B_GRID 150        /* BatchedMapGPU: 150 x 150 cells of 0.2 m over a 30 m map, row = y, column = x      */

/* extra dynamic per-env fields of the live task (AoSoA like the base state) */
enum {
  USV_BS_PREV_H = 0,          /* prev_heading_error                                                                */
  USV_BS_PREV_POT,            /* prev_potential                                                                    */
  USV_BS_OUTCOME,             /* int32 bit pattern: bit0 _done_success, bit1 _done_collision                       */
  USV_BS_COUNT
};
/* extra per-episode constants of the live task */
enum {
  USV_BC_COM_X = 0, USV_BC_COM_Y, USV_BC_COM_Z,   /* MDD.platforms_CoM (observed only)                             */
  USV_BC_OBST = 3,            /* xunlian_pos[:, j, 0:2] at USV_BC_OBST + 2*j, +1   (env-local frame)               */
  USV_BC_COUNT = USV_BC_OBST + 2 * USV_B_OBSTACLES
};
/* optional episode_sums of the live task [ref: USV_capture_xy_static_obs.py:130-187,720-765 ;                     */
/* OIGE/tasks/USV/USV_task_rewards.py Penalties.update_statistics ; OIGE/tasks/USV_Virtual.py:1187-1220]           */
enum {
  USV_BST_TOTAL_REWARD = 0, USV_BST_DISTANCE_REWARD, USV_BST_ALIGNMENT_REWARD, USV_BST_HEADING_IMPROVE_REWARD,
  USV_BST_POTENTIAL_SHAPING_REWARD, USV_BST_SPEED_REWARD, USV_BST_ANGULAR_REWARD, USV_BST_TURN_HAZARD_PENALTY,
  USV_BST_GOAL_REWARD, USV_BST_COLLISION_REWARD, USV_BST_TIME_REWARD, USV_BST_POSITION_ERROR, USV_BST_BOUNDARY_PENALTY,
  USV_BST_DANGER_MEAN, USV_BST_DANGER_HI_RATE, USV_BST_G_GATE_MEAN,
  USV_BST_LINEAR_VEL_PENALTY, USV_BST_ANGULAR_VEL_PENALTY, USV_BST_ANGULAR_VEL_VARIATION_PENALTY,
  USV_BST_ENERGY_PENALTY, USV_BST_ACTION_VARIATION_PENALTY,
  USV_BST_NORMED_LINEAR_VEL, USV_BST_NORMED_ANGULAR_VEL, USV_BST_ACTIONS_SUM,
  USV_BST_CMD_NEG_RATE, USV_BST_THRUSTER_FORCE_NEG_RATE, USV_BST_U_MEAN, USV_BST_U_LOW_RATE, USV_BST_U_SUM,
  USV_BST_COUNT      /* "success" / "collision" are read from USV_BS_OUTCOME before the reset (USV_Virtual.py:1508-1516,1581-1588) */
};

enum { USV_PRIV_RAW = 0, USV_PRIV_CENTERED = 1, USV_PRIV_MINMAX = 2 };
/* tasks behind the live USVVirtual's 33-dim observation (task_data = obs[3:23]); 1-3 are SURVEY row T (Tier 3):
 *   [ref: OIGE/tasks/USV/USV_go_to_pose.py:81-209 ; USV_keep_xy.py:80-179 ; USV_track_xy_velocity.py:64-128 ;
 *         OIGE/tasks/USV/USV_task_rewards.py:170-325 ; USV_task_parameters.py:95-177]                                    */
enum { USV_TASK_CAPTURE_OBSTACLES = 0, USV_TASK_GO_TO_POSE = 1, USV_TASK_KEEP_XY = 2, USV_TASK_TRACK_XY_VELOCITY = 3 };
/* per-episode task constants of tasks 1-3 live in the (otherwise unused) obstacle slots of bconsts */
enum { USV_BC_TARGET_HEADING = 3 /* GoToPose: _target_headings */, USV_BC_TARGET_VX = 3, USV_BC_TARGET_VY = 4 /* TrackXYVelocity */ };

typedef struct {
  /* privileged tail [ref: OIGE/tasks/USV_Virtual.py:837-984 ; USV_disturbances.py:153-194] */
  int32_t priv_mode;            /* USV_PRIV_*                                                       */
  int32_t mass_obs_relative;    /* 1: (m - base)/max(|base|,eps) ; 0: raw                            */
  int32_t com_obs_scaled;       /* 1: com / (scale + eps)                                            */
  float com_scale_eps[3];       /* fp32 (scale + 1e-6)                                               */
  /* [k_drag, thr_L, thr_R, k_Iz]: raw -> x ; centered -> clamp((x - a)/b, +-1) with a = nominal, b = max(|min-nom|,|max-nom|,eps) ;
   * minmax -> active ? clamp(2*((x - a)/b) - 1, +-1) : 0 with a = min, b = max - min  (USV_Virtual.py:97-151,905-970) */
  float priv_a[4], priv_b[4]; int32_t priv_active[4];
  /* CoM re-draw at reset [ref: USV_disturbances.py:88-124] (observation only: the planar integrator has no CoM offset) */
  int32_t com_rand; float com_base[3], com_disp[3];   /* com_rand: 0 off, 1 box +-com_disp per axis, 2 legacy XY disc of radius com_disp[0] */
  /* task */
  float collision_threshold;    /* 1.2  (:103)                                                       */
  float map_size;               /* 30.0                                                              */
  int32_t fixed_horizon_eval;   /* is_done ignores `die` (USV_Virtual.py:1229-1233)                  */
  /* Tier-3 tasks (task != 0): no obstacles / potential field; UsvStepParams.reward_mode, exponential_reward_coeff and
   * position_scale parameterise the position (or velocity) reward                                    */
  int32_t task;                 /* USV_TASK_*                                                        */
  int32_t heading_reward_mode;  /* GoToPoseReward.heading_reward_mode (USV_REWARD_*)                  */
  float heading_exponential_reward_coeff, heading_scale, sig_gain;
  float goal_random_velocity, lin_vel_tolerance;   /* TrackXYVelocityParameters                       */
  /* mass.masscom_obs_source == "base" (evaluation ablation, USV_Virtual.py:840-880; USV_disturbances.py:196-250): the tail shows
   * every env the BASE mass / CoM encodings and the encodings of priv_neutral[] (minmax: mid-range, else 1.0) instead of the
   * simulated values; the dynamics stay randomised                                                   */
  int32_t masscom_obs_base; float priv_neutral[4];
  /* width of the privileged tail: 8 = [mass, CoM(3), k_drag, thr_L, thr_R, k_Iz] (obs 33 wide) or 4 = [mass, CoM(3)] (obs 29 wide:
   * env.mass_dim / priv_dim = 4)  [ref: OIGE/tasks/USV_Virtual.py:484-488,854-856 ; OIGE/tasks/USV/USV_core.py:23-52,127-170].
   * The obs tensor handed to usv_step_live_f32 is [n, 25 + priv_dim]; 0 reads as 8 (round-1 callers). */
  int32_t priv_dim;
} UsvLiveParams;

typedef struct {
  float* bstate;  int64_t bstate_stride;   /* [stride/32][USV_BS_COUNT][32]                              */
  float* bconsts; int64_t bconsts_stride;  /* [stride/32][USV_BC_COUNT][32]                              */
  float* bstats;  int64_t bstats_stride;   /* [stride/32][USV_BST_COUNT][32] or NULL                     */
  float* field;                            /* [n][150][150] global_potential_field                       */
  /* "a reset happened" epoch words, uint64[2] (reference quirk: reset() sets prev_potential=None for EVERY env, so the
   * potential shaping of the next reward is zero for all envs).  The step kernel of control step s stores s+1 into word
   * (s+1)&1 when any env finishes; the kernel of step s+1 treats word[(s+1)&1] == its step_counter as "some env was reset
   * on entry" (two words: readers and writers of one launch never share a word).  The host stores step_counter into word
   * step_counter&1 when it sets reset_buf itself. */
  uint64_t* reset_epoch;
} UsvLiveBuffers;

/* one control step of the live task for n envs.  Same dynamics / action path as usv_step_fused_f32 (p->action_affine etc.);
 * env resets are split: the in-kernel part re-draws the episode constants and the spawn pose, obstacles + potential field of
 * the envs flagged in reset_buf must have been rebuilt by usv_live_reset_scene_f32 BEFORE this call.                        */
int usv_step_live_f32(const UsvEnvBuffers* b, const UsvLiveBuffers* lb, const float* actions /*[n,2]*/,
                      float* obs /*[n,33]*/, float* rew /*[n]*/, int64_t n, const UsvStepParams* p,
                      const UsvLiveParams* lp, void* stream);

/* B5 + B6: for every env flagged in b->reset_buf re-draw the 16 obstacles (rejection sampling against the spawn point the
 * step kernel will draw for the same (seed, env, step) and against the CURRENT target) and rebuild its potential field.
 * The batch-global maxima of the reference's builder (d_multi_gemini.py:204-210,257-260) are taken over the envs that reset
 * in this call.  Call before usv_step_live_f32 with the same p->step_counter.  cell_centres = torch.linspace(-14.9,14.9,150);
 * workspace: usv_live_scene_workspace_bytes(n) bytes, 16 B aligned (counters, the compacted reset list and 32 B of per-scene
 * statistics that the cost kernel hands to the field kernel).
 *     [ref: USV_capture_xy_static_obs.py:936-1060 ; d_multi_gemini.py:66-271]                                               */
int64_t usv_live_scene_workspace_bytes(int64_t n);
int usv_live_reset_scene_f32(const UsvEnvBuffers* b, const UsvLiveBuffers* lb, const float* cell_centres /*[150]*/,
                             void* workspace, int64_t n, const UsvStepParams* p, void* stream);
/* B6 alone on a dense batch (BatchedMapGPU.compute_occupancy_and_sdf -> compute_cost_field_wavefront -> compute_potential_field);
 * workspace: usv_live_scene_workspace_bytes(m) bytes, 16 B aligned */
int usv_live_build_fields_f32(const float* obstacles /*[m,16,2]*/, const float* targets /*[m,2]*/,
                              const float* cell_centres /*[150]*/, float* field /*[m,150,150]*/,
                              float* cost_out /*[m,150,150] raw cost-to-go or NULL*/, void* workspace, int64_t m, void* stream);

/* ------------------------------------------------------------------------- */
/* P1  A2CBase.discount_values (GAE) + returns                                */
/*     [ref: RLG/common/a2c_common.py:525-540,761-763]                        */
int ppo_gae_f32(const float* rewards /*[T,n]*/, const float* values /*[T,n]*/,
                const uint8_t* dones /*[T,n] flag entering step t*/, const float* last_values /*[n]*/,
                const uint8_t* last_dones /*[n]*/, float gamma, float tau,
                float* advantages /*[T,n]*/, float* returns /*[T,n] or NULL*/,
                int32_t T, int64_t n, void* stream);

/* P6  play_steps bookkeeping of one control step, fused: rewards_out = rew*scale (DefaultRewardsShaper), dones_out = uint8(dones),   */
/*   current_rewards += rew, current_lengths += 1, sums over the finished envs into episode_acc (fp64: return, length, count) and    */
/*   into the two windowed AverageMeters (mean, current_size), then the finished envs' running values are zeroed.                    */
/*     [ref: RLG/common/a2c_common.py:708-747 ; RLG/algos_torch/torch_ext.py:281-307]                                                */
int ppo_rollout_bookkeep_f32(const float* rew /*[n]*/, const int64_t* dones /*[n]*/, float scale, float* rewards_out /*[n]*/,
                             uint8_t* dones_out /*[n]*/, float* cur_rew /*[n]*/, float* cur_len /*[n]*/, double* episode_acc /*[3]*/,
                             float* meter_r, float* meter_r_size, float* meter_l, float* meter_l_size, float max_size, int64_t n,
                             void* stream);

/* ------------------------------------------------------------------------- */
/* P4/P5  USV_PPOcontinuous_MLP: shared-trunk actor-critic                     */
/*   obs(D) -> RunningMeanStd norm (clamp +-5) -> Linear(D,128)+tanh -> Linear(128,128)+tanh -> {mu: Linear(128,2),  */
/*   value: Linear(128,1)}, state-independent logstd parameter (2,)                                                */
/*     [ref: RLG/algos_torch/models.py:366-401 ; RLG/algos_torch/network_builder.py:1480-1678 ;                    */
/*           RLG/algos_torch/running_mean_std.py:81-117 ; OIGE/cfg/train/USV/USV_PPOcontinuous_MLP.yaml]           */
/* All parameters live in ONE flat fp32 buffer in rl_games' model.parameters() order (Adam state and the gradient  */
/* all-reduce work on the same span):                                                                              */
/*   sigma[2] | actor_mlp.0.weight[128,D] | .bias[128] | actor_mlp.2.weight[128,128] | .bias[128] |                 */
/*   value.weight[1,128] | value.bias[1] | mu.weight[2,128] | mu.bias[2]            (18 693 floats for D = 13)      */
#define PPO_HIDDEN 128
#define PPO_ACTIONS 2
#define PPO_MAX_OBS 64
int64_t ppo_param_count(int32_t obs_dim);

/* rollout inference (is_train=False): a = mu + sigma*N(0,1) (Philox, Box-Muller), neglogp, de-normalised value   */
/* any output pointer may be NULL; with actions==NULL no sampling happens (get_values)                            */
int ppo_policy_forward_f32(const float* params, const float* obs /*[M,D]*/, int32_t obs_dim,
                           const float* obs_mean /*[D] fp32 copy of the fp64 running mean*/, const float* obs_var /*[D]*/,
                           const float* value_mean /*[1]*/, const float* value_var /*[1]*/,
                           uint64_t seed, uint64_t counter, const uint64_t* counter_offset /*device addend to `counter` or NULL (graph replay)*/,
                           int64_t row_offset,
                           float* actions /*[M,2]*/, float* neglogp /*[M]*/, float* values /*[M] de-normalised*/,
                           float* mus /*[M,2]*/, float* sigmas /*[M,2]*/, int64_t M, void* stream);

/* the same contract on the tcgen05 tensor cores (TF32 operands, fp32 accumulation in TMEM, tanh.approx): ~1e-3 relative
 * of the fp32 entry point above; obs_dim <= 47: the first GEMM runs with K = 16 (obs_dim <= 15, classic task) or K = 48 (live task, 33),
 * one padded K column carries the first-layer bias */
int64_t ppo_packed_weight_floats(void);
/* params -> weight operand tiles pre-arranged in the kernels' shared-memory order (staged by TMA bulk copies); call after
 * every parameter update.  `packed`: ppo_packed_weight_floats() floats, 16 B aligned */
int ppo_pack_weights_tc(const float* params, int32_t obs_dim, float* packed, void* stream);
int ppo_policy_forward_tc(const float* params, const float* packed, const float* obs, int32_t obs_dim, const float* obs_mean, const float* obs_var,
                          const float* value_mean, const float* value_var, uint64_t seed, uint64_t counter, const uint64_t* counter_offset,
                          int64_t row_offset, float* actions, float* neglogp, float* values, float* mus, float* sigmas, int64_t M, void* stream);

typedef struct {
  float e_clip;            /* 0.2  */
  float critic_coef;       /* 0.5 (the loss uses 0.5*c_loss*critic_coef) */
  float entropy_coef;      /* 0.0  */
  float bounds_loss_coef;  /* 1e-4 */
  float bound_soft;        /* 1.1  */
  int32_t clip_value;      /* 1    */
} PpoLossParams;

/* layout of the small statistics vector the train kernels fill (means over the minibatch) */
enum { PPO_STAT_A_LOSS = 0, PPO_STAT_C_LOSS, PPO_STAT_ENTROPY, PPO_STAT_B_LOSS, PPO_STAT_KL, PPO_STAT_LOSS,
       PPO_STAT_GRAD_NORM, PPO_STAT_LR, PPO_STAT_COUNT };

/* one PPO minibatch: forward (train mode), clipped surrogate / clipped value / bound losses, backward.           */
/*   [ref: RLG/algos_torch/a2c_continuous.py:78-196 ; RLG/common/common_losses.py:10-48 ; torch_ext.py:27-36]     */
/* grads[P+PPO_STAT_COUNT]: d(loss)/d(params) followed by the statistics (so one all-reduce carries both);        */
/* new_mu/new_sigma are what PPODataset.update_mu_sigma stores back.  scratch: ppo_train_scratch_floats(D) floats */
int64_t ppo_train_scratch_floats(int32_t obs_dim);
int ppo_minibatch_grad_f32(const float* params, const float* obs /*[M,D]*/, int32_t obs_dim,
                           const float* obs_mean, const float* obs_var,
                           const float* actions /*[M,2]*/, const float* old_neglogp /*[M]*/, const float* advantages /*[M]*/,
                           const float* old_values /*[M] normalised*/, const float* returns /*[M] normalised*/,
                           float* old_mu /*[M,2] in: KL reference, out: new mu*/, float* old_sigma /*[M,2] in/out*/,
                           const PpoLossParams* lp, float* grads /*[P+PPO_STAT_COUNT]*/, float* scratch,
                           int64_t M, void* stream);

/* the same minibatch step with every GEMM (forward, dH, and the weight gradients, which accumulate in TMEM across the
 * CTA's tiles) on the tcgen05 tensor cores in TF32; obs_dim <= 47 */
int ppo_minibatch_grad_tc(const float* params, const float* packed, const float* obs, int32_t obs_dim, const float* obs_mean, const float* obs_var,
                          const float* actions, const float* old_neglogp, const float* advantages, const float* old_values,
                          const float* returns, float* old_mu, float* old_sigma, const PpoLossParams* lp, float* grads,
                          float* scratch, float* workspace /*ppo_train_tc_workspace_floats(M) floats, 16 B aligned*/,
                          int64_t M, void* stream);
int64_t ppo_train_tc_workspace_floats(int64_t M);


/* gradient-norm clip + Adam + adaptive-KL learning rate, all on device (no kl.item() host sync)                  */
/*   [ref: RLG/common/a2c_common.py:308-330 ; torch.optim.Adam ; RLG/common/schedulers.py:19-32]                  */
typedef struct {
  float beta1, beta2, eps;        /* 0.9, 0.999, 1e-8 */
  float grad_norm;                /* 1.0; <=0 disables truncation */
  float inv_world;                /* 1/world_size applied to the (summed) gradient and statistics */
  int32_t adaptive_lr;            /* 1: lr/=1.5 if kl > 2*thr ; lr*=1.5 if kl < 0.5*thr ; clamp [min_lr,max_lr] */
  float kl_threshold, min_lr, max_lr;
} PpoAdamParams;
int ppo_adam_step_f32(float* params, float* grads /*[P+PPO_STAT_COUNT], scaled in place*/, float* exp_avg, float* exp_avg_sq,
                      float* lr /*device float[2]: [0] current lr (updated), [1] scratch*/,
                      int32_t* step /*device int32[2]: [0] Adam step count (incremented), [1] scratch*/,
                      int64_t P, const PpoAdamParams* ap, void* stream);
/* one whole minibatch step on a single rank: ppo_minibatch_grad_tc + ppo_adam_step_f32 + ppo_pack_weights_tc with the second-stage
 * reduction, clip, Adam, adaptive lr, the lr / step roll and the refresh of the packed operand tiles fused into ONE cooperative launch:
 * T1 + T2 + tail = 3 launches per minibatch instead of 7 */
int ppo_minibatch_step_tc(float* params, float* packed, const float* obs, int32_t obs_dim, const float* obs_mean, const float* obs_var,
                          const float* actions, const float* old_neglogp, const float* advantages, const float* old_values,
                          const float* returns, float* old_mu, float* old_sigma, const PpoLossParams* lp, float* grads, float* scratch,
                          float* workspace, float* exp_avg, float* exp_avg_sq, float* lr, int32_t* step, const PpoAdamParams* ap,
                          int64_t M, void* stream);

/* ------------------------------------------------------------------------- */
/* Gradient all-reduce over NVLink peer memory (SURVEY 8(e) collective (1)+(2)): replaces dist.all_reduce(grads) of
 *   [ref: RLG/common/a2c_common.py:308-323] with ONE kernel per minibatch that exchanges the span through CUDA-IPC mapped
 *   windows (P2P stores / loads, release / acquire flags), sums in rank order (bit-identical on every rank) and never leaves the
 *   stream -- so the PPO update phase stays one CUDA graph on every rank.  Windows are the one thing this library allocates
 *   itself (cudaMalloc: IPC handles need whole allocations); the 64-byte handles travel through torch.distributed. */
typedef struct {
  float* windows[16];          /* windows[r] = rank r's window mapped into THIS process (windows[rank] = the local one) */
  int64_t cap;                 /* floats per payload buffer (>= count)                                          */
  int32_t world, rank;
} PpoPeerComm;
int64_t ppo_peer_window_bytes(int64_t cap);
int ppo_peer_window_alloc(int64_t cap, void** window_out, unsigned char* handle64_out);
int ppo_peer_window_open(const unsigned char* handle64, void** window_out);
int ppo_peer_window_close(void* window, int32_t owned);
/* dst[i] = sum over ranks of src_r[i]; seq_dev: device uint32 sequence counter (starts at 0, same on every rank);
 * err_flag: device word OR-ed with 1 if a peer did not arrive within the spin bound (result then undefined)          */
int ppo_peer_allreduce_f32(const PpoPeerComm* c, const float* src, float* dst, int64_t count, uint32_t* seq_dev,
                           uint32_t* err_flag, void* stream);

/* ppo_minibatch_step_tc on `world` ranks: the gradient all-reduce of trancate_gradients_and_step [ref: RLG/common/a2c_common.py:308-323]
 * runs INSIDE the cooperative tail kernel -- every 64-entry block of the span [gradient | loss statistics | KL] is pushed to the peers
 * as 8-byte {value, sequence} packets (P2P stores over NVLink, payload and flag in one word), summed in rank order as the packets
 * arrive, then clipped / Adam-stepped / re-packed by the same CTA: T1 + T2 + tail = 3 launches per minibatch at any world size.
 * comm: windows from ppo_peer_window_alloc/open with cap >= world * ppo_minibatch_step_peer_entries(obs_dim) * 2 floats;
 * seq_dev as in ppo_peer_allreduce_f32 (its own counter); err_flag: set when a peer does not arrive within 10 s -- the parameters
 * are then left untouched by this and every later step until the host clears the flag.                                          */
int64_t ppo_minibatch_step_peer_entries(int32_t obs_dim);
int ppo_minibatch_step_peer_tc(float* params, float* packed, const float* obs, int32_t obs_dim, const float* obs_mean, const float* obs_var,
                               const float* actions, const float* old_neglogp, const float* advantages, const float* old_values,
                               const float* returns, float* old_mu, float* old_sigma, const PpoLossParams* lp, float* grads, float* scratch,
                               float* workspace, float* exp_avg, float* exp_avg_sq, float* lr, int32_t* step, const PpoAdamParams* ap,
                               const PpoPeerComm* comm, uint32_t* seq_dev, uint32_t* err_flag, int64_t M, void* stream);

/* RunningMeanStd training-mode update, fused: batch moments of x[M,D] + Chan merge into the fp64 running state + fp32 copies
 *   [ref: RLG/algos_torch/running_mean_std.py:69-89] */
int ppo_rms_update_f64(const float* x /*[M,D]*/, int64_t M, int32_t D, double* mean /*[D]*/, double* var /*[D]*/, double* count /*[1]*/,
                       float* mean32 /*[D]*/, float* var32 /*[D]*/, void* stream);

/* ------------------------------------------------------------------------- */
/* L  the loopz PPO learner (SURVEY 8(f) row 4): what OIGE/scripts/rlgames_train_loopz.py trains with                       */
/*   actor and critic are separate MLPEncode networks over obs = [speed | task | mass(Md)]:                                  */
/*     mass -> Linear(Md,64)+LeakyReLU -> Linear(64,16)+LeakyReLU -> Linear(16,8)+LeakyReLU = latent                         */
/*     cat(speed, task, latent) -> Linear(D-Md+8,128)+LeakyReLU -> Linear(128,128)+LeakyReLU -> Linear(128,OUT) [+tanh]      */
/*   actor OUT = 2 (+ tanh when tanh_out), critic OUT = 1; actions ~ tanh(Normal(mean, std)) * action_scale, std a free      */
/*   parameter (NOT a log-std).      [ref: OIGE/algo/ppo/module.py:54-115,184-361,517-659 ; rlgames_train_loopz.py:784-842]  */
/* ONE flat fp32 parameter vector in the order of PPO's optimiser ([*actor.parameters(), *critic.parameters()], ppo.py:60): */
/*   actor: mass_encoder.{0,2,4}.{weight,bias} | action_mlp.{0,2,4}.{weight,bias} | std[2] | critic: the same twelve tensors  */
#define PPO_LOOPZ_ENC1 64
#define PPO_LOOPZ_ENC2 16
#define PPO_LOOPZ_LATENT 8
#define PPO_LOOPZ_MAX_MASS 8
typedef struct {
  int32_t obs_dim;      /* D (33 for the live task)                                   */
  int32_t mass_dim;     /* Md: privileged tail width, 4 or 8 (cfg.yaml environment.mass_dim) */
  int32_t tanh_out;     /* architecture.activation == 'tanh': tanh on the actor output */
  float action_scale;   /* task.env.clipActions                                       */
  float eps;            /* 1e-6                                                       */
} PpoLoopzNet;
typedef struct {
  float clip_param;         /* 0.2 */
  float value_loss_coef;    /* 0.5 */
  float entropy_coef;       /* 0.0 ("entropy" is -log_prob of the stored action, module.py:632-637) */
  int32_t use_clipped_value_loss;
} PpoLoopzLossParams;
typedef struct {
  float beta1, beta2, eps;  /* torch.optim.Adam defaults 0.9, 0.999, 1e-8 */
  float max_grad_norm;      /* 0.5 */
} PpoLoopzAdamParams;
enum { PPO_LOOPZ_STAT_SURROGATE = 0, PPO_LOOPZ_STAT_VALUE_LOSS, PPO_LOOPZ_STAT_LOG_PROB, PPO_LOOPZ_STAT_LOSS, PPO_LOOPZ_STAT_GRAD_NORM,
       PPO_LOOPZ_STAT_SKIPPED, PPO_LOOPZ_STAT_COUNT };

int64_t ppo_loopz_param_count(const PpoLoopzNet* net);          /* P; < 0: unsupported shape */
int64_t ppo_loopz_actor_param_count(const PpoLoopzNet* net);    /* std lives at [PA, PA+2), the critic starts at PA+2 */
int64_t ppo_loopz_train_scratch_floats(const PpoLoopzNet* net);
int64_t ppo_loopz_returns_scratch_bytes(void);

/* PPO.observe / PPO.step: actor.sample(actor_obs) -> (actions, log_prob) and critic.predict(critic_obs) -> values.            */
/* The actor runs when actions, means or eval_actions is given, the critic when values is given (one launch, blockIdx.y =      */
/* network).  With eval_actions ([M,2]) nothing is sampled: log_prob receives the log-probability of those actions              */
/* (Actor.evaluate, module.py:72-74,586-637).                                                                                   */
/*   [ref: OIGE/algo/ppo/ppo.py:97-148 ; module.py:67-70,104-105,568-583]                                                     */
int ppo_loopz_act_f32(const float* params, const PpoLoopzNet* net, const float* actor_obs /*[M,D]*/, const float* critic_obs /*[M,D]*/,
                      uint64_t seed, uint64_t counter, const uint64_t* counter_offset /*device addend or NULL*/, int64_t row_offset,
                      const float* eval_actions /*[M,2] or NULL*/, float* actions /*[M,2]*/, float* log_prob /*[M]*/,
                      float* means /*[M,2] noiseless action*/, float* values /*[M]*/,
                      int64_t M, void* stream);

/* RolloutStorage.compute_returns: GAE with the done flag of the SAME step, returns = A + V, advantages = returns - values      */
/* standardised over the whole batch ((x - mean) / (unbiased std + 1e-8)), non-finite inputs / outputs zeroed.                  */
/*   [ref: OIGE/algo/ppo/storage.py:92-124]                                                                                     */
int ppo_loopz_returns_f32(const float* rewards /*[T,n]*/, const float* values /*[T,n]*/, const uint8_t* dones /*[T,n]*/,
                          const float* last_values /*[n]*/, float gamma, float lam, float* returns /*[T,n]*/, float* advantages /*[T,n]*/,
                          void* scratch /*ppo_loopz_returns_scratch_bytes()*/, int32_t T, int64_t n, void* stream);

/* one minibatch of PPO._train_step: clipped surrogate on the actor, (clipped) value loss on the critic, full backward.         */
/* index (optional): row ids of the minibatch inside the [T*n] storage (mini_batch_generator_shuffle); NULL = rows [0, M) of     */
/* the pointers given (mini_batch_generator_inorder: pass pointers offset to the minibatch).                                     */
/* grads[P + PPO_LOOPZ_STAT_COUNT]: gradient of mean(surrogate + value_loss_coef*value_loss - entropy_coef*entropy) + SUMS of    */
/* the per-sample statistics (ppo_loopz_adam_step_f32 turns them into means).   [ref: OIGE/algo/ppo/ppo.py:232-284]              */
int ppo_loopz_minibatch_grad_f32(const float* params, const PpoLoopzNet* net, const float* actor_obs, const float* critic_obs,
                                 const float* actions /*[.,2]*/, const float* old_log_prob, const float* advantages,
                                 const float* target_values, const float* returns, const int64_t* index /*[M] or NULL*/,
                                 const PpoLoopzLossParams* lp, float* grads, float* scratch, int64_t M, void* stream);

/* the same minibatch gradient with the two 128-wide layers of each network on the tcgen05 tensor cores (TF32 operands, fp32        */
/* accumulation in TMEM; ~1e-3 relative of the fp32 entry point above, which stays the numerics reference).  In-order minibatches  */
/* only (no index list); obs_dim - mass_dim + 8 <= 47.  workspace: ppo_loopz_tc_workspace_floats(net, M) floats, 16 B aligned.    */
int64_t ppo_loopz_tc_workspace_floats(const PpoLoopzNet* net, int64_t M);
int ppo_loopz_minibatch_grad_tc(const float* params, const PpoLoopzNet* net, const float* actor_obs, const float* critic_obs,
                                const float* actions, const float* old_log_prob, const float* advantages, const float* target_values,
                                const float* returns, const PpoLoopzLossParams* lp, float* grads, float* workspace, int64_t M,
                                void* stream);

/* clip_grad_norm_(max_grad_norm) + Adam on the whole flat vector; skipped (parameters, moments and step count untouched) when   */
/* the loss is not finite.  step: device int32[2], the current count is step[parity] and the new one is written to               */
/* step[1-parity] (the caller alternates parity: no CTA can observe another CTA's update); lr: device float (the host owns the   */
/* schedule); accum: device float[3] += (value loss, surrogate, 1) of the valid updates or NULL.   [ref: ppo.py:286-318]         */
int ppo_loopz_adam_step_f32(float* params, float* grads, float* exp_avg, float* exp_avg_sq, const float* lr, int32_t* step,
                            int32_t parity, float* accum, int64_t P, int64_t M, const PpoLoopzLossParams* lp,
                            const PpoLoopzAdamParams* ap, void* stream);

/* SquashedGaussianDiagonalCovariance.enforce_minimum_std   [ref: module.py:649-659] */
int ppo_loopz_enforce_min_std_f32(float* std, const float* min_std, int32_t dim, void* stream);

/* The loopz learner on `world` ranks (one process per GPU): each rank holds n envs of a W x n batch, and two exchanges over the         */
/* PpoPeerComm windows make a W-rank update equal to the one-rank update over all W x n envs (up to summation order), with bit-identical */
/* results on every rank.  Every entry travels as an 8-byte {fp32 value, sequence} packet stored into each peer's window and the values  */
/* are added in rank order.  comm: windows from ppo_peer_window_alloc/open with cap >= world * ppo_loopz_peer_entries(net) * 2 floats,  */
/* shared by both exchanges; seq_dev: device uint32[2], zero at start, shared by both exchanges and the same on every rank; err_flag:     */
/* device word OR-ed with 1 when a peer does not arrive within 10 s -- sticky: later exchanges stop waiting, the gradient exchange then   */
/* makes Adam skip its step, and the advantages come out zero.  Every rank must issue the same sequence of exchanges.                   */
int64_t ppo_loopz_peer_entries(const PpoLoopzNet* net);   /* packets per rank and parity; < 0: unsupported shape */
/* ppo_loopz_returns_f32 with the advantage moments (fp64 sum a, sum a^2) summed over the ranks: advantages are standardised over the */
/* whole W x T x n batch.                                                                                                             */
int ppo_loopz_returns_peer_f32(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, float gamma,
                               float lam, float* returns, float* advantages, void* scratch /*ppo_loopz_returns_scratch_bytes()*/, int32_t T,
                               int64_t n, const PpoPeerComm* comm, uint32_t* seq_dev, uint32_t* err_flag, void* stream);
/* between ppo_loopz_minibatch_grad_f32 / _tc and ppo_loopz_adam_step_f32 (called with M = world x the local minibatch): grads[0, P) */
/* becomes the mean of the ranks' gradients, the three statistic sums behind it their sum.                                          */
int ppo_loopz_grad_exchange_f32(const PpoPeerComm* comm, const PpoLoopzNet* net, float* grads, uint32_t* seq_dev, uint32_t* err_flag,
                                void* stream);

/* ------------------------------------------------------------------------- */
/* D  the USV SysID / DAgger student (SURVEY 8(f) row 4, second half): what OIGE/scripts/dagger_usv_sysid_loopz.py trains   */
/*   StateHistoryEncoder: hist[M, tsteps*In] -> per-step Linear(In,32)+LeakyReLU -> RESHAPE (bs,32,T) (the reference's      */
/*   reshape, not a transpose) -> Conv1d stack (tsteps 50: (8,4),(5,1),(5,1); 20: (6,2),(4,2); 10: (4,2),(2,1)) + LeakyReLU */
/*   -> flatten 96 -> Linear(96,Out)+LeakyReLU.     [ref: OIGE/algo/ppo/module.py:392-448]                                   */
/*   Flat fp32 parameters in StateHistoryEncoder.parameters() order: encoder.0.{weight,bias} | conv_layers.{0,2,(4)}.        */
/*   {weight [32,32,k], bias} | linear_output.0.{weight [Out,96], bias}.  In <= 32, Out <= 8.                                */
int64_t dagger_history_encoder_param_count(int32_t input_size, int32_t tsteps, int32_t output_size);   /* < 0: unsupported */
int64_t dagger_train_scratch_floats(int32_t input_size, int32_t tsteps, int32_t output_size);
/* id_encoder(history): latent[M, Out]; hist rows are hist_ld floats apart (sysid_obs = [history_flat | current] is read in place) */
int dagger_history_encoder_forward_f32(const float* params, const float* hist /*[M, hist_ld]*/, int64_t hist_ld, int32_t input_size,
                                       int32_t tsteps, int32_t output_size, float* latent /*[M, Out]*/, int64_t M, void* stream);
/* one minibatch of USVSysIDTrainer._train_step: pred = id_encoder(hist); loss = MSELoss(pred, zstar); backward; Adam.step()    */
/* (torch defaults: betas 0.9 / 0.999, eps 1e-8, no weight decay, no clipping).  grads[P + 1] = [gradient | the minibatch MSE];  */
/* lr: device float (the host owns StepLR); step: device int32[2], current count in step[parity], new count to step[1 - parity]; */
/* mse_accum: device float += MSE or NULL.  Deterministic (fixed summation order).   [ref: OIGE/algo/ppo/dagger.py:125-196]      */
int dagger_sysid_minibatch_step_f32(float* params, const float* hist, int64_t hist_ld, const float* zstar /*[M, Out]*/, int32_t input_size,
                                    int32_t tsteps, int32_t output_size, float* grads, float* scratch, float* exp_avg, float* exp_avg_sq,
                                    const float* lr, int32_t* step, int32_t parity, float* mse_accum, int64_t M, void* stream);
/* a small dense MLP (<= 3 nn.Linear layers, widths <= 128, LeakyReLU between them) out of a flat parameter vector: the frozen     */
/* teacher mass encoder (priv tail -> z*) and the frozen action head ([current obs | z^] -> action) of USVSysIDAgent.              */
/* last_activation: 0 LeakyReLU, 1 tanh, 2 none.   [ref: OIGE/algo/ppo/dagger.py:50-66]                                            */
int dagger_mlp_forward_f32(const float* params, int32_t n_layers, const int32_t* dims /*host [n_layers + 1]*/,
                           const int32_t* w_offsets /*host [n_layers]*/, const int32_t* b_offsets /*host [n_layers]*/,
                           int32_t last_activation, const float* x /*[M, x_ld]*/, int64_t x_ld, float* y /*[M, dims[n_layers]]*/,
                           int64_t M, void* stream);
/* The deployed student's control step in one launch (USVSysIDStudentPolicy): append obs[:, :obs_nonpriv_dim] (rows obs_ld floats   */
/* apart) to each env's history ring, run the id_encoder on the window in chronological order and the frozen action head on           */
/* [frame | z^].  mu_out[M, head_dims[head_layers]] and latent_out[M, latent_dim] (or NULL) are bit-identical to                     */
/* dagger_mlp_forward_f32(head, [frame | dagger_history_encoder_forward_f32(history)]) on the unrolled history.                       */
/* ring: device [M, tsteps, obs_nonpriv_dim]; slot: device int32[2] = {slot of the oldest frame, 0}, zeroed with the ring: the launch */
/* overwrites that slot and advances the index on the device (graph-capturable).  The window follows USVSysIDVecEnv: init = 1 is    */
/* its reset() (fill_mode 0 "zeros": zeros then the frame last; 1 "repeat": the frame in every slot), init = 0 a step; dones (int64  */
/* [M] or NULL, the flags of the step that produced obs) refill a finished env's window with the frame in "repeat" mode only.        */
/* head_*: as dagger_mlp_forward_f32; head_dims[0] must be obs_nonpriv_dim + latent_dim.  Every argument is checked before any CUDA    */
/* call.   [ref: OIGE/envs/usv_raisim_vecenv.py:387-617, OIGE/algo/ppo/dagger.py:50-66]                                               */
int dagger_student_act_f32(const float* encoder_params, const float* head_params, int32_t head_layers, const int32_t* head_dims /*host*/,
                           const int32_t* head_w_offsets /*host*/, const int32_t* head_b_offsets /*host*/, int32_t head_last_activation,
                           float* ring, int32_t* slot, const float* obs /*[M, obs_ld]*/, int64_t obs_ld, int32_t obs_nonpriv_dim,
                           int32_t tsteps, int32_t latent_dim, const int64_t* dones, int32_t fill_mode, int32_t init, float* mu_out,
                           float* latent_out, int64_t M, void* stream);
/* Distillation from a frame store (USVSysIDDistiller).  Over a rollout of H steps the store keeps each frame once:                   */
/*   store  device [M, tsteps - 1 + H, obs_nonpriv_dim]: index t + tsteps - 1 is the frame of rollout step t; indices 0 .. tsteps - 1 */
/*          hold the whole window of step 0;                                                                                         */
/*   refill device int32 [H, M]: the store index of the last "repeat" refill at or before step t, 0 when there was none;              */
/*   row t * M + e (time-major, as ObsStorage flattens its samples) is the window of step t for env e, whose element k (oldest       */
/*   first) is store[e][max(t + k, refill[t][e])].                                                                                    */
/* dagger_sysid_collect_f32: dagger_student_act_f32 on rollout step t in [0, H) (init = 1 only at t = 0), plus the window into the   */
/* store, refill[t], and the label zstar[t] (device [H, M, latent_dim]) = the teacher's mass encoder (teacher_*: as                  */
/* dagger_mlp_forward_f32, teacher_dims[teacher_layers] = latent_dim) on obs[:, obs_nonpriv_dim : obs_nonpriv_dim + teacher_dims[0]], */
/* bit-identical to dagger_mlp_forward_f32 on that slice.  One launch.  Every argument is checked before any CUDA call.               */
int dagger_sysid_collect_f32(const float* encoder_params, const float* head_params, int32_t head_layers, const int32_t* head_dims /*host*/,
                             const int32_t* head_w_offsets /*host*/, const int32_t* head_b_offsets /*host*/, int32_t head_last_activation,
                             const float* teacher_params, int32_t teacher_layers, const int32_t* teacher_dims /*host*/,
                             const int32_t* teacher_w_offsets /*host*/, const int32_t* teacher_b_offsets /*host*/,
                             int32_t teacher_last_activation, float* ring, int32_t* slot, const float* obs /*[M, obs_ld]*/, int64_t obs_ld,
                             int32_t obs_nonpriv_dim, int32_t tsteps, int32_t latent_dim, const int64_t* dones, int32_t fill_mode, int32_t init,
                             float* store, int32_t* refill, float* zstar, int32_t t, int32_t horizon, float* mu_out, int64_t M, void* stream);
/* dagger_history_encoder_forward_f32 / dagger_sysid_minibatch_step_f32 on the store's rows [row0, row0 + M) of horizon * num_envs  */
/* (input_size = obs_nonpriv_dim); zstar is the whole label buffer [horizon * num_envs, Out].  Same bits as the row versions on the */
/* unrolled windows.                                                                                                                  */
int dagger_history_encoder_forward_store_f32(const float* params, const float* store, const int32_t* refill, int64_t num_envs, int32_t horizon,
                                             int64_t row0, int32_t input_size, int32_t tsteps, int32_t output_size, float* latent /*[M, Out]*/,
                                             int64_t M, void* stream);
int dagger_sysid_minibatch_step_store_f32(float* params, const float* store, const int32_t* refill, int64_t num_envs, int32_t horizon, int64_t row0,
                                          const float* zstar, int32_t input_size, int32_t tsteps, int32_t output_size, float* grads, float* scratch,
                                          float* exp_avg, float* exp_avg_sq, const float* lr, int32_t* step, int32_t parity, float* mse_accum,
                                          int64_t M, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* USV_B200_H_ */

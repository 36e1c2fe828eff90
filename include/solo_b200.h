/*
 * solo_b200.h — C-ABI of the B200-native batched Solo8/Solo12 environment step.
 *
 * This is the drop-in boundary for the ONE hot path of michel-aractingi/soloRL:
 * the vectorised env step that the reference drives, one OS process per env,
 * through PyBullet (`agents/ppo/envs.py:91-95` -> `baseEnv.py:42-68` ->
 * `solo.py:224-274` -> `p.stepSimulation()`).  Every entry point below names the
 * reference interface it replaces (file:line into the reference tree).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - every function returns 0 on success, a negative SOLO_E_* code otherwise;
 *     solo_last_error() returns a human-readable string for the last failure
 *     (per handle when a handle exists, otherwise a thread-local global).
 *   - all `d_*` pointers are DEVICE pointers owned by the caller; all `h_*`
 *     pointers are HOST pointers.  Launches go onto the caller-supplied stream
 *     (`void* stream` is a cudaStream_t; NULL = legacy default stream) and the
 *     device-pointer calls never synchronise the host.
 *   - a handle is not thread-safe; different handles are independent.
 *   - there is NO CPU fallback: without a CUDA device solo_create fails with
 *     SOLO_E_CUDA.  (The double-precision CPU restatement under oracle/ is test
 *     infrastructure and is never linked into this library.)
 *
 * Layouts at the boundary (all row-major, float32 unless noted)
 *   actions  [N, A]   A = nj (+2 for control == SOLO_CONTROL_VPD)   (solo.py:224-259)
 *   obs      [N, D]   D = D0*(1+H), D0 = 1+3+6+2*nj+4 (+4 pointgoal) (solo.py:186-222)
 *   reward   [N]      (baseEnv.py:91-157; caller views it as [N,1], envs.py:195)
 *   done     [N]      float 0/1 (envs.py:194)
 *   state    [N, 13+2*nj] = pos(3) quat xyzw(4) linvel(3) angvel(3) q(nj) qd(nj)
 *            (what getBasePositionAndOrientation/getBaseVelocity/getJointState
 *             return, solo.py:201-210)
 */
#ifndef SOLO_B200_H
#define SOLO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOLO_ABI_VERSION 3

#define SOLO_MAX_LINKS 20
#define SOLO_MAX_FEET 4

/* error codes */
#define SOLO_OK 0
#define SOLO_E_ARG (-1)      /* bad argument */
#define SOLO_E_MODEL (-2)    /* model table not supported by the kernels */
#define SOLO_E_CUDA (-3)     /* CUDA runtime failure / no device */
#define SOLO_E_STATE (-4)    /* step before reset (baseEnv.py:43) */

/* joint types in the model table */
#define SOLO_JOINT_FIXED 0
#define SOLO_JOINT_REVOLUTE 1

/* control modes (solo.py:228-254) */
#define SOLO_CONTROL_TORQUE 0
#define SOLO_CONTROL_PD 1      /* 'pd', 'fpd', 'fixed_pd' */
#define SOLO_CONTROL_VPD 2     /* 'vpd', 'variable_pd' */

/* tasks (baseEnv.py:93-138) */
#define SOLO_TASK_STAND 0
#define SOLO_TASK_WALK 1
#define SOLO_TASK_POINTGOAL 2

/* reset modes */
#define SOLO_RESET_CACHED 0    /* settle trajectories memoised per settle count (bit-identical) */
#define SOLO_RESET_SIMULATE 1  /* settle steps simulated in the step kernel */

/*
 * Flattened kinematic tree, the result of parsing a solo_description URDF once
 * (replaces p.loadURDF + p.getJointInfo iteration, solo.py:69-110).
 * Links are in URDF <joint> order (= PyBullet link index); parents precede children.
 * All joint origins must have rpy = 0 (true for solo.urdf and solo12.urdf).
 */
typedef struct SoloModelTable {
  int32_t abi_version;               /* SOLO_ABI_VERSION */
  int32_t num_links;                 /* links excluding the base */
  int32_t parent[SOLO_MAX_LINKS];    /* -1 = base */
  int32_t jtype[SOLO_MAX_LINKS];     /* SOLO_JOINT_* */
  double axis[SOLO_MAX_LINKS][3];    /* joint axis in the link frame */
  double origin[SOLO_MAX_LINKS][3];  /* joint origin xyz in the parent link frame */
  double mass[SOLO_MAX_LINKS];
  double com[SOLO_MAX_LINKS][3];     /* inertial origin in the link frame */
  double inertia[SOLO_MAX_LINKS][6]; /* ixx ixy ixz iyy iyz izz about the COM, link axes */
  double base_mass;
  double base_com[3];                /* must be 0 (true for both URDFs) */
  double base_inertia[6];
  int32_t num_feet;                  /* links whose joint name contains "ANKLE" (solo.py:99-106) */
  int32_t foot_link[SOLO_MAX_FEET];  /* link index of each foot */
  double foot_center[SOLO_MAX_FEET][3]; /* collision-sphere centre in the foot link frame */
  double foot_radius;                /* collision-sphere radius */
} SoloModelTable;

/*
 * Simulation + task parameters.  Physics defaults restate Bullet/PyBullet defaults
 * (third-party, not in the reference tree; see DESIGN.md "Bullet step restatement");
 * env defaults restate solo.py:17-53 and baseEnv.py:8-16.
 */
typedef struct SoloSimParams {
  int32_t abi_version;
  /* physics (simulation.py:19,33; solo.py:22) */
  double dt;                 /* 1/240 */
  int32_t frame_skip;        /* 4 */
  double gravity_z;          /* -9.81 */
  double lin_damping;        /* 0.04  Bullet btMultiBody linear damping  */
  double ang_damping;        /* 0.04  Bullet btMultiBody angular damping */
  double max_coord_vel;      /* 100   Bullet m_maxCoordinateVelocity */
  int32_t solver_iters;      /* 50    PyBullet numSolverIterations (iteration cap) */
  double solver_residual_threshold; /* 1e-7  PyBullet solverResidualThreshold: the sweep loop stops once
                                     * the largest squared row velocity residual of an iteration is <= this;
                                     * 0 = always run solver_iters iterations */
  double contact_erp;        /* 0.2   contact error-reduction parameter */
  double contact_slop;       /* 1e-5  linear slop added to the contact distance */
  double contact_margin;     /* 0.02  contact point exists while distance < margin */
  double friction;           /* 1.0   combined lateral friction (foot 1.0 x plane 1.0) */
  int32_t cone_friction;     /* 1     implicit cone (Bullet default) ; 0 = pyramid */
  int32_t torque_hold;       /* 0     torque acts in substep 1 only (SURVEY F4); 1 = all substeps */
  /* action front end (solo.py:224-259, controllers/PD.py:3-10) */
  int32_t control;           /* SOLO_CONTROL_* */
  double kp, kd;             /* gains for SOLO_CONTROL_PD */
  double max_torque;         /* 3   (solo.py:53) */
  double joint_state_limit;  /* 10  (solo.py:109) */
  double joint_vel_limit;    /* 100 (solo.py:110) */
  /* task (baseEnv.py) */
  int32_t task;              /* SOLO_TASK_* */
  int32_t episode_length;    /* configs: 400 */
  int32_t num_history_stack; /* H */
  double initial_z;          /* 0.35 (solo.py:52) */
  int32_t settle_min;        /* 5  np.random.randint(low=5, high=12) (baseEnv.py:79) */
  int32_t settle_max;        /* 12 (exclusive) */
  double goal_radius;        /* 2.0 (solo.py:141) */
  double goal_reach_dist;    /* 0.5 (solo.py:270) */
  double pointgoal_dt;       /* frame_skip*dt; stands in for the undefined scene.dt (baseEnv.py:137) */
  double contact_flag_force; /* 0.2 (solo.py:320, tuple index 9 = normal force) */
  double fall_z;             /* 0.05 (baseEnv.py:169) */
  double stand_z;            /* 0.2 (baseEnv.py:96) */
  int32_t reset_mode;        /* SOLO_RESET_* */
  /* joint-limit rows: [3P] PyBullet's URDF importer adds a btMultiBodyJointLimitConstraint per revolute joint
   * with lower <= upper (here +-joint_state_limit, solo.urdf:47); while q is beyond a limit the solver gets a
   * unilateral row on that joint, swept before the contact normals (see DESIGN.md) */
  int32_t joint_limits;           /* 1: on (reference behaviour); 0: joints are unlimited */
  int32_t limit_rows_per_leg;     /* 1: at most one row per leg, the most violated joint (what the kernels
                                   * solve); 0: one row per violated joint (Bullet; oracle only) */
  double joint_limit_erp;         /* 0.2   btContactSolverInfo::m_erp */
  double joint_limit_max_impulse; /* 100   btMultiBodyConstraint m_maxAppliedImpulse default */
  double split_impulse_threshold; /* -0.04 violations deeper than this get no positional correction */
  /* contacts of links other than the feet with the flat ground (SURVEY §8f n4): in Bullet a collapsed robot rests
   * on its knees / base box (convex hulls of the visual meshes, solo.py:72-73) and may stay above the z < 0.05
   * termination height (baseEnv.py:169) until the timeout.  Collision primitives, [3P] stand-ins for those hulls:
   * one sphere per knee (centre = KFE joint origin, on the lower-leg link) and the eight corners of the base box
   * (points).  Contact points are ordered feet, knees, lower base corners, upper base corners (leg order inside
   * each group); normals of all points are swept first, then the friction pair of each point. */
  int32_t body_contacts;          /* 0: feet only (default, what round 1 built); 1: knees and base corners too */
  double knee_radius;             /* 0.015: the lower-leg mesh reaches 0.0135 m above the KFE axis (SURVEY App. A) */
  double base_half_x, base_half_y;/* 0.2241 x 0.1095 (Solo12), 0.212 x 0.1046 (Solo8) */
  double base_z_lo, base_z_hi;    /* -0.025, 0.028: bottom / top of the base box relative to the base origin */
  /* Randomised dynamics (domain randomisation for sim-to-real).  With randomize = 1 every reset (full, masked,
   * or the auto-reset inside solo_step) draws three values per env, each uniform in [lo, hi] from the env's own
   * RNG stream, fixed for the episode:
   *   friction        the combined lateral friction of the env's contact rows (replaces `friction`);
   *   base_mass_scale base mass and base inertia tensor times this (the legs keep theirs);
   *   motor_strength  the torque of every action mode times this (max_torque; kp, kd and the clamp under PD / VPD).
   * They act in the control steps of solo_step / solo_step_host, solo_substep, solo_forward_dynamics and
   * solo_action_to_torque.  The settle steps of a reset run with the nominal values (so cached resets stay
   * exact); solo_actuator_step (gait envs) does not use them.  Not available in the wide build.
   * randomize = 0 (default): the ranges are not read.  With randomize = 1 all six bounds must be set
   * (0 <= friction_lo <= friction_hi, 0 < lo <= hi for the scales); solo_default_params leaves them 0. */
  int32_t randomize;
  double friction_lo, friction_hi;
  double base_mass_scale_lo, base_mass_scale_hi;
  double motor_strength_lo, motor_strength_hi;
  /* Random pushes: a horizontal force on the base, in base axes at the base origin, held as a rectangular pulse
   * through every substep of push_duration consecutive control steps once in every push_interval control steps.
   * With t = the env's control steps completed in its episode, j = t / push_interval and r = t % push_interval,
   * one draw of the env's RNG stream per (episode, j) gives the window's start s in [0, interval - duration] and
   * the force (fx, fy, 0), fx and fy uniform in [-push_force, push_force]; step t is pushed iff s <= r < s + D.
   * The schedule starts again at t = 0 with every episode.  Pushes act in the control steps of solo_step /
   * solo_step_host only: not in the settle steps of a reset (so cached resets stay exact), solo_substep,
   * solo_forward_dynamics, solo_action_to_torque or solo_actuator_step.  Not available in the wide build.
   *   push_force     F in N, finite, >= 0;
   *   push_interval  I in control steps; 0 = pushes off (default), and then the other two are not read;
   *   push_duration  D in control steps, 1 <= D <= I.
   * solo_create also rejects episode_length / I >= 2^30. */
  double push_force;
  int32_t push_interval;
  int32_t push_duration;
} SoloSimParams;

/* Per-env episode record, valid for envs whose `done` was 1 at the last step
 * (the info dict of baseEnv.py:63-66,162-187). */
typedef struct SoloEpisodeStats {
  float episode_reward;  /* reward of the terminal step (baseEnv.py:65, SURVEY F8) */
  float episode_return;  /* sum of rewards over the episode (_reward_sum, baseEnv.py:62) */
  int32_t episode_length;
  int32_t success;       /* info['success'] */
  int32_t timeout;       /* info['timeout'] */
  int32_t goals_reached;
  float dr_stand, dr_joint_pose, dr_torque, dr_balance, dr_progress; /* the 'dr/...' sums */
  int32_t nan;           /* 1: the episode was ended by the non-finite-state guard (the reference only
                          * guards its gait envs, baseControlEnv.py:171-175,389-397: zero obs, done, hard reset) */
} SoloEpisodeStats;

typedef struct SoloHandle SoloHandle;

/* Fill *p with the reference defaults (solo.py:17-53, baseEnv.py:8-16, Bullet defaults). */
int solo_default_params(SoloSimParams* p);

/* Dimensions implied by (model, params): nj, action dim A, base obs dim D0, obs dim D. */
int solo_dims(const SoloModelTable* m, const SoloSimParams* p,
              int32_t* nj, int32_t* act_dim, int32_t* obs_dim0, int32_t* obs_dim);

/* Replaces SoloBaseEnv.__init__ / SoloBase.load for N envs at once
 * (baseEnv.py:6-40, solo.py:55-152, simulation.py:13-35).
 * env_id_offset: global id of env 0 on this rank (per-env RNG stream = global id,
 * so results do not depend on how envs are sharded over GPUs). */
int solo_create(const SoloModelTable* model, const SoloSimParams* params,
                int32_t num_envs, int32_t device, uint64_t seed, int64_t env_id_offset,
                SoloHandle** out);
int solo_destroy(SoloHandle* h);
const char* solo_last_error(const SoloHandle* h_or_null);

/* Replaces VecEnvWrapper.reset -> SoloBaseEnv.reset (agents/ppo/envs.py:97-100,
 * baseEnv.py:70-82, solo.py:166-181,291-296).  d_mask: optional uint8[N], reset only
 * envs with mask != 0; NULL = all.  d_obs_out may be NULL. */
int solo_reset(SoloHandle* h, const uint8_t* d_mask, float* d_obs_out, void* stream);

/* Replaces VecEnvWrapper.step -> simple_worker step + auto-reset
 * (agents/ppo/envs.py:36-40,91-95, baseEnv.py:42-68). */
int solo_step(SoloHandle* h, const float* d_actions, float* d_obs, float* d_reward,
              float* d_done, void* stream);

/* Same call with HOST buffers (the reference boundary is host numpy arrays,
 * agents/ppo/envs.py:189-196): H2D actions, step, obs/reward/done back on the host, then one
 * stream synchronise.  When the three output buffers are pinned (page-locked) the step kernel writes
 * them itself through their device-mapped alias, as whole 128-byte lines while the launch is still
 * running; pageable buffers go through device staging and three D2H copies. */
int solo_step_host(SoloHandle* h, const float* h_actions, float* h_obs, float* h_reward,
                   float* h_done, void* stream);

/* Replaces get_observation (agents/ppo/envs.py:102-105, solo.py:186-196). */
int solo_get_observation(SoloHandle* h, float* d_obs, void* stream);

/* State injection / extraction for parity tests: replaces
 * getBasePositionAndOrientation/getBaseVelocity/getJointState and
 * resetBasePositionAndOrientation/resetJointState (solo.py:201-210,291-296).
 * set_state also clears the contact set and refills the history with the current
 * state (solo.py:170-171). */
int solo_get_state(SoloHandle* h, float* d_state, void* stream);
int solo_set_state(SoloHandle* h, const float* d_state, void* stream);

/* Pointgoal only: overwrite the goal of every env (d_goals float[N,2]) and recompute the
 * potential (solo.py:277-279); parity tests use it to give oracle and GPU the same goal. */
int solo_set_goals(SoloHandle* h, const float* d_goals, void* stream);

/* Contact record of the last substep: per env, per foot: flag (0/1 as in
 * solo.py:310-323), has_point, normal force [N]. d_out float[N, 4, 3]. */
int solo_get_contacts(SoloHandle* h, float* d_out, void* stream);

/* Parity hook: overwrite the contact record that solo_get_contacts / the observation's contact flags read
 * (what p.getContactPoints would return at solo.py:313-317): d_force float[N, 4] = normal force per foot,
 * a negative value = no contact point.  Lets the 1e-6 observation test inject contact sets on both sides of
 * the 0.2 N flag threshold (solo.py:310-323, SURVEY F5); solo_set_state clears the record again. */
int solo_set_contacts(SoloHandle* h, const float* d_force, void* stream);

/* Measurement hook: work done by the last env step, per env: d_out int32[N,2] =
 * (sum over substeps of feet in contact, sum over substeps of feet-in-contact x PGS sweeps run).
 * bench.py turns these into the algorithmic FLOPs of the launch. */
int solo_get_work_counters(SoloHandle* h, int32_t* d_out, void* stream);

/* Contact-free forward dynamics on given states: qdd [N, 6+nj] =
 * (base angular acc (world), base linear acc (world), joint acc) for joint torques
 * tau [N, nj]; includes gravity and Bullet damping terms.  The 1e-5 test hook. */
int solo_forward_dynamics(SoloHandle* h, const float* d_state, const float* d_tau,
                          float* d_qdd, void* stream);

/* One Bullet-equivalent substep (collision, ABA, contact PGS, integrate) on the
 * handle's own state with joint torques tau [N, nj].  The 1e-3 contact-step hook
 * (replaces p.stepSimulation, solo.py:265). */
int solo_substep(SoloHandle* h, const float* d_tau, void* stream);

/* Action -> joint torque exactly as solo.py:224-259 + controllers/PD.py:3-10 on the
 * handle's current state (times the env's motor strength on a randomised handle). d_tau [N, nj]. */
int solo_action_to_torque(SoloHandle* h, const float* d_actions, float* d_tau, void* stream);

/* The dynamics each env runs its episode with, d_out float[N, 3] = (friction, base_mass_scale, motor_strength):
 * the values the last reset drew on a randomised handle (privileged critic inputs, logging), the nominal
 * (friction, 1, 1) otherwise and before the first reset. */
int solo_get_env_params(SoloHandle* h, float* d_out, void* stream);

/* The push the next solo_step applies to each env (SoloSimParams.push_*), d_out float[N, 3] = (fx, fy, 0) in N,
 * base axes: zero outside a push window and on a handle without pushes.  A pure function of the env's episode
 * and step count (privileged critic inputs, logging). */
int solo_get_push_force(SoloHandle* h, float* d_out, void* stream);

/* Gait envs (SURVEY §8f n2): n_ticks simulator ticks under the joint-level PD + feed-forward actuator
 * that the external PyBulletSimulator exposes to baseControlEnv.py:256-270
 * (SetDesiredJointPDgains / Position / Velocity / Torque + SendCommand):
 *   tau = clip(P (q_des - q) + D (v_des - v) + tau_ff, +-max_torque), recomputed before every tick,
 * then one Bullet-equivalent step at params.dt (create the handle with dt = 0.002, the gait envs' tick).
 * d_cmd float[N, 5, nj] = q_des, v_des, P, D, tau_ff.  State is read back with solo_get_state.
 * Runs with the nominal dynamics: SoloSimParams.randomize does not apply to the gait envs. */
int solo_actuator_step(SoloHandle* h, const float* d_cmd, int32_t n_ticks, void* stream);

/* Gait envs: external force on the base for the following solo_actuator_step calls, d_force float[N, 3] in base
 * (link-frame) axes, acting at the base origin -- the random pushes of baseControlEnv.py:276-289, which the
 * external simulator applies with pyb.applyExternalForce(robot, -1, F, [0,0,0], LINK_FRAME) [3P].  Stays in
 * force until overwritten; zero after solo_create.  solo_step / solo_substep ignore it: the RL envs' step has
 * pushes of its own (SoloSimParams.push_*). */
int solo_set_external_force(SoloHandle* h, const float* d_force, void* stream);

/* World-frame centres of the four foot collision spheres, d_out float[N, 4, 3]
 * (replaces get_feet_positions, baseControlEnv.py:410-414). */
int solo_get_feet(SoloHandle* h, float* d_out, void* stream);

/* Episode records of the last step (see SoloEpisodeStats). d_stats: SoloEpisodeStats[N]. */
int solo_episode_stats(SoloHandle* h, SoloEpisodeStats* d_stats, void* stream);

/* Fold the episode records of the envs whose d_done flag is set (the flags solo_step just wrote) into
 * running totals on the device — the trainer's episode logging (agents/ppo/train.py:90-100,
 * agents/td3/train.py:108-115) without reading an info dict per env and step.
 * d_acc double[13]: [0] episodes, [1] sum episode_reward, [2] sum episode_return, [3] sum length,
 * [4] sum success, [5..9] sums of the five dr/ terms, [10] min return, [11] max return, [12] max length.
 * The caller initialises d_acc (zeros; +inf / -inf / 0 for [10..12]). */
int solo_accumulate_episode_stats(SoloHandle* h, const float* d_done, double* d_acc, void* stream);

/* Curriculum hook (increment_goal_radius, solo.py:332-334).  The radius is kept in device memory, so steps
 * already captured into a CUDA graph see the new value; the call waits for the device to drain first. */
int solo_set_goal_radius(SoloHandle* h, double goal_radius);

/* Reverse-scan GAE over a device-resident rollout, replaces
 * OPBuffer.compute_returns (agents/ppo/storage.py:35-55).
 * rewards [T,N], values [T+1,N] (values[T] = bootstrap), masks [T+1,N], returns [T+1,N].
 * use_gae == 0 selects the discounted-return branch (storage.py:51-55), which reads
 * returns[T] as the bootstrap value. */
int solo_gae(const float* d_rewards, const float* d_values, const float* d_masks,
             float* d_returns, int32_t T, int32_t N, float gamma, float lam,
             int32_t use_gae, void* stream);

/* Number of kernel launches issued through this handle so far (bench evidence). */
int64_t solo_launch_count(const SoloHandle* h);

/* Which build of the step kernel this handle launches ("latency", "throughput", "wide", or "body" when
 * SoloSimParams.body_contacts is set; "+rand" appended on a randomised handle, then "+push" on a handle with
 * pushes): chosen at create time from the batch size, SOLO_STEP_VARIANT overrides (bench / profile evidence). */
const char* solo_step_variant(const SoloHandle* h);

#ifdef __cplusplus
}
#endif
#endif /* SOLO_B200_H */

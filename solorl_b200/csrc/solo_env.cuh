/*
 * solo_env.cuh — env-level arithmetic of the step (observation, reward, termination,
 * episode bookkeeping) as lane-level host/device functions.  Restates the reference's
 * baseEnv.py:42-187 and solo.py:186-340 in fp32; citations are file:line into the
 * reference tree.
 */
#pragma once
#include "solo_core.cuh"

namespace solo {

/* Per-env episode bookkeeping (baseEnv.py:30-38, solo.py:138-145), one record per env. */
struct EnvBook {
  int32_t timestep;      /* baseEnv.py:32 */
  int32_t goals_env;     /* SoloBaseEnv._goals_reached */
  int32_t goals;         /* SoloBase.goals_reached */
  int32_t settle_left;   /* simulate-mode reset: control steps still to settle */
  uint32_t episode;      /* rng stream position */
  uint32_t draw;
  float reward_sum;      /* baseEnv.py:33 */
  float dr[5];           /* stand, joint_pose, torque, balance, progress (baseEnv.py:34-38) */
  /* work done by the last env step (measurement only): sum over substeps of the number of feet
   * in contact, and of (feet in contact x PGS sweeps executed) */
  int32_t nc_sum, sweep_feet;
};

/* layout of the base record base[env][16] */
enum { kBaseP = 0, kBaseQ = 3, kBaseV = 7, kBaseW = 10, kBaseGoal = 13, kBasePot = 15, kBaseStride = 16 };

/* index helpers into one D0 row of the observation (solo.py:198-222) */
SOLO_HD int idx_q(int njl, int leg, int k) { return 10 + leg * njl + k; }
SOLO_HD int idx_qd(int njl, int leg, int k) { return 10 + 4 * njl + leg * njl + k; }
SOLO_HD int idx_flag(int njl, int leg) { return 10 + 8 * njl + leg; }
SOLO_HD int idx_pg(int njl) { return 14 + 8 * njl; }
SOLO_HD int obs_dim0(int njl, int task) { return 14 + 8 * njl + (task == 2 ? 4 : 0); }

/* solo.py:310-323 with tuple index 9 = normal force (SURVEY F5); cforce < 0 = no contact point */
SOLO_HD float contact_flag(const SimConst& sc, float cforce) {
  return (cforce >= 0.f && cforce < sc.flag_force) ? 1.0f : 0.0f;
}

/* base part of get_current_state (solo.py:201-206): z, euler map, linear vel, angular vel */
SOLO_HD void cur_base(const BaseState& st, float* out10) {
  float rpy[3];
  quat_to_euler(st.q, rpy);
  out10[0] = st.p[2];
  out10[1] = euler_obs(rpy[0]); out10[2] = euler_obs(rpy[1]); out10[3] = euler_obs(rpy[2]);
  out10[4] = st.v[0]; out10[5] = st.v[1]; out10[6] = st.v[2];
  out10[7] = st.w[0]; out10[8] = st.w[1]; out10[9] = st.w[2];
}
/* solo.py:337-340 */
SOLO_HD void cur_pointgoal(const BaseState& st, const float* goal, float* out4) {
  out4[0] = st.p[0] / 2.0f; out4[1] = st.p[1] / 2.0f; out4[2] = goal[0] / 2.0f; out4[3] = goal[1] / 2.0f;
}
SOLO_HD float calc_potential(const BaseState& st, const float* goal) { /* solo.py:277-279 */
  float dx = st.p[0] - goal[0], dy = st.p[1] - goal[1];
  return sqrtf(dx * dx + dy * dy);
}

struct StepOutcome {
  float reward;
  int done, success, timeout;
};

/* get_reward + is_episode_finished + the done overrides of step (baseEnv.py:50-62,91-180).
 * sum_q  = sum over joints of |q| (stand) or q^2 (walk, pointgoal);  sum_a2 = sum a^2 over the raw action.
 * progress = robot.progress (pointgoal).  Updates book (timestep must already be incremented). */
SOLO_HD StepOutcome step_outcome(const SimConst& sc, const BaseState& st, int nj, float sum_q,
                                 float sum_a2, float progress_pg, EnvBook& bk, bool bad_state = false) {
  StepOutcome o;
  if (bad_state) {
    /* non-finite state (NaN/Inf actions or a blown-up solve): end the episode as a failure and let the
     * auto-reset replace the state; nothing non-finite enters the episode sums */
    o.reward = -10.f; o.done = 1; o.success = 0; o.timeout = 0;
    bk.reward_sum = isfinite(bk.reward_sum) ? bk.reward_sum + o.reward : o.reward;
    for (int i = 0; i < 5; i++) bk.dr[i] = isfinite(bk.dr[i]) ? bk.dr[i] : 0.f;
    return o;
  }
  float z = st.p[2];
  float stand = (z > sc.stand_z ? 1.0f : 0.0f) * 0.5f;            /* :96 */
  float jp = -0.1f * (sum_q / (float)nj);                         /* :101,:113,:131 */
  float balance = 0.f, progress = 0.f, torque = 0.f;
  if (sc.task == 1) {                                             /* walk :115-119 */
    if (z > sc.stand_z) {
      float vx = st.v[0];
      float sg = (vx > 0.f ? 1.f : 0.f) - (vx < 0.f ? 1.f : 0.f);
      progress = 2.f * sg * vx * vx;
    }
  } else if (sc.task == 2) {                                      /* pointgoal :133-140 */
    float rpy[3];
    quat_to_euler(st.q, rpy);
    balance = -0.1f * (fabsf(rpy[0]) + fabsf(rpy[1]));
    if (z > sc.stand_z) progress = progress_pg * sc.inv_pg_dt;
  }
  if (sc.control == 0) torque = -0.01f * sum_a2;                  /* :142-146 (F9a: else 0) */
  float r = stand + jp + balance + progress + torque;             /* :148 */
  bk.dr[0] += stand; bk.dr[1] += jp; bk.dr[2] += torque; bk.dr[3] += balance; bk.dr[4] += progress;
  o.done = 0; o.success = 0; o.timeout = 0;
  if (bk.timestep >= sc.episode_length) {                         /* :164-167 */
    o.done = 1; o.timeout = 1; o.success = (sc.task != 2);
  } else if (z < sc.fall_z) {                                     /* :169-172 */
    o.done = 1;
  } else if (sc.task == 2 && bk.goals > bk.goals_env) {           /* :174-178 */
    bk.goals_env = bk.goals; o.done = 1; o.success = 1;
  }
  if (o.done) {                                                   /* :52-60 */
    if (o.success) { if (sc.task == 2) r = 0.1f * (float)(sc.episode_length - bk.timestep); }
    else if (!o.timeout) r = -10.f;
  }
  bk.reward_sum += r;                                             /* :62 */
  o.reward = r;
  return o;
}

SOLO_HD void book_clear_episode(EnvBook& bk) { /* baseEnv.py:72-77 */
  bk.timestep = 0; bk.goals_env = 0; bk.reward_sum = 0.f;
  for (int i = 0; i < 5; i++) bk.dr[i] = 0.f;
}

/* Ranges of the randomised dynamics (SoloSimParams.friction_lo .. motor_strength_hi, narrowed to float). */
struct EnvRanges {
  float mu_lo, mu_hi, sm_lo, sm_hi, st_lo, st_hi;
};

/* Philox draw indices of the dynamics draw and of the push draws: the per-episode draws (settle count and goal at
 * the reset, new goals while stepping) count up from 0 and never reach kDynDraw; the push draw of interval j is
 * kPushDraw + j, and solo_create keeps j below 2^30, so it never reaches back to kDynDraw or wraps to 0.  Every
 * draw therefore stays what it is without randomisation or pushes. */
constexpr uint32_t kDynDraw = 0x80000000u;
constexpr uint32_t kPushDraw = 0xC0000000u;

/* The dynamics of env `gid` for episode `episode`: each value uniform in its range.  fmaf keeps the device and a
 * host replay bit-identical; fminf keeps a rounded-up product inside the range. */
SOLO_HD float dyn_uniform(float lo, float hi, uint32_t w) { return fminf(fmaf(hi - lo, u01(w), lo), hi); }
SOLO_HD EnvDyn sample_env_dyn(const EnvRanges& r, uint32_t seed_lo, uint32_t seed_hi, long long gid,
                              uint32_t episode) {
  uint32_t w[4] = {(uint32_t)((unsigned long long)gid & 0xffffffffull), (uint32_t)((unsigned long long)gid >> 32),
                   episode, kDynDraw};
  philox4x32_10(w, seed_lo, seed_hi);
  EnvDyn p;
  p.mu = dyn_uniform(r.mu_lo, r.mu_hi, w[0]);
  p.sm = dyn_uniform(r.sm_lo, r.sm_hi, w[1]);
  p.st = dyn_uniform(r.st_lo, r.st_hi, w[2]);
  return p;
}

/* Random pushes (SoloSimParams.push_*, narrowed to float / int): interval 0 = off. */
struct PushParams {
  float force;
  int32_t interval, duration;
};
struct PushSample {
  bool on;
  float fx, fy;   /* base axes; 0 when !on */
};

/* The push of env `gid` in control step t (steps completed in episode `episode`): interval j = t / I draws the
 * window start s = w[0] % (I - D + 1) and the force from one Philox block; step t is pushed iff s <= t % I < s + D. */
SOLO_HD PushSample sample_push(const PushParams& pp, uint32_t seed_lo, uint32_t seed_hi, long long gid,
                               uint32_t episode, int32_t t) {
  PushSample ps;
  ps.on = false; ps.fx = 0.f; ps.fy = 0.f;
  if (pp.interval <= 0) return ps;
  const uint32_t I = (uint32_t)pp.interval, j = (uint32_t)t / I, r = (uint32_t)t % I;
  uint32_t w[4] = {(uint32_t)((unsigned long long)gid & 0xffffffffull), (uint32_t)((unsigned long long)gid >> 32),
                   episode, kPushDraw + j};
  philox4x32_10(w, seed_lo, seed_hi);
  const uint32_t s = w[0] % (I - (uint32_t)pp.duration + 1u);
  if (s <= r && r < s + (uint32_t)pp.duration) {
    ps.on = true;
    ps.fx = dyn_uniform(-pp.force, pp.force, w[1]);
    ps.fy = dyn_uniform(-pp.force, pp.force, w[2]);
  }
  return ps;
}

/* robot_specific_reset (solo.py:291-296): base -> (0,0,initial_z), identity, zero velocity */
SOLO_HD void reset_pose(const SimConst& sc, BaseState& st) {
  st.p[0] = 0.f; st.p[1] = 0.f; st.p[2] = sc.initial_z;
  st.q[0] = 0.f; st.q[1] = 0.f; st.q[2] = 0.f; st.q[3] = 1.f;
  for (int i = 0; i < 3; i++) { st.v[i] = 0.f; st.w[i] = 0.f; }
}

}  // namespace solo

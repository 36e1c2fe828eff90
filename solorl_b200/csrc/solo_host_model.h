/*
 * solo_host_model.h — host-side conversion of the public tables (include/solo_b200.h)
 * into the kernel constants of solo_core.cuh: validates that the tree is
 * "floating base + 4 legs of NJL revolute joints + one fixed foot link each" (what
 * solo.urdf / solo12.urdf describe), merges each fixed FOOT link into its lower leg
 * (exact for the dynamics; the two bodies keep separate Bullet damping terms) and
 * narrows to float.  Replaces what p.loadURDF builds internally (reference solo.py:73).
 */
#pragma once
#include <math.h>
#include <string.h>

#include <string>

#include "../../include/solo_b200.h"
#include "solo_core.cuh"
#include "solo_env.cuh"

namespace solo {

inline int build_model_const(const SoloModelTable& t, ModelConst& mc, std::string& err) {
  memset(&mc, 0, sizeof(mc));
  if (t.abi_version != SOLO_ABI_VERSION) { err = "model table ABI version mismatch"; return SOLO_E_ARG; }
  if (t.num_links <= 0 || t.num_links > SOLO_MAX_LINKS) { err = "bad num_links"; return SOLO_E_MODEL; }
  if (t.num_feet != 4) { err = "model must have exactly 4 feet (ANKLE joints)"; return SOLO_E_MODEL; }
  for (int k = 0; k < 3; k++)
    if (t.base_com[k] != 0.0) { err = "base COM must be at the base origin"; return SOLO_E_MODEL; }
  /* dof numbering = revolute links in table order */
  int dof_of[SOLO_MAX_LINKS], nj = 0;
  for (int i = 0; i < t.num_links; i++) dof_of[i] = (t.jtype[i] == SOLO_JOINT_REVOLUTE) ? nj++ : -1;
  if (nj != 8 && nj != 12) { err = "expected 8 or 12 actuated joints"; return SOLO_E_MODEL; }
  const int njl = nj / 4;
  mc.njl = njl;
  for (int leg = 0; leg < 4; leg++) {
    int foot = t.foot_link[leg];
    if (foot < 0 || foot >= t.num_links || t.jtype[foot] != SOLO_JOINT_FIXED) {
      err = "foot link must hang off a fixed joint"; return SOLO_E_MODEL;
    }
    int chain[kMaxJL];
    int l = t.parent[foot];
    for (int k = njl - 1; k >= 0; k--) {
      if (l < 0 || t.jtype[l] != SOLO_JOINT_REVOLUTE) { err = "leg chain is not revolute up to the base"; return SOLO_E_MODEL; }
      chain[k] = l;
      l = t.parent[l];
    }
    if (l != -1) { err = "leg chain longer than expected"; return SOLO_E_MODEL; }
    LegConst& lc = mc.leg[leg];
    for (int k = 0; k < njl; k++) {
      int li = chain[k];
      if (dof_of[li] != leg * njl + k) { err = "joints must be ordered leg-major in the URDF"; return SOLO_E_MODEL; }
      int ax = (njl == 3 && k == 0) ? 0 : 1;
      for (int c = 0; c < 3; c++)
        if (t.axis[li][c] != (c == ax ? 1.0 : 0.0)) { err = "joint axis pattern must be (x,)y,y"; return SOLO_E_MODEL; }
      for (int c = 0; c < 3; c++) { lc.jo[k][c] = (float)t.origin[li][c]; lc.c[k][c] = (float)t.com[li][c]; }
      lc.m[k] = (float)t.mass[li];
      for (int c = 0; c < 6; c++) lc.I[k][c] = (float)t.inertia[li][c];
    }
    /* merge the foot into the last link (double precision, then narrow) */
    int last = chain[njl - 1];
    double m1 = t.mass[last], m2 = t.mass[foot], m = m1 + m2;
    double c1[3], c2[3], c[3];
    for (int k = 0; k < 3; k++) {
      c1[k] = t.com[last][k];
      c2[k] = t.origin[foot][k] + t.com[foot][k];
      c[k] = (m1 * c1[k] + m2 * c2[k]) / m;
    }
    double I[6];
    for (int k = 0; k < 6; k++) I[k] = t.inertia[last][k] + t.inertia[foot][k];
    const double* cs[2] = {c1, c2};
    const double ms[2] = {m1, m2};
    for (int b = 0; b < 2; b++) {
      double d[3] = {cs[b][0] - c[0], cs[b][1] - c[1], cs[b][2] - c[2]};
      double dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
      I[0] += ms[b] * (dd - d[0] * d[0]); I[1] += ms[b] * (-d[0] * d[1]); I[2] += ms[b] * (-d[0] * d[2]);
      I[3] += ms[b] * (dd - d[1] * d[1]); I[4] += ms[b] * (-d[1] * d[2]); I[5] += ms[b] * (dd - d[2] * d[2]);
    }
    lc.m[njl - 1] = (float)m;
    for (int k = 0; k < 3; k++) lc.c[njl - 1][k] = (float)c[k];
    for (int k = 0; k < 6; k++) lc.I[njl - 1][k] = (float)I[k];
    lc.m_own = (float)m1; lc.m_foot = (float)m2;
    for (int k = 0; k < 3; k++) {
      lc.c_own[k] = (float)c1[k];
      lc.c_foot[k] = (float)c2[k];
      lc.foot_ctr[k] = (float)(t.origin[foot][k] + t.foot_center[leg][k]);
    }
    for (int k = 0; k < 6; k++) lc.Idamp[k] = (float)(t.inertia[last][k] + t.inertia[foot][k]);
  }
  /* every link must be accounted for: 4*(njl+1) */
  if (t.num_links != 4 * (njl + 1)) { err = "unexpected extra links"; return SOLO_E_MODEL; }
  mc.base_m = (float)t.base_mass;
  for (int k = 0; k < 6; k++) mc.base_I[k] = (float)t.base_inertia[k];
  mc.foot_r = (float)t.foot_radius;
  return SOLO_OK;
}

inline int build_sim_const(const SoloSimParams& p, SimConst& sc, std::string& err) {
  memset(&sc, 0, sizeof(sc));
  if (p.abi_version != SOLO_ABI_VERSION) { err = "params ABI version mismatch"; return SOLO_E_ARG; }
  if (p.dt <= 0 || p.frame_skip <= 0 || p.solver_iters < 0 || p.episode_length <= 0 ||
      p.num_history_stack < 0 || p.settle_max < p.settle_min || p.settle_min < 0 ||
      p.solver_residual_threshold < 0) {
    err = "bad simulation parameters"; return SOLO_E_ARG;
  }
  if (p.control < 0 || p.control > 2 || p.task < 0 || p.task > 2) { err = "bad control/task"; return SOLO_E_ARG; }
  sc.dt = (float)p.dt; sc.inv_dt = (float)(1.0 / p.dt); sc.gz = (float)p.gravity_z;
  sc.klin = (float)p.lin_damping; sc.kang = (float)p.ang_damping; sc.vmax = (float)p.max_coord_vel;
  sc.erp = (float)p.contact_erp; sc.slop = (float)p.contact_slop; sc.margin = (float)p.contact_margin;
  sc.mu = (float)p.friction; sc.iters = p.solver_iters; sc.cone = p.cone_friction;
  sc.res_thr = (float)p.solver_residual_threshold;
  sc.frame_skip = p.frame_skip; sc.torque_hold = p.torque_hold;
  sc.control = p.control; sc.kp = (float)p.kp; sc.kd = (float)p.kd;
  sc.max_torque = (float)p.max_torque; sc.q_limit = (float)p.joint_state_limit;
  sc.qd_limit = (float)p.joint_vel_limit;
  sc.task = p.task; sc.episode_length = p.episode_length; sc.H = p.num_history_stack;
  sc.initial_z = (float)p.initial_z; sc.settle_min = p.settle_min;
  sc.settle_span = p.settle_max - p.settle_min;
  sc.goal_reach = (float)p.goal_reach_dist; sc.inv_pg_dt = (float)(1.0 / p.pointgoal_dt);
  sc.flag_force = (float)p.contact_flag_force; sc.fall_z = (float)p.fall_z; sc.stand_z = (float)p.stand_z;
  sc.reset_mode = p.reset_mode;
  sc.joint_limits = p.joint_limits ? 1 : 0;
  sc.lim_erp = (float)p.joint_limit_erp; sc.lim_max_impulse = (float)p.joint_limit_max_impulse;
  sc.lim_split_thr = (float)p.split_impulse_threshold;
  sc.body_contacts = p.body_contacts ? 1 : 0;
  if (p.body_contacts && (p.knee_radius < 0 || p.base_half_x <= 0 || p.base_half_y <= 0 || p.base_z_hi < p.base_z_lo)) {
    err = "body_contacts: bad knee radius / base box"; return SOLO_E_ARG;
  }
  sc.knee_r = (float)p.knee_radius; sc.base_hx = (float)p.base_half_x; sc.base_hy = (float)p.base_half_y;
  sc.base_zlo = (float)p.base_z_lo; sc.base_zhi = (float)p.base_z_hi;
  return SOLO_OK;
}

/* Ranges of the randomised dynamics, checked when SoloSimParams.randomize is set (and left 0 otherwise). */
inline int build_env_ranges(const SoloSimParams& p, EnvRanges& r, std::string& err) {
  memset(&r, 0, sizeof(r));
  if (!p.randomize) return SOLO_OK;
  if (!(p.friction_lo >= 0 && p.friction_lo <= p.friction_hi)) {
    err = "randomize: friction range must satisfy 0 <= friction_lo <= friction_hi"; return SOLO_E_ARG;
  }
  if (!(p.base_mass_scale_lo > 0 && p.base_mass_scale_lo <= p.base_mass_scale_hi)) {
    err = "randomize: base mass scale range must satisfy 0 < lo <= hi"; return SOLO_E_ARG;
  }
  if (!(p.motor_strength_lo > 0 && p.motor_strength_lo <= p.motor_strength_hi)) {
    err = "randomize: motor strength range must satisfy 0 < lo <= hi"; return SOLO_E_ARG;
  }
  r.mu_lo = (float)p.friction_lo; r.mu_hi = (float)p.friction_hi;
  r.sm_lo = (float)p.base_mass_scale_lo; r.sm_hi = (float)p.base_mass_scale_hi;
  r.st_lo = (float)p.motor_strength_lo; r.st_hi = (float)p.motor_strength_hi;
  return SOLO_OK;
}

/* Random pushes, checked when push_interval > 0 (and left 0 otherwise).  episode_length / interval < 2^30 keeps
 * the push draw index kPushDraw + j from wrapping. */
inline int build_push_params(const SoloSimParams& p, PushParams& pp, std::string& err) {
  memset(&pp, 0, sizeof(pp));
  if (!(isfinite(p.push_force) && p.push_force >= 0)) {
    err = "push: push_force must be finite and >= 0"; return SOLO_E_ARG;
  }
  if (p.push_interval < 0) { err = "push: push_interval must be >= 0 (0 = pushes off)"; return SOLO_E_ARG; }
  if (p.push_interval == 0) return SOLO_OK;
  if (p.push_duration < 1 || p.push_duration > p.push_interval) {
    err = "push: push_duration must satisfy 1 <= push_duration <= push_interval"; return SOLO_E_ARG;
  }
  if (p.episode_length / p.push_interval >= (1 << 30)) {
    err = "push: episode_length / push_interval must be below 2^30"; return SOLO_E_ARG;
  }
  pp.force = (float)p.push_force; pp.interval = p.push_interval; pp.duration = p.push_duration;
  return SOLO_OK;
}

inline void fill_default_params(SoloSimParams* p) {
  memset(p, 0, sizeof(*p));
  p->abi_version = SOLO_ABI_VERSION;
  p->dt = 1.0 / 240.0; p->frame_skip = 4; p->gravity_z = -9.81;
  p->lin_damping = 0.04; p->ang_damping = 0.04; p->max_coord_vel = 100.0;
  p->solver_iters = 50; p->solver_residual_threshold = 1e-7; p->contact_erp = 0.2; p->contact_slop = 1e-5; p->contact_margin = 0.02;
  p->friction = 1.0; p->cone_friction = 1; p->torque_hold = 0;
  p->control = SOLO_CONTROL_TORQUE; p->kp = 0; p->kd = 0; p->max_torque = 3.0;
  p->joint_state_limit = 10.0; p->joint_vel_limit = 100.0;
  p->task = SOLO_TASK_STAND; p->episode_length = 400; p->num_history_stack = 0;
  p->initial_z = 0.35; p->settle_min = 5; p->settle_max = 12;
  p->goal_radius = 2.0; p->goal_reach_dist = 0.5; p->pointgoal_dt = 4.0 / 240.0;
  p->contact_flag_force = 0.2; p->fall_z = 0.05; p->stand_z = 0.2;
  p->reset_mode = SOLO_RESET_CACHED;
  p->joint_limits = 1;
  p->limit_rows_per_leg = 1;
  p->joint_limit_erp = 0.2;
  p->joint_limit_max_impulse = 100.0;
  p->split_impulse_threshold = -0.04;
  p->body_contacts = 0;
  p->knee_radius = 0.015;
  p->base_half_x = 0.2241; p->base_half_y = 0.1095;
  p->base_z_lo = -0.025; p->base_z_hi = 0.028;
}

}  // namespace solo

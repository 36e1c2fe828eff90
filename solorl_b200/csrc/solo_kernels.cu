/*
 * solo_kernels.cu — sm_100a kernels and the C-ABI (include/solo_b200.h) of the batched
 * Solo8/Solo12 env step.
 *
 * step_kernel: ONE launch per env step.  Thread t of a warp = (env t/4, leg t%4): four lanes
 * per environment, eight environments per warp, 4 or 8 warps per block (two builds, see the comment
 * above step_kernel).  At 4096 envs that is 512 warps for the 592 warp schedulers of a B200: the step
 * is a dependent-latency problem, so the design minimises the per-warp instruction chain rather than
 * occupancy.  All cross-leg traffic — the sum of the four legs' articulated inertias into the
 * floating base, the exchange of IA0^-1 P blocks for the Delassus rows, and the one-value
 * broadcast per projected-Gauss-Seidel row relaxation — is full-mask register shuffles of a
 * converged warp.  Shared memory holds the per-leg model constants and one staging tile per warp
 * through which action words arrive and observation rows leave as whole 128-byte lines; the one
 * block barrier per substep keeps the warps of an SM on the same instruction-cache lines.
 *
 * HBM layout (structure of arrays, fp32):
 *   base  [cap][16]  : pos3 quat4 linvel3 angvel3 goal2 potential1   (4 x float4 per env)
 *   q,qd  [NJL][cap][4] : joint k of leg l of env e at ((k*cap+e)*4+l)  (one float4 per env and k,
 *                      consecutive threads read consecutive words)
 *   cforce[cap][4]   : normal force of the last substep per foot, <0 = no contact point
 *   hist  [H][cap][D0], currow [cap][D0], book [cap] (EnvBook), stats [cap] (SoloEpisodeStats)
 */
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/solo_b200.h"
#include "solo_core.cuh"
#include "solo_body.cuh"
#include "solo_env.cuh"
#include "solo_host_model.h"

namespace solo {

constexpr int kBlockThreads = 32;   /* threads per env warp: eight envs x four legs */

enum { MODE_STEP = 0, MODE_SETTLE = 1, MODE_SUBSTEP = 2 };
enum { VARIANT_LATENCY = 0, VARIANT_THROUGHPUT = 1, VARIANT_WIDE = 2 };

struct DevArrays {
  float* base;
  float* q;
  float* qd;
  float* cforce;
  float* hist;
  float* currow;     /* [cap][D0] get_current_state() of the env as it stands (the row the next step pushes into the history) */
  EnvBook* book;
  SoloEpisodeStats* stats;
  /* reset cache: one row per settle count (settle_min + row) */
  float* rc_base;    /* [K][16] */
  float* rc_q;       /* [K][12] leg-major */
  float* rc_qd;
  float* rc_cforce;  /* [K][4] */
  float* rc_hist;    /* [K][H][D0] */
  /* run-time mutable scalars, read by the kernels from device memory so that a captured CUDA graph of the
   * step sees later updates: [0] = pointgoal goal radius (increment_goal_radius, solo.py:332-334) */
  const float* mut;
  /* gait envs: external force on the base, base axes, acting at the base origin ([3P] the random pushes of
   * baseControlEnv.py:276-289 go through pyb.applyExternalForce(robot, -1, F, 0, LINK_FRAME)); [cap][4], zero by
   * default; read by the actuator kernel only */
  float* fext;
  int cap;
};
enum { kMutGoalRadius = 0, kMutCount = 4 };

struct StepArgs {
  DevArrays d;
  SimConst sc;
  ModelConst mc;
  int n, mode;
  int D0, D, A;
  const float* in;   /* actions [n][A] (STEP) or joint torques [n][nj] (SUBSTEP) */
  float* obs;
  float* reward;
  float* done;
  uint32_t seed_lo, seed_hi;
  long long env_id_offset;
  int reset_simulate; /* 1: done envs restart from the reset pose with settle_left = k */
  int force_settle;   /* >=0: cache generation, env i settles settle_min + i steps, goal far away */
};

/* Randomised dynamics of a handle: per-env (mu, base mass scale, motor strength, 0) and the ranges a reset draws
 * them from; envp == nullptr: randomisation off.  A kernel parameter of its own, after StepArgs, so that the
 * kernels without randomisation keep their parameter layout.  push: the random pushes (interval 0 = off), last
 * so that nothing before it moves. */
struct DynArgs {
  float4* envp;
  EnvRanges ranges;
  PushParams push;
};

struct ResetArgs {
  DevArrays d;
  SimConst sc;
  int n, njl, D0, D;
  const uint8_t* mask;
  float* obs;
  uint32_t seed_lo, seed_hi;
  long long env_id_offset;
  int reset_simulate, force_settle;
  DynArgs dyn;
};

/* Observation rows of the eight envs of a warp are assembled in shared memory and leave the SM as
 * whole 128-byte lines (8 x D contiguous floats per warp): the row pieces come from four lanes in
 * 4-byte scraps, which is tolerable for HBM but not for the host-mapped output buffers of
 * solo_step_host, where every store is a PCIe write. */
constexpr int kStageD = 128;   /* rows up to 128 floats are staged (D = 76 / 84 for H = 1); longer ones go direct */
struct Smem {
  LegConst leg[4];
};

/* sum over the four lanes of an env (xor butterfly; the whole warp is converged) */
__device__ __forceinline__ float sum4(float x) {
  x += __shfl_xor_sync(0xffffffffu, x, 1);
  x += __shfl_xor_sync(0xffffffffu, x, 2);
  return x;
}
__device__ __forceinline__ void sum4_sym6(Sym6& I) {
#pragma unroll
  for (int i = 0; i < 6; i++) I.A[i] = sum4(I.A[i]);
#pragma unroll
  for (int i = 0; i < 9; i++) I.H[i] = sum4(I.H[i]);
#pragma unroll
  for (int i = 0; i < 6; i++) I.M[i] = sum4(I.M[i]);
}

/* ---- the pieces of one D0-row of the observation that a lane produces -------------- */
template <int NJL>
struct RowPieces {
  float base[10], pg[4], qn[NJL], qdn[NJL], flag;
};
template <int NJL>
__device__ __forceinline__ void make_pieces(const SimConst& sc, const BaseState& st, const Lane<NJL>& ln,
                                            float cforce, const float* goal, RowPieces<NJL>& r) {
  cur_base(st, r.base);
#pragma unroll
  for (int k = 0; k < NJL; k++) { r.qn[k] = ln.q[k] / sc.q_limit; r.qdn[k] = ln.qd[k] / sc.qd_limit; }
  r.flag = contact_flag(sc, cforce);
  if (sc.task == 2) cur_pointgoal(st, goal, r.pg);
  else { r.pg[0] = r.pg[1] = r.pg[2] = r.pg[3] = 0.f; }
}
template <int NJL>
__device__ __forceinline__ void store_pieces(float* row, int leg, int task, const RowPieces<NJL>& r) {
#pragma unroll
  for (int k = 0; k < NJL; k++) { row[idx_q(NJL, leg, k)] = r.qn[k]; row[idx_qd(NJL, leg, k)] = r.qdn[k]; }
  row[idx_flag(NJL, leg)] = r.flag;
  if (leg == 0) {
#pragma unroll
    for (int i = 0; i < 10; i++) row[i] = r.base[i];
    if (task == 2) {
#pragma unroll
      for (int i = 0; i < 4; i++) row[idx_pg(NJL) + i] = r.pg[i];
    }
  }
}
template <int NJL>
__device__ __forceinline__ void load_pieces(const float* row, int leg, int task, RowPieces<NJL>& r) {
#pragma unroll
  for (int k = 0; k < NJL; k++) { r.qn[k] = row[idx_q(NJL, leg, k)]; r.qdn[k] = row[idx_qd(NJL, leg, k)]; }
  r.flag = row[idx_flag(NJL, leg)];
  if (leg == 0) {
#pragma unroll
    for (int i = 0; i < 10; i++) r.base[i] = row[i];
    if (task == 2) {
#pragma unroll
      for (int i = 0; i < 4; i++) r.pg[i] = row[idx_pg(NJL) + i];
    }
  }
}
template <int NJL>
__device__ __forceinline__ void diff_pieces(const RowPieces<NJL>& a, const RowPieces<NJL>& b, RowPieces<NJL>& o) {
#pragma unroll
  for (int i = 0; i < 10; i++) o.base[i] = a.base[i] - b.base[i];
#pragma unroll
  for (int i = 0; i < 4; i++) o.pg[i] = a.pg[i] - b.pg[i];
#pragma unroll
  for (int k = 0; k < NJL; k++) { o.qn[k] = a.qn[k] - b.qn[k]; o.qdn[k] = a.qdn[k] - b.qdn[k]; }
  o.flag = a.flag - b.flag;
}

__device__ __forceinline__ float* hist_row(const DevArrays& d, int D0, int h, int e) {
  return d.hist + ((size_t)h * d.cap + e) * D0;
}

/* get_current_state() of every env is kept as a row of its own (currow), refreshed wherever the state changes
 * (step / settle / substep epilogue, reset, set_state, set_contacts, set_goals).  The history push at the start of
 * a step (solo.py:262) then copies that row instead of re-deriving it: the observation arithmetic (Euler angles
 * from the quaternion, ...) is ~600 SASS instructions per inlined copy, and the step is bound by instruction
 * fetch (profiles/r2_icache_probe.txt). */
__device__ __forceinline__ float* cur_row(const DevArrays& d, int D0, int e) { return d.currow + (size_t)e * D0; }

/* deque(maxlen=H).append(get_current_state()) (solo.py:262) */
template <int NJL>
__device__ __forceinline__ void push_history(const DevArrays& d, const SimConst& sc, int D0, int e, int leg,
                                             const RowPieces<NJL>& cur) {
  for (int h = sc.H - 1; h > 0; h--) {
    RowPieces<NJL> t;
    load_pieces<NJL>(hist_row(d, D0, h - 1, e), leg, sc.task, t);
    store_pieces<NJL>(hist_row(d, D0, h, e), leg, sc.task, t);
  }
  if (sc.H > 0) store_pieces<NJL>(hist_row(d, D0, 0, e), leg, sc.task, cur);
}

/* calc_state (solo.py:186-196): [cur, cur - hist[0], cur - hist[1], ...] */
template <int NJL>
__device__ __forceinline__ void write_obs_row(const DevArrays& d, const SimConst& sc, int D0, int e, int leg,
                                              const RowPieces<NJL>& cur, float* row) {
  store_pieces<NJL>(row, leg, sc.task, cur);
  for (int h = 0; h < sc.H; h++) {
    RowPieces<NJL> old, df;
    load_pieces<NJL>(hist_row(d, D0, h, e), leg, sc.task, old);
    diff_pieces<NJL>(cur, old, df);
    store_pieces<NJL>(row + (size_t)(1 + h) * D0, leg, sc.task, df);
  }
}
template <int NJL>
__device__ __forceinline__ void write_obs(const DevArrays& d, const SimConst& sc, int D0, int D, int e, int leg,
                                          const RowPieces<NJL>& cur, float* obs) {
  float* row = obs + (size_t)e * D;
  store_pieces<NJL>(row, leg, sc.task, cur);
  for (int h = 0; h < sc.H; h++) {
    RowPieces<NJL> old, df;
    load_pieces<NJL>(hist_row(d, D0, h, e), leg, sc.task, old);
    diff_pieces<NJL>(cur, old, df);
    store_pieces<NJL>(row + (size_t)(1 + h) * D0, leg, sc.task, df);
  }
}

__device__ __forceinline__ void env_rng(uint32_t seed_lo, uint32_t seed_hi, long long gid, EnvBook& bk, uint32_t* w) {
  w[0] = (uint32_t)((unsigned long long)gid & 0xffffffffull);
  w[1] = (uint32_t)((unsigned long long)gid >> 32);
  w[2] = bk.episode;
  w[3] = bk.draw++;
  philox4x32_10(w, seed_lo, seed_hi);
}

__device__ __forceinline__ void load_base(const float* base, int e, BaseState& st, float* goal, float& potential) {
  const float4* b = reinterpret_cast<const float4*>(base + (size_t)e * kBaseStride);
  float4 b0 = b[0], b1 = b[1], b2 = b[2], b3 = b[3];
  st.p[0] = b0.x; st.p[1] = b0.y; st.p[2] = b0.z;
  st.q[0] = b0.w; st.q[1] = b1.x; st.q[2] = b1.y; st.q[3] = b1.z;
  st.v[0] = b1.w; st.v[1] = b2.x; st.v[2] = b2.y;
  st.w[0] = b2.z; st.w[1] = b2.w; st.w[2] = b3.x;
  goal[0] = b3.y; goal[1] = b3.z; potential = b3.w;
}
__device__ __forceinline__ void store_base(float* base, int e, const BaseState& st, const float* goal, float potential) {
  float4* b = reinterpret_cast<float4*>(base + (size_t)e * kBaseStride);
  b[0] = make_float4(st.p[0], st.p[1], st.p[2], st.q[0]);
  b[1] = make_float4(st.q[1], st.q[2], st.q[3], st.v[0]);
  b[2] = make_float4(st.v[1], st.v[2], st.w[0], st.w[1]);
  b[3] = make_float4(st.w[2], goal[0], goal[1], potential);
}

/* SoloBaseEnv.reset up to (not including) the settle loop (baseEnv.py:70-77, solo.py:166-181),
 * or — cached mode — the memoised result of the whole reset for the drawn settle count. */
template <int NJL>
__device__ __forceinline__ void begin_reset(const DevArrays& d, const SimConst& sc, int D0, int e, int leg,
                                            long long gid, uint32_t seed_lo, uint32_t seed_hi, float goal_radius,
                                            int reset_simulate, int force_settle, BaseState& st, Lane<NJL>& ln,
                                            float& cforce, float* goal, float& potential, EnvBook& bk,
                                            const DynArgs* dyn = nullptr) {
  bk.episode += 1; bk.draw = 0;
  uint32_t w[4];
  env_rng(seed_lo, seed_hi, gid, bk, w);
  if (dyn != nullptr && dyn->envp != nullptr && leg == 0) {    /* the new episode's dynamics */
    const EnvDyn p = sample_env_dyn(dyn->ranges, seed_lo, seed_hi, gid, bk.episode);
    dyn->envp[e] = make_float4(p.mu, p.sm, p.st, 0.f);
  }
  if (sc.task == 2) sample_goal(w, goal_radius, goal);          /* solo.py:173-174 */
  int k = sc.settle_min + (sc.settle_span > 0 ? (int)(w[0] % (uint32_t)sc.settle_span) : 0); /* baseEnv.py:79 */
  if (force_settle >= 0) { k = sc.settle_min + (e % (sc.settle_span > 0 ? sc.settle_span : 1)); goal[0] = 1.0e3f; goal[1] = 1.0e3f; }
  book_clear_episode(bk);
  bk.goals = 0;
  if (reset_simulate) {
    reset_pose(sc, st);
#pragma unroll
    for (int j = 0; j < NJL; j++) { ln.q[j] = 0.f; ln.qd[j] = 0.f; }
    cforce = -1.0f;                                              /* contact set cleared */
    RowPieces<NJL> cur;
    make_pieces<NJL>(sc, st, ln, cforce, goal, cur);
    for (int h = 0; h < sc.H; h++) store_pieces<NJL>(hist_row(d, D0, h, e), leg, sc.task, cur); /* solo.py:170-171 */
    store_pieces<NJL>(cur_row(d, D0, e), leg, sc.task, cur);
    bk.settle_left = k;
  } else {
    const int row = k - sc.settle_min;
    float g2[2], pot;
    load_base(d.rc_base, row, st, g2, pot);
#pragma unroll
    for (int j = 0; j < NJL; j++) {
      ln.q[j] = d.rc_q[row * 12 + leg * NJL + j];
      ln.qd[j] = d.rc_qd[row * 12 + leg * NJL + j];
    }
    cforce = d.rc_cforce[row * 4 + leg];
    for (int h = 0; h < sc.H; h++) {
      RowPieces<NJL> t;
      load_pieces<NJL>(d.rc_hist + ((size_t)row * sc.H + h) * D0, leg, sc.task, t);
      t.pg[2] = goal[0] / 2.0f; t.pg[3] = goal[1] / 2.0f;
      store_pieces<NJL>(hist_row(d, D0, h, e), leg, sc.task, t);
    }
    bk.settle_left = 0;
  }
  potential = (sc.task == 2) ? calc_potential(st, goal) : 0.f;   /* solo.py:176 */
}

/* The projected Gauss-Seidel sweep loop of one env over its four lanes (PgsLane: each lane owns the
 * three rows of its foot).  Per row relaxation: the owner's candidate, ONE shuffle broadcast of the
 * impulse change inside the 4-lane group, three FMAs in every lane.  An env whose sweep met Bullet's
 * residual test keeps relaxing until the whole warp is done (no per-row select on the dependent chain);
 * its impulses are latched into lam3 at the sweep that converged, so the result is exactly that of
 * stopping there.  CONE selects Bullet's implicit-cone friction rows or the pyramid ones. */
template <bool CONE>
__device__ __forceinline__ void pgs_sweeps(PgsLane& pl, const SimConst& sc, int leg, unsigned gbase, unsigned amask,
                                           int nc, float* lam3, int& sweep_feet, const EnvDyn* dyn) {
  const unsigned kFull = 0xffffffffu;
  bool conv = (amask == 0);          /* env-uniform: the sweep loop of this env has ended */
  lam3[0] = lam3[1] = lam3[2] = 0.f;
  for (int it = 0; it < sc.iters; it++) {
    float res_own = 0.f;             /* largest |velocity residual| among the rows this lane relaxed */
    sweep_feet += conv ? 0 : nc;
#pragma unroll
    for (int f = 0; f < 4; f++) {   /* feet without contact hold zero rows: no skip branches (measured: warp-uniform
                                     * skips of the rows no still-iterating env holds cost more than they save:
                                     * 105.6 vs 90.1 us per step at 4096 envs, profiles/r2_experiments.txt) */
      float nv, d, rv;
      pgs_normal_candidate(pl, nv, d, rv);
      const float db = __shfl_sync(kFull, d, gbase + f);
      if (leg == f) { pgs_normal_commit(pl, nv); res_own = fmaxf(res_own, fabsf(rv)); }
      pgs_apply(pl, row_of(f, 0), db);
    }
#pragma unroll
    for (int f = 0; f < 4; f++) {
      if (CONE) {
        float nA, nB, dA, dB, rv;
        pgs_cone_candidate(pl, env_mu(sc, dyn), nA, nB, dA, dB, rv);
        const float dAb = __shfl_sync(kFull, dA, gbase + f);
        const float dBb = __shfl_sync(kFull, dB, gbase + f);
        if (leg == f) { pl.lam[1] = nA; pl.lam[2] = nB; res_own = fmaxf(res_own, fabsf(rv)); }
        pgs_apply(pl, row_of(f, 1), dAb);
        pgs_apply(pl, row_of(f, 2), dBb);
      } else {
#pragma unroll
        for (int q = 0; q < 2; q++) {
          float nv, d, rv;
          pgs_pyramid_candidate(pl, env_mu(sc, dyn), q, nv, d, rv);
          const float db = __shfl_sync(kFull, d, gbase + f);
          if (leg == f) { pl.lam[1 + q] = nv; res_own = fmaxf(res_own, fabsf(rv)); }
          pgs_apply(pl, row_of(f, 1 + q), db);
        }
      }
    }
    if (!conv) { lam3[0] = pl.lam[0]; lam3[1] = pl.lam[1]; lam3[2] = pl.lam[2]; }
    /* end of sweep, Bullet's exit test: the env is done when every row residual of the sweep is
     * within the threshold, i.e. when each of its four lanes is; one ballot serves the env test
     * and the warp-wide loop exit */
    const unsigned okb = __ballot_sync(kFull, conv || (res_own * res_own <= sc.res_thr));
    conv = conv || (((okb >> gbase) & 0xFu) == 0xFu);
    if (okb == kFull) break;
  }
}

/* The sweep loop when some env of the warp holds a joint-limit row: a fourth row per lane, relaxed first in
 * every sweep like Bullet's non-contact rows (under random actions 11 % of env steps hold a limit row). */
template <bool CONE>
__device__ __forceinline__ void pgs_sweeps4(PgsLane4& pl, const SimConst& sc, int leg, unsigned gbase, unsigned amask,
                                            unsigned lmask, unsigned lwarp, int nc, float* lam4, int& sweep_feet,
                                            const EnvDyn* dyn) {
  const unsigned kFull = 0xffffffffu;
  bool conv = (amask == 0) && (lmask == 0);
  lam4[0] = lam4[1] = lam4[2] = lam4[3] = 0.f;
  for (int it = 0; it < sc.iters; it++) {
    float res_own = 0.f;
    sweep_feet += conv ? 0 : nc;
    {   /* (a warp-uniform `if (lwarp)` around this block was measured slower: 94.6 vs 90.1 us at 4096 envs) */
      /* the (at most four) limit rows of an env belong to different legs and are relaxed as ONE group: every
       * lane takes its candidate from the same state, the four changes are exchanged in one shuffle round.
       * With a single limit row per env (99.5 % of the cases under random actions) this IS Bullet's
       * sequential order; with several it is a Jacobi step among rows that couple only through the base. */
      float nv, d, rv;
      pgs_limit_candidate(pl, sc.lim_max_impulse, nv, d, rv);
      pgs_limit_commit(pl, sc.lim_max_impulse, nv);
      res_own = fmaxf(res_own, fabsf(rv));
      const float d0 = __shfl_sync(kFull, d, gbase + 0), d1 = __shfl_sync(kFull, d, gbase + 1);
      const float d2 = __shfl_sync(kFull, d, gbase + 2), d3 = __shfl_sync(kFull, d, gbase + 3);
      pgs_apply(pl, limit_col(0), d0);
      pgs_apply(pl, limit_col(1), d1);
      pgs_apply(pl, limit_col(2), d2);
      pgs_apply(pl, limit_col(3), d3);
    }
#pragma unroll
    for (int f = 0; f < 4; f++) {
      float nv, d, rv;
      pgs_normal_candidate(pl, nv, d, rv);
#ifdef SOLO_EXP_NOSHFL_NORMALS   /* timing experiment only (wrong results): the normal rounds without their shuffle */
      const float db = d;
#else
      const float db = __shfl_sync(kFull, d, gbase + f);
#endif
      if (leg == f) { pgs_normal_commit(pl, nv); res_own = fmaxf(res_own, fabsf(rv)); }
      pgs_apply(pl, row_of(f, 0), db);
    }
#pragma unroll
    for (int f = 0; f < 4; f++) {
      if (CONE) {
        float nA, nB, dA, dB, rv;
        pgs_cone_candidate(pl, env_mu(sc, dyn), nA, nB, dA, dB, rv);
        const float dAb = __shfl_sync(kFull, dA, gbase + f);
        const float dBb = __shfl_sync(kFull, dB, gbase + f);
        if (leg == f) { pl.lam[1] = nA; pl.lam[2] = nB; res_own = fmaxf(res_own, fabsf(rv)); }
        pgs_apply(pl, row_of(f, 1), dAb);
        pgs_apply(pl, row_of(f, 2), dBb);
      } else {
#pragma unroll
        for (int q = 0; q < 2; q++) {
          float nv, d, rv;
          pgs_pyramid_candidate(pl, env_mu(sc, dyn), q, nv, d, rv);
          const float db = __shfl_sync(kFull, d, gbase + f);
          if (leg == f) { pl.lam[1 + q] = nv; res_own = fmaxf(res_own, fabsf(rv)); }
          pgs_apply(pl, row_of(f, 1 + q), db);
        }
      }
    }
    if (!conv) { lam4[0] = pl.lam[0]; lam4[1] = pl.lam[1]; lam4[2] = pl.lam[2]; lam4[3] = pl.lam[3]; }
    const unsigned okb = __ballot_sync(kFull, conv || (res_own * res_own <= sc.res_thr));
    conv = conv || (((okb >> gbase) & 0xFu) == 0xFu);
    if (okb == kFull) break;
  }
}

/* SOLO_TRACE builds (tools only): cycle stamps inside the substeps of the narrow builds, lane 0 of every block */
#ifdef SOLO_TRACE
__device__ long long g_narrow_trace[1024][8][8];
__device__ int g_trace_substep;
#define NSTAMP(i) do { if (threadIdx.x == 0 && blockIdx.x < 1024) g_narrow_trace[blockIdx.x][g_trace_sub & 7][i] = clock64(); } while (0)
/* kernel-level stamps (slot 4 of the block's record): 0 entry, 1 after step_load, 2 before step_finish, 3 end */
#define KSTAMP(i) do { if (threadIdx.x == 0 && blockIdx.x < 1024) g_narrow_trace[blockIdx.x][4][i] = clock64(); } while (0)
#else
#define NSTAMP(i) do { } while (0)
#define KSTAMP(i) do { } while (0)
#endif

/* Second half of a substep for the four lanes of an env: contact / joint-limit rows -> Delassus rows ->
 * projected Gauss-Seidel -> impulses -> position update.  In: ln (P, K, sP, Lm, b, dist, active of the own
 * foot and the ABA by-products r, ax, h, invD), bw (pre-update rotation, LDL factor), the limit-row selection. */
template <int NJL, bool LIMITS, bool BODY>
__device__ __forceinline__ void contact_solve(const SimConst& sc, int leg, BaseState& st, const BaseWork& bw,
                                              Lane<NJL>& ln, bool lim_env, int kL, float dirL, float penL,
                                              float& cforce, int& nc_sum, int& sweep_feet, int g_trace_sub = 0,
                                              float* body_rows = nullptr, const EnvDyn* dyn = nullptr) {
  const unsigned kFull = 0xffffffffu;
  const unsigned lane = threadIdx.x & 31u;
  const unsigned gbase = lane & ~3u;
  /* BODY (SoloSimParams.body_contacts): an env with a knee or a base corner on the ground solves ALL its rows on
   * the general path (solo_body.cuh) and takes part in the register path below with empty rows -- the choice is
   * per env, never per warp, so an env's result does not depend on its neighbours */
  const int foot_on = ln.active;
  bool body_env = false;
  unsigned pmask = 0;
  BodyLaneGeom<NJL> bg;
  if (BODY) {
    body_lane_geometry<NJL>(sc, st, bw, ln, leg, bg);
    const unsigned bf = __ballot_sync(kFull, foot_on != 0), bk = __ballot_sync(kFull, bg.kn_on);
    const unsigned b0 = __ballot_sync(kFull, bg.c_on[0]), b1 = __ballot_sync(kFull, bg.c_on[1]);
    pmask = ((bf >> gbase) & 0xFu) | (((bk >> gbase) & 0xFu) << 4) | (((b0 >> gbase) & 0xFu) << 8) |
            (((b1 >> gbase) & 0xFu) << 12);
    body_env = (pmask >> 4) != 0;
    if (body_env) ln.active = 0;
  }
  const bool lim_any = lim_env && !body_env;
  const unsigned ball = __ballot_sync(kFull, ln.active != 0);
  const unsigned amask = (ball >> gbase) & 0xFu;                 /* feet in contact of this env */
  const unsigned wmask = (ball | (ball >> 4) | (ball >> 8) | (ball >> 12) | (ball >> 16) | (ball >> 20) |
                          (ball >> 24) | (ball >> 28)) & 0xFu;     /* ... of any env of the warp */
  const unsigned lball = __ballot_sync(kFull, lim_any);
  const unsigned lmask = (lball >> gbase) & 0xFu;
  const unsigned lwarp = (lball | (lball >> 4) | (lball >> 8) | (lball >> 12) | (lball >> 16) | (lball >> 20) |
                          (lball >> 24) | (lball >> 28)) & 0xFu;
  float lam3[3] = {0.f, 0.f, 0.f};
  /* LIMITS (joint_limits on, the reference behaviour): every warp with a contact or a limit row takes the
   * four-row path, so that one env step executes ONE solve path -- the step is bound by instruction fetch
   * (profiles/r2_icache_probe.txt), and a block whose warps split over the three-row and the four-row code
   * streams both through the instruction caches every substep */
  if (LIMITS ? (lwarp | wmask) != 0 : false) {   /* warp-uniform */
    LimitRow<NJL> lr;
    limit_setup<NJL>(sc, bw, ln, lim_any, kL, dirL, penL, lr);
    PgsLane4 pl;
    {
      float rows[4][kRowsL];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        float Kj[3][6], KLj[6];
#pragma unroll
        for (int n = 0; n < 3; n++) {
#pragma unroll
          for (int i = 0; i < 6; i++) Kj[n][i] = __shfl_sync(kFull, ln.K[n][i], gbase + j);
        }
        const bool col_on = ((lwarp >> j) & 1u) != 0;   /* warp-uniform */
#pragma unroll
        for (int i = 0; i < 6; i++) KLj[i] = col_on ? __shfl_sync(kFull, lr.K[i], gbase + j) : 0.f;
        assemble_block4<NJL>(ln, lr, leg, j, Kj, KLj, col_on, rows);
      }
      pgs_lane_init4<NJL>(ln, lr, leg, rows, amask, lmask, sc.lim_max_impulse, pl);
    }
    const int nc = __popc(amask);
    nc_sum += nc;
    float lam4[4];
    NSTAMP(3);
    if (sc.cone) pgs_sweeps4<true>(pl, sc, leg, gbase, amask, lmask, lwarp, nc, lam4, sweep_feet, dyn);
    else pgs_sweeps4<false>(pl, sc, leg, gbase, amask, lmask, lwarp, nc, lam4, sweep_feet, dyn);
    NSTAMP(4);
    lam3[0] = lam4[0]; lam3[1] = lam4[1]; lam3[2] = lam4[2];
    float part[6], dv0[6];
    impulse_base_part4<NJL>(ln, lr, lam4, part);
#pragma unroll
    for (int i = 0; i < 6; i++) dv0[i] = sum4(part[i]);
    impulse_leg4<NJL>(ln, lr, sc, lam4, dv0);
    float dw[3], dvl[3];
    mat3_mulv(bw.R, dv0, dw);
    mat3_mulv(bw.R, dv0 + 3, dvl);
    base_add_velocity(sc, st, dw, dvl, 1.0f);
  } else if (!LIMITS && wmask) {   /* warp-uniform */
    PgsLane pl;
    {
      float rows[3][kRows];
#pragma unroll
      for (int j = 0; j < 4; j++) {
        float Kj[3][6];
#pragma unroll
        for (int n = 0; n < 3; n++) {
#pragma unroll
          for (int i = 0; i < 6; i++) Kj[n][i] = __shfl_sync(kFull, ln.K[n][i], gbase + j);
        }
        assemble_block<NJL>(ln, leg, j, Kj, rows);
      }
      pgs_lane_init<NJL>(ln, leg, rows, amask, pl);
    }
    const int nc = __popc(amask);
    nc_sum += nc;
    if (sc.cone) pgs_sweeps<true>(pl, sc, leg, gbase, amask, nc, lam3, sweep_feet, dyn);
    else pgs_sweeps<false>(pl, sc, leg, gbase, amask, nc, lam3, sweep_feet, dyn);
    float part[6], dv0[6];
    impulse_base_part<NJL>(ln, lam3, part);
#pragma unroll
    for (int i = 0; i < 6; i++) dv0[i] = sum4(part[i]);
    impulse_leg<NJL>(ln, sc, lam3, dv0);
    float dw[3], dvl[3];
    mat3_mulv(bw.R, dv0, dw);
    mat3_mulv(bw.R, dv0 + 3, dvl);
    base_add_velocity(sc, st, dw, dvl, 1.0f);
  }
  if (BODY) {
    ln.active = foot_on;
    if (body_env) {                  /* diverges between the envs of a warp; the four lanes of an env stay together */
      const unsigned gmask = 0xFu << gbase;
      const unsigned lm_all = (__ballot_sync(gmask, lim_env) >> gbase) & 0xFu;
      LimitRow<NJL> lr;
      lr.active = 0;
      if (LIMITS) limit_setup<NJL>(sc, bw, ln, lim_env, kL, dirL, penL, lr);
      body_lane_fill<NJL>(sc, st, bw, ln, LIMITS ? &lr : nullptr, leg, foot_on != 0, bg, body_rows);
      __syncwarp(gmask);
      float dv0[6], us[3];
      const int sweeps = sc.cone ? body_pgs_lanes<true>(body_rows, lm_all, pmask, sc, gmask, gbase, leg, dv0, us, dyn)
                                 : body_pgs_lanes<false>(body_rows, lm_all, pmask, sc, gmask, gbase, leg, dv0, us, dyn);
      body_apply_leg<NJL>(ln, sc, us, dv0);
      float dw[3], dvl[3];
      mat3_mulv(bw.R, dv0, dw);
      mat3_mulv(bw.R, dv0 + 3, dvl);
      base_add_velocity(sc, st, dw, dvl, 1.0f);
      lam3[0] = foot_on ? body_rows[body_slot(leg, 0) * kBodyRowW + kBrLam] : 0.f;
      const int np = __popc(pmask);
      nc_sum += np;
      sweep_feet += np * sweeps;
      __syncwarp(gmask);
    }
    __syncwarp();
  }
  cforce = ln.active ? lam3[0] * sc.inv_dt : -1.0f;
  integrate_base(sc, st);
#pragma unroll
  for (int k = 0; k < NJL; k++) ln.q[k] += sc.dt * ln.qd[k];
}

/* One Bullet-equivalent substep for the four lanes of an env (see solo_core.cuh).
 * Control flow is kept WARP-uniform (skip masks and the sweep-loop exit are warp votes, envs that
 * have nothing to do contribute exact zeros) so that every shuffle is a full-mask shuffle of a
 * converged warp: group-masked shuffles cost a WARPSYNC each and let the 4-lane groups drift apart. */
template <int NJL, bool LIMITS, bool BODY = false>
__device__ __forceinline__ void group_substep(const LegConst& lc, const ModelConst& mc, const SimConst& sc,
                                              int leg, BaseState& st, Lane<NJL>& ln, const float* tau, float& cforce,
                                              int& nc_sum, int& sweep_feet, int g_trace_sub = 0,
                                              const float* fext = nullptr, float* body_rows = nullptr,
                                              const EnvDyn* dyn = nullptr) {
  NSTAMP(0);
  BaseWork bw;
  base_prepare(st, bw);
  Sym6 IA;
  float pA[6], a0[6];
  leg_inward<NJL>(lc, sc, bw, ln, tau, IA, pA);
  sum4_sym6(IA);
#pragma unroll
  for (int i = 0; i < 6; i++) pA[i] = sum4(pA[i]);
  if (fext != nullptr) {               /* external force on the base (gait envs): enters the bias force with a minus */
#pragma unroll
    for (int i = 0; i < 3; i++) pA[3 + i] -= fext[i];
  }
  base_solve(mc, sc, bw, IA, pA, a0, dyn);
  {
    float qdd[NJL], aw[3], al[3];
    leg_outward<NJL>(ln, a0, qdd);
    base_world_acc(sc, bw, a0, aw, al);
    base_add_velocity(sc, st, aw, al, sc.dt);
#pragma unroll
    for (int k = 0; k < NJL; k++) ln.qd[k] = clampf(ln.qd[k] + sc.dt * qdd[k], -sc.vmax, sc.vmax);
  }
  NSTAMP(1);
  contact_setup<NJL>(lc, mc, sc, st, bw, ln);
  NSTAMP(2);
  /* joint-limit rows (positions of the start of the substep, velocities after the unconstrained update) */
  int kL;
  float dirL, penL;
  const bool lim_any = LIMITS && limit_select<NJL>(sc, ln, kL, dirL, penL);
  contact_solve<NJL, LIMITS, BODY>(sc, leg, st, bw, ln, lim_any, kL, dirL, penL, cforce, nc_sum, sweep_feet, g_trace_sub,
                                   body_rows, dyn);
  NSTAMP(5);
}

/* Everything an (env, leg) lane carries in registers through one env step. */
template <int NJL>
struct EnvLane {
  BaseState st;
  float goal[2], potential;
  Lane<NJL> ln;
  float cforce;
  EnvBook bk;
  float tau[NJL], act[NJL];
  EnvDyn dyn;          /* RAND builds only */
  int e, el, leg, tid;
  long long gid;
  bool valid, active;
};
typedef float StageTile[8][kStageD];

/* Step prologue of one lane: state load, apply_action (solo.py:224-259), history push (solo.py:262).
 * wslot = index of this lane's warp among the env warps of the grid (eight envs per warp). */
template <int NJL, bool RAND = false, bool PUSH = false>
__device__ __forceinline__ void step_load(const StepArgs& args, int wslot, int tid, StageTile& stage, EnvLane<NJL>& L,
                                          const DynArgs* dyn = nullptr) {
  const SimConst& sc = args.sc;
  const DevArrays& d = args.d;
  L.tid = tid;
  L.el = tid >> 2; L.leg = tid & 3;
  const int env = wslot * 8 + L.el;
  L.valid = env < args.n;
  L.e = L.valid ? env : args.n - 1;
  L.gid = args.env_id_offset + L.e;
  const int e = L.e, leg = L.leg;
  load_base(d.base, e, L.st, L.goal, L.potential);
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    L.ln.q[k] = d.q[((size_t)k * d.cap + e) * 4 + leg];
    L.ln.qd[k] = d.qd[((size_t)k * d.cap + e) * 4 + leg];
  }
  L.cforce = d.cforce[e * 4 + leg];
  L.bk = d.book[e];
  L.active = L.valid && (args.mode != MODE_SETTLE || L.bk.settle_left > 0);
  if (RAND) {
    /* the settle steps of a reset run with the nominal dynamics, so that a cached reset stays exact */
    if (args.mode == MODE_SETTLE || (PUSH && dyn->envp == nullptr)) { L.dyn.mu = sc.mu; L.dyn.sm = 1.f; L.dyn.st = 1.f; }
    else { const float4 p = dyn->envp[e]; L.dyn.mu = p.x; L.dyn.sm = p.y; L.dyn.st = p.z; }
  }
#pragma unroll
  for (int k = 0; k < NJL; k++) { L.tau[k] = 0.f; L.act[k] = 0.f; }
  if (args.mode == MODE_STEP) {                     /* apply_action (solo.py:224-259) */
    /* the warp's 8 x A action words arrive as whole lines through the (still unused) observation stage:
     * the actions may live in host-mapped memory (solo_step_host), where scattered 4-byte reads would each
     * be a PCIe round trip */
    const int e0w = wslot * 8;
    const bool tile_ok = (e0w + 8 <= args.n);       /* warp-uniform; ragged / idle warps read directly */
    const float* a = args.in + (size_t)e * args.A;
    if (tile_ok) {
      float* tile = &stage[0][0];
      const float* src = args.in + (size_t)e0w * args.A;
      for (int j = tid; j < 8 * args.A; j += 32) tile[j] = src[j];
      __syncwarp();
      a = tile + L.el * args.A;
    }
    float kp = sc.kp, kd = sc.kd;
    if (sc.control == 2) { kp = a[4 * NJL]; kd = a[4 * NJL + 1]; }
#pragma unroll
    for (int k = 0; k < NJL; k++) {
      L.act[k] = a[leg * NJL + k];
      L.tau[k] = action_to_torque(sc, L.act[k], L.ln.q[k], L.ln.qd[k], kp, kd);
      if (RAND) L.tau[k] *= L.dyn.st;
    }
    __syncwarp();                                   /* the stage is reused for the observation rows */
  } else if (args.mode == MODE_SUBSTEP) {
#pragma unroll
    for (int k = 0; k < NJL; k++) L.tau[k] = args.in[(size_t)e * 4 * NJL + leg * NJL + k];
  }
  if (PUSH) {
    /* The env's push for this launch, held in its row of the warp's stage (idle until step_finish writes the
     * observation rows) rather than in registers.  Pushes act in the control steps only: the settle steps
     * (cached resets stay exact) and the substep hook run unpushed.  t = the steps this episode has completed,
     * before step_finish counts this one. */
    if (leg == 0) {
      PushSample ps;
      ps.fx = 0.f; ps.fy = 0.f;
      if (args.mode == MODE_STEP) ps = sample_push(dyn->push, args.seed_lo, args.seed_hi, L.gid, L.bk.episode, L.bk.timestep);
      stage[L.el][0] = ps.fx; stage[L.el][1] = ps.fy; stage[L.el][2] = 0.f;
    }
    __syncwarp();
  }
  if (args.mode != MODE_SUBSTEP && L.active && sc.H > 0) {   /* simulator_step: history push (solo.py:262) */
    RowPieces<NJL> cur;
    load_pieces<NJL>(cur_row(d, args.D0, e), leg, sc.task, cur);
    push_history<NJL>(d, sc, args.D0, e, leg, cur);
  }
  L.bk.nc_sum = 0; L.bk.sweep_feet = 0;
}

/* Step epilogue of one lane: pointgoal bookkeeping (solo.py:267-272), observation, reward / termination
 * (baseEnv.py:47-68), episode record, worker auto-reset (agents/ppo/envs.py:38-40), state store. */
template <int NJL, bool RAND = false>
__device__ __forceinline__ void step_finish(const StepArgs& args, int wslot, StageTile& stage, EnvLane<NJL>& L,
                                            const DynArgs* dyn = nullptr) {
  const SimConst& sc = args.sc;
  const DevArrays& d = args.d;
  const int e = L.e, leg = L.leg, el = L.el, tid = L.tid, D0 = args.D0;
  const bool valid = L.valid;
  BaseState& st = L.st;
  Lane<NJL>& ln = L.ln;
  EnvBook& bk = L.bk;
  float* goal = L.goal;
  float& potential = L.potential;
  float& cforce = L.cforce;
  float progress = 0.f;
  if (args.mode != MODE_SUBSTEP && sc.task == 2) {  /* pointgoal bookkeeping (solo.py:267-272) */
    const float oldp = potential;
    potential = calc_potential(st, goal);
    progress = oldp - potential;
    if (potential < sc.goal_reach) {
      bk.goals += 1;
      uint32_t w[4];
      env_rng(args.seed_lo, args.seed_hi, L.gid, bk, w);
      sample_goal(w, d.mut[kMutGoalRadius], goal);
    }
  }

  if (args.mode == MODE_STEP) {
    bk.timestep += 1;                               /* baseEnv.py:47 */
    float sq = 0.f, sa = 0.f;
#pragma unroll
    for (int k = 0; k < NJL; k++) {
      sq += (sc.task == 0) ? fabsf(ln.q[k]) : ln.q[k] * ln.q[k];
      sa += L.act[k] * L.act[k];
    }
    /* non-finite-state guard: 0 * x is NaN exactly when x is NaN or Inf */
    float chk = st.p[0] + st.p[1] + st.p[2] + st.q[0] + st.q[1] + st.q[2] + st.q[3] + st.v[0] + st.v[1] + st.v[2] +
                st.w[0] + st.w[1] + st.w[2] + sa;
#pragma unroll
    for (int k = 0; k < NJL; k++) chk += ln.q[k] + ln.qd[k];
    sq = sum4(sq); sa = sum4(sa); chk = sum4(chk * 0.f);
    const bool bad_state = !(chk == 0.f);
    StepOutcome o = step_outcome(sc, st, 4 * NJL, sq, sa, progress, bk, bad_state);
    if (valid && leg == 0) {
      args.reward[e] = o.reward;
      args.done[e] = o.done ? 1.0f : 0.0f;
    }
    if (o.done) {
      if (valid && leg == 0) {                      /* info dict (baseEnv.py:63-66) */
        SoloEpisodeStats s;
        s.episode_reward = o.reward; s.episode_return = bk.reward_sum;
        s.episode_length = bk.timestep; s.success = o.success; s.timeout = o.timeout;
        s.goals_reached = bk.goals_env;
        s.dr_stand = bk.dr[0]; s.dr_joint_pose = bk.dr[1]; s.dr_torque = bk.dr[2];
        s.dr_balance = bk.dr[3]; s.dr_progress = bk.dr[4];
        s.nan = bad_state ? 1 : 0;
        d.stats[e] = s;
      }
      /* worker auto-reset (agents/ppo/envs.py:38-40): the terminal observation is never returned
       * (baseEnv.py:54), the reset one is.  Simulate mode: the settle launches that follow rewrite the row. */
      if (valid)
        begin_reset<NJL>(d, sc, D0, e, leg, L.gid, args.seed_lo, args.seed_hi, d.mut[kMutGoalRadius],
                         args.reset_simulate, -1, st, ln, cforce, goal, potential, bk, RAND ? dyn : nullptr);
    }
    /* ONE derivation of get_current_state per step, after the reset decision: it is the observation's first
     * block, and the row the next step pushes into the history */
    RowPieces<NJL> cur;
    make_pieces<NJL>(sc, st, ln, cforce, goal, cur);
    const bool staged = args.D <= kStageD;           /* uniform */
    float* const row = staged ? &stage[el][0] : args.obs + (size_t)e * args.D;
    if (valid) {
      write_obs_row<NJL>(d, sc, D0, e, leg, cur, row);
      store_pieces<NJL>(cur_row(d, D0, e), leg, sc.task, cur);
    }
    if (staged) {                                     /* the warp's 8 x D floats leave as whole lines */
      __syncwarp();
      const int e0 = wslot * 8;
      const int nv = min(8, args.n - e0);
      if ((args.D & 3) == 0) {
        const int d4 = args.D >> 2;
        for (int r = 0; r < nv; r++) {
          float4* dst = reinterpret_cast<float4*>(args.obs + (size_t)(e0 + r) * args.D);
          const float4* src = reinterpret_cast<const float4*>(&stage[r][0]);
          for (int j = tid; j < d4; j += 32) dst[j] = src[j];
        }
      } else {
        for (int r = 0; r < nv; r++)
          for (int j = tid; j < args.D; j += 32) args.obs[(size_t)(e0 + r) * args.D + j] = stage[r][j];
      }
    }
  } else if (L.active) {                              /* settle step of a simulated reset, or the substep hook */
    RowPieces<NJL> cur;
    make_pieces<NJL>(sc, st, ln, cforce, goal, cur);
    store_pieces<NJL>(cur_row(d, D0, e), leg, sc.task, cur);
    if (args.mode == MODE_SETTLE) {
      bk.settle_left -= 1;
      if (bk.settle_left == 0 && args.obs != nullptr) write_obs<NJL>(d, sc, D0, args.D, e, leg, cur, args.obs);
    }
  }

  if (L.active) {
    if (leg == 0) { store_base(d.base, e, st, goal, potential); d.book[e] = bk; }
#pragma unroll
    for (int k = 0; k < NJL; k++) {
      d.q[((size_t)k * d.cap + e) * 4 + leg] = ln.q[k];
      d.qd[((size_t)k * d.cap + e) * 4 + leg] = ln.qd[k];
    }
    d.cforce[e * 4 + leg] = cforce;
  }
}

/* Builds of the step kernel, chosen per handle from the batch size (choose_variant):
 *   latency    WPB = 4 warps per block, 254 registers (8 warps per SM): shortest per-warp dependent
 *              chain; best while the batch is a single resident wave (<= 8k envs);
 *   throughput WPB = 8, capped at 128 registers (16 warps per SM, 320 B of spills): +30 % once
 *              several waves are resident.
 * WPB > 1 with a block barrier per substep keeps the warps of an SM on the same instruction lines:
 * the substep body is ~54 KB of straight-line SASS against a 32 KB L1.5 instruction cache, so every
 * substep streams its code from L2, and warps that drift apart each pay for the fetch
 * (profiles/r1_sweep_wpb.txt: +6 % at 4096 envs, +38 % at 64k envs against one warp per block).
 * Eight envs per warp always: narrower warps were measured slower at every size
 * (profiles/r1_sweep_epw.txt).
 * RAND (SoloSimParams.randomize): every lane holds its env's dynamics (EnvDyn) in registers for the launch; the
 * builds without it are the code of a handle that has never heard of randomisation.
 * PUSH (SoloSimParams.push_interval > 0), instantiated with RAND only: step_load puts the env's push for the
 * launch into the warp's stage, and every substep reads it from there as the external force on the base; a handle
 * with pushes and without randomisation passes envp == nullptr and runs the nominal dynamics. */
template <int NJL, int MINB, int WPB, bool LIMITS, bool BODY = false, bool RAND = false, bool PUSH = false>
__global__ void __launch_bounds__(kBlockThreads * WPB, MINB) step_kernel(const __grid_constant__ StepArgs args,
                                                                         const __grid_constant__ DynArgs dyn) {
  __shared__ Smem sm;
  __shared__ __align__(16) StageTile stage[WPB];
  extern __shared__ __align__(16) float body_smem[];   /* BODY: the row records of the block's 8 x WPB envs */
  if (blockIdx.x * (8 * WPB) >= args.n) return;   /* padding blocks of an experiment grid (SOLO_GRID_MIN) */
  KSTAMP(0);
  const int tid = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;      /* warp in block */
  const SimConst& sc = args.sc;
  {
    const float* src = reinterpret_cast<const float*>(&args.mc.leg[0]);
    float* dst = reinterpret_cast<float*>(&sm.leg[0]);
    for (int i = threadIdx.x; i < (int)(sizeof(LegConst) * 4 / sizeof(float)); i += kBlockThreads * WPB) dst[i] = src[i];
  }
  __syncthreads();
  const int nsub = (args.mode == MODE_SUBSTEP) ? 1 : sc.frame_skip;
  const int wslot = blockIdx.x * WPB + wib;
  EnvLane<NJL> L;
  step_load<NJL, RAND, PUSH>(args, wslot, tid, stage[wib], L, &dyn);
  KSTAMP(1);
  for (int s = 0; s < nsub; s++) {                  /* frame_skip x p.stepSimulation() (solo.py:264-265) */
    if (WPB > 1) __syncthreads();   /* keep the warps of a block on the same instruction lines */
    const bool torque_on = (s == 0) || sc.torque_hold; /* SURVEY F4 */
    float tau_s[NJL];
#pragma unroll
    for (int k = 0; k < NJL; k++) tau_s[k] = torque_on ? L.tau[k] : 0.f;
    group_substep<NJL, LIMITS, BODY>(sm.leg[L.leg], args.mc, sc, L.leg, L.st, L.ln, tau_s, L.cforce, L.bk.nc_sum,
                                     L.bk.sweep_feet, s, PUSH ? &stage[wib][L.el][0] : nullptr,
                                     BODY ? body_smem + (size_t)(wib * 8 + L.el) * kBodyEnvStride : nullptr,
                                     RAND ? &L.dyn : nullptr);
  }
  KSTAMP(2);
  if (PUSH) __syncwarp();                           /* every lane has read the push before the stage is reused */
  step_finish<NJL, RAND>(args, wslot, stage[wib], L, &dyn);
  KSTAMP(3);
}

}  // namespace solo
#include "solo_wide.cuh"
namespace solo {

/* The wide build (solo_wide.cuh): warpgroup 0 runs the env step of 32 envs exactly like a 4-warp block of the
 * narrow builds, with the substep replaced by its phase-split form; warpgroups 1..3 serve it. */
template <int NJL, bool LIMITS>
__global__ void __launch_bounds__(kWThreads, 1) wide_step_kernel(const __grid_constant__ StepArgs args) {
  extern __shared__ __align__(16) unsigned char wide_raw[];
  WideShared& S = *reinterpret_cast<WideShared*>(wide_raw);
  __shared__ Smem sm;
  __shared__ __align__(16) StageTile stage[4];
  if (blockIdx.x * kWEnvs >= args.n) return;      /* padding blocks of an experiment grid (SOLO_GRID_MIN) */
  const SimConst& sc = args.sc;
  {
    const float* src = reinterpret_cast<const float*>(&args.mc.leg[0]);
    float* dst = reinterpret_cast<float*>(&sm.leg[0]);
    for (int i = threadIdx.x; i < (int)(sizeof(LegConst) * 4 / sizeof(float)); i += kWThreads) dst[i] = src[i];
  }
  __syncthreads();
  const int nsub = (args.mode == MODE_SUBSTEP) ? 1 : sc.frame_skip;
  const int wg = threadIdx.x >> 7, t4 = threadIdx.x & (kWE4 - 1);
  if (wg == 0) {
    wide_regs_grow();
    const int tid = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int wslot = blockIdx.x * 4 + wib;
    EnvLane<NJL> L;
    step_load<NJL>(args, wslot, tid, stage[wib], L);
    for (int s = 0; s < nsub; s++) {                /* frame_skip x p.stepSimulation() (solo.py:264-265) */
      const bool torque_on = (s == 0) || sc.torque_hold; /* SURVEY F4 */
      float tau_s[NJL];
#pragma unroll
      for (int k = 0; k < NJL; k++) tau_s[k] = torque_on ? L.tau[k] : 0.f;
      wide_leg_substep<NJL, LIMITS>(sm.leg[L.leg], args.mc, sc, S, t4, L.leg, L.st, L.ln, tau_s, L.cforce, L.bk.nc_sum,
                            L.bk.sweep_feet);
    }
    step_finish<NJL>(args, wslot, stage[wib], L);
  } else {
    wide_regs_shrink();
    for (int s = 0; s < nsub; s++) wide_helper_substep<NJL>(sm.leg[t4 & 3], sc, S, t4, wg - 1);
  }
}

/* n_ticks simulator ticks under the joint-level PD + feed-forward actuator (SURVEY §8f n2): the
 * torque is recomputed from the current joint state before every tick, as the external simulator's
 * SendCommand does once per control tick (baseControlEnv.py:256-270).  cmd [n][5][nj] = q_des, v_des,
 * P, D, tau_ff.  No env bookkeeping: the gait-env shell on top owns reward / termination. */
template <int NJL, bool BODY>
__global__ void __launch_bounds__(kBlockThreads) actuator_kernel(const __grid_constant__ StepArgs args, int n_ticks) {
  __shared__ Smem sm;
  extern __shared__ __align__(16) float body_smem[];   /* BODY: the row records of the warp's eight envs */
  const int tid = threadIdx.x;
  const SimConst& sc = args.sc;
  {
    const float* src = reinterpret_cast<const float*>(&args.mc.leg[0]);
    float* dst = reinterpret_cast<float*>(&sm.leg[0]);
    for (int i = tid; i < (int)(sizeof(LegConst) * 4 / sizeof(float)); i += kBlockThreads) dst[i] = src[i];
  }
  __syncthreads();
  const DevArrays& d = args.d;
  const int el = tid >> 2, leg = tid & 3;
  const int env = blockIdx.x * 8 + el;
  const bool valid = env < args.n;
  const int e = valid ? env : args.n - 1;
  BaseState st;
  float goal[2], potential;
  load_base(d.base, e, st, goal, potential);
  Lane<NJL> ln;
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    ln.q[k] = d.q[((size_t)k * d.cap + e) * 4 + leg];
    ln.qd[k] = d.qd[((size_t)k * d.cap + e) * 4 + leg];
  }
  float cforce = d.cforce[e * 4 + leg];
  const int nj = 4 * NJL;
  const float* c = args.in + (size_t)e * 5 * nj + leg * NJL;
  float qdes[NJL], vdes[NJL], P[NJL], D[NJL], tff[NJL];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    qdes[k] = c[k]; vdes[k] = c[nj + k]; P[k] = c[2 * nj + k]; D[k] = c[3 * nj + k]; tff[k] = c[4 * nj + k];
  }
  int nc_sum = 0, sweep_feet = 0;
  const float4 fx = reinterpret_cast<const float4*>(d.fext)[e];
  const float fext[3] = {fx.x, fx.y, fx.z};
  for (int s = 0; s < n_ticks; s++) {
    float tau[NJL];
#pragma unroll
    for (int k = 0; k < NJL; k++) tau[k] = actuator_torque(sc, ln.q[k], ln.qd[k], qdes[k], vdes[k], P[k], D[k], tff[k]);
    float* const rows = BODY ? body_smem + (size_t)el * kBodyEnvStride : nullptr;
    if (sc.joint_limits) group_substep<NJL, true, BODY>(sm.leg[leg], args.mc, sc, leg, st, ln, tau, cforce, nc_sum, sweep_feet, 0, fext, rows);
    else group_substep<NJL, false, BODY>(sm.leg[leg], args.mc, sc, leg, st, ln, tau, cforce, nc_sum, sweep_feet, 0, fext, rows);
  }
  if (valid) {
    if (leg == 0) store_base(d.base, e, st, goal, potential);
#pragma unroll
    for (int k = 0; k < NJL; k++) {
      d.q[((size_t)k * d.cap + e) * 4 + leg] = ln.q[k];
      d.qd[((size_t)k * d.cap + e) * 4 + leg] = ln.qd[k];
    }
    d.cforce[e * 4 + leg] = cforce;
  }
}

/* world-frame centres of the four foot collision spheres, out [n][4][3] */
template <int NJL>
__global__ void feet_kernel(DevArrays d, ModelConst mc, int n, float* out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t >> 2, leg = t & 3;
  if (e >= n) return;
  BaseState st;
  float goal[2], potential;
  load_base(d.base, e, st, goal, potential);
  float q[NJL], fb[3], fw[3], R[9];
#pragma unroll
  for (int k = 0; k < NJL; k++) q[k] = d.q[((size_t)k * d.cap + e) * 4 + leg];
  leg_foot_center<NJL>(mc.leg[leg], q, fb);
  quat_to_rot(st.q, R);
  mat3_mulv(R, fb, fw);
  float* o = out + ((size_t)e * 4 + leg) * 3;
  o[0] = st.p[0] + fw[0]; o[1] = st.p[1] + fw[1]; o[2] = st.p[2] + fw[2];
}

/* VecEnvWrapper.reset (agents/ppo/envs.py:97-100): masked begin_reset, four lanes per env */
template <int NJL>
__global__ void reset_kernel(const __grid_constant__ ResetArgs args) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t >> 2, leg = t & 3;
  if (e >= args.n) return;
  if (args.mask != nullptr && args.mask[e] == 0) return;
  const DevArrays& d = args.d;
  BaseState st;
  float goal[2], potential;
  load_base(d.base, e, st, goal, potential);
  Lane<NJL> ln;
  float cforce;
  EnvBook bk = d.book[e];
  begin_reset<NJL>(d, args.sc, args.D0, e, leg, args.env_id_offset + e, args.seed_lo, args.seed_hi,
                   d.mut[kMutGoalRadius], args.reset_simulate, args.force_settle, st, ln, cforce, goal, potential, bk,
                   &args.dyn);
  if (!args.reset_simulate) {
    RowPieces<NJL> cur;
    make_pieces<NJL>(args.sc, st, ln, cforce, goal, cur);
    store_pieces<NJL>(cur_row(d, args.D0, e), leg, args.sc.task, cur);
    if (args.obs != nullptr) write_obs<NJL>(d, args.sc, args.D0, args.D, e, leg, cur, args.obs);
  }
  if (leg == 0) { store_base(d.base, e, st, goal, potential); d.book[e] = bk; }
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    d.q[((size_t)k * d.cap + e) * 4 + leg] = ln.q[k];
    d.qd[((size_t)k * d.cap + e) * 4 + leg] = ln.qd[k];
  }
  d.cforce[e * 4 + leg] = cforce;
}

/* get_observation (agents/ppo/envs.py:102-105) */
template <int NJL>
__global__ void obs_kernel(DevArrays d, SimConst sc, int n, int D0, int D, float* obs) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t >> 2, leg = t & 3;
  if (e >= n) return;
  BaseState st;
  float goal[2], potential;
  load_base(d.base, e, st, goal, potential);
  Lane<NJL> ln;
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    ln.q[k] = d.q[((size_t)k * d.cap + e) * 4 + leg];
    ln.qd[k] = d.qd[((size_t)k * d.cap + e) * 4 + leg];
  }
  RowPieces<NJL> cur;
  make_pieces<NJL>(sc, st, ln, d.cforce[e * 4 + leg], goal, cur);
  write_obs<NJL>(d, sc, D0, D, e, leg, cur, obs);
}

/* state [n][13+2nj] <-> SoA */
template <int NJL>
__global__ void get_state_kernel(DevArrays d, int n, float* state) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t >> 2, leg = t & 3;
  if (e >= n) return;
  const int nj = 4 * NJL, W = 13 + 2 * nj;
  float* s = state + (size_t)e * W;
  if (leg == 0) {
    for (int i = 0; i < 13; i++) s[i] = d.base[(size_t)e * kBaseStride + i];
  }
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    s[13 + leg * NJL + k] = d.q[((size_t)k * d.cap + e) * 4 + leg];
    s[13 + nj + leg * NJL + k] = d.qd[((size_t)k * d.cap + e) * 4 + leg];
  }
}
template <int NJL>
__global__ void set_state_kernel(DevArrays d, SimConst sc, int n, int D0, const float* state) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t >> 2, leg = t & 3;
  if (e >= n) return;
  const int nj = 4 * NJL, W = 13 + 2 * nj;
  const float* s = state + (size_t)e * W;
  BaseState st;
  float goal[2], potential;
  load_base(d.base, e, st, goal, potential);
  for (int i = 0; i < 3; i++) { st.p[i] = s[i]; st.v[i] = s[7 + i]; st.w[i] = s[10 + i]; }
  for (int i = 0; i < 4; i++) st.q[i] = s[3 + i];
  normalize_quat(st.q);
  Lane<NJL> ln;
#pragma unroll
  for (int k = 0; k < NJL; k++) { ln.q[k] = s[13 + leg * NJL + k]; ln.qd[k] = s[13 + nj + leg * NJL + k]; }
  const float cforce = -1.0f;
  RowPieces<NJL> cur;
  make_pieces<NJL>(sc, st, ln, cforce, goal, cur);
  for (int h = 0; h < sc.H; h++) store_pieces<NJL>(hist_row(d, D0, h, e), leg, sc.task, cur);
  store_pieces<NJL>(cur_row(d, D0, e), leg, sc.task, cur);
  potential = (sc.task == 2) ? calc_potential(st, goal) : 0.f;
  if (leg == 0) {
    store_base(d.base, e, st, goal, potential);
    EnvBook bk = d.book[e];
    book_clear_episode(bk);
    bk.settle_left = 0;
    d.book[e] = bk;
  }
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    d.q[((size_t)k * d.cap + e) * 4 + leg] = ln.q[k];
    d.qd[((size_t)k * d.cap + e) * 4 + leg] = ln.qd[k];
  }
  d.cforce[e * 4 + leg] = cforce;
}

__global__ void set_goal_kernel(DevArrays d, int n, int njl, int D0, int task, const float* goals) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float* b = d.base + (size_t)e * kBaseStride;
  b[kBaseGoal] = goals[2 * e]; b[kBaseGoal + 1] = goals[2 * e + 1];
  float dx = b[0] - goals[2 * e], dy = b[1] - goals[2 * e + 1];
  b[kBasePot] = sqrtf(dx * dx + dy * dy);
  if (task == 2) {                                   /* the goal is part of the pointgoal state row (solo.py:337-340) */
    float* row = cur_row(d, D0, e);
    row[idx_pg(njl) + 2] = goals[2 * e] / 2.0f; row[idx_pg(njl) + 3] = goals[2 * e + 1] / 2.0f;
  }
}

__global__ void set_fext_kernel(DevArrays d, int n, const float* f) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  reinterpret_cast<float4*>(d.fext)[e] = make_float4(f[3 * e], f[3 * e + 1], f[3 * e + 2], 0.f);
}

/* parity hook: overwrite the per-foot contact record (normal force, < 0 = no contact point) */
__global__ void set_contacts_kernel(DevArrays d, SimConst sc, int n, int njl, int D0, const float* force) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * 4) return;
  d.cforce[t] = force[t];
  cur_row(d, D0, t >> 2)[idx_flag(njl, t & 3)] = contact_flag(sc, force[t]);
}

__global__ void work_kernel(DevArrays d, int n, int* out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  out[2 * e] = d.book[e].nc_sum;
  out[2 * e + 1] = d.book[e].sweep_feet;
}

__global__ void contacts_kernel(DevArrays d, SimConst sc, int n, float* out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * 4) return;
  const float f = d.cforce[t];
  out[t * 3 + 0] = contact_flag(sc, f);
  out[t * 3 + 1] = f >= 0.f ? 1.f : 0.f;
  out[t * 3 + 2] = f >= 0.f ? f : 0.f;
}

/* contact-free forward dynamics on caller-provided states (test hook) */
template <int NJL>
__global__ void fd_kernel(ModelConst mc, SimConst sc, int n, const float* state, const float* tau_in, float* out,
                          const float4* envp) {
  __shared__ LegConst sleg[4];
  {
    const float* src = reinterpret_cast<const float*>(&mc.leg[0]);
    float* dst = reinterpret_cast<float*>(&sleg[0]);
    for (int i = threadIdx.x; i < (int)(sizeof(LegConst) * 4 / sizeof(float)); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int env = t >> 2, leg = t & 3;
  const int e = env < n ? env : n - 1;
  const int nj = 4 * NJL, W = 13 + 2 * nj;
  const float* s = state + (size_t)e * W;
  BaseState st;
  for (int i = 0; i < 3; i++) { st.p[i] = s[i]; st.v[i] = s[7 + i]; st.w[i] = s[10 + i]; }
  for (int i = 0; i < 4; i++) st.q[i] = s[3 + i];
  normalize_quat(st.q);
  Lane<NJL> ln;
  float tau[NJL];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    ln.q[k] = s[13 + leg * NJL + k]; ln.qd[k] = s[13 + nj + leg * NJL + k];
    tau[k] = tau_in[(size_t)e * nj + leg * NJL + k];
  }
  BaseWork bw;
  base_prepare(st, bw);
  Sym6 IA;
  float pA[6], a0[6], qdd[NJL], aw[3], al[3];
  leg_inward<NJL>(sleg[leg], sc, bw, ln, tau, IA, pA);
  sum4_sym6(IA);
#pragma unroll
  for (int i = 0; i < 6; i++) pA[i] = sum4(pA[i]);
  EnvDyn dyn;
  if (envp != nullptr) { const float4 p = envp[e]; dyn.mu = p.x; dyn.sm = p.y; dyn.st = p.z; }
  base_solve(mc, sc, bw, IA, pA, a0, envp != nullptr ? &dyn : nullptr);
  leg_outward<NJL>(ln, a0, qdd);
  base_world_acc(sc, bw, a0, aw, al);
  if (env < n) {
    float* o = out + (size_t)e * (6 + nj);
    if (leg == 0) { for (int i = 0; i < 3; i++) { o[i] = aw[i]; o[3 + i] = al[i]; } }
#pragma unroll
    for (int k = 0; k < NJL; k++) o[6 + leg * NJL + k] = qdd[k];
  }
}

template <int NJL>
__global__ void torque_kernel(DevArrays d, SimConst sc, int n, int A, const float* actions, float* tau,
                              const float4* envp) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t >> 2, leg = t & 3;
  if (e >= n) return;
  const float* a = actions + (size_t)e * A;
  float kp = sc.kp, kd = sc.kd;
  if (sc.control == 2) { kp = a[4 * NJL]; kd = a[4 * NJL + 1]; }
  const float st = envp != nullptr ? envp[e].z : 1.f;
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    float q = d.q[((size_t)k * d.cap + e) * 4 + leg], qd = d.qd[((size_t)k * d.cap + e) * 4 + leg];
    float t = action_to_torque(sc, a[leg * NJL + k], q, qd, kp, kd);
    if (envp != nullptr) t *= st;
    tau[(size_t)e * 4 * NJL + leg * NJL + k] = t;
  }
}

/* solo_get_env_params: envp [n] float4 -> out [n][3] */
__global__ void env_params_kernel(const float4* envp, int n, float* out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const float4 p = envp[e];
  out[3 * e] = p.x; out[3 * e + 1] = p.y; out[3 * e + 2] = p.z;
}

/* solo_get_push_force: the push of each env's next control step, from its episode record -> out [n][3] */
__global__ void push_force_kernel(const EnvBook* book, PushParams pp, uint32_t seed_lo, uint32_t seed_hi,
                                  long long env_id_offset, int n, float* out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const EnvBook bk = book[e];
  const PushSample ps = sample_push(pp, seed_lo, seed_hi, env_id_offset + e, bk.episode, bk.timestep);
  out[3 * e] = ps.fx; out[3 * e + 1] = ps.fy; out[3 * e + 2] = 0.f;
}

/* copy env rows 0..K-1 into the reset cache */
template <int NJL>
__global__ void fill_cache_kernel(DevArrays d, int K, int H, int D0) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= K) return;
  for (int i = 0; i < kBaseStride; i++) d.rc_base[t * kBaseStride + i] = d.base[(size_t)t * kBaseStride + i];
  for (int leg = 0; leg < 4; leg++) {
    for (int k = 0; k < NJL; k++) {
      d.rc_q[t * 12 + leg * NJL + k] = d.q[((size_t)k * d.cap + t) * 4 + leg];
      d.rc_qd[t * 12 + leg * NJL + k] = d.qd[((size_t)k * d.cap + t) * 4 + leg];
    }
    d.rc_cforce[t * 4 + leg] = d.cforce[t * 4 + leg];
  }
  for (int h = 0; h < H; h++)
    for (int i = 0; i < D0; i++) d.rc_hist[((size_t)t * H + h) * D0 + i] = d.hist[((size_t)h * d.cap + t) * D0 + i];
}

/* Trainer-side episode logging without a host round trip (agents/ppo/train.py:90-100 reads an info
 * dict per finished env and step): fold the records of envs whose done flag is set into running
 * totals.  acc[0..9] = count, sum episode_reward, sum episode_return, sum length, sum success, the
 * five dr/ sums; acc[10..12] = min return, max return, max length.  Few envs finish per step, so
 * plain atomics are enough. */
__device__ __forceinline__ void atomic_min_double(double* addr, double v) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *a, assumed;
  do {
    assumed = old;
    if (__longlong_as_double((long long)assumed) <= v) break;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
  } while (assumed != old);
}
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(addr);
  unsigned long long old = *a, assumed;
  do {
    assumed = old;
    if (__longlong_as_double((long long)assumed) >= v) break;
    old = atomicCAS(a, assumed, (unsigned long long)__double_as_longlong(v));
  } while (assumed != old);
}
__global__ void episode_accumulate_kernel(const SoloEpisodeStats* __restrict__ stats, const float* __restrict__ done,
                                          int n, double* acc) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n || done[e] <= 0.5f) return;
  const SoloEpisodeStats s = stats[e];
  atomicAdd(acc + 0, 1.0);
  atomicAdd(acc + 1, (double)s.episode_reward);
  atomicAdd(acc + 2, (double)s.episode_return);
  atomicAdd(acc + 3, (double)s.episode_length);
  atomicAdd(acc + 4, (double)s.success);
  atomicAdd(acc + 5, (double)s.dr_stand);
  atomicAdd(acc + 6, (double)s.dr_joint_pose);
  atomicAdd(acc + 7, (double)s.dr_torque);
  atomicAdd(acc + 8, (double)s.dr_balance);
  atomicAdd(acc + 9, (double)s.dr_progress);
  atomic_min_double(acc + 10, (double)s.episode_return);
  atomic_max_double(acc + 11, (double)s.episode_return);
  atomic_max_double(acc + 12, (double)s.episode_length);
}

/* Reverse-scan GAE (agents/ppo/storage.py:35-55), HBM-bound: 20 B per (t, env) = 4 reads + 1 write of fp32.
 * The recurrence A_t = delta_t + gamma lam m_{t+1} A_{t+1} is serial in t, but nothing it READS depends on it:
 * delta_t = r_t + gamma V_{t+1} m_{t+1} - V_t and the factor c_t = gamma lam m_{t+1} are known up front.
 * A block owns kGaeEnvs consecutive envs and kGaeChunks time chunks of L steps.  Thread (c, e)
 *   1. loads ITS chunk's rewards / values / masks -- all kGaeChunks x kGaeEnvs x 3L loads of the block are
 *      independent and in flight together -- and turns them into (c_t, delta_t) in registers;
 *   2. the chunks then run the recurrence one after the other, newest first; on the serial path a step is ONE
 *      fused multiply-add (the round-2 profile of the previous form, profiles/r2_gae_kernel_ncu.txt, showed 40
 *      instructions per step there -- 64-bit address arithmetic and the store -- and 16 warps waiting for them);
 *      the running value is handed to the next chunk through shared memory BEFORE the chunk's results are stored;
 *   3. every thread stores its L returns (coalesced 128-byte rows), overlapping the later chunks' turns.
 * Steps beyond T hold (c, delta) = (1, 0), i.e. leave the running value untouched, so the serial loop carries
 * no predicate.  masks are 0/1, so folding them into c_t is exact and the arithmetic (and its rounding) is that
 * of the serial walk below and of the oracle's storage.py-order loop. */
constexpr int kGaeEnvs = 32;      /* one 128-byte line per [t] row and block */
constexpr int kGaeChunks = 16;
constexpr int kGaeMaxL = 32;      /* time steps per chunk held in registers: T <= 512 takes the chunked path */
template <int L>
__global__ void __launch_bounds__(kGaeEnvs * kGaeChunks)
gae_chunked_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                   const float* __restrict__ masks, float* __restrict__ returns, int T, int N,
                   float gamma, float lam, int use_gae) {
  __shared__ float carry[kGaeEnvs];
  const int e = threadIdx.x & (kGaeEnvs - 1), c = threadIdx.x / kGaeEnvs;
  const int n = blockIdx.x * kGaeEnvs + e;
  const bool valid = n < N;
  const int nn = valid ? n : N - 1;
  /* chunk c covers t in [t0, t1), chunk kGaeChunks-1 is the newest */
  const int t0 = c * L, t1 = min(T, t0 + L);
  const size_t stride = (size_t)N;
  const float* pr = rewards + (size_t)t0 * stride + nn;
  const float* pv = values + (size_t)t0 * stride + nn;
  const float* pm = masks + (size_t)(t0 + 1) * stride + nn;
  float cf[L], dl[L], vv[L + 1];
#pragma unroll
  for (int i = 0; i < L; i++) {         /* the loads: nothing below depends on another thread */
    const bool on = t0 + i < t1;
    dl[i] = on ? pr[(size_t)i * stride] : 0.f;
    cf[i] = on ? pm[(size_t)i * stride] : 0.f;
  }
#pragma unroll
  for (int i = 0; i <= L; i++) vv[i] = (use_gae && t0 + i <= T && t0 < t1) ? pv[(size_t)i * stride] : 0.f;
  if (c == kGaeChunks - 1) carry[e] = use_gae ? 0.f : returns[(size_t)T * stride + nn];
  /* (c_t, delta_t) with the roundings of the reference's tensor expression (every product and sum rounded on
   * its own: storage.py:45-47 / :52-53), no fused multiply-add */
  const float gl = __fmul_rn(gamma, lam);
#pragma unroll
  for (int i = 0; i < L; i++) {
    const bool on = t0 + i < t1;
    const float m = cf[i];
    if (use_gae) {
      dl[i] = on ? __fsub_rn(__fadd_rn(dl[i], __fmul_rn(__fmul_rn(gamma, vv[i + 1]), m)), vv[i]) : 0.f;
      cf[i] = on ? __fmul_rn(gl, m) : 1.f;
    } else {
      cf[i] = on ? __fmul_rn(gamma, m) : 1.f;       /* ret = ret * gamma * m + r */
    }
  }
  for (int turn = kGaeChunks - 1; turn >= 0; turn--) {
    __syncthreads();
    if (turn == c) {
      float acc = carry[e];
#pragma unroll
      for (int i = L - 1; i >= 0; i--) {
        acc = __fadd_rn(__fmul_rn(cf[i], acc), dl[i]);
        dl[i] = acc;
      }
      carry[e] = acc;
    }
  }
  if (valid) {
    float* po = returns + (size_t)t0 * stride + n;
#pragma unroll
    for (int i = 0; i < L; i++)
      if (t0 + i < t1) po[(size_t)i * stride] = __fadd_rn(dl[i], vv[i]);
  }
}

/* any T: the serial walk (one thread per env) */
__global__ void gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                           const float* __restrict__ masks, float* __restrict__ returns, int T, int N,
                           float gamma, float lam, int use_gae) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  if (use_gae) {          /* same roundings as the chunked kernel (and the reference's tensor expression) */
    float gae = 0.f;
    float v_next = values[(size_t)T * N + n];
    const float gl = __fmul_rn(gamma, lam);
    for (int t = T - 1; t >= 0; t--) {
      const float m = masks[(size_t)(t + 1) * N + n];
      const float v = values[(size_t)t * N + n];
      const float delta = __fsub_rn(__fadd_rn(rewards[(size_t)t * N + n], __fmul_rn(__fmul_rn(gamma, v_next), m)), v);
      gae = __fadd_rn(__fmul_rn(__fmul_rn(gl, m), gae), delta);
      returns[(size_t)t * N + n] = __fadd_rn(gae, v);
      v_next = v;
    }
  } else {
    float ret = returns[(size_t)T * N + n];
    for (int t = T - 1; t >= 0; t--) {
      ret = __fadd_rn(__fmul_rn(__fmul_rn(gamma, masks[(size_t)(t + 1) * N + n]), ret), rewards[(size_t)t * N + n]);
      returns[(size_t)t * N + n] = ret;
    }
  }
}

}  // namespace solo

/* ===================================================================== C-ABI */
using namespace solo;

struct SoloHandle {
  SoloModelTable model;
  SoloSimParams params;
  ModelConst mc;
  SimConst sc;
  int n, njl, nj, A, D0, D, device, K, cap;
  int variant;     /* which build of the step kernel this handle launches (choose_variant) */
  uint64_t seed;
  long long env_id_offset;
  float goal_radius;
  DevArrays d;
  bool was_reset;
  long long launches;
  std::string err;
  /* staging for solo_step_host */
  float *s_act, *s_obs, *s_rew, *s_done;
  int host_zero_copy;   /* SOLO_HOST_ZERO_COPY != 0 */
  /* randomised dynamics: per-env (mu, base mass scale, motor strength, 0), nominal until a reset draws them */
  int randomize;
  DynArgs dyn;
  int push;        /* random pushes on (push_interval > 0): the step launches the PUSH builds */
};

static thread_local std::string g_err;

static int fail(SoloHandle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  g_err = msg;
  return code;
}
#define CUDA_TRY(h, call)                                                                   \
  do {                                                                                      \
    cudaError_t _e = (call);                                                                \
    if (_e != cudaSuccess) return fail(h, SOLO_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e)); \
  } while (0)

static StepArgs make_step_args(SoloHandle* h, int mode, int n, const float* in, float* obs, float* rew, float* done) {
  StepArgs a;
  a.d = h->d; a.sc = h->sc; a.mc = h->mc; a.n = n; a.mode = mode;
  a.D0 = h->D0; a.D = h->D; a.A = h->A;
  a.in = in; a.obs = obs; a.reward = rew; a.done = done;
  a.seed_lo = (uint32_t)(h->seed & 0xffffffffu); a.seed_hi = (uint32_t)(h->seed >> 32);
  a.env_id_offset = h->env_id_offset;
  a.reset_simulate = (h->params.reset_mode == SOLO_RESET_SIMULATE);
  a.force_settle = -1;
  return a;
}
static int grid_min() {
  static int v = -1;
  if (v < 0) { const char* ev = getenv("SOLO_GRID_MIN"); v = ev ? atoi(ev) : 0; }
  return v;
}
/* the DynArgs of a launch: envp only on a randomised handle (a handle with pushes alone runs the nominal
 * dynamics, and its resets draw nothing) */
static DynArgs dyn_args(const SoloHandle* h) {
  DynArgs a = h->dyn;
  if (!h->randomize) a.envp = nullptr;
  return a;
}
template <int MINB, int WPB, bool RAND, bool PUSH = false>
static void launch_step_variant(SoloHandle* h, const StepArgs& a, cudaStream_t s) {
  int blocks = (a.n + 8 * WPB - 1) / (8 * WPB);
  if (blocks < grid_min()) blocks = grid_min();
  const bool lim = h->sc.joint_limits != 0;
  const DynArgs dyn = dyn_args(h);
  if (h->njl == 3) {
    if (lim) step_kernel<3, MINB, WPB, true, false, RAND, PUSH><<<blocks, kBlockThreads * WPB, 0, s>>>(a, dyn);
    else step_kernel<3, MINB, WPB, false, false, RAND, PUSH><<<blocks, kBlockThreads * WPB, 0, s>>>(a, dyn);
  } else {
    if (lim) step_kernel<2, MINB, WPB, true, false, RAND, PUSH><<<blocks, kBlockThreads * WPB, 0, s>>>(a, dyn);
    else step_kernel<2, MINB, WPB, false, false, RAND, PUSH><<<blocks, kBlockThreads * WPB, 0, s>>>(a, dyn);
  }
}
/* shape of the throughput build: warps per block and resident blocks per SM (the register cap follows:
 * 65536 / (32 WPB MINB)); overridable for experiments (tools/gpu_ab.py) */
#ifndef SOLO_TP_WPB
#define SOLO_TP_WPB 8
#endif
#ifndef SOLO_TP_MINB
#define SOLO_TP_MINB 2
#endif
/* body_contacts: the latency shape (4 warps per block) plus the row records in dynamic shared memory */
constexpr int kBodyWPB = 4;
constexpr size_t kBodySmemBytes = (size_t)kBodyWPB * 8 * kBodyEnvStride * sizeof(float);
template <bool RAND, bool PUSH = false>
static void launch_step_body(SoloHandle* h, const StepArgs& a, cudaStream_t s) {
  int blocks = (a.n + 8 * kBodyWPB - 1) / (8 * kBodyWPB);
  const bool lim = h->sc.joint_limits != 0;
  const int threads = kBlockThreads * kBodyWPB;
  const DynArgs dyn = dyn_args(h);
  if (h->njl == 3) {
    if (lim) step_kernel<3, 1, kBodyWPB, true, true, RAND, PUSH><<<blocks, threads, kBodySmemBytes, s>>>(a, dyn);
    else step_kernel<3, 1, kBodyWPB, false, true, RAND, PUSH><<<blocks, threads, kBodySmemBytes, s>>>(a, dyn);
  } else {
    if (lim) step_kernel<2, 1, kBodyWPB, true, true, RAND, PUSH><<<blocks, threads, kBodySmemBytes, s>>>(a, dyn);
    else step_kernel<2, 1, kBodyWPB, false, true, RAND, PUSH><<<blocks, threads, kBodySmemBytes, s>>>(a, dyn);
  }
}
/* builds: PUSH only with RAND (a handle with pushes and nominal dynamics passes envp == nullptr) */
static void launch_step(SoloHandle* h, const StepArgs& a, cudaStream_t s) {
  if (h->sc.body_contacts) {
    if (h->push) launch_step_body<true, true>(h, a, s);
    else if (h->randomize) launch_step_body<true>(h, a, s);
    else launch_step_body<false>(h, a, s);
    h->launches++;
    return;
  }
  if (h->variant == VARIANT_WIDE) {
    int blocks = (a.n + kWEnvs - 1) / kWEnvs;
    if (blocks < grid_min()) blocks = grid_min();
    const bool lim = h->sc.joint_limits != 0;
    if (h->njl == 3) {
      if (lim) wide_step_kernel<3, true><<<blocks, kWThreads, sizeof(WideShared), s>>>(a);
      else wide_step_kernel<3, false><<<blocks, kWThreads, sizeof(WideShared), s>>>(a);
    } else {
      if (lim) wide_step_kernel<2, true><<<blocks, kWThreads, sizeof(WideShared), s>>>(a);
      else wide_step_kernel<2, false><<<blocks, kWThreads, sizeof(WideShared), s>>>(a);
    }
  } else if (h->variant == VARIANT_THROUGHPUT) {
    if (h->push) launch_step_variant<SOLO_TP_MINB, SOLO_TP_WPB, true, true>(h, a, s);
    else if (h->randomize) launch_step_variant<SOLO_TP_MINB, SOLO_TP_WPB, true>(h, a, s);
    else launch_step_variant<SOLO_TP_MINB, SOLO_TP_WPB, false>(h, a, s);
  } else {
    if (h->push) launch_step_variant<1, 4, true, true>(h, a, s);
    else if (h->randomize) launch_step_variant<1, 4, true>(h, a, s);
    else launch_step_variant<1, 4, false>(h, a, s);
  }
  h->launches++;
}
/* latency build up to 8192 envs (one resident wave of 8 warps per SM), throughput build beyond;
 * SOLO_STEP_VARIANT=latency|throughput overrides.  Results are bit-reproducible within a build
 * (and therefore across shardings that stay within one); the two builds differ in the last bits
 * because the compiler contracts and schedules the arithmetic differently. */
static int choose_variant(int n) {
  const char* ev = getenv("SOLO_STEP_VARIANT");
  if (ev && ev[0] == 'l') return VARIANT_LATENCY;
  if (ev && ev[0] == 't') return VARIANT_THROUGHPUT;
  if (ev && ev[0] == 'w') return VARIANT_WIDE;
  return n > 8192 ? VARIANT_THROUGHPUT : VARIANT_LATENCY;
}
static ResetArgs make_reset_args(SoloHandle* h, int n, const uint8_t* mask, float* obs) {
  ResetArgs a;
  a.d = h->d; a.sc = h->sc; a.n = n; a.njl = h->njl; a.D0 = h->D0; a.D = h->D;
  a.mask = mask; a.obs = obs;
  a.seed_lo = (uint32_t)(h->seed & 0xffffffffu); a.seed_hi = (uint32_t)(h->seed >> 32);
  a.env_id_offset = h->env_id_offset;
  a.reset_simulate = (h->params.reset_mode == SOLO_RESET_SIMULATE);
  a.force_settle = -1;
  a.dyn = dyn_args(h);
  return a;
}
static void launch_reset(SoloHandle* h, const ResetArgs& a, cudaStream_t s) {
  const int threads = 128, blocks = (a.n * 4 + threads - 1) / threads;
  if (h->njl == 3) reset_kernel<3><<<blocks, threads, 0, s>>>(a);
  else reset_kernel<2><<<blocks, threads, 0, s>>>(a);
  h->launches++;
}
/* the settle loop of SoloBaseEnv.reset (baseEnv.py:79-80), simulate mode: the longest settle
 * count bounds the number of launches; envs that are done settling idle */
static void launch_settle(SoloHandle* h, int n, float* obs, cudaStream_t s) {
  const int kmax = h->params.settle_max - 1;
  for (int i = 0; i < kmax; i++) {
    StepArgs a = make_step_args(h, MODE_SETTLE, n, nullptr, obs, nullptr, nullptr);
    launch_step(h, a, s);
  }
}

extern "C" {

int solo_default_params(SoloSimParams* p) {
  if (!p) return fail(nullptr, SOLO_E_ARG, "null params");
  fill_default_params(p);
  return SOLO_OK;
}

int solo_dims(const SoloModelTable* m, const SoloSimParams* p, int32_t* nj, int32_t* act_dim,
              int32_t* obs_dim0, int32_t* obs_dim) {
  if (!m || !p) return fail(nullptr, SOLO_E_ARG, "null argument");
  int n = 0;
  for (int i = 0; i < m->num_links; i++) n += (m->jtype[i] == SOLO_JOINT_REVOLUTE);
  const int d0 = 1 + 3 + 6 + 2 * n + 4 + (p->task == SOLO_TASK_POINTGOAL ? 4 : 0);
  if (nj) *nj = n;
  if (act_dim) *act_dim = n + (p->control == SOLO_CONTROL_VPD ? 2 : 0);
  if (obs_dim0) *obs_dim0 = d0;
  if (obs_dim) *obs_dim = d0 * (1 + p->num_history_stack);
  return SOLO_OK;
}

const char* solo_last_error(const SoloHandle* h) { return h ? h->err.c_str() : g_err.c_str(); }

int solo_destroy(SoloHandle* h) {
  if (!h) return SOLO_OK;
  cudaSetDevice(h->device);
  cudaFree(h->d.base); cudaFree(h->d.q); cudaFree(h->d.qd); cudaFree(h->d.cforce); cudaFree(h->d.hist); cudaFree(h->d.currow); cudaFree(h->d.fext);
  cudaFree(h->d.book); cudaFree(h->d.stats);
  cudaFree(h->d.rc_base); cudaFree(h->d.rc_q); cudaFree(h->d.rc_qd); cudaFree(h->d.rc_cforce); cudaFree(h->d.rc_hist);
  cudaFree(const_cast<float*>(h->d.mut));
  cudaFree(h->s_act); cudaFree(h->s_obs); cudaFree(h->s_rew); cudaFree(h->s_done);
  cudaFree(h->dyn.envp);
  delete h;
  return SOLO_OK;
}

static int allocate_and_prime(SoloHandle* h, const SoloSimParams* params);

int solo_create(const SoloModelTable* model, const SoloSimParams* params, int32_t num_envs, int32_t device,
                uint64_t seed, int64_t env_id_offset, SoloHandle** out) {
  if (!model || !params || !out || num_envs <= 0) return fail(nullptr, SOLO_E_ARG, "bad argument to solo_create");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(nullptr, SOLO_E_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(nullptr, SOLO_E_ARG, "bad device index");
  SoloHandle* h = new SoloHandle();
  h->model = *model; h->params = *params;
  std::string err;
  int rc = build_model_const(*model, h->mc, err);
  if (rc == SOLO_OK) rc = build_sim_const(*params, h->sc, err);
  if (rc == SOLO_OK && params->num_history_stack > 8) { rc = SOLO_E_ARG; err = "num_history_stack > 8"; }
  if (rc == SOLO_OK && params->joint_limits && params->limit_rows_per_leg != 1) {
    rc = SOLO_E_ARG; err = "joint_limits: the kernels solve one limit row per leg (limit_rows_per_leg must be 1)";
  }
  if (rc == SOLO_OK) rc = build_env_ranges(*params, h->dyn.ranges, err);
  h->randomize = params->randomize ? 1 : 0;
  if (rc == SOLO_OK && h->randomize && !params->body_contacts && choose_variant(num_envs) == VARIANT_WIDE) {
    rc = SOLO_E_ARG; err = "randomize: the wide build (SOLO_STEP_VARIANT=wide) has no randomised dynamics";
  }
  if (rc == SOLO_OK) rc = build_push_params(*params, h->dyn.push, err);
  h->push = params->push_interval > 0 ? 1 : 0;
  if (rc == SOLO_OK && h->push && !params->body_contacts && choose_variant(num_envs) == VARIANT_WIDE) {
    rc = SOLO_E_ARG; err = "push: the wide build (SOLO_STEP_VARIANT=wide) has no random pushes";
  }
  if (rc != SOLO_OK) { delete h; return fail(nullptr, rc, err); }
  h->n = num_envs; h->njl = h->mc.njl; h->nj = 4 * h->njl;
  h->A = h->nj + (params->control == SOLO_CONTROL_VPD ? 2 : 0);
  h->D0 = obs_dim0(h->njl, params->task);
  h->D = h->D0 * (1 + params->num_history_stack);
  h->device = device; h->seed = seed; h->env_id_offset = env_id_offset;
  h->goal_radius = (float)params->goal_radius;
  h->was_reset = false; h->launches = 0;
  h->variant = choose_variant(num_envs);
  h->K = params->settle_max - params->settle_min; if (h->K < 1) h->K = 1;
  h->cap = num_envs > h->K ? num_envs : h->K;
  h->s_act = h->s_obs = h->s_rew = h->s_done = nullptr;
  h->dyn.envp = nullptr;
  { const char* ev = getenv("SOLO_HOST_ZERO_COPY"); h->host_zero_copy = !(ev && ev[0] == '0'); }
  memset(&h->d, 0, sizeof(h->d));
  h->d.cap = h->cap;
  rc = allocate_and_prime(h, params);
  if (rc != SOLO_OK) {            /* no leak on a failed create: free whatever was allocated */
    const std::string msg = h->err;
    solo_destroy(h);
    return fail(nullptr, rc, msg);
  }
  *out = h;
  return SOLO_OK;
}

}  // extern "C"

static int allocate_and_prime(SoloHandle* h, const SoloSimParams* params) {
  const int H = params->num_history_stack;
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->variant == VARIANT_WIDE) {     /* 104 KB of exchange arrays: above the 48 KB default */
    const int bytes = (int)sizeof(WideShared);
    CUDA_TRY(h, cudaFuncSetAttribute(wide_step_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(wide_step_kernel<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(wide_step_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(wide_step_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  }
  if (h->sc.body_contacts) {            /* 160 KB of row records: above the 48 KB default */
    const int bytes = (int)kBodySmemBytes;
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<3, 1, kBodyWPB, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<3, 1, kBodyWPB, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<2, 1, kBodyWPB, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<2, 1, kBodyWPB, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<3, 1, kBodyWPB, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<3, 1, kBodyWPB, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<2, 1, kBodyWPB, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<2, 1, kBodyWPB, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<3, 1, kBodyWPB, true, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<3, 1, kBodyWPB, false, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<2, 1, kBodyWPB, true, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    CUDA_TRY(h, cudaFuncSetAttribute(step_kernel<2, 1, kBodyWPB, false, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  }
  const size_t cap = (size_t)h->cap;
  {
    float* mut = nullptr;
    CUDA_TRY(h, cudaMalloc(&mut, kMutCount * sizeof(float)));
    h->d.mut = mut;
    const float init[kMutCount] = {h->goal_radius, 0.f, 0.f, 0.f};
    CUDA_TRY(h, cudaMemcpy(mut, init, sizeof(init), cudaMemcpyHostToDevice));
  }
  CUDA_TRY(h, cudaMalloc(&h->d.base, cap * kBaseStride * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.q, cap * 4 * h->njl * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.qd, cap * 4 * h->njl * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.cforce, cap * 4 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.hist, (cap * (H > 0 ? H : 1)) * h->D0 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.fext, cap * 4 * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.fext, 0, cap * 4 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->dyn.envp, cap * sizeof(float4)));
  CUDA_TRY(h, cudaMalloc(&h->d.currow, cap * h->D0 * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.currow, 0, cap * h->D0 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.book, cap * sizeof(EnvBook)));
  CUDA_TRY(h, cudaMalloc(&h->d.stats, cap * sizeof(SoloEpisodeStats)));
  CUDA_TRY(h, cudaMalloc(&h->d.rc_base, (size_t)h->K * kBaseStride * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.rc_q, (size_t)h->K * 12 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.rc_qd, (size_t)h->K * 12 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.rc_cforce, (size_t)h->K * 4 * sizeof(float)));
  CUDA_TRY(h, cudaMalloc(&h->d.rc_hist, (size_t)h->K * (H > 0 ? H : 1) * h->D0 * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.base, 0, cap * kBaseStride * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.q, 0, cap * 4 * h->njl * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.qd, 0, cap * 4 * h->njl * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.cforce, 0, cap * 4 * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.hist, 0, (cap * (H > 0 ? H : 1)) * h->D0 * sizeof(float)));
  CUDA_TRY(h, cudaMemset(h->d.book, 0, cap * sizeof(EnvBook)));
  CUDA_TRY(h, cudaMemset(h->d.stats, 0, cap * sizeof(SoloEpisodeStats)));

  /* Reset cache: the reset trajectory (fixed pose, zero torque, k control steps) depends only
   * on k, so it is simulated ONCE per k with the very kernel that simulate-mode resets use
   * (same binary code => the cached rows are bit-identical to simulating them), and a
   * reset during stepping becomes a table lookup. */
  {
    cudaStream_t s = 0;
    ResetArgs ra = make_reset_args(h, h->K, nullptr, nullptr);
    ra.reset_simulate = 1; ra.force_settle = 1;
    launch_reset(h, ra, s);
    const int kmax = params->settle_max - 1;
    for (int i = 0; i < kmax; i++) {
      StepArgs a = make_step_args(h, MODE_SETTLE, h->K, nullptr, nullptr, nullptr, nullptr);
      a.reset_simulate = 1;
      launch_step(h, a, s);
    }
    const int fc_blocks = (h->K + 31) / 32;   /* any settle span, not just the default 7 rows */
    if (h->njl == 3) fill_cache_kernel<3><<<fc_blocks, 32, 0, s>>>(h->d, h->K, H, h->D0);
    else fill_cache_kernel<2><<<fc_blocks, 32, 0, s>>>(h->d, h->K, H, h->D0);
    h->launches++;
    /* the cache-generation envs leave no trace: counters, goals and states start from zero */
    CUDA_TRY(h, cudaMemsetAsync(h->d.book, 0, cap * sizeof(EnvBook), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d.base, 0, cap * kBaseStride * sizeof(float), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d.q, 0, cap * 4 * h->njl * sizeof(float), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d.qd, 0, cap * 4 * h->njl * sizeof(float), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d.cforce, 0, cap * 4 * sizeof(float), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d.hist, 0, (cap * (H > 0 ? H : 1)) * h->D0 * sizeof(float), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d.currow, 0, cap * h->D0 * sizeof(float), s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    CUDA_TRY(h, cudaGetLastError());
  }
  {   /* nominal dynamics until the first reset (this also drops what the cache generation drew) */
    const std::vector<float4> nominal(cap, make_float4(h->sc.mu, 1.f, 1.f, 0.f));
    CUDA_TRY(h, cudaMemcpy(h->dyn.envp, nominal.data(), cap * sizeof(float4), cudaMemcpyHostToDevice));
  }
  return SOLO_OK;
}

extern "C" {

int solo_reset(SoloHandle* h, const uint8_t* d_mask, float* d_obs_out, void* stream) {
  if (!h) return fail(nullptr, SOLO_E_ARG, "null handle");
  cudaStream_t s = (cudaStream_t)stream;
  ResetArgs ra = make_reset_args(h, h->n, d_mask, d_obs_out);
  launch_reset(h, ra, s);
  if (ra.reset_simulate) launch_settle(h, h->n, d_obs_out, s);
  if (d_mask == nullptr) h->was_reset = true;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_step(SoloHandle* h, const float* d_actions, float* d_obs, float* d_reward, float* d_done, void* stream) {
  if (!h || !d_actions || !d_obs || !d_reward || !d_done) return fail(h, SOLO_E_ARG, "null argument to solo_step");
  if (!h->was_reset) return fail(h, SOLO_E_STATE, "env.reset() must be called before step"); /* baseEnv.py:43 */
  cudaStream_t s = (cudaStream_t)stream;
  StepArgs a = make_step_args(h, MODE_STEP, h->n, d_actions, d_obs, d_reward, d_done);
  launch_step(h, a, s);
  if (a.reset_simulate) launch_settle(h, h->n, d_obs, s);
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

/* device-visible alias of a pinned (page-locked, UVA-mapped) host buffer, or NULL */
static float* mapped_alias(float* host) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr) return nullptr;
  return static_cast<float*>(at.devicePointer);
}

int solo_step_host(SoloHandle* h, const float* h_actions, float* h_obs, float* h_reward, float* h_done, void* stream) {
  if (!h || !h_actions || !h_obs || !h_reward || !h_done) return fail(h, SOLO_E_ARG, "null argument to solo_step_host");
  if (!h->was_reset) return fail(h, SOLO_E_STATE, "env.reset() must be called before step");
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)h->n;
  if (!h->s_act) {
    CUDA_TRY(h, cudaMalloc(&h->s_act, n * h->A * sizeof(float)));
    CUDA_TRY(h, cudaMalloc(&h->s_obs, n * h->D * sizeof(float)));
    CUDA_TRY(h, cudaMalloc(&h->s_rew, n * sizeof(float)));
    CUDA_TRY(h, cudaMalloc(&h->s_done, n * sizeof(float)));
  }
  /* Pinned output buffers are written by the step kernel itself (whole 128-byte lines over PCIe as the
   * warps finish, overlapping the rest of the launch) instead of by three copies after it; pageable
   * buffers, and the simulate-mode reset whose settle launches rewrite observation rows, take the staged
   * path.  SOLO_HOST_ZERO_COPY=0 forces the staged path. */
  /* queried on every call (measured: no visible cost): a cached answer would go stale if the caller
   * freed a pinned buffer and a pageable one landed on the same address */
  float *z_obs = mapped_alias(h_obs), *z_rew = mapped_alias(h_reward), *z_done = mapped_alias(h_done);
  const bool zero_copy = h->host_zero_copy && z_obs && z_rew && z_done && h->D <= kStageD &&
                         h->params.reset_mode == SOLO_RESET_CACHED;
  /* likewise a pinned action buffer is read by the kernel directly (three 128-byte lines per warp) */
  const float* z_act = zero_copy ? mapped_alias(const_cast<float*>(h_actions)) : nullptr;
  if (!z_act) CUDA_TRY(h, cudaMemcpyAsync(h->s_act, h_actions, n * h->A * sizeof(float), cudaMemcpyHostToDevice, s));
  if (zero_copy) {
    int rc = solo_step(h, z_act ? z_act : h->s_act, z_obs, z_rew, z_done, stream);
    if (rc != SOLO_OK) return rc;
  } else {
    int rc = solo_step(h, h->s_act, h->s_obs, h->s_rew, h->s_done, stream);
    if (rc != SOLO_OK) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(h_obs, h->s_obs, n * h->D * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(h, cudaMemcpyAsync(h_reward, h->s_rew, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(h, cudaMemcpyAsync(h_done, h->s_done, n * sizeof(float), cudaMemcpyDeviceToHost, s));
  }
  CUDA_TRY(h, cudaStreamSynchronize(s));
  return SOLO_OK;
}

int solo_get_observation(SoloHandle* h, float* d_obs, void* stream) {
  if (!h || !d_obs) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128, blocks = (h->n * 4 + threads - 1) / threads;
  if (h->njl == 3) obs_kernel<3><<<blocks, threads, 0, s>>>(h->d, h->sc, h->n, h->D0, h->D, d_obs);
  else obs_kernel<2><<<blocks, threads, 0, s>>>(h->d, h->sc, h->n, h->D0, h->D, d_obs);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_get_state(SoloHandle* h, float* d_state, void* stream) {
  if (!h || !d_state) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128, blocks = (h->n * 4 + threads - 1) / threads;
  if (h->njl == 3) get_state_kernel<3><<<blocks, threads, 0, s>>>(h->d, h->n, d_state);
  else get_state_kernel<2><<<blocks, threads, 0, s>>>(h->d, h->n, d_state);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_set_state(SoloHandle* h, const float* d_state, void* stream) {
  if (!h || !d_state) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128, blocks = (h->n * 4 + threads - 1) / threads;
  if (h->njl == 3) set_state_kernel<3><<<blocks, threads, 0, s>>>(h->d, h->sc, h->n, h->D0, d_state);
  else set_state_kernel<2><<<blocks, threads, 0, s>>>(h->d, h->sc, h->n, h->D0, d_state);
  h->launches++;
  h->was_reset = true;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_set_goals(SoloHandle* h, const float* d_goals, void* stream) {
  if (!h || !d_goals) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  set_goal_kernel<<<(h->n + 127) / 128, 128, 0, s>>>(h->d, h->n, h->njl, h->D0, h->params.task, d_goals);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_get_contacts(SoloHandle* h, float* d_out, void* stream) {
  if (!h || !d_out) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  contacts_kernel<<<(h->n * 4 + 127) / 128, 128, 0, s>>>(h->d, h->sc, h->n, d_out);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_set_contacts(SoloHandle* h, const float* d_force, void* stream) {
  if (!h || !d_force) return fail(h, SOLO_E_ARG, "null argument");
  set_contacts_kernel<<<(h->n * 4 + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d, h->sc, h->n, h->njl, h->D0, d_force);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_get_work_counters(SoloHandle* h, int32_t* d_out, void* stream) {
  if (!h || !d_out) return fail(h, SOLO_E_ARG, "null argument");
  work_kernel<<<(h->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d, h->n, d_out);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_forward_dynamics(SoloHandle* h, const float* d_state, const float* d_tau, float* d_qdd, void* stream) {
  if (!h || !d_state || !d_tau || !d_qdd) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128, blocks = (h->n * 4 + threads - 1) / threads;
  const float4* envp = h->randomize ? h->dyn.envp : nullptr;
  if (h->njl == 3) fd_kernel<3><<<blocks, threads, 0, s>>>(h->mc, h->sc, h->n, d_state, d_tau, d_qdd, envp);
  else fd_kernel<2><<<blocks, threads, 0, s>>>(h->mc, h->sc, h->n, d_state, d_tau, d_qdd, envp);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_substep(SoloHandle* h, const float* d_tau, void* stream) {
  if (!h || !d_tau) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  StepArgs a = make_step_args(h, MODE_SUBSTEP, h->n, d_tau, nullptr, nullptr, nullptr);
  launch_step(h, a, s);
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_actuator_step(SoloHandle* h, const float* d_cmd, int32_t n_ticks, void* stream) {
  if (!h || !d_cmd || n_ticks <= 0) return fail(h, SOLO_E_ARG, "bad argument to solo_actuator_step");
  if (!h->was_reset) return fail(h, SOLO_E_STATE, "env.reset() must be called before step");
  cudaStream_t s = (cudaStream_t)stream;
  StepArgs a = make_step_args(h, MODE_SUBSTEP, h->n, d_cmd, nullptr, nullptr, nullptr);
  const int blocks = (h->n + 7) / 8;
  if (h->sc.body_contacts) {      /* 8 envs x 5 KB of row records per one-warp block: below the 48 KB default */
    const size_t smem = (size_t)8 * kBodyEnvStride * sizeof(float);
    if (h->njl == 3) actuator_kernel<3, true><<<blocks, kBlockThreads, smem, s>>>(a, n_ticks);
    else actuator_kernel<2, true><<<blocks, kBlockThreads, smem, s>>>(a, n_ticks);
  } else {
    if (h->njl == 3) actuator_kernel<3, false><<<blocks, kBlockThreads, 0, s>>>(a, n_ticks);
    else actuator_kernel<2, false><<<blocks, kBlockThreads, 0, s>>>(a, n_ticks);
  }
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_set_external_force(SoloHandle* h, const float* d_force, void* stream) {
  if (!h || !d_force) return fail(h, SOLO_E_ARG, "null argument");
  set_fext_kernel<<<(h->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d, h->n, d_force);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_get_feet(SoloHandle* h, float* d_out, void* stream) {
  if (!h || !d_out) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128, blocks = (h->n * 4 + threads - 1) / threads;
  if (h->njl == 3) feet_kernel<3><<<blocks, threads, 0, s>>>(h->d, h->mc, h->n, d_out);
  else feet_kernel<2><<<blocks, threads, 0, s>>>(h->d, h->mc, h->n, d_out);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_action_to_torque(SoloHandle* h, const float* d_actions, float* d_tau, void* stream) {
  if (!h || !d_actions || !d_tau) return fail(h, SOLO_E_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  const int threads = 128, blocks = (h->n * 4 + threads - 1) / threads;
  const float4* envp = h->randomize ? h->dyn.envp : nullptr;
  if (h->njl == 3) torque_kernel<3><<<blocks, threads, 0, s>>>(h->d, h->sc, h->n, h->A, d_actions, d_tau, envp);
  else torque_kernel<2><<<blocks, threads, 0, s>>>(h->d, h->sc, h->n, h->A, d_actions, d_tau, envp);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_get_env_params(SoloHandle* h, float* d_out, void* stream) {
  if (!h || !d_out) return fail(h, SOLO_E_ARG, "null argument");
  env_params_kernel<<<(h->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->dyn.envp, h->n, d_out);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_get_push_force(SoloHandle* h, float* d_out, void* stream) {
  if (!h || !d_out) return fail(h, SOLO_E_ARG, "null argument");
  push_force_kernel<<<(h->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      h->d.book, h->dyn.push, (uint32_t)(h->seed & 0xffffffffu), (uint32_t)(h->seed >> 32), h->env_id_offset, h->n,
      d_out);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_episode_stats(SoloHandle* h, SoloEpisodeStats* d_stats, void* stream) {
  if (!h || !d_stats) return fail(h, SOLO_E_ARG, "null argument");
  CUDA_TRY(h, cudaMemcpyAsync(d_stats, h->d.stats, (size_t)h->n * sizeof(SoloEpisodeStats),
                              cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return SOLO_OK;
}

int solo_accumulate_episode_stats(SoloHandle* h, const float* d_done, double* d_acc, void* stream) {
  if (!h || !d_done || !d_acc) return fail(h, SOLO_E_ARG, "null argument");
  episode_accumulate_kernel<<<(h->n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(h->d.stats, d_done, h->n, d_acc);
  h->launches++;
  CUDA_TRY(h, cudaGetLastError());
  return SOLO_OK;
}

int solo_set_goal_radius(SoloHandle* h, double goal_radius) {
  if (!h) return fail(nullptr, SOLO_E_ARG, "null handle");
  h->goal_radius = (float)goal_radius;
  /* The radius lives in device memory (DevArrays::mut) because a step captured into a CUDA graph bakes its
   * kernel parameters: a by-value radius would stay at its capture-time value.  The call has no stream
   * argument and is rare (one curriculum increment per so many updates), so it simply orders itself after
   * everything in flight on the device and writes synchronously. */
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaDeviceSynchronize());
  CUDA_TRY(h, cudaMemcpy(const_cast<float*>(h->d.mut) + kMutGoalRadius, &h->goal_radius, sizeof(float),
                         cudaMemcpyHostToDevice));
  return SOLO_OK;
}

int solo_gae(const float* d_rewards, const float* d_values, const float* d_masks, float* d_returns, int32_t T,
             int32_t N, float gamma, float lam, int32_t use_gae, void* stream) {
  if (!d_rewards || !d_values || !d_masks || !d_returns || T <= 0 || N <= 0)
    return fail(nullptr, SOLO_E_ARG, "bad argument to solo_gae");
  cudaStream_t s = (cudaStream_t)stream;
  const int blocks = (N + kGaeEnvs - 1) / kGaeEnvs, threads = kGaeEnvs * kGaeChunks;
  const char* ev = getenv("SOLO_GAE_SERIAL");
  const bool serial = (ev && ev[0] == '1') || T > kGaeChunks * kGaeMaxL;
  if (serial)
    gae_kernel<<<(N + 127) / 128, 128, 0, s>>>(d_rewards, d_values, d_masks, d_returns, T, N, gamma, lam, use_gae);
  else if (T <= kGaeChunks * 8)
    gae_chunked_kernel<8><<<blocks, threads, 0, s>>>(d_rewards, d_values, d_masks, d_returns, T, N, gamma, lam, use_gae);
  else if (T <= kGaeChunks * 16)
    gae_chunked_kernel<16><<<blocks, threads, 0, s>>>(d_rewards, d_values, d_masks, d_returns, T, N, gamma, lam, use_gae);
  else if (T <= kGaeChunks * 25)      /* T = 400, the episode length of every shipped config */
    gae_chunked_kernel<25><<<blocks, threads, 0, s>>>(d_rewards, d_values, d_masks, d_returns, T, N, gamma, lam, use_gae);
  else
    gae_chunked_kernel<kGaeMaxL><<<blocks, threads, 0, s>>>(d_rewards, d_values, d_masks, d_returns, T, N, gamma, lam, use_gae);
  if (cudaGetLastError() != cudaSuccess) return fail(nullptr, SOLO_E_CUDA, "gae_kernel launch failed");
  return SOLO_OK;
}

int64_t solo_launch_count(const SoloHandle* h) { return h ? h->launches : 0; }

#ifdef SOLO_TRACE
/* tools only: copy the phase stamps of the last wide step to the host (int64 [1024][8]) */
int solo_debug_wide_trace(long long* h_out) {
  return cudaMemcpyFromSymbol(h_out, solo::g_wide_trace, sizeof(long long) * 1024 * 8) == cudaSuccess ? 0 : -3;
}
int solo_debug_narrow_trace(long long* h_out) {
  return cudaMemcpyFromSymbol(h_out, solo::g_narrow_trace, sizeof(long long) * 1024 * 8 * 8) == cudaSuccess ? 0 : -3;
}
int solo_debug_wide_trace_helpers(long long* h_out) {
  return cudaMemcpyFromSymbol(h_out, solo::g_wide_trace_h, sizeof(long long) * 1024 * 3 * 8) == cudaSuccess ? 0 : -3;
}
#endif

const char* solo_step_variant(const SoloHandle* h) {
  if (!h) return "";
  static const char* const kNames[3][4] = {
      {"latency", "latency+rand", "latency+push", "latency+rand+push"},
      {"throughput", "throughput+rand", "throughput+push", "throughput+rand+push"},
      {"body", "body+rand", "body+push", "body+rand+push"}};   /* body: the latency shape + the general contact path */
  const int opts = (h->randomize ? 1 : 0) + (h->push ? 2 : 0);
  if (h->sc.body_contacts) return kNames[2][opts];
  if (h->variant == VARIANT_WIDE) return "wide";
  return kNames[h->variant == VARIANT_THROUGHPUT ? 1 : 0][opts];
}

}  // extern "C"

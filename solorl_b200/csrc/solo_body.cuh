/*
 * solo_body.cuh — contacts of links other than the feet with the flat ground (SURVEY §8f n4,
 * SoloSimParams.body_contacts): one sphere per knee (centre = KFE joint origin, on the lower-leg link) and the
 * eight corners of the base box.  In Bullet a collapsed robot rests on the convex hulls of its knees / base
 * (solo.py:72-73) and may stay above the z < 0.05 termination height (baseEnv.py:169) until the timeout.
 *
 * An env that holds such a point leaves the register-resident Delassus path (at most 16 rows per env) for the
 * general one below: up to 16 contact points (feet, knees, lower and upper base corners) x 3 rows + 4
 * joint-limit rows = 52 rows, kept as row RECORDS in shared memory.  A record holds what one row needs of the
 * articulated-body response, in the same base-axes formulation as the foot rows (solo_core.cuh):
 *   P  base wrench per unit row impulse, K = IA0^-1 P, sP[k] = S_k . (the impulse's wrench at joint k of the
 *   row's leg; zero for rows of the base itself), g[k] = sP[k] / D_k, b = target relative velocity,
 *   diag = P.K + sum_k sP[k] g[k] (the row's Delassus diagonal).
 * With  dv0 = sum_c K_c lambda_c  (base velocity change, base axes) and  s[leg][k] = sum_{c on leg} sP_c[k]
 * lambda_c  the product of Delassus row r with lambda is  P_r . dv0 + g_r . s[leg_r]  -- no 52 x 52 matrix is
 * ever formed -- and dv0, s are exactly what the impulse application needs afterwards.
 * The sweep (body_pgs) restates the same Bullet order as the foot-only path and the oracle
 * (btMultiBodyConstraintSolver::solveSingleIteration [3P]): joint-limit rows, the normals of all points, then
 * the friction pair of each point; points ordered feet, knees, lower corners, upper corners, legs 0..3 inside
 * each group (oracle/solo_oracle.c:detect_contacts).
 * The four lanes of an env run the sweep redundantly on the shared records: no shuffle and no warp-wide
 * convergence is needed, so envs of one warp may take the general path independently of each other, and an
 * env's result does not depend on which envs share its warp (shard invariance stays bitwise).
 */
#pragma once
#include "solo_core.cuh"

namespace solo {

constexpr int kBodyPts = 16;                        /* feet 0-3, knees 4-7, lower corners 8-11, upper corners 12-15 */
constexpr int kBodySlots = 4 + 3 * kBodyPts;        /* slot l < 4: limit row of leg l; 4 + 3 p + m: row m of point p */
constexpr int kBodyRowW = 24;                       /* floats per row record (six float4) */
constexpr int kBodyEnvStride = kBodySlots * kBodyRowW + 4;   /* +4 words: the eight envs of a warp start four banks apart */
/* record layout */
enum { kBrP = 0, kBrB = 6, kBrDinv = 7, kBrG = 8, kBrDiag = 11, kBrK = 12, kBrSP = 18, kBrLam = 21 };

SOLO_HD constexpr int body_slot(int point, int m) { return 4 + 3 * point + m; }

/* The four lanes of an env run the sweep on the same records and each writes the (identical) new impulse back:
 * a lane that ran ahead must not overwrite an impulse before its siblings have read the old value, so the group
 * is synchronised between the read and the write of every row relaxation (nothing to do in the host replay). */
SOLO_HD void body_group_sync(unsigned gmask) {
#if defined(__CUDA_ARCH__)
  __syncwarp(gmask);
#else
  (void)gmask;
#endif
}

SOLO_HD int body_ctz(unsigned x) {
#if defined(__CUDA_ARCH__)
  return __ffs((int)x) - 1;
#else
  return __builtin_ctz(x);
#endif
}

struct BodyRowR {
  float P[6], b, dinv, g[3], diag, K[6], sP[3];
};
SOLO_HD void body_row_load(const float* r, BodyRowR& o) {
#if defined(__CUDA_ARCH__)
  const float4* v = reinterpret_cast<const float4*>(r);
  const float4 a = v[0], c = v[1], d = v[2], e = v[3], f = v[4];
  o.P[0] = a.x; o.P[1] = a.y; o.P[2] = a.z; o.P[3] = a.w;
  o.P[4] = c.x; o.P[5] = c.y; o.b = c.z; o.dinv = c.w;
  o.g[0] = d.x; o.g[1] = d.y; o.g[2] = d.z; o.diag = d.w;
  o.K[0] = e.x; o.K[1] = e.y; o.K[2] = e.z; o.K[3] = e.w;
  o.K[4] = f.x; o.K[5] = f.y; o.sP[0] = f.z; o.sP[1] = f.w;
  o.sP[2] = r[kBrSP + 2];
#else
  for (int i = 0; i < 6; i++) { o.P[i] = r[kBrP + i]; o.K[i] = r[kBrK + i]; }
  for (int i = 0; i < 3; i++) { o.g[i] = r[kBrG + i]; o.sP[i] = r[kBrSP + i]; }
  o.b = r[kBrB]; o.dinv = r[kBrDinv]; o.diag = r[kBrDiag];
#endif
}

/* write the record of one row; sP has NJL entries (nullptr: a row of the base itself) */
template <int NJL>
SOLO_HD void body_row_store(float* r, const float* P, const float* K, const float* sP, const float* invD, float b) {
  float diag = dot6(P, K);
#pragma unroll
  for (int i = 0; i < 6; i++) { r[kBrP + i] = P[i]; r[kBrK + i] = K[i]; }
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float s = (sP != nullptr && k < NJL) ? sP[k] : 0.f;
    const float g = (sP != nullptr && k < NJL) ? s * invD[k] : 0.f;
    r[kBrSP + k] = s; r[kBrG + k] = g;
    diag += s * g;
  }
  r[kBrB] = b; r[kBrDiag] = diag; r[kBrDinv] = solo_rcp(diag); r[kBrLam] = 0.f;
  r[kBrLam + 1] = 0.f; r[kBrLam + 2] = 0.f;
}

/* spatial velocity of the last link of a leg about O_last with the UPDATED velocities, base axes
 * (the velocity part of contact_geometry) */
template <int NJL>
SOLO_HD void last_link_velocity(const BaseState& st, const BaseWork& bw, const Lane<NJL>& ln, float* v6) {
  mat3T_mulv(bw.R, st.w, v6);
  mat3T_mulv(bw.R, st.v, v6 + 3);
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    cross3_add(v6, ln.r[k], v6 + 3);
    v6[0] += ln.ax[k][0] * ln.qd[k]; v6[1] += ln.ax[k][1] * ln.qd[k]; v6[2] += ln.ax[k][2] * ln.qd[k];
  }
}
/* knee sphere: centre = O_last (the KFE joint origin), radius knee_r; rc = contact point relative to O_last */
template <int NJL>
SOLO_HD bool knee_geometry(const SimConst& sc, const BaseState& st, const BaseWork& bw, const Lane<NJL>& ln,
                           float* rc, float& dist) {
  const float nb[3] = {bw.R[6], bw.R[7], bw.R[8]};          /* world z in base coordinates */
  dist = st.p[2] + dot3(nb, ln.ol) - sc.knee_r;
  rc[0] = -sc.knee_r * nb[0]; rc[1] = -sc.knee_r * nb[1]; rc[2] = -sc.knee_r * nb[2];
  return dist < sc.margin;
}
/* corner `leg` of the lower (g = 0) / upper (g = 1) face of the base box: FL (+x,+y) FR (+x,-y) HL (-x,+y) HR (-x,-y);
 * rc = the corner relative to the base origin, base axes */
SOLO_HD bool corner_geometry(const SimConst& sc, const BaseState& st, const BaseWork& bw, int leg, int g, float* rc,
                             float& dist) {
  rc[0] = (leg < 2) ? sc.base_hx : -sc.base_hx;
  rc[1] = (leg & 1) ? -sc.base_hy : sc.base_hy;
  rc[2] = g ? sc.base_zhi : sc.base_zlo;
  const float nb[3] = {bw.R[6], bw.R[7], bw.R[8]};
  dist = st.p[2] + dot3(nb, rc);
  return dist < sc.margin;
}
/* one row (m = 0 normal, 1 / 2 friction) of a contact point of the base link: no joint between the point and
 * the base, so P is the impulse's wrench about the base origin itself */
SOLO_HD void base_point_row(const SimConst& sc, const float* R, const Ldl6& F, const float* rc, const float* vb6,
                            float dist, int m, float* P, float* K, float& b) {
  float d[3];
  if (m == 0) { d[0] = R[6]; d[1] = R[7]; d[2] = R[8]; }
  else if (m == 1) { d[0] = -R[3]; d[1] = -R[4]; d[2] = -R[5]; }
  else { d[0] = R[0]; d[1] = R[1]; d[2] = R[2]; }
  cross3(rc, d, P);
  P[3] = d[0]; P[4] = d[1]; P[5] = d[2];
  const float vel = dot6(P, vb6);
#pragma unroll
  for (int i = 0; i < 6; i++) K[i] = P[i];
  ldl6_solve(F, K);
  if (m == 0) {
    const float pen = dist + sc.slop;
    b = -vel - pen * (pen > 0.f ? sc.inv_dt : sc.erp * sc.inv_dt);
  } else {
    b = -vel;
  }
}

/* s[leg][k] with a run-time leg: selects, so that s stays in registers */
SOLO_HD float body_sel(const float (*s)[3], int leg, int k) {
  return leg == 0 ? s[0][k] : (leg == 1 ? s[1][k] : (leg == 2 ? s[2][k] : s[3][k]));
}
SOLO_HD float body_resid(const BodyRowR& r, const float* dv0, const float (*s)[3], int leg) {
  const float a = r.P[0] * dv0[0] + r.P[1] * dv0[1] + r.P[2] * dv0[2];
  const float c = r.P[3] * dv0[3] + r.P[4] * dv0[4] + r.P[5] * dv0[5];
  const float d = r.g[0] * body_sel(s, leg, 0) + r.g[1] * body_sel(s, leg, 1) + r.g[2] * body_sel(s, leg, 2);
  return r.b - ((a + c) + d);
}
SOLO_HD void body_apply(const BodyRowR& r, float d, float* dv0, float (*s)[3], int leg) {
#pragma unroll
  for (int i = 0; i < 6; i++) dv0[i] = fmaf(r.K[i], d, dv0[i]);
#pragma unroll
  for (int j = 0; j < 4; j++) {
#pragma unroll
    for (int k = 0; k < 3; k++) s[j][k] = fmaf((leg == j) ? r.sP[k] : 0.f, d, s[j][k]);
  }
}

/* The sweep loop of one env over its row records (`rows` = the env's region, lambda lives in the records).
 * lmask: legs holding a joint-limit row; pmask: contact points present.  Returns the number of sweeps. */
template <bool CONE>
SOLO_HD int body_pgs(float* rows, unsigned lmask, unsigned pmask, const SimConst& sc, unsigned gmask, float* dv0,
                     float (*s)[3]) {
#pragma unroll
  for (int i = 0; i < 6; i++) dv0[i] = 0.f;
#pragma unroll
  for (int j = 0; j < 4; j++) { s[j][0] = 0.f; s[j][1] = 0.f; s[j][2] = 0.f; }
  int it = 0;
  for (; it < sc.iters;) {
    float res = 0.f;           /* largest |velocity residual| of the sweep */
    it++;
    if (lmask) {
      /* the limit rows of an env (one per leg at most) are relaxed as one simultaneous group, like the
       * foot-only path (pgs_sweeps4) and the oracle under limit_rows_per_leg = 1 */
      float dl[4], nl[4];
#pragma unroll
      for (int l = 0; l < 4; l++) {
        dl[l] = 0.f; nl[l] = 0.f;
        if ((lmask >> l) & 1u) {
          const float* rr = rows + l * kBodyRowW;
          BodyRowR r;
          body_row_load(rr, r);
          const float lam = rr[kBrLam];
          nl[l] = fminf(fmaxf(fmaf(body_resid(r, dv0, s, l), r.dinv, lam), 0.f), sc.lim_max_impulse);
          dl[l] = nl[l] - lam;
          res = fmaxf(res, fabsf(dl[l] * r.diag));
        }
      }
      body_group_sync(gmask);
#pragma unroll
      for (int l = 0; l < 4; l++) {
        if ((lmask >> l) & 1u) {
          float* rr = rows + l * kBodyRowW;
          BodyRowR r;
          body_row_load(rr, r);
          rr[kBrLam] = nl[l];
          body_apply(r, dl[l], dv0, s, l);
        }
      }
    }
    for (unsigned m = pmask; m; m &= m - 1) {                 /* normals of all points */
      const int p = body_ctz(m);
      float* rr = rows + body_slot(p, 0) * kBodyRowW;
      BodyRowR r;
      body_row_load(rr, r);
      const float lam = rr[kBrLam];
      const float nv = fmaxf(fmaf(body_resid(r, dv0, s, p & 3), r.dinv, lam), 0.f);
      const float d = nv - lam;
      body_group_sync(gmask);
      rr[kBrLam] = nv;
      res = fmaxf(res, fabsf(d * r.diag));
      body_apply(r, d, dv0, s, p & 3);
    }
    for (unsigned m = pmask; m; m &= m - 1) {                 /* friction pair of each point */
      const int p = body_ctz(m);
      const int leg = p & 3;
      float* rn = rows + body_slot(p, 0) * kBodyRowW;
      float* ra = rn + kBodyRowW;
      float* rb = ra + kBodyRowW;
      const float lim = sc.mu * rn[kBrLam];
      BodyRowR A, B;
      body_row_load(ra, A);
      body_row_load(rb, B);
      const float lamA = ra[kBrLam], lamB = rb[kBrLam];
      body_group_sync(gmask);
      if (CONE) {      /* both candidates from the same state, scaled back onto the circle (pgs_cone_candidate) */
        const float sA = fmaf(body_resid(A, dv0, s, leg), A.dinv, lamA);
        const float sB = fmaf(body_resid(B, dv0, s, leg), B.dinv, lamB);
        const float n2 = fmaf(sB, sB, fmaf(sA, sA, 1e-30f));
        const float scl = fminf(lim * solo_rsqrt(n2), 1.0f);
        const float nA = sA * scl, nB = sB * scl;
        const float dA = nA - lamA, dB = nB - lamB;
        ra[kBrLam] = nA; rb[kBrLam] = nB;
        res = fmaxf(res, fabsf(dA * A.diag + dB * B.diag));
        body_apply(A, dA, dv0, s, leg);
        body_apply(B, dB, dv0, s, leg);
      } else {
        const float nA = clampf(fmaf(body_resid(A, dv0, s, leg), A.dinv, lamA), -lim, lim);
        const float dA = nA - lamA;
        ra[kBrLam] = nA;
        res = fmaxf(res, fabsf(dA * A.diag));
        body_apply(A, dA, dv0, s, leg);
        const float nB = clampf(fmaf(body_resid(B, dv0, s, leg), B.dinv, lamB), -lim, lim);
        const float dB = nB - lamB;
        rb[kBrLam] = nB;
        res = fmaxf(res, fabsf(dB * B.diag));
        body_apply(B, dB, dv0, s, leg);
      }
    }
    if (res * res <= sc.res_thr) break;
  }
  return it;
}

#if defined(__CUDACC__)
/* The same sweep as body_pgs for the four lanes of an env on the GPU, without the run-time-indexed s[leg]:
 * lane `me` keeps only the impulse sums of its own leg (s_me), so the candidate of a row is right in the lane of
 * the row's leg alone and is handed to the siblings with one shuffle inside the group; everything else (dv0, the
 * residual test, the record updates) is computed redundantly and identically by the four lanes.  Same arithmetic,
 * operand for operand, as body_pgs (which the host replay runs), so the two agree bit for bit up to the
 * compiler's FMA contraction. */
__device__ __forceinline__ float body_resid_me(const BodyRowR& r, const float* dv0, const float* s_me) {
  const float a = r.P[0] * dv0[0] + r.P[1] * dv0[1] + r.P[2] * dv0[2];
  const float c = r.P[3] * dv0[3] + r.P[4] * dv0[4] + r.P[5] * dv0[5];
  const float d = r.g[0] * s_me[0] + r.g[1] * s_me[1] + r.g[2] * s_me[2];
  return r.b - ((a + c) + d);
}
__device__ __forceinline__ void body_apply_me(const BodyRowR& r, float d, bool mine, float* dv0, float* s_me) {
#pragma unroll
  for (int i = 0; i < 6; i++) dv0[i] = fmaf(r.K[i], d, dv0[i]);
  const float dm = mine ? d : 0.f;
#pragma unroll
  for (int k = 0; k < 3; k++) s_me[k] = fmaf(r.sP[k], dm, s_me[k]);
}
template <bool CONE>
__device__ __forceinline__ int body_pgs_lanes(float* rows, unsigned lmask, unsigned pmask, const SimConst& sc,
                                              unsigned gmask, unsigned gbase, int me, float* dv0, float* s_me,
                                              const EnvDyn* dyn = nullptr) {
#pragma unroll
  for (int i = 0; i < 6; i++) dv0[i] = 0.f;
  s_me[0] = s_me[1] = s_me[2] = 0.f;
  int it = 0;
  for (; it < sc.iters;) {
    float res = 0.f;
    it++;
    if (lmask) {
      float dl[4], nl[4];
      {
        float nv = 0.f;
        if ((lmask >> me) & 1u) {
          const float* rr = rows + me * kBodyRowW;
          BodyRowR r;
          body_row_load(rr, r);
          nv = fminf(fmaxf(fmaf(body_resid_me(r, dv0, s_me), r.dinv, rr[kBrLam]), 0.f), sc.lim_max_impulse);
        }
#pragma unroll
        for (int l = 0; l < 4; l++) nl[l] = __shfl_sync(gmask, nv, gbase + l);
      }
#pragma unroll
      for (int l = 0; l < 4; l++) {
        dl[l] = 0.f;
        if ((lmask >> l) & 1u) {
          const float* rr = rows + l * kBodyRowW;
          dl[l] = nl[l] - rr[kBrLam];
          res = fmaxf(res, fabsf(dl[l] * rr[kBrDiag]));
        }
      }
      __syncwarp(gmask);
#pragma unroll
      for (int l = 0; l < 4; l++) {
        if ((lmask >> l) & 1u) {
          float* rr = rows + l * kBodyRowW;
          BodyRowR r;
          body_row_load(rr, r);
          rr[kBrLam] = nl[l];
          body_apply_me(r, dl[l], l == me, dv0, s_me);
        }
      }
    }
    for (unsigned m = pmask; m; m &= m - 1) {                 /* normals of all points */
      const int p = body_ctz(m);
      const int leg = p & 3;
      float* rr = rows + body_slot(p, 0) * kBodyRowW;
      BodyRowR r;
      body_row_load(rr, r);
      const float lam = rr[kBrLam];
      const float nv = __shfl_sync(gmask, fmaxf(fmaf(body_resid_me(r, dv0, s_me), r.dinv, lam), 0.f), gbase + leg);
      const float d = nv - lam;
      rr[kBrLam] = nv;                                        /* the shuffle above ordered the siblings' reads */
      res = fmaxf(res, fabsf(d * r.diag));
      body_apply_me(r, d, leg == me, dv0, s_me);
    }
    for (unsigned m = pmask; m; m &= m - 1) {                 /* friction pair of each point */
      const int p = body_ctz(m);
      const int leg = p & 3;
      float* rn = rows + body_slot(p, 0) * kBodyRowW;
      float* ra = rn + kBodyRowW;
      float* rb = ra + kBodyRowW;
      const float lim = env_mu(sc, dyn) * rn[kBrLam];
      BodyRowR A, B;
      body_row_load(ra, A);
      body_row_load(rb, B);
      const float lamA = ra[kBrLam], lamB = rb[kBrLam];
      if (CONE) {
        const float sA = fmaf(body_resid_me(A, dv0, s_me), A.dinv, lamA);
        const float sB = fmaf(body_resid_me(B, dv0, s_me), B.dinv, lamB);
        const float n2 = fmaf(sB, sB, fmaf(sA, sA, 1e-30f));
        const float scl = fminf(lim * solo_rsqrt(n2), 1.0f);
        const float nA = __shfl_sync(gmask, sA * scl, gbase + leg), nB = __shfl_sync(gmask, sB * scl, gbase + leg);
        const float dA = nA - lamA, dB = nB - lamB;
        ra[kBrLam] = nA; rb[kBrLam] = nB;
        res = fmaxf(res, fabsf(dA * A.diag + dB * B.diag));
        body_apply_me(A, dA, leg == me, dv0, s_me);
        body_apply_me(B, dB, leg == me, dv0, s_me);
      } else {
        const float nA = __shfl_sync(gmask, clampf(fmaf(body_resid_me(A, dv0, s_me), A.dinv, lamA), -lim, lim), gbase + leg);
        const float dA = nA - lamA;
        ra[kBrLam] = nA;
        res = fmaxf(res, fabsf(dA * A.diag));
        body_apply_me(A, dA, leg == me, dv0, s_me);
        const float nB = __shfl_sync(gmask, clampf(fmaf(body_resid_me(B, dv0, s_me), B.dinv, lamB), -lim, lim), gbase + leg);
        const float dB = nB - lamB;
        rb[kBrLam] = nB;
        res = fmaxf(res, fabsf(dB * B.diag));
        body_apply_me(B, dB, leg == me, dv0, s_me);
      }
    }
    if (res * res <= sc.res_thr) break;
  }
  return it;
}
#endif

/* Joint velocity change of one leg for the joint-space impulses us[k] = s[leg][k] accumulated on it and the
 * base velocity change dv0 (impulse_leg with the impulse sums already formed). */
template <int NJL>
SOLO_HD void body_apply_leg(Lane<NJL>& ln, const SimConst& sc, const float* us, const float* dv0) {
  float a[6];
#pragma unroll
  for (int i = 0; i < 6; i++) a[i] = dv0[i];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    cross3_add(a, ln.r[k], a + 3);
    const float dq = (us[k] - dot6(ln.h[k], a)) * ln.invD[k];
    a[0] += ln.ax[k][0] * dq; a[1] += ln.ax[k][1] * dq; a[2] += ln.ax[k][2] * dq;
    ln.qd[k] = clampf(ln.qd[k] + dq, -sc.vmax, sc.vmax);
  }
}

/* Records of the rows this lane (= leg) owns: its limit row, its foot, its knee and its two base corners. */
template <int NJL>
struct BodyLaneGeom {
  float kn_rc[3], kn_dist, c_rc[2][3], c_dist[2];
  bool kn_on, c_on[2];
};
template <int NJL>
SOLO_HD void body_lane_geometry(const SimConst& sc, const BaseState& st, const BaseWork& bw, const Lane<NJL>& ln,
                                int leg, BodyLaneGeom<NJL>& g) {
  g.kn_on = knee_geometry<NJL>(sc, st, bw, ln, g.kn_rc, g.kn_dist);
  g.c_on[0] = corner_geometry(sc, st, bw, leg, 0, g.c_rc[0], g.c_dist[0]);
  g.c_on[1] = corner_geometry(sc, st, bw, leg, 1, g.c_rc[1], g.c_dist[1]);
}
template <int NJL>
SOLO_HD void body_lane_fill(const SimConst& sc, const BaseState& st, const BaseWork& bw, const Lane<NJL>& ln,
                            const LimitRow<NJL>* lr, int leg, bool foot_on, const BodyLaneGeom<NJL>& g, float* rows) {
  if (lr != nullptr && lr->active)
    body_row_store<NJL>(rows + leg * kBodyRowW, lr->P, lr->K, lr->U, ln.invD, lr->b);
  if (foot_on) {
#pragma unroll
    for (int m = 0; m < 3; m++) {
      float sPm[NJL];
#pragma unroll
      for (int k = 0; k < NJL; k++) sPm[k] = ln.sP[k][m];
      body_row_store<NJL>(rows + body_slot(leg, m) * kBodyRowW, ln.P[m], ln.K[m], sPm, ln.invD, ln.b[m]);
    }
  }
  if (g.kn_on) {
    float v6[6];
    last_link_velocity<NJL>(st, bw, ln, v6);
    for (int m = 0; m < 3; m++) {
      float sPm[NJL], P[6], K[6], b;
      contact_row<NJL>(sc, bw.R, bw.F, ln.ax, ln.r, ln.h, ln.invD, g.kn_rc, v6, g.kn_dist, m, sPm, P, K, b);
      body_row_store<NJL>(rows + body_slot(4 + leg, m) * kBodyRowW, P, K, sPm, ln.invD, b);
    }
  }
  if (g.c_on[0] || g.c_on[1]) {
    float vb6[6];
    mat3T_mulv(bw.R, st.w, vb6);
    mat3T_mulv(bw.R, st.v, vb6 + 3);
    for (int c = 0; c < 2; c++) {
      if (!g.c_on[c]) continue;
      for (int m = 0; m < 3; m++) {
        float P[6], K[6], b;
        base_point_row(sc, bw.R, bw.F, g.c_rc[c], vb6, g.c_dist[c], m, P, K, b);
        body_row_store<NJL>(rows + body_slot(8 + 4 * c + leg, m) * kBodyRowW, P, K, nullptr, ln.invD, b);
      }
    }
  }
}

}  // namespace solo

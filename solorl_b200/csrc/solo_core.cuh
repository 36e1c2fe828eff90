/*
 * solo_core.cuh — per-lane math of the fused Solo8/Solo12 substep (sm_100a FP32 SIMT).
 *
 * Mapping: ONE LANE PER LEG, four lanes per environment.  Every spatial quantity of an
 * environment is expressed in the AXES of the base link frame; the quantities of link k
 * are taken about that link's own joint origin O_k (a point on the joint axis).  So a
 * joint's motion subspace is S = (axis, 0), no rotation is ever applied to a 6x6
 * inertia, and going from a link to its parent is a pure translation by r_k = O_k -
 * O_{k-1}.  Taking moments about the joint's own origin is what keeps fp32 within 1e-5
 * of the fp64 oracle: the joint-axis inertia D = a.A.a is a sum of positive terms
 * instead of the difference of large m|r|^2 terms it would be about the base origin.
 * The four legs are summed into the floating base with two xor-shuffles and the 6x6 base
 * solve is done redundantly by the four lanes.  Contacts are solved in Delassus form
 * A = P^T IA0^-1 P + blockdiag(L): each lane keeps the three rows of its own foot in
 * registers and the projected Gauss-Seidel sweep broadcasts one impulse change per row
 * relaxation with a shuffle inside the four-lane group (see PgsLane); a leg whose joint is
 * at a URDF limit carries a fourth row (see LimitRow / PgsLane4).
 *
 * This formulation is deliberately different from the CPU oracle (oracle/solo_oracle.c:
 * link-COM frames, 6x6 transforms, one impulse-response pass per contact row), which is
 * what makes the parity tests meaningful.  What is computed is the same physics as the
 * reference's `p.stepSimulation()` (reference solo.py:265) restated in DESIGN.md.
 *
 * Everything here is `__host__ __device__` so that tests/emu can replay the exact lane
 * program on the CPU in fp32 (the `-m "not gpu"` check of the kernel math); the product
 * only ever runs it on the GPU.
 */
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define SOLO_HD __host__ __device__ __forceinline__
#else
#define SOLO_HD inline
#endif

namespace solo {

constexpr int kMaxJL = 3;  /* joints per leg: 2 (Solo8: HFE,KFE) or 3 (Solo12: HAA,HFE,KFE) */
constexpr int kRows = 12;  /* 4 feet x (normal, 2 friction) */

/* joint axis of leg joint k: Solo12 = (x,y,y), Solo8 = (y,y) (solo12.urdf:48,91,134; solo.urdf:49,94) */
template <int NJL>
SOLO_HD constexpr int axis_of(int k) { return (NJL == 3 && k == 0) ? 0 : 1; }

struct LegConst {
  float jo[kMaxJL][3];  /* joint origin in the parent link frame */
  float m[kMaxJL];      /* link mass (last link: lower leg + foot merged) */
  float c[kMaxJL][3];   /* COM in the link frame (merged for the last link) */
  float I[kMaxJL][6];   /* inertia about the COM: xx xy xz yy yz zz (merged for the last link) */
  /* Bullet damps every URDF link separately, so the merged last link keeps two damping bodies */
  float m_own, c_own[3];
  float m_foot, c_foot[3];
  float Idamp[6];       /* I_own + I_foot, each about its own COM */
  float foot_ctr[3];    /* collision-sphere centre in the last link frame */
};

struct ModelConst {
  LegConst leg[4];
  float base_m;
  float base_I[6];
  float foot_r;
  int njl;
};

struct SimConst {
  float dt, inv_dt, gz, klin, kang, vmax, erp, slop, margin, mu;
  int iters, cone, frame_skip, torque_hold;
  float res_thr;   /* squared velocity residual below which the PGS sweep loop stops (0 = never) */
  int control;
  float kp, kd, max_torque, q_limit, qd_limit;
  int task, episode_length, H;
  float initial_z;
  int settle_min, settle_span;
  float goal_reach, inv_pg_dt, flag_force, fall_z, stand_z;
  int reset_mode;
  /* joint-limit rows ([3P] btMultiBodyJointLimitConstraint) */
  int joint_limits;
  float lim_erp, lim_max_impulse, lim_split_thr;
  /* contacts of knees and base-box corners with the ground (solo_body.cuh) */
  int body_contacts;
  float knee_r, base_hx, base_hy, base_zlo, base_zhi;
};

/* Dynamics of one env of a randomised handle (SoloSimParams.randomize): contact friction, base mass / inertia
 * scale, motor strength.  Wherever a `const EnvDyn*` is taken, nullptr means the nominal values of SimConst /
 * ModelConst, and the code is then exactly that of a handle without randomisation. */
struct EnvDyn {
  float mu, sm, st;
};
SOLO_HD float env_mu(const SimConst& sc, const EnvDyn* dyn) { return dyn != nullptr ? dyn->mu : sc.mu; }

/* ------------------------------------------------------------------ small helpers */
SOLO_HD float dot3(const float* a, const float* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
SOLO_HD void cross3(const float* a, const float* b, float* o) {
  float x = a[1] * b[2] - a[2] * b[1];
  float y = a[2] * b[0] - a[0] * b[2];
  float z = a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z;
}
SOLO_HD void cross3_add(const float* a, const float* b, float* o) {
  o[0] += a[1] * b[2] - a[2] * b[1];
  o[1] += a[2] * b[0] - a[0] * b[2];
  o[2] += a[0] * b[1] - a[1] * b[0];
}
SOLO_HD float dot6(const float* a, const float* b) {
  return (a[0] * b[0] + a[1] * b[1] + a[2] * b[2]) + (a[3] * b[3] + a[4] * b[4] + a[5] * b[5]);
}
SOLO_HD float clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }
/* Two dot6 against the same vector at once: on the GPU as packed FP32 (sm_100 mul / fma / add .f32x2 = SASS FMUL2 /
 * FFMA2 / FADD2, the common operand k[i] broadcast by the instruction's scalar form), in exactly dot6's order of
 * operations per half -- same bits, half the instructions.  The straight-line part of a substep is bound by
 * instruction fetch (profiles/r2_icache_probe.txt), so instructions saved are cycles saved. */
SOLO_HD void dot6_pair(const float* a, const float* b, const float* k, float& ra, float& rb) {
#if defined(__CUDA_ARCH__)
  /* nvcc contracts dot6's (x0 + x1 + x2) + (x3 + x4 + x5), x_i = a_i k_i, as fma(a2,k2, fma(a0,k0, a1*k1)) per
   * half-sum: the packed form follows that order so that the bits do not change */
  unsigned long long t, u, x, s;
#define SOLO_PK(i) asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(a[i]), "f"(b[i])); asm("mov.b64 %0, {%1, %1};" : "=l"(s) : "f"(k[i]))
  SOLO_PK(1); asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(x), "l"(s));
  SOLO_PK(0); asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(t) : "l"(x), "l"(s));
  SOLO_PK(2); asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(t) : "l"(x), "l"(s));
  SOLO_PK(4); asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(u) : "l"(x), "l"(s));
  SOLO_PK(3); asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(u) : "l"(x), "l"(s));
  SOLO_PK(5); asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(u) : "l"(x), "l"(s));
#undef SOLO_PK
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(t) : "l"(u));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(ra), "=f"(rb) : "l"(t));
#else
  ra = dot6(a, k); rb = dot6(b, k);
#endif
}
SOLO_HD float solo_rsqrt(float x) {   /* x >= 1e-30: one MUFU.RSQ, no denormal fix-up code */
#if defined(__CUDA_ARCH__)
  float y;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return 1.0f / sqrtf(x);
#endif
}
/* Joint-angle sine/cosine to ~1 ulp without sincosf's slow-path code: three-part Cody-Waite reduction
 * by pi/2 (exact for |x| <= 100 rad; the joint range is +-10) and the Cephes single-precision minimax
 * polynomials on [-pi/4, pi/4].  ~25 instructions.  (MUFU.SIN/COS would be 10, but their 4e-7 absolute
 * error becomes a 1e-7 m foot-height error, which the contact rows amplify by 1/dt: measured, it doubled
 * the median single-substep error against the oracle and produced rare 2e-3 outliers.)  The same code
 * runs on the host, so the CPU replay of the lane program stays bit-comparable. */
SOLO_HD void solo_sincos(float x, float* s, float* c) {
  const float kf = rintf(x * 0.63661977236758134f);
  const int k = (int)kf;
  float r = fmaf(kf, -1.5703125f, x);
  r = fmaf(kf, -4.837512969970703125e-4f, r);
  r = fmaf(kf, -7.54978995489188216e-8f, r);
  const float z = r * r;
  float sp = fmaf(fmaf(fmaf(-1.9515295891e-4f, z, 8.3321608736e-3f), z, -1.6666654611e-1f), z * r, r);
  float cp = fmaf(fmaf(fmaf(2.443315711809948e-5f, z, -1.388731625493765e-3f), z, 4.166664568298827e-2f), z * z,
                  fmaf(-0.5f, z, 1.0f));
  const bool swap = (k & 1) != 0;
  float sv = swap ? cp : sp;
  float cv = swap ? sp : cp;
  *s = (k & 2) ? -sv : sv;
  *c = ((k + 1) & 2) ? -cv : cv;
}
/* 1/x to within an ulp: MUFU.RCP and one Newton step, no denormal/slow-path code (x is a joint-axis
 * inertia, an LDL pivot or a Delassus diagonal: positive and far from the denormal range). */
SOLO_HD float solo_rcp(float x) {
#if defined(__CUDA_ARCH__)
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return fmaf(r, fmaf(-x, r, 1.0f), r);
#else
  return 1.0f / x;
#endif
}
/* norm for the Bullet damping factors k (1 + |v|): k = 0.04, so 2 ulp of the norm are immaterial */
SOLO_HD float solo_sqrt_approx(float x) {
#if defined(__CUDA_ARCH__)
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return sqrtf(x);
#endif
}
/* sym 3x3 stored xx xy xz yy yz zz times vector */
SOLO_HD void sym3_mulv(const float* S, const float* x, float* y) {
  y[0] = S[0] * x[0] + S[1] * x[1] + S[2] * x[2];
  y[1] = S[1] * x[0] + S[3] * x[1] + S[4] * x[2];
  y[2] = S[2] * x[0] + S[4] * x[1] + S[5] * x[2];
}
/* row-major 3x3 */
SOLO_HD void mat3_mulv(const float* R, const float* x, float* y) {
  float a = R[0] * x[0] + R[1] * x[1] + R[2] * x[2];
  float b = R[3] * x[0] + R[4] * x[1] + R[5] * x[2];
  float c = R[6] * x[0] + R[7] * x[1] + R[8] * x[2];
  y[0] = a; y[1] = b; y[2] = c;
}
SOLO_HD void mat3T_mulv(const float* R, const float* x, float* y) {
  float a = R[0] * x[0] + R[3] * x[1] + R[6] * x[2];
  float b = R[1] * x[0] + R[4] * x[1] + R[7] * x[2];
  float c = R[2] * x[0] + R[5] * x[1] + R[8] * x[2];
  y[0] = a; y[1] = b; y[2] = c;
}
SOLO_HD void quat_to_rot(const float* q, float* R) { /* (x,y,z,w), base -> world */
  float x = q[0], y = q[1], z = q[2], w = q[3];
  R[0] = 1.f - 2.f * (y * y + z * z); R[1] = 2.f * (x * y - w * z);       R[2] = 2.f * (x * z + w * y);
  R[3] = 2.f * (x * y + w * z);       R[4] = 1.f - 2.f * (x * x + z * z); R[5] = 2.f * (y * z - w * x);
  R[6] = 2.f * (x * z - w * y);       R[7] = 2.f * (y * z + w * x);       R[8] = 1.f - 2.f * (x * x + y * y);
}

SOLO_HD void normalize_quat(float* q) {
  float inv = 1.0f / sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  q[0] *= inv; q[1] *= inv; q[2] *= inv; q[3] *= inv;
}

/* Symmetric 6x6 spatial inertia in (angular, linear) block form:
 *   f_ang = A w + H v ,  f_lin = H^T w + M v ;  A, M symmetric (6 floats), H full (9). */
struct Sym6 {
  float A[6], H[9], M[6];
};
SOLO_HD void sym6_zero(Sym6& I) {
  for (int i = 0; i < 6; i++) { I.A[i] = 0.f; I.M[i] = 0.f; }
  for (int i = 0; i < 9; i++) I.H[i] = 0.f;
}
SOLO_HD void sym6_mulv(const Sym6& I, const float* x, float* y) {
  float a[3], b[3];
  sym3_mulv(I.A, x, a);
  mat3_mulv(I.H, x + 3, b);
  y[0] = a[0] + b[0]; y[1] = a[1] + b[1]; y[2] = a[2] + b[2];
  mat3T_mulv(I.H, x, a);
  sym3_mulv(I.M, x + 3, b);
  y[3] = a[0] + b[0]; y[4] = a[1] + b[1]; y[5] = a[2] + b[2];
}
/* I -= h h^T * s */
SOLO_HD void sym6_rank1_sub(Sym6& I, const float* h, float s) {
  float g[6];
  for (int i = 0; i < 6; i++) g[i] = h[i] * s;
  I.A[0] -= g[0] * h[0]; I.A[1] -= g[0] * h[1]; I.A[2] -= g[0] * h[2];
  I.A[3] -= g[1] * h[1]; I.A[4] -= g[1] * h[2]; I.A[5] -= g[2] * h[2];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) I.H[3 * i + j] -= g[i] * h[3 + j];
  I.M[0] -= g[3] * h[3]; I.M[1] -= g[3] * h[4]; I.M[2] -= g[3] * h[5];
  I.M[3] -= g[4] * h[4]; I.M[4] -= g[4] * h[5]; I.M[5] -= g[5] * h[5];
}
/* I += rigid body (mass m, COM c, inertia about COM Ic in the common frame) */
SOLO_HD void sym6_add_rigid(Sym6& I, float m, const float* c, const float* Ic) {
  float cc = dot3(c, c);
  float mx = m * c[0], my = m * c[1], mz = m * c[2];
  I.A[0] += Ic[0] + m * cc - mx * c[0];
  I.A[1] += Ic[1] - mx * c[1];
  I.A[2] += Ic[2] - mx * c[2];
  I.A[3] += Ic[3] + m * cc - my * c[1];
  I.A[4] += Ic[4] - my * c[2];
  I.A[5] += Ic[5] + m * cc - mz * c[2];
  /* H = m [c]x */
  I.H[1] -= mz; I.H[2] += my;
  I.H[3] += mz; I.H[5] -= mx;
  I.H[6] -= my; I.H[7] += mx;
  I.M[0] += m; I.M[3] += m; I.M[5] += m;
}

/* Re-express a spatial inertia taken about O' = O + r about O (pure translation):
 *   M stays, H <- H + [r]x M =: T,  A <- A + [r]x H^T - T [r]x   (old H on the right-hand side). */
SOLO_HD void sym6_shift(Sym6& I, const float* r) {
  const float M[9] = {I.M[0], I.M[1], I.M[2], I.M[1], I.M[3], I.M[4], I.M[2], I.M[4], I.M[5]};
  float T[9];
  /* columns of [r]x M = r x (columns of M) */
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const float mc[3] = {M[j], M[3 + j], M[6 + j]};
    float t[3];
    cross3(r, mc, t);
    T[j] = I.H[j] + t[0]; T[3 + j] = I.H[3 + j] + t[1]; T[6 + j] = I.H[6 + j] + t[2];
  }
  /* X = [r]x H^T : column j of H^T is row j of H */
  float X[9];
#pragma unroll
  for (int j = 0; j < 3; j++) {
    const float hr[3] = {I.H[3 * j], I.H[3 * j + 1], I.H[3 * j + 2]};
    float t[3];
    cross3(r, hr, t);
    X[j] = t[0]; X[3 + j] = t[1]; X[6 + j] = t[2];
  }
  /* Y = T [r]x : row i of Y = (row i of T) x r  */
  float Y[9];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const float tr[3] = {T[3 * i], T[3 * i + 1], T[3 * i + 2]};
    float t[3];
    cross3(tr, r, t);
    Y[3 * i] = t[0]; Y[3 * i + 1] = t[1]; Y[3 * i + 2] = t[2];
  }
  I.A[0] += X[0] - Y[0];
  I.A[1] += 0.5f * ((X[1] - Y[1]) + (X[3] - Y[3]));
  I.A[2] += 0.5f * ((X[2] - Y[2]) + (X[6] - Y[6]));
  I.A[3] += X[4] - Y[4];
  I.A[4] += 0.5f * ((X[5] - Y[5]) + (X[7] - Y[7]));
  I.A[5] += X[8] - Y[8];
#pragma unroll
  for (int i = 0; i < 9; i++) I.H[i] = T[i];
}

/* LDL^T factor of the 6x6 base articulated inertia */
struct Ldl6 {
  float L[15];   /* strictly lower, row-major: (1,0) (2,0) (2,1) (3,0) ... (5,4) */
  float dinv[6];
};
SOLO_HD constexpr int ldl_idx(int i, int j) { return i * (i - 1) / 2 + j; }
/* column J of the factorisation; J is a template constant so that every loop has a constant trip
 * count and all indices fold: the factor lives in registers (a run-time j left L, d and the 6x6 copy
 * in local memory, with LDL/STL round trips on the dependent chain) */
template <int J>
SOLO_HD void ldl6_column(const float (&a)[6][6], Ldl6& F, float (&d)[6]) {
  float s = a[J][J];
#pragma unroll
  for (int k = 0; k < J; k++) s -= F.L[ldl_idx(J, k)] * F.L[ldl_idx(J, k)] * d[k];
  d[J] = s;
  F.dinv[J] = solo_rcp(s);
#pragma unroll
  for (int i = J + 1; i < 6; i++) {
    float t = a[i][J];
#pragma unroll
    for (int k = 0; k < J; k++) t -= F.L[ldl_idx(i, k)] * F.L[ldl_idx(J, k)] * d[k];
    F.L[ldl_idx(i, J)] = t * F.dinv[J];
  }
}
SOLO_HD void ldl6_factor(const Sym6& I, Ldl6& F) {
  float a[6][6];
  a[0][0] = I.A[0]; a[1][0] = I.A[1]; a[2][0] = I.A[2]; a[1][1] = I.A[3]; a[2][1] = I.A[4]; a[2][2] = I.A[5];
#pragma unroll
  for (int i = 0; i < 3; i++) {
#pragma unroll
    for (int j = 0; j < 3; j++) a[3 + i][j] = I.H[3 * j + i]; /* lower-left block = H^T */
  }
  a[3][3] = I.M[0]; a[4][3] = I.M[1]; a[5][3] = I.M[2]; a[4][4] = I.M[3]; a[5][4] = I.M[4]; a[5][5] = I.M[5];
  float d[6];
  ldl6_column<0>(a, F, d);
  ldl6_column<1>(a, F, d);
  ldl6_column<2>(a, F, d);
  ldl6_column<3>(a, F, d);
  ldl6_column<4>(a, F, d);
  ldl6_column<5>(a, F, d);
}
SOLO_HD void ldl6_solve(const Ldl6& F, float* x) { /* in place */
#pragma unroll
  for (int i = 1; i < 6; i++) {
#pragma unroll
    for (int k = 0; k < i; k++) x[i] -= F.L[ldl_idx(i, k)] * x[k];
  }
#pragma unroll
  for (int i = 0; i < 6; i++) x[i] *= F.dinv[i];
#pragma unroll
  for (int i = 4; i >= 0; i--) {
#pragma unroll
    for (int k = i + 1; k < 6; k++) x[i] -= F.L[ldl_idx(k, i)] * x[k];
  }
}

/* ------------------------------------------------------------------ state */
struct BaseState {        /* world frame; replicated in the four lanes of an env */
  float p[3], q[4], v[3], w[3];
};
struct BaseWork {
  float R[9];             /* base -> world */
  float wb[3], vb[3];     /* base velocity in base coordinates */
  Ldl6 F;                 /* factor of the base articulated inertia */
};
template <int NJL>
struct Lane {             /* one leg */
  float q[NJL], qd[NJL];
  float ax[NJL][3];       /* joint axis in base axes */
  float r[NJL][3];        /* O_k - O_{k-1} in base axes (O_{-1} = base origin) */
  float cJ[NJL][6], h[NJL][6], invD[NJL], u[NJL];
  float Rl[9], ol[3];     /* rotation of the last link, and O_last relative to the base origin */
  /* contact */
  float sP[NJL][3];       /* S_k . (wrench of unit impulse m propagated to joint k) */
  float P[3][6], K[3][6]; /* base wrench per unit impulse, IA0^-1 P */
  float Lm[6];            /* leg-local 3x3 block (sym): sum_k sP sP^T invD */
  float b[3];             /* target relative velocity (rhs before scaling) */
  float dist;
  int active;
};

SOLO_HD void base_prepare(const BaseState& s, BaseWork& w) {
  quat_to_rot(s.q, w.R);
  mat3T_mulv(w.R, s.w, w.wb);
  mat3T_mulv(w.R, s.v, w.vb);
}

/* Kinematic state carried down a leg while walking outward from the base: rotation of the current link,
 * position O_k of its joint origin relative to the base origin, and the spatial velocity (angular, linear
 * velocity of the point at O_k) of the current link -- all in base axes. */
struct LegKin {
  float R[9], o[3], va[3], vl[3];
};
SOLO_HD void legkin_init(const BaseWork& bw, LegKin& kn) {
  const float I3[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
#pragma unroll
  for (int i = 0; i < 9; i++) kn.R[i] = I3[i];
#pragma unroll
  for (int i = 0; i < 3; i++) { kn.o[i] = 0.f; kn.va[i] = bw.wb[i]; kn.vl[i] = bw.vb[i]; }
}
/* Step through joint k (k is a compile-time constant after unrolling at every call site): r = O_k - O_{k-1},
 * a = joint axis, cJ = velocity-product acceleration v x (a qd, 0); kn ends up describing link k. */
template <int NJL>
SOLO_HD void legkin_joint(const LegConst& lc, int k, float q, float qd, LegKin& kn, float* r, float* a, float* cJ) {
  float* R = kn.R;
  mat3_mulv(R, lc.jo[k], r);
  kn.o[0] += r[0]; kn.o[1] += r[1]; kn.o[2] += r[2];
  cross3_add(kn.va, r, kn.vl);                           /* move the reference point to O_k */
  constexpr int kAxX = 0;
  const int ax = axis_of<NJL>(k);
  a[0] = R[ax]; a[1] = R[3 + ax]; a[2] = R[6 + ax];
  float sn, cs;
  solo_sincos(q, &sn, &cs);
  if (ax == kAxX) { /* R <- R Rx(q): col1' = c col1 + s col2 ; col2' = -s col1 + c col2 */
#pragma unroll
    for (int i = 0; i < 3; i++) {
      float c1 = R[3 * i + 1], c2 = R[3 * i + 2];
      R[3 * i + 1] = cs * c1 + sn * c2;
      R[3 * i + 2] = cs * c2 - sn * c1;
    }
  } else {          /* R <- R Ry(q): col0' = c col0 - s col2 ; col2' = s col0 + c col2 */
#pragma unroll
    for (int i = 0; i < 3; i++) {
      float c0 = R[3 * i + 0], c2 = R[3 * i + 2];
      R[3 * i + 0] = cs * c0 - sn * c2;
      R[3 * i + 2] = sn * c0 + cs * c2;
    }
  }
  /* joint velocity (a qd, 0) and velocity-product acceleration cJ = v x (a qd, 0) */
  float wJ[3] = {a[0] * qd, a[1] * qd, a[2] * qd};
  cross3(kn.va, wJ, cJ);
  cross3(kn.vl, wJ, cJ + 3);
  kn.va[0] += wJ[0]; kn.va[1] += wJ[1]; kn.va[2] += wJ[2];
}
/* Per-link quantities of link k at the kinematic state kn: COM relative to O_k, inertia about the COM in base
 * axes, and the bias wrench pk = v x* (I v) + Bullet link damping, moments about O_k. */
template <int NJL>
SOLO_HD void link_bias(const LegConst& lc, const SimConst& sc, int k, const LegKin& kn, float* com, float* Ic,
                       float* pk) {
  const float* R = kn.R;
  const float* va = kn.va;
  const float* vl = kn.vl;
  mat3_mulv(R, lc.c[k], com);
  {
    const float* I = lc.I[k];
    float T[9];
#pragma unroll
    for (int i = 0; i < 3; i++) {
      T[3 * i + 0] = R[3 * i] * I[0] + R[3 * i + 1] * I[1] + R[3 * i + 2] * I[2];
      T[3 * i + 1] = R[3 * i] * I[1] + R[3 * i + 1] * I[3] + R[3 * i + 2] * I[4];
      T[3 * i + 2] = R[3 * i] * I[2] + R[3 * i + 1] * I[4] + R[3 * i + 2] * I[5];
    }
    Ic[0] = T[0] * R[0] + T[1] * R[1] + T[2] * R[2];
    Ic[1] = T[0] * R[3] + T[1] * R[4] + T[2] * R[5];
    Ic[2] = T[0] * R[6] + T[1] * R[7] + T[2] * R[8];
    Ic[3] = T[3] * R[3] + T[4] * R[4] + T[5] * R[5];
    Ic[4] = T[3] * R[6] + T[4] * R[7] + T[5] * R[8];
    Ic[5] = T[6] * R[6] + T[7] * R[7] + T[8] * R[8];
  }
  /* momentum and velocity-product bias  p = v x* (I v), moments about O_k */
  float vc[3], l[3], nc[3], nO[3];
  cross3(va, com, vc);
  vc[0] += vl[0]; vc[1] += vl[1]; vc[2] += vl[2];
  float m = lc.m[k];
  l[0] = m * vc[0]; l[1] = m * vc[1]; l[2] = m * vc[2];
  sym3_mulv(Ic, va, nc);
  cross3(com, l, nO);
  nO[0] += nc[0]; nO[1] += nc[1]; nO[2] += nc[2];
  cross3(va, nO, pk);
  cross3_add(vl, l, pk);
  cross3(va, l, pk + 3);
  /* Bullet link damping: drag  m v_c (k + k|v_c|)  and  I w (k + k|w|)  per URDF link */
  float wn = solo_sqrt_approx(dot3(va, va));
  float sa = sc.kang + sc.kang * wn;
  if (k < NJL - 1) {
    float sl = sc.klin + sc.klin * solo_sqrt_approx(dot3(vc, vc));
    float f[3] = {l[0] * sl, l[1] * sl, l[2] * sl};
    pk[3] += f[0]; pk[4] += f[1]; pk[5] += f[2];
    cross3_add(com, f, pk);
    pk[0] += nc[0] * sa; pk[1] += nc[1] * sa; pk[2] += nc[2] * sa;
  } else {
    float cb[3], vb2[3], f[3];
    /* lower leg proper */
    mat3_mulv(R, lc.c_own, cb);
    cross3(va, cb, vb2);
    vb2[0] += vl[0]; vb2[1] += vl[1]; vb2[2] += vl[2];
    float sl = lc.m_own * (sc.klin + sc.klin * solo_sqrt_approx(dot3(vb2, vb2)));
    f[0] = vb2[0] * sl; f[1] = vb2[1] * sl; f[2] = vb2[2] * sl;
    pk[3] += f[0]; pk[4] += f[1]; pk[5] += f[2];
    cross3_add(cb, f, pk);
    /* foot */
    mat3_mulv(R, lc.c_foot, cb);
    cross3(va, cb, vb2);
    vb2[0] += vl[0]; vb2[1] += vl[1]; vb2[2] += vl[2];
    sl = lc.m_foot * (sc.klin + sc.klin * solo_sqrt_approx(dot3(vb2, vb2)));
    f[0] = vb2[0] * sl; f[1] = vb2[1] * sl; f[2] = vb2[2] * sl;
    pk[3] += f[0]; pk[4] += f[1]; pk[5] += f[2];
    cross3_add(cb, f, pk);
    /* angular: R Idamp R^T w */
    float wl[3], Iw[3], tw[3];
    mat3T_mulv(R, va, wl);
    sym3_mulv(lc.Idamp, wl, Iw);
    mat3_mulv(R, Iw, tw);
    pk[0] += tw[0] * sa; pk[1] += tw[1] * sa; pk[2] += tw[2] * sa;
  }
}
/* Inward pass over one leg: carry the articulated inertia up the chain, translating it from O_k to O_{k-1}
 * after each joint.  In: ln.ax, ln.r, ln.cJ and the per-link com / Ic / pk.  Out: ln.h, ln.invD, ln.u and the
 * leg's articulated inertia and bias force as seen by the base (about the base origin, base axes). */
template <int NJL>
SOLO_HD void leg_recursion(const LegConst& lc, Lane<NJL>& ln, const float* tau, const float (*pk)[6],
                           const float (*com)[3], const float (*Ic)[6], Sym6& IAleg, float* pAleg) {
  sym6_zero(IAleg);
#pragma unroll
  for (int i = 0; i < 6; i++) pAleg[i] = 0.f;
#pragma unroll
  for (int k = NJL - 1; k >= 0; k--) {
    sym6_add_rigid(IAleg, lc.m[k], com[k], Ic[k]);
#pragma unroll
    for (int i = 0; i < 6; i++) pAleg[i] += pk[k][i];
    const float* a = ln.ax[k];
    float* h = ln.h[k];
    sym3_mulv(IAleg.A, a, h);          /* h = IA (a, 0) */
    mat3T_mulv(IAleg.H, a, h + 3);
    float D = dot3(a, h);
    float invD = solo_rcp(D);
    ln.invD[k] = invD;
    float u = tau[k] - dot3(a, pAleg);
    ln.u[k] = u;
    sym6_rank1_sub(IAleg, h, invD);
    float Ic6[6];
    sym6_mulv(IAleg, ln.cJ[k], Ic6);
    float ud = u * invD;
#pragma unroll
    for (int i = 0; i < 6; i++) pAleg[i] += Ic6[i] + h[i] * ud;
    /* translate to the parent's origin */
    sym6_shift(IAleg, ln.r[k]);
    cross3_add(ln.r[k], pAleg + 3, pAleg);
  }
}

/* Passes 1+2 of the articulated-body algorithm for one leg (outward kinematics and bias
 * forces, then inward articulated inertia).  Result: the leg's articulated inertia and
 * bias force as seen by the base (IAleg, pAleg), about the base origin, base axes. */
template <int NJL>
SOLO_HD void leg_inward(const LegConst& lc, const SimConst& sc, const BaseWork& bw, Lane<NJL>& ln,
                        const float* tau, Sym6& IAleg, float* pAleg) {
  LegKin kn;
  legkin_init(bw, kn);
  float pk[NJL][6], com[NJL][3], Ic[NJL][6];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    legkin_joint<NJL>(lc, k, ln.q[k], ln.qd[k], kn, ln.r[k], ln.ax[k], ln.cJ[k]);
    link_bias<NJL>(lc, sc, k, kn, com[k], Ic[k], pk[k]);
  }
#pragma unroll
  for (int i = 0; i < 9; i++) ln.Rl[i] = kn.R[i];
  ln.ol[0] = kn.o[0]; ln.ol[1] = kn.o[1]; ln.ol[2] = kn.o[2];
  leg_recursion<NJL>(lc, ln, tau, pk, com, Ic, IAleg, pAleg);
}

/* The base body's inertia added to IA0, its angular momentum (base axes) nb and linear momentum l. */
SOLO_HD void base_rigid(float m, const float* I, const BaseWork& bw, Sym6& IA0, float* nb, float* l) {
  const float zero3[3] = {0.f, 0.f, 0.f};
  sym6_add_rigid(IA0, m, zero3, I);
  sym3_mulv(I, bw.wb, nb);
  l[0] = m * bw.vb[0]; l[1] = m * bw.vb[1]; l[2] = m * bw.vb[2];
}

/* Base rigid body: add to the summed leg inertias / bias, factor, solve a0 = -IA0^-1 pA0.
 * dyn: base mass and inertia scaled by dyn->sm (randomised dynamics). */
SOLO_HD void base_solve(const ModelConst& mc, const SimConst& sc, BaseWork& bw, Sym6& IA0,
                        float* pA0, float* a0, const EnvDyn* dyn = nullptr) {
  float nb[3], l[3];
  if (dyn == nullptr) {
    base_rigid(mc.base_m, mc.base_I, bw, IA0, nb, l);
  } else {
    float I[6];
#pragma unroll
    for (int i = 0; i < 6; i++) I[i] = mc.base_I[i] * dyn->sm;
    base_rigid(mc.base_m * dyn->sm, I, bw, IA0, nb, l);
  }
  float sa = sc.kang + sc.kang * solo_sqrt_approx(dot3(bw.wb, bw.wb));
  float sl = sc.klin + sc.klin * solo_sqrt_approx(dot3(bw.vb, bw.vb));
  float pb[6];
  cross3(bw.wb, nb, pb);
  cross3(bw.wb, l, pb + 3);
  pb[0] += nb[0] * sa; pb[1] += nb[1] * sa; pb[2] += nb[2] * sa;
  pb[3] += l[0] * sl; pb[4] += l[1] * sl; pb[5] += l[2] * sl;
#pragma unroll
  for (int i = 0; i < 6; i++) pA0[i] += pb[i];
  ldl6_factor(IA0, bw.F);
#pragma unroll
  for (int i = 0; i < 6; i++) a0[i] = -pA0[i];
  ldl6_solve(bw.F, a0);
}

/* Pass 3: joint accelerations of one leg from the base spatial acceleration. */
template <int NJL>
SOLO_HD void leg_outward(const Lane<NJL>& ln, const float* a0, float* qdd) {
  float a[6];
#pragma unroll
  for (int i = 0; i < 6; i++) a[i] = a0[i];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    cross3_add(a, ln.r[k], a + 3);                   /* reference point -> O_k */
#pragma unroll
    for (int i = 0; i < 6; i++) a[i] += ln.cJ[k][i];
    float qa = (ln.u[k] - dot6(ln.h[k], a)) * ln.invD[k];
    qdd[k] = qa;
    a[0] += ln.ax[k][0] * qa; a[1] += ln.ax[k][1] * qa; a[2] += ln.ax[k][2] * qa;
  }
}

/* World-frame base acceleration from the spatial one: gravity enters here (uniform field:
 * it does not change relative accelerations), and w x v converts the derivative of
 * body-frame velocity coordinates into the classical acceleration of the base origin. */
SOLO_HD void base_world_acc(const SimConst& sc, const BaseWork& bw, const float* a0,
                            float* angacc_w, float* linacc_w) {
  float al[3];
  cross3(bw.wb, bw.vb, al);
  /* gravity in base coordinates = gz * (third row of R) */
  al[0] += a0[3] + sc.gz * bw.R[6];
  al[1] += a0[4] + sc.gz * bw.R[7];
  al[2] += a0[5] + sc.gz * bw.R[8];
  mat3_mulv(bw.R, a0, angacc_w);
  mat3_mulv(bw.R, al, linacc_w);
}

SOLO_HD void base_add_velocity(const SimConst& sc, BaseState& s, const float* dw, const float* dv,
                               float scale) {
#pragma unroll
  for (int i = 0; i < 3; i++) {
    s.w[i] = clampf(s.w[i] + scale * dw[i], -sc.vmax, sc.vmax);
    s.v[i] = clampf(s.v[i] + scale * dv[i], -sc.vmax, sc.vmax);
  }
}

/* Contact geometry of one foot: distance of the collision sphere to the plane (ln.dist, ln.active), the contact
 * point relative to O_last (rc) and the spatial velocity of the last link about O_last with the UPDATED
 * velocities (v6), all in base coordinates.  bw holds the PRE-update rotation (poses do not change between the
 * ABA and the constraint solve), st the POST-update velocity v*. */
template <int NJL>
SOLO_HD void contact_geometry(const LegConst& lc, const ModelConst& mc, const SimConst& sc, const BaseState& st,
                              const BaseWork& bw, Lane<NJL>& ln, float* rc, float* v6) {
  float rfl[3];                                             /* sphere centre relative to O_last */
  mat3_mulv(ln.Rl, lc.foot_ctr, rfl);
  const float nb[3] = {bw.R[6], bw.R[7], bw.R[8]};          /* world z in base coordinates */
  float rf[3] = {ln.ol[0] + rfl[0], ln.ol[1] + rfl[1], ln.ol[2] + rfl[2]};
  float height = st.p[2] + dot3(nb, rf);
  ln.dist = height - mc.foot_r;
  ln.active = ln.dist < sc.margin;
  rc[0] = rfl[0] - mc.foot_r * nb[0]; rc[1] = rfl[1] - mc.foot_r * nb[1]; rc[2] = rfl[2] - mc.foot_r * nb[2];
  /* spatial velocity of the last link about O_last with the updated velocities */
  mat3T_mulv(bw.R, st.w, v6);
  mat3T_mulv(bw.R, st.v, v6 + 3);
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    cross3_add(v6, ln.r[k], v6 + 3);
    v6[0] += ln.ax[k][0] * ln.qd[k]; v6[1] += ln.ax[k][1] * ln.qd[k]; v6[2] += ln.ax[k][2] * ln.qd[k];
  }
}
/* One contact row (m = 0 normal, 1 / 2 the friction directions of btPlaneSpace1((0,0,1)) = (0,-1,0), (1,0,0)):
 * unit impulse along direction m at the contact point, propagated up the leg (sPm[k] = S_k . wrench at joint k)
 * to the base (P), K = IA0^-1 P, and the target relative velocity b. */
template <int NJL>
SOLO_HD void contact_row(const SimConst& sc, const float* R, const Ldl6& F, const float (*ax)[3],
                         const float (*r)[3], const float (*h)[6], const float* invD, const float* rc,
                         const float* v6, float dist, int m, float* sPm, float* P, float* K, float& b) {
  float d[3];
  if (m == 0) { d[0] = R[6]; d[1] = R[7]; d[2] = R[8]; }
  else if (m == 1) { d[0] = -R[3]; d[1] = -R[4]; d[2] = -R[5]; }
  else { d[0] = R[0]; d[1] = R[1]; d[2] = R[2]; }
  float w[6];
  cross3(rc, d, w);
  w[3] = d[0]; w[4] = d[1]; w[5] = d[2];
  float vel = dot6(w, v6);
#pragma unroll
  for (int k = NJL - 1; k >= 0; k--) {
    float s = dot3(ax[k], w);
    sPm[k] = s;
    float g = s * invD[k];
#pragma unroll
    for (int i = 0; i < 6; i++) w[i] -= h[k][i] * g;
    cross3_add(r[k], w + 3, w);                        /* moments about the parent's origin */
  }
#pragma unroll
  for (int i = 0; i < 6; i++) { P[i] = w[i]; K[i] = w[i]; }
  ldl6_solve(F, K);
  if (m == 0) {
    float pen = dist + sc.slop;
    /* speculative contact while separated, ERP push-out while penetrating */
    b = -vel - pen * (pen > 0.f ? sc.inv_dt : sc.erp * sc.inv_dt);
  } else {
    b = -vel;
  }
}
/* leg-local block L = sum_k sP_k sP_k^T invD_k  (xx xy xz yy yz zz over m,n) */
template <int NJL>
SOLO_HD void contact_local_block(Lane<NJL>& ln) {
#pragma unroll
  for (int i = 0; i < 6; i++) ln.Lm[i] = 0.f;
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    float g0 = ln.sP[k][0] * ln.invD[k], g1 = ln.sP[k][1] * ln.invD[k], g2 = ln.sP[k][2] * ln.invD[k];
    ln.Lm[0] += g0 * ln.sP[k][0]; ln.Lm[1] += g0 * ln.sP[k][1]; ln.Lm[2] += g0 * ln.sP[k][2];
    ln.Lm[3] += g1 * ln.sP[k][1]; ln.Lm[4] += g1 * ln.sP[k][2]; ln.Lm[5] += g2 * ln.sP[k][2];
  }
}
/* Contact rows of one foot (the three functions above, one lane doing all of it). */
template <int NJL>
SOLO_HD void contact_setup(const LegConst& lc, const ModelConst& mc, const SimConst& sc,
                           const BaseState& st, const BaseWork& bw, Lane<NJL>& ln) {
  float rc[3], v6[6];
  contact_geometry<NJL>(lc, mc, sc, st, bw, ln, rc, v6);
#pragma unroll
  for (int m = 0; m < 3; m++) {
    float sPm[NJL];
    contact_row<NJL>(sc, bw.R, bw.F, ln.ax, ln.r, ln.h, ln.invD, rc, v6, ln.dist, m, sPm, ln.P[m], ln.K[m], ln.b[m]);
#pragma unroll
    for (int k = 0; k < NJL; k++) ln.sP[k][m] = sPm[k];
  }
  contact_local_block<NJL>(ln);
}

/* ------------------------------------------------------------------ joint-limit rows
 * [3P] PyBullet's URDF importer gives every revolute joint with lower <= upper a
 * btMultiBodyJointLimitConstraint; while the joint position is at or beyond a limit
 * (createConstraintRows: `if (penetration > 0) continue;`) the solver holds a unilateral row on that joint,
 * impulse in [0, maxAppliedImpulse], target velocity erp*|penetration|/dt (no positional part beyond the
 * split-impulse threshold), relaxed BEFORE the contact normals in every sweep.  The kernels carry at most
 * one such row per leg: the most violated joint (first on ties); SoloSimParams.limit_rows_per_leg = 1 makes
 * the oracle do the same. */
template <int NJL>
struct LimitRow {
  float U[NJL];          /* generalized force the unit row impulse puts on joint k of the leg (0 above the joint) */
  float P[6], K[6];      /* base wrench per unit impulse, IA0^-1 P */
  float b;               /* target relative velocity */
  float LL;              /* leg-local diagonal term  sum_k U_k^2 invD_k */
  float Lc[3];           /* leg-local coupling with the foot's contact rows  sum_k U_k sP_k[m] invD_k */
  int active;
};

/* which joint of the leg, if any: dir = +1 at the lower bound, -1 at the upper, pen <= 0 */
template <int NJL>
SOLO_HD bool limit_select(const SimConst& sc, const Lane<NJL>& ln, int& kL, float& dir, float& pen) {
  bool any = false;
  kL = 0; dir = 0.f; pen = 0.f;
  if (!sc.joint_limits) return false;
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    const float lo = ln.q[k] + sc.q_limit, hi = sc.q_limit - ln.q[k];
    /* lower row first, then upper, in joint order; strictly-more-violated replaces */
    if (!(lo > 0.f) && (!any || lo < pen)) { any = true; kL = k; dir = 1.f; pen = lo; }
    if (!(hi > 0.f) && (!any || hi < pen)) { any = true; kL = k; dir = -1.f; pen = hi; }
  }
  return any;
}

/* Row data of the selected joint.  Same propagation as a contact row (contact_setup), with the unit impulse
 * entering as a generalized force on joint kL instead of a wrench at the foot.  kL is a run-time value: every
 * per-joint array is indexed by the unrolled k and selected with predicates, never by kL. */
template <int NJL>
SOLO_HD void limit_setup(const SimConst& sc, const BaseWork& bw, const Lane<NJL>& ln, bool any, int kL, float dir,
                         float pen, LimitRow<NJL>& lr) {
  float w[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float qdL = 0.f;
  lr.LL = 0.f; lr.Lc[0] = lr.Lc[1] = lr.Lc[2] = 0.f;
#pragma unroll
  for (int k = NJL - 1; k >= 0; k--) {
    const bool at = any && (k == kL);
    float s = dot3(ln.ax[k], w) + (at ? dir : 0.f);       /* w is still zero above the joint */
    s = (any && k <= kL) ? s : 0.f;
    lr.U[k] = s;
    qdL = at ? ln.qd[k] : qdL;
    const float g = s * ln.invD[k];
#pragma unroll
    for (int i = 0; i < 6; i++) w[i] -= ln.h[k][i] * g;
    cross3_add(ln.r[k], w + 3, w);                        /* moments about the parent's origin */
    lr.LL += g * s;
#pragma unroll
    for (int m = 0; m < 3; m++) lr.Lc[m] += g * ln.sP[k][m];
  }
#pragma unroll
  for (int i = 0; i < 6; i++) { lr.P[i] = w[i]; lr.K[i] = w[i]; }
  ldl6_solve(bw.F, lr.K);
  const float rel_vel = dir * qdL;
  const float positional = (pen > sc.lim_split_thr) ? -pen * sc.lim_erp * sc.inv_dt : 0.f;
  lr.b = positional - rel_vel;
  lr.active = any ? 1 : 0;
}

/* Global row index of (foot i, direction m): normals first, then friction pairs
 * (the order btMultiBodyConstraintSolver sweeps them). */
SOLO_HD constexpr int row_of(int foot, int m) { return m == 0 ? foot : 4 + 2 * foot + (m - 1); }

/* Rows of the scaled Delassus matrix owned by one foot, built one column block at a time:
 *   A = P^T IA0^-1 P + blockdiag(L),  B[m][c] = A[r_m][c] / A[r_m][r_m],  g0[m] = b[m] / A[r_m][r_m].
 * assemble_block adds the 3x3 block against foot j (Kj = K of foot j, fetched from that lane). */
SOLO_HD constexpr int sym3_idx(int m, int n) { return m == n ? (m == 0 ? 0 : (m == 1 ? 3 : 5)) : (m + n == 1 ? 1 : (m + n == 2 ? 2 : 4)); }
/* `foot` (this lane's leg) is a run-time value and j a compile-time one: the own-foot block is picked
 * with selects, never by indexing `rows` with `foot`, so the rows stay in registers. */
template <int NJL>
SOLO_HD void assemble_block(const Lane<NJL>& ln, int foot, int j, const float Kj[3][6], float rows[3][kRows]) {
  const bool own = (j == foot);
#pragma unroll
  for (int m = 0; m < 3; m++) {
#pragma unroll
    for (int n = 0; n < 3; n++) rows[m][row_of(j, n)] = dot6(ln.P[m], Kj[n]) + (own ? ln.Lm[sym3_idx(m, n)] : 0.f);
  }
}

/* Projected Gauss-Seidel state of one foot (= one lane): its three rows of B, and for those
 * rows  g[m] = lambda[m] + (rhs[m] - sum_c A[m][c] lambda[c]) / A[m][m],  the value the row would
 * take if relaxed now.  Relaxing row r anywhere changes g[m] by -B[m][r] * dlambda_r, so a sweep is:
 * owner clamps its g, the impulse change is broadcast to the env's four lanes, every lane applies
 * three FMAs.  Sweep order and projections restate btMultiBodyConstraintSolver::solveSingleIteration
 * [3P]: all normal rows (lambda >= 0), then per contact the friction pair, both candidates taken from
 * the same state and projected radially onto the circle of radius mu*lambda_n
 * (resolveConeFrictionConstraintRows; its atan2/sin/cos == the x/|x| scaling used here), or row by
 * row onto [-mu lambda_n, mu lambda_n] when cone friction is off.  No warm start.  The sweep loop
 * ends after solver_iters iterations or once the largest squared velocity residual
 * (dlambda * A[r][r])^2 of an iteration is <= solver_residual_threshold. */
template <int NR, int NC>
struct PgsLaneT {
  float B[NR][NC];
  float g[NR], lam[NR], diag[NR];
  /* The clamped rows (normal row 0, limit row 3) keep h = g - lambda in g[], the distance of the candidate from the
   * current impulse, so that the impulse CHANGE is one min/max of h against pre-negated bounds -- max(h, -lambda),
   * and min(., max - lambda) for a limit row -- instead of clamp-then-subtract: one dependent operation less per
   * row relaxation on the sweep's chain (profiles/r2_experiments.txt item 11).  Relaxing the row
   * itself moves h by -dlambda, which rides in the apply step as B[own row][own column] = 1. */
  float nl0;        /* -lambda of the normal row */
  float nl3, ul3;   /* limit row: -lambda and max_impulse - lambda */
};
typedef PgsLaneT<3, kRows> PgsLane;
/* with joint-limit rows: a fourth row per lane (the leg's limit row), columns 12..15 = the four limit rows */
constexpr int kRowsL = kRows + 4;
typedef PgsLaneT<4, kRowsL> PgsLane4;
SOLO_HD constexpr int limit_col(int leg) { return kRows + leg; }
template <int NJL>
SOLO_HD void pgs_lane_init(const Lane<NJL>& ln, int foot, float rows[3][kRows], unsigned active_mask,
                           PgsLane& pl) {
#pragma unroll
  for (int m = 0; m < 3; m++) {
    float d = 1.0f;
#pragma unroll
    for (int j = 0; j < 4; j++) d = (j == foot) ? rows[m][row_of(j, m)] : d;
    const float invd = ln.active ? solo_rcp(d) : 0.f;
    pl.diag[m] = ln.active ? d : 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
      for (int n = 0; n < 3; n++) {
        const int c = row_of(j, n);
        const bool own_diag = (j == foot) && (n == m);
        pl.B[m][c] = (((active_mask >> j) & 1u) && !own_diag) ? -(rows[m][c] * invd) : 0.f;   /* stored negated */
        if (own_diag && m == 0) pl.B[m][c] = ln.active ? -1.0f : 0.f;    /* h-row: see PgsLaneT */
      }
    }
    pl.g[m] = ln.b[m] * invd;
    pl.lam[m] = 0.f;
  }
  pl.nl0 = 0.f; pl.nl3 = 0.f; pl.ul3 = 0.f;
}
/* candidate for this lane's normal row: new value, impulse change, velocity residual */
template <class PL>
SOLO_HD void pgs_normal_candidate(const PL& pl, float& nv, float& d, float& rv) {
  d = fmaxf(pl.g[0], pl.nl0);          /* g[0] = candidate - lambda (h-row): lambda + d = max(candidate, 0) */
  nv = pl.lam[0] + d;
  rv = d * pl.diag[0];
}
/* the owner of the row takes the new impulse (the row's h moves in the apply step) */
template <class PL>
SOLO_HD void pgs_normal_commit(PL& pl, float nv) {
  pl.lam[0] = nv;
  pl.nl0 = -nv;
}
/* candidates of one friction pair (cone) from the state of its two rows: candidates sA, sB, impulses lA, lB,
 * diagonals dgA, dgB; lamn = the foot's normal impulse */
SOLO_HD void cone_candidate(float mu, float lamn, float sA, float sB, float lA, float lB, float dgA, float dgB,
                            float& nA, float& nB, float& dA, float& dB, float& rv) {
  /* Bullet clamps sA to +-|lim sin(atan2(sA,sB))| and sB to +-|lim cos(.)|, i.e. it scales the pair
   * (sA,sB) back onto the circle of radius lim when it lies outside: (sA,sB) * min(1, lim/|s|).
   * Written for the shortest dependent chain from g to the impulse change: the 1e-30 guard rides in
   * the first FMA instead of a max, and d = s*scale - lambda is one FMA instead of multiply + subtract. */
  const float lim = mu * lamn;
  const float n2 = fmaf(sB, sB, fmaf(sA, sA, 1e-30f));
  const float sc = fminf(lim * solo_rsqrt(n2), 1.0f);
  nA = sA * sc;
  nB = sB * sc;
  dA = fmaf(sA, sc, -lA);
  dB = fmaf(sB, sc, -lB);
  rv = dA * dgA + dB * dgB;
}
/* candidate of one friction row (pyramid): candidate s, impulse l, diagonal dg */
SOLO_HD void pyramid_candidate(float mu, float lamn, float s, float l, float dg, float& nv, float& d, float& rv) {
  const float lim = mu * lamn;
  nv = clampf(s, -lim, lim);
  d = nv - l;
  rv = d * dg;
}
/* candidates for this lane's friction pair (cone) */
template <class PL>
SOLO_HD void pgs_cone_candidate(const PL& pl, float mu, float& nA, float& nB, float& dA, float& dB,
                                float& rv) {
  cone_candidate(mu, pl.lam[0], pl.g[1], pl.g[2], pl.lam[1], pl.lam[2], pl.diag[1], pl.diag[2], nA, nB, dA, dB, rv);
}
/* candidate for one friction row (pyramid), q = 0/1 */
template <class PL>
SOLO_HD void pgs_pyramid_candidate(const PL& pl, float mu, int q, float& nv, float& d, float& rv) {
  pyramid_candidate(mu, pl.lam[0], pl.g[1 + q], pl.lam[1 + q], pl.diag[1 + q], nv, d, rv);
}
/* Apply the impulse change d of global row `col` to this lane's rows: g[m] += (-B[m][col]) d, B being stored negated.
 * On the GPU two rows go through ONE packed FFMA2 (sm_100 fma.rn.f32x2, the scalar d broadcast by the instruction's
 * .F32 operand form, no packing moves): the sweep is sensitive to its instruction count -- a lone warp issues a
 * three-register FFMA every second cycle -- and the applies are 64 of its ~146 instructions
 * (profiles/r2_experiments.txt items 12-13).  Each half is an ordinary fused multiply-add: same bits as two FFMAs. */
SOLO_HD void pgs_fma_pair(float& g0, float& g1, float b0, float b1, float d) {
#if defined(__CUDA_ARCH__)
  unsigned long long rg, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(rg) : "f"(g0), "f"(g1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b0), "f"(b1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(rd) : "f"(d));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(rg) : "l"(rb), "l"(rd));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(g0), "=f"(g1) : "l"(rg));
#else
  g0 += b0 * d; g1 += b1 * d;
#endif
}
SOLO_HD void pgs_apply(PgsLane& pl, int col, float d) {
  pgs_fma_pair(pl.g[0], pl.g[1], pl.B[0][col], pl.B[1][col], d);
  pl.g[2] += pl.B[2][col] * d;
}
SOLO_HD void pgs_apply(PgsLane4& pl, int col, float d) {
  pgs_fma_pair(pl.g[0], pl.g[1], pl.B[0][col], pl.B[1][col], d);
  pgs_fma_pair(pl.g[2], pl.g[3], pl.B[2][col], pl.B[3][col], d);
}
/* candidate for this lane's joint-limit row: impulse in [0, max], otherwise like a normal row */
SOLO_HD void pgs_limit_candidate(const PgsLane4& pl, float max_impulse, float& nv, float& d, float& rv) {
  (void)max_impulse;
  d = fminf(fmaxf(pl.g[3], pl.nl3), pl.ul3);   /* h-row: lambda + d = min(max(candidate, 0), max_impulse) */
  nv = pl.lam[3] + d;
  rv = d * pl.diag[3];
}
SOLO_HD void pgs_limit_commit(PgsLane4& pl, float max_impulse, float nv) {
  pl.lam[3] = nv;
  pl.nl3 = -nv;
  pl.ul3 = max_impulse - nv;
}

/* Four-row versions of assemble_block / pgs_lane_init: row 3 / column 12+j is the limit row of leg j.
 * Kj[n] (n < 3) and KLj are K of the contact rows and of the limit row of lane j. */
template <int NJL>
SOLO_HD void assemble_block4(const Lane<NJL>& ln, const LimitRow<NJL>& lr, int foot, int j, const float Kj[3][6],
                             const float* KLj, bool limit_col_on, float rows[4][kRowsL]) {
  const bool own = (j == foot);
  /* the four rows of this lane (three contact rows, the limit row) against one column at a time, two rows per
   * packed dot product */
#pragma unroll
  for (int n = 0; n < 3; n++) {
    float d0, d1, d2, d3;
    dot6_pair(ln.P[0], ln.P[1], Kj[n], d0, d1);
    dot6_pair(ln.P[2], lr.P, Kj[n], d2, d3);
    rows[0][row_of(j, n)] = d0 + (own ? ln.Lm[sym3_idx(0, n)] : 0.f);
    rows[1][row_of(j, n)] = d1 + (own ? ln.Lm[sym3_idx(1, n)] : 0.f);
    rows[2][row_of(j, n)] = d2 + (own ? ln.Lm[sym3_idx(2, n)] : 0.f);
    rows[3][row_of(j, n)] = d3 + (own ? lr.Lc[n] : 0.f);
  }
  if (limit_col_on) {   /* uniform: some env of the warp has a limit row on leg j */
    float d0, d1, d2, d3;
    dot6_pair(ln.P[0], ln.P[1], KLj, d0, d1);
    dot6_pair(ln.P[2], lr.P, KLj, d2, d3);
    rows[0][limit_col(j)] = d0 + (own ? lr.Lc[0] : 0.f);
    rows[1][limit_col(j)] = d1 + (own ? lr.Lc[1] : 0.f);
    rows[2][limit_col(j)] = d2 + (own ? lr.Lc[2] : 0.f);
    rows[3][limit_col(j)] = d3 + (own ? lr.LL : 0.f);
  } else {
#pragma unroll
    for (int m = 0; m < 4; m++) rows[m][limit_col(j)] = 0.f;
  }
}
template <int NJL>
SOLO_HD void pgs_lane_init4(const Lane<NJL>& ln, const LimitRow<NJL>& lr, int foot, float rows[4][kRowsL],
                            unsigned active_mask, unsigned limit_mask, float max_impulse, PgsLane4& pl) {
#pragma unroll
  for (int m = 0; m < 4; m++) {
    const bool row_on = (m < 3) ? (ln.active != 0) : (lr.active != 0);
    float d = 1.0f;
#pragma unroll
    for (int j = 0; j < 4; j++) d = (j == foot) ? rows[m][m < 3 ? row_of(j, m) : limit_col(j)] : d;
    const float invd = row_on ? solo_rcp(d) : 0.f;
    pl.diag[m] = row_on ? d : 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++) {
#pragma unroll
      for (int n = 0; n < 4; n++) {
        const int c = (n < 3) ? row_of(j, n) : limit_col(j);
        const bool col_on = (n < 3) ? (((active_mask >> j) & 1u) != 0) : (((limit_mask >> j) & 1u) != 0);
        const bool own_diag = (j == foot) && (n == m);
        pl.B[m][c] = (col_on && !own_diag) ? -(rows[m][c] * invd) : 0.f;         /* stored negated */
        if (own_diag && (m == 0 || m == 3)) pl.B[m][c] = row_on ? -1.0f : 0.f;  /* h-rows: see PgsLaneT */
      }
    }
    pl.g[m] = ((m < 3) ? ln.b[m] : lr.b) * invd;
    pl.lam[m] = 0.f;
  }
  pl.nl0 = 0.f; pl.nl3 = 0.f; pl.ul3 = max_impulse;
}

/* Wrench on the base produced by this foot's impulses, already multiplied by IA0^-1:
 * dv0_part = K lambda (sum over feet = base velocity change, base coordinates). */
template <int NJL>
SOLO_HD void impulse_base_part(const Lane<NJL>& ln, const float* lam3, float* dv0_part) {
#pragma unroll
  for (int i = 0; i < 6; i++)
    dv0_part[i] = ln.K[0][i] * lam3[0] + ln.K[1][i] * lam3[1] + ln.K[2][i] * lam3[2];
}

/* Joint velocity change of one leg for its own impulses and the base velocity change. */
template <int NJL>
SOLO_HD void impulse_leg(Lane<NJL>& ln, const SimConst& sc, const float* lam3, const float* dv0) {
  float a[6];
#pragma unroll
  for (int i = 0; i < 6; i++) a[i] = dv0[i];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    cross3_add(a, ln.r[k], a + 3);
    float us = ln.sP[k][0] * lam3[0] + ln.sP[k][1] * lam3[1] + ln.sP[k][2] * lam3[2];
    float dq = (us - dot6(ln.h[k], a)) * ln.invD[k];
    a[0] += ln.ax[k][0] * dq; a[1] += ln.ax[k][1] * dq; a[2] += ln.ax[k][2] * dq;
    ln.qd[k] = clampf(ln.qd[k] + dq, -sc.vmax, sc.vmax);
  }
}

/* Forward kinematics of one leg: centre of the foot collision sphere in base coordinates
 * (the kinematic part of leg_inward, for the feet-position query of the gait envs). */
template <int NJL>
SOLO_HD void leg_foot_center(const LegConst& lc, const float* q, float* out) {
  float R[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
  float o[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    float r[3];
    mat3_mulv(R, lc.jo[k], r);
    o[0] += r[0]; o[1] += r[1]; o[2] += r[2];
    float sn, cs;
    solo_sincos(q[k], &sn, &cs);
    if (axis_of<NJL>(k) == 0) {
#pragma unroll
      for (int i = 0; i < 3; i++) {
        float c1 = R[3 * i + 1], c2 = R[3 * i + 2];
        R[3 * i + 1] = cs * c1 + sn * c2;
        R[3 * i + 2] = cs * c2 - sn * c1;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 3; i++) {
        float c0 = R[3 * i + 0], c2 = R[3 * i + 2];
        R[3 * i + 0] = cs * c0 - sn * c2;
        R[3 * i + 2] = sn * c0 + cs * c2;
      }
    }
  }
  float f[3];
  mat3_mulv(R, lc.foot_ctr, f);
  out[0] = o[0] + f[0]; out[1] = o[1] + f[1]; out[2] = o[2] + f[2];
}

/* Joint-level PD + feed-forward actuator of the gait envs' simulator ([3P] PyBulletSimulator.SendCommand
 * of LAAS quadruped-reactive-walking, the surface baseControlEnv.py:256-270 drives):
 * tau = P (q_des - q) + D (v_des - v) + tau_ff, saturated at the motor limit. */
SOLO_HD float actuator_torque(const SimConst& sc, float q, float qd, float q_des, float v_des, float P, float D,
                              float tau_ff) {
  return clampf(P * (q_des - q) + D * (v_des - qd) + tau_ff, -sc.max_torque, sc.max_torque);
}

/* the same two steps when the leg also carries a joint-limit impulse lamL */
template <int NJL>
SOLO_HD void impulse_base_part4(const Lane<NJL>& ln, const LimitRow<NJL>& lr, const float* lam4, float* dv0_part) {
#pragma unroll
  for (int i = 0; i < 6; i++)
    dv0_part[i] = ln.K[0][i] * lam4[0] + ln.K[1][i] * lam4[1] + ln.K[2][i] * lam4[2] + lr.K[i] * lam4[3];
}
template <int NJL>
SOLO_HD void impulse_leg4(Lane<NJL>& ln, const LimitRow<NJL>& lr, const SimConst& sc, const float* lam4,
                          const float* dv0) {
  float a[6];
#pragma unroll
  for (int i = 0; i < 6; i++) a[i] = dv0[i];
#pragma unroll
  for (int k = 0; k < NJL; k++) {
    cross3_add(a, ln.r[k], a + 3);
    float us = ln.sP[k][0] * lam4[0] + ln.sP[k][1] * lam4[1] + ln.sP[k][2] * lam4[2] + lr.U[k] * lam4[3];
    float dq = (us - dot6(ln.h[k], a)) * ln.invD[k];
    a[0] += ln.ax[k][0] * dq; a[1] += ln.ax[k][1] * dq; a[2] += ln.ax[k][2] * dq;
    ln.qd[k] = clampf(ln.qd[k] + dq, -sc.vmax, sc.vmax);
  }
}

/* Semi-implicit Euler position update ([3P] btMultiBody::stepPositionsMultiDof). */
SOLO_HD void integrate_base(const SimConst& sc, BaseState& s) {
#pragma unroll
  for (int i = 0; i < 3; i++) s.p[i] += sc.dt * s.v[i];
  /* rotation by w dt as the quaternion (w sin(ha)/|w|, cos(ha)), ha = |w| dt / 2 <= 0.36 (|w_i| <= 100 rad/s,
   * dt <= 1/240): even Taylor polynomials in ha^2 are exact to 1e-8 there, need no |w| and no division */
  const float h2 = 0.25f * sc.dt * sc.dt * dot3(s.w, s.w);
  const float sinc = 1.0f + h2 * (-1.0f / 6.0f + h2 * (1.0f / 120.0f + h2 * (-1.0f / 5040.0f + h2 * (1.0f / 362880.0f))));
  const float cs = 1.0f + h2 * (-0.5f + h2 * (1.0f / 24.0f + h2 * (-1.0f / 720.0f + h2 * (1.0f / 40320.0f))));
  const float k = 0.5f * sc.dt * sinc;
  float dx = s.w[0] * k, dy = s.w[1] * k, dz = s.w[2] * k, dw = cs;
  float x = s.q[0], y = s.q[1], z = s.q[2], w = s.q[3];
  float nx = dw * x + dx * w + dy * z - dz * y;
  float ny = dw * y - dx * z + dy * w + dz * x;
  float nz = dw * z + dx * y - dy * x + dz * w;
  float nw = dw * w - dx * x - dy * y - dz * z;
  float inv = solo_rsqrt(nx * nx + ny * ny + nz * nz + nw * nw);
  s.q[0] = nx * inv; s.q[1] = ny * inv; s.q[2] = nz * inv; s.q[3] = nw * inv;
}

/* ------------------------------------------------------------------ env arithmetic */
/* [3P] p.getEulerFromQuaternion = btQuaternion::getEulerZYX -> roll, pitch, yaw */
SOLO_HD void quat_to_euler(const float* q, float* rpy) {
  const float kHalfPi = 1.57079632679489661923f;
  float x = q[0], y = q[1], z = q[2], w = q[3];
  float sqx = x * x, sqy = y * y, sqz = z * z, sqw = w * w;
  float sarg = -2.f * (x * z - w * y);
  if (sarg <= -0.99999f) {
    rpy[1] = -kHalfPi; rpy[0] = 0.f; rpy[2] = 2.f * atan2f(x, -y);
  } else if (sarg >= 0.99999f) {
    rpy[1] = kHalfPi; rpy[0] = 0.f; rpy[2] = 2.f * atan2f(-x, y);
  } else {
    rpy[1] = asinf(sarg);
    rpy[0] = atan2f(2.f * (y * z + w * x), sqw - sqx - sqy + sqz);
    rpy[2] = atan2f(2.f * (x * y + w * z), sqw + sqx - sqy - sqz);
  }
}
/* solo.py:206: (e % 2*pi) / (2*pi) == ((e mod 2) * pi) / (2 pi) with Python's floor-mod (SURVEY F6) */
SOLO_HD float euler_obs(float e) {
  float r = fmodf(e, 2.0f);
  if (r < 0.f) r += 2.0f;
  return r * 0.5f;
}
/* solo.py:224-259 + controllers/PD.py:3-10 for one joint */
SOLO_HD float action_to_torque(const SimConst& sc, float a, float q, float qd, float kp, float kd) {
  float ac = clampf(a, -1.f, 1.f);
  if (sc.control == 0) return ac * sc.max_torque;
  float t = kp * (ac * sc.q_limit - q) - kd * qd;
  return clampf(t, -sc.max_torque, sc.max_torque);
}

/* Philox4x32-10, counter = (env id lo, env id hi, episode, draw), key = seed */
SOLO_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
SOLO_HD void philox4x32_10(uint32_t* c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    uint32_t h0 = mulhi32(0xD2511F53u, c[0]), l0 = 0xD2511F53u * c[0];
    uint32_t h1 = mulhi32(0xCD9E8D57u, c[2]), l1 = 0xCD9E8D57u * c[2];
    uint32_t n0 = h1 ^ c[1] ^ k0, n2 = h0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = l1; c[2] = n2; c[3] = l0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
SOLO_HD float u01(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }
/* solo.py:325-330 */
SOLO_HD void sample_goal(const uint32_t* w, float goal_radius, float* g) {
  float gx = 1.0f + (goal_radius - 1.0f) * u01(w[1]);
  float gy = 1.0f + (goal_radius - 1.0f) * u01(w[2]);
  g[0] = (w[3] & 1u) ? gx : -gx;
  g[1] = (w[3] & 2u) ? gy : -gy;
}

}  // namespace solo

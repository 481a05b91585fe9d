// Articulated-body form of the step: the same linear system the reference solves with
// the assembled matrices,
//     Z q'+ = M q'/dt + g + J^T f ,   Z = M/dt + B + N                   (core.py:813-818, 975-976)
// solved WITHOUT assembling M, N, B or Z, in O(ndof) per right-hand side.
//
// Derivation (each identity is checked against the real reference by the parity tests).
// Body Jacobians obey  J_c = X_c J_p (+ own columns S_c),  X_c = Ad(H_pc^-1), and the
// reference's  dJ_c = dAd_cp J_p + X_c dJ_p (+ own columns dS_c)  (core.py:1309-1313) with
//     dAd_cp = Ad_cn Ad_nr adjacency(-Ad_nr T_nr) Ad_rp = adjacency(tau_c) X_c ,
//     tau_c  = -Ad_cn Ad_nr Ad_nr T_nr                                  (rigidmotion.py:49-75).
// Summing along a root path gives, with theta_c = X_c theta_p + tau_c,
//     dJ_b[:,k] = adjacency(theta_b) J_b[:,k] + X_(b<-c_k) s^_k ,  s^_k = ds_k - adjacency(theta_(c_k)) s_k
// so that with  Jh_b[:,k] = X_(b<-c_k) s^_k  (a second "Jacobian" with the same recursion)
//     Z = sum_b J_b^T ( A_b J_b + M_b Jh_b ) ,   A_b = M_b/dt + B_b + N_b + M_b adjacency(theta_b)
// (N_b from core.py:1276-1288).  For a vector x the body quantities V_b = J_b x, Vh_b = Jh_b x
// follow  V_c = X_c V_p + S_c x_c,  Vh_c = X_c Vh_p + S^_c x_c,  and  (Z x)_k = s_k^T F_(c_k) with
// F_b = A_b V_b + M_b Vh_b + sum_children X^T F.  Eliminating the dofs leaf-to-root, one
// scalar dof at a time (exact Gaussian elimination, no fill-in), keeps F of the form
//     F_b = IA_b V_b + IM_b Vh_b + beta_b :
//     U_k = IA s_k + IM s^_k ,  d_k = s_k^T U_k ,  x_k = (tau_k - s_k^T(IA V + IM Vh + beta)) / d_k
//     IA <- IA - U_k (s_k^T IA)/d_k ,  IM <- IM - U_k (s_k^T IM)/d_k ,  beta <- beta + U_k u_k
//     parent:  IA_p += X^T IA X ,  IM_p += X^T IM X ,  beta_p += X^T beta .
// Right-hand sides are generalized forces tau_k plus body wrenches w_b (beta_b starts at -w_b):
// the free motion uses w_b = M_b (T_b/dt + gravity_b)  (M q' = sum J_b^T M_b T_b,
// controllers.py:43-60), the constraint generators use unit wrenches on the bodies that
// carry constraint frames, and the final velocity uses the Gauss-Seidel wrenches.
//
// One world per lane; scratch arrays are tiled [W/32][elem][32] (each access of a warp is one
// 256-byte segment).
#pragma once
#include "arb_constraints.cuh"
#include "arb_joints.cuh"
#include "arb_math.cuh"
#include "arb_types.h"

// Addressing.  FT = fused scratch: tile layout [W/32][elem][32] reached through per-thread
// pre-offset pointers (fused_tile_view, arb_fused.cuh), so an element index costs no 64-bit
// arithmetic -- with a compile-time index the load is one LDG with an immediate offset.
// ST = caller-owned state arrays, [elem][W] (the ABI layout of include/arboris_b200.h).
#define FT(ptr, idx) (ptr)[(idx) * ARB_TILE]
#define ST(ptr, idx) (ptr)[(int64_t)(idx) * b.W + w]
// State reads.  With sorted worlds (arb_fused.cu) the 32 lanes of a warp read 32 different
// sectors: do not let them allocate in L1, which the stages use as the landing zone of their
// scratch prefetches.
ARB_D double arb_ld_state(const double* p) {
#ifdef __CUDA_ARCH__
  double v;
  asm volatile("ld.global.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
#else
  return *p;
#endif
}
#define ST_LD(ptr, idx) arb_ld_state(&ST(ptr, idx))

// y = X^T x for a wrench x = [m; f], X = Ad(H^-1):  [R m + p x (R f) ; R f]
ARB_HD void wrench_up(const Se3& h, const double* x, double* y) {
  double rm[3], rf[3], c[3];
  m3_mulv(h.R, x, rm);
  m3_mulv(h.R, x + 3, rf);
  cross3(h.p, rf, c);
  y[0] = rm[0] + c[0]; y[1] = rm[1] + c[1]; y[2] = rm[2] + c[2];
  y[3] = rf[0]; y[4] = rf[1]; y[5] = rf[2];
}
// A <- X^T A X  (6x6 row-major), X = Ad(H^-1)
ARB_HD void congruence_up(const Se3& h, double* A) {
#pragma unroll
  for (int r = 0; r < 6; ++r) {  // rows:  row_r(A X) = (X^T row_r(A)^T)^T
    double y[6];
    wrench_up(h, A + 6 * r, y);
#pragma unroll
    for (int i = 0; i < 6; ++i) A[6 * r + i] = y[i];
  }
#pragma unroll
  for (int c = 0; c < 6; ++c) {  // columns
    double x[6], y[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) x[i] = A[6 * i + c];
    wrench_up(h, x, y);
#pragma unroll
    for (int i = 0; i < 6; ++i) A[6 * i + c] = y[i];
  }
}
// y = adjacency(t) x = [w x xw ; v x xw + w x xv]      (twistvector.py:26-33)
ARB_HD void adj_apply(const double* t, const double* x, double* y) {
  double a[3], b2[3], c[3];
  cross3(t, x, a);
  cross3(t + 3, x, b2);
  cross3(t, x + 3, c);
  y[0] = a[0]; y[1] = a[1]; y[2] = a[2];
  y[3] = b2[0] + c[0]; y[4] = b2[1] + c[1]; y[5] = b2[2] + c[2];
}

ARB_D void load_se3(const double* arr, int j, Se3& h) {
#pragma unroll
  for (int i = 0; i < 9; ++i) h.R[i] = FT(arr, j * 12 + i);
#pragma unroll
  for (int i = 0; i < 3; ++i) h.p[i] = FT(arr, j * 12 + 9 + i);
}
ARB_D void store_se3(double* arr, int j, const Se3& h) {
#pragma unroll
  for (int i = 0; i < 9; ++i) FT(arr, j * 12 + i) = h.R[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) FT(arr, j * 12 + 9 + i) = h.p[i];
}

// L1 prefetch of one 8-byte element per lane (a 256-byte row per warp); no-op on the host.
// The passes below walk the joints in a fixed order and every operand of joint j was written
// long before (by another pass): asking for the next joint's rows while working on this one
// hides most of the DRAM / L2 latency that the 8 resident warps per SM cannot.
#ifndef ARB_PREFETCH_MODE
#define ARB_PREFETCH_MODE 1     /* 0: none, 1: into L1, 2: into L2 only (A/B builds) */
#endif
ARB_D void arb_prefetch(const double* p) {
#if defined(__CUDA_ARCH__) && ARB_PREFETCH_MODE == 1
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
#elif defined(__CUDA_ARCH__) && ARB_PREFETCH_MODE == 2
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#elif defined(__CUDA_ARCH__) && ARB_PREFETCH_MODE == 3
  // prefetch.global.L1 does not allocate in the L1 on sm_100a (profiles/micro/prefetch_probe.cu: the
  // load that follows takes 503 cycles, an L2 hit; 892 cold; 46 after a real load).  An asynchronous
  // copy through the L1 does (cp.async.ca: 46 cycles afterwards) and holds no register either: the 8
  // bytes go to a per-CTA dump row of shared memory that nobody reads.
  __shared__ double arb_prefetch_dump[32];
  const unsigned d = (unsigned)__cvta_generic_to_shared(&arb_prefetch_dump[threadIdx.x & 31u]);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(p));
#endif
}
// the asynchronous-copy form whatever ARB_PREFETCH_MODE says (device only)
#ifdef __CUDACC__
__device__ __forceinline__ void arb_prefetch_l1(const double* p) {
  __shared__ double arb_prefetch_dump2[32];
  const unsigned d = (unsigned)__cvta_generic_to_shared(&arb_prefetch_dump2[threadIdx.x & 31u]);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(p));
}
#endif
template <int N>
ARB_D void arb_prefetch_rows(const double* p) {
#pragma unroll
  for (int i = 0; i < N; ++i) arb_prefetch(p + i * ARB_TILE);
}
// Rows of the scratch that were just read for the LAST time before they are written again (the
// children's slots of the factorisation, the (V, V^) a body hands to its children): tell the L2 to
// drop them instead of writing them back to HBM (discard.global.L2, 128 bytes per instruction:
// lanes 0 and 16 cover the 256-byte row of the warp's 32 worlds).  The barrier orders the other
// lanes' loads of the row before the discard.  Contents are undefined afterwards, until rewritten.
#ifndef ARB_DISCARD
#define ARB_DISCARD 1
#endif
template <int N>
ARB_D void arb_discard_rows(const double* p) {
#if defined(__CUDA_ARCH__) && ARB_DISCARD
  __syncwarp(__activemask());
  if ((threadIdx.x & 15) == 0) {
#pragma unroll
    for (int i = 0; i < N; ++i) asm volatile("discard.global.L2 [%0], 128;" ::"l"(p + i * ARB_TILE) : "memory");
  }
#endif
}
// per-dof rows of joint j in the four arrays a0..a3 (6 rows per dof each)
ARB_D void artic_prefetch_dofs(const DevModel& m, int j, const double* a0, const double* a1,
                               const double* a2, const double* a3) {
  const int nd = arb_joint_ndof(m.jtype[j]);
  const int off = m.jdof[j] * (6 * ARB_TILE);
  for (int c = 0; c < nd; ++c) {
    const int o = off + c * (6 * ARB_TILE);
    arb_prefetch_rows<6>(a0 + o);
    arb_prefetch_rows<6>(a1 + o);
    if (a2) arb_prefetch_rows<6>(a2 + o);
    if (a3) arb_prefetch_rows<6>(a3 + o);
  }
}

// ---------------------------------------------------------------------------------------
// root-to-leaf pass: body poses and twists (core.py:1295-1308), theta, X, s, s^
#ifndef ARTIC_KIN_PRELOAD
#define ARTIC_KIN_PRELOAD 1     /* the next joint's coordinates are requested before this joint's arithmetic (A/B builds: 0) */
#endif
ARB_D void artic_kinematics(const DevModel& m, const DevBatch& b, int64_t w) {
#if ARTIC_KIN_PRELOAD
  // The state is read once, from HBM, joint after joint: ask for the NEXT joint's coordinates and
  // velocities (at most three each, except for a free joint) before this joint's arithmetic, so that
  // their latency is not paid at the head of every iteration (ncu: 6 % of the stage's stall samples).
  double qn[3] = {0., 0., 0.}, dqn[3] = {0., 0., 0.};
  bool pre = false;
#endif
  for (int j = 0; j < m.nj; ++j) {
    const int type = m.jtype[j];
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(type);
    const int dof = m.jdof[j];
    double q[16], dq[6];
#if ARTIC_KIN_PRELOAD
    if (pre) {
#pragma unroll
      for (int i = 0; i < 3; ++i) { q[i] = qn[i]; dq[i] = dqn[i]; }
    } else
#endif
    {
      for (int i = 0; i < arb_joint_ngpos(type); ++i) q[i] = ST_LD(b.gpos, m.jgpos[j] + i);
      for (int i = 0; i < nd; ++i) dq[i] = ST_LD(b.gvel, dof + i);
    }
#if ARTIC_KIN_PRELOAD
    pre = false;
    if (j + 1 < m.nj && m.jtype[j + 1] != ARB_JOINT_FREE) {
      const int tn = m.jtype[j + 1], gn = m.jgpos[j + 1], dn = m.jdof[j + 1];
      const int ngn = arb_joint_ngpos(tn), ndn = arb_joint_ndof(tn);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (i < ngn) qn[i] = ST_LD(b.gpos, gn + i);
        if (i < ndn) dqn[i] = ST_LD(b.gvel, dn + i);
      }
      pre = true;
    }
#endif
    JointKin k;
    joint_kinematics(type, q, dq, k);
    const bool ident = m.hcn_ident[j] != 0;
    Se3 Hpr, Hcn, Hpc, Hgc, t0;
    load_se3_const(m.Hpr, j, Hpr);
    se3_mul(Hpr, k.H, t0);
    if (ident) {
      Hpc = t0;
      se3_identity(Hcn);
    } else {
      Se3 HcnInv;
      load_se3_const(m.HcnInv, j, HcnInv);
      load_se3_const(m.Hcn, j, Hcn);
      se3_mul(t0, HcnInv, Hpc);
    }
    double Tp[6], thp[6];
    if (par == 0) {
      Hgc = Hpc;
#pragma unroll
      for (int i = 0; i < 6; ++i) { Tp[i] = 0.; thp[i] = 0.; }
    } else {
      Se3 Hgp;
      load_se3(b.fpose, par - 1, Hgp);
      se3_mul(Hgp, Hpc, Hgc);
#pragma unroll
      for (int i = 0; i < 6; ++i) { Tp[i] = FT(b.atw, (par - 1) * 6 + i); thp[i] = FT(b.ath, (par - 1) * 6 + i); }
    }
    store_se3(b.fpose, j, Hgc);
    store_se3(b.aX, j, Hpc);
    // child twist = Ad_cp T_p + Ad_cn T_nr                               (core.py:1308)
    double ta[6], tb[6], th[6];
    iad_apply(Hpc, Tp, ta);
    if (ident) {
#pragma unroll
      for (int i = 0; i < 6; ++i) tb[i] = k.T[i];
    } else {
      ad_apply(Hcn, k.T, tb);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) FT(b.atw, j * 6 + i) = ta[i] + tb[i];
    // theta_c = X_c theta_p - Ad_cn Ad_nr Ad_nr T_nr
    {
      Se3 Hnr;
      se3_inv(k.H, Hnr);
      double t1[6], t2[6], tau[6];
      ad_apply(Hnr, k.T, t1);
      ad_apply(Hnr, t1, t2);
      if (ident) {
#pragma unroll
        for (int i = 0; i < 6; ++i) tau[i] = t2[i];
      } else {
        ad_apply(Hcn, t2, tau);
      }
      iad_apply(Hpc, thp, ta);
#pragma unroll
      for (int i = 0; i < 6; ++i) { th[i] = ta[i] - tau[i]; FT(b.ath, j * 6 + i) = th[i]; }
    }
    // own columns: s = Ad_cn S, s^ = Ad_cn dS - adjacency(theta) s         (core.py:1310,1313)
    for (int c = 0; c < nd; ++c) {
      double s0[6], ds0[6], s[6], ds[6], as[6];
      if (type == ARB_JOINT_FREE) {
#pragma unroll
        for (int i = 0; i < 6; ++i) { s0[i] = (i == c) ? 1. : 0.; ds0[i] = 0.; }
      } else {
#pragma unroll
        for (int i = 0; i < 6; ++i) { s0[i] = k.S[6 * c + i]; ds0[i] = k.dS[6 * c + i]; }
      }
      if (ident) {
#pragma unroll
        for (int i = 0; i < 6; ++i) { s[i] = s0[i]; ds[i] = ds0[i]; }
      } else {
        ad_apply(Hcn, s0, s);
        ad_apply(Hcn, ds0, ds);
      }
      adj_apply(th, s, as);
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        FT(b.aS, (dof + c) * 6 + i) = s[i];
        FT(b.aSh, (dof + c) * 6 + i) = ds[i] - as[i];
      }
    }
  }
}

// generalized force of the (diagonal) PD controllers on dof k        (controllers.py:141-159)
// Per-world parameters (arb_batch_bind_controller_params) are indexed by WORLD: under a sorted
// assignment the thread's column w is a slot, its world is perm[w].
ARB_D int64_t artic_param_world(const DevBatch& b, int64_t w) { return b.perm ? (int64_t)b.perm[w] : w; }
ARB_D double artic_pd_param(const double* per_world, const double* model, const DevModel& m, const DevBatch& b,
                            int64_t w, int k) {
  return per_world ? per_world[(int64_t)m.pd_index[k] * b.W + artic_param_world(b, w)] : model[k];
}
ARB_D double artic_tau(const DevModel& m, const DevBatch& b, int64_t w, int k) {
  if (!m.has_pd || m.pd_gpos[k] < 0) return 0.;
  const double q = ST_LD(b.gpos, m.pd_gpos[k]);
  if (!(b.pkp || b.pkd || b.pqd || b.pdqd)) return m.pd_kp[k] * (m.pd_qd[k] - q) + m.pd_c[k];
  return artic_pd_param(b.pkp, m.pd_kp, m, b, w, k) * (artic_pd_param(b.pqd, m.pd_qd, m, b, w, k) - q) +
         artic_pd_param(b.pkd, m.pd_kd, m, b, w, k) * artic_pd_param(b.pdqd, m.pd_dqd, m, b, w, k);
}
// diagonal impedance of the PD controller on dof k: dt kp + kd
ARB_D double artic_pd_diag(const DevModel& m, const DevBatch& b, int64_t w, int k, double dt) {
  if (m.pd_gpos[k] < 0) return 0.;
  return dt * artic_pd_param(b.pkp, m.pd_kp, m, b, w, k) + artic_pd_param(b.pkd, m.pd_kd, m, b, w, k);
}

// ---------------------------------------------------------------------------------------
// leaf-to-root pass: elimination of every dof (stores U, LA, LM, 1/d) together with the
// reduced right-hand side u of the free motion (w_b = M_b (T_b/dt + gravity_b) + applied wrench,
// tau = PD + applied generalized force).  APPLIED = false: the instantiation without the applied-force
// terms, which the fused step runs while none are bound (with them ptxas spills 48 more bytes in the
// prepare kernel, a cost the unbound step need not pay).
template <bool APPLIED>
ARB_D bool artic_factor(const DevModel& m, const DevBatch& b, int64_t w, double dt, const DevApplied& ap) {
  bool ok = true;
  // 1/dt once per world: the 36 M_b/dt per body are mostly 0/dt, which sends the fp64 division
  // through its slow path (a quarter of this stage's instructions before)
  const double idt = 1. / dt;
  const double gt[6] = {0., 0., 0., m.gravity * m.up[0], m.gravity * m.up[1], m.gravity * m.up[2]};
  // Along a chain (joint j+1 hangs on the body of joint j, the usual case in depth-first order) the
  // child's contribution X^T IA X, X^T IM X, X^T beta stays in registers for the next iteration
  // instead of going through its scratch slot: `carry`.
  double IA[36], IM[36], beta[6];
  bool carry = false;
  for (int j = m.nj - 1; j >= 0; --j) {
    if (j > 0) {
      arb_prefetch_rows<6>(b.atw + (j - 1) * (6 * ARB_TILE));
      arb_prefetch_rows<6>(b.ath + (j - 1) * (6 * ARB_TILE));
      arb_prefetch_rows<12>(b.aX + (j - 1) * (12 * ARB_TILE));
      arb_prefetch_rows<12>(b.fpose + (j - 1) * (12 * ARB_TILE));
      artic_prefetch_dofs(m, j - 1, b.aS, b.aSh, nullptr, nullptr);
    }
    const int type = m.jtype[j];
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(type);
    const int dof = m.jdof[j];
    const int flags = m.bflags[j];
    const double* Mb = m.bmass + 36 * j;
    if (!carry) {
#pragma unroll
      for (int i = 0; i < 36; ++i) { IA[i] = 0.; IM[i] = 0.; }
#pragma unroll
      for (int i = 0; i < 6; ++i) beta[i] = 0.;
    }
    double T[6], th[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) { T[i] = FT(b.atw, j * 6 + i); th[i] = FT(b.ath, j * 6 + i); }
    if (flags & ARB_BODY_HASMASS) {
      // A_b = M_b/dt + B_b + Omega(T) M_b + M_b adjacency(theta)
      double X3[9];
      {
        double wx[9], t1[9], t2[9];
        skew3(T, wx);
        m3_mul(m.brx + 9 * j, wx, t1);
        m3_mul(wx, m.brx + 9 * j, t2);
#pragma unroll
        for (int i = 0; i < 9; ++i) X3[i] = t1[i] - t2[i];
      }
#pragma unroll
      for (int c = 0; c < 6; ++c) {  // Omega M, column by column
        double top[3] = {Mb[c], Mb[6 + c], Mb[12 + c]}, bot[3] = {Mb[18 + c], Mb[24 + c], Mb[30 + c]};
        double a[3], x2[3], d[3];
        cross3(T, top, a);
        m3_mulv(X3, bot, x2);
        cross3(T, bot, d);
#pragma unroll
        for (int i = 0; i < 3; ++i) { IA[6 * i + c] += a[i] + x2[i]; IA[6 * (i + 3) + c] += d[i]; }
      }
#pragma unroll
      for (int r = 0; r < 6; ++r) {  // M adjacency(theta), row by row: [a1 x w + a2 x v, a2 x w]
        const double* a1 = Mb + 6 * r;
        const double* a2 = Mb + 6 * r + 3;
        double c1[3], c2[3], c3[3];
        cross3(a1, th, c1);
        cross3(a2, th + 3, c2);
        cross3(a2, th, c3);
#pragma unroll
        for (int i = 0; i < 3; ++i) { IA[6 * r + i] += c1[i] + c2[i]; IA[6 * r + 3 + i] += c3[i]; }
      }
#pragma unroll
      for (int i = 0; i < 36; ++i) { IA[i] += Mb[i] * idt; IM[i] += Mb[i]; }
      // -w_b = -M_b (T/dt + gravity_b)
      double a[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) a[i] = T[i] * idt;
      if ((flags & ARB_BODY_MASSIVE) && m.nweight > 0) {
        Se3 H;
        load_se3(b.fpose, j, H);
        double g[6];
        iad_apply(H, gt, g);
#pragma unroll
        for (int i = 0; i < 6; ++i) a[i] += g[i];
      }
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        double t = 0.;
#pragma unroll
        for (int c = 0; c < 6; ++c) t += Mb[6 * r + c] * a[c];
        beta[r] -= t;
      }
    }
    if (flags & ARB_BODY_HASVISC) {
      const double* Bb = m.bvisc + 36 * j;
#pragma unroll
      for (int i = 0; i < 36; ++i) IA[i] += Bb[i];
    }
    // applied wrench (arb_batch_bind_applied_forces), on massless bodies too: -[R^T torque; R^T force]
    if (APPLIED && ap.wrench) {
      const int row = ap.row[j];
      if (row >= 0) {
        const double* wp = ap.wrench + (int64_t)(6 * row) * b.W + artic_param_world(b, w);
        double R[9], wg[6], wr[6];
#pragma unroll
        for (int i = 0; i < 9; ++i) R[i] = FT(b.fpose, j * 12 + i);
#pragma unroll
        for (int i = 0; i < 6; ++i) wg[i] = arb_ld_state(wp + (int64_t)i * b.W);
        m3t_mulv(R, wg, wr);
        m3t_mulv(R, wg + 3, wr + 3);
#pragma unroll
        for (int i = 0; i < 6; ++i) beta[i] -= wr[i];
      }
    }
    // children's contributions: every child joint c left X^T IA X, X^T IM X, X^T beta in ITS
    // OWN slot (no read-modify-write on the way up), summed here
    for (int c = m.jchild0[j]; c >= 0; c = m.jsib[c]) {
      if (carry && c == j + 1) continue;        // already in IA, IM, beta
      const double* pa = b.aIA + c * (36 * ARB_TILE);
      const double* pm = b.aIM + c * (36 * ARB_TILE);
      const double* pb = b.abeta + c * (6 * ARB_TILE);
#pragma unroll
      for (int i = 0; i < 36; ++i) { IA[i] += pa[i * ARB_TILE]; IM[i] += pm[i * ARB_TILE]; }
#pragma unroll
      for (int i = 0; i < 6; ++i) beta[i] += pb[i * ARB_TILE];
      arb_discard_rows<36>(pa);      // dead until joint c writes its slot again in the next step
      arb_discard_rows<36>(pm);
      arb_discard_rows<6>(pb);
    }
    for (int c = nd - 1; c >= 0; --c) {
      const int k = dof + c;
      double s[6], sh[6], U[6], LA[6], LM[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) { s[i] = FT(b.aS, k * 6 + i); sh[i] = FT(b.aSh, k * 6 + i); }
      double d = 0., sb = 0.;
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        double t = 0.;
#pragma unroll
        for (int i = 0; i < 6; ++i) t += IA[6 * r + i] * s[i] + IM[6 * r + i] * sh[i];
        U[r] = t;
        d += s[r] * t;
        sb += s[r] * beta[r];
      }
      if (m.has_pd) d += artic_pd_diag(m, b, w, k, dt);
      if (!(fabs(d) > 0.)) ok = false;
      const double dinv = 1. / d;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        double ta = 0., tm = 0.;
#pragma unroll
        for (int r = 0; r < 6; ++r) { ta += s[r] * IA[6 * r + i]; tm += s[r] * IM[6 * r + i]; }
        LA[i] = ta * dinv;
        LM[i] = tm * dinv;
      }
      double tau = artic_tau(m, b, w, k);
      if (APPLIED && ap.tau) tau += arb_ld_state(ap.tau + (int64_t)k * b.W + artic_param_world(b, w));
      const double u = (tau - sb) * dinv;
      FT(b.au, k) = u;
      FT(b.adinv, k) = dinv;
#pragma unroll
      for (int i = 0; i < 6; ++i) { FT(b.aU, k * 6 + i) = U[i]; FT(b.aLA, k * 6 + i) = LA[i]; FT(b.aLM, k * 6 + i) = LM[i]; }
      if (c > 0 || par != 0) {
#pragma unroll
        for (int r = 0; r < 6; ++r) {
#pragma unroll
          for (int i = 0; i < 6; ++i) { IA[6 * r + i] -= U[r] * LA[i]; IM[6 * r + i] -= U[r] * LM[i]; }
          beta[r] += U[r] * u;
        }
      }
    }
    if (par != 0) {
      Se3 X;
      load_se3(b.aX, j, X);
      congruence_up(X, IA);
      congruence_up(X, IM);
      double bu[6];
      wrench_up(X, beta, bu);
      carry = (par == j);       // the parent body is the one of joint j-1: next iteration
      if (carry) {
#pragma unroll
        for (int i = 0; i < 6; ++i) beta[i] = bu[i];
      } else {
        double* pa = b.aIA + j * (36 * ARB_TILE);
        double* pm = b.aIM + j * (36 * ARB_TILE);
        double* pb = b.abeta + j * (6 * ARB_TILE);
#pragma unroll
        for (int i = 0; i < 36; ++i) { pa[i * ARB_TILE] = IA[i]; pm[i * ARB_TILE] = IM[i]; }
#pragma unroll
        for (int i = 0; i < 6; ++i) pb[i * ARB_TILE] = bu[i];
      }
    } else {
      carry = false;
    }
  }
  return ok;
}

// ---------------------------------------------------------------------------------------
// The root-to-leaf passes below visit the joints in depth-first order, so most joints hang on the
// body of the joint visited just before: its (V, V^) are still in registers (`prev`).  A body's
// values go through aV only when another child reads them later, or when the generator rows read
// them (fused_gen_rows).
ARB_D bool artic_child_reads_aV(const DevModel& m, int j, int next, bool marked_only) {
  for (int c = m.jchild0[j]; c >= 0; c = m.jsib[c])
    if (c != next && (!marked_only || m.jmark[c])) return true;
  return false;
}
ARB_D bool artic_is_gen_body(const DevModel& m, int j) {
  for (int g = 0; g < m.ngen; ++g)
    if (m.gen_body[g] == j + 1) return true;
  return false;
}
// doubles per joint in aV
ARB_D int artic_vstride(const DevModel& m) { return 72 * (m.ngen > 1 ? m.ngen : 1); }
// (V, V^) of the child: X applied in place
ARB_D void artic_down(const Se3& X, double* V, double* Vh) {
  double a[6], c[6];
  iad_apply(X, V, a);
  iad_apply(X, Vh, c);
#pragma unroll
  for (int i = 0; i < 6; ++i) { V[i] = a[i]; Vh[i] = c[i]; }
}

// ---------------------------------------------------------------------------------------
// root-to-leaf pass for ONE right-hand side over ALL joints:  x_k = u_k - LA_k V - LM_k Vh.
// u_k is read from `u` for marked joints (or all joints if !marked_u), else 0.  x is written
// to `x`; (V, Vh) of the bodies other passes read is kept in aV[j][0..11].
// NE "extra" right-hand sides ride along over the marked joints when `ext` is set (the rows
// LA, LM, s, s^ are read once for all of them): unit generalized forces on the dofs ek[e], whose
// reduced right-hand sides artic_backward_generators left in au[1 + e]; solutions to ax[e],
// (V, Vh) to aV[j][12 (1 + e) ..].
// PF: prefetch the next joint's rows (pays in the prepare stage; the finish stage, which only runs
// this one pass over rows nothing else touched for a whole Gauss-Seidel, is 12 % faster without).
template <bool MARKED_U, int NE, bool PF = true>
ARB_D void artic_forward_full(const DevModel& m, const DevBatch& b, int64_t w, const double* u, double* x,
                              bool ext = false, const int* ek = nullptr) {
  const int n = m.ndof;
  const int VS = artic_vstride(m);
  double V[1 + NE][6], Vh[1 + NE][6];
  int eoff[NE > 0 ? NE : 1], ekc[NE > 0 ? NE : 1];
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    eoff[e] = ext ? m.coloff[m.dofbody[ek[e]]] : 0;
    ekc[e] = ext ? m.dofpos[ek[e]] + 1 : 0;
  }
  int prev = -2;
  for (int j = 0; j < m.nj; ++j) {
    if (PF && j + 1 < m.nj) {
      arb_prefetch_rows<12>(b.aX + (j + 1) * (12 * ARB_TILE));
      artic_prefetch_dofs(m, j + 1, b.aLA, b.aLM, b.aS, b.aSh);
    }
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(m.jtype[j]);
    const int dof = m.jdof[j];
    const bool ex = NE > 0 && ext && m.jmark[j];
    if (par == 0) {
#pragma unroll
      for (int r = 0; r < 1 + NE; ++r)
#pragma unroll
        for (int i = 0; i < 6; ++i) { V[r][i] = 0.; Vh[r][i] = 0.; }
    } else {
      Se3 X;
      load_se3(b.aX, j, X);
      const bool reload = (par - 1 != prev);
      if (reload) {
#pragma unroll
        for (int i = 0; i < 6; ++i) { V[0][i] = FT(b.aV, (par - 1) * VS + i); Vh[0][i] = FT(b.aV, (par - 1) * VS + 6 + i); }
      }
      artic_down(X, V[0], Vh[0]);
      if (ex) {
#pragma unroll
        for (int e = 1; e < 1 + NE; ++e) {
          if (reload) {
#pragma unroll
            for (int i = 0; i < 6; ++i) {
              V[e][i] = FT(b.aV, (par - 1) * VS + e * 12 + i);
              Vh[e][i] = FT(b.aV, (par - 1) * VS + e * 12 + 6 + i);
            }
          }
          artic_down(X, V[e], Vh[e]);
        }
      }
    }
    const bool useu = !MARKED_U || m.jmark[j];
    for (int c = 0; c < nd; ++c) {
      const int k = dof + c;
      double LA[6], LM[6], s[6], sh[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        LA[i] = FT(b.aLA, k * 6 + i); LM[i] = FT(b.aLM, k * 6 + i);
        s[i] = FT(b.aS, k * 6 + i); sh[i] = FT(b.aSh, k * 6 + i);
      }
      double t = useu ? FT(u, k) : 0.;
      if (par != 0 || c > 0) {
#pragma unroll
        for (int i = 0; i < 6; ++i) t -= LA[i] * V[0][i] + LM[i] * Vh[0][i];
      }
      FT(x, k) = t;
#pragma unroll
      for (int i = 0; i < 6; ++i) { V[0][i] += s[i] * t; Vh[0][i] += sh[i] * t; }
      if (ex) {
        const int pos = m.dofpos[k];
#pragma unroll
        for (int e = 0; e < NE; ++e) {
          const bool onpath = pos < ekc[e] && m.pathdof[eoff[e] + pos] == k;
          double te = onpath ? FT(b.au, (1 + e) * n + k) : 0.;
          if (par != 0 || c > 0) {
#pragma unroll
            for (int i = 0; i < 6; ++i) te -= LA[i] * V[1 + e][i] + LM[i] * Vh[1 + e][i];
          }
          FT(b.ax, e * n + k) = te;
#pragma unroll
          for (int i = 0; i < 6; ++i) { V[1 + e][i] += s[i] * te; Vh[1 + e][i] += sh[i] * te; }
        }
      }
    }
    const bool gen = !MARKED_U && m.jmark[j] && artic_is_gen_body(m, j);
    if (gen || artic_child_reads_aV(m, j, j + 1, false)) {
#pragma unroll
      for (int i = 0; i < 6; ++i) { FT(b.aV, j * VS + i) = V[0][i]; FT(b.aV, j * VS + 6 + i) = Vh[0][i]; }
    }
    if (ex && (gen || artic_child_reads_aV(m, j, j + 1, true))) {
#pragma unroll
      for (int e = 1; e < 1 + NE; ++e)
#pragma unroll
        for (int i = 0; i < 6; ++i) { FT(b.aV, j * VS + e * 12 + i) = V[e][i]; FT(b.aV, j * VS + e * 12 + 6 + i) = Vh[e][i]; }
    }
    prev = j;
  }
}

// ---------------------------------------------------------------------------------------
// NR right-hand sides that start on ONE root path (unit wrenches on body `body`, or a unit
// generalized force on dof `kstart`): leaf-to-root along the path, reduced right-hand sides u
// to au[ubase + r][k] for the path dofs.
// `rot` (9 doubles, row-major, or nullptr): the unit wrenches are those of the rotated generator
// basis G' = blockdiag(R, R) G of a contact-aligned body, i.e. wrench r is row r of blockdiag(R, R).
template <int NR>
ARB_D void artic_backward_generators(const DevModel& m, const DevBatch& b, int64_t w, int body, int kstart,
                                     const double* rot = nullptr, int ubase = 0) {
  const int n = m.ndof;
  const int off = m.coloff[body];
  double beta[NR][6];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int i = 0; i < 6; ++i) beta[r][i] = (kstart < 0 && i == r) ? -1. : 0.;
  if (rot != nullptr && NR == 6) {
#pragma unroll
    for (int r = 0; r < NR; ++r)
#pragma unroll
      for (int i = 0; i < 6; ++i) beta[r][i] = ((r < 3) == (i < 3)) ? -rot[3 * (r % 3) + (i % 3)] : 0.;
  }
  const int l0 = (kstart < 0) ? m.kcols[body] - 1 : m.dofpos[kstart];
  for (int l = l0; l >= 0; --l) {
    const int k = m.pathdof[off + l];
    const int j = m.dofjoint[k];
    if (l > 0) {
      const int kn = m.pathdof[off + l - 1];
      arb_prefetch_rows<6>(b.aS + kn * (6 * ARB_TILE));
      arb_prefetch_rows<6>(b.aU + kn * (6 * ARB_TILE));
      arb_prefetch(b.adinv + kn * ARB_TILE);
    }
    double s[6], U[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) { s[i] = FT(b.aS, k * 6 + i); U[i] = FT(b.aU, k * 6 + i); }
    const double dinv = FT(b.adinv, k);
    const bool last = (l == 0);
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      double sb = 0.;
#pragma unroll
      for (int i = 0; i < 6; ++i) sb += s[i] * beta[r][i];
      const double tau = (k == kstart) ? 1. : 0.;
      const double u = (tau - sb) * dinv;
      FT(b.au, (ubase + r) * n + k) = u;
      if (!last) {
#pragma unroll
        for (int i = 0; i < 6; ++i) beta[r][i] += U[i] * u;
      }
    }
    if (k == m.jdof[j] && m.jparent[j] != 0) {
      Se3 X;
      load_se3(b.aX, j, X);
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        double y[6];
        wrench_up(X, beta[r], y);
#pragma unroll
        for (int i = 0; i < 6; ++i) beta[r][i] = y[i];
      }
    }
  }
}

// The NR solutions of artic_backward_generators' right-hand sides (ubase 0) over the marked joints:
// x to ax[r][k]; V of the generator bodies (and (V, V^) of the bodies a later joint reads) to
// aV[j][r*12 ..].  CARRY = false: every body's (V, V^) goes through aV (less register pressure).
template <int NR, bool CARRY>
ARB_D void artic_forward_generators(const DevModel& m, const DevBatch& b, int64_t w, int body, int kstart) {
  const int n = m.ndof;
  const int VS = artic_vstride(m);
  const int off = m.coloff[body];
  const int kc = ((kstart < 0) ? m.kcols[body] - 1 : m.dofpos[kstart]) + 1;   // path dofs 0..kc-1 carry a non-zero u
  double V[NR][6], Vh[NR][6];
  int prev = -2;
  for (int j = 0; j < m.nj; ++j) {
    if (!m.jmark[j]) continue;
    int jn = j + 1;                       // the next joint of this pass
    while (jn < m.nj && !m.jmark[jn]) ++jn;
    if (jn < m.nj) {
      arb_prefetch_rows<12>(b.aX + jn * (12 * ARB_TILE));
      artic_prefetch_dofs(m, jn, b.aLA, b.aLM, b.aS, b.aSh);
    }
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(m.jtype[j]);
    const int dof = m.jdof[j];
    if (par == 0) {
#pragma unroll
      for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int i = 0; i < 6; ++i) { V[r][i] = 0.; Vh[r][i] = 0.; }
    } else {
      Se3 X;
      load_se3(b.aX, j, X);
      const bool reload = !CARRY || (par - 1 != prev);
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        if (reload) {
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            V[r][i] = FT(b.aV, (par - 1) * VS + r * 12 + i);
            Vh[r][i] = FT(b.aV, (par - 1) * VS + r * 12 + 6 + i);
          }
        }
        artic_down(X, V[r], Vh[r]);
      }
    }
    for (int c = 0; c < nd; ++c) {
      const int k = dof + c;
      const int pos = m.dofpos[k];
      const bool onpath = pos < kc && m.pathdof[off + pos] == k;
      double LA[6], LM[6], s[6], sh[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        LA[i] = FT(b.aLA, k * 6 + i); LM[i] = FT(b.aLM, k * 6 + i);
        s[i] = FT(b.aS, k * 6 + i); sh[i] = FT(b.aSh, k * 6 + i);
      }
#pragma unroll
      for (int r = 0; r < NR; ++r) {
        double t = onpath ? FT(b.au, r * n + k) : 0.;
        if (par != 0 || c > 0) {
#pragma unroll
          for (int i = 0; i < 6; ++i) t -= LA[i] * V[r][i] + LM[i] * Vh[r][i];
        }
        FT(b.ax, r * n + k) = t;
#pragma unroll
        for (int i = 0; i < 6; ++i) { V[r][i] += s[i] * t; Vh[r][i] += sh[i] * t; }
      }
    }
    if (!CARRY || artic_child_reads_aV(m, j, jn, true)) {
#pragma unroll
      for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          FT(b.aV, j * VS + r * 12 + i) = V[r][i];
          FT(b.aV, j * VS + r * 12 + 6 + i) = Vh[r][i];
        }
    } else if (artic_is_gen_body(m, j)) {
#pragma unroll
      for (int r = 0; r < NR; ++r)
#pragma unroll
        for (int i = 0; i < 6; ++i) FT(b.aV, j * VS + r * 12 + i) = V[r][i];
    }
    prev = j;
  }
}

// The six-column solves of ALL generator bodies (right-hand sides of artic_backward_generators with
// ubase = 6 gi) in ONE root-to-leaf pass over the marked joints: the rows LA, LM, s, s^ and X of a
// joint come from DRAM once and are re-read from the L1 for the other bodies, instead of once per
// body in passes far enough apart to miss the L2.  Body gi uses au / ax rows 6 gi .. 6 gi + 5 and
// aV[j][12 (6 gi + r) ..]; nothing stays in registers from one body to the next.
ARB_D void artic_forward_generators_all(const DevModel& m, const DevBatch& b, int64_t w) {
  const int n = m.ndof;
  const int VS = artic_vstride(m);
  for (int j = 0; j < m.nj; ++j) {
    if (!m.jmark[j]) continue;
    int jn = j + 1;                       // the next joint of this pass
    while (jn < m.nj && !m.jmark[jn]) ++jn;
    if (jn < m.nj) {
      arb_prefetch_rows<12>(b.aX + jn * (12 * ARB_TILE));
      artic_prefetch_dofs(m, jn, b.aLA, b.aLM, b.aS, b.aSh);
    }
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(m.jtype[j]);
    const int dof = m.jdof[j];
    for (int gi = 0; gi < m.ngen; ++gi) {
      const int off = m.coloff[m.gen_body[gi]];
      const int kc = m.kcols[m.gen_body[gi]];   // path dofs 0..kc-1 carry a non-zero u
      const int rb = 6 * gi;
      double V[6][6], Vh[6][6];
      if (par == 0) {
#pragma unroll
        for (int r = 0; r < 6; ++r)
#pragma unroll
          for (int i = 0; i < 6; ++i) { V[r][i] = 0.; Vh[r][i] = 0.; }
      } else {
        Se3 X;
        load_se3(b.aX, j, X);
#pragma unroll
        for (int r = 0; r < 6; ++r) {
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            V[r][i] = FT(b.aV, (par - 1) * VS + (rb + r) * 12 + i);
            Vh[r][i] = FT(b.aV, (par - 1) * VS + (rb + r) * 12 + 6 + i);
          }
          artic_down(X, V[r], Vh[r]);
        }
        // last reader of the parent's (V, V^): the generator rows read V (first 6 of 12) of generator
        // bodies later, everything else is dead
        if (m.jmarkfirst[j]) {
          const bool pgen = artic_is_gen_body(m, par - 1);
#pragma unroll
          for (int r = 0; r < 6; ++r) {
            const double* pv = b.aV + ((par - 1) * VS + (rb + r) * 12) * ARB_TILE;
            if (!pgen) arb_discard_rows<6>(pv);
            arb_discard_rows<6>(pv + 6 * ARB_TILE);
          }
        }
      }
      for (int c = 0; c < nd; ++c) {
        const int k = dof + c;
        const int pos = m.dofpos[k];
        const bool onpath = pos < kc && m.pathdof[off + pos] == k;
        double LA[6], LM[6], s[6], sh[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          LA[i] = FT(b.aLA, k * 6 + i); LM[i] = FT(b.aLM, k * 6 + i);
          s[i] = FT(b.aS, k * 6 + i); sh[i] = FT(b.aSh, k * 6 + i);
        }
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          double t = onpath ? FT(b.au, (rb + r) * n + k) : 0.;
          if (par != 0 || c > 0) {
#pragma unroll
            for (int i = 0; i < 6; ++i) t -= LA[i] * V[r][i] + LM[i] * Vh[r][i];
          }
          if (m.doflim[k]) FT(b.ax, (rb + r) * n + k) = t;     // (only joint-limit rows read a solution back)
#pragma unroll
          for (int i = 0; i < 6; ++i) { V[r][i] += s[i] * t; Vh[r][i] += sh[i] * t; }
        }
      }
      // (V, V^) for the children; a leaf of the marked tree only hands V to the generator rows
      const bool vh_read = m.jmarkchild[j] != 0;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int i = 0; i < 6; ++i) {
          FT(b.aV, j * VS + (rb + r) * 12 + i) = V[r][i];
          if (vh_read) FT(b.aV, j * VS + (rb + r) * 12 + 6 + i) = Vh[r][i];
        }
    }
  }
}

// Carrying (V, V^) of SIX right-hand sides along chains keeps 144 registers live across the joint
// loop: measured slower (spills, prepare 4.80 vs 4.65 ms per 262144 worlds), so the six-column
// solves go through aV; the one- to three-column pass above carries.
#ifndef ARTIC_GEN_CARRY
#define ARTIC_GEN_CARRY 0
#endif
template <int NR>
ARB_D void artic_solve_generators(const DevModel& m, const DevBatch& b, int64_t w, int body, int kstart,
                                  const double* rot = nullptr) {
  artic_backward_generators<NR>(m, b, w, body, kstart, rot, 0);
  artic_forward_generators<NR, (ARTIC_GEN_CARRY != 0)>(m, b, w, body, kstart);
}

// row `g` of the generator matrix G applied to the solution r of the last solve:
// body generators read V of their body, joint-limit generators the dof itself.
ARB_D double artic_gen_value(const DevModel& m, const DevBatch& b, int64_t w, int g, int r, const double* x) {
  if (g < 6 * m.ngen) return FT(b.aV, (m.gen_body[g / 6] - 1) * artic_vstride(m) + r * 12 + g % 6);
  return FT(x, r * m.ndof + m.glimdof[g - 6 * m.ngen]);
}
// the 6 rows of generator body gi applied to solution r: V of the body, rotated into the
// contact-aligned frame (rot = R_e, 9 doubles) when the body is aligned
ARB_D void artic_gen_block(const DevModel& m, const DevBatch& b, int gi, int r, const double* rot, double* out) {
  double V[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) V[i] = FT(b.aV, (m.gen_body[gi] - 1) * artic_vstride(m) + r * 12 + i);
  if (rot != nullptr) {
    m3_mulv(rot, V, out);
    m3_mulv(rot, V + 3, out + 3);
  } else {
#pragma unroll
    for (int i = 0; i < 6; ++i) out[i] = V[i];
  }
}

// ---------------------------------------------------------------------------------------
// leaf-to-root pass over the marked joints for the Gauss-Seidel result y (wrenches on the
// generator bodies, generalized forces on the limited dofs): u -> au[0][k] (marked dofs).
ARB_D void artic_backward_wrenches(const DevModel& m, const DevBatch& b, int64_t w, const double* y) {
  const int NG6 = 6 * m.ngen;
  for (int j = m.nj - 1; j >= 0; --j) {
    if (!m.jmark[j]) continue;
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(m.jtype[j]);
    const int dof = m.jdof[j];
    double beta[6] = {0., 0., 0., 0., 0., 0.};
    for (int g = 0; g < m.ngen; ++g)
      if (m.gen_body[g] == j + 1) {
        if (m.gen_aligned[g]) {     // y is in the contact-aligned frame: wrench = blockdiag(R_e, R_e)^T y
          double Re[9], yy[6], t[6];
#pragma unroll
          for (int i = 0; i < 9; ++i) Re[i] = FT(b.fRe, 9 * g + i);
#pragma unroll
          for (int i = 0; i < 6; ++i) yy[i] = FT(y, 6 * g + i);
          m3t_mulv(Re, yy, t);
          m3t_mulv(Re, yy + 3, t + 3);
#pragma unroll
          for (int i = 0; i < 6; ++i) beta[i] -= t[i];
        } else {
#pragma unroll
          for (int i = 0; i < 6; ++i) beta[i] -= FT(y, 6 * g + i);
        }
      }
    for (int c = m.jchild0[j]; c >= 0; c = m.jsib[c])
      if (m.jmark[c]) {
#pragma unroll
        for (int i = 0; i < 6; ++i) beta[i] += FT(b.abeta, c * 6 + i);
      }
    for (int c = nd - 1; c >= 0; --c) {
      const int k = dof + c;
      double tau = 0.;
      for (int g = NG6; g < m.ngrows; ++g)
        if (m.glimdof[g - NG6] == k) tau += FT(y, g);
      double sb = 0.;
#pragma unroll
      for (int i = 0; i < 6; ++i) sb += FT(b.aS, k * 6 + i) * beta[i];
      const double u = (tau - sb) * FT(b.adinv, k);
      FT(b.au, k) = u;
      if (c > 0 || par != 0) {
#pragma unroll
        for (int i = 0; i < 6; ++i) beta[i] += FT(b.aU, k * 6 + i) * u;
      }
    }
    if (par != 0) {
      Se3 X;
      load_se3(b.aX, j, X);
      double bu[6];
      wrench_up(X, beta, bu);
#pragma unroll
      for (int i = 0; i < 6; ++i) FT(b.abeta, j * 6 + i) = bu[i];
    }
  }
}

// One world per thread ("lane-per-world"): the four phases of the reference
// step written as scalar routines over structure-of-arrays memory
// (element index major, world index fastest, so the 32 lanes of a warp touch
// 256 contiguous bytes).  These are the API-shaped phases -- every intermediate
// the reference exposes (body pose/jacobian/..., M, N, B, Z, Y, constraint
// state) is left in HBM scratch for the arb_get_* read-backs.
//
// Reference lines followed:
//   world_update_dynamic      core.py:716-734 and Body.update_dynamic core.py:1272-1315
//   world_update_controllers  core.py:811-818, controllers.py:43-60, :141-159
//   world_update_constraints  core.py:910-937, constraints.py (see arb_constraints.cuh)
//   world_integrate           core.py:974-980, core.py:238-240, joints.py:54-57
#pragma once
#include "arb_constraints.cuh"
#include "arb_joints.cuh"
#include "arb_math.cuh"
#include "arb_types.h"

#define AT(ptr, idx) (ptr)[(int64_t)(idx) * W + w]

ARB_D void load_pose(const DevBatch& b, int body, int64_t w, Se3& h) {
  const int64_t W = b.W;
  if (body == 0) { se3_identity(h); return; }
  const int o = (body - 1) * 12;
#pragma unroll
  for (int i = 0; i < 9; ++i) h.R[i] = AT(b.pose, o + i);
#pragma unroll
  for (int i = 0; i < 3; ++i) h.p[i] = AT(b.pose, o + 9 + i);
}
ARB_D void load_twist(const DevBatch& b, int body, int64_t w, double* t) {
  const int64_t W = b.W;
#pragma unroll
  for (int i = 0; i < 6; ++i) t[i] = (body == 0) ? 0. : AT(b.twist, (body - 1) * 6 + i);
}

// The world's own M_b, rx and body flags of body j+1 (arb_batch_bind_body_inertia) when PARAMS and the
// body is bound; the model's otherwise.  Mw, rxw: storage for the world's values.
template <bool PARAMS>
ARB_D int world_body_mass(const DevModel& m, const DevApplied& ap, int j, int64_t W, int64_t w,
                          const double*& Mb, const double*& rx, double* Mw, double* rxw) {
  Mb = m.bmass + 36 * j;
  rx = m.brx + 9 * j;
  int flags = m.bflags[j];
  if constexpr (PARAMS) {
    const int row = ap.inertia ? ap.irow[j] : -1;
    if (row >= 0) {
      double v[10];
#pragma unroll
      for (int i = 0; i < 10; ++i) v[i] = ap.inertia[(int64_t)(10 * row + i) * W + w];
      flags = (flags & ARB_BODY_HASVISC) | body_inertia_matrix(v, Mw, rxw);
      Mb = Mw;
      rx = rxw;
    }
  }
  return flags;
}

// ---------------------------------------------------------------------------
// PARAMS: with the world's body inertia (arb_batch_bind_body_inertia, ap.inertia)
template <bool PARAMS = false>
ARB_D void world_update_dynamic(const DevModel& m, const DevBatch& b, int64_t w,
                                const DevApplied& ap = DevApplied{nullptr, nullptr, nullptr}) {
  const int64_t W = b.W;
  const int n = m.ndof;
  for (int i = 0; i < n * n; ++i) {
    AT(b.M, i) = 0.;
    AT(b.N, i) = 0.;
    AT(b.B, i) = 0.;
  }
  for (int j = 0; j < m.nj; ++j) {
    const int type = m.jtype[j];
    const int par = m.jparent[j];
    const int nd = arb_joint_ndof(type);
    double q[16], dq[6];
    for (int i = 0; i < arb_joint_ngpos(type); ++i) q[i] = AT(b.gpos, m.jgpos[j] + i);
    for (int i = 0; i < nd; ++i) dq[i] = AT(b.gvel, m.jdof[j] + i);
    JointKin k;
    joint_kinematics(type, q, dq, k);
    const bool ident = m.hcn_ident[j] != 0;
    // H_pc = H_pr H_rn inv(H_cn), child pose = H_gp H_pc            (core.py:1295-1299)
    Se3 Hpr, Hcn, Hpc, Hgp, Hgc, t0;
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
    load_pose(b, par, w, Hgp);
    se3_mul(Hgp, Hpc, Hgc);
#pragma unroll
    for (int i = 0; i < 9; ++i) AT(b.pose, j * 12 + i) = Hgc.R[i];
#pragma unroll
    for (int i = 0; i < 3; ++i) AT(b.pose, j * 12 + 9 + i) = Hgc.p[i];
    // child twist = Ad_cp T_p + Ad_cn T_nr                              (core.py:1308)
    double Tp[6], Tc[6], ta[6], tb[6];
    load_twist(b, par, w, Tp);
    iad_apply(Hpc, Tp, ta);
    if (ident) {
#pragma unroll
      for (int i = 0; i < 6; ++i) tb[i] = k.T[i];
    } else {
      ad_apply(Hcn, k.T, tb);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) { Tc[i] = ta[i] + tb[i]; AT(b.twist, j * 6 + i) = Tc[i]; }
    // dAd_cp = Ad_cn . (Ad(H_nr) adjacency(-Ad(H_nr) T_nr)) . Ad_rp       (core.py:1300-1304,
    //                                                                    rigidmotion.py:49-75)
    Blk6 dAd;
    {
      Se3 Hnr, HprInv;
      se3_inv(k.H, Hnr);
      double it[6];
      ad_apply(Hnr, k.T, it);
#pragma unroll
      for (int i = 0; i < 6; ++i) it[i] = -it[i];
      Blk6 iAd, adj, t1, Adrp;
      blk_from_se3(Hnr, iAd);
      blk_adjacency(it, adj);
      blk_mul(iAd, adj, t1);
      load_se3_const(m.HprInv, j, HprInv);
      blk_from_se3(HprInv, Adrp);
      if (ident) {
        blk_mul(t1, Adrp, dAd);
      } else {
        Blk6 t2, Adcn;
        blk_mul(t1, Adrp, t2);
        blk_from_se3(Hcn, Adcn);
        blk_mul(Adcn, t2, dAd);
      }
    }
    // Jacobian / hessian columns of the child                         (core.py:1309-1313)
    const int kp = m.kcols[par], offp = m.coloff[par], offc = m.coloff[j + 1];
    for (int l = 0; l < kp; ++l) {
      double Jp[6], dJp[6], Jc[6], dJc[6], t1[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) { Jp[i] = AT(b.J, (offp + l) * 6 + i); dJp[i] = AT(b.dJ, (offp + l) * 6 + i); }
      iad_apply(Hpc, Jp, Jc);
      blk_apply(dAd, Jp, dJc);
      iad_apply(Hpc, dJp, t1);
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        AT(b.J, (offc + l) * 6 + i) = Jc[i];
        AT(b.dJ, (offc + l) * 6 + i) = dJc[i] + t1[i];
      }
    }
    for (int c = 0; c < nd; ++c) {
      double s[6], ds[6], Jc[6], dJc[6];
      if (type == ARB_JOINT_FREE) {
#pragma unroll
        for (int i = 0; i < 6; ++i) { s[i] = (i == c) ? 1. : 0.; ds[i] = 0.; }
      } else {
#pragma unroll
        for (int i = 0; i < 6; ++i) { s[i] = k.S[6 * c + i]; ds[i] = k.dS[6 * c + i]; }
      }
      if (ident) {
#pragma unroll
        for (int i = 0; i < 6; ++i) { Jc[i] = s[i]; dJc[i] = ds[i]; }
      } else {
        ad_apply(Hcn, s, Jc);
        ad_apply(Hcn, ds, dJc);
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        AT(b.J, (offc + kp + c) * 6 + i) = Jc[i];
        AT(b.dJ, (offc + kp + c) * 6 + i) = dJc[i];
      }
    }
    // M += J^T M_b J ; B += J^T B_b J ; N += J^T (M_b dJ + N_b J)          (core.py:725-734)
    // with N_b = [[w^, rx w^ - w^ rx],[0, w^]] M_b                        (core.py:1276-1288)
    const double *Mb, *rx;
    double Mw[36], rxw[9];
    const int flags = world_body_mass<PARAMS>(m, ap, j, W, w, Mb, rx, Mw, rxw);
    if (flags & (ARB_BODY_HASMASS | ARB_BODY_HASVISC)) {
      const double* Bb = m.bvisc + 36 * j;
      double wx[9], X[9];
      {
        double t1[9], t2[9];
        skew3(Tc, wx);
        m3_mul(rx, wx, t1);
        m3_mul(wx, rx, t2);
#pragma unroll
        for (int i = 0; i < 9; ++i) X[i] = t1[i] - t2[i];
      }
      const int kc = kp + nd;
      for (int l = 0; l < kc; ++l) {
        double Jl[6], dJl[6], P[6], Q[6], V[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) { Jl[i] = AT(b.J, (offc + l) * 6 + i); dJl[i] = AT(b.dJ, (offc + l) * 6 + i); }
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          double p = 0., qq = 0., v = 0.;
#pragma unroll
          for (int c = 0; c < 6; ++c) {
            p += Mb[6 * r + c] * Jl[c];
            qq += Mb[6 * r + c] * dJl[c];
            v += Bb[6 * r + c] * Jl[c];
          }
          P[r] = p; Q[r] = qq; V[r] = v;
        }
        {  // Q += Omega P
          double a[3], c2[3], d[3];
          m3_mulv(wx, P, a);
          m3_mulv(X, P + 3, c2);
          m3_mulv(wx, P + 3, d);
#pragma unroll
          for (int i = 0; i < 3; ++i) { Q[i] += a[i] + c2[i]; Q[3 + i] += d[i]; }
        }
        const int dl = m.pathdof[offc + l];
        for (int mm = 0; mm < kc; ++mm) {
          const int dm = m.pathdof[offc + mm];
          double am = 0., an = 0., ab = 0.;
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            double jm = AT(b.J, (offc + mm) * 6 + i);
            am += jm * P[i];
            an += jm * Q[i];
            ab += jm * V[i];
          }
          AT(b.M, dm * n + dl) += am;
          AT(b.N, dm * n + dl) += an;
          if (flags & ARB_BODY_HASVISC) AT(b.B, dm * n + dl) += ab;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// In-place inverse of the n x n matrix at Y (row-major, SoA) by Gauss-Jordan
// elimination with partial pivoting (what numpy.linalg.inv -> dgesv does up to
// operation order).  perm: n ints of per-thread scratch stored as doubles.
ARB_D bool world_invert(double* Y, double* perm, int n, int64_t W, int64_t w) {
  bool ok = true;
  for (int k = 0; k < n; ++k) {
    int piv = k;
    double best = fabs(AT(Y, k * n + k));
    for (int i = k + 1; i < n; ++i) {
      double v = fabs(AT(Y, i * n + k));
      if (v > best) { best = v; piv = i; }
    }
    AT(perm, k) = (double)piv;
    if (best == 0.) { ok = false; continue; }
    if (piv != k)
      for (int j = 0; j < n; ++j) {
        double t = AT(Y, k * n + j);
        AT(Y, k * n + j) = AT(Y, piv * n + j);
        AT(Y, piv * n + j) = t;
      }
    double inv = 1. / AT(Y, k * n + k);
    AT(Y, k * n + k) = 1.;
    for (int j = 0; j < n; ++j) AT(Y, k * n + j) *= inv;
    for (int i = 0; i < n; ++i) {
      if (i == k) continue;
      double f = AT(Y, i * n + k);
      if (f == 0.) continue;
      AT(Y, i * n + k) = 0.;
      for (int j = 0; j < n; ++j) AT(Y, i * n + j) -= f * AT(Y, k * n + j);
    }
  }
  for (int k = n - 1; k >= 0; --k) {
    int piv = (int)AT(perm, k);
    if (piv != k)
      for (int i = 0; i < n; ++i) {
        double t = AT(Y, i * n + k);
        AT(Y, i * n + k) = AT(Y, i * n + piv);
        AT(Y, i * n + piv) = t;
      }
  }
  return ok;
}

// ap: the applied forces of arb_batch_bind_applied_forces (none by default); PARAMS: with the world's
// body inertia and gravity (ap.inertia, ap.gravity)
template <bool PARAMS = false>
ARB_D void world_update_controllers(const DevModel& m, const DevBatch& b, int64_t w, double dt,
                                    const DevApplied& ap = DevApplied{nullptr, nullptr, nullptr}) {
  const int64_t W = b.W;
  const int n = m.ndof;
  for (int i = 0; i < n; ++i) AT(b.gforce, i) = 0.;
  // Z = M/dt + B + N                                                   (core.py:813)
  for (int i = 0; i < n * n; ++i) AT(b.Z, i) = AT(b.M, i) / dt + AT(b.B, i) + AT(b.N, i);
  bool weighed = false;     // (PARAMS) the world's gravity is evaluated once, at the first WeightController
  for (int a = 0; a < m.na; ++a) {
    if (m.atype[a] == ARB_CTRL_WEIGHT) {
      // gforce += J_b^T M_b Ad(pose_b^-1) [0,0,0, g up]                  (controllers.py:43-60)
      const double grav = m.adbl[4 * a];
      double gt[6] = {0., 0., 0., grav * m.up[0], grav * m.up[1], grav * m.up[2]};
      if constexpr (PARAMS) {
        if (ap.gravity) {
          if (weighed) continue;
          weighed = true;
#pragma unroll
          for (int i = 0; i < 3; ++i) gt[3 + i] = ap.gravity[(int64_t)i * W + w];
        }
      }
      for (int j = 0; j < m.nj; ++j) {
        const double *Mb, *rx;
        double Mw[36], rxw[9];
        if (!(world_body_mass<PARAMS>(m, ap, j, W, w, Mb, rx, Mw, rxw) & ARB_BODY_MASSIVE)) continue;
        Se3 H;
        load_pose(b, j + 1, w, H);
        double g[6], wr[6];
        iad_apply(H, gt, g);
#pragma unroll
        for (int r = 0; r < 6; ++r) {
          double t = 0.;
#pragma unroll
          for (int c = 0; c < 6; ++c) t += Mb[6 * r + c] * g[c];
          wr[r] = t;
        }
        const int off = m.coloff[j + 1], kc = m.kcols[j + 1];
        for (int l = 0; l < kc; ++l) {
          double t = 0.;
#pragma unroll
          for (int i = 0; i < 6; ++i) t += AT(b.J, (off + l) * 6 + i) * wr[i];
          AT(b.gforce, m.pathdof[off + l]) += t;
        }
      }
    } else {
      // PD: gforce[dofs] += kp (q_d - q) + kd dq_d ; Z[dofs,dofs] += dt kp + kd  (controllers.py:141-159)
      const int mm = m.aint[4 * a], off = m.aint[4 * a + 1];
      const double* dofs = m.ablob + off;
      const double* gmap = dofs + mm;
      const double* kp = gmap + mm;
      const double* kd = kp + mm * mm;
      const double* qd = kd + mm * mm;
      const double* dqd = qd + mm;
      // per-world parameters (arb_batch_bind_controller_params): rows prow + i of [npd][W] arrays
      // replace gpos_des, gvel_des and the DIAGONAL gains of this controller
      int prow = 0;
      for (int a2 = 0; a2 < a; ++a2)
        if (m.atype[a2] == ARB_CTRL_PD) prow += m.aint[4 * a2];
      for (int i = 0; i < mm; ++i) {
        double t = 0.;
        for (int j = 0; j < mm; ++j) {
          const double kpij = (i == j && b.pkp) ? b.pkp[(int64_t)(prow + j) * W + w] : kp[i * mm + j];
          const double qdj = b.pqd ? b.pqd[(int64_t)(prow + j) * W + w] : qd[j];
          t += kpij * (qdj - AT(b.gpos, (int)gmap[j]));
        }
        double t2 = 0.;
        for (int j = 0; j < mm; ++j) {
          const double kdij = (i == j && b.pkd) ? b.pkd[(int64_t)(prow + j) * W + w] : kd[i * mm + j];
          const double dqdj = b.pdqd ? b.pdqd[(int64_t)(prow + j) * W + w] : dqd[j];
          t2 += kdij * dqdj;
        }
        AT(b.gforce, (int)dofs[i]) += t + t2;
        for (int j = 0; j < mm; ++j) {
          const double kpij = (i == j && b.pkp) ? b.pkp[(int64_t)(prow + j) * W + w] : kp[i * mm + j];
          const double kdij = (i == j && b.pkd) ? b.pkd[(int64_t)(prow + j) * W + w] : kd[i * mm + j];
          AT(b.Z, (int)dofs[i] * n + (int)dofs[j]) -= -(dt * kpij + kdij);
        }
      }
    }
  }
  // applied forces (arb_batch_bind_applied_forces), a controller registered after the model's with
  // no impedance: gforce += tau + sum_b J_b^T [R_b^T torque_b; R_b^T force_b]
  if (ap.tau)
    for (int k = 0; k < n; ++k) AT(b.gforce, k) += ap.tau[(int64_t)k * W + w];
  if (ap.wrench)
    for (int j = 0; j < m.nj; ++j) {
      const int row = ap.row[j];
      if (row < 0) continue;
      Se3 H;
      load_pose(b, j + 1, w, H);
      double wg[6], wr[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) wg[i] = ap.wrench[(int64_t)(6 * row + i) * W + w];
      m3t_mulv(H.R, wg, wr);
      m3t_mulv(H.R, wg + 3, wr + 3);
      const int off = m.coloff[j + 1], kc = m.kcols[j + 1];
      for (int l = 0; l < kc; ++l) {
        double t = 0.;
#pragma unroll
        for (int i = 0; i < 6; ++i) t += AT(b.J, (off + l) * 6 + i) * wr[i];
        AT(b.gforce, m.pathdof[off + l]) += t;
      }
    }
  // Y = Z^-1                                                            (core.py:818)
  for (int i = 0; i < n * n; ++i) AT(b.Y, i) = AT(b.Z, i);
  if (!world_invert(b.Y, b.tmp, n, W, w)) b.status[w] |= ARB_STATUS_SINGULAR;
}

// ---------------------------------------------------------------------------
ARB_D void world_integrate(const DevModel& m, const DevBatch& b, int64_t w, double dt) {
  const int64_t W = b.W;
  const int n = m.ndof;
  // gvel = Y (M gvel/dt + gforce)                                       (core.py:975-976)
  for (int i = 0; i < n; ++i) {
    double t = 0.;
    for (int j = 0; j < n; ++j) t += AT(b.M, i * n + j) * (AT(b.gvel, j) / dt);
    AT(b.tmp, i) = t + AT(b.gforce, i);
  }
  bool finite = true;
  for (int i = 0; i < n; ++i) {
    double t = 0.;
    for (int j = 0; j < n; ++j) t += AT(b.Y, i * n + j) * AT(b.tmp, j);
    AT(b.tmp, n + i) = t;
    finite = finite && isfinite(t);
  }
  for (int i = 0; i < n; ++i) AT(b.gvel, i) = AT(b.tmp, n + i);
  for (int j = 0; j < m.nj; ++j) {
    const int type = m.jtype[j];
    const int g = m.jgpos[j], d = m.jdof[j];
    if (type == ARB_JOINT_FREE) {
      // gpos = gpos . exp(dt gvel)                                       (joints.py:54-57)
      double q[16], tw[6];
      for (int i = 0; i < 16; ++i) q[i] = AT(b.gpos, g + i);
#pragma unroll
      for (int i = 0; i < 6; ++i) tw[i] = dt * AT(b.gvel, d + i);
      Se3 H, E, R;
      se3_from16(q, H);
      se3_exp(tw, E);
      se3_mul(H, E, R);
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) AT(b.gpos, g + 4 * r + c) = R.R[3 * r + c];
        AT(b.gpos, g + 4 * r + 3) = R.p[r];
      }
      // last row stays [0 0 0 1]
    } else {
      // gpos += dt gvel                                                  (core.py:238-240)
      const int nd = arb_joint_ndof(type);
      for (int i = 0; i < nd; ++i) AT(b.gpos, g + i) += dt * AT(b.gvel, d + i);
    }
  }
  if (!finite) b.status[w] |= ARB_STATUS_NONFINITE;
}

// The fused step, stage by stage.  Same results as the four API phases
// (core.py:1356-1363) but organised for the GPU:
//
//  prepare : kinematics, then -- instead of assembling M, N, B, Z = M/dt + B + N and the
//            explicit 42x42 inverse (core.py:722-734, 813-818) -- the articulated-body
//            elimination of arb_artic.cuh (O(ndof), nothing bigger than a 6x6 block), the
//            unconstrained velocity q_free = Z^-1 (M q'/dt + g), and the constraint problem
//            reduced to "generator" space: constraint Jacobians are
//            J_c = T1_c J_body1 - T0_c J_body0, so with G = stacked body Jacobians of the few
//            bodies that carry constraint frames (the two feet for human36) plus one unit row
//            per limited joint, only  Lambda = G Z^-1 G^T  and  v0 = G q_free  are needed:
//            J_c Y J_d^T = T_c Lambda T_d^T  (core.py:925-927).
//  gs      : the 20 sequential Gauss-Seidel sweeps (core.py:929-935) in generator space,
//            one world per lane; u = v0 + Lambda y is kept up to date, y = sum T_c^T f_c.
//  finish  : q'+ = q_free + Z^-1 G^T y (equals core.py:975-976) by one more articulated
//            solve, and joint integration.
#pragma once
#include "arb_artic.cuh"
#include "arb_constraints.cuh"
#include "arb_world.cuh"

// Per-thread view of the fused scratch: every pointer moved to this world's slot of its tile
// (see FT in arb_artic.cuh).  All double arrays share one record per tile of ARB_TILE worlds
// (frec doubles per world), all int arrays another (firec), so one offset serves each kind.
ARB_D DevBatch fused_tile_view(const DevBatch& b, int64_t w) {
  DevBatch t = b;
  const int64_t tile = w / ARB_TILE, lane = w % ARB_TILE;
  const int64_t od = tile * b.frec * ARB_TILE + lane, oi = tile * b.firec * ARB_TILE + lane;
  t.fq += od; t.fLam += od; t.fv0 += od; t.fT1 += od; t.fT0 += od; t.fu += od; t.fy += od;
  t.fAcc += od; t.fP += od; t.faux += od; t.fpose += od; t.ff += od; t.fRe += od;
  t.aX += od; t.atw += od; t.ath += od; t.aS += od; t.aSh += od; t.aU += od; t.aLA += od;
  t.aLM += od; t.adinv += od; t.aIA += od; t.aIM += od; t.abeta += od; t.au += od; t.ax += od;
  t.aV += od; t.fK += od;
  t.factive += oi; t.fbranch += oi; t.fzidx += oi;
  return t;
}

// Per-constraint update from body poses/twists: activation, aux (sdist / pos0 / q) and the
// maps T1 (from body1's twist) and T0 (from body0's twist) to the constraint rows.
// Returns the active flag.  pose/twist accessors go through P (12 doubles) and TW (6).
// `aligned` (contact of a contact-aligned generator body, arb_model_host.h): instead of the 4x6
// maps only the translation t_c = R_c^T (p_body1 - p_c0) is returned in T1[0..2]; in the frame
// R_e = R_c^T R_body1 the map is rows 2:6 of Ad([I, t_c])  (H_01 Ad(bpose1^-1) = Ad(H_gc0^-1 pose1)).
ARB_D bool constraint_update(const DevModel& m, int c, const Se3& P0, const Se3& P1, const double* TW0,
                             const double* TW1, double q, double dt, double* aux, double* T1,
                             double* T0, int* zidx, bool aligned = false) {
  const int type = m.ctype[c];
  const double* cd = m.cdbl + ARB_CONS_NDBL * c;
  if (type == ARB_CONS_JOINT_LIMITS) {
    aux[0] = q;
    return (q - cd[0] < cd[2]) || (cd[1] - q < cd[2]);
  }
  Se3 bp0, bp1;
  se3_from16(cd, bp0);
  se3_from16(cd + 16, bp1);
  Se3 cb0, cb1;  // frames on the two bodies between which the constraint acts
  int r0, nr;
  bool active;
  if (type == ARB_CONS_BALL_SOCKET) {
    cb0 = bp0; cb1 = bp1; r0 = 3; nr = 3; active = true;
  } else {
    Se3 Hg0, Hgp;
    se3_mul(P0, bp0, Hg0);
    se3_mul(P1, bp1, Hgp);
    Se3 Hc0, Hc1, P0i, P1i, Hc0i, Hc0c1;
    const double sdist = contact_collide(m.cint[ARB_CONS_NINT * c + 2], cd, Hg0, Hgp, Hc0, Hc1, zidx);
    se3_inv(P0, P0i);
    se3_inv(P1, P1i);
    se3_mul(P0i, Hc0, cb0);
    se3_mul(P1i, Hc1, cb1);
    double f0t[6], f1t[6], y[6];
    iad_apply(cb0, TW0, f0t);
    iad_apply(cb1, TW1, f1t);
    se3_inv(Hc0, Hc0i);
    se3_mul(Hc0i, Hc1, Hc0c1);
    ad_apply(Hc0c1, f1t, y);
    const double dsdist = y[5] - f0t[5];
    active = (sdist + dsdist * dt < cd[40]);
    aux[0] = sdist;
    r0 = 2; nr = 4;
    if (!active) return false;
    if (aligned) {
      const double d[3] = {P1.p[0] - Hc0.p[0], P1.p[1] - Hc0.p[1], P1.p[2] - Hc0.p[2]};
      m3t_mulv(Hc0.R, d, T1);
      return true;
    }
  }
  // H_01 = inv(pose0 cb0) (pose1 cb1);  T1 = (Ad(H_01) Ad(cb1^-1))[rows], T0 = Ad(cb0^-1)[rows]
  Se3 F0, F1, F0i, H01;
  se3_mul(P0, cb0, F0);
  se3_mul(P1, cb1, F1);
  se3_inv(F0, F0i);
  se3_mul(F0i, F1, H01);
  if (type == ARB_CONS_BALL_SOCKET) {
#pragma unroll
    for (int i = 0; i < 3; ++i) aux[i] = H01.p[i];
  }
#pragma unroll
  for (int col = 0; col < 6; ++col) {
    double e[6] = {0., 0., 0., 0., 0., 0.}, y[6], z[6];
    e[col] = 1.;
    iad_apply(cb1, e, y);
    ad_apply(H01, y, z);
    for (int r = 0; r < nr; ++r) T1[r * 6 + col] = z[r0 + r];
    iad_apply(cb0, e, y);
    for (int r = 0; r < nr; ++r) T0[r * 6 + col] = y[r0 + r];
  }
  return true;
}

// G applied to the NR solutions of the last articulated solve (x = solutions of the joint-limit
// rows, V of the generator bodies in aV[..][rv0 + r]): out[g * stride + col0 + r] for every generator row g.
template <int NR>
ARB_D void fused_gen_rows(const DevModel& m, const DevBatch& b, int64_t w, const double* x, double* out,
                          int stride, int col0, int rv0 = 0) {
  for (int gj = 0; gj < m.ngen; ++gj) {
    double Re[9];
    const bool al = m.gen_aligned[gj] != 0;
    if (al) {
#pragma unroll
      for (int i = 0; i < 9; ++i) Re[i] = FT(b.fRe, 9 * gj + i);
    }
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      double v[6];
      artic_gen_block(m, b, gj, rv0 + r, al ? Re : nullptr, v);
#pragma unroll
      for (int i = 0; i < 6; ++i) FT(out, (6 * gj + i) * stride + col0 + r) = v[i];
    }
  }
  for (int g = 6 * m.ngen; g < m.ngrows; ++g)
#pragma unroll
    for (int r = 0; r < NR; ++r) FT(out, g * stride + col0 + r) = FT(x, r * m.ndof + m.glimdof[g - 6 * m.ngen]);
}

// ---------------------------------------------------------------------------------------
// prepare: see the header.  Reads the bound state only; writes the fused scratch.
// APPLIED: with the applied-force terms (arb_batch_bind_applied_forces; artic_factor); PARAMS (with
// APPLIED): with the world's body inertia and gravity (arb_batch_bind_body_inertia / _gravity).
template <bool APPLIED = false, bool PARAMS = false>
ARB_D void world_fused_prepare(const DevModel& m, const DevBatch& b, int64_t w, double dt,
                               const DevApplied& ap = DevApplied{nullptr, nullptr, nullptr}) {
  const int NG = m.ngrows;
  artic_kinematics(m, b, w);
  if (!artic_factor<APPLIED, PARAMS>(m, b, w, dt, ap)) b.status[w] |= ARB_STATUS_SINGULAR;
  // frames of the contact-aligned generator bodies: R_e = R_c^T R_body
  for (int gi = 0; gi < m.ngen; ++gi) {
    if (!m.gen_aligned[gi]) continue;
    double Rc[9], Rb[9], Re[9];
    int zi[3];
    zaligned(m.cdbl + ARB_CONS_NDBL * m.gen_c0[gi] + 32, Rc, zi);
#pragma unroll
    for (int i = 0; i < 9; ++i) Rb[i] = FT(b.fpose, (m.gen_body[gi] - 1) * 12 + i);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) Re[3 * i + j] = Rc[i] * Rb[j] + Rc[3 + i] * Rb[3 + j] + Rc[6 + i] * Rb[6 + j];
#pragma unroll
    for (int i = 0; i < 9; ++i) FT(b.fRe, 9 * gi + i) = Re[i];
  }
  // constraints: activation, T maps
  bool any = false;
  for (int c = 0; c < m.nc; ++c) {
    const int* ci = m.cint + ARB_CONS_NINT * c;
    const int type = m.ctype[c];
    const int r0 = m.crow[c];
    FT(b.factive, c) = 0;
    FT(b.fbranch, c) = 0;
    if (!ci[3]) continue;
    double aux[4] = {0., 0., 0., 0.}, T1[24], T0[24];
    int zi[3] = {0, 0, 0};
    bool act;
    if (type == ARB_CONS_JOINT_LIMITS) {
      Se3 I;
      se3_identity(I);
      act = constraint_update(m, c, I, I, nullptr, nullptr, ST_LD(b.gpos, ci[2]), dt, aux, T1, T0, zi);
      ST(b.cforce, r0) = 0.;
    } else {
      Se3 P0, P1;
      double TW0[6], TW1[6];
      if (ci[0] == 0) se3_identity(P0); else load_se3(b.fpose, ci[0] - 1, P0);
      if (ci[1] == 0) se3_identity(P1); else load_se3(b.fpose, ci[1] - 1, P1);
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        TW0[i] = (ci[0] == 0) ? 0. : FT(b.atw, (ci[0] - 1) * 6 + i);
        TW1[i] = (ci[1] == 0) ? 0. : FT(b.atw, (ci[1] - 1) * 6 + i);
      }
      const bool aligned = m.caligned[c] != 0;
      act = constraint_update(m, c, P0, P1, TW0, TW1, 0., dt, aux, T1, T0, zi, aligned);
      if (type == ARB_CONS_SOFT_FINGER_PLANE_POINT) {
#pragma unroll
        for (int i = 0; i < 4; ++i) ST(b.cforce, r0 + i) = 0.;
#pragma unroll
        for (int i = 0; i < 3; ++i) FT(b.fzidx, 3 * c + i) = zi[i];
      }
      if (act) {
        if (aligned) {
#pragma unroll
          for (int i = 0; i < 3; ++i) FT(b.fT1, c * 24 + i) = T1[i];
        } else {
          const int nr = arb_cons_ndol(type);
          for (int i = 0; i < nr * 6; ++i) { FT(b.fT1, c * 24 + i) = T1[i]; FT(b.fT0, c * 24 + i) = T0[i]; }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) FT(b.faux, 4 * c + i) = aux[i];
    FT(b.factive, c) = act ? 1 : 0;
    any = any || act;
  }
  // q_free; the first two joint-limit generators (unit generalized forces) ride along in the same
  // root-to-leaf pass
  const int nlim = NG - 6 * m.ngen;
  const int nm = nlim >= 2 ? 2 : 0;
  if (nm == 2) {
    const int ek[2] = {m.glimdof[0], m.glimdof[1]};
    if (any) {
      artic_backward_generators<1>(m, b, w, m.dofbody[ek[0]], ek[0], nullptr, 1);
      artic_backward_generators<1>(m, b, w, m.dofbody[ek[1]], ek[1], nullptr, 2);
    }
    artic_forward_full<false, 2>(m, b, w, b.au, b.fq, any, ek);
  } else {
    artic_forward_full<false, 0>(m, b, w, b.au, b.fq);
  }
  if (!any) return;
  // generator space: v0 = G q_free, Lambda = G Z^-1 G^T (column block by column block)
  // (rows of a contact-aligned body are taken in its frame R_e: G' = blockdiag(R_e, R_e) G)
  fused_gen_rows<1>(m, b, w, b.fq, b.fv0, 1, 0);
  for (int e = 0; e < nm; ++e)
    fused_gen_rows<1>(m, b, w, b.ax + e * m.ndof * ARB_TILE, b.fLam, NG, 6 * m.ngen + e, 1 + e);
#ifndef PREP_GEN_SEPARATE
  // the generator bodies: leaf-to-root per body, then one root-to-leaf pass for all of them
  for (int gi = 0; gi < m.ngen; ++gi) {
    if (m.gen_aligned[gi]) {
      double Re[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) Re[i] = FT(b.fRe, 9 * gi + i);
      artic_backward_generators<6>(m, b, w, m.gen_body[gi], -1, Re, 6 * gi);
    } else {
      artic_backward_generators<6>(m, b, w, m.gen_body[gi], -1, nullptr, 6 * gi);
    }
  }
  artic_forward_generators_all(m, b, w);
  for (int gi = 0; gi < m.ngen; ++gi)
    fused_gen_rows<6>(m, b, w, b.ax + 6 * gi * m.ndof * ARB_TILE, b.fLam, NG, 6 * gi, 6 * gi);
#else
  for (int gi = 0; gi < m.ngen; ++gi) {
    if (m.gen_aligned[gi]) {
      double Re[9];
#pragma unroll
      for (int i = 0; i < 9; ++i) Re[i] = FT(b.fRe, 9 * gi + i);
      artic_solve_generators<6>(m, b, w, m.gen_body[gi], -1, Re);
    } else {
      artic_solve_generators<6>(m, b, w, m.gen_body[gi], -1);
    }
    fused_gen_rows<6>(m, b, w, b.ax, b.fLam, NG, 6 * gi);
  }
#endif
  for (int h = 6 * m.ngen + nm; h < NG; ++h) {
    const int k = m.glimdof[h - 6 * m.ngen];
    artic_solve_generators<1>(m, b, w, m.dofbody[k], k);
    fused_gen_rows<1>(m, b, w, b.ax, b.fLam, NG, h);
  }
}

// ---------------------------------------------------------------------------------------
// Gauss-Seidel in generator space, one world per lane.
//
// The generator rows of ONE body (or one limited dof) are kept in registers while the sweep
// visits the constraints attached to it: u_F (its twist), Lambda_FF (its 6x6 diagonal block)
// and dy_F (the wrench accumulated since the block was loaded).  Rows outside the block are
// brought up to date lazily, when the sweep moves to another body:
//     u[r] += Lambda[r, F] dy_F ,   y[F] += dy_F .
// For human36 the sweep order is 4 contacts of the right foot, 4 of the left foot, 2 knee
// limits (registration order, core.py:929-935): two block switches per sweep instead of a
// 14x6 update through memory per constraint.
#ifdef __CUDA_ARCH__
#define arb_warp_any(pred) (__any_sync(__activemask(), (pred)) != 0)
#else
#define arb_warp_any(pred) (pred)
#endif

// operands of the visit of constraint c: T rows, diagonal block, pseudo-inverse, forces
ARB_D void gs_prefetch_visit(const DevModel& m, const DevBatch& b, int c) {
  const int r0 = m.crow[c];
  const double* Tp = ((m.cgen1[c] < 0) ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
  const double* pA = b.fAcc + r0 * (4 * ARB_TILE);
  const double* pP = b.fP + r0 * (4 * ARB_TILE);
  if (m.caligned[c]) {
#pragma unroll
    for (int i = 0; i < 3; ++i) arb_prefetch(Tp + i * ARB_TILE);
  } else {
#pragma unroll
    for (int i = 0; i < 24; ++i) arb_prefetch(Tp + i * ARB_TILE);
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) { arb_prefetch(pA + i * ARB_TILE); arb_prefetch(pP + i * ARB_TILE); }
}

struct GsCache {
  int g, n;          // first generator row of the cached block and its size (6 or 1); g < 0: empty
  double u[6], dy[6];
  double* L;         // Lambda_FF, element i at L[i * ls]: shared memory on the device ([36][threads],
  int ls;            // conflict-free), a plain array on the host -- 72 registers the visit needs
};
#define GSL(k, i) (k).L[(i) * (k).ls]

// (Cached blocks are the 6 generator rows of a body: joint limits are visited through memory,
// gs_visit_limit, so no other size exists; k.n is 6 whenever k.g >= 0.)
ARB_D void gs_cache_flush(const DevModel& m, const DevBatch& b, int64_t w, GsCache& k) {
  const int NG = m.ngrows;
  if (k.g < 0) return;
  bool any = false;
#pragma unroll
  for (int p = 0; p < 6; ++p) any = any || (k.dy[p] != 0.);
  double* pu = b.fu + k.g * ARB_TILE;
  if (any) {
    // (the accumulated wrench y is not maintained during the sweeps: gs_final_wrench forms it from
    // the final forces, as the reference forms gforce += J^T f, core.py:936-937)
    const double* pl = b.fLam + k.g * ARB_TILE;        // Lambda[r, g + p] = pl[(r NG + p) TILE]
    const int rowstride = NG * ARB_TILE;
    // Rows outside the block, four at a time: the loads of four rows are in flight together
    // (the switch is bound by memory latency), and the loop is NOT unrolled further -- this code
    // sits in the sweep loop, whose instructions must fit the SM's 32 KB instruction cache
    // together with the sliding solve.  Row i of the outside rows is i (< g) or i + 6.
    const int nout = NG - 6;
#pragma unroll 1
    for (int i0 = 0; i0 < nout; i0 += 4) {
      double acc[4], uu[4];
      int rr[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ii = i0 + i < nout ? i0 + i : nout - 1;
        rr[i] = ii < k.g ? ii : ii + 6;
        const double* q = pl + rr[i] * rowstride;
        uu[i] = b.fu[rr[i] * ARB_TILE];       // (in flight with the Lambda rows: one round trip, not two)
        double a = 0.;
#pragma unroll
        for (int p = 0; p < 6; ++p) a += q[p * ARB_TILE] * k.dy[p];
        acc[i] = a;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i0 + i < nout) b.fu[rr[i] * ARB_TILE] = uu[i] + acc[i];
    }
  }
#pragma unroll
  for (int p = 0; p < 6; ++p) pu[p * ARB_TILE] = k.u[p];
  k.g = -1;
}

template <bool WITH_U>
ARB_D void gs_cache_load(const DevModel& m, const DevBatch& b, int64_t w, GsCache& k, int g, int n) {
  const int NG = m.ngrows;
  k.g = g;
  k.n = 6;
  const double* pu = b.fu + g * ARB_TILE;
  const double* pl = b.fLam + (g * NG + g) * ARB_TILE;
  const int rowstride = NG * ARB_TILE;
#pragma unroll
  for (int p = 0; p < 6; ++p) k.dy[p] = 0.;
#pragma unroll
  for (int p = 0; p < 6; ++p) {
    k.u[p] = WITH_U ? pu[p * ARB_TILE] : 0.;
#pragma unroll
    for (int q = 0; q < 6; ++q) GSL(k, 6 * p + q) = pl[q * ARB_TILE];
    pl += rowstride;
  }
}

// Block switch F -> G in one memory round trip (used by the staged Gauss-Seidel).  gs_cache_flush
// followed by gs_cache_load is a chain of three: the flush loads Lambda[r, F] and u[r] of the outside
// rows, stores u[r], and the load then reads the u rows of G back through the L2 (and only then asks
// for Lambda_GG) -- ncu: ~3 000 cycles per switch, showing up at the first use of the new block's u.
// Here the new block's rows are updated in registers and handed over directly (their memory copy is
// not read while the block is cached, and is rewritten when it leaves), Lambda_GG is requested before
// anything else, and the remaining outside rows follow.  Same arithmetic per row, same bits.
ARB_D void gs_cache_switch(const DevModel& m, const DevBatch& b, int64_t w, GsCache& k, int g2, int n2) {
  if (k.g < 0 || g2 < 0) {
    gs_cache_flush(m, b, w, k);
    if (g2 >= 0) gs_cache_load<true>(m, b, w, k, g2, n2);
    return;
  }
  const int NG = m.ngrows, g = k.g;
  const int rowstride = NG * ARB_TILE;
  bool any = false;
#pragma unroll
  for (int p = 0; p < 6; ++p) any = any || (k.dy[p] != 0.);
  double un[6];
  const double* pun = b.fu + g2 * ARB_TILE;
  const double* plg = b.fLam + (g2 * NG + g2) * ARB_TILE;      // Lambda[g2 + p, g2 + q]
  const double* plf = b.fLam + (g2 * NG + g) * ARB_TILE;       // Lambda[g2 + p, g + q]
  double* pu = b.fu + g * ARB_TILE;
#pragma unroll
  for (int p = 0; p < 6; ++p) {
    un[p] = pun[p * ARB_TILE];
#pragma unroll
    for (int q = 0; q < 6; ++q) GSL(k, 6 * p + q) = plg[p * rowstride + q * ARB_TILE];
  }
  if (any) {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double a = 0.;
#pragma unroll
      for (int q = 0; q < 6; ++q) a += plf[p * rowstride + q * ARB_TILE] * k.dy[q];
      un[p] = un[p] + a;
    }
    // the rows outside both blocks, as in gs_cache_flush
    const double* pl = b.fLam + g * ARB_TILE;
    const int nrest = NG - 12;
    const int lo = g < g2 ? g : g2, hi = g < g2 ? g2 : g;
#pragma unroll 1
    for (int i0 = 0; i0 < nrest; i0 += 4) {
      double acc[4];
      int rr[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int r = i0 + i < nrest ? i0 + i : nrest - 1;
        if (r >= lo) r += 6;
        if (r >= hi) r += 6;
        rr[i] = r;
        const double* q = pl + r * rowstride;
        const double uu = b.fu[r * ARB_TILE];
        double a = 0.;
#pragma unroll
        for (int p = 0; p < 6; ++p) a += q[p * ARB_TILE] * k.dy[p];
        acc[i] = uu + a;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i0 + i < nrest) b.fu[rr[i] * ARB_TILE] = acc[i];
    }
  }
#pragma unroll
  for (int p = 0; p < 6; ++p) pu[p * ARB_TILE] = k.u[p];
#pragma unroll
  for (int p = 0; p < 6; ++p) { k.u[p] = un[p]; k.dy[p] = 0.; }
  k.g = g2;
  k.n = 6;
}

// one visit of a constraint that touches TWO generator bodies (e.g. a ball-and-socket joint
// between two moving bodies): everything through memory.  FRIC: a contact's mu is the world's, in aux[2]
// (world_friction_gather), not the model's.
template <bool FRIC = false>
ARB_NOINLINE void gs_visit_two_body(const DevModel& m, const DevBatch& b, int64_t w, int c, double dt, int* status) {
  const int NG = m.ngrows;
  const int type = m.ctype[c];
  const double* cd = m.cdbl + ARB_CONS_NDBL * c;
  const int r0 = m.crow[c];
  const int g1 = m.cgen1[c], g0 = m.cgen0[c];
  const int nd = arb_cons_ndol(type);
  double v[4], f[4], df[4];
  for (int i = 0; i < nd; ++i) {
    double acc = 0.;
    if (g1 >= 0)
#pragma unroll
      for (int p = 0; p < 6; ++p) acc += FT(b.fT1, c * 24 + i * 6 + p) * FT(b.fu, g1 + p);
    if (g0 >= 0)
#pragma unroll
      for (int p = 0; p < 6; ++p) acc -= FT(b.fT0, c * 24 + i * 6 + p) * FT(b.fu, g0 + p);
    v[i] = acc;
    f[i] = FT(b.ff, r0 + i);
  }
  if (type == ARB_CONS_BALL_SOCKET) {
    double rhs3[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) rhs3[i] = v[i] + FT(b.faux, 4 * c + i) / dt;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double t = 0.;
#pragma unroll
      for (int j = 0; j < 3; ++j) t += FT(b.fP, r0 * 4 + 3 * i + j) * rhs3[j];
      df[i] = -t;
      FT(b.ff, r0 + i) = f[i] + df[i];
    }
  } else {
    double A4[16], P4[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { A4[i] = FT(b.fAcc, r0 * 4 + i); P4[i] = FT(b.fP, r0 * 4 + i); }
    const double mu = FRIC ? FT(b.faux, 4 * c + 2) : cd[36];
    const int br = softfinger_solve(v, A4, P4, FT(b.faux, 4 * c), mu, cd + 37, dt, f, df, status);
#pragma unroll
    for (int i = 0; i < 4; ++i) FT(b.ff, r0 + i) = f[i];
    FT(b.fbranch, c) = br;
  }
  // y += T^T df ; u += Lambda[:, g..g+5] (T^T df)
  for (int s = 0; s < 2; ++s) {
    const int gs = s ? g0 : g1;
    if (gs < 0) continue;
    const double* Ts = s ? b.fT0 : b.fT1;
    const double sign = s ? -1. : 1.;
    double wv[6];
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double acc = 0.;
      for (int i = 0; i < nd; ++i) acc += FT(Ts, c * 24 + i * 6 + p) * df[i];
      wv[p] = sign * acc;
    }
    for (int g = 0; g < NG; ++g) {
      double acc = 0.;
#pragma unroll
      for (int p = 0; p < 6; ++p) acc += FT(b.fLam, g * NG + gs + p) * wv[p];
      FT(b.fu, g) += acc;
    }
  }
}

// Contact-aligned blocks (arb_model_host.h): the cached twist u = [w; v] of the body is expressed
// in the frame R_e, where contact c is the translation t = (pt[0], pt[TILE], pt[2 TILE]):
//   rows [w_z, v_x, v_y, v_z] of Ad([I, t]) u  =  [w_z ; v + t x w]
//   T^T df = [(0, 0, df_0) + df_123 x t ; df_123]
// 3 operands per visit instead of the 24 of a general 4x6 map (read twice).
ARB_D void gs_aligned_rows(const double* pt, const double* u, double* v) {
  const double t0 = pt[0], t1 = pt[ARB_TILE], t2 = pt[2 * ARB_TILE];
  v[0] = u[2];
  v[1] = u[3] + (t1 * u[2] - t2 * u[1]);
  v[2] = u[4] + (t2 * u[0] - t0 * u[2]);
  v[3] = u[5] + (t0 * u[1] - t1 * u[0]);
}
ARB_D void gs_aligned_wrench(const double* pt, const double* df, double* wv) {
  const double t0 = pt[0], t1 = pt[ARB_TILE], t2 = pt[2 * ARB_TILE];
  wv[0] = df[2] * t2 - df[3] * t1;
  wv[1] = df[3] * t0 - df[1] * t2;
  wv[2] = (df[1] * t1 - df[2] * t0) + df[0];
  wv[3] = df[1]; wv[4] = df[2]; wv[5] = df[3];
}
// SoftFingerContact.solve (constraints.py:780-836) on tiled operands: pA / pP point at the 4x4
// diagonal Delassus block and its pseudo-inverse (element i at [i TILE]); they are read where
// they are used so that neither stays in registers across the sliding solve.
// sd_dt = sdist / dt is formed once per step (gs_prologue leaves it in aux[1]), not in every visit;
// with eps = (1, 1, 1) -- the value the reference fixes, constraints.py:423 -- nf / eps is nf exactly
// and the three divisions are skipped: four fp64 divisions less per contact visit, the same bits.
ARB_D int softfinger_solve_tiled(const double* v, const double* pA, const double* pP, double sdist,
                                 double sd_dt, double mu, const double* eps, double dt, double* f,
                                 double* df, int* status) {
  // (only the normal row of A is needed unless the contact slides)
  double vnf3;
  {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += pA[(12 + j) * ARB_TILE] * f[j];
    vnf3 = v[3] - t;
  }
  if (sdist + dt * vnf3 > 0.) {  // separating: release
#pragma unroll
    for (int i = 0; i < 4; ++i) { df[i] = -f[i]; f[i] = 0.; }
    return 1;
  }
  const double rhs[4] = {v[0], v[1], v[2], v[3] + sd_dt};
  double nf[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += -pP[(4 * i + j) * ARB_TILE] * rhs[j];
    df[i] = t;
    nf[i] = f[i] + t;
  }
  double lhs = 0.;
  if (eps[0] == 1. && eps[1] == 1. && eps[2] == 1.) {
#pragma unroll
    for (int i = 0; i < 3; ++i) lhs += nf[i] * nf[i];
  } else {
#pragma unroll
    for (int i = 0; i < 3; ++i) { const double t = nf[i] / eps[i]; lhs += t * t; }
  }
  const double rr = nf[3] * mu;
  if (lhs <= rr * rr) {
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = nf[i];
    return 2;
  }
  // sliding (only some lanes of the warp get here)
#ifdef ARB_X_NOSLIDE   /* timing experiment only (wrong results): what the sliding solves cost */
#pragma unroll
  for (int i = 0; i < 4; ++i) f[i] = nf[i];
  return 3;
#endif
  double A[16], alpha[4];
#pragma unroll
  for (int i = 0; i < 16; ++i) A[i] = pA[i * ARB_TILE];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += A[4 * i + j] * f[j];
    alpha[i] = v[i] - t;
  }
  alpha[3] = vnf3 + sd_dt;
  double newf[4];
  softfinger_sliding(A, alpha, mu, eps, newf, status);
#pragma unroll
  for (int i = 0; i < 4; ++i) { df[i] = newf[i] - f[i]; f[i] = newf[i]; }
  return 3;
}

// one visit of a constraint whose rows depend on ONE generator body (the other frame is on
// the ground): ND rows, block in the cache
// returns the solver branch (soft-finger contacts; 0 otherwise).  FRIC: mu from aux[2], as gs_visit_two_body.
template <int ND, bool FRIC = false>
ARB_D int gs_visit_one_body(const DevModel& m, const DevBatch& b, int64_t w, int c, double dt,
                            GsCache& k, int* status) {
  const double* cd = m.cdbl + ARB_CONS_NDBL * c;
  const int r0 = m.crow[c];
  const bool side0 = m.cgen1[c] < 0;          // the moving body is body0: rows enter with a minus sign
  const double* Tp = (side0 ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
  const double sign = side0 ? -1. : 1.;
  double* pf = b.ff + r0 * ARB_TILE;
  const double* paux = b.faux + c * (4 * ARB_TILE);
  const bool al = ND == 4 && m.caligned[c] != 0;
  int br = 0;
  double v[4], f[ND], df[4];
  if (al) {
    gs_aligned_rows(Tp, k.u, v);
#pragma unroll
    for (int i = 0; i < ND; ++i) f[i] = pf[i * ARB_TILE];
  } else {
#pragma unroll
    for (int i = 0; i < ND; ++i) {
      double acc = 0.;
#pragma unroll
      for (int p = 0; p < 6; ++p) acc += Tp[(i * 6 + p) * ARB_TILE] * k.u[p];
      v[i] = sign * acc;
      f[i] = pf[i * ARB_TILE];
    }
  }
  if (ND == 3) {
    const double* pP = b.fP + r0 * (4 * ARB_TILE);
    double rhs3[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) rhs3[i] = v[i] + paux[i * ARB_TILE] / dt;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double t = 0.;
#pragma unroll
      for (int j = 0; j < 3; ++j) t += pP[(3 * i + j) * ARB_TILE] * rhs3[j];
      df[i] = -t;
      pf[i * ARB_TILE] = f[i] + df[i];
    }
  } else {
    br = softfinger_solve_tiled(v, b.fAcc + r0 * (4 * ARB_TILE), b.fP + r0 * (4 * ARB_TILE),
                                paux[0], paux[ARB_TILE], FRIC ? paux[2 * ARB_TILE] : cd[36], cd + 37, dt, f, df, status);
#pragma unroll
    for (int i = 0; i < ND; ++i) pf[i * ARB_TILE] = f[i];
    b.fbranch[c * ARB_TILE] = br;
  }
  double wv[6];
  if (al) {
    gs_aligned_wrench(Tp, df, wv);
#pragma unroll
    for (int p = 0; p < 6; ++p) k.dy[p] += wv[p];
  } else {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double acc = 0.;
#pragma unroll
      for (int i = 0; i < ND; ++i) acc += Tp[(i * 6 + p) * ARB_TILE] * df[i];
      wv[p] = sign * acc;
      k.dy[p] += wv[p];
    }
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    double acc = 0.;
#pragma unroll
    for (int p = 0; p < 6; ++p) acc += GSL(k, 6 * q + p) * wv[p];
    k.u[q] += acc;
  }
  return br;
}

// diagonal Delassus block A_cc = T Lambda_FF T^T of a one-body constraint and its pseudo-inverse
template <int ND>
ARB_D void gs_diag_one_body(const DevModel& m, const DevBatch& b, int64_t w, int c, const GsCache& k) {
  const int r0 = m.crow[c];
  const double* Tp = ((m.cgen1[c] < 0) ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
  double T[ND * 6], A[ND * ND], P[ND * ND];
#pragma unroll
  for (int i = 0; i < ND * 6; ++i) T[i] = Tp[i * ARB_TILE];
#pragma unroll
  for (int i = 0; i < ND; ++i) {
    double tl[6];
#pragma unroll
    for (int q = 0; q < 6; ++q) {
      double acc = 0.;
#pragma unroll
      for (int p = 0; p < 6; ++p) acc += T[i * 6 + p] * GSL(k, 6 * p + q);
      tl[q] = acc;
    }
#pragma unroll
    for (int j = 0; j < ND; ++j) {
      double acc = 0.;
#pragma unroll
      for (int q = 0; q < 6; ++q) acc += tl[q] * T[j * 6 + q];
      A[i * ND + j] = acc;
    }
  }
  pinv_small<ND>(A, P);
#pragma unroll
  for (int i = 0; i < ND * ND; ++i) { FT(b.fAcc, r0 * 4 + i) = A[i]; FT(b.fP, r0 * 4 + i) = P[i]; }
}

// the same for a contact of a contact-aligned block: T = [e_z^T 0 ; t^ I] is sparse, so
// A_cc = (T Lambda_FF) T^T costs 60 multiply-adds instead of 240 (and a quarter of the code)
ARB_D void gs_diag_aligned(const DevModel& m, const DevBatch& b, int c, const GsCache& k) {
  const int r0 = m.crow[c];
  const double* pt = b.fT1 + c * (24 * ARB_TILE);
  const double t0 = pt[0], t1 = pt[ARB_TILE], t2 = pt[2 * ARB_TILE];
  double W[24], A[16], P[16];
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    W[q] = GSL(k, 12 + q);
    W[6 + q] = (t1 * GSL(k, 12 + q) - t2 * GSL(k, 6 + q)) + GSL(k, 18 + q);
    W[12 + q] = (t2 * GSL(k, q) - t0 * GSL(k, 12 + q)) + GSL(k, 24 + q);
    W[18 + q] = (t0 * GSL(k, 6 + q) - t1 * GSL(k, q)) + GSL(k, 30 + q);
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    A[4 * r] = W[6 * r + 2];
    A[4 * r + 1] = (t1 * W[6 * r + 2] - t2 * W[6 * r + 1]) + W[6 * r + 3];
    A[4 * r + 2] = (t2 * W[6 * r] - t0 * W[6 * r + 2]) + W[6 * r + 4];
    A[4 * r + 3] = (t0 * W[6 * r + 1] - t1 * W[6 * r]) + W[6 * r + 5];
  }
  pinv_small<4>(A, P);
#pragma unroll
  for (int i = 0; i < 16; ++i) { FT(b.fAcc, r0 * 4 + i) = A[i]; FT(b.fP, r0 * 4 + i) = P[i]; }
}

// Start of the Gauss-Seidel of one world: diagonal Delassus blocks and their pseudo-inverses,
// y0 = sum T_c^T f_c (only ball-and-socket forces persist across steps), u = v0 + Lambda y0.
ARB_NOINLINE void gs_prologue(const DevModel& m, const DevBatch& b, int64_t w, double dt) {
  const int NG = m.ngrows;
  GsCache k;       // own cache and block storage: nothing of the caller's escapes into this call,
  double Lp[36];   // so the sweep loop's cache stays in registers
  k.g = -1;
  k.n = 0;
  k.L = Lp;
  k.ls = 1;
  // y0 = sum T_c^T f_c (warm start of ball-and-socket forces), diagonal blocks and pinv
  bool warm = false;
  for (int c = 0; c < m.nc; ++c) {
    if (!FT(b.factive, c)) continue;
    const int type = m.ctype[c];
    const int nd = arb_cons_ndol(type);
    const int r0 = m.crow[c];
    const int g1 = m.cgen1[c], g0 = m.cgen0[c];
    if (type == ARB_CONS_SOFT_FINGER_PLANE_POINT) FT(b.faux, 4 * c + 1) = FT(b.faux, 4 * c) / dt;
    if (type == ARB_CONS_JOINT_LIMITS) {
      const double a = FT(b.fLam, g1 * NG + g1);
      double p;
      pinv_small<1>(&a, &p);
      FT(b.fAcc, r0 * 4) = a;
      FT(b.fP, r0 * 4) = p;
      const double f0 = FT(b.ff, r0);
      if (f0 != 0.) { FT(b.fy, g1) += f0; warm = true; }
      continue;
    }
    if (g1 < 0 || g0 < 0) {
      const int gF = g1 < 0 ? g0 : g1;
      if (k.g != gF) gs_cache_load<false>(m, b, w, k, gF, 6);
      if (nd == 3) gs_diag_one_body<3>(m, b, w, c, k);
      else if (m.caligned[c]) gs_diag_aligned(m, b, c, k);
      else gs_diag_one_body<4>(m, b, w, c, k);
    } else {
      // A_cc = sum over sides s,t of  sign * T_s Lambda[g_s, g_t] T_t^T
      double A[16];
      for (int i = 0; i < nd * nd; ++i) A[i] = 0.;
      for (int s = 0; s < 2; ++s) {
        const int gs = s ? g0 : g1;
        const double* Ts = s ? b.fT0 : b.fT1;
        for (int t = 0; t < 2; ++t) {
          const int gt = t ? g0 : g1;
          const double* Tt = t ? b.fT0 : b.fT1;
          const double sign = (s == t) ? 1. : -1.;
          for (int i = 0; i < nd; ++i) {
            double tl[6];  // row i of T_s Lambda[gs.., gt..]
#pragma unroll
            for (int q = 0; q < 6; ++q) {
              double acc = 0.;
#pragma unroll
              for (int p = 0; p < 6; ++p) acc += FT(Ts, c * 24 + i * 6 + p) * FT(b.fLam, (gs + p) * NG + gt + q);
              tl[q] = acc;
            }
            for (int j = 0; j < nd; ++j) {
              double acc = 0.;
#pragma unroll
              for (int q = 0; q < 6; ++q) acc += tl[q] * FT(Tt, c * 24 + j * 6 + q);
              A[i * nd + j] += sign * acc;
            }
          }
        }
      }
      double P[16];
      if (nd == 3) pinv_small<3>(A, P); else pinv_small<4>(A, P);
      for (int i = 0; i < nd * nd; ++i) { FT(b.fAcc, r0 * 4 + i) = A[i]; FT(b.fP, r0 * 4 + i) = P[i]; }
    }
    if (type == ARB_CONS_BALL_SOCKET) {   // the only forces that persist across steps
      for (int s = 0; s < 2; ++s) {
        const int gs = s ? g0 : g1;
        if (gs < 0) continue;
        const double* Ts = s ? b.fT0 : b.fT1;
        const double sign = s ? -1. : 1.;
#pragma unroll
        for (int p = 0; p < 6; ++p) {
          double acc = 0.;
          for (int i = 0; i < nd; ++i) acc += FT(Ts, c * 24 + i * 6 + p) * FT(b.ff, r0 + i);
          FT(b.fy, gs + p) += sign * acc;
        }
      }
      warm = true;
    }
  }
  // u = v0 + Lambda y0
  for (int g = 0; g < NG; ++g) {
    double t = FT(b.fv0, g);
    if (warm)
      for (int h = 0; h < NG; ++h) {
        const double yh = FT(b.fy, h);
        if (yh != 0.) t += FT(b.fLam, g * NG + h) * yh;
      }
    FT(b.fu, g) = t;
  }
}

// JointLimits.solve (constraints.py:73-90) on the cached 1-row block
// JointLimits visit (constraints.py:35-90).  The generator row of a limited dof is NOT cached: whatever
// block the sweep holds stays where it is.  The row's velocity is its memory copy plus what the cached
// block's pending wrench would add at its flush, u_g = u[g] + Lambda[g, F] dy_F (6 loads), and the
// force increment goes straight into u: the rows of the cached block in registers, the others in memory
// (u[r] += Lambda[r, g] df).  Round 2 cached the row as a 1-row block, which made every limit two block
// switches (flush the body's block: 8 rows x 6 loads + stores, load the row, flush it again: 13 rows,
// reload the body's block: 42 loads) -- four switches per sweep for human36's two feet and two knees
// where two are needed, each a chain of three memory round trips.
ARB_D void gs_visit_limit(const DevModel& m, const DevBatch& b, int c, double dt, GsCache& k) {
  const int NG = m.ngrows;
  const double* cd = m.cdbl + ARB_CONS_NDBL * c;
  const int r0 = m.crow[c];
  const int g = m.cgen1[c];
  const int rowstride = NG * ARB_TILE;
  const double a = FT(b.fAcc, r0 * 4), p = FT(b.fP, r0 * 4);
  const double f = FT(b.ff, r0), q = FT(b.faux, 4 * c);
  double v = FT(b.fu, g);
  if (k.g >= 0) {
    bool any = false;
#pragma unroll
    for (int i = 0; i < 6; ++i) any = any || (k.dy[i] != 0.);
    if (any) {
      const double* pl = b.fLam + (g * NG + k.g) * ARB_TILE;
      double acc = 0.;
#pragma unroll
      for (int i = 0; i < 6; ++i)
        acc += pl[i * ARB_TILE] * k.dy[i];
      v = v + acc;
    }
  }
  const double pred = q + dt * (v - a * f);
  double nf;
  int br;
  if (pred <= cd[0]) { nf = p * ((cd[0] - pred) / dt); br = 2; }
  else if (cd[1] <= pred) { nf = p * ((cd[1] - pred) / dt); br = 3; }
  else { nf = 0.; br = 1; }
  const double df = nf - f;
  FT(b.ff, r0) = nf;
  FT(b.fbranch, c) = br;
  if (df != 0.) {
    const double* col = b.fLam + g * ARB_TILE;          // Lambda[r, g] = col[r rowstride]
    const int kg = k.g, kn = k.g >= 0 ? 6 : 0;
    if (kg >= 0) {
#pragma unroll
      for (int i = 0; i < 6; ++i) k.u[i] += col[(kg + i) * rowstride] * df;
    }
    const int nout = NG - kn;
#pragma unroll 1
    for (int i0 = 0; i0 < nout; i0 += 4) {
      double lam[4], uu[4];
      int rr[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ii = i0 + i < nout ? i0 + i : nout - 1;
        rr[i] = (kn > 0 && ii >= kg) ? ii + kn : ii;
        lam[i] = col[rr[i] * rowstride];
        uu[i] = b.fu[rr[i] * ARB_TILE];
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i0 + i < nout) b.fu[rr[i] * ARB_TILE] = uu[i] + lam[i] * df;
    }
  }
}

// y = sum_c T_c^T f_c from the FINAL constraint forces (generator-space image of the reference's
// gforce += J^T f, core.py:936-937): what the finish stage solves with.
ARB_D void gs_final_wrench(const DevModel& m, const DevBatch& b) {
  const int NG = m.ngrows;
  for (int g = 0; g < NG; ++g) FT(b.fy, g) = 0.;
  for (int c = 0; c < m.nc; ++c) {
    if (!FT(b.factive, c)) continue;
    const int type = m.ctype[c];
    const int r0 = m.crow[c];
    if (type == ARB_CONS_JOINT_LIMITS) {
      FT(b.fy, m.cgen1[c]) += FT(b.ff, r0);
      continue;
    }
    const int nd = arb_cons_ndol(type);
    double f[4] = {0., 0., 0., 0.};
    for (int i = 0; i < nd; ++i) f[i] = FT(b.ff, r0 + i);
    for (int s = 0; s < 2; ++s) {
      const int gs = s ? m.cgen0[c] : m.cgen1[c];
      if (gs < 0) continue;
      const double* Ts = (s ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
      double wv[6];
      if (m.caligned[c]) {
        gs_aligned_wrench(Ts, f, wv);
      } else {
        const double sign = s ? -1. : 1.;
#pragma unroll
        for (int p = 0; p < 6; ++p) {
          double acc = 0.;
          for (int i = 0; i < nd; ++i) acc += Ts[(i * 6 + p) * ARB_TILE] * f[i];
          wv[p] = sign * acc;
        }
      }
#pragma unroll
      for (int p = 0; p < 6; ++p) FT(b.fy, gs + p) += wv[p];
    }
  }
}

#ifdef ARB_HOSTTEST_COUNTERS
static unsigned* arb_dbg_slidemask = nullptr;   // host unit tests only: [W][sweeps] mask of contacts that slid
#endif
// Returns the world's sort key for the next steps (arb_fused.cu): contacts that took the sliding
// branch in some sweep (high part) and active constraints (low part), first 32 constraints.
ARB_D unsigned long long gs_sort_key(const DevModel& m, unsigned slid, unsigned amask) {
  const int nb = m.nc < 32 ? m.nc : 32;
  return ((unsigned long long)slid << nb) | (unsigned long long)amask;
}
// the prepare stage's hand-over (v0 and the diagonal of Lambda) holds a NaN or an Inf
ARB_D bool gs_world_nonfinite(const DevModel& m, const DevBatch& b) {
  const int NG = m.ngrows;
  double chk = 0.;
  for (int g = 0; g < NG; ++g) chk += FT(b.fv0, g) + FT(b.fLam, g * NG + g);
  return !isfinite(chk);
}
// Per-world friction (arb_batch_bind_contact_friction): the world's mu of every soft-finger contact,
// or the model's where none is bound, into aux[2] of the contact's scratch, once per step between the
// prepare and the Gauss-Seidel stage.  The sweeps then read mu by slot next to sdist (in the staged
// kernel through the same bulk copy) instead of gathering it through perm at every visit.  wp: the
// world's column in fr.mu.
ARB_D void world_friction_gather(const DevModel& m, const DevBatch& b, int64_t wp, const DevFriction& fr) {
  for (int c = 0; c < m.nc; ++c) {
    if (m.ctype[c] != ARB_CONS_SOFT_FINGER_PLANE_POINT) continue;
    const int row = fr.row[c];
    FT(b.faux, 4 * c + 2) = row >= 0 ? arb_ld_state(fr.mu + (int64_t)row * b.W + wp) : m.cdbl[ARB_CONS_NDBL * c + 36];
  }
}

// FRIC: the instantiation that reads each contact's mu from aux[2] (world_friction_gather)
template <bool FRIC = false>
ARB_D unsigned long long world_fused_gs(const DevModel& m, const DevBatch& b, int64_t w, double dt,
                                        double* Lstore, int Lstride) {
  const int NG = m.ngrows;
  int status = 0;
  unsigned slid = 0u;
  bool any = false;
  for (int c = 0; c < m.nc; ++c) any = any || FT(b.factive, c);
  for (int g = 0; g < NG; ++g) FT(b.fy, g) = 0.;
  if (!any) return 0ull;
  // A world whose state has gone non-finite (the uncontrolled humanoid can blow up: the
  // reference's own sliding solve diverges) gets NaN out of the reference too; here it must not
  // cost more than a healthy world: with NaN operands every root finder and the QR fallback of
  // the sliding solve run to their iteration caps in every visit (8 ms per world-step measured,
  // a tail that kept one SM busy for 80 ms).  Flag it and leave: the finish stage propagates the
  // NaN of q_free into the state exactly as the reference's arithmetic would.
  if (gs_world_nonfinite(m, b)) {
    b.status[w] |= ARB_STATUS_NONFINITE;
    return 0ull;
  }
  // constraint forces live in tiled scratch during the sweeps (ball-and-socket rows carry
  // the warm start, the others were reset by the prepare stage)
  for (int r = 0; r < m.nrows; ++r) FT(b.ff, r) = ST_LD(b.cforce, r);
  GsCache k;
  k.g = -1;
  k.n = 0;
  k.L = Lstore;
  k.ls = Lstride;
  gs_prologue(m, b, w, dt);
  // active flags as a bit mask (first 32 constraints; the rest are read from memory)
  unsigned amask = 0u;
  for (int c = 0; c < m.nc && c < 32; ++c)
    if (FT(b.factive, c)) amask |= 1u << c;
#ifndef ARB_X_SWEEPS
#define ARB_X_SWEEPS ARB_GS_SWEEPS   /* timing experiments only */
#endif
  // One walk over (sweep, constraint) pairs plus a final pseudo-visit that only flushes: the
  // block-switch code (flush + load, ~2.5 KB of SASS) exists ONCE -- the sweep loop has to fit
  // the 32 KB instruction cache of the SM together with the sliding solve.
  const int nvis = ARB_X_SWEEPS * m.nc;
  for (int v = 0, c = 0, sweep = 0; v <= nvis; ++v, ++c) {
    if (c == m.nc) { c = 0; ++sweep; }
    const bool last = v == nvis;
    const bool act = !last && (c < 32 ? ((amask >> c) & 1u) != 0u : FT(b.factive, c) != 0);
    // Block switches are decided per WORLD and per RUN of constraints that share a cached block
    // (crunmask): a lane takes part in the switch at the first constraint of a run iff one of ITS
    // OWN constraints in the run is active -- so all the lanes of a warp that need the block switch
    // together (the flush / load code runs once per run and warp), and the sequence of flushes,
    // hence the rounding of the lazily updated rows, depends on the world's own active set alone:
    // results are bit-identical whatever the batch size, the position in the batch or the sorting.
    // (Decided per warp, a lane flushed early whenever a neighbour needed another block:
    // u += L dy1 then u += L dy2 instead of u += L (dy1 + dy2) -- results depended on the warp's
    // composition in the last bits.)
    const bool needs = last || (c < 32 ? (amask & m.crunmask[c]) != 0u : act);
    if (!needs) continue;
    const int type = last ? -1 : m.ctype[c];
    const int g1 = last ? -1 : m.cgen1[c], g0 = last ? -1 : m.cgen0[c];
    // the block this visit needs in the cache: a limited dof (1 row), the moving body of a
    // one-body constraint (6 rows), or none (two-body constraints go through memory; the end)
    int gneed = -1, nneed = 0;
    const bool keep = type == ARB_CONS_JOINT_LIMITS;      // a limit visit works with whatever block is cached
    if (!last && !keep && !(g1 >= 0 && g0 >= 0)) { gneed = g1 < 0 ? g0 : g1; nneed = 6; }
    if (!keep && k.g != gneed) {
      gs_cache_flush(m, b, w, k);
      if (gneed >= 0) gs_cache_load<true>(m, b, w, k, gneed, nneed);
    }
    if (!act) continue;
    {   // operands of the next visit, also from a joint-limit visit and across the end of a sweep
      const int cn = (c + 1 < m.nc) ? c + 1 : 0;
      if (m.ctype[cn] != ARB_CONS_JOINT_LIMITS) gs_prefetch_visit(m, b, cn);
    }
    if (type == ARB_CONS_JOINT_LIMITS) {
      gs_visit_limit(m, b, c, dt, k);
    } else if (gneed < 0) {
      gs_visit_two_body<FRIC>(m, b, w, c, dt, &status);
    } else {
      if (type == ARB_CONS_BALL_SOCKET) gs_visit_one_body<3>(m, b, w, c, dt, k, &status);
      else if (gs_visit_one_body<4, FRIC>(m, b, w, c, dt, k, &status) == 3 && c < 32) slid |= 1u << c;
#ifdef ARB_HOSTTEST_COUNTERS
      if (arb_dbg_slidemask && c < 32 && FT(b.fbranch, c) == 3) arb_dbg_slidemask[w * ARB_GS_SWEEPS + sweep] |= 1u << c;
#endif
    }
  }
  gs_final_wrench(m, b);
  for (int r = 0; r < m.nrows; ++r) ST(b.cforce, r) = FT(b.ff, r);
  if (status) b.status[w] |= status;
  return gs_sort_key(m, slid, amask);
}

// ---------------------------------------------------------------------------------------
// Gauss-Seidel with the contact operands staged in shared memory by TMA (device only).
//
// Same arithmetic, same order as world_fused_gs above.  What changes is where a contact visit finds
// its operands.  In world_fused_gs the 4x4 Delassus block A_cc, its pseudo-inverse, the contact map
// and sdist are ~35 global loads per lane that the L1 prefetch of the previous visit brings no closer
// than the L2 (ncu: their first uses hold a quarter of the stage's stall samples).  Here
//  * the warp walks the (sweep, constraint) sequence in lockstep over a warp-uniform schedule (the
//    constraints SOME world of the warp visits; the active sets do not change during the sweeps, so
//    the schedule is a bit mask formed once) -- lanes whose world does not take part in a visit idle;
//  * the tile layout [W/32][elem][32] makes A_cc, pinv(A_cc), t_c and (sdist, sdist/dt) of the warp's
//    32 worlds contiguous blocks (4 KB, 4 KB, 768 B, 512 B), which one elected lane copies into the
//    warp's shared-memory buffer with cp.async.bulk (TMA, completion on the warp's mbarrier) as soon
//    as every lane has read the operands of the current visit -- before the sliding solves of that
//    visit, one whole visit ahead of their use, holding no registers;
//  * the per-constraint model tables (type, rows, generator block, friction) are one 64-byte record
//    per constraint in shared memory instead of eight dependent look-ups through the L1.
#ifdef __CUDACC__
#ifndef GS_STAGE_PF_F
#define GS_STAGE_PF_F 0
#endif
#ifndef GS_STAGE_COOP_ROOT
#define GS_STAGE_COOP_ROOT 1  /* the sliding lanes of a visit are balloted before the solve and enter it together, the mask goes
                                 down to sliding_root_structured (which then has no early exits, and can share the
                                 sampling search of ARB_SAMPLE_ROOT): gs 7.15 -> 6.93 ms at 262144 worlds, 1.85 -> 1.73 at
                                 32768 with the ballot alone (profiles/ab_r04/r04o_*; 0: A/B builds) */
#endif
#ifndef GS_STAGE_PF_SWITCH
#define GS_STAGE_PF_SWITCH 0  /* 1: the rows of an upcoming block switch's flush prefetched into the L1 (A/B builds) */
#endif
#ifndef GS_STAGE_SWITCH
#define GS_STAGE_SWITCH 0     /* 0: flush, then load; 1: one round trip (gs_cache_switch); 2: Lambda_GG requested before the flush (A/B builds) */
#endif
struct GsDesc {           // one constraint, as the sweep loop needs it (shared memory, filled once per CTA)
  int type, g1, g0, row;
  int aligned, gneed, nneed, staged;
  double mu, eps[3];
};
#define GS_STAGE_AP_BYTES (2 * 16 * ARB_TILE * 8)      /* A_cc, pinv(A_cc) */
#define GS_STAGE_T_BYTES (3 * ARB_TILE * 8)            /* t_c of an aligned contact, double-buffered */
// aux rows: sdist, sdist / dt, and with FRIC the world's mu (world_friction_gather)
template <bool FRIC> __host__ __device__ constexpr unsigned gs_stage_aux_rows() { return FRIC ? 3u : 2u; }
template <bool FRIC> __host__ __device__ constexpr unsigned gs_stage_aux_bytes() { return gs_stage_aux_rows<FRIC>() * ARB_TILE * 8; }
template <bool FRIC> __host__ __device__ constexpr unsigned gs_stage_warp_bytes() {
  return GS_STAGE_AP_BYTES + 2 * GS_STAGE_T_BYTES + gs_stage_aux_bytes<FRIC>();
}
struct GsStage {
  double* buf;          // the warp's staging buffer: A (16 rows of 32 lanes), P (16), aux (2, or 3 with FRIC), T (2 x 3)
  unsigned buf_s;       // ... its shared-space address
  unsigned bar_s;       // shared-space address of the warp's mbarrier (one arrival per refill)
  unsigned parity;      // phase the next wait looks for (warp-uniform)
  unsigned tsel;        // which T buffer the CURRENT visit reads (warp-uniform)
  unsigned lane;
  const GsDesc* desc;   // [nc] in shared memory
  const double* const* wbase;   // [5] in shared memory: lane 0's pointers into the warp's tile (fAcc, fP, faux, fT1, fT0)
};
__device__ __forceinline__ void gs_bulk_g2s(unsigned dst_s, const double* src, unsigned bytes, unsigned bar_s) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_s), "l"(src), "r"(bytes), "r"(bar_s) : "memory");
}
// refill for constraint c; tnext: the T buffer the visit of c will read.  One lane issues; the source
// addresses come from the warp's tile pointers in shared memory (assembling them from the lane's own
// view -- spilled 64-bit pointers minus the lane index -- was 95 instructions per visit, 7 % of the kernel's)
template <bool FRIC>
__device__ __forceinline__ void gs_stage_issue(const GsStage& st, int c, unsigned tnext) {
  const unsigned AUXB = gs_stage_aux_bytes<FRIC>();
  const GsDesc& d = st.desc[c];
  const unsigned tb = d.aligned ? (unsigned)GS_STAGE_T_BYTES : 0u;
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
               ::"r"(st.bar_s), "r"((unsigned)(GS_STAGE_AP_BYTES + AUXB) + tb) : "memory");
  gs_bulk_g2s(st.buf_s, st.wbase[0] + d.row * (4 * ARB_TILE), 16 * ARB_TILE * 8, st.bar_s);
  gs_bulk_g2s(st.buf_s + 16 * ARB_TILE * 8, st.wbase[1] + d.row * (4 * ARB_TILE), 16 * ARB_TILE * 8, st.bar_s);
  gs_bulk_g2s(st.buf_s + GS_STAGE_AP_BYTES, st.wbase[2] + c * (4 * ARB_TILE), AUXB, st.bar_s);
  if (d.aligned)
    gs_bulk_g2s(st.buf_s + GS_STAGE_AP_BYTES + AUXB + tnext * GS_STAGE_T_BYTES,
                st.wbase[d.g1 < 0 ? 4 : 3] + c * (24 * ARB_TILE), GS_STAGE_T_BYTES, st.bar_s);
}
__device__ __forceinline__ void gs_stage_wait(const GsStage& st) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "GS_STAGE_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@!p bra GS_STAGE_WAIT_%=;\n"
      "}\n" ::"r"(st.bar_s), "r"(st.parity) : "memory");
}

// SoftFingerContact.solve up to the sliding solve (softfinger_solve_tiled, first part): returns 1
// (separating), 2 (static) with f, df updated, or 3 with the sliding problem (A, alpha) copied out of
// the staging buffer -- the caller releases the buffer, then solves.
__device__ __forceinline__ int softfinger_begin_tiled(const double* v, const double* pA, const double* pP, double sdist,
                                                      double sd_dt, double mu, const double* eps, double dt, double* f,
                                                      double* df, double* A, double* alpha) {
  double vnf3;
  {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += pA[(12 + j) * ARB_TILE] * f[j];
    vnf3 = v[3] - t;
  }
  if (sdist + dt * vnf3 > 0.) {  // separating: release
#pragma unroll
    for (int i = 0; i < 4; ++i) { df[i] = -f[i]; f[i] = 0.; }
    return 1;
  }
  const double rhs[4] = {v[0], v[1], v[2], v[3] + sd_dt};
  double nf[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += -pP[(4 * i + j) * ARB_TILE] * rhs[j];
    df[i] = t;
    nf[i] = f[i] + t;
  }
  double lhs = 0.;
  if (eps[0] == 1. && eps[1] == 1. && eps[2] == 1.) {
#pragma unroll
    for (int i = 0; i < 3; ++i) lhs += nf[i] * nf[i];
  } else {
#pragma unroll
    for (int i = 0; i < 3; ++i) { const double t = nf[i] / eps[i]; lhs += t * t; }
  }
  const double rr = nf[3] * mu;
  if (lhs <= rr * rr) {
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = nf[i];
    return 2;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) A[i] = pA[i * ARB_TILE];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += A[4 * i + j] * f[j];
    alpha[i] = v[i] - t;
  }
  alpha[3] = vnf3 + sd_dt;
  return 3;
}

// gs_visit_one_body<4> with staged operands.  vmask: the lanes of the warp that take part in this
// visit (all of them are here); cn: the warp's next staged contact (-1: none left).  FRIC: the lane's
// own mu from the staged aux[2] instead of the descriptor's warp-uniform one; read before the refill
// of the buffer, it is the one value of the operands held across the sliding solve.
template <bool PLAIN, bool FRIC>
__device__ __forceinline__ int gs_visit_contact_staged(const DevBatch& b, int c, double dt, GsCache& k, int* status,
                                                       const GsStage& st, unsigned vmask, int cn) {
  const GsDesc& d = st.desc[c];
  const bool side0 = d.g1 < 0;
  const double* Tg = (side0 ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
  const double sign = side0 ? -1. : 1.;
  double* pf = b.ff + d.row * ARB_TILE;
  const bool al = PLAIN || d.aligned != 0;
  const double* sA = st.buf + st.lane;
  const double* sP = sA + 16 * ARB_TILE;
  const double* sAux = sA + 32 * ARB_TILE;
  const double* sT = sA + (32 + gs_stage_aux_rows<FRIC>()) * ARB_TILE + st.tsel * (3 * ARB_TILE);
  double v[4], f[4], df[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) f[i] = pf[i * ARB_TILE];
  gs_stage_wait(st);
  if (al) {
    gs_aligned_rows(sT, k.u, v);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double acc = 0.;
#pragma unroll
      for (int p = 0; p < 6; ++p) acc += Tg[(i * 6 + p) * ARB_TILE] * k.u[p];
      v[i] = sign * acc;
    }
  }
  double A[16], alpha[4];
  const double mu = FRIC ? sAux[2 * ARB_TILE] : d.mu;
  int br = softfinger_begin_tiled(v, sA, sP, sAux[0], sAux[ARB_TILE], mu, d.eps, dt, f, df, A, alpha);
  // every lane of the visit has read what it needs of A, P, aux: refill them (and the OTHER T buffer)
  // for the warp's next contact visit while this one's sliding solves run
  __syncwarp(vmask);
  if (cn >= 0 && st.lane == (unsigned)(__ffs(vmask) - 1)) gs_stage_issue<FRIC>(st, cn, st.tsel ^ 1u);
#if GS_STAGE_PF_F
  // the forces of the next contact (written by this lane one sweep ago, read first thing in its visit):
  // into the L1 by an asynchronous copy to the dump row (arb_prefetch_l1)
  if (cn >= 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) arb_prefetch_l1(b.ff + (st.desc[cn].row + i) * ARB_TILE);
  }
#endif
#if GS_STAGE_COOP_ROOT
  const unsigned slmask = __ballot_sync(vmask, br == 3);      // the lanes that solve a sliding problem now
#else
  const unsigned slmask = 0u;
#endif
  if (br == 3) {
    double newf[4];
    softfinger_sliding(A, alpha, FRIC ? mu : d.mu, d.eps, newf, status, slmask);
#pragma unroll
    for (int i = 0; i < 4; ++i) { df[i] = newf[i] - f[i]; f[i] = newf[i]; }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) pf[i * ARB_TILE] = f[i];
  b.fbranch[c * ARB_TILE] = br;
  double wv[6];
  if (al) {
    gs_aligned_wrench(sT, df, wv);
#pragma unroll
    for (int p = 0; p < 6; ++p) k.dy[p] += wv[p];
  } else {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double acc = 0.;
#pragma unroll
      for (int i = 0; i < 4; ++i) acc += Tg[(i * 6 + p) * ARB_TILE] * df[i];
      wv[p] = sign * acc;
      k.dy[p] += wv[p];
    }
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    double acc = 0.;
#pragma unroll
    for (int p = 0; p < 6; ++p) acc += GSL(k, 6 * q + p) * wv[p];
    k.u[q] += acc;
  }
  return br;
}

// fills the CTA's descriptor table (threads c < nc), the caller synchronises the CTA afterwards
__device__ __forceinline__ void gs_desc_fill(const DevModel& m, GsDesc* desc, int c) {
  GsDesc d;
  d.type = m.ctype[c]; d.g1 = m.cgen1[c]; d.g0 = m.cgen0[c]; d.row = m.crow[c];
  d.aligned = m.caligned[c];
  d.gneed = -1; d.nneed = 0;
  if (d.type == ARB_CONS_JOINT_LIMITS) { d.gneed = -2; }      // (-2: keeps whatever block is cached)
  else if (!(d.g1 >= 0 && d.g0 >= 0)) { d.gneed = d.g1 < 0 ? d.g0 : d.g1; d.nneed = 6; }
  // operands through the staging buffer: soft-finger contacts with one moving body
  d.staged = d.type == ARB_CONS_SOFT_FINGER_PLANE_POINT && d.gneed >= 0;
  const double* cd = m.cdbl + ARB_CONS_NDBL * c;
  d.mu = cd[36]; d.eps[0] = cd[37]; d.eps[1] = cd[38]; d.eps[2] = cd[39];
  desc[c] = d;
}

// All 32 lanes of the warp call this together (valid = false: a lane beyond the batch, given the view
// of the last world and kept from writing); m.nc <= 32.
// PLAIN: the model holds nothing but joint limits and contacts of contact-aligned bodies (human36 on a
// ground plane): the instantiation without the general visits (ball-and-socket, two-body constraints,
// 4x6 contact maps), whose code the sweep loop then does not carry through the instruction cache.
// FRIC: the world's contact friction (world_friction_gather), staged with sdist.
template <bool PLAIN, bool FRIC>
__device__ unsigned long long world_fused_gs_staged(const DevModel& m, const DevBatch& b, int64_t w, bool valid, double dt,
                                                    double* Lstore, int Lstride, GsStage& st) {
  const unsigned FULL = 0xffffffffu;
  const int NG = m.ngrows;
  const int nc = m.nc;
  int status = 0;
  unsigned slid = 0u;
  bool live = false;
  if (valid) {
    for (int c = 0; c < nc; ++c) live = live || FT(b.factive, c);
    for (int g = 0; g < NG; ++g) FT(b.fy, g) = 0.;
    if (live && gs_world_nonfinite(m, b)) {      // (see world_fused_gs)
      b.status[w] |= ARB_STATUS_NONFINITE;
      live = false;
    }
  }
  const unsigned wlive = __ballot_sync(FULL, live);
  if (wlive == 0u) return 0ull;
  GsCache k;
  k.g = -1;
  k.n = 0;
  k.L = Lstore;
  k.ls = Lstride;
  // amask: this world's active constraints; nmask: the visits it takes part in (its own, and the
  // block switch at the head of a run of constraints in which it has an active one, see world_fused_gs)
  unsigned amask = 0u, nmask = 0u;
  if (live) {
    for (int r = 0; r < m.nrows; ++r) FT(b.ff, r) = ST_LD(b.cforce, r);
    gs_prologue(m, b, w, dt);
    for (int c = 0; c < nc; ++c)
      if (FT(b.factive, c)) amask |= 1u << c;
    for (int c = 0; c < nc; ++c)
      if ((amask & m.crunmask[c]) != 0u) nmask |= 1u << c;
  }
  unsigned smask = 0u;
  for (int c = 0; c < nc; ++c)
    if (st.desc[c].staged) smask |= 1u << c;
  const unsigned wvis = __reduce_or_sync(FULL, nmask);              // the warp's schedule of a sweep
  const unsigned wmask = __reduce_or_sync(FULL, amask) & smask;     // ... its staged contact visits
  // the prologue wrote A_cc, pinv(A_cc), sdist/dt with ordinary stores: order them before the async proxy's reads
  asm volatile("fence.proxy.async.global;" ::: "memory");
  asm volatile("fence.proxy.async;" ::: "memory");
  __syncwarp();
  st.tsel = 0u;
  if (wmask != 0u && st.lane == (unsigned)(__ffs(wlive) - 1)) gs_stage_issue<FRIC>(st, __ffs(wmask) - 1, 0u);
  for (int sweep = 0; sweep < ARB_X_SWEEPS; ++sweep) {
    for (unsigned mm = wvis; mm != 0u; mm &= mm - 1u) {
      const int c = __ffs(mm) - 1;
      const GsDesc& d = st.desc[c];
      const bool act = ((amask >> c) & 1u) != 0u;
      if (((nmask >> c) & 1u) != 0u && d.gneed != -2 && k.g != d.gneed) {
#if GS_STAGE_SWITCH == 1
        gs_cache_switch(m, b, w, k, d.gneed, d.nneed);
#elif GS_STAGE_SWITCH == 2
        // Lambda_GG is asked for before the flush (the old block's copy is dead by now): its round
        // trip overlaps the flush's instead of following it
        if (d.gneed >= 0) {
          const double* pl = b.fLam + (d.gneed * NG + d.gneed) * ARB_TILE;
          if (d.nneed == 6) {
#pragma unroll
            for (int p = 0; p < 6; ++p)
#pragma unroll
              for (int q = 0; q < 6; ++q) GSL(k, 6 * p + q) = pl[(p * NG + q) * ARB_TILE];
          } else {
            GSL(k, 0) = pl[0];
          }
        }
        gs_cache_flush(m, b, w, k);
        if (d.gneed >= 0) {
          const double* pu = b.fu + d.gneed * ARB_TILE;
          k.g = d.gneed;
          k.n = d.nneed;
#pragma unroll
          for (int p = 0; p < 6; ++p) { k.dy[p] = 0.; k.u[p] = (p < d.nneed) ? pu[p * ARB_TILE] : 0.; }
        }
#else
        gs_cache_flush(m, b, w, k);
        if (d.gneed >= 0) gs_cache_load<true>(m, b, w, k, d.gneed, d.nneed);
#endif
      }
      const unsigned vmask = __ballot_sync(FULL, act);
      if (vmask == 0u) continue;
      const bool staged = ((wmask >> c) & 1u) != 0u;
      int cn = -1;      // the warp's next staged contact visit
      if (staged) {
        const unsigned hi = (wmask >> c) >> 1;
        if (hi != 0u) cn = c + __ffs(hi);
        else if (sweep + 1 < ARB_X_SWEEPS) cn = __ffs(wmask) - 1;
      }
      if (act) {
#if GS_STAGE_PF_SWITCH
        {   // a block switch follows this visit: ask for the rows its flush will read (true L1 prefetch)
          const unsigned rest = (wvis >> c) >> 1;
          const int c2 = rest != 0u ? c + __ffs(rest) : __ffs(wvis) - 1;
          if (st.desc[c2].gneed != d.gneed && k.g >= 0) {
            const int nout = NG - k.n;
            const double* pl = b.fLam + k.g * ARB_TILE;
#pragma unroll 1
            for (int i = 0; i < nout; ++i) {
              const int r = i < k.g ? i : i + k.n;
              const double* q = pl + r * (NG * ARB_TILE);
              if (k.n == 6) {
#pragma unroll
                for (int p = 0; p < 6; ++p) arb_prefetch_l1(q + p * ARB_TILE);
              } else {
                arb_prefetch_l1(q);
              }
            }
          }
        }
#endif
        if (d.type == ARB_CONS_JOINT_LIMITS) {
          gs_visit_limit(m, b, c, dt, k);
        } else if (!PLAIN && d.gneed < 0) {
          gs_visit_two_body<FRIC>(m, b, w, c, dt, &status);
        } else if (!PLAIN && d.type == ARB_CONS_BALL_SOCKET) {
          gs_visit_one_body<3>(m, b, w, c, dt, k, &status);
        } else if (gs_visit_contact_staged<PLAIN, FRIC>(b, c, dt, k, &status, st, vmask, cn) == 3) {
          slid |= 1u << c;
        }
      }
      if (staged) { st.parity ^= 1u; st.tsel ^= 1u; }
    }
  }
  if (!live) return 0ull;
  gs_cache_flush(m, b, w, k);
  gs_final_wrench(m, b);
  for (int r = 0; r < m.nrows; ++r) ST(b.cforce, r) = FT(b.ff, r);
  if (status) b.status[w] |= status;
  return gs_sort_key(m, slid, amask);
}
#endif  // __CUDACC__

// ---------------------------------------------------------------------------------------
// Gauss-Seidel, block-cooperative form (the one the CUDA kernel runs).
//
// Same arithmetic per world as world_fused_gs above, but the worlds of one thread block walk
// the (sweep, constraint) sequence in lockstep and the SLIDING-friction solves of a visit --
// needed by ~20 % of the contacts in steady state, ~5x the cost of the rest of the visit, and
// therefore executed at 3-7 active lanes per warp when each lane solves its own -- are pooled:
// the lanes that need one push (A, alpha, mu) into a shared-memory queue, the block meets at a
// barrier, the first n threads solve the n problems with full warps, a second barrier, and the
// owners pick their forces up.  The order of operations inside each world is unchanged
// (constraint order of core.py:929-935), so results are bit-identical to the per-lane form.
#define ARB_SLIDE_NDBL 21      /* A (16), alpha (4), mu */
struct GsCoop {
  double* q;                 // [ARB_SLIDE_NDBL][cap] problems, element-major
  double* r;                 // [4][cap] new forces
  int* rs;                   // [cap] status bits of each solve
  int* cnt;                  // [2] problem counters, alternating between visits
  unsigned long long* bm;    // [1] OR of the active masks of the block's worlds
  int cap, tid, nthr, parity;
};
ARB_D void coop_sync() {
#ifdef __CUDA_ARCH__
  __syncthreads();
#endif
}
ARB_D int coop_inc(int* p) {
#ifdef __CUDA_ARCH__
  return atomicAdd(p, 1);
#else
  return (*p)++;
#endif
}
ARB_D void coop_or(unsigned long long* p, unsigned long long v) {
#ifdef __CUDA_ARCH__
  if (v) atomicOr(p, v);
#else
  *p |= v;
#endif
}
// barrier, the first n threads solve the n queued problems, barrier
ARB_D void coop_solve_sliding(GsCoop& co, const double* eps) {
  coop_sync();
  const int n = co.cnt[co.parity] < co.cap ? co.cnt[co.parity] : co.cap;
  for (int s = co.tid; s < n; s += co.nthr) {
    double A[16], alpha[4], newf[4];
#pragma unroll
    for (int i = 0; i < 16; ++i) A[i] = co.q[i * co.cap + s];
#pragma unroll
    for (int i = 0; i < 4; ++i) alpha[i] = co.q[(16 + i) * co.cap + s];
    const double mu = co.q[20 * co.cap + s];
    int st = 0;
    softfinger_sliding(A, alpha, mu, eps, newf, &st);
#pragma unroll
    for (int i = 0; i < 4; ++i) co.r[i * co.cap + s] = newf[i];
    co.rs[s] = st;
  }
  if (co.tid == 0) co.cnt[co.parity ^ 1] = 0;
  coop_sync();
  co.parity ^= 1;
}

// soft-finger visit, part 1 (before the pooled solve): returns the branch (1 separating,
// 2 static, 3 sliding: problem queued in *slot); f is updated for branches 1 and 2.  FRIC: mu from
// aux[2] (world_friction_gather); the queue carries it per problem either way.
template <bool FRIC = false>
ARB_D int gs_softfinger_begin(const DevModel& m, const DevBatch& b, int c, double dt, const GsCache& k,
                              GsCoop& co, double* f, double* df, int* slot, int* status) {
  const double* cd = m.cdbl + ARB_CONS_NDBL * c;
  const int r0 = m.crow[c];
  const bool side0 = m.cgen1[c] < 0;
  const double* Tp = (side0 ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
  const double sign = side0 ? -1. : 1.;
  const double* pf = b.ff + r0 * ARB_TILE;
  const double* pA = b.fAcc + r0 * (4 * ARB_TILE);
  const double* pP = b.fP + r0 * (4 * ARB_TILE);
  const double sdist = b.faux[c * (4 * ARB_TILE)];
  const double mu = FRIC ? b.faux[(c * 4 + 2) * ARB_TILE] : cd[36];
  const double* eps = cd + 37;
  double v[4], vnf[4];
  if (m.caligned[c]) {
    gs_aligned_rows(Tp, k.u, v);
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = pf[i * ARB_TILE];
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double acc = 0.;
#pragma unroll
      for (int p = 0; p < 6; ++p) acc += Tp[(i * 6 + p) * ARB_TILE] * k.u[p];
      v[i] = sign * acc;
      f[i] = pf[i * ARB_TILE];
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += pA[(4 * i + j) * ARB_TILE] * f[j];
    vnf[i] = v[i] - t;
  }
  if (sdist + dt * vnf[3] > 0.) {  // separating: release          (constraints.py:781-785)
#pragma unroll
    for (int i = 0; i < 4; ++i) { df[i] = -f[i]; f[i] = 0.; }
    return 1;
  }
  const double sd_dt = b.faux[(c * 4 + 1) * ARB_TILE];
  const double rhs[4] = {v[0], v[1], v[2], v[3] + sd_dt};
  double nf[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += -pP[(4 * i + j) * ARB_TILE] * rhs[j];
    df[i] = t;
    nf[i] = f[i] + t;
  }
  double lhs = 0.;
  if (eps[0] == 1. && eps[1] == 1. && eps[2] == 1.) {
#pragma unroll
    for (int i = 0; i < 3; ++i) lhs += nf[i] * nf[i];
  } else {
#pragma unroll
    for (int i = 0; i < 3; ++i) { const double t = nf[i] / eps[i]; lhs += t * t; }
  }
  const double rr = nf[3] * mu;
  if (lhs <= rr * rr) {            // static friction holds          (constraints.py:795-802)
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = nf[i];
    return 2;
  }
  // sliding: queue (A, alpha, mu)                                  (constraints.py:803-836)
  const int s = coop_inc(&co.cnt[co.parity]);
  *slot = s;
  if (s < co.cap) {
#pragma unroll
    for (int i = 0; i < 16; ++i) co.q[i * co.cap + s] = pA[i * ARB_TILE];
#pragma unroll
    for (int i = 0; i < 3; ++i) co.q[(16 + i) * co.cap + s] = vnf[i];
    co.q[19 * co.cap + s] = vnf[3] + sd_dt;
    co.q[20 * co.cap + s] = mu;
  } else {
    // queue full (more sliding contacts in this visit than it holds): solve in place
    double A[16], newf[4];
#pragma unroll
    for (int i = 0; i < 16; ++i) A[i] = pA[i * ARB_TILE];
    const double alpha[4] = {vnf[0], vnf[1], vnf[2], vnf[3] + sd_dt};
    softfinger_sliding(A, alpha, mu, eps, newf, status);
#pragma unroll
    for (int i = 0; i < 4; ++i) { df[i] = newf[i] - f[i]; f[i] = newf[i]; }
  }
  return 3;
}

// soft-finger visit, part 2: pick up the pooled result, store the force, update the block
ARB_D void gs_softfinger_end(const DevModel& m, const DevBatch& b, int c, GsCache& k, const GsCoop& co,
                             int br, int slot, double* f, double* df, int* status) {
  const int r0 = m.crow[c];
  const bool side0 = m.cgen1[c] < 0;
  const double* Tp = (side0 ? b.fT0 : b.fT1) + c * (24 * ARB_TILE);
  const double sign = side0 ? -1. : 1.;
  double* pf = b.ff + r0 * ARB_TILE;
  if (br == 3 && slot < co.cap) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double nf = co.r[i * co.cap + slot];
      df[i] = nf - f[i];
      f[i] = nf;
    }
    *status |= co.rs[slot];
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) pf[i * ARB_TILE] = f[i];
  b.fbranch[c * ARB_TILE] = br;
  double wv[6];
  if (m.caligned[c]) {
    gs_aligned_wrench(Tp, df, wv);
#pragma unroll
    for (int p = 0; p < 6; ++p) k.dy[p] += wv[p];
  } else {
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      double acc = 0.;
#pragma unroll
      for (int i = 0; i < 4; ++i) acc += Tp[(i * 6 + p) * ARB_TILE] * df[i];
      wv[p] = sign * acc;
      k.dy[p] += wv[p];
    }
  }
#pragma unroll
  for (int q = 0; q < 6; ++q) {
    double acc = 0.;
#pragma unroll
    for (int p = 0; p < 6; ++p) acc += GSL(k, 6 * q + p) * wv[p];
    k.u[q] += acc;
  }
}

// `valid`: this thread has a world (w < W); threads without one only take part in the barriers.
// Supports up to 64 constraints (the active set is a bit mask).  FRIC: as world_fused_gs.
template <bool FRIC = false>
ARB_D unsigned long long world_fused_gs_coop(const DevModel& m, const DevBatch& b, int64_t w, bool valid,
                                             double dt, GsCoop& co, double* Lstore, int Lstride) {
  const int NG = m.ngrows;
  int status = 0;
  unsigned slid = 0u;
  unsigned long long amask = 0ull;
  if (valid) {
    for (int c = 0; c < m.nc; ++c)
      if (FT(b.factive, c)) amask |= 1ull << c;
    for (int g = 0; g < NG; ++g) FT(b.fy, g) = 0.;
  }
  if (valid && amask != 0ull && gs_world_nonfinite(m, b)) {   // see world_fused_gs
    b.status[w] |= ARB_STATUS_NONFINITE;
    amask = 0ull;
  }
  if (co.tid == 0) { *co.bm = 0ull; co.cnt[0] = 0; co.cnt[1] = 0; }
  coop_sync();
  coop_or(co.bm, amask);
  coop_sync();
  const unsigned long long bm = *co.bm;
  if (bm == 0ull) return 0ull;               // no world of this block has an active constraint
  const bool live = amask != 0ull;
  GsCache k;
  k.g = -1;
  k.n = 0;
  k.L = Lstore;
  k.ls = Lstride;
  if (live) {
    for (int r = 0; r < m.nrows; ++r) FT(b.ff, r) = ST_LD(b.cforce, r);
    gs_prologue(m, b, w, dt);
  }
  k.g = -1;
  for (int sweep = 0; sweep < ARB_GS_SWEEPS; ++sweep) {
    for (int c = 0; c < m.nc; ++c) {
      if (!((bm >> c) & 1ull)) continue;     // block-uniform: everybody walks the same sequence
      const bool act = ((amask >> c) & 1ull) != 0ull;
      const int type = m.ctype[c];
      const int g1 = m.cgen1[c], g0 = m.cgen0[c];
      // block switches per world and per run of constraints, as in world_fused_gs
      const bool needs = c < 32 ? (amask & (unsigned long long)m.crunmask[c]) != 0ull : act;
      if (type == ARB_CONS_JOINT_LIMITS) {
        if (act) gs_visit_limit(m, b, c, dt, k);
        continue;
      }
      if (g1 >= 0 && g0 >= 0) {
        if (act) {
          gs_cache_flush(m, b, w, k);
          gs_visit_two_body<FRIC>(m, b, w, c, dt, &status);
        }
        continue;
      }
      const int gF = g1 < 0 ? g0 : g1;
      if (needs && k.g != gF) {
        gs_cache_flush(m, b, w, k);
        gs_cache_load<true>(m, b, w, k, gF, 6);
      }
      if (type == ARB_CONS_BALL_SOCKET) {
        if (act) gs_visit_one_body<3>(m, b, w, c, dt, k, &status);
        continue;
      }
      double f[4], df[4];
      int br = 0, slot = 0;
      if (act) {
        if (c + 1 < m.nc) gs_prefetch_visit(m, b, c + 1);
        br = gs_softfinger_begin<FRIC>(m, b, c, dt, k, co, f, df, &slot, &status);
      }
      coop_solve_sliding(co, m.cdbl + ARB_CONS_NDBL * c + 37);
      if (act) gs_softfinger_end(m, b, c, k, co, br, slot, f, df, &status);
      if (br == 3 && c < 32) slid |= 1u << c;
    }
  }
  if (live) {
    gs_cache_flush(m, b, w, k);
    gs_final_wrench(m, b);
    for (int r = 0; r < m.nrows; ++r) ST(b.cforce, r) = FT(b.ff, r);
    if (status) b.status[w] |= status;
  }
  return gs_sort_key(m, slid, (unsigned)(amask & 0xffffffffull));
}

// ---------------------------------------------------------------------------------------
ARB_D void world_fused_finish(const DevModel& m, const DevBatch& b, int64_t w, double dt) {
  bool any = false;
  for (int c = 0; c < m.nc; ++c) any = any || FT(b.factive, c);
  // q'+ = q_free + Z^-1 G^T y
  if (any) {
    artic_backward_wrenches(m, b, w, b.fy);
    artic_forward_full<true, 0, false>(m, b, w, b.au, b.ax);
  }
  bool finite = true;
  for (int j = 0; j < m.nj; ++j) {
    const int type = m.jtype[j];
    const int g = m.jgpos[j], d = m.jdof[j];
    const int nd = arb_joint_ndof(type);
    double nv[6];
    for (int i = 0; i < nd; ++i) {
      double t = FT(b.fq, d + i);
      if (any) t += FT(b.ax, d + i);
      ST(b.gvel, d + i) = t;
      finite = finite && isfinite(t);
      nv[i] = t;
    }
    if (type == ARB_JOINT_FREE) {
      double q[16], tw[6];
      for (int i = 0; i < 16; ++i) q[i] = ST_LD(b.gpos, g + i);
#pragma unroll
      for (int i = 0; i < 6; ++i) tw[i] = dt * nv[i];
      Se3 H, E, R;
      se3_from16(q, H);
      se3_exp(tw, E);
      se3_mul(H, E, R);
#pragma unroll
      for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) ST(b.gpos, g + 4 * r + c) = R.R[3 * r + c];
        ST(b.gpos, g + 4 * r + 3) = R.p[r];
      }
    } else {
      for (int i = 0; i < nd; ++i) ST(b.gpos, g + i) = ST_LD(b.gpos, g + i) + dt * nv[i];
    }
  }
  if (!finite) b.status[w] |= ARB_STATUS_NONFINITE;
}

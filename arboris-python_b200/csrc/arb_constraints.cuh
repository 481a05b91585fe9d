// Constraints phase, one world per thread: collision + activation, constraint
// Jacobians, Delassus operator, and the 20 sequential Gauss-Seidel sweeps in
// the reference's registration order (parallel only across worlds).
//
// Reference lines followed:
//   World.update_constraints                 core.py:910-937
//   JointLimits.update/is_active/solve       constraints.py:65-90
//   BallAndSocketConstraint.update/jacobian/solve   constraints.py:164-237
//   PointContact.update                      constraints.py:277-295
//   plane/point collision                    collisions.py:105-111, 161-205 (radius 0)
//   zaligned (argsort index work)            homogeneousmatrix.py:201-232
//   SoftFingerContact.jacobian/solve         constraints.py:429-433, 780-836
//   _SubFrame.pose/twist/jacobian            core.py:1017-1032
#pragma once
#include "arb_math.cuh"
#include "arb_smallmat.cuh"
#include "arb_types.h"

#ifndef AT
#define AT(ptr, idx) (ptr)[(int64_t)(idx) * W + w]
#endif

ARB_D void load_pose(const DevBatch& b, int body, int64_t w, Se3& h);
ARB_D void load_twist(const DevBatch& b, int body, int64_t w, double* t);

ARB_D void se3_from_cdbl(const double* d, Se3& h) { se3_from16(d, h); }

// Stable argsort of |z| for 3 elements (numpy.argsort on a length-3 array is an
// insertion sort, hence stable) and the frame zaligned() builds from it.
ARB_D void zaligned(const double* z, double* R, int* idx) {
  double a[3] = {fabs(z[0]), fabs(z[1]), fabs(z[2])};
  int i0 = 0, i1 = 1, i2 = 2, t;
  if (a[i1] < a[i0]) { t = i0; i0 = i1; i1 = t; }
  if (a[i2] < a[i1]) {
    t = i1; i1 = i2; i2 = t;
    if (a[i1] < a[i0]) { t = i0; i0 = i1; i1 = t; }
  }
  idx[0] = i0; idx[1] = i1; idx[2] = i2;
  double x[3];
  x[i0] = 0.;
  x[i1] = z[i2];
  x[i2] = -z[i1];
  double nx = sqrt(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
  x[0] /= nx; x[1] /= nx; x[2] /= nx;
  double y[3];
  cross3(z, x, y);
#pragma unroll
  for (int i = 0; i < 3; ++i) { R[3 * i] = x[i]; R[3 * i + 1] = y[i]; R[3 * i + 2] = z[i]; }
}

// Collision solvers of the point contacts (collisions.py): shape 0 with frame Hg0 (world pose of
// the shape frame), shape 1 with frame Hg1; cd = the constraint's parameters (arboris_b200.h).
// Returns the signed distance and the two contact frames (same orientation zaligned(normal),
// z along the contact normal), exactly as the reference composes them -- including its habit of
// using plane-frame / box-frame coordinates of the normal as world coordinates.
//   pair 0  _plane_sphere_collision   collisions.py:161-205  (Point = radius 0)
//   pair 1  _sphere_sphere_collision  collisions.py:113-159  (Point = radius 0)
//   pair 2  _box_sphere_collision     collisions.py:207-299  (argmin index work at :274)
ARB_D double contact_collide(int pair, const double* cd, const Se3& Hg0, const Se3& Hg1, Se3& Hc0, Se3& Hc1,
                             int* zidx) {
  const double r0 = cd[41], r1 = cd[42];
  double sdist;
  if (pair == ARB_PAIR_SPHERE_SPHERE) {
    double vec[3], nrm = 0.;
#pragma unroll
    for (int i = 0; i < 3; ++i) { vec[i] = Hg1.p[i] - Hg0.p[i]; nrm += vec[i] * vec[i]; }
    nrm = sqrt(nrm);
    sdist = nrm - r0 - r1;
    double normal[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) normal[i] = vec[i] / nrm;
    zaligned(normal, Hc0.R, zidx);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double z = Hc0.R[3 * i + 2];
      Hc0.p[i] = Hg0.p[i] + r0 * z;
      Hc1.p[i] = Hc0.p[i] + sdist * z;
    }
  } else {
    Se3 Hg0i;
    se3_inv(Hg0, Hg0i);
    double p01[3], t3[3];
    m3_mulv(Hg0i.R, Hg1.p, t3);
#pragma unroll
    for (int i = 0; i < 3; ++i) p01[i] = t3[i] + Hg0i.p[i];
    if (pair == ARB_PAIR_BOX_SPHERE) {
      const double* he = cd + 32;
      double f0[3], fg[3], normal[3] = {0., 0., 0.};
      const bool inside = fabs(p01[0]) <= he[0] && fabs(p01[1]) <= he[1] && fabs(p01[2]) <= he[2];
      if (inside) {     // nearest face: argmin over (he - p, he + p), first minimum (numpy.argmin)
        int im = 0;
        double best = he[0] - p01[0];
#pragma unroll
        for (int i = 1; i < 6; ++i) {
          const double v = i < 3 ? he[i] - p01[i] : he[i - 3] + p01[i - 3];
          if (v < best) { best = v; im = i; }
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) f0[i] = p01[i];
        if (im < 3) { f0[im] = he[im]; normal[im] = 1.; }
        else { f0[im - 3] = -he[im - 3]; normal[im - 3] = -1.; }
        m3_mulv(Hg0.R, f0, fg);
        double d2 = 0.;
#pragma unroll
        for (int i = 0; i < 3; ++i) { fg[i] += Hg0.p[i]; const double d = fg[i] - Hg1.p[i]; d2 += d * d; }
        sdist = -sqrt(d2) - r1;
      } else {          // nearest point of the box to the sphere centre
#pragma unroll
        for (int i = 0; i < 3; ++i) f0[i] = fmax(fmin(he[i], p01[i]), -he[i]);
        m3_mulv(Hg0.R, f0, fg);
        double vec[3], nrm = 0.;
#pragma unroll
        for (int i = 0; i < 3; ++i) { fg[i] += Hg0.p[i]; vec[i] = Hg1.p[i] - fg[i]; nrm += vec[i] * vec[i]; }
        nrm = sqrt(nrm);
#pragma unroll
        for (int i = 0; i < 3; ++i) normal[i] = vec[i] / nrm;
        sdist = nrm - r1;
      }
      zaligned(normal, Hc0.R, zidx);
#pragma unroll
      for (int i = 0; i < 3; ++i) { Hc0.p[i] = fg[i]; Hc1.p[i] = Hg1.p[i] - r1 * normal[i]; }
    } else {            // plane (coefficients in the plane's frame) against a sphere / point
      const double* coef = cd + 32;
      const double csdist = (coef[0] * p01[0] + coef[1] * p01[1] + coef[2] * p01[2]) - coef[3];
      sdist = csdist - r1;
      zaligned(coef, Hc0.R, zidx);
      const double sg = sdist > 0. ? 1. : (sdist < 0. ? -1. : 0.);     // numpy.sign
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        Hc0.p[i] = p01[i] - csdist * coef[i];
        Hc1.p[i] = p01[i] - (sg * r1) * coef[i];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) Hc1.R[i] = Hc0.R[i];
  return sdist;
}

// rows [r0, r0+nr) of  Ad(H_01) Ad(bpose1^-1) J_body1  -  Ad(bpose0^-1) J_body0  written to
// the compacted constraint Jacobian starting at row `dol` (rows pre-zeroed).
ARB_D void write_frame_pair_jac(const DevModel& m, const DevBatch& b, int64_t w, int b0, int b1,
                                const Se3& bp0, const Se3& bp1, const Se3& H01, int r0, int nr,
                                int dol) {
  const int64_t W = b.W;
  const int n = m.ndof;
  if (b1 > 0) {
    const int off = m.coloff[b1], kc = m.kcols[b1];
    for (int l = 0; l < kc; ++l) {
      double x[6], y[6], z[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) x[i] = AT(b.J, (off + l) * 6 + i);
      iad_apply(bp1, x, y);
      ad_apply(H01, y, z);
      const int d = m.pathdof[off + l];
      for (int r = 0; r < nr; ++r) AT(b.cjac, (dol + r) * n + d) += z[r0 + r];
    }
  }
  if (b0 > 0) {
    const int off = m.coloff[b0], kc = m.kcols[b0];
    for (int l = 0; l < kc; ++l) {
      double x[6], y[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) x[i] = AT(b.J, (off + l) * 6 + i);
      iad_apply(bp0, x, y);
      const int d = m.pathdof[off + l];
      for (int r = 0; r < nr; ++r) AT(b.cjac, (dol + r) * n + d) -= y[r0 + r];
    }
  }
}

// general solve of the sliding branch: pivoted LU of the 4x4 system (out of line: rare)
ARB_NOINLINE void softfinger_sliding_lu(const double* A, const double* alpha, double s, const double* eps,
                                        double* newf, int* status) {
  double A2[16], nalpha[4];
#pragma unroll
  for (int i = 0; i < 16; ++i) A2[i] = A[i];
#pragma unroll
  for (int i = 0; i < 3; ++i) A2[5 * i] -= s * (1. / (eps[i] * eps[i]));
#pragma unroll
  for (int i = 0; i < 4; ++i) nalpha[i] = -alpha[i];
  if (!solve_small<4>(A2, nalpha, newf)) *status |= ARB_STATUS_SINGULAR;
}

// Sliding branch of SoftFingerContact.solve (constraints.py:803-836): s = smallest real
// eigenvalue <= 0 of B (with the reference's scalar inner products), then
// newf = (A - s diag(eps^-2, 0))^-1 (-alpha).
// coop: see sliding_root_structured (the lanes of the warp that make this call together; 0: unknown)
ARB_NOINLINE void softfinger_sliding(const double* A, const double* alpha, double mu, const double* eps,
                              double* newf, int* status, unsigned coop = 0u) {
  double s = 0.;
  bool found = false;
  const bool unit_eps = (eps[0] == 1. && eps[1] == 1. && eps[2] == 1.);
  if (!(unit_eps && sliding_root_structured(A, alpha, mu, &s, &found, coop))) {
    const double Yc[3] = {A[3], A[7], A[11]};
    const double yn = A[15];
    double beta[3], bb[3];
    const double a = mu / yn * alpha[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      beta[i] = alpha[i] - alpha[3] / yn * Yc[i];
      bb[i] = mu / yn * Yc[i];
    }
    const double ycyc = Yc[0] * Yc[0] + Yc[1] * Yc[1] + Yc[2] * Yc[2];
    const double betab = beta[0] * bb[0] + beta[1] * bb[1] + beta[2] * bb[2];
    const double betabeta = beta[0] * beta[0] + beta[1] * beta[1] + beta[2] * beta[2];
    const double bdotb = bb[0] * bb[0] + bb[1] * bb[1] + bb[2] * bb[2];
    double Bm[36];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const double e2 = eps[i] * eps[i];
        const double yhat = A[4 * i + j] - ycyc / yn;
        Bm[6 * (3 + i) + 3 + j] = e2 * yhat;
        Bm[6 * i + j] = e2 * (yhat + 2. / a * betab);
        // dot(E, scalar) is E*scalar in numpy: these two blocks are DIAGONAL
        Bm[6 * i + 3 + j] = (i == j) ? -(e2 * (betabeta / (a * a))) : 0.;
        Bm[6 * (3 + i) + j] = (i == j) ? e2 * bdotb - 1. : 0.;
      }
    double wr[6], wi[6];
    if (!eig_real_general6(Bm, wr, wi)) *status |= ARB_STATUS_EIG_NOCONV;
    found = false;
    s = 0.;
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (wi[i] == 0. && wr[i] <= 0.) {
        if (!found || wr[i] < s) s = wr[i];
        found = true;
      }
  }
  if (!found) { s = -1e10; *status |= ARB_STATUS_EIG_NOROOT; }
  if (s < -1e10) s = -1e10;
  // newf = (A - s diag(eps^-2, 0))^-1 (-alpha)        (numpy.linalg.solve, constraints.py:834)
  // by elimination of the normal row (its pivot y_n = A[3][3] > 0 is the normal admittance) and
  // Cramer's rule on the 3x3 Schur complement -- a third of the code of the pivoted 4x4 LU, which
  // matters in the sweep loop (instruction cache); the LU is the fallback when the complement
  // is badly scaled.
  double B[9];
  const double idn = 1. / A[15];
  double ie2[3] = {1., 1., 1.};          // eps^-2; with eps = 1 (constraints.py:423) s * 1 is s: no division
  if (!unit_eps) {
#pragma unroll
    for (int i = 0; i < 3; ++i) ie2[i] = 1. / (eps[i] * eps[i]);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      B[3 * i + j] = (A[4 * i + j] - ((i == j) ? s * ie2[i] : 0.)) - (A[4 * i + 3] * idn) * A[12 + j];
  const double rhs[3] = {-alpha[0] + (A[3] * idn) * alpha[3], -alpha[1] + (A[7] * idn) * alpha[3],
                         -alpha[2] + (A[11] * idn) * alpha[3]};
  const double c00 = B[4] * B[8] - B[5] * B[7], c01 = B[5] * B[6] - B[3] * B[8], c02 = B[3] * B[7] - B[4] * B[6];
  const double det = B[0] * c00 + B[1] * c01 + B[2] * c02;
  const double scale = (fabs(B[0]) + fabs(B[4]) + fabs(B[8])) * (1. / 3.);
  if (fabs(det) > 1e-9 * scale * scale * scale && fabs(A[15]) > 0.) {
    const double c10 = B[2] * B[7] - B[1] * B[8], c11 = B[0] * B[8] - B[2] * B[6], c12 = B[1] * B[6] - B[0] * B[7];
    const double c20 = B[1] * B[5] - B[2] * B[4], c21 = B[2] * B[3] - B[0] * B[5], c22 = B[0] * B[4] - B[1] * B[3];
    const double id = 1. / det;
    // x = adj(B) rhs / det,  adj(B)_ij = cofactor_ji
    newf[0] = (c00 * rhs[0] + c10 * rhs[1] + c20 * rhs[2]) * id;
    newf[1] = (c01 * rhs[0] + c11 * rhs[1] + c21 * rhs[2]) * id;
    newf[2] = (c02 * rhs[0] + c12 * rhs[1] + c22 * rhs[2]) * id;
    newf[3] = (-alpha[3] - (A[12] * newf[0] + A[13] * newf[1] + A[14] * newf[2])) * idn;
  } else {
    softfinger_sliding_lu(A, alpha, s, eps, newf, status);
  }
}

// SoftFingerContact.solve (constraints.py:780-836).  v: constraint velocity (4),
// A: 4x4 diagonal block of the Delassus operator, P: its pseudo-inverse, f: force
// (updated), df: returned increment.  Returns the branch id.
ARB_D int softfinger_solve(const double* v, const double* A, const double* P, double sdist,
                           double mu, const double* eps, double dt, double* f, double* df,
                           int* status) {
  double vnf[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += A[4 * i + j] * f[j];
    vnf[i] = v[i] - t;
  }
  if (sdist + dt * vnf[3] > 0.) {  // separating: release
#pragma unroll
    for (int i = 0; i < 4; ++i) { df[i] = -f[i]; f[i] = 0.; }
    return 1;
  }
  // static friction attempt: df = -pinv(A) [v_t, v_n + sdist/dt]
  double rhs[4] = {v[0], v[1], v[2], v[3] + sdist / dt};
  double nf[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double t = 0.;
#pragma unroll
    for (int j = 0; j < 4; ++j) t += -P[4 * i + j] * rhs[j];
    df[i] = t;
    nf[i] = f[i] + t;
  }
  double lhs = 0.;
#pragma unroll
  for (int i = 0; i < 3; ++i) { double t = nf[i] / eps[i]; lhs += t * t; }
  double rr = nf[3] * mu;
  if (lhs <= rr * rr) {
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = nf[i];
    return 2;
  }
  double alpha[4] = {vnf[0], vnf[1], vnf[2], vnf[3] + sdist / dt};
  double newf[4];
  softfinger_sliding(A, alpha, mu, eps, newf, status);
#pragma unroll
  for (int i = 0; i < 4; ++i) { df[i] = newf[i] - f[i]; f[i] = newf[i]; }
  return 3;
}

// FRIC: the friction coefficients of the contacts in fr.row are the world's own
// (arb_batch_bind_contact_friction, fr.mu); the instantiation launched only while they are bound
template <bool FRIC = false>
ARB_D void world_update_constraints(const DevModel& m, const DevBatch& b, int64_t w, double dt,
                                    const DevFriction& fr = DevFriction{nullptr, nullptr}) {
  const int64_t W = b.W;
  const int n = m.ndof;
  int L = 0;
  int status = 0;
  // ---- update(): activation + Jacobian rows (core.py:913-923) ------------------
  for (int c = 0; c < m.nc; ++c) {
    const int type = m.ctype[c];
    const int* ci = m.cint + ARB_CONS_NINT * c;
    const double* cd = m.cdbl + ARB_CONS_NDBL * c;
    const int r0 = m.crow[c];
    const int nd = arb_cons_ndol(type);
    AT(b.cactive, c) = 0;
    AT(b.cbranch, c) = 0;
    AT(b.cdol, c) = -1;
    if (!ci[3]) continue;  // disabled
    bool active = false;
    if (type == ARB_CONS_JOINT_LIMITS) {
      const double q = AT(b.gpos, ci[2]);
      AT(b.cforce, r0) = 0.;
      active = (q - cd[0] < cd[2]) || (cd[1] - q < cd[2]);
      AT(b.caux, 4 * c) = q;
      if (active) {
        for (int j = 0; j < n; ++j) AT(b.cjac, L * n + j) = 0.;
        AT(b.cjac, L * n + ci[1]) = 1.;
      }
    } else if (type == ARB_CONS_BALL_SOCKET) {
      Se3 bp0, bp1, P0, P1, F0, F1, F0i, H01;
      se3_from_cdbl(cd, bp0);
      se3_from_cdbl(cd + 16, bp1);
      load_pose(b, ci[0], w, P0);
      load_pose(b, ci[1], w, P1);
      se3_mul(P0, bp0, F0);
      se3_mul(P1, bp1, F1);
      se3_inv(F0, F0i);
      se3_mul(F0i, F1, H01);
#pragma unroll
      for (int i = 0; i < 3; ++i) AT(b.caux, 4 * c + i) = H01.p[i];
      active = true;
      for (int r = 0; r < 3; ++r)
        for (int j = 0; j < n; ++j) AT(b.cjac, (L + r) * n + j) = 0.;
      write_frame_pair_jac(m, b, w, ci[0], ci[1], bp0, bp1, H01, 3, 3, L);
    } else {
      // shape 0 (frame bp0 on body b0) against shape 1 (frame bp1 on body b1)
      Se3 bp0, bp1, P0, P1, Hg0, Hgp;
      se3_from_cdbl(cd, bp0);
      se3_from_cdbl(cd + 16, bp1);
      load_pose(b, ci[0], w, P0);
      load_pose(b, ci[1], w, P1);
      se3_mul(P0, bp0, Hg0);
      se3_mul(P1, bp1, Hgp);
      Se3 Hc0, Hc1;
      int zi[3];
      const double sdist = contact_collide(ci[2], cd, Hg0, Hgp, Hc0, Hc1, zi);
#pragma unroll
      for (int i = 0; i < 3; ++i) AT(b.czidx, 3 * c + i) = zi[i];
      // contact frames become subframes of their bodies (constraints.py:285-288)
      Se3 P0i, P1i, cb0, cb1, F0, F1, F0i, H01, Hc0i, Hc0c1;
      se3_inv(P0, P0i);
      se3_inv(P1, P1i);
      se3_mul(P0i, Hc0, cb0);
      se3_mul(P1i, Hc1, cb1);
      double T0[6], T1[6], f0t[6], f1t[6], y[6];
      load_twist(b, ci[0], w, T0);
      load_twist(b, ci[1], w, T1);
      iad_apply(cb0, T0, f0t);
      iad_apply(cb1, T1, f1t);
      se3_inv(Hc0, Hc0i);
      se3_mul(Hc0i, Hc1, Hc0c1);
      ad_apply(Hc0c1, f1t, y);
      const double dsdist = y[5] - f0t[5];
      active = (sdist + dsdist * dt < cd[40]);
      AT(b.caux, 4 * c) = sdist;
#pragma unroll
      for (int i = 0; i < 4; ++i) AT(b.cforce, r0 + i) = 0.;
      if (active) {
        se3_mul(P0, cb0, F0);
        se3_mul(P1, cb1, F1);
        se3_inv(F0, F0i);
        se3_mul(F0i, F1, H01);
        for (int r = 0; r < 4; ++r)
          for (int j = 0; j < n; ++j) AT(b.cjac, (L + r) * n + j) = 0.;
        write_frame_pair_jac(m, b, w, ci[0], ci[1], cb0, cb1, H01, 2, 4, L);
      }
    }
    if (active) {
      AT(b.cactive, c) = 1;
      AT(b.cdol, c) = L;
      L += nd;
    }
  }
  // ---- vel = J Y (M gvel/dt + gforce + sum J_c^T f_c),  A = J Y J^T  (core.py:920-927)
  double* rhs = b.tmp;        // [n]
  double* u = b.tmp + n * W;  // [n]
  for (int i = 0; i < n; ++i) {
    double t = 0.;
    for (int j = 0; j < n; ++j) t += AT(b.M, i * n + j) * (AT(b.gvel, j) / dt);
    AT(rhs, i) = t;
  }
  for (int i = 0; i < n; ++i) {
    double g = AT(b.gforce, i);
    for (int c = 0; c < m.nc; ++c) {
      const int dol = AT(b.cdol, c);
      if (dol < 0) continue;
      const int nd = arb_cons_ndol(m.ctype[c]);
      double t = 0.;
      for (int r = 0; r < nd; ++r) t += AT(b.cjac, (dol + r) * n + i) * AT(b.cforce, m.crow[c] + r);
      g += t;
    }
    AT(rhs, i) += g;
  }
  for (int i = 0; i < n; ++i) {
    double t = 0.;
    for (int j = 0; j < n; ++j) t += AT(b.Y, i * n + j) * AT(rhs, j);
    AT(u, i) = t;
  }
  const int LD = m.nrows;  // leading dimension of cA / cT
  for (int r = 0; r < L; ++r) {
    double t = 0.;
    for (int j = 0; j < n; ++j) t += AT(b.cjac, r * n + j) * AT(u, j);
    AT(b.cvel, r) = t;
  }
  for (int i = 0; i < n; ++i)
    for (int r = 0; r < L; ++r) {
      double t = 0.;
      for (int j = 0; j < n; ++j) t += AT(b.Y, i * n + j) * AT(b.cjac, r * n + j);
      AT(b.cT, i * LD + r) = t;
    }
  for (int r = 0; r < L; ++r)
    for (int s = 0; s < L; ++s) {
      double t = 0.;
      for (int j = 0; j < n; ++j) t += AT(b.cjac, r * n + j) * AT(b.cT, j * LD + s);
      AT(b.cA, r * LD + s) = t;
    }
  // pseudo-inverse of each diagonal block: constant over the sweeps
  for (int c = 0; c < m.nc; ++c) {
    const int dol = AT(b.cdol, c);
    if (dol < 0) continue;
    const int type = m.ctype[c];
    const int r0 = m.crow[c];
    if (type == ARB_CONS_JOINT_LIMITS) {
      double a = AT(b.cA, dol * LD + dol), p;
      pinv_small<1>(&a, &p);
      AT(b.cpinv, r0 * 4) = p;
    } else if (type == ARB_CONS_BALL_SOCKET) {
      double a[9], p[9];
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) a[3 * i + j] = AT(b.cA, (dol + i) * LD + dol + j);
      pinv_small<3>(a, p);
      for (int i = 0; i < 9; ++i) AT(b.cpinv, r0 * 4 + i) = p[i];
    } else {
      double a[16], p[16];
      for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) a[4 * i + j] = AT(b.cA, (dol + i) * LD + dol + j);
      pinv_small<4>(a, p);
      for (int i = 0; i < 16; ++i) AT(b.cpinv, r0 * 4 + i) = p[i];
    }
  }
  // ---- Gauss-Seidel: 20 sweeps, fixed (core.py:929-935) ---------------------------
  for (int sweep = 0; sweep < ARB_GS_SWEEPS; ++sweep) {
    for (int c = 0; c < m.nc; ++c) {
      const int dol = AT(b.cdol, c);
      if (dol < 0) continue;
      const int type = m.ctype[c];
      const double* cd = m.cdbl + ARB_CONS_NDBL * c;
      const int r0 = m.crow[c];
      double df[4];
      int nd;
      if (type == ARB_CONS_JOINT_LIMITS) {
        nd = 1;
        const double a = AT(b.cA, dol * LD + dol), p = AT(b.cpinv, r0 * 4);
        const double f = AT(b.cforce, r0), v = AT(b.cvel, dol), q = AT(b.caux, 4 * c);
        const double pred = q + dt * (v - a * f);
        double nf;
        int br;
        if (pred <= cd[0]) { nf = p * ((cd[0] - pred) / dt); br = 2; }
        else if (cd[1] <= pred) { nf = p * ((cd[1] - pred) / dt); br = 3; }
        else { nf = 0.; br = 1; }
        df[0] = nf - f;
        if (br == 1) df[0] = -f;
        AT(b.cforce, r0) = nf;
        AT(b.cbranch, c) = br;
      } else if (type == ARB_CONS_BALL_SOCKET) {
        nd = 3;
        double rhs3[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) rhs3[i] = AT(b.cvel, dol + i) + AT(b.caux, 4 * c + i) / dt;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          double t = 0.;
#pragma unroll
          for (int j = 0; j < 3; ++j) t += AT(b.cpinv, r0 * 4 + 3 * i + j) * rhs3[j];
          df[i] = -t;
          AT(b.cforce, r0 + i) += df[i];
        }
      } else {
        nd = 4;
        double v[4], A4[16], P4[16], f[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          v[i] = AT(b.cvel, dol + i);
          f[i] = AT(b.cforce, r0 + i);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            A4[4 * i + j] = AT(b.cA, (dol + i) * LD + dol + j);
            P4[4 * i + j] = AT(b.cpinv, r0 * 4 + 4 * i + j);
          }
        }
        double mu = cd[36];
        if constexpr (FRIC) {
          const int row = fr.row[c];
          if (row >= 0) mu = fr.mu[(int64_t)row * W + w];
        }
        const int br = softfinger_solve(v, A4, P4, AT(b.caux, 4 * c), mu, cd + 37, dt, f, df, &status);
#pragma unroll
        for (int i = 0; i < 4; ++i) AT(b.cforce, r0 + i) = f[i];
        AT(b.cbranch, c) = br;
      }
      // vel += A[:, rows] df                                              (core.py:935)
      for (int r = 0; r < L; ++r) {
        double t = 0.;
        for (int i = 0; i < nd; ++i) t += AT(b.cA, r * LD + dol + i) * df[i];
        AT(b.cvel, r) += t;
      }
    }
  }
  // ---- gforce += sum J_c^T f_c                                          (core.py:936-937)
  for (int i = 0; i < n; ++i) {
    double g = 0.;
    for (int c = 0; c < m.nc; ++c) {
      const int dol = AT(b.cdol, c);
      if (dol < 0) continue;
      const int nd = arb_cons_ndol(m.ctype[c]);
      double t = 0.;
      for (int r = 0; r < nd; ++r) t += AT(b.cjac, (dol + r) * n + i) * AT(b.cforce, m.crow[c] + r);
      g += t;
    }
    AT(b.gforce, i) += g;
  }
  if (status) b.status[w] |= status;
}

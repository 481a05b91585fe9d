// Closed forms of the nine stock joints: relative pose H_rn, joint Jacobian S
// (6 x ndof, twist of n relative to r in n) and its time derivative dS.
// Device counterpart of arboris/joints.py:10-384; the rotation products are the
// closed forms of arboris/homogeneousmatrix.py:32-199.
#pragma once
#include "arb_math.cuh"
#include "arb_types.h"

struct JointKin {
  Se3 H;          // H_rn(q)
  double S[18];   // S[6*c + r], column-major, up to 3 columns (FreeJoint handled apart)
  double dS[18];
  double T[6];    // T_nr = S dq  (Joint.twist core.py:197-201; FreeJoint joints.py:42-44)
};

ARB_D void joint_kinematics(int type, const double* q, const double* dq, JointKin& k) {
#pragma unroll
  for (int i = 0; i < 18; ++i) { k.S[i] = 0.; k.dS[i] = 0.; }
  se3_identity(k.H);
  double* R = k.H.R;
  switch (type) {
    case ARB_JOINT_FREE: {
      se3_from16(q, k.H);
#pragma unroll
      for (int i = 0; i < 6; ++i) k.T[i] = dq[i];
      return;
    }
    case ARB_JOINT_RZRYRX: {  // joints.py:59-104, rotzyx homogeneousmatrix.py:32-58
      double sz, cz, sy, cy, sx, cx;
      sincos(q[0], &sz, &cz); sincos(q[1], &sy, &cy); sincos(q[2], &sx, &cx);
      R[0] = cz * cy; R[1] = cz * sy * sx - sz * cx; R[2] = cz * sy * cx + sz * sx;
      R[3] = sz * cy; R[4] = sz * sy * sx + cz * cx; R[5] = sz * sy * cx - cz * sx;
      R[6] = -sy;     R[7] = cy * sx;                R[8] = cy * cx;
      double dx = dq[2], dy = dq[1];
      k.S[0] = -sy; k.S[1] = sx * cy; k.S[2] = cx * cy;   // column 0
      k.S[6 + 1] = cx; k.S[6 + 2] = -sx;                  // column 1
      k.S[12 + 0] = 1.;                                   // column 2
      k.dS[0] = -dy * cy;
      k.dS[1] = dx * cx * cy - dy * sx * sy;
      k.dS[2] = -dx * sx * cy - dy * cx * sy;
      k.dS[6 + 1] = -dx * sx; k.dS[6 + 2] = -dx * cx;
      break;
    }
    case ARB_JOINT_RZRY: {  // joints.py:107-146
      double sz, cz, sy, cy;
      sincos(q[0], &sz, &cz); sincos(q[1], &sy, &cy);
      R[0] = cz * cy; R[1] = -sz; R[2] = cz * sy;
      R[3] = sz * cy; R[4] = cz;  R[5] = sz * sy;
      R[6] = -sy;     R[7] = 0.;  R[8] = cy;
      double dy = dq[1];
      k.S[0] = -sy; k.S[2] = cy; k.S[6 + 1] = 1.;
      k.dS[0] = -dy * cy; k.dS[2] = -dy * sy;
      break;
    }
    case ARB_JOINT_RZRX: {  // joints.py:149-185
      double sz, cz, sx, cx;
      sincos(q[0], &sz, &cz); sincos(q[1], &sx, &cx);
      R[0] = cz; R[1] = -sz * cx; R[2] = sz * sx;
      R[3] = sz; R[4] = cz * cx;  R[5] = -cz * sx;
      R[6] = 0.; R[7] = sx;       R[8] = cx;
      double dx = dq[1];
      k.S[1] = sx; k.S[2] = cx; k.S[6 + 0] = 1.;
      k.dS[1] = dx * cx; k.dS[2] = -dx * sx;
      break;
    }
    case ARB_JOINT_RYRX: {  // joints.py:188-224
      double sy, cy, sx, cx;
      sincos(q[0], &sy, &cy); sincos(q[1], &sx, &cx);
      R[0] = cy;  R[1] = sy * sx; R[2] = sy * cx;
      R[3] = 0.;  R[4] = cx;      R[5] = -sx;
      R[6] = -sy; R[7] = cy * sx; R[8] = cy * cx;
      double dx = dq[1];
      k.S[1] = cx; k.S[2] = -sx; k.S[6 + 0] = 1.;
      k.dS[1] = -dx * sx; k.dS[2] = -dx * cx;
      break;
    }
    case ARB_JOINT_RZ: {  // joints.py:227-303
      double s, c;
      sincos(q[0], &s, &c);
      R[0] = c; R[1] = -s; R[3] = s; R[4] = c;
      k.S[2] = 1.;
      break;
    }
    case ARB_JOINT_RY: {  // joints.py:305-326
      double s, c;
      sincos(q[0], &s, &c);
      R[0] = c; R[2] = s; R[6] = -s; R[8] = c;
      k.S[1] = 1.;
      break;
    }
    case ARB_JOINT_RX: {  // joints.py:328-349
      double s, c;
      sincos(q[0], &s, &c);
      R[4] = c; R[5] = -s; R[7] = s; R[8] = c;
      k.S[0] = 1.;
      break;
    }
    case ARB_JOINT_TXTYTZ: {  // joints.py:352-384
      k.H.p[0] = q[0]; k.H.p[1] = q[1]; k.H.p[2] = q[2];
      k.S[3] = 1.; k.S[6 + 4] = 1.; k.S[12 + 5] = 1.;
      break;
    }
    default: break;
  }
  int nd = arb_joint_ndof(type);
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    double t = 0.;
    for (int c = 0; c < nd; ++c) t += k.S[6 * c + r] * dq[c];
    k.T[r] = t;
  }
}

// ---------------------------------------------------------------------------------------
// Per-world inertia of one body (arb_batch_bind_body_inertia): the 10 numbers
// v = [m, m c_x, m c_y, m c_z, I_xx, I_yy, I_zz, I_xy, I_xz, I_yz] placed into the body's 6x6 mass
// matrix ([angular; linear], row-major), M = [[I, skew(m c)], [skew(m c)^T, m 1]], without
// arithmetic; rx = M[0:3,3:6]/M[3,3] or 0 (core.py:1280-1283).  Returns the MASSIVE / HASMASS flags
// by the rules build_host_model (arb_model_host.h) applies to the model's matrices.
ARB_D int body_inertia_matrix(const double* v, double* M, double* rx) {
  const double m = v[0], cx = v[1], cy = v[2], cz = v[3];
  const double Mv[36] = {v[4], v[7], v[8], 0., -cz, cy,
                         v[7], v[5], v[9], cz, 0., -cx,
                         v[8], v[9], v[6], -cy, cx, 0.,
                         0., cz, -cy, m, 0., 0.,
                         -cz, 0., cx, 0., m, 0.,
                         cy, -cx, 0., 0., 0., m};
  int fl = 0;
#pragma unroll
  for (int i = 0; i < 36; ++i) {
    M[i] = Mv[i];
    if (Mv[i] > 0.) fl |= ARB_BODY_MASSIVE;
    if (Mv[i] != 0.) fl |= ARB_BODY_HASMASS;
  }
  const bool light = m <= 1e-10;    // (core.py:1280)
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) rx[3 * r + c] = light ? 0. : Mv[6 * r + 3 + c] / m;
  return fl;
}

// Device-side view of a flattened model and of a batch's memory.
#pragma once
#include <stdint.h>
#include "../../include/arboris_b200.h"

#ifdef __CUDACC__
#define ARB_HDI __host__ __device__ __forceinline__
#else
#define ARB_HDI inline
#endif

ARB_HDI int arb_joint_ndof(int t) {
  return t == ARB_JOINT_FREE ? 6 : (t == ARB_JOINT_RZRYRX || t == ARB_JOINT_TXTYTZ) ? 3
         : (t == ARB_JOINT_RZRY || t == ARB_JOINT_RZRX || t == ARB_JOINT_RYRX) ? 2 : 1;
}
ARB_HDI int arb_joint_ngpos(int t) { return t == ARB_JOINT_FREE ? 16 : arb_joint_ndof(t); }
ARB_HDI int arb_cons_ndol(int t) {
  return t == ARB_CONS_JOINT_LIMITS ? 1 : t == ARB_CONS_BALL_SOCKET ? 3 : 4;
}

#ifndef ARB_TILE
#define ARB_TILE 32          /* worlds per tile of the fused scratch ([W/32][elem][32]) */
#endif

#define ARB_BODY_MASSIVE 1   /* some entry of the mass matrix > 0 (WeightController.init, controllers.py:37) */
#define ARB_BODY_HASMASS 2   /* mass matrix not identically zero */
#define ARB_BODY_HASVISC 4   /* viscosity matrix not identically zero */

// Per-world shared-memory record of the group prepare stage (arb_group.cuh): offsets in doubles.
struct GroupLayout {
  int X, S, Sh, U, LA, LM, dinv, u0;   // what the solves read: X [nj][12]; S, Sh, U, LA, LM [n][6]; 1/d, u [n]
  int kin;                             // kinematics area: pose [nj][12], T [nj][6], theta [nj][6]; dead after the
  int slot;                            //   body terms and aliased with the children slots [nslot][78] of the factorisation
  int ex;                              // exchange buffers of the factorisation (204) + flags (4)
  int ab;                              // body terms [nj][42] (factorisation), aliased with
  int au, av;                          //   reduced right-hand sides [16][maxpath] and branch-point (V, V^) [nvslot][16][12]
  int re;                              // [ngen][9] frames of the contact-aligned generator bodies
  int total;                           // doubles per world (odd, so that two worlds' records do not share banks)
  int nslot, nvslot, maxpath, nlev;
};

// Read-only tables, device (or host, in the CPU unit-test build) pointers.
struct DevModel {
  int ndof, ngpos, nj, nc, na, nrows;
  int ncols;      // sum over bodies of the number of ancestor dofs (packed Jacobian columns)
  int maxk;       // longest root path, in dofs
  int anyvisc;
  const int *jtype, *jparent, *jdof, *jgpos;
  const double *Hpr, *HprInv, *Hcn, *HcnInv;   // [nj][12]  (R row-major, p)
  const int *hcn_ident;                        // [nj]
  const double *bmass, *bvisc;                 // [nj][36]
  const double *brx;                           // [nj][9]  M[0:3,3:6]/M[3,3] or 0 (core.py:1280-1283)
  const int *bflags;                           // [nj]
  const int *coloff;                           // [nj+1] first packed column of body b (b = 0 ground)
  const int *kcols;                            // [nj+1] number of path columns of body b
  const int *pathdof;                          // [ncols] dof of each packed column
  const int *ctype, *cint, *crow;              // constraints
  const double *cdbl;
  const int *atype, *aint;                     // controllers
  const double *adbl, *ablob;
  double up[3];
  // ---- fused path tables -------------------------------------------------------------
  // Z = M/dt + B + N has the tree's sparsity: Z[i][j] != 0 only if dofs i and j lie on a
  // common root path.  dof k sits at position dofpos[k] of the path of body dofbody[k];
  // its ancestors are pathdof[coloff[dofbody[k]] + 0 .. dofpos[k]-1].
  const int *dofbody, *dofpos;                 // [ndof]
  // "generators" of the constraint space: 6 rows (a body twist) per distinct moving body
  // that carries a constraint frame, 1 row per limited joint dof.
  int ngen, ngrows;                            // generator bodies, total rows NG
  const int *gen_body;                         // [ngen]
  const int *cgen1, *cgen0;                    // [nc] first generator row of body1 / body0 (or -1)
  const int *gen_aligned;                      // [ngen] rows kept in the contact-aligned frame (arb_model_host.h)
  const int *gen_c0;                           // [ngen] first contact of an aligned generator (its plane normal)
  const int *caligned;                         // [nc] contact of an aligned generator: T is a translation
  const unsigned *crunmask;                    // [nc] constraints (first 32) visited on the same cached Gauss-Seidel block, consecutively
  // ---- articulated-body tables (arb_artic.cuh) -----------------------------------------
  const int *dofjoint;                         // [ndof] joint of each dof
  const int *jhaschild;                        // [nj] body j+1 has child joints
  const int *jaccfirst;                        // [nj] joint j is the highest-numbered child of its parent body
  const int *jmark;                            // [nj] body j+1 lies on the root path of a generator
  const int *jmarkfirst;                       // [nj] highest-numbered MARKED child of its parent body
  const int *jmarkchild;                       // [nj] body j+1 has marked child joints
  const int *jchild0, *jsib;                   // [nj] first child joint of body j+1 / next sibling joint (-1: none)
  const int *glimdof;                          // [ngrows - 6 ngen] dof of each joint-limit generator row
  const int *doflim;                           // [ndof] the dof carries a joint-limit generator row (its solutions are read back)
  // diagonal PD controllers folded per dof: tau = kp (qd - q) + c, Z[k][k] += dt kp + kd
  int has_pd;
  const double *pd_kp, *pd_kd, *pd_qd, *pd_c, *pd_dqd;  // [ndof]
  const int *pd_gpos;                          // [ndof] gpos index of the dof (or -1)
  const int *pd_index;                         // [ndof] row of the dof in the per-world controller parameters (or -1)
  int npd;                                     // dofs driven by PD controllers (rows of the per-world parameters)
  double gravity;                              // sum of the WeightControllers' gravity
  int nweight;
  // ---- group prepare stage (arb_group.cuh) ------------------------------------------------
  GroupLayout gl;
  const int *glev_off, *glev_joint;            // [nlev + 1], [nj] joints by depth (root-to-leaf scan)
  const int *gslot;                            // [nj] children slot of joint j in the factorisation (or -1: carried / root)
  const int *gvslot;                           // [nj] slot of body j+1's (V, V^) in the forward pass (or -1: never re-read)
};

// Applied forces of a batch (arb_batch_bind_applied_forces), by WORLD index; nullptr: none.  A kernel
// argument of their own, given only to the kernels that add them: in DevBatch they change ptxas's
// register allocation of the Gauss-Seidel kernels, which never read them (more spills, 0.3 % slower).
struct DevApplied {
  const double *tau;     // [ndof][W]     generalized forces (caller-owned)
  const double *wrench;  // [nsel][6][W]  [torque; force] in ground axes at the body origin (caller-owned)
  const int *row;        // [nj]          wrench row of body j+1, or -1 (library-owned table)
};

// Per-batch memory: caller-owned state and the phase-API scratch are [elem][W]; the fused
// scratch (f*, a*) is tiled [W/32][elem][32].
struct DevBatch {
  int64_t W;
  double *gpos, *gvel, *cforce;        // state (bound)
  // per-world PD controller parameters, [npd][W] by WORLD index (arb_batch_bind_controller_params);
  // nullptr: the model's value for every world
  const double *pkp, *pkd, *pqd, *pdqd;
  // update_dynamic outputs
  double *pose;      // [nj][12]
  double *twist;     // [nj][6]
  double *J, *dJ;    // [ncols][6]
  double *M, *N, *B; // [n][n]
  // update_controllers outputs
  double *Z, *Y;     // [n][n]
  double *gforce;    // [n]
  // update_constraints
  double *cjac;      // [nrows][n]   active rows compacted
  double *cvel;      // [nrows]
  double *cA;        // [nrows][nrows]
  double *cT;        // [n][nrows]   Y J^T
  double *cpinv;     // [nrows][4]   pinv of each constraint's diagonal block
  double *caux;      // [nc][4]      sdist / pos0
  double *tmp;       // [2n]
  int *cactive, *cbranch, *cdol, *czidx /*[nc][3]*/;
  int *status;       // [W]
  // ---- fused path (arb_fused.cuh): what the prepare stage hands to the Gauss-Seidel
  // and finish stages, [elem][W] ------------------------------------------------------
  double *fq;        // [n]        velocity without constraint forces  Z^-1 (M gvel/dt + gforce)
  double *fLam;      // [NG][NG]   G Z^-1 G^T
  double *fv0;       // [NG]       G fq
  double *fT1, *fT0; // [nc][24]   d_c x 6 maps from the body twists to the constraint rows
  double *fu, *fy;   // [NG]       generator-space velocity / accumulated wrench
  double *fAcc, *fP; // [nrows][4] diagonal Delassus blocks and their pseudo-inverses
  double *faux;      // [nc][4]
  double *fpose;     // [nj][12]   body poses (for contacts and gravity)
  double *ff;        // [nrows]    constraint forces during the sweeps
  double *fRe;       // [ngen][9]  R_e = R_c^T R_body of the contact-aligned generator bodies
  int *factive, *fbranch;  // [nc]
  int *fzidx;              // [nc][3]  argsort indices of zaligned() of the last prepare stage
  int64_t frec, firec;     // doubles / ints per world in the tiled fused scratch
  // world sorting (arb_fused.cu): the thread (and scratch slot) s works on world perm[s]; the
  // Gauss-Seidel stage leaves a sort key per slot (contacts that slid, active contacts)
  const int *perm;              // [W] slot -> world, or nullptr (identity)
  unsigned long long *fkey;     // [W] by slot, or nullptr
  // ---- articulated-body factorisation of Z (arb_artic.cuh), [elem][W] ------------------
  double *aX;        // [nj][12]   H_pc of each joint
  double *atw, *ath; // [nj][6]    body twist T_b and the accumulated joint term theta_b
  double *aS, *aSh;  // [n][6]     joint axis s_k in the child body frame and s^_k = ds_k - ad(theta) s_k
  double *aU, *aLA, *aLM;  // [n][6]  U_k = IA s_k + IM s^_k ; rows s_k^T IA / d_k, s_k^T IM / d_k
  double *adinv;     // [n]        1 / d_k,  d_k = s_k^T U_k (+ PD diagonal)
  double *aIA, *aIM; // [nj][36]   children's contributions to the articulated matrices of body j+1
  double *abeta;     // [nj][6]    children's contributions to the bias wrench
  double *au;        // [6 ngen][n]     reduced right-hand sides u_k, 6 per generator body
  double *ax;        // [6 ngen][n]     solutions
  double *aV;        // [nj][72 ngen]   (V, V^) of each body for 6 right-hand sides per generator body
  // ---- group prepare stage: K = Z^-1 G^T, the generator solutions over ALL dofs -----------
  double *fK;        // [n][NG]   (tiled like the rest of the fused scratch)
};

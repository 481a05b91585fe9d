// Host-side preprocessing of an arb_model_desc into the tables the kernels read
// (inverse constant frames, packed Jacobian column layout, body flags).  Plain
// C++, shared by the CUDA library (arb_api.cu) and the CPU unit-test build.
#pragma once
#include <cmath>
#include <cstring>
#include <string>
#include <vector>
#include "arb_math.cuh"
#include "arb_types.h"

struct HostModel {
  int ndof = 0, ngpos = 0, nj = 0, nc = 0, na = 0, nrows = 0, ncols = 0, maxk = 0, anyvisc = 0;
  std::vector<int> jtype, jparent, jdof, jgpos, hcn_ident, bflags, coloff, kcols, pathdof;
  std::vector<int> ctype, cint, crow, atype, aint;
  std::vector<int> dofbody, dofpos, gen_body, cgen1, cgen0;
  std::vector<int> gen_aligned, gen_c0, caligned;   // contact-aligned generator blocks (arb_fused.cuh)
  std::vector<int> doflim;
  std::vector<unsigned> crunmask;                   // runs of constraints on one cached Gauss-Seidel block
  int ngen = 0, ngrows = 0;
  // articulated-body tables
  std::vector<int> dofjoint, jhaschild, jaccfirst, jmark, jmarkfirst, jmarkchild, glimdof, pd_gpos;
  std::vector<int> pd_index, pd_dofs;   // per-world controller parameters: dof -> row (or -1), row -> dof
  int has_warm = 0;                     // some constraint force is state across steps (ball and socket)
  std::vector<int> glev_off, glev_joint, gslot, gvslot;   // group prepare stage (arb_group.cuh)
  GroupLayout gl;
  std::vector<int> jchild0, jsib;   // first child joint of body j+1 / next sibling joint (-1: none), ascending
  std::vector<double> pd_kp, pd_kd, pd_qd, pd_c, pd_dqd;
  int has_pd = 0, nweight = 0;
  double gravity = 0.;
  int fused_ok = 1;            // 0: a controller couples dofs in a way the fused step does not support
  std::string fused_why;
  std::vector<double> Hpr, HprInv, Hcn, HcnInv, bmass, bvisc, brx, cdbl, adbl, ablob;
  double up[3] = {0., 1., 0.};
};

static inline void se3_to12(const Se3& h, double* o) {
  for (int i = 0; i < 9; ++i) o[i] = h.R[i];
  for (int i = 0; i < 3; ++i) o[9 + i] = h.p[i];
}

static inline int build_host_model(const arb_model_desc* d, HostModel& m, std::string& err) {
  if (!d) { err = "null model description"; return -1; }
  if (d->njoints < 0 || d->ndof < 0 || d->nconstraints < 0 || d->ncontrollers < 0) {
    err = "negative size in model description"; return -1;
  }
  m.ndof = d->ndof; m.ngpos = d->ngpos; m.nj = d->njoints; m.nc = d->nconstraints;
  m.na = d->ncontrollers; m.nrows = d->nrows;
  const int nj = m.nj;
  m.jtype.assign(d->joint_type, d->joint_type + nj);
  m.jparent.assign(d->joint_parent, d->joint_parent + nj);
  m.jdof.assign(d->joint_dof, d->joint_dof + nj);
  m.jgpos.assign(d->joint_gpos, d->joint_gpos + nj);
  m.Hpr.resize(12 * nj); m.HprInv.resize(12 * nj); m.Hcn.resize(12 * nj); m.HcnInv.resize(12 * nj);
  m.hcn_ident.resize(nj);
  m.bmass.assign(d->body_mass, d->body_mass + 36 * nj);
  m.bvisc.assign(d->body_visc, d->body_visc + 36 * nj);
  m.brx.assign(9 * nj, 0.);
  m.bflags.assign(nj, 0);
  m.coloff.assign(nj + 1, 0);
  m.kcols.assign(nj + 1, 0);
  int ndof = 0, ngpos = 0;
  std::vector<std::vector<int>> path(nj + 1);
  for (int j = 0; j < nj; ++j) {
    const int t = m.jtype[j];
    if (t < 0 || t > ARB_JOINT_TXTYTZ) { err = "unknown joint type"; return -2; }
    const int p = m.jparent[j];
    if (p < 0 || p > j) { err = "joint parent must precede the joint (depth-first order)"; return -2; }
    if (m.jdof[j] != ndof || m.jgpos[j] != ngpos) { err = "dof/gpos offsets are not contiguous"; return -2; }
    ndof += arb_joint_ndof(t);
    ngpos += arb_joint_ngpos(t);
    Se3 h, hi;
    se3_from16(d->joint_Hpr + 16 * j, h);
    se3_inv(h, hi);
    se3_to12(h, &m.Hpr[12 * j]);
    se3_to12(hi, &m.HprInv[12 * j]);
    se3_from16(d->joint_Hcn + 16 * j, h);
    se3_inv(h, hi);
    se3_to12(h, &m.Hcn[12 * j]);
    se3_to12(hi, &m.HcnInv[12 * j]);
    bool ident = true;
    for (int i = 0; i < 16; ++i)
      if (d->joint_Hcn[16 * j + i] != ((i % 5 == 0) ? 1. : 0.)) ident = false;
    m.hcn_ident[j] = ident ? 1 : 0;
    const double* M = &m.bmass[36 * j];
    int fl = 0;
    for (int i = 0; i < 36; ++i) {
      if (M[i] > 0.) fl |= ARB_BODY_MASSIVE;
      if (M[i] != 0.) fl |= ARB_BODY_HASMASS;
      if (m.bvisc[36 * j + i] != 0.) fl |= ARB_BODY_HASVISC;
    }
    if (fl & ARB_BODY_HASVISC) m.anyvisc = 1;
    m.bflags[j] = fl;
    if (!(M[6 * 3 + 3] <= 1e-10))  // core.py:1280
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) m.brx[9 * j + 3 * r + c] = M[6 * r + 3 + c] / M[6 * 3 + 3];
    path[j + 1] = path[p];
    for (int i = 0; i < arb_joint_ndof(t); ++i) path[j + 1].push_back(m.jdof[j] + i);
  }
  if (ndof != m.ndof || ngpos != m.ngpos) { err = "ndof/ngpos do not match the joint list"; return -2; }
  for (int b = 0; b <= nj; ++b) {
    m.coloff[b] = (int)m.pathdof.size();
    m.kcols[b] = (int)path[b].size();
    if (m.kcols[b] > m.maxk) m.maxk = m.kcols[b];
    m.pathdof.insert(m.pathdof.end(), path[b].begin(), path[b].end());
  }
  m.ncols = (int)m.pathdof.size();
  m.ctype.assign(d->cons_type, d->cons_type + m.nc);
  m.cint.assign(d->cons_int, d->cons_int + ARB_CONS_NINT * m.nc);
  m.cdbl.assign(d->cons_dbl, d->cons_dbl + ARB_CONS_NDBL * m.nc);
  m.crow.assign(d->cons_row, d->cons_row + m.nc);
  int rows = 0;
  for (int c = 0; c < m.nc; ++c) {
    const int t = m.ctype[c];
    if (t < 0 || t > ARB_CONS_SOFT_FINGER_PLANE_POINT) { err = "unknown constraint type"; return -3; }
    if (m.crow[c] != rows) { err = "constraint rows are not contiguous"; return -3; }
    rows += arb_cons_ndol(t);
    const int* ci = &m.cint[ARB_CONS_NINT * c];
    if (t == ARB_CONS_BALL_SOCKET) m.has_warm = 1;
    if (t == ARB_CONS_JOINT_LIMITS) {
      if (ci[0] < 0 || ci[0] >= nj || arb_joint_ndof(m.jtype[ci[0]]) != 1) {
        err = "JointLimits needs a 1-dof joint"; return -3;
      }
      if (ci[1] != m.jdof[ci[0]] || ci[2] != m.jgpos[ci[0]]) {
        err = "JointLimits dof / gpos index does not match its joint"; return -3;
      }
    } else if (ci[0] < 0 || ci[0] > nj || ci[1] < 0 || ci[1] > nj) {
      err = "constraint body index out of range"; return -3;
    } else if (t == ARB_CONS_SOFT_FINGER_PLANE_POINT && (ci[2] < 0 || ci[2] > ARB_PAIR_BOX_SPHERE)) {
      err = "unknown contact shape pair"; return -3;
    }
  }
  if (rows != m.nrows) { err = "nrows does not match the constraint list"; return -3; }
  m.atype.assign(d->ctrl_type, d->ctrl_type + m.na);
  m.aint.assign(d->ctrl_int, d->ctrl_int + 4 * m.na);
  m.adbl.assign(d->ctrl_dbl, d->ctrl_dbl + 4 * m.na);
  if (d->nblob > 0) m.ablob.assign(d->ctrl_blob, d->ctrl_blob + d->nblob);
  for (int a = 0; a < m.na; ++a) {
    if (m.atype[a] != ARB_CTRL_WEIGHT && m.atype[a] != ARB_CTRL_PD) { err = "unknown controller type"; return -4; }
    if (m.atype[a] != ARB_CTRL_PD) continue;
    // PD blob: {dof map[m], gpos map[m], kp[m*m], kd[m*m], gpos_des[m], gvel_des[m]}
    const long mm = m.aint[4 * a], off = m.aint[4 * a + 1];
    if (mm < 0 || off < 0 || off + 4 * mm + 2 * mm * mm > (long)d->nblob) {
      err = "PD controller blob out of range"; return -4;
    }
    for (long i = 0; i < mm; ++i) {
      const double kd_ = m.ablob[off + i], kg = m.ablob[off + mm + i];
      if (!(kd_ >= 0. && kd_ < m.ndof && kd_ == (double)(int)kd_) || !(kg >= 0. && kg < m.ngpos && kg == (double)(int)kg)) {
        err = "PD controller dof / gpos index out of range"; return -4;
      }
    }
  }
  for (int i = 0; i < 3; ++i) m.up[i] = d->up[i];
  // fused-path tables
  m.dofbody.assign(m.ndof, 0);
  m.dofpos.assign(m.ndof, 0);
  for (int j = 0; j < nj; ++j)
    for (int i = 0; i < arb_joint_ndof(m.jtype[j]); ++i) {
      m.dofbody[m.jdof[j] + i] = j + 1;
      m.dofpos[m.jdof[j] + i] = m.kcols[m.jparent[j]] + i;
    }
  m.cgen1.assign(m.nc, -1);
  m.cgen0.assign(m.nc, -1);
  std::vector<int> body_gen(nj + 1, -1);
  for (int c = 0; c < m.nc; ++c) {   // 6-row generators first, in order of first use
    if (m.ctype[c] == ARB_CONS_JOINT_LIMITS) continue;
    const int* ci = &m.cint[ARB_CONS_NINT * c];
    for (int side = 1; side >= 0; --side) {
      const int b = ci[side];
      if (b == 0) continue;
      if (body_gen[b] < 0) { body_gen[b] = 6 * (int)m.gen_body.size(); m.gen_body.push_back(b); }
      (side ? m.cgen1 : m.cgen0)[c] = body_gen[b];
    }
  }
  m.ngen = (int)m.gen_body.size();
  m.ngrows = 6 * m.ngen;
  // A generator body is "contact-aligned" when every constraint attached to it is a plane/point
  // soft-finger contact whose plane is carried by the ground and all those planes share one
  // normal: the contact frames of the body then share one orientation R_c (zaligned(normal),
  // collisions.py:200-204), and the Gauss-Seidel keeps the body's rows in the frame
  // R_e = R_c^T R_body, where each contact is a pure translation t_c (3 numbers instead of a
  // 4x6 map).  See "contact-aligned blocks" in arb_fused.cuh.
  m.gen_aligned.assign(m.ngen > 0 ? m.ngen : 1, 0);
  m.gen_c0.assign(m.ngen > 0 ? m.ngen : 1, -1);
  m.caligned.assign(m.nc > 0 ? m.nc : 1, 0);
  for (int g = 0; g < m.ngen; ++g) {
    bool ok = true;
    int first = -1;
    for (int c = 0; c < m.nc && ok; ++c) {
      if (m.ctype[c] == ARB_CONS_JOINT_LIMITS) continue;
      if (m.cgen1[c] != 6 * g && m.cgen0[c] != 6 * g) continue;
      if (m.ctype[c] != ARB_CONS_SOFT_FINGER_PLANE_POINT || m.cgen1[c] != 6 * g || m.cgen0[c] >= 0 ||
          m.cint[ARB_CONS_NINT * c + 2] != ARB_PAIR_PLANE_SPHERE) { ok = false; break; }
      if (first < 0) first = c;
      for (int i = 0; i < 3; ++i)
        if (m.cdbl[ARB_CONS_NDBL * c + 32 + i] != m.cdbl[ARB_CONS_NDBL * first + 32 + i]) ok = false;
    }
    if (ok && first >= 0) {
      m.gen_aligned[g] = 1;
      m.gen_c0[g] = first;
      for (int c = 0; c < m.nc; ++c)
        if (m.ctype[c] != ARB_CONS_JOINT_LIMITS && m.cgen1[c] == 6 * g) m.caligned[c] = 1;
    }
  }
  for (int c = 0; c < m.nc; ++c)
    if (m.ctype[c] == ARB_CONS_JOINT_LIMITS) {
      m.cgen1[c] = m.ngrows++;
      m.glimdof.push_back(m.cint[ARB_CONS_NINT * c + 1]);
    }
  m.doflim.assign(m.ndof > 0 ? m.ndof : 1, 0);
  for (size_t i = 0; i < m.glimdof.size(); ++i) m.doflim[m.glimdof[i]] = 1;
  // Runs of the Gauss-Seidel sweep: consecutive constraints that work on the same cached generator
  // block (the moving body of a one-body constraint).  A world switches to the block at the first
  // constraint of the run iff one of ITS constraints in the run is active.  Joint limits work with
  // whatever block is cached (gs_visit_limit): they neither form nor break a run.
  {
    m.crunmask.assign(m.nc > 0 ? m.nc : 1, 0u);
    auto block_of = [&](int c) {
      if (m.cgen1[c] >= 0 && m.cgen0[c] >= 0) return -1 - c;      // two-body constraint: no cached block, its own run
      return m.cgen1[c] < 0 ? m.cgen0[c] : m.cgen1[c];
    };
    const int nb = m.nc < 32 ? m.nc : 32;
    for (int c = 0; c < nb; ) {
      if (m.ctype[c] == ARB_CONS_JOINT_LIMITS) { m.crunmask[c] = 1u << c; ++c; continue; }
      unsigned mask = 1u << c;
      int e = c + 1;
      while (e < nb && (m.ctype[e] == ARB_CONS_JOINT_LIMITS || block_of(e) == block_of(c))) {
        if (m.ctype[e] != ARB_CONS_JOINT_LIMITS) mask |= 1u << e;
        ++e;
      }
      while (e > c + 1 && m.ctype[e - 1] == ARB_CONS_JOINT_LIMITS) --e;    // trailing limits belong to no run
      for (int i = c; i < e; ++i)
        m.crunmask[i] = (m.ctype[i] == ARB_CONS_JOINT_LIMITS) ? (1u << i) : mask;
      c = e;
    }
  }
  // articulated-body tables: tree shape, generator paths, controllers folded per dof
  m.dofjoint.assign(m.ndof, 0);
  for (int k = 0; k < m.ndof; ++k) m.dofjoint[k] = m.dofbody[k] - 1;
  m.jhaschild.assign(nj, 0); m.jaccfirst.assign(nj, 0);
  m.jmark.assign(nj, 0); m.jmarkfirst.assign(nj, 0); m.jmarkchild.assign(nj, 0);
  m.jchild0.assign(nj, -1); m.jsib.assign(nj, -1);
  for (int j = nj - 1; j >= 0; --j) {
    const int p = m.jparent[j];
    if (p == 0) continue;
    m.jsib[j] = m.jchild0[p - 1];
    m.jchild0[p - 1] = j;
  }
  {
    std::vector<int> seen(nj + 1, 0);
    for (int j = nj - 1; j >= 0; --j) {
      const int p = m.jparent[j];
      if (p == 0) continue;
      m.jhaschild[p - 1] = 1;
      if (!seen[p]) { seen[p] = 1; m.jaccfirst[j] = 1; }
    }
    auto mark_path = [&](int body) {
      while (body > 0) { m.jmark[body - 1] = 1; body = m.jparent[body - 1]; }
    };
    for (int g = 0; g < m.ngen; ++g) mark_path(m.gen_body[g]);
    for (size_t i = 0; i < m.glimdof.size(); ++i) mark_path(m.dofbody[m.glimdof[i]]);
    std::vector<int> seenm(nj + 1, 0);
    for (int j = nj - 1; j >= 0; --j) {
      const int p = m.jparent[j];
      if (p == 0 || !m.jmark[j]) continue;
      m.jmarkchild[p - 1] = 1;
      if (!seenm[p]) { seenm[p] = 1; m.jmarkfirst[j] = 1; }
    }
  }
  // ---- group prepare stage: joints by depth, children slots, branch-point slots, shared-memory layout
  {
    std::vector<int> depth(nj, 0);
    int nlev = 0;
    for (int j = 0; j < nj; ++j) {
      depth[j] = m.jparent[j] == 0 ? 0 : depth[m.jparent[j] - 1] + 1;
      if (depth[j] + 1 > nlev) nlev = depth[j] + 1;
    }
    m.glev_off.assign(nlev + 1, 0);
    m.glev_joint.clear();
    for (int l = 0; l < nlev; ++l) {
      m.glev_off[l] = (int)m.glev_joint.size();
      for (int j = 0; j < nj; ++j)
        if (depth[j] == l) m.glev_joint.push_back(j);
    }
    m.glev_off[nlev] = (int)m.glev_joint.size();
    if (m.glev_joint.empty()) m.glev_joint.push_back(0);
    m.gslot.assign(nj > 0 ? nj : 1, -1);
    m.gvslot.assign(nj > 0 ? nj : 1, -1);
    int nslot = 0, nvslot = 0;
    for (int j = 0; j < nj; ++j) {
      const int p = m.jparent[j];
      if (p != 0 && p != j) m.gslot[j] = nslot++;           // (p == j: the parent body is the one of joint j-1, carried)
      bool reread = false;                                    // a child other than joint j+1 reads (V, V^) of body j+1
      for (int c = m.jchild0[j]; c >= 0; c = m.jsib[c])
        if (c != j + 1) reread = true;
      if (reread) m.gvslot[j] = nvslot++;
    }
    int maxpath = 1;
    for (int g = 0; g < m.ngen; ++g)
      if (m.kcols[m.gen_body[g]] > maxpath) maxpath = m.kcols[m.gen_body[g]];
    for (size_t i = 0; i < m.glimdof.size(); ++i)
      if (m.dofpos[m.glimdof[i]] + 1 > maxpath) maxpath = m.dofpos[m.glimdof[i]] + 1;
    GroupLayout& L = m.gl;
    const int n = m.ndof > 0 ? m.ndof : 1, njj = nj > 0 ? nj : 1;
    int o = 0;
    auto take = [&](int k) { int r = o; o += k; return r; };
    L.X = take(12 * njj);
    L.S = take(6 * n); L.Sh = take(6 * n); L.U = take(6 * n); L.LA = take(6 * n); L.LM = take(6 * n);
    L.dinv = take(n); L.u0 = take(n);
    const int kin = 24 * njj, slots = 78 * nslot;
    L.kin = L.slot = take(kin > slots ? kin : slots);
    L.ex = take(208);
    const int ab = 42 * njj, solve = 16 * maxpath + 16 * 12 * nvslot;
    L.ab = L.au = take(ab > solve ? ab : solve);
    L.av = L.au + 16 * maxpath;
    L.re = take(9 * (m.ngen > 0 ? m.ngen : 1));
    L.total = o | 1;
    L.nslot = nslot; L.nvslot = nvslot; L.maxpath = maxpath; L.nlev = nlev;
  }
  m.pd_kp.assign(m.ndof, 0.); m.pd_kd.assign(m.ndof, 0.); m.pd_qd.assign(m.ndof, 0.);
  m.pd_c.assign(m.ndof, 0.); m.pd_dqd.assign(m.ndof, 0.); m.pd_gpos.assign(m.ndof, -1);
  m.pd_index.assign(m.ndof > 0 ? m.ndof : 1, -1);
  for (int a = 0; a < m.na; ++a) {
    if (m.atype[a] == ARB_CTRL_WEIGHT) { m.gravity += m.adbl[4 * a]; m.nweight++; continue; }
    m.has_pd = 1;
    const int mm = m.aint[4 * a], off = m.aint[4 * a + 1];
    const double* dofs = &m.ablob[off];
    const double* gmap = dofs + mm;
    const double* kp = gmap + mm;
    const double* kd = kp + mm * mm;
    const double* qd = kd + mm * mm;
    const double* dqd = qd + mm;
    for (int i = 0; i < mm; ++i) {
      const int k = (int)dofs[i];
      for (int j = 0; j < mm; ++j)
        if (i != j && (kp[i * mm + j] != 0. || kd[i * mm + j] != 0.)) {
          m.fused_ok = 0;
          m.fused_why = "PD controller with off-diagonal gains";
        }
      if (m.pd_gpos[k] >= 0) { m.fused_ok = 0; m.fused_why = "two PD controllers on one dof"; }
      if (m.pd_index[k] < 0) m.pd_index[k] = (int)m.pd_dofs.size();   // (a second controller on the dof shares the row)
      m.pd_dofs.push_back(k);
      m.pd_gpos[k] = (int)gmap[i];
      m.pd_kp[k] = kp[i * mm + i];
      m.pd_kd[k] = kd[i * mm + i];
      m.pd_qd[k] = qd[i];
      m.pd_c[k] = kd[i * mm + i] * dqd[i];
      m.pd_dqd[k] = dqd[i];
    }
  }
  return 0;
}

// Sizes (in doubles / ints per world) of the per-batch scratch arrays, in the order
// of the DevBatch members.
struct ScratchSizes {
  int64_t pose, twist, J, dJ, M, N, B, Z, Y, gforce, cjac, cvel, cA, cT, cpinv, caux, tmp;
  int64_t cactive, cbranch, cdol, czidx;
  int64_t total_doubles() const {
    return pose + twist + J + dJ + M + N + B + Z + Y + gforce + cjac + cvel + cA + cT + cpinv + caux + tmp;
  }
  int64_t total_ints() const { return cactive + cbranch + cdol + czidx; }
};
static inline ScratchSizes scratch_sizes(const HostModel& m) {
  ScratchSizes s;
  const int64_t n = m.ndof, nj = m.nj, nr = m.nrows > 0 ? m.nrows : 1, nc = m.nc > 0 ? m.nc : 1;
  s.pose = nj * 12; s.twist = nj * 6; s.J = (int64_t)m.ncols * 6; s.dJ = s.J;
  s.M = s.N = s.B = s.Z = s.Y = n * n; s.gforce = n;
  s.cjac = nr * n; s.cvel = nr; s.cA = nr * nr; s.cT = n * nr; s.cpinv = nr * 4; s.caux = nc * 4;
  s.tmp = 2 * n;
  s.cactive = s.cbranch = s.cdol = nc; s.czidx = nc * 3;
  return s;
}
struct FusedSizes {
  int64_t fq, fLam, fv0, fT1, fT0, fu, fy, fAcc, fP, faux, fpose, ff, fRe, factive, fbranch, fzidx;
  int64_t aX, atw, ath, aS, aSh, aU, aLA, aLM, adinv, aIA, aIM, abeta, au, ax, aV, fK;
  int64_t total_doubles() const {
    return fq + fLam + fv0 + fT1 + fT0 + fu + fy + fAcc + fP + faux + fpose + ff + fRe +
           aX + atw + ath + aS + aSh + aU + aLA + aLM + adinv + aIA + aIM + abeta + au + ax + aV + fK;
  }
  int64_t total_ints() const { return factive + fbranch + fzidx; }
};
static inline FusedSizes fused_sizes(const HostModel& m) {
  FusedSizes s;
  const int64_t n = m.ndof, NG = m.ngrows > 0 ? m.ngrows : 1, nc = m.nc > 0 ? m.nc : 1,
                nr = m.nrows > 0 ? m.nrows : 1;
  const int64_t nj = m.nj > 0 ? m.nj : 1, nn = n > 0 ? n : 1;
  s.fq = nn; s.fLam = NG * NG; s.fv0 = NG; s.fT1 = nc * 24; s.fT0 = nc * 24;
  s.fu = NG; s.fy = NG; s.fAcc = nr * 4; s.fP = nr * 4; s.faux = nc * 4; s.fpose = nj * 12; s.ff = nr;
  s.fRe = 9 * (m.ngen > 0 ? m.ngen : 1);
  s.factive = nc; s.fbranch = nc; s.fzidx = 3 * nc;
  s.aX = nj * 12; s.atw = nj * 6; s.ath = nj * 6;
  s.aS = s.aSh = s.aU = s.aLA = s.aLM = nn * 6; s.adinv = nn;
  s.aIA = s.aIM = nj * 36; s.abeta = nj * 6;
  const int64_t ng1 = m.ngen > 1 ? m.ngen : 1;   // six right-hand sides per generator body, all bodies in one pass
  s.au = 6 * ng1 * nn; s.ax = 6 * ng1 * nn; s.aV = nj * 72 * ng1;
  s.fK = nn * NG;
  return s;
}
// Tiled layout: tile t of ARB_TILE worlds owns doubles [t*R*ARB_TILE, (t+1)*R*ARB_TILE), array X
// starts offX*ARB_TILE into the tile; the pointers stored here are those of tile 0 (the kernels
// add the per-thread tile offset, fused_tile_view).  Allocate for fused_padded_worlds(W).
static inline int64_t fused_padded_worlds(int64_t W) { return (W + ARB_TILE - 1) / ARB_TILE * ARB_TILE; }
static inline void carve_fused(const FusedSizes& s, double* dbl, int* ints, DevBatch& b) {
  double* p = dbl;
  auto take = [&](int64_t k) { double* r = p; p += k * ARB_TILE; return r; };
  b.fq = take(s.fq); b.fLam = take(s.fLam); b.fv0 = take(s.fv0);
  b.fT1 = take(s.fT1); b.fT0 = take(s.fT0); b.fu = take(s.fu); b.fy = take(s.fy);
  b.fAcc = take(s.fAcc); b.fP = take(s.fP); b.faux = take(s.faux); b.fpose = take(s.fpose);
  b.ff = take(s.ff); b.fRe = take(s.fRe);
  b.aX = take(s.aX); b.atw = take(s.atw); b.ath = take(s.ath);
  b.aS = take(s.aS); b.aSh = take(s.aSh); b.aU = take(s.aU); b.aLA = take(s.aLA); b.aLM = take(s.aLM);
  b.adinv = take(s.adinv); b.aIA = take(s.aIA); b.aIM = take(s.aIM); b.abeta = take(s.abeta);
  b.au = take(s.au); b.ax = take(s.ax); b.aV = take(s.aV);
  b.fK = take(s.fK);
  int* q = ints;
  auto takei = [&](int64_t k) { int* r = q; q += k * ARB_TILE; return r; };
  b.factive = takei(s.factive); b.fbranch = takei(s.fbranch); b.fzidx = takei(s.fzidx);
  b.frec = s.total_doubles();
  b.firec = s.total_ints();
}
// Body -> wrench row table of arb_batch_bind_applied_forces: rows[j] = i if bodies[i] == j + 1,
// else -1.  Refuses the ground, bodies out of range, duplicates and a wrench without bodies.  The same
// table for the body inertia of arb_batch_bind_body_inertia, with `what` naming the array.
static inline int applied_wrench_rows(const HostModel& m, int nbodies, const int32_t* bodies, bool has_wrench,
                                      std::vector<int>& rows, std::string& err, const char* what = "wrench") {
  const std::string w(what);
  if (nbodies < 0) { err = "negative number of " + w + " bodies"; return -1; }
  if (nbodies > 0 && !bodies) { err = "null body list"; return -1; }
  if (has_wrench && nbodies == 0) {
    err = (std::string("aeiou").find(w[0]) != std::string::npos ? "an " : "a ") + w + " array needs its bodies";
    return -1;
  }
  rows.assign(m.nj > 0 ? m.nj : 1, -1);
  for (int i = 0; i < nbodies; ++i) {
    const int body = bodies[i];
    if (body == 0) { err = "no " + w + " can be applied to the ground (body 0)"; return -1; }
    if (body < 0 || body > m.nj) { err = w + " body " + std::to_string(body) + " out of range"; return -1; }
    if (rows[body - 1] >= 0) { err = w + " body " + std::to_string(body) + " listed twice"; return -1; }
    rows[body - 1] = i;
  }
  return 0;
}
// Constraint -> mu row table of arb_batch_bind_contact_friction: rows[c] = i if constraints[i] == c,
// else -1.  Refuses indices out of range, constraints that are not soft-finger contacts, duplicates
// and mu without constraints.
static inline int friction_rows(const HostModel& m, int ncontacts, const int32_t* constraints, bool has_mu,
                                std::vector<int>& rows, std::string& err) {
  if (ncontacts < 0) { err = "negative number of mu constraints"; return -1; }
  if (ncontacts > 0 && !constraints) { err = "null constraint list"; return -1; }
  if (has_mu && ncontacts == 0) { err = "a mu array needs its constraints"; return -1; }
  rows.assign(m.nc > 0 ? m.nc : 1, -1);
  for (int i = 0; i < ncontacts; ++i) {
    const int c = constraints[i];
    const std::string cs = std::to_string(c);
    if (c < 0 || c >= m.nc) { err = "mu constraint " + cs + " out of range"; return -1; }
    if (m.ctype[c] != ARB_CONS_SOFT_FINGER_PLANE_POINT) { err = "mu constraint " + cs + " is not a contact"; return -1; }
    if (rows[c] >= 0) { err = "mu constraint " + cs + " listed twice"; return -1; }
    rows[c] = i;
  }
  return 0;
}

// carve `dbl` (doubles) and `ints` into the DevBatch members; W worlds
static inline void carve_scratch(const ScratchSizes& s, int64_t W, double* dbl, int* ints, DevBatch& b) {
  double* p = dbl;
  auto take = [&](int64_t k) { double* r = p; p += k * W; return r; };
  b.pose = take(s.pose); b.twist = take(s.twist); b.J = take(s.J); b.dJ = take(s.dJ);
  b.M = take(s.M); b.N = take(s.N); b.B = take(s.B); b.Z = take(s.Z); b.Y = take(s.Y);
  b.gforce = take(s.gforce); b.cjac = take(s.cjac); b.cvel = take(s.cvel); b.cA = take(s.cA);
  b.cT = take(s.cT); b.cpinv = take(s.cpinv); b.caux = take(s.caux); b.tmp = take(s.tmp);
  int* q = ints;
  auto takei = [&](int64_t k) { int* r = q; q += k * W; return r; };
  b.cactive = takei(s.cactive); b.cbranch = takei(s.cbranch); b.cdol = takei(s.cdol);
  b.czidx = takei(s.czidx);
}

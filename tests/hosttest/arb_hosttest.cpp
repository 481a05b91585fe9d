// TEST INFRASTRUCTURE ONLY.  CPU build of the per-world scalar routines of
// arboris-python_b200/csrc (the same source the CUDA kernels compile), so that
// `pytest -m "not gpu"` can check the arithmetic against the oracle without a
// GPU.  Built by tests/hosttest/build.py into tests/hosttest/_build/; the
// arboris_b200 package never loads it (the product path is CUDA only).
#define ARB_HOSTTEST_COUNTERS 1
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>
#include "../../arboris-python_b200/csrc/arb_model_host.h"
#include "../../arboris-python_b200/csrc/arb_world.cuh"
#include "../../arboris-python_b200/csrc/arb_fused.cuh"
#include "../../arboris-python_b200/csrc/arb_group.cuh"

static DevModel view(const HostModel& h) {
  DevModel m;
  m.ndof = h.ndof; m.ngpos = h.ngpos; m.nj = h.nj; m.nc = h.nc; m.na = h.na; m.nrows = h.nrows;
  m.ncols = h.ncols; m.maxk = h.maxk; m.anyvisc = h.anyvisc;
  m.jtype = h.jtype.data(); m.jparent = h.jparent.data(); m.jdof = h.jdof.data(); m.jgpos = h.jgpos.data();
  m.Hpr = h.Hpr.data(); m.HprInv = h.HprInv.data(); m.Hcn = h.Hcn.data(); m.HcnInv = h.HcnInv.data();
  m.hcn_ident = h.hcn_ident.data(); m.bmass = h.bmass.data(); m.bvisc = h.bvisc.data(); m.brx = h.brx.data();
  m.bflags = h.bflags.data(); m.coloff = h.coloff.data(); m.kcols = h.kcols.data(); m.pathdof = h.pathdof.data();
  m.ctype = h.ctype.data(); m.cint = h.cint.data(); m.crow = h.crow.data(); m.cdbl = h.cdbl.data();
  m.atype = h.atype.data(); m.aint = h.aint.data(); m.adbl = h.adbl.data(); m.ablob = h.ablob.data();
  for (int i = 0; i < 3; ++i) m.up[i] = h.up[i];
  m.dofbody = h.dofbody.data(); m.dofpos = h.dofpos.data(); m.ngen = h.ngen; m.ngrows = h.ngrows;
  m.gen_body = h.gen_body.data(); m.cgen1 = h.cgen1.data(); m.cgen0 = h.cgen0.data();
  m.gen_aligned = h.gen_aligned.data(); m.gen_c0 = h.gen_c0.data(); m.caligned = h.caligned.data(); m.crunmask = h.crunmask.data(); m.doflim = h.doflim.data();
  m.dofjoint = h.dofjoint.data(); m.jhaschild = h.jhaschild.data(); m.jaccfirst = h.jaccfirst.data();
  m.jmark = h.jmark.data(); m.jmarkfirst = h.jmarkfirst.data(); m.jmarkchild = h.jmarkchild.data();
  m.jchild0 = h.jchild0.data(); m.jsib = h.jsib.data();
  m.glimdof = h.glimdof.data(); m.pd_gpos = h.pd_gpos.data(); m.pd_kp = h.pd_kp.data();
  m.pd_kd = h.pd_kd.data(); m.pd_qd = h.pd_qd.data(); m.pd_c = h.pd_c.data();
  m.pd_dqd = h.pd_dqd.data(); m.pd_index = h.pd_index.data(); m.npd = (int)h.pd_dofs.size();
  m.has_pd = h.has_pd; m.gravity = h.gravity; m.nweight = h.nweight;
  m.gl = h.gl; m.glev_off = h.glev_off.data(); m.glev_joint = h.glev_joint.data();
  m.gslot = h.gslot.data(); m.gvslot = h.gvslot.data();
  return m;
}

struct HostBatch {
  HostModel hm;
  DevModel dm;
  DevBatch b;
  std::vector<double> dbl, fdbl;
  std::vector<int> ints, fints, status;
  int coop = 1;
};

extern "C" {
void* ht_create(const arb_model_desc* d, int64_t W, char* errbuf, int errlen) {
  HostBatch* hb = new HostBatch();
  std::string err;
  if (build_host_model(d, hb->hm, err) != 0) {
    strncpy(errbuf, err.c_str(), errlen - 1);
    delete hb;
    return nullptr;
  }
  hb->dm = view(hb->hm);
  ScratchSizes s = scratch_sizes(hb->hm);
  hb->dbl.assign(s.total_doubles() * W, 0.);
  hb->ints.assign(s.total_ints() * W, 0);
  hb->status.assign(W, 0);
  memset(&hb->b, 0, sizeof(DevBatch));
  hb->b.W = W;
  carve_scratch(s, W, hb->dbl.data(), hb->ints.data(), hb->b);
  hb->b.status = hb->status.data();
  FusedSizes fs = fused_sizes(hb->hm);
  hb->fdbl.assign(fs.total_doubles() * fused_padded_worlds(W), 0.);
  hb->fints.assign(fs.total_ints() * fused_padded_worlds(W), 0);
  carve_fused(fs, hb->fdbl.data(), hb->fints.data(), hb->b);
  return hb;
}
void ht_destroy(void* p) { delete (HostBatch*)p; }
void ht_set_coop(void* p, int v) { ((HostBatch*)p)->coop = v; }
void ht_bind(void* p, double* gpos, double* gvel, double* cforce) {
  HostBatch* hb = (HostBatch*)p;
  hb->b.gpos = gpos; hb->b.gvel = gvel; hb->b.cforce = cforce;
}
void ht_bind_params(void* p, const double* kp, const double* kd, const double* qd, const double* dqd) {
  HostBatch* hb = (HostBatch*)p;
  hb->b.pkp = kp; hb->b.pkd = kd; hb->b.pqd = qd; hb->b.pdqd = dqd;
}
void ht_update_dynamic(void* p) {
  HostBatch* hb = (HostBatch*)p;
  for (int64_t w = 0; w < hb->b.W; ++w) world_update_dynamic(hb->dm, hb->b, w);
}
void ht_update_controllers(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  for (int64_t w = 0; w < hb->b.W; ++w) world_update_controllers(hb->dm, hb->b, w, dt);
}
void ht_update_constraints(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  for (int64_t w = 0; w < hb->b.W; ++w) world_update_constraints(hb->dm, hb->b, w, dt);
}
void ht_integrate(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  for (int64_t w = 0; w < hb->b.W; ++w) world_integrate(hb->dm, hb->b, w, dt);
}
// the fused step with the group prepare stage (16 emulated lanes per world, arb_group.cuh), the
// per-lane Gauss-Seidel and the K-matrix finish stage
void ht_fused_step_group(void* p, double dt, int write_poses) {
  HostBatch* hb = (HostBatch*)p;
  std::vector<double> sm(hb->dm.gl.total, 0.);
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const DevBatch t = fused_tile_view(hb->b, w);
    for (size_t i = 0; i < sm.size(); ++i) sm[i] = 1e300;     // nothing may be read before it is written
    GroupCtx g;
    g.sm = sm.data(); g.lane = 0; g.mask = 0;
    group_prepare(hb->dm, t, w, dt, g, write_poses != 0);
    double Lst[36];
    world_fused_gs(hb->dm, t, w, dt, Lst, 1);
    world_fused_finish_k(hb->dm, t, w, dt);
  }
}
int ht_group_doubles(void* p) { return ((HostBatch*)p)->dm.gl.total; }
// the fused step in its scalar form: update_dynamic, prepare, gs, finish
void ht_fused_step(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const DevBatch t = fused_tile_view(hb->b, w);
    world_fused_prepare(hb->dm, t, w, dt);
    double Lst[36];
    if (hb->coop) {       // block-cooperative form with a "block" of one thread
      double q[ARB_SLIDE_NDBL], r[4];
      int rs[1], cnt[2];
      unsigned long long bm;
      GsCoop co;
      co.q = q; co.r = r; co.rs = rs; co.cnt = cnt; co.bm = &bm;
      co.cap = 1; co.tid = 0; co.nthr = 1; co.parity = 0;
      world_fused_gs_coop(hb->dm, t, w, true, dt, co, Lst, 1);
    } else {
      world_fused_gs(hb->dm, t, w, dt, Lst, 1);
    }
    world_fused_finish(hb->dm, t, w, dt);
  }
}
// The prepare stage followed by the Gauss-Seidel's prologue only (diagonal Delassus blocks, the warm
// start y0 = sum T_c^T f_c): the hand-over of the prepare stage without the sweeps, for
// tests/test_prepare_reference.py (arb_hosttest_applied.cpp: the instantiation with applied forces).
extern "C++" template <bool APPLIED, bool PARAMS>
void fused_prepare_worlds(HostBatch* hb, double dt, const DevApplied& ap) {
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const DevBatch b = fused_tile_view(hb->b, w);
    world_fused_prepare<APPLIED, PARAMS>(hb->dm, b, w, dt, ap);
    bool any = false;
    for (int c = 0; c < hb->dm.nc; ++c) any = any || FT(b.factive, c);
    for (int g = 0; g < hb->dm.ngrows; ++g) FT(b.fy, g) = 0.;
    if (!any) continue;
    for (int r = 0; r < hb->dm.nrows; ++r) FT(b.ff, r) = ST_LD(b.cforce, r);
    gs_prologue(hb->dm, b, w, dt);
  }
}
void ht_fused_prepare(void* p, double dt) {
  fused_prepare_worlds<false, false>((HostBatch*)p, dt, DevApplied{nullptr, nullptr, nullptr});
}
// the finish stage alone, with the wrench y the caller left in fy (ht_fused_dbl_set)
void ht_fused_finish(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  for (int64_t w = 0; w < hb->b.W; ++w) world_fused_finish(hb->dm, fused_tile_view(hb->b, w), w, dt);
}
static double* fused_dbl(HostBatch* hb, const std::string& s) {
  const DevBatch& b = hb->b;
  if (s == "fq") return b.fq; if (s == "fv0") return b.fv0; if (s == "fLam") return b.fLam;
  if (s == "fRe") return b.fRe; if (s == "fy") return b.fy; if (s == "fAcc") return b.fAcc;
  if (s == "adinv") return b.adinv;
  return nullptr;
}
// fused double outputs are tiled: copied out as [elem][W] (ht_fused_dbl) or in from it (ht_fused_dbl_set)
int ht_fused_dbl(void* p, const char* name, int nelem, double* out) {
  HostBatch* hb = (HostBatch*)p;
  const double* base = fused_dbl(hb, name);
  if (!base) return -1;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const double* t = base + (w / ARB_TILE) * hb->b.frec * ARB_TILE + w % ARB_TILE;
    for (int e = 0; e < nelem; ++e) out[e * hb->b.W + w] = t[e * ARB_TILE];
  }
  return 0;
}
int ht_fused_dbl_set(void* p, const char* name, int nelem, const double* in) {
  HostBatch* hb = (HostBatch*)p;
  double* base = fused_dbl(hb, name);
  if (!base) return -1;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    double* t = base + (w / ARB_TILE) * hb->b.frec * ARB_TILE + w % ARB_TILE;
    for (int e = 0; e < nelem; ++e) t[e * ARB_TILE] = in[e * hb->b.W + w];
  }
  return 0;
}
// raw scratch access: which = index into the DevBatch double members in declaration order
double* ht_array(void* p, const char* name) {
  HostBatch* hb = (HostBatch*)p;
  DevBatch& b = hb->b;
  std::string s(name);
  if (s == "pose") return b.pose; if (s == "twist") return b.twist; if (s == "J") return b.J;
  if (s == "dJ") return b.dJ; if (s == "M") return b.M; if (s == "N") return b.N; if (s == "B") return b.B;
  if (s == "Z") return b.Z; if (s == "Y") return b.Y; if (s == "gforce") return b.gforce;
  if (s == "cjac") return b.cjac; if (s == "cvel") return b.cvel; if (s == "cA") return b.cA;
  if (s == "caux") return b.caux;
  return nullptr;
}
// fused int outputs are tiled: copy out as [elem][W]
void ht_fused_ints(void* p, const char* name, int nelem, int* out) {
  HostBatch* hb = (HostBatch*)p;
  const std::string s(name);
  const int* base = s == "factive" ? hb->b.factive : hb->b.fbranch;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const int* t = base + (w / ARB_TILE) * hb->b.firec * ARB_TILE + w % ARB_TILE;
    for (int e = 0; e < nelem; ++e) out[e * hb->b.W + w] = t[e * ARB_TILE];
  }
}
int* ht_iarray(void* p, const char* name) {
  HostBatch* hb = (HostBatch*)p;
  DevBatch& b = hb->b;
  std::string s(name);
  if (s == "cactive") return b.cactive; if (s == "cbranch") return b.cbranch; if (s == "cdol") return b.cdol;
  if (s == "czidx") return b.czidx; if (s == "status") return b.status;
  return nullptr;
}
void ht_pinv(int n, const double* a, double* out) {
  if (n == 1) pinv_small<1>(a, out);
  else if (n == 2) pinv_small<2>(a, out);
  else if (n == 3) pinv_small<3>(a, out);
  else pinv_small<4>(a, out);
}
int ht_eig6(const double* a, double* wr, double* wi) {
  double tmp[36];
  memcpy(tmp, a, sizeof(tmp));
  return eig_real_general6(tmp, wr, wi) ? 1 : 0;
}
// structured sliding root: returns 1 if the structured path applied
int ht_sliding_root(const double* A, const double* alpha, double mu, double* s, int* found) {
  bool f = false;
  bool ok = sliding_root_structured(A, alpha, mu, s, &f);
  *found = f ? 1 : 0;
  return ok ? 1 : 0;
}
// the sextic routines of the sliding root, one polynomial at a time (p[0..5], monic)
int ht_poly6_positive(const double* p) { return poly6_positive_on_halfline(p) ? 1 : 0; }
int ht_poly6_fast(const double* p, double* root) {
  double c[7];      // (the bracket refinement reads the leading coefficient too)
  for (int k = 0; k < 6; ++k) c[k] = p[k];
  c[6] = 1.;
  return poly6_largest_root_fast(c, root);
}
int ht_poly6_slow(const double* p, double* root) {
  double T = 0.;
  for (int k = 0; k < 6; ++k) T = fmax(T, fabs(p[k]));
  T += 1.;
  double roots[6], c[7];
  for (int k = 0; k < 6; ++k) c[k] = p[k];
  c[6] = 1.;
  const int nr = poly6_roots_slow(c, T, roots);
  if (nr) *root = roots[nr - 1];
  return nr;
}
long ht_fastroot_hits() { return arb_fastroot_hits; }
long ht_fastroot_fail(int i) { return arb_fastroot_fail[i]; }
void ht_set_slidemask(unsigned* p) { arb_dbg_slidemask = p; }
// number of generator bodies; flags[g] = 1 for contact-aligned ones, caligned[c] per constraint
int ht_aligned(void* p, int* flags, int* caligned) {
  HostBatch* hb = (HostBatch*)p;
  for (int g = 0; g < hb->hm.ngen; ++g) flags[g] = hb->hm.gen_aligned[g];
  for (int c = 0; c < hb->hm.nc; ++c) caligned[c] = hb->hm.caligned[c];
  return hb->hm.ngen;
}
// generator layout: counts = {ngen, NG}; body, aligned, c0 [ngen]; limdof [NG - 6 ngen] (NULL: counts only)
void ht_generators(void* p, int* counts, int* body, int* aligned, int* c0, int* limdof) {
  const HostModel& h = ((HostBatch*)p)->hm;
  counts[0] = h.ngen;
  counts[1] = h.ngrows;
  if (!body) return;     // counts only
  for (int g = 0; g < h.ngen; ++g) { body[g] = h.gen_body[g]; aligned[g] = h.gen_aligned[g]; c0[g] = h.gen_c0[g]; }
  for (size_t i = 0; i < h.glimdof.size(); ++i) limdof[i] = h.glimdof[i];
}
int ht_solve4(const double* a, const double* b, double* x) { return solve_small<4>(a, b, x) ? 1 : 0; }
void ht_exp(const double* tw, double* out12) {
  Se3 h;
  se3_exp(tw, h);
  se3_to12(h, out12);
}
// SoftFingerContact.solve, phase form: f (4) in/out, df (4) out, *status out; returns the branch
int ht_softfinger_solve(const double* v, const double* A, const double* P, double sdist, double mu, const double* eps,
                        double dt, double* f, double* df, int* status) {
  *status = 0;
  return softfinger_solve(v, A, P, sdist, mu, eps, dt, f, df, status);
}
double ht_inv_cond4(const double* a, double* out) { return inv_small_cond<4>(a, out); }
int ht_certify(const double* p, double x) { return poly6_certify(p, x) ? 1 : 0; }
void ht_zaligned(const double* z, double* R, int* idx) { zaligned(z, R, idx); }
// contact_collide, frames as 12 doubles (R row-major, p); cd: ARB_CONS_NDBL doubles
double ht_collide(int pair, const double* cd, const double* h0, const double* h1, double* c0, double* c1, int* zi) {
  Se3 g0, g1, o0, o1;
  for (int k = 0; k < 9; ++k) { g0.R[k] = h0[k]; g1.R[k] = h1[k]; }
  for (int k = 0; k < 3; ++k) { g0.p[k] = h0[9 + k]; g1.p[k] = h1[9 + k]; }
  const double sd = contact_collide(pair, cd, g0, g1, o0, o1, zi);
  se3_to12(o0, c0);
  se3_to12(o1, c1);
  return sd;
}
}

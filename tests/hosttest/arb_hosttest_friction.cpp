// TEST INFRASTRUCTURE ONLY.  The CPU build of arb_hosttest.cpp plus per-world contact friction
// (arb_batch_bind_contact_friction; DevFriction), for tests/test_contact_friction.py: binding with the
// library's own validation, the phase routines and the fused step with the world's friction.  Built
// by that test into tests/hosttest/_build/.
#include <map>
#include "arb_hosttest.cpp"

namespace {
struct Friction {
  std::vector<int> rows;
  DevFriction fr = {nullptr, nullptr};
};
std::map<void*, Friction> g_friction;   // by host batch
}

extern "C" {
// arb_batch_bind_contact_friction on a host array; returns 0 or -1 with the message in errbuf (the
// previous binding kept)
int ht_bind_friction(void* p, int ncontacts, const int32_t* constraints, const double* mu, char* errbuf, int errlen) {
  HostBatch* hb = (HostBatch*)p;
  std::vector<int> rows;
  std::string err;
  if (friction_rows(hb->hm, ncontacts, constraints, mu != nullptr, rows, err)) {
    strncpy(errbuf, err.c_str(), errlen - 1);
    return -1;
  }
  Friction& a = g_friction[p];
  a.rows = rows;
  a.fr.mu = ncontacts > 0 ? mu : nullptr;
  a.fr.row = a.rows.data();
  return 0;
}
void ht_release_friction(void* p) { g_friction.erase(p); }
// the phase routine and the fused step with the instantiations the device picks (launch_update_constraints
// in arb_api.cu, launch_gs in arb_fused.cu)
void ht_fr_update_constraints(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  const DevFriction fr = g_friction[p].fr;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    if (fr.mu) world_update_constraints<true>(hb->dm, hb->b, w, dt, fr);
    else world_update_constraints<false>(hb->dm, hb->b, w, dt, fr);
  }
}
// group = 1: the group prepare stage (16 emulated lanes) and the K-matrix finish, as ht_fused_step_group
void ht_fr_fused_step(void* p, double dt, int group) {
  HostBatch* hb = (HostBatch*)p;
  const DevFriction fr = g_friction[p].fr;
  std::vector<double> sm(hb->dm.gl.total, 0.);
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const DevBatch t = fused_tile_view(hb->b, w);
    if (group) {
      for (size_t i = 0; i < sm.size(); ++i) sm[i] = 1e300;
      GroupCtx g;
      g.sm = sm.data(); g.lane = 0; g.mask = 0;
      group_prepare(hb->dm, t, w, dt, g, false);
    } else {
      world_fused_prepare(hb->dm, t, w, dt);
    }
    if (fr.mu) world_friction_gather(hb->dm, t, w, fr);
    double Lst[36];
    if (hb->coop) {       // block-cooperative form with a "block" of one thread
      double q[ARB_SLIDE_NDBL], r[4];
      int rs[1], cnt[2];
      unsigned long long bm;
      GsCoop co;
      co.q = q; co.r = r; co.rs = rs; co.cnt = cnt; co.bm = &bm;
      co.cap = 1; co.tid = 0; co.nthr = 1; co.parity = 0;
      if (fr.mu) world_fused_gs_coop<true>(hb->dm, t, w, true, dt, co, Lst, 1);
      else world_fused_gs_coop<false>(hb->dm, t, w, true, dt, co, Lst, 1);
    } else {
      if (fr.mu) world_fused_gs<true>(hb->dm, t, w, dt, Lst, 1);
      else world_fused_gs<false>(hb->dm, t, w, dt, Lst, 1);
    }
    if (group) world_fused_finish_k(hb->dm, t, w, dt);
    else world_fused_finish(hb->dm, t, w, dt);
  }
}
}

// TEST INFRASTRUCTURE ONLY.  The CPU build of arb_hosttest.cpp plus per-world body inertia and
// gravity (arb_batch_bind_body_inertia, arb_batch_bind_gravity; DevApplied), for
// tests/test_body_params.py: binding with the library's own validation, the phase routines and the
// fused step with the world's parameters.  Built by that test into tests/hosttest/_build/.
#include <map>
#include "arb_hosttest.cpp"

namespace {
struct BodyParams {
  std::vector<int> rows;
  DevApplied ap = {nullptr, nullptr, nullptr};
};
std::map<void*, BodyParams> g_params;   // by host batch
bool bound(const DevApplied& ap) { return ap.inertia || ap.gravity; }
}

extern "C" {
// arb_batch_bind_body_inertia and arb_batch_bind_gravity on host arrays; returns 0 or -1 with the
// message in errbuf (the previous binding kept)
int ht_bind_body_params(void* p, int nbodies, const int32_t* bodies, const double* inertia, const double* gravity,
                        char* errbuf, int errlen) {
  HostBatch* hb = (HostBatch*)p;
  std::vector<int> rows;
  std::string err;
  if (applied_wrench_rows(hb->hm, nbodies, bodies, inertia != nullptr, rows, err, "inertia") == 0 &&
      gravity && hb->hm.nweight == 0)
    err = "the model has no WeightController: there is no gravity to replace";
  if (!err.empty()) {
    strncpy(errbuf, err.c_str(), errlen - 1);
    return -1;
  }
  BodyParams& a = g_params[p];
  a.rows = rows;
  a.ap.inertia = nbodies > 0 ? inertia : nullptr;
  a.ap.irow = a.rows.data();
  a.ap.gravity = gravity;
  return 0;
}
void ht_release_body_params(void* p) { g_params.erase(p); }
// the phase routines and the fused step with the instantiations the device picks (arb_api.cu,
// launch_prepare_lane in arb_fused.cu)
void ht_bp_update_dynamic(void* p) {
  HostBatch* hb = (HostBatch*)p;
  const DevApplied ap = g_params[p].ap;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    if (bound(ap)) world_update_dynamic<true>(hb->dm, hb->b, w, ap);
    else world_update_dynamic<false>(hb->dm, hb->b, w, ap);
  }
}
void ht_bp_update_controllers(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  const DevApplied ap = g_params[p].ap;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    if (bound(ap)) world_update_controllers<true>(hb->dm, hb->b, w, dt, ap);
    else world_update_controllers<false>(hb->dm, hb->b, w, dt, ap);
  }
}
void ht_bp_fused_step(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  const DevApplied ap = g_params[p].ap;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const DevBatch t = fused_tile_view(hb->b, w);
    if (bound(ap)) world_fused_prepare<true, true>(hb->dm, t, w, dt, ap);
    else world_fused_prepare<false, false>(hb->dm, t, w, dt, ap);
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
}

// TEST INFRASTRUCTURE ONLY.  The CPU build of arb_hosttest.cpp plus the applied forces of
// arb_batch_bind_applied_forces (DevApplied), for tests/test_applied_forces.py: binding with the
// library's own validation, update_controllers and the fused step with the forces.  Built by that
// test into tests/hosttest/_build/.
#include <map>
#include "arb_hosttest.cpp"

namespace {
struct Applied {
  std::vector<int> rows;
  DevApplied ap = {nullptr, nullptr, nullptr};
};
std::map<void*, Applied> g_applied;   // by host batch
}

extern "C" {
// arb_batch_bind_applied_forces on host arrays; returns 0 or -1 with the message in errbuf
int ht_bind_applied(void* p, const double* tau, int nbodies, const int32_t* bodies, const double* wrench,
                    char* errbuf, int errlen) {
  HostBatch* hb = (HostBatch*)p;
  std::vector<int> rows;
  std::string err;
  if (applied_wrench_rows(hb->hm, nbodies, bodies, wrench != nullptr, rows, err)) {
    strncpy(errbuf, err.c_str(), errlen - 1);
    return -1;
  }
  Applied& a = g_applied[p];
  a.rows = rows;
  a.ap.tau = tau;
  a.ap.wrench = nbodies > 0 ? wrench : nullptr;
  a.ap.row = a.rows.data();
  return 0;
}
void ht_release_applied(void* p) { g_applied.erase(p); }
void ht_applied_update_controllers(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  const DevApplied ap = g_applied[p].ap;
  for (int64_t w = 0; w < hb->b.W; ++w) world_update_controllers(hb->dm, hb->b, w, dt, ap);
}
// ht_fused_step with the prepare instantiation the device picks (launch_prepare_lane, arb_fused.cu)
void ht_applied_fused_step(void* p, double dt) {
  HostBatch* hb = (HostBatch*)p;
  const DevApplied ap = g_applied[p].ap;
  for (int64_t w = 0; w < hb->b.W; ++w) {
    const DevBatch t = fused_tile_view(hb->b, w);
    if (ap.tau || ap.wrench) world_fused_prepare<true>(hb->dm, t, w, dt, ap);
    else world_fused_prepare<false>(hb->dm, t, w, dt, ap);
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

// C ABI of arboris_b200 (include/arboris_b200.h) and the lane-per-world kernels.
// sm_100a, fp64.  The fused step (lane-per-world stages, and the 16-lanes-per-world prepare stage of
// arb_group.cuh) lives in arb_fused.cu.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "arb_model_host.h"
#include "arb_world.cuh"
#include "arb_internal.h"

static thread_local std::string g_err;
const char* arb_set_error(const std::string& s) { g_err = s; return g_err.c_str(); }

#define CUDA_OK(call)                                                               \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      arb_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));            \
      return -100;                                                                  \
    }                                                                               \
  } while (0)

extern "C" const char* arb_last_error(void) { return g_err.c_str(); }
extern "C" int arb_version(void) { return 100; }

// ---------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------
template <class T>
static int upload(const std::vector<T>& v, const T** out, std::vector<void*>& owned) {
  size_t bytes = (v.size() ? v.size() : 1) * sizeof(T);
  void* p = nullptr;
  CUDA_OK(cudaMalloc(&p, bytes));
  owned.push_back(p);
  if (v.size()) CUDA_OK(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = (const T*)p;
  return 0;
}

static int model_to_device(arb_model* mo, int device) {
  if (mo->dev_ready.count(device)) return 0;
  CUDA_OK(cudaSetDevice(device));
  const HostModel& h = mo->host;
  DevModel m;
  memset(&m, 0, sizeof(m));
  m.ndof = h.ndof; m.ngpos = h.ngpos; m.nj = h.nj; m.nc = h.nc; m.na = h.na; m.nrows = h.nrows;
  m.ncols = h.ncols; m.maxk = h.maxk; m.anyvisc = h.anyvisc;
  std::vector<void*>& own = mo->dev_owned[device];
  int rc = 0;
  rc |= upload(h.jtype, &m.jtype, own);   rc |= upload(h.jparent, &m.jparent, own);
  rc |= upload(h.jdof, &m.jdof, own);     rc |= upload(h.jgpos, &m.jgpos, own);
  rc |= upload(h.Hpr, &m.Hpr, own);       rc |= upload(h.HprInv, &m.HprInv, own);
  rc |= upload(h.Hcn, &m.Hcn, own);       rc |= upload(h.HcnInv, &m.HcnInv, own);
  rc |= upload(h.hcn_ident, &m.hcn_ident, own);
  rc |= upload(h.bmass, &m.bmass, own);   rc |= upload(h.bvisc, &m.bvisc, own);
  rc |= upload(h.brx, &m.brx, own);       rc |= upload(h.bflags, &m.bflags, own);
  rc |= upload(h.coloff, &m.coloff, own); rc |= upload(h.kcols, &m.kcols, own);
  rc |= upload(h.pathdof, &m.pathdof, own);
  rc |= upload(h.ctype, &m.ctype, own);   rc |= upload(h.cint, &m.cint, own);
  rc |= upload(h.crow, &m.crow, own);     rc |= upload(h.cdbl, &m.cdbl, own);
  rc |= upload(h.atype, &m.atype, own);   rc |= upload(h.aint, &m.aint, own);
  rc |= upload(h.adbl, &m.adbl, own);     rc |= upload(h.ablob, &m.ablob, own);
  rc |= upload(h.dofbody, &m.dofbody, own); rc |= upload(h.dofpos, &m.dofpos, own);
  rc |= upload(h.gen_body, &m.gen_body, own);
  rc |= upload(h.cgen1, &m.cgen1, own);   rc |= upload(h.cgen0, &m.cgen0, own);
  rc |= upload(h.gen_aligned, &m.gen_aligned, own); rc |= upload(h.gen_c0, &m.gen_c0, own);
  rc |= upload(h.caligned, &m.caligned, own);
  rc |= upload(h.crunmask, &m.crunmask, own);
  rc |= upload(h.doflim, &m.doflim, own);
  m.ngen = h.ngen; m.ngrows = h.ngrows;
  rc |= upload(h.dofjoint, &m.dofjoint, own);   rc |= upload(h.jhaschild, &m.jhaschild, own);
  rc |= upload(h.jaccfirst, &m.jaccfirst, own); rc |= upload(h.jmark, &m.jmark, own);
  rc |= upload(h.jmarkfirst, &m.jmarkfirst, own); rc |= upload(h.jmarkchild, &m.jmarkchild, own);
  rc |= upload(h.jchild0, &m.jchild0, own);       rc |= upload(h.jsib, &m.jsib, own);
  rc |= upload(h.glimdof, &m.glimdof, own);     rc |= upload(h.pd_gpos, &m.pd_gpos, own);
  rc |= upload(h.pd_kp, &m.pd_kp, own);         rc |= upload(h.pd_kd, &m.pd_kd, own);
  rc |= upload(h.pd_qd, &m.pd_qd, own);         rc |= upload(h.pd_c, &m.pd_c, own);
  rc |= upload(h.pd_dqd, &m.pd_dqd, own);       rc |= upload(h.pd_index, &m.pd_index, own);
  m.npd = (int)h.pd_dofs.size();
  rc |= upload(h.glev_off, &m.glev_off, own);   rc |= upload(h.glev_joint, &m.glev_joint, own);
  rc |= upload(h.gslot, &m.gslot, own);         rc |= upload(h.gvslot, &m.gvslot, own);
  m.gl = h.gl;
  m.has_pd = h.has_pd; m.gravity = h.gravity; m.nweight = h.nweight;
  if (rc) return -100;
  for (int i = 0; i < 3; ++i) m.up[i] = h.up[i];
  mo->dev[device] = m;
  mo->dev_ready.insert(device);
  return 0;
}

extern "C" int arb_model_create(const arb_model_desc* desc, arb_model** out) {
  if (!out) { arb_set_error("null output pointer"); return -1; }
  arb_model* mo = new arb_model();
  std::string err;
  int rc = build_host_model(desc, mo->host, err);
  if (rc != 0) {
    arb_set_error(err);
    delete mo;
    return rc;
  }
  *out = mo;
  return 0;
}

extern "C" void arb_model_destroy(arb_model* mo) {
  if (!mo) return;
  for (auto& kv : mo->dev_owned) {
    cudaSetDevice(kv.first);
    for (void* p : kv.second) cudaFree(p);
  }
  delete mo;
}

// ---------------------------------------------------------------------------------
// batch
// ---------------------------------------------------------------------------------
extern "C" int arb_batch_create(const arb_model* model, int64_t nworlds, int device, void* stream,
                                arb_batch** out) {
  if (!model || !out) { arb_set_error("null argument"); return -1; }
  if (nworlds <= 0) { arb_set_error("nworlds must be positive"); return -1; }
  int ndev = 0;
  CUDA_OK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) { arb_set_error("no such CUDA device"); return -1; }
  arb_model* mo = const_cast<arb_model*>(model);
  int rc = model_to_device(mo, device);
  if (rc) return rc;
  arb_batch* b = new arb_batch();
  b->model = mo;
  b->device = device;
  b->stream = (cudaStream_t)stream;
  b->m = mo->dev[device];
  memset(&b->d, 0, sizeof(DevBatch));
  b->d.W = nworlds;
  CUDA_OK(cudaSetDevice(device));
  CUDA_OK(cudaMalloc((void**)&b->d.status, sizeof(int) * nworlds));
  CUDA_OK(cudaMemset(b->d.status, 0, sizeof(int) * nworlds));
  *out = b;
  return 0;
}

// The API-shaped phases keep every intermediate in HBM; that scratch (about
// 114 KB per human36 world) is only allocated when a phase call needs it.
int arb_ensure_phase_scratch(arb_batch* b) {
  if (b->scratch_dbl) return 0;
  CUDA_OK(cudaSetDevice(b->device));
  ScratchSizes s = scratch_sizes(b->model->host);
  const int64_t W = b->d.W;
  CUDA_OK(cudaMalloc((void**)&b->scratch_dbl, sizeof(double) * s.total_doubles() * W));
  CUDA_OK(cudaMalloc((void**)&b->scratch_int, sizeof(int) * s.total_ints() * W));
  CUDA_OK(cudaMemsetAsync(b->scratch_dbl, 0, sizeof(double) * s.total_doubles() * W, b->stream));
  CUDA_OK(cudaMemsetAsync(b->scratch_int, 0, sizeof(int) * s.total_ints() * W, b->stream));
  carve_scratch(s, W, b->scratch_dbl, b->scratch_int, b->d);
  return 0;
}

extern "C" void arb_batch_destroy(arb_batch* b) {
  if (!b) return;
  cudaSetDevice(b->device);
  cudaFree(b->scratch_dbl);
  cudaFree(b->scratch_int);
  cudaFree(b->d.status);
  cudaFree(b->applied_rows);
  cudaFree(b->inertia_rows);
  cudaFree(b->friction_rows);
  arb_fused_release(b);
  delete b;
}

extern "C" int arb_batch_set_stream(arb_batch* b, void* stream) {
  if (!b) { arb_set_error("null batch"); return -1; }
  b->stream = (cudaStream_t)stream;
  return 0;
}

extern "C" int arb_batch_set_option(arb_batch* b, const char* name, int value) {
  if (!b || !name) { arb_set_error("null argument"); return -1; }
  const std::string s(name);
  if (s == "force_phases") b->force_phases = value;
  else if (s == "gs_coop") b->gs_coop = value;
  else if (s == "gs_stage") b->gs_stage = value;
  else if (s == "gs_plain") b->gs_plain_allow = value;
  else if (s == "sort_period") b->sort_period = value < 0 ? 0 : value;
  else if (s == "prepare_group") b->prepare_group = value;
  else if (s == "time_stages") {
    b->time_stages = value;
    for (int i = 0; i < 4; ++i) b->stage_ms[i] = 0.;
  }
  else { arb_set_error("unknown option " + s); return -1; }
  return 0;
}

extern "C" int arb_batch_bind_state(arb_batch* b, double* gpos, double* gvel, double* cforce) {
  if (!b || !gpos || !gvel) { arb_set_error("null state pointer"); return -1; }
  if (b->model->host.nrows > 0 && !cforce) { arb_set_error("cforce is required when the model has constraints"); return -1; }
  b->d.gpos = gpos; b->d.gvel = gvel; b->d.cforce = cforce;
  return 0;
}

extern "C" int arb_model_pd_dofs(const arb_model* model, int32_t* dofs, int cap) {
  if (!model) { arb_set_error("null model"); return -1; }
  const std::vector<int>& v = model->host.pd_dofs;
  if (dofs)
    for (int i = 0; i < (int)v.size() && i < cap; ++i) dofs[i] = v[i];
  return (int)v.size();
}

extern "C" int arb_batch_bind_controller_params(arb_batch* b, const double* kp, const double* kd,
                                                const double* gpos_des, const double* gvel_des) {
  if (!b) { arb_set_error("null batch"); return -1; }
  if ((kp || kd || gpos_des || gvel_des) && b->model->host.pd_dofs.empty()) {
    arb_set_error("the model has no ProportionalDerivativeController"); return -2;
  }
  b->d.pkp = kp; b->d.pkd = kd; b->d.pqd = gpos_des; b->d.pdqd = gvel_des;
  return 0;
}

extern "C" int arb_batch_bind_applied_forces(arb_batch* b, const double* gforce, int nbodies, const int32_t* bodies,
                                             const double* wrench) {
  if (!b) { arb_set_error("null batch"); return -1; }
  std::vector<int> rows;
  std::string err;
  if (applied_wrench_rows(b->model->host, nbodies, bodies, wrench != nullptr, rows, err)) {
    arb_set_error(err);
    return -1;
  }
  CUDA_OK(cudaSetDevice(b->device));
  if (!b->applied_rows) CUDA_OK(cudaMalloc((void**)&b->applied_rows, sizeof(int) * rows.size()));
  // in stream order: the steps already enqueued read the previous table
  CUDA_OK(cudaMemcpyAsync(b->applied_rows, rows.data(), sizeof(int) * rows.size(), cudaMemcpyHostToDevice, b->stream));
  CUDA_OK(cudaStreamSynchronize(b->stream));
  b->applied.tau = gforce;
  b->applied.wrench = nbodies > 0 ? wrench : nullptr;
  b->applied.row = b->applied_rows;
  return 0;
}

extern "C" int arb_batch_bind_body_inertia(arb_batch* b, int nbodies, const int32_t* bodies, const double* inertia) {
  if (!b) { arb_set_error("null batch"); return -1; }
  std::vector<int> rows;
  std::string err;
  if (applied_wrench_rows(b->model->host, nbodies, bodies, inertia != nullptr, rows, err, "inertia")) {
    arb_set_error(err);
    return -1;
  }
  CUDA_OK(cudaSetDevice(b->device));
  if (!b->inertia_rows) CUDA_OK(cudaMalloc((void**)&b->inertia_rows, sizeof(int) * rows.size()));
  // in stream order: the steps already enqueued read the previous table
  CUDA_OK(cudaMemcpyAsync(b->inertia_rows, rows.data(), sizeof(int) * rows.size(), cudaMemcpyHostToDevice, b->stream));
  CUDA_OK(cudaStreamSynchronize(b->stream));
  b->applied.inertia = nbodies > 0 ? inertia : nullptr;
  b->applied.irow = b->inertia_rows;
  return 0;
}

extern "C" int arb_batch_bind_gravity(arb_batch* b, const double* gravity) {
  if (!b) { arb_set_error("null batch"); return -1; }
  if (gravity && b->model->host.nweight == 0) {
    arb_set_error("the model has no WeightController: there is no gravity to replace");
    return -1;
  }
  b->applied.gravity = gravity;
  return 0;
}

extern "C" int arb_batch_bind_contact_friction(arb_batch* b, int ncontacts, const int32_t* constraints, const double* mu) {
  if (!b) { arb_set_error("null batch"); return -1; }
  std::vector<int> rows;
  std::string err;
  if (friction_rows(b->model->host, ncontacts, constraints, mu != nullptr, rows, err)) {
    arb_set_error(err);
    return -1;
  }
  CUDA_OK(cudaSetDevice(b->device));
  if (!b->friction_rows) CUDA_OK(cudaMalloc((void**)&b->friction_rows, sizeof(int) * rows.size()));
  // in stream order: the steps already enqueued read the previous table
  CUDA_OK(cudaMemcpyAsync(b->friction_rows, rows.data(), sizeof(int) * rows.size(), cudaMemcpyHostToDevice, b->stream));
  CUDA_OK(cudaStreamSynchronize(b->stream));
  b->friction.mu = ncontacts > 0 ? mu : nullptr;
  b->friction.row = b->friction_rows;
  return 0;
}

/* 1: arb_step runs the fused stages; 0: it runs the four phase kernels (a controller couples dofs
 * in a way the fused stages do not fold, or "force_phases" is set); *why (optional) names the reason */
extern "C" int arb_batch_step_path(const arb_batch* b, const char** why) {
  if (!b) { arb_set_error("null batch"); return -1; }
  const bool fused = !b->force_phases && arb_fused_supported(b);
  if (why) *why = fused ? "" : (b->force_phases ? "force_phases option" : b->model->host.fused_why.c_str());
  return fused ? 1 : 0;
}

static int check_bound(arb_batch* b) {
  if (!b) { arb_set_error("null batch"); return -1; }
  if (!b->d.gpos) { arb_set_error("state not bound: call arb_batch_bind_state first"); return -2; }
  return 0;
}

// ---------------------------------------------------------------------------------
// lane-per-world kernels
// ---------------------------------------------------------------------------------
#define LPW_THREADS 64

// PARAMS: the instantiations with the world's body inertia and gravity, launched only while either
// is bound (arb_batch_bind_body_inertia / _gravity)
template <bool PARAMS>
__global__ void __launch_bounds__(LPW_THREADS) k_update_dynamic(DevModel m, DevBatch b, DevApplied ap) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < b.W) world_update_dynamic<PARAMS>(m, b, w, ap);
}
template <bool PARAMS>
__global__ void __launch_bounds__(LPW_THREADS) k_update_controllers(DevModel m, DevBatch b, double dt, DevApplied ap) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < b.W) world_update_controllers<PARAMS>(m, b, w, dt, ap);
}
// FRIC: the instantiation with the world's contact friction, launched only while it is bound
// (arb_batch_bind_contact_friction)
template <bool FRIC>
__global__ void __launch_bounds__(LPW_THREADS) k_update_constraints(DevModel m, DevBatch b, double dt, DevFriction fr) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < b.W) world_update_constraints<FRIC>(m, b, w, dt, fr);
}
__global__ void __launch_bounds__(LPW_THREADS) k_integrate(DevModel m, DevBatch b, double dt) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < b.W) world_integrate(m, b, w, dt);
}

static inline unsigned lpw_grid(int64_t W) { return (unsigned)((W + LPW_THREADS - 1) / LPW_THREADS); }
static inline bool params_bound(const arb_batch* b) { return b->applied.inertia || b->applied.gravity; }
static void launch_update_dynamic(arb_batch* b) {
  if (params_bound(b)) k_update_dynamic<true><<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, b->applied);
  else k_update_dynamic<false><<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, b->applied);
}
static void launch_update_controllers(arb_batch* b, double dt) {
  if (params_bound(b))
    k_update_controllers<true><<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, dt, b->applied);
  else k_update_controllers<false><<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, dt, b->applied);
}
static void launch_update_constraints(arb_batch* b, double dt) {
  if (b->friction.mu)
    k_update_constraints<true><<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, dt, b->friction);
  else k_update_constraints<false><<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, dt, b->friction);
}

#define LAUNCH_CHECK(b)                                                        \
  do {                                                                         \
    (b)->launches++;                                                           \
    cudaError_t e_ = cudaGetLastError();                                       \
    if (e_ != cudaSuccess) {                                                   \
      arb_set_error(std::string("kernel launch: ") + cudaGetErrorString(e_)); \
      return -101;                                                             \
    }                                                                          \
  } while (0)

extern "C" int arb_update_dynamic(arb_batch* b) {
  int rc = check_bound(b); if (rc) return rc;
  CUDA_OK(cudaSetDevice(b->device));
  rc = arb_ensure_phase_scratch(b); if (rc) return rc;
  launch_update_dynamic(b);
  LAUNCH_CHECK(b);
  b->last_fused = 0;
  b->half_open = 0;
  return 0;
}
extern "C" int arb_update_controllers(arb_batch* b, double dt) {
  int rc = check_bound(b); if (rc) return rc;
  if (!(dt > 0)) { arb_set_error("dt must be > 0"); return -3; }
  CUDA_OK(cudaSetDevice(b->device));
  rc = arb_ensure_phase_scratch(b); if (rc) return rc;
  launch_update_controllers(b, dt);
  LAUNCH_CHECK(b);
  return 0;
}
extern "C" int arb_update_constraints(arb_batch* b, double dt) {
  int rc = check_bound(b); if (rc) return rc;
  if (!(dt > 0)) { arb_set_error("dt must be > 0"); return -3; }
  CUDA_OK(cudaSetDevice(b->device));
  rc = arb_ensure_phase_scratch(b); if (rc) return rc;
  launch_update_constraints(b, dt);
  LAUNCH_CHECK(b);
  b->last_fused = 0;
  return 0;
}
extern "C" int arb_integrate(arb_batch* b, double dt) {
  int rc = check_bound(b); if (rc) return rc;
  if (!(dt > 0)) { arb_set_error("dt must be > 0"); return -3; }
  CUDA_OK(cudaSetDevice(b->device));
  rc = arb_ensure_phase_scratch(b); if (rc) return rc;
  k_integrate<<<lpw_grid(b->d.W), LPW_THREADS, 0, b->stream>>>(b->m, b->d, dt);
  LAUNCH_CHECK(b);
  return 0;
}

// nsteps of the simulate() loop through the four phase kernels (used when the
// fused stages do not support the model, and by tests).
int arb_step_phases(arb_batch* b, const double* dts, int nsteps) {
  int rc = arb_ensure_phase_scratch(b); if (rc) return rc;
  const unsigned g = lpw_grid(b->d.W);
  for (int s = 0; s < nsteps; ++s) {
    const double dt = dts[s];
    if (!(dt > 0)) { arb_set_error("dt must be > 0"); return -3; }
    launch_update_dynamic(b);
    launch_update_controllers(b, dt);
    launch_update_constraints(b, dt);
    k_integrate<<<g, LPW_THREADS, 0, b->stream>>>(b->m, b->d, dt);
    b->launches += 3;
    LAUNCH_CHECK(b);
  }
  if (nsteps > 0) b->last_fused = 0;
  return 0;
}

extern "C" int arb_step(arb_batch* b, const double* dts, int nsteps) {
  int rc = check_bound(b); if (rc) return rc;
  if (nsteps < 0 || (nsteps > 0 && !dts)) { arb_set_error("bad dts/nsteps"); return -3; }
  CUDA_OK(cudaSetDevice(b->device));
  if (b->force_phases || !arb_fused_supported(b)) return arb_step_phases(b, dts, nsteps);
  rc = arb_fused_step(b, dts, nsteps);
  if (rc == 0 && nsteps > 0) b->last_fused = 1;
  return rc;
}

extern "C" int arb_step_begin(arb_batch* b, double dt) {
  int rc = check_bound(b); if (rc) return rc;
  if (!(dt > 0)) { arb_set_error("dt must be > 0"); return -3; }
  CUDA_OK(cudaSetDevice(b->device));
  if (b->force_phases || !arb_fused_supported(b)) {
    rc = arb_update_dynamic(b); if (rc) return rc;
    rc = arb_update_controllers(b, dt); if (rc) return rc;
    return arb_update_constraints(b, dt);
  }
  rc = arb_fused_step_half(b, dt, 0);
  if (rc == 0) { b->last_fused = 1; b->half_open = 1; }
  return rc;
}
extern "C" int arb_step_end(arb_batch* b, double dt) {
  int rc = check_bound(b); if (rc) return rc;
  if (!(dt > 0)) { arb_set_error("dt must be > 0"); return -3; }
  CUDA_OK(cudaSetDevice(b->device));
  if (!b->half_open) return arb_integrate(b, dt);   // arb_step_begin ran the phase kernels
  b->half_open = 0;
  return arb_fused_step_half(b, dt, 1);
}

extern "C" int arb_step_host(arb_batch* b, double* h_gpos, double* h_gvel, double* h_cforce,
                             const double* dts, int nsteps) {
  int rc = check_bound(b); if (rc) return rc;
  if (!h_gpos || !h_gvel) { arb_set_error("null host state pointer"); return -1; }
  CUDA_OK(cudaSetDevice(b->device));
  const HostModel& h = b->model->host;
  const size_t W = (size_t)b->d.W;
  CUDA_OK(cudaMemcpyAsync(b->d.gpos, h_gpos, sizeof(double) * h.ngpos * W, cudaMemcpyHostToDevice, b->stream));
  CUDA_OK(cudaMemcpyAsync(b->d.gvel, h_gvel, sizeof(double) * h.ndof * W, cudaMemcpyHostToDevice, b->stream));
  // constraint forces are inputs only where the reference keeps them across steps (ball-and-socket
  // warm start, constraints.py:164-182); contact and joint-limit rows are reset by every step
  if (h.nrows > 0 && h_cforce && h.has_warm)
    CUDA_OK(cudaMemcpyAsync(b->d.cforce, h_cforce, sizeof(double) * h.nrows * W, cudaMemcpyHostToDevice, b->stream));
  rc = arb_step(b, dts, nsteps);
  if (rc) return rc;
  CUDA_OK(cudaMemcpyAsync(h_gpos, b->d.gpos, sizeof(double) * h.ngpos * W, cudaMemcpyDeviceToHost, b->stream));
  CUDA_OK(cudaMemcpyAsync(h_gvel, b->d.gvel, sizeof(double) * h.ndof * W, cudaMemcpyDeviceToHost, b->stream));
  if (h.nrows > 0 && h_cforce)
    CUDA_OK(cudaMemcpyAsync(h_cforce, b->d.cforce, sizeof(double) * h.nrows * W, cudaMemcpyDeviceToHost, b->stream));
  CUDA_OK(cudaStreamSynchronize(b->stream));
  return 0;
}

extern "C" int arb_step_host_strided(arb_batch* b, double* h_gpos, double* h_gvel, double* h_cforce,
                                     int64_t host_ld, const double* dts, int nsteps, int synchronize) {
  int rc = check_bound(b); if (rc) return rc;
  if (!h_gpos || !h_gvel) { arb_set_error("null host state pointer"); return -1; }
  if (host_ld < b->d.W) { arb_set_error("host_ld smaller than the number of worlds"); return -1; }
  CUDA_OK(cudaSetDevice(b->device));
  const HostModel& h = b->model->host;
  const size_t W = (size_t)b->d.W, dp = sizeof(double) * W, hp = sizeof(double) * (size_t)host_ld;
  double* dev[3] = {b->d.gpos, b->d.gvel, b->d.cforce};
  double* host[3] = {h_gpos, h_gvel, h_cforce};
  const int rows[3] = {h.ngpos, h.ndof, h_cforce ? h.nrows : 0};
  for (int a = 0; a < 3; ++a)
    if (rows[a] > 0 && (a < 2 || h.has_warm))     // cforce: host -> device only when it is state
      CUDA_OK(cudaMemcpy2DAsync(dev[a], dp, host[a], hp, dp, rows[a], cudaMemcpyHostToDevice, b->stream));
  rc = arb_step(b, dts, nsteps);
  if (rc) return rc;
  for (int a = 0; a < 3; ++a)
    if (rows[a] > 0)
      CUDA_OK(cudaMemcpy2DAsync(host[a], hp, dev[a], dp, dp, rows[a], cudaMemcpyDeviceToHost, b->stream));
  if (synchronize) CUDA_OK(cudaStreamSynchronize(b->stream));
  return 0;
}
extern "C" int arb_state_copy_host_strided(arb_batch* b, double* h_gpos, double* h_gvel, double* h_cforce,
                                           int64_t host_ld, int to_device, void* stream) {
  int rc = check_bound(b); if (rc) return rc;
  if (!h_gpos || !h_gvel) { arb_set_error("null host state pointer"); return -1; }
  if (host_ld < b->d.W) { arb_set_error("host_ld smaller than the number of worlds"); return -1; }
  CUDA_OK(cudaSetDevice(b->device));
  const HostModel& h = b->model->host;
  const size_t W = (size_t)b->d.W, dp = sizeof(double) * W, hp = sizeof(double) * (size_t)host_ld;
  double* dev[3] = {b->d.gpos, b->d.gvel, b->d.cforce};
  double* host[3] = {h_gpos, h_gvel, h_cforce};
  const int rows[3] = {h.ngpos, h.ndof, h_cforce ? h.nrows : 0};
  cudaStream_t st = (cudaStream_t)stream;
  for (int a = 0; a < 3; ++a) {
    if (rows[a] <= 0) continue;
    if (to_device && a == 2 && !h.has_warm) continue;   // cforce is an output only (no ball-and-socket rows)
    if (to_device) CUDA_OK(cudaMemcpy2DAsync(dev[a], dp, host[a], hp, dp, rows[a], cudaMemcpyHostToDevice, st));
    else CUDA_OK(cudaMemcpy2DAsync(host[a], hp, dev[a], dp, dp, rows[a], cudaMemcpyDeviceToHost, st));
  }
  return 0;
}
extern "C" int arb_batch_synchronize(arb_batch* b) {
  if (!b) { arb_set_error("null argument"); return -1; }
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaStreamSynchronize(b->stream));
  return 0;
}

// ---------------------------------------------------------------------------------
// read-backs: SoA scratch -> world-major output
// ---------------------------------------------------------------------------------
__global__ void k_gather(const double* __restrict__ src, double* __restrict__ out, int cnt,
                         int64_t W, int64_t w0, int64_t nw) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw * cnt) return;
  int64_t w = i / cnt;
  int e = (int)(i - w * cnt);
  out[i] = src[(int64_t)e * W + w0 + w];
}
__global__ void k_gather_int(const int* __restrict__ src, int* __restrict__ out, int cnt,
                             int64_t W, int64_t w0, int64_t nw) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw * cnt) return;
  int64_t w = i / cnt;
  int e = (int)(i - w * cnt);
  out[i] = src[(int64_t)e * W + w0 + w];
}
// the same from the fused scratch, tiled [W/32][record][32]; `first`/`stride` select elements
// first, first + stride, ... of the array that starts `off` elements into the record
template <class T>
__global__ void k_gather_tiled(const T* __restrict__ src, T* __restrict__ out, int cnt, int stride,
                               int64_t rec, int64_t w0, int64_t nw, const int* __restrict__ slots) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw * cnt) return;
  int64_t w = i / cnt;
  int e = (int)(i - w * cnt);
  const int64_t ww = slots ? (int64_t)slots[w0 + w] : w0 + w;   // the scratch belongs to the thread slot
  out[i] = src[(ww / ARB_TILE) * rec * ARB_TILE + (int64_t)e * stride * ARB_TILE + ww % ARB_TILE];
}
__global__ void k_get_body(DevModel m, DevBatch b, DevApplied ap, int which, int body, double* out, int64_t w0, int64_t nw) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw) return;
  const int64_t w = w0 + i, W = b.W;
  const int n = m.ndof;
  if (which == ARB_BODY_POSE) {
    Se3 h;
    load_pose(b, body, w, h);
    double* o = out + i * 16;
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) o[4 * r + c] = h.R[3 * r + c];
      o[4 * r + 3] = h.p[r];
    }
    o[12] = o[13] = o[14] = 0.; o[15] = 1.;
  } else if (which == ARB_BODY_TWIST) {
    double t[6];
    load_twist(b, body, w, t);
    for (int r = 0; r < 6; ++r) out[i * 6 + r] = t[r];
  } else if (which == ARB_BODY_JAC || which == ARB_BODY_DJAC) {
    double* o = out + i * 6 * n;
    for (int r = 0; r < 6 * n; ++r) o[r] = 0.;
    const double* src = (which == ARB_BODY_JAC) ? b.J : b.dJ;
    const int off = m.coloff[body], kc = m.kcols[body];
    for (int l = 0; l < kc; ++l)
      for (int r = 0; r < 6; ++r) o[r * n + m.pathdof[off + l]] = AT(src, (off + l) * 6 + r);
  } else if (which == ARB_BODY_NLE) {
    // N_b = [[w^, rx w^ - w^ rx],[0, w^]] M_b   (core.py:1276-1288)
    double* o = out + i * 36;
    double t[6], wx[9], t1[9], t2[9], Om[36];
    load_twist(b, body, w, t);
    for (int r = 0; r < 36; ++r) { Om[r] = 0.; o[r] = 0.; }
    if (body == 0) return;
    skew3(t, wx);
    const double *Mb, *rx;
    double Mw[36], rxw[9];
    world_body_mass<true>(m, ap, body - 1, W, w, Mb, rx, Mw, rxw);   // the world's own M_b if bound
    m3_mul(rx, wx, t1);
    m3_mul(wx, rx, t2);
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) {
        Om[6 * r + c] = wx[3 * r + c];
        Om[6 * (r + 3) + c + 3] = wx[3 * r + c];
        Om[6 * r + c + 3] = t1[3 * r + c] - t2[3 * r + c];
      }
    for (int r = 0; r < 6; ++r)
      for (int c = 0; c < 6; ++c) {
        double s = 0.;
        for (int k = 0; k < 6; ++k) s += Om[6 * r + k] * Mb[6 * k + c];
        o[6 * r + c] = s;
      }
  }
}

static int check_range(arb_batch* b, const void* out, int64_t w0, int64_t w1, bool fused_ok = false) {
  if (!b || !out) { arb_set_error("null argument"); return -1; }
  if (w0 < 0 || w1 > b->d.W || w0 >= w1) { arb_set_error("world range out of bounds"); return -1; }
  if (fused_ok && b->last_fused) return 0;
  if (!b->scratch_dbl) { arb_set_error("nothing to read: no phase call was made on this batch yet"); return -2; }
  if (b->last_fused) {
    // the phase scratch is stale by any number of fused steps: refuse instead of returning old data
    arb_set_error("not formed by the fused step: call arb_update_dynamic / arb_update_controllers first");
    return -2;
  }
  return 0;
}

extern "C" int arb_get_matrix(arb_batch* b, int which, double* out, int64_t w0, int64_t w1) {
  int rc = check_range(b, out, w0, w1); if (rc) return rc;
  CUDA_OK(cudaSetDevice(b->device));
  const double* src = which == ARB_MASS ? b->d.M : which == ARB_NLEFFECTS ? b->d.N
                    : which == ARB_VISCOSITY ? b->d.B : which == ARB_IMPEDANCE ? b->d.Z
                    : which == ARB_ADMITTANCE ? b->d.Y : nullptr;
  if (!src) { arb_set_error("unknown matrix id"); return -1; }
  const int cnt = b->m.ndof * b->m.ndof;
  const int64_t tot = (w1 - w0) * cnt;
  if (tot == 0) return 0;
  k_gather<<<(unsigned)((tot + 255) / 256), 256, 0, b->stream>>>(src, out, cnt, b->d.W, w0, w1 - w0);
  LAUNCH_CHECK(b);
  return 0;
}
extern "C" int arb_get_vector(arb_batch* b, int which, double* out, int64_t w0, int64_t w1) {
  int rc = check_range(b, out, w0, w1); if (rc) return rc;
  CUDA_OK(cudaSetDevice(b->device));
  if (which != ARB_VEC_GFORCE) { arb_set_error("unknown vector id"); return -1; }
  const int cnt = b->m.ndof;
  const int64_t tot = (w1 - w0) * cnt;
  if (tot == 0) return 0;
  k_gather<<<(unsigned)((tot + 255) / 256), 256, 0, b->stream>>>(b->d.gforce, out, cnt, b->d.W, w0, w1 - w0);
  LAUNCH_CHECK(b);
  return 0;
}
// pose (4x4 row-major) / twist of a body from the fused scratch (fpose [nj][12], atw [nj][6])
__global__ void k_get_body_fused(DevBatch b, int which, int body, double* __restrict__ out, int64_t w0, int64_t nw,
                                 const int* __restrict__ slots) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw) return;
  const int64_t s = slots ? (int64_t)slots[w0 + i] : w0 + i;
  const int64_t base = (s / ARB_TILE) * b.frec * ARB_TILE + s % ARB_TILE;
  if (which == ARB_BODY_POSE) {
    double* o = out + i * 16;
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c)
        o[4 * r + c] = body == 0 ? (r == c ? 1. : 0.) : b.fpose[base + (int64_t)((body - 1) * 12 + 3 * r + c) * ARB_TILE];
      o[4 * r + 3] = body == 0 ? 0. : b.fpose[base + (int64_t)((body - 1) * 12 + 9 + r) * ARB_TILE];
    }
    o[12] = o[13] = o[14] = 0.; o[15] = 1.;
  } else {
    for (int r = 0; r < 6; ++r)
      out[i * 6 + r] = body == 0 ? 0. : b.atw[base + (int64_t)((body - 1) * 6 + r) * ARB_TILE];
  }
}
extern "C" int arb_get_body(arb_batch* b, int which, int body, double* out, int64_t w0, int64_t w1) {
  const bool from_fused = b && b->last_fused && (which == ARB_BODY_POSE || which == ARB_BODY_TWIST);
  int rc = check_range(b, out, w0, w1, from_fused); if (rc) return rc;
  CUDA_OK(cudaSetDevice(b->device));
  if (body < 0 || body > b->m.nj) { arb_set_error("body index out of range"); return -1; }
  if (which < ARB_BODY_POSE || which > ARB_BODY_NLE) { arb_set_error("unknown body quantity"); return -1; }
  const int64_t nw = w1 - w0;
  if (from_fused && !b->poses_valid) {
    arb_set_error("body poses / twists are not kept by arb_step with the group prepare stage: use arb_step_begin / arb_step_end");
    return -2;
  }
  if (from_fused) {
    k_get_body_fused<<<(unsigned)((nw + 127) / 128), 128, 0, b->stream>>>(b->d, which, body, out, w0, nw,
                                                                          arb_fused_world_slots(b));
    LAUNCH_CHECK(b);
    return 0;
  }
  k_get_body<<<(unsigned)((nw + 127) / 128), 128, 0, b->stream>>>(b->m, b->d, b->applied, which, body, out, w0, nw);
  LAUNCH_CHECK(b);
  return 0;
}
extern "C" int arb_get_constraint(arb_batch* b, int which, void* out, int64_t w0, int64_t w1) {
  int rc = check_range(b, out, w0, w1, true); if (rc) return rc;
  CUDA_OK(cudaSetDevice(b->device));
  const int nc = b->m.nc;
  if (nc == 0) return 0;
  const int64_t nw = w1 - w0;
  if (b->last_fused) {      // last step ran fused: the quantities live in the tiled fused scratch
    const int cnt = which == ARB_CONS_ZIDX ? 3 * nc : nc;
    const unsigned g = (unsigned)((nw * cnt + 255) / 256);
    const int* slots = arb_fused_world_slots(b);
    if (which == ARB_CONS_SDIST)
      k_gather_tiled<double><<<g, 256, 0, b->stream>>>(b->d.faux, (double*)out, nc, 4, b->d.frec, w0, nw, slots);
    else if (which == ARB_CONS_ACTIVE)
      k_gather_tiled<int><<<g, 256, 0, b->stream>>>(b->d.factive, (int*)out, nc, 1, b->d.firec, w0, nw, slots);
    else if (which == ARB_CONS_BRANCH)
      k_gather_tiled<int><<<g, 256, 0, b->stream>>>(b->d.fbranch, (int*)out, nc, 1, b->d.firec, w0, nw, slots);
    else if (which == ARB_CONS_ZIDX)
      k_gather_tiled<int><<<g, 256, 0, b->stream>>>(b->d.fzidx, (int*)out, cnt, 1, b->d.firec, w0, nw, slots);
    else { arb_set_error("unknown constraint quantity"); return -1; }
    LAUNCH_CHECK(b);
    return 0;
  }
  if (which == ARB_CONS_SDIST) {
    // caux is [nc][4]: gather element 4c
    std::vector<double> dummy;
    const int64_t tot = nw * nc * 4;
    double* tmp = nullptr;
    CUDA_OK(cudaMallocAsync((void**)&tmp, sizeof(double) * tot, b->stream));
    k_gather<<<(unsigned)((tot + 255) / 256), 256, 0, b->stream>>>(b->d.caux, tmp, nc * 4, b->d.W, w0, nw);
    CUDA_OK(cudaMemcpy2DAsync(out, sizeof(double), tmp, 4 * sizeof(double), sizeof(double), nw * nc,
                              cudaMemcpyDeviceToDevice, b->stream));
    CUDA_OK(cudaFreeAsync(tmp, b->stream));
    LAUNCH_CHECK(b);
    return 0;
  }
  const int* src = which == ARB_CONS_ACTIVE ? b->d.cactive : which == ARB_CONS_BRANCH ? b->d.cbranch
                 : which == ARB_CONS_ZIDX ? b->d.czidx : nullptr;
  if (!src) { arb_set_error("unknown constraint quantity"); return -1; }
  const int cnt = which == ARB_CONS_ZIDX ? 3 * nc : nc;
  const int64_t tot = nw * cnt;
  k_gather_int<<<(unsigned)((tot + 255) / 256), 256, 0, b->stream>>>(src, (int*)out, cnt, b->d.W, w0, nw);
  LAUNCH_CHECK(b);
  return 0;
}

// the fused hand-over of worlds [w0, w0 + nw): element e of the array `src` (a base pointer of the tiled
// fused scratch), through the world -> slot map; NaN where generator space was skipped (no active
// constraint, world_fused_prepare) and the identity for the frames of generator bodies that are not aligned
__global__ void k_get_fused(DevModel m, DevBatch b, int which, const double* __restrict__ src, int cnt,
                            double* __restrict__ out, int64_t w0, int64_t nw, const int* __restrict__ slots) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nw * cnt) return;
  const int64_t w = i / cnt;
  const int e = (int)(i - w * cnt);
  const int64_t s = slots ? (int64_t)slots[w0 + w] : w0 + w;
  const int64_t tile = s / ARB_TILE, lane = s % ARB_TILE;
  if (which == ARB_FUSED_GFRAME && !m.gen_aligned[e / 9]) {
    out[i] = (e % 9) % 4 == 0 ? 1. : 0.;
    return;
  }
  if (which != ARB_FUSED_QFREE && which != ARB_FUSED_GFRAME) {
    const int* act = b.factive + tile * b.firec * ARB_TILE + lane;
    bool any = false;
    for (int c = 0; c < m.nc; ++c) any = any || act[c * ARB_TILE];
    if (!any) {
      out[i] = CUDART_NAN;
      return;
    }
  }
  out[i] = src[tile * b.frec * ARB_TILE + (int64_t)e * ARB_TILE + lane];
}
extern "C" int arb_get_fused(arb_batch* b, int which, double* out, int64_t w0, int64_t w1) {
  if (!b || !out) { arb_set_error("null argument"); return -1; }
  if (w0 < 0 || w1 > b->d.W || w0 >= w1) { arb_set_error("world range out of bounds"); return -1; }
  if (!b->fused || !b->last_fused) {
    arb_set_error("no fused hand-over to read: the last step ran the phase kernels, or no fused step was made");
    return -1;
  }
  const DevModel& m = b->m;
  const int NG = m.ngrows;
  const double* src = nullptr;
  int cnt = 0;
  switch (which) {
    case ARB_FUSED_QFREE: src = b->d.fq; cnt = m.ndof; break;
    case ARB_FUSED_V0: src = b->d.fv0; cnt = NG; break;
    case ARB_FUSED_LAMBDA: src = b->d.fLam; cnt = NG * NG; break;
    case ARB_FUSED_GFRAME: src = b->d.fRe; cnt = 9 * m.ngen; break;
    case ARB_FUSED_Y: src = b->d.fy; cnt = NG; break;
    case ARB_FUSED_DELASSUS: src = b->d.fAcc; cnt = 4 * m.nrows; break;
    case ARB_FUSED_K:
      if (!b->last_group) {
        arb_set_error("K = Z^-1 G^T is formed by the prepare_group prepare stage only, and the last step did not run it");
        return -1;
      }
      src = b->d.fK; cnt = m.ndof * NG; break;
    default: arb_set_error("unknown fused quantity"); return -1;
  }
  if (cnt == 0) return 0;
  CUDA_OK(cudaSetDevice(b->device));
  const int64_t nw = w1 - w0;
  k_get_fused<<<(unsigned)((nw * cnt + 255) / 256), 256, 0, b->stream>>>(m, b->d, which, src, cnt, out, w0, nw,
                                                                          arb_fused_world_slots(b));
  LAUNCH_CHECK(b);
  return 0;
}

extern "C" int arb_model_generators(const arb_model* model, int32_t* ngen, int32_t* ngrows, int32_t* gen_body,
                                    int32_t* gen_aligned, int32_t* gen_c0, int32_t* glimdof) {
  if (!model) { arb_set_error("null model"); return -1; }
  const HostModel& h = model->host;
  if (ngen) *ngen = h.ngen;
  if (ngrows) *ngrows = h.ngrows;
  for (int g = 0; g < h.ngen; ++g) {
    if (gen_body) gen_body[g] = h.gen_body[g];
    if (gen_aligned) gen_aligned[g] = h.gen_aligned[g];
    if (gen_c0) gen_c0[g] = h.gen_c0[g];
  }
  if (glimdof)
    for (size_t i = 0; i < h.glimdof.size(); ++i) glimdof[i] = h.glimdof[i];
  return 0;
}

extern "C" int arb_batch_status(arb_batch* b, int32_t* flags) {
  if (!b || !flags) { arb_set_error("null argument"); return -1; }
  CUDA_OK(cudaSetDevice(b->device));
  CUDA_OK(cudaMemcpyAsync(flags, b->d.status, sizeof(int) * b->d.W, cudaMemcpyDeviceToDevice, b->stream));
  CUDA_OK(cudaMemsetAsync(b->d.status, 0, sizeof(int) * b->d.W, b->stream));
  return 0;
}

extern "C" int64_t arb_batch_launch_count(const arb_batch* b) { return b ? b->launches : 0; }

extern "C" int arb_batch_stage_ms(const arb_batch* b, double* out4) {
  if (!b || !out4) { arb_set_error("null argument"); return -1; }
  for (int i = 0; i < 4; ++i) out4[i] = b->stage_ms[i];
  return 0;
}

// ---------------------------------------------------------------------------------
// fp64 FMA peak micro-benchmark (roofline denominator; MEASURED_PEAKS.json has no fp64 entry)
// ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dfma_peak(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 12345.678) out[0] = s;
}

extern "C" int arb_measure_fp64_peak(int device, double* flops_per_s) {
  if (!flops_per_s) { arb_set_error("null argument"); return -1; }
  CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  double* d = nullptr;
  CUDA_OK(cudaMalloc((void**)&d, 8));
  const int blocks = prop.multiProcessorCount * 8, iters = 1 << 15;
  cudaEvent_t e0, e1;
  CUDA_OK(cudaEventCreate(&e0));
  CUDA_OK(cudaEventCreate(&e1));
  double best = 0.;
  for (int rep = 0; rep < 4; ++rep) {
    CUDA_OK(cudaEventRecord(e0));
    k_dfma_peak<<<blocks, 256>>>(d, iters, 0.999999, 1e-9);
    CUDA_OK(cudaEventRecord(e1));
    CUDA_OK(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_OK(cudaEventElapsedTime(&ms, e0, e1));
    double fl = 2.0 * 8.0 * iters * 256.0 * blocks / (ms * 1e-3);
    if (rep > 0 && fl > best) best = fl;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  *flops_per_s = best;
  return 0;
}

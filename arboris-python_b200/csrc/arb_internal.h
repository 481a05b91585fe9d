// Library-private definitions of the opaque ABI handles.
#pragma once
#include <cuda_runtime.h>
#include <map>
#include <set>
#include <string>
#include <vector>
#include "arb_model_host.h"
#include "arb_types.h"

struct arb_model {
  HostModel host;
  std::map<int, DevModel> dev;                 // per CUDA device
  std::map<int, std::vector<void*>> dev_owned;
  std::set<int> dev_ready;
};

struct FusedState;  // arb_fused.cu

struct arb_batch {
  arb_model* model = nullptr;
  int device = 0;
  cudaStream_t stream = nullptr;
  DevModel m;
  DevBatch d;
  double* scratch_dbl = nullptr;   // phase-API scratch (lazy)
  int* scratch_int = nullptr;
  int64_t launches = 0;
  int force_phases = 0;            // tests: run arb_step through the four phase kernels
  int gs_coop = 0;                 // 1: block-cooperative Gauss-Seidel kernel (pooled sliding solves) instead of the per-lane one
  int gs_stage = 1;                // 1 (default): Gauss-Seidel kernel with the contact operands staged in shared memory by TMA
                                   // (world_fused_gs_staged; models of at most 32 constraints), 0: operands loaded from global memory
  int gs_plain = 0;                // set by the fused state: the model qualifies for the plain instantiation of the staged kernel
  int gs_plain_allow = 1;          // option gs_plain (set before the first step): 0 keeps the general instantiation
  int time_stages = 0;             // 1: CUDA events around every fused stage (diagnostic, synchronises per step)
  double stage_ms[4] = {0., 0., 0., 0.};   // accumulated prepare / gs / finish milliseconds, [3] = steps timed
  FusedState* fused = nullptr;
  int sort_period = 2;             // fused path: re-sort the worlds by contact state every N steps (0: never)
  int poses_valid = 1;             // the fused scratch holds the body poses / twists of the last fused step
  int half_group = 0;              // arb_step_begin ran the group prepare stage: arb_step_end runs the K-matrix finish
  int half_open = 0;               // arb_step_begin ran the fused stages: arb_step_end must run the finish stage
  int prepare_group = 0;           // 1: prepare stage with 16 lanes per world and on-chip scratch (arb_group.cuh) + K-matrix finish
  int last_fused = 0;              // 1: the constraint read-backs come from the fused scratch (last step was fused)
  int last_group = 0;              // 1: that step ran the group prepare stage (the scratch holds K, arb_get_fused)
  DevApplied applied = {nullptr, nullptr, nullptr};   // arb_batch_bind_applied_forces
  int* applied_rows = nullptr;     // device [nj]: applied.row (allocated on the first bind)
  int* inertia_rows = nullptr;     // device [nj]: applied.irow (arb_batch_bind_body_inertia, allocated on the first bind)
  DevFriction friction = {nullptr, nullptr};   // arb_batch_bind_contact_friction
  int* friction_rows = nullptr;    // device [nc]: friction.row (allocated on the first bind)
};

const char* arb_set_error(const std::string& s);
int arb_step_phases(arb_batch* b, const double* dts, int nsteps);
int arb_ensure_phase_scratch(arb_batch* b);
// fused step (arb_fused.cu)
bool arb_fused_supported(const arb_batch* b);
int arb_fused_step(arb_batch* b, const double* dts, int nsteps);
void arb_fused_release(arb_batch* b);
const int* arb_fused_world_slots(arb_batch* b);
int arb_fused_step_half(arb_batch* b, double dt, int half);   // 0: prepare + gs, 1: finish

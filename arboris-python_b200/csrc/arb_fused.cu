// Fused step driver: prepare -> gs -> finish per time step (see arb_fused.cuh).
// All three stages are lane-per-world (one world per thread); the scratch between them is tiled
// [W/32][elem][32] (arb_types.h).
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <string>

#include "arb_fused.cuh"
#include "arb_group.cuh"
#include "arb_internal.h"

// World sorting.  The Gauss-Seidel stage is executed warp by warp: a warp pays for a contact
// visit if ANY of its 32 worlds has that contact active, and for the (5x dearer) sliding-friction
// solve if any of them slides there.  Which contacts are active / sliding changes slowly from one
// 1 ms step to the next, so every `sort_period` steps the worlds are re-assigned to threads in the
// order of the key the last Gauss-Seidel left (contacts that slid, active contacts): warps then hold
// worlds in the same contact state.  Only the thread <-> world assignment changes; the arithmetic
// of a world does not depend on its slot, results are bit-identical with and without sorting.
// While an assignment other than the identity is in force the stages work on a PRIVATE copy of
// the state laid out by slot ([elem][slot], coalesced like everything else): it is gathered
// from the caller's arrays (through `perm`) at the start of arb_step and after every re-sort,
// and scattered back before every re-sort and at the end of arb_step, by two pure copy kernels
// -- the 32 lanes of a warp never touch 32 different sectors inside the stages.
struct FusedState {
  double* dbl = nullptr;
  int* ints = nullptr;
  int* perm[2] = {nullptr, nullptr};          // slot -> world, double-buffered
  int* inv = nullptr;                         // world -> slot (read-backs), rebuilt on demand
  unsigned long long* key[2] = {nullptr, nullptr};
  void* cub_tmp = nullptr;
  size_t cub_bytes = 0;
  int cur = 0;
  bool inv_valid = false;
  bool sorted = false;                        // an assignment other than the identity is in force
  int64_t steps = 0;
  double* pstate = nullptr;                   // private state by slot: gpos, gvel, cforce
  int* pstatus = nullptr;                     // status bits by slot, merged into the caller's on scatter
  bool has_K = false;                         // the scratch holds K = Z^-1 G^T (group prepare stage only: 4.7 KB per human36 world)
};

#define CUDA_OKF(call)                                                            \
  do {                                                                            \
    cudaError_t e_ = (call);                                                      \
    if (e_ != cudaSuccess) {                                                      \
      arb_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));          \
      return -100;                                                                \
    }                                                                             \
  } while (0)

#define FUSED_THREADS 64
#ifndef GS_L_SMEM
#define GS_L_SMEM 0     /* 1: the cached Lambda_FF block of the per-lane Gauss-Seidel lives in shared memory */
#endif

#ifndef PREP_MINBLOCKS
#define PREP_MINBLOCKS 1    /* resident-CTA floor of the prepare kernel: 4 = 255 registers, 6 = 168, 8 = 128 */
#endif
#ifndef GS_STAGE_CARVEOUT
#define GS_STAGE_CARVEOUT 40   /* per cent of the SM's 228 KB for shared memory: 2 CTAs x 43 KB (A/B builds) */
#endif
#ifndef GS_STAGE_PLAIN
#define GS_STAGE_PLAIN 1       /* 0: always the general instantiation of the staged kernel (A/B builds) */
#endif
#ifndef GS_CARVEOUT
#define GS_CARVEOUT 0          /* the unstaged kernel uses no shared memory (A/B builds: what a smaller L1 costs) */
#endif
#ifndef GS_MINBLOCKS
#define GS_MINBLOCKS 1
#endif
// s: thread slot = scratch slot = column of the state arrays the kernel was given (the caller's
// arrays under the identity assignment, the private by-slot copy otherwise)
#define FUSED_SLOT_WORLD()                                                  \
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;         \
  const int64_t w = s

// 128-thread CTAs for the lane stages (prepare 4.79 against 4.86 ms with 64 and 5.11 with 32; finish
// 0.739 against 0.773): same resident warps, fewer CTA slots idling behind a CTA's last warp
#ifndef PREP_THREADS
#define PREP_THREADS 128
#endif
#ifndef FINISH_THREADS
#define FINISH_THREADS 128
#endif
template <bool APPLIED>
__global__ void __launch_bounds__(PREP_THREADS, PREP_MINBLOCKS) k_fused_prepare_lane(DevModel m, DevBatch b, double dt, DevApplied ap) {
  FUSED_SLOT_WORLD();
  if (s >= b.W) return;
  world_fused_prepare<APPLIED>(m, fused_tile_view(b, s), w, dt, ap);
}
// the instantiation with the applied-force terms only while some are bound
static void launch_prepare_lane(const arb_batch* b, const DevBatch& d, double dt) {
  const unsigned grid = (unsigned)((d.W + PREP_THREADS - 1) / PREP_THREADS);
  if (b->applied.tau || b->applied.wrench)
    k_fused_prepare_lane<true><<<grid, PREP_THREADS, 0, b->stream>>>(b->m, d, dt, b->applied);
  else k_fused_prepare_lane<false><<<grid, PREP_THREADS, 0, b->stream>>>(b->m, d, dt, b->applied);
}
// Threads per CTA of the Gauss-Seidel kernel: 128 (8.87 ms against 9.01 with 64 and 9.11 with 32 at
// 262144 worlds; end to end, with seven column blocks on three streams, 1.406e7 world-steps/s against
// 1.37e7 / 1.36e7: fewer, fatter CTAs waste less of an SM while a CTA's last warp finishes).  At 255
// registers per thread all three keep 8 resident warps per SM; 96 / 160 / 224 threads (6 / 5 / 7 warps)
// are slower.  GS_THREADS builds another size (A/B).
#ifndef GS_THREADS
#define GS_THREADS 128
#endif
template <int THREADS>
__global__ void __launch_bounds__(THREADS, GS_MINBLOCKS) k_fused_gs(DevModel m, DevBatch b, double dt) {
  FUSED_SLOT_WORLD();
  if (s >= b.W) return;
#if GS_L_SMEM
  __shared__ double sL[36 * THREADS];
  const unsigned long long key = world_fused_gs(m, fused_tile_view(b, s), w, dt, sL + threadIdx.x, THREADS);
#else
  double Lr[36];
  const unsigned long long key = world_fused_gs(m, fused_tile_view(b, s), w, dt, Lr, 1);
#endif
  if (b.fkey != nullptr) b.fkey[s] = key;
}
// Gauss-Seidel with the contact operands staged by TMA (world_fused_gs_staged): 10 KB of shared memory
// and one mbarrier per warp, a 64-byte descriptor per constraint
template <int THREADS, bool PLAIN>
__global__ void __launch_bounds__(THREADS, GS_MINBLOCKS) k_fused_gs_staged(DevModel m, DevBatch b, double dt) {
  __shared__ __align__(128) double sbuf[(THREADS / 32) * (GS_STAGE_WARP_BYTES / 8)];
  __shared__ __align__(16) GsDesc sdesc[32];
  __shared__ __align__(8) unsigned long long sbar[THREADS / 32];
  __shared__ const double* swbase[THREADS / 32][5];
  const unsigned lane = threadIdx.x & 31u, wp = threadIdx.x >> 5;
  GsStage st;
  st.buf = sbuf + wp * (GS_STAGE_WARP_BYTES / 8);
  st.buf_s = (unsigned)__cvta_generic_to_shared(st.buf);
  st.bar_s = (unsigned)__cvta_generic_to_shared(&sbar[wp]);
  st.parity = 0u;
  st.tsel = 0u;
  st.lane = lane;
  st.desc = sdesc;
  st.wbase = swbase[wp];
  if (lane == 0u) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(st.bar_s) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const int64_t s0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // the first slot of the warp's tile
    if (s0 < b.W) {
      const DevBatch t = fused_tile_view(b, s0);
      swbase[wp][0] = t.fAcc; swbase[wp][1] = t.fP; swbase[wp][2] = t.faux; swbase[wp][3] = t.fT1; swbase[wp][4] = t.fT0;
    }
  }
  if ((int)threadIdx.x < m.nc) gs_desc_fill(m, sdesc, threadIdx.x);
  __syncthreads();
  FUSED_SLOT_WORLD();
  (void)w;
  const bool valid = s < b.W;
  const int64_t sv = valid ? s : b.W - 1;
  double Lr[36];
  const unsigned long long key = world_fused_gs_staged<PLAIN>(m, fused_tile_view(b, sv), sv, valid, dt, Lr, 1, st);
  if (valid && b.fkey != nullptr) b.fkey[s] = key;
}
static void launch_gs(const arb_batch* b, const DevBatch& d, double dt) {
  const int64_t W = d.W;
  const unsigned grid = (unsigned)((W + GS_THREADS - 1) / GS_THREADS);
  if (b->gs_stage && b->m.nc <= 32) {
    if (b->gs_plain) k_fused_gs_staged<GS_THREADS, true><<<grid, GS_THREADS, 0, b->stream>>>(b->m, d, dt);
    else k_fused_gs_staged<GS_THREADS, false><<<grid, GS_THREADS, 0, b->stream>>>(b->m, d, dt);
  }
  else
    k_fused_gs<GS_THREADS><<<grid, GS_THREADS, 0, b->stream>>>(b->m, d, dt);
}
// block-cooperative Gauss-Seidel: the sliding-friction solves of a visit are pooled over the
// block through shared memory (world_fused_gs_coop)
#define GS_COOP_THREADS 128
#define GS_COOP_CAP 48        /* queue slots: ~0.2 x 128 sliding contacts per visit in steady state, + 4 sigma */
#ifndef GS_COOP_MINBLOCKS
#define GS_COOP_MINBLOCKS 3
#endif
#define GS_COOP_SMEM (((ARB_SLIDE_NDBL + 4) * GS_COOP_CAP + 1) * sizeof(double) + \
                      (GS_COOP_CAP + 2) * sizeof(int))
__global__ void __launch_bounds__(GS_COOP_THREADS, GS_COOP_MINBLOCKS) k_fused_gs_coop(DevModel m, DevBatch b, double dt) {
  extern __shared__ double smem[];
  GsCoop co;
  co.q = smem;                                         // [21][cap]
  co.r = co.q + ARB_SLIDE_NDBL * GS_COOP_CAP;          // [4][cap]
  co.bm = (unsigned long long*)(co.r + 4 * GS_COOP_CAP);
  co.rs = (int*)(co.bm + 1);                           // [cap]
  co.cnt = co.rs + GS_COOP_CAP;                        // [2]
  co.cap = GS_COOP_CAP; co.tid = threadIdx.x; co.nthr = GS_COOP_THREADS; co.parity = 0;
  FUSED_SLOT_WORLD();
  const bool valid = s < b.W;
  double Lr[36];     // cached Lambda_FF block: registers (shared memory would shrink the L1)
  const unsigned long long key = world_fused_gs_coop(m, fused_tile_view(b, valid ? s : b.W - 1), w, valid, dt, co, Lr, 1);
  if (valid && b.fkey != nullptr) b.fkey[s] = key;
}

__global__ void __launch_bounds__(FINISH_THREADS) k_fused_finish(DevModel m, DevBatch b, double dt) {
  FUSED_SLOT_WORLD();
  if (s < b.W) world_fused_finish(m, fused_tile_view(b, s), w, dt);
}

// prepare stage with a group of 16 lanes per world and the world's intermediates in shared memory
// (arb_group.cuh); GROUP_WPC worlds per CTA, one record of m.gl.total doubles each
#ifndef GROUP_WPC
#define GROUP_WPC 2
#endif
__global__ void __launch_bounds__(GROUP_WPC * ARB_GL) k_fused_prepare_group(DevModel m, DevBatch b, double dt, int write_poses) {
  extern __shared__ double gsm[];
  const int gidx = threadIdx.x / ARB_GL;
  const int64_t s = (int64_t)blockIdx.x * GROUP_WPC + gidx;
  if (s >= b.W) return;
  GroupCtx g;
  g.sm = gsm + (size_t)gidx * m.gl.total;
  g.lane = threadIdx.x % ARB_GL;
  g.mask = 0xFFFFu << ((threadIdx.x & 31) & 16);
  group_prepare(m, fused_tile_view(b, s), s, dt, g, write_poses != 0);
}
__global__ void __launch_bounds__(FUSED_THREADS) k_fused_finish_k(DevModel m, DevBatch b, double dt) {
  FUSED_SLOT_WORLD();
  if (s < b.W) world_fused_finish_k(m, fused_tile_view(b, s), w, dt);
}
static size_t group_smem_bytes(const arb_batch* b) { return sizeof(double) * (size_t)b->m.gl.total * GROUP_WPC; }
// the group stage needs its per-world record to fit the SM's shared memory
static bool group_supported(const arb_batch* b) { return group_smem_bytes(b) <= 227 * 1024; }
// the group prepare stage has no applied-force term: refused rather than stepping without the forces
static int group_refuses_applied(const arb_batch* b) {
  if (!(b->prepare_group && group_supported(b) && (b->applied.tau || b->applied.wrench))) return 0;
  arb_set_error("the prepare_group option does not support applied forces (arb_batch_bind_applied_forces): "
                "unbind them or clear the option");
  return -1;
}

// private by-slot state <- caller's state (GATHER) or the reverse; one thread per slot and
// ELEMS_PER_BLOCK_Y elements, the by-slot side coalesced
#define STATE_EPB 8
template <bool GATHER>
__global__ void k_state_copy(double* __restrict__ caller, double* __restrict__ priv, const int* __restrict__ perm,
                             int nelem, int64_t W) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= W) return;
  const int64_t w = perm[s];
  const int e0 = blockIdx.y * STATE_EPB;
#pragma unroll
  for (int i = 0; i < STATE_EPB; ++i) {
    const int e = e0 + i;
    if (e < nelem) {
      if (GATHER) priv[(int64_t)e * W + s] = caller[(int64_t)e * W + w];
      else caller[(int64_t)e * W + w] = priv[(int64_t)e * W + s];
    }
  }
}
__global__ void k_status_merge(int* __restrict__ caller, int* __restrict__ priv, const int* __restrict__ perm, int64_t W) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= W) return;
  const int v = priv[s];
  if (v) { caller[perm[s]] |= v; priv[s] = 0; }
}
__global__ void k_iota(int* p, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (int)i;
}
__global__ void k_invert_perm(const int* __restrict__ perm, int* __restrict__ inv, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) inv[perm[i]] = (int)i;
}

// the fused stages fold controllers per dof: PD gains must be diagonal (arb_model_host.h)
bool arb_fused_supported(const arb_batch* b) { return b->model->host.fused_ok != 0; }

static int ensure_fused_scratch(arb_batch* b) {
  if (b->fused) return 0;
  FusedSizes s = fused_sizes(b->model->host);
  const int64_t W = fused_padded_worlds(b->d.W);
  FusedState* f = new FusedState();
  f->has_K = b->prepare_group != 0;           // (the option must be set before the first step)
  if (!f->has_K) s.fK = 0;
  CUDA_OKF(cudaMalloc((void**)&f->dbl, sizeof(double) * s.total_doubles() * W));
  CUDA_OKF(cudaMalloc((void**)&f->ints, sizeof(int) * s.total_ints() * W));
  CUDA_OKF(cudaMemsetAsync(f->dbl, 0, sizeof(double) * s.total_doubles() * W, b->stream));
  CUDA_OKF(cudaMemsetAsync(f->ints, 0, sizeof(int) * s.total_ints() * W, b->stream));
  carve_fused(s, f->dbl, f->ints, b->d);
  // world sorting: only models with constraints (the key comes from the Gauss-Seidel stage);
  // 32-bit world indices
  if (b->m.nc > 0 && b->d.W < (int64_t)1 << 31) {
    const int64_t n = b->d.W;
    for (int i = 0; i < 2; ++i) {
      CUDA_OKF(cudaMalloc((void**)&f->perm[i], sizeof(int) * n));
      CUDA_OKF(cudaMalloc((void**)&f->key[i], sizeof(unsigned long long) * n));
    }
    CUDA_OKF(cudaMalloc((void**)&f->inv, sizeof(int) * n));
    CUDA_OKF(cudaMemsetAsync(f->key[0], 0, sizeof(unsigned long long) * n, b->stream));
    k_iota<<<(unsigned)((n + 255) / 256), 256, 0, b->stream>>>(f->perm[0], n);
    k_iota<<<(unsigned)((n + 255) / 256), 256, 0, b->stream>>>(f->inv, n);
    f->inv_valid = true;
    CUDA_OKF(cub::DeviceRadixSort::SortPairsDescending(nullptr, f->cub_bytes, f->key[0], f->key[1], f->perm[0], f->perm[1],
                                             (int)n, 0, 64, b->stream));
    CUDA_OKF(cudaMalloc(&f->cub_tmp, f->cub_bytes ? f->cub_bytes : 1));
    const HostModel& h = b->model->host;
    CUDA_OKF(cudaMalloc((void**)&f->pstate, sizeof(double) * (h.ngpos + h.ndof + (h.nrows > 0 ? h.nrows : 1)) * n));
    CUDA_OKF(cudaMalloc((void**)&f->pstatus, sizeof(int) * n));
    CUDA_OKF(cudaMemsetAsync(f->pstatus, 0, sizeof(int) * n, b->stream));
    b->d.perm = f->perm[0];
    b->d.fkey = f->key[0];
  }
  CUDA_OKF(cudaFuncSetAttribute(k_fused_gs_coop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GS_COOP_SMEM));
  if (group_supported(b))
    CUDA_OKF(cudaFuncSetAttribute(k_fused_prepare_group, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)group_smem_bytes(b)));
  // the per-lane stages live on L1 (operands re-read every sweep / pass): no shared-memory carve-out
  CUDA_OKF(cudaFuncSetAttribute(k_fused_gs<GS_THREADS>, cudaFuncAttributePreferredSharedMemoryCarveout, GS_L_SMEM ? 20 : GS_CARVEOUT));
  // (staged: 2 CTAs x 43 KB per SM; the driver rounds the carve-out up to the next configuration)
  CUDA_OKF(cudaFuncSetAttribute(k_fused_gs_staged<GS_THREADS, false>, cudaFuncAttributePreferredSharedMemoryCarveout, GS_STAGE_CARVEOUT));
  CUDA_OKF(cudaFuncSetAttribute(k_fused_gs_staged<GS_THREADS, true>, cudaFuncAttributePreferredSharedMemoryCarveout, GS_STAGE_CARVEOUT));
  {   // the plain instantiation serves models of joint limits and contact-aligned one-body contacts only
    const HostModel& hm = b->model->host;
    bool plain = GS_STAGE_PLAIN != 0 && b->gs_plain_allow != 0;
    for (int c = 0; c < hm.nc; ++c) {
      const bool lim = hm.ctype[c] == ARB_CONS_JOINT_LIMITS;
      const bool alc = hm.ctype[c] == ARB_CONS_SOFT_FINGER_PLANE_POINT && hm.caligned[c] != 0 &&
                       ((hm.cgen1[c] >= 0) != (hm.cgen0[c] >= 0));
      plain = plain && (lim || alc);
    }
    b->gs_plain = plain ? 1 : 0;
  }
  CUDA_OKF(cudaFuncSetAttribute(k_fused_prepare_lane<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  CUDA_OKF(cudaFuncSetAttribute(k_fused_prepare_lane<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  CUDA_OKF(cudaFuncSetAttribute(k_fused_finish, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
  b->fused = f;
  return 0;
}



// caller's state <-> private by-slot state through the current assignment
static int fused_state_sync(arb_batch* b, bool gather) {
  FusedState* f = b->fused;
  const HostModel& h = b->model->host;
  const int64_t W = b->d.W;
  const int* perm = f->perm[f->cur];
  double* priv = f->pstate;
  double* caller[3] = {b->d.gpos, b->d.gvel, b->d.cforce};
  const int nelem[3] = {h.ngpos, h.ndof, h.nrows};
  for (int a = 0; a < 3; ++a) {
    if (nelem[a] > 0) {
      const dim3 grid((unsigned)((W + 255) / 256), (unsigned)((nelem[a] + STATE_EPB - 1) / STATE_EPB));
      if (gather) k_state_copy<true><<<grid, 256, 0, b->stream>>>(caller[a], priv, perm, nelem[a], W);
      else k_state_copy<false><<<grid, 256, 0, b->stream>>>(caller[a], priv, perm, nelem[a], W);
      b->launches += 1;
    }
    priv += (int64_t)(a == 2 ? 0 : nelem[a]) * W;
  }
  if (!gather) {
    k_status_merge<<<(unsigned)((W + 255) / 256), 256, 0, b->stream>>>(b->d.status, f->pstatus, perm, W);
    b->launches += 1;
  }
  const cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) { arb_set_error(std::string("state copy launch: ") + cudaGetErrorString(e)); return -101; }
  return 0;
}

int arb_fused_step(arb_batch* b, const double* dts, int nsteps) {
  for (int s = 0; s < nsteps; ++s)       // before anything is enqueued: a bad dt leaves the state untouched
    if (!(dts[s] > 0)) { arb_set_error("dt must be > 0"); return -3; }
  int rc = group_refuses_applied(b);
  if (rc) return rc;
  rc = ensure_fused_scratch(b);
  if (rc) return rc;
  FusedState* f = b->fused;
  const HostModel& h = b->model->host;
  const int64_t W = b->d.W;
  const unsigned g = (unsigned)((W + FUSED_THREADS - 1) / FUSED_THREADS);
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  if (f->sorted && b->sort_period <= 0) {       // sorting switched off: back to the identity
    k_iota<<<(unsigned)((W + 255) / 256), 256, 0, b->stream>>>(f->perm[f->cur], W);
    f->sorted = false;
    f->inv_valid = false;
  }
  // the batch the stages see: the caller's state arrays under the identity assignment,
  // the private by-slot copy otherwise
  DevBatch d = b->d;
  auto point_at_private = [&]() {
    d.gpos = f->pstate;
    d.gvel = d.gpos + (int64_t)h.ngpos * W;
    d.cforce = d.gvel + (int64_t)h.ndof * W;
    d.status = f->pstatus;
  };
  bool priv_valid = false;
  // every exit goes through here: the live state goes back to the caller's arrays (the steps
  // already enqueued are not lost when a later call fails) and the timing events are released
  auto leave = [&](int code) {
    if (f->sorted && priv_valid) {
      const int rs = fused_state_sync(b, false);
      if (code == 0) code = rs;
    }
    for (int i = 0; i < 4; ++i)
      if (ev[i]) cudaEventDestroy(ev[i]);
    return code;
  };
#define CUDA_OKL(call)                                                            \
  do {                                                                            \
    cudaError_t e_ = (call);                                                      \
    if (e_ != cudaSuccess) {                                                      \
      arb_set_error(std::string(#call) + ": " + cudaGetErrorString(e_));          \
      return leave(-100);                                                         \
    }                                                                             \
  } while (0)
  if (b->time_stages)
    for (int i = 0; i < 4; ++i) CUDA_OKL(cudaEventCreate(&ev[i]));
  // (a call whose first step re-sorts anyway does not gather first: the caller's arrays are the
  // state at that point -- one gather and one scatter less per sort for callers that step once per
  // call, like the end-to-end pipeline)
  const bool sort_first = nsteps > 0 && f->perm[0] != nullptr && b->sort_period > 0 && f->steps > 0 &&
                          (f->steps % b->sort_period) == 0;
  if (f->sorted && !sort_first) {
    rc = fused_state_sync(b, true);
    if (rc) return leave(rc);
    point_at_private();
    priv_valid = true;
  }
  for (int s = 0; s < nsteps; ++s) {
    const double dt = dts[s];
    if (f->perm[0] != nullptr && b->sort_period > 0 && f->steps > 0 && (f->steps % b->sort_period) == 0) {
      // re-assign worlds to threads by the key of the previous step, DESCENDING: the CTAs of the
      // worlds with the most contact work are dispatched first and the grid's tail is made of the
      // cheap ones (stable: ties keep their order).  Done BEFORE the step, so that after a step the scratch read-backs
      // (arb_get_constraint) still see the assignment the step ran with.
      if (f->sorted && priv_valid) {
        priv_valid = false;
        rc = fused_state_sync(b, false);
        if (rc) return leave(rc);
      }
      const int nb = b->m.nc < 32 ? b->m.nc : 32;
      const int c = f->cur;
      CUDA_OKL(cub::DeviceRadixSort::SortPairsDescending(f->cub_tmp, f->cub_bytes, f->key[c], f->key[c ^ 1], f->perm[c],
                                               f->perm[c ^ 1], (int)W, 0, 2 * nb, b->stream));
      f->cur = c ^ 1;
      b->d.perm = d.perm = f->perm[f->cur];
      b->d.fkey = d.fkey = f->key[f->cur];     // (the sorted keys are overwritten by the next Gauss-Seidel)
      f->inv_valid = false;
      f->sorted = true;
      b->launches += 1;
      rc = fused_state_sync(b, true);
      if (rc) return leave(rc);
      point_at_private();
      priv_valid = true;
    }
    const bool grp = b->prepare_group && group_supported(b);
    if (grp && !f->has_K) {
      arb_set_error("set the prepare_group option before the batch's first step (its scratch has no room for K)");
      return leave(-3);
    }
    b->poses_valid = grp ? 0 : 1;      // (the group stage keeps poses on chip unless asked: arb_step_begin)
    if (ev[0]) cudaEventRecord(ev[0], b->stream);
    if (grp)
      k_fused_prepare_group<<<(unsigned)((W + GROUP_WPC - 1) / GROUP_WPC), GROUP_WPC * ARB_GL, group_smem_bytes(b), b->stream>>>(b->m, d, dt, 0);
    else
      launch_prepare_lane(b, d, dt);
    if (ev[0]) cudaEventRecord(ev[1], b->stream);
    if (b->m.nc > 0) {
      if (b->m.nc <= 64 && b->gs_coop)
        k_fused_gs_coop<<<(unsigned)((W + GS_COOP_THREADS - 1) / GS_COOP_THREADS), GS_COOP_THREADS,
                          GS_COOP_SMEM, b->stream>>>(b->m, d, dt);
      else
        launch_gs(b, d, dt);
    }
    if (ev[0]) cudaEventRecord(ev[2], b->stream);
    if (grp) k_fused_finish_k<<<g, FUSED_THREADS, 0, b->stream>>>(b->m, d, dt);
    else k_fused_finish<<<(unsigned)((W + FINISH_THREADS - 1) / FINISH_THREADS), FINISH_THREADS, 0, b->stream>>>(b->m, d, dt);
    b->launches += (b->m.nc > 0) ? 3 : 2;
    ++f->steps;
    if (ev[0]) {   // diagnostic mode: per-stage device time of this step
      cudaEventRecord(ev[3], b->stream);
      CUDA_OKL(cudaEventSynchronize(ev[3]));
      for (int i = 0; i < 3; ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
        b->stage_ms[i] += ms;
      }
      b->stage_ms[3] += 1.;
    }
  }
#undef CUDA_OKL
  rc = leave(0);
  if (rc) return rc;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { arb_set_error(std::string("kernel launch: ") + cudaGetErrorString(e)); return -101; }
  return 0;
}

// One step in two halves (arb_step_begin / arb_step_end): identity assignment, the caller's
// state arrays, so that everything the caller reads between the halves is in place.
int arb_fused_step_half(arb_batch* b, double dt, int half) {
  int rc = half == 0 ? group_refuses_applied(b) : 0;
  if (rc) return rc;
  rc = ensure_fused_scratch(b);
  if (rc) return rc;
  FusedState* f = b->fused;
  const int64_t W = b->d.W;
  const unsigned g = (unsigned)((W + FUSED_THREADS - 1) / FUSED_THREADS);
  if (f->sorted) {
    k_iota<<<(unsigned)((W + 255) / 256), 256, 0, b->stream>>>(f->perm[f->cur], W);
    f->sorted = false;
    f->inv_valid = false;
  }
  const bool grp = b->prepare_group && group_supported(b);
  if (grp && !f->has_K) {
    arb_set_error("set the prepare_group option before the batch's first step (its scratch has no room for K)");
    return -3;
  }
  if (half == 0) {
    b->half_group = grp ? 1 : 0;       // the finish half must match the prepare half
    b->poses_valid = 1;
    if (grp)
      k_fused_prepare_group<<<(unsigned)((W + GROUP_WPC - 1) / GROUP_WPC), GROUP_WPC * ARB_GL, group_smem_bytes(b), b->stream>>>(b->m, b->d, dt, 1);
    else
      launch_prepare_lane(b, b->d, dt);
    if (b->m.nc > 0) launch_gs(b, b->d, dt);
    b->launches += (b->m.nc > 0) ? 2 : 1;
  } else {
    if (b->half_group) k_fused_finish_k<<<g, FUSED_THREADS, 0, b->stream>>>(b->m, b->d, dt);
    else k_fused_finish<<<(unsigned)((W + FINISH_THREADS - 1) / FINISH_THREADS), FINISH_THREADS, 0, b->stream>>>(b->m, b->d, dt);
    b->launches += 1;
    ++f->steps;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { arb_set_error(std::string("kernel launch: ") + cudaGetErrorString(e)); return -101; }
  return 0;
}

// world -> slot map of the current assignment (device pointer), or nullptr for the identity
const int* arb_fused_world_slots(arb_batch* b) {
  FusedState* f = b->fused;
  if (!f || !f->perm[0]) return nullptr;
  if (!f->inv_valid) {
    const int64_t n = b->d.W;
    k_invert_perm<<<(unsigned)((n + 255) / 256), 256, 0, b->stream>>>(f->perm[f->cur], f->inv, n);
    f->inv_valid = true;
  }
  return f->inv;
}

void arb_fused_release(arb_batch* b) {
  if (!b->fused) return;
  cudaFree(b->fused->dbl);
  cudaFree(b->fused->ints);
  for (int i = 0; i < 2; ++i) { cudaFree(b->fused->perm[i]); cudaFree(b->fused->key[i]); }
  cudaFree(b->fused->inv);
  cudaFree(b->fused->cub_tmp);
  cudaFree(b->fused->pstate);
  cudaFree(b->fused->pstatus);
  delete b->fused;
  b->fused = nullptr;
}

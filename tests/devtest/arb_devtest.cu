// TEST INFRASTRUCTURE ONLY.  Device unit harness of the small dense routines and the soft-finger
// contact solve (arboris-python_b200/csrc), one problem per thread in 128-thread blocks, inputs and
// outputs element-major [elem][N].  Built by tests/devtest/harness.py with the package's nvcc flags
// (plus optional -D variant flags) into tests/devtest/_build/; the package never loads it.
//
// Caveat: a test kernel is a separate compilation context.  ptxas may contract and inline the
// routines differently here than inside k_fused_gs_staged or k_fused_gs_coop, so this harness tests
// the DEVICE ARITHMETIC of the routines (FMA contraction, the MUFU seeds of the Laguerre step, the
// ballot and shared-memory-queue call forms), not the SASS of the product kernels.  The world-level
// GPU tests remain the check on the product kernels.
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../arboris-python_b200/csrc/arb_fused.cuh"
#include "../../arboris-python_b200/csrc/arb_group.cuh"
#include "../../arboris-python_b200/csrc/arb_internal.h"

#define DT_THREADS 128
#define DT_CAP 48        /* queue slots of the pooled sliding solve, as GS_COOP_CAP */
#define EL(p, e) (p)[(int64_t)(e) * N + i]

static inline int dt_blocks(int N) { return (N + DT_THREADS - 1) / DT_THREADS; }
static inline int dt_err() { return (int)cudaGetLastError(); }

// SoftFingerContact.solve, phase-kernel form (P = pinv(A) given)
__global__ void __launch_bounds__(DT_THREADS) k_softfinger_solve(int N, const double* v, const double* A, const double* P,
                                                                 const double* sdist, const double* mu, const double* eps,
                                                                 double dt, double* f, double* df, int* br, int* st) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double vv[4], a[16], p[16], e[3], ff[4], d[4];
  for (int k = 0; k < 4; ++k) { vv[k] = EL(v, k); ff[k] = EL(f, k); }
  for (int k = 0; k < 16; ++k) { a[k] = EL(A, k); p[k] = EL(P, k); }
  for (int k = 0; k < 3; ++k) e[k] = EL(eps, k);
  int status = 0;
  const int b = softfinger_solve(vv, a, p, EL(sdist, 0), EL(mu, 0), e, dt, ff, d, &status);
  for (int k = 0; k < 4; ++k) { EL(f, k) = ff[k]; EL(df, k) = d[k]; }
  EL(br, 0) = b;
  EL(st, 0) = status;
}

// The fused Gauss-Seidel form: softfinger_begin_tiled on a tiled shared-memory copy of A and P,
// then softfinger_sliding in one of three call forms that must give identical bits:
//   mode 0: per lane, coop = 0;
//   mode 1: with the ballot mask of the sliding lanes (gs_visit_contact_staged, GS_STAGE_COOP_ROOT);
//   mode 2: pooled through a GsCoop queue in shared memory (gs_softfinger_begin, coop_solve_sliding).
// eps (3 doubles) is uniform over the launch: a constraint's eps is a model constant.  Threads past N
// take the last problem and do not write, as the product kernels do with lanes beyond the batch.
__global__ void __launch_bounds__(DT_THREADS) k_softfinger_fused(int N, int mode, const double* v, const double* A,
                                                                 const double* P, const double* aux, const double* mu,
                                                                 const double* eps, double dt, double* f, double* df,
                                                                 int* br, int* st) {
  __shared__ double tile[DT_THREADS / 32][32][ARB_TILE];      // per warp: A (16 rows), P (16 rows)
  __shared__ double cq[(ARB_SLIDE_NDBL + 4) * DT_CAP];
  __shared__ int crs[DT_CAP], ccnt[2];
  __shared__ unsigned long long cbm;
  const int64_t gi = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  const bool valid = gi < N;
  const int64_t i = valid ? gi : N - 1;
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  for (int k = 0; k < 16; ++k) { tile[warp][k][lane] = EL(A, k); tile[warp][16 + k][lane] = EL(P, k); }
  if (threadIdx.x == 0) { ccnt[0] = ccnt[1] = 0; cbm = 0ull; }
  __syncthreads();
  double vv[4], ff[4], d[4], e[3], a[16], alpha[4];
  for (int k = 0; k < 4; ++k) { vv[k] = EL(v, k); ff[k] = EL(f, k); }
  for (int k = 0; k < 3; ++k) e[k] = eps[k];
  const double m = EL(mu, 0);
  int status = 0;
  const int b = softfinger_begin_tiled(vv, &tile[warp][0][lane], &tile[warp][16][lane], EL(aux, 0), EL(aux, 1), m, e,
                                       dt, ff, d, a, alpha);
  if (mode == 2) {
    GsCoop co;
    co.q = cq;
    co.r = cq + ARB_SLIDE_NDBL * DT_CAP;
    co.rs = crs; co.cnt = ccnt; co.bm = &cbm;
    co.cap = DT_CAP; co.tid = threadIdx.x; co.nthr = DT_THREADS; co.parity = 0;
    int slot = -1;
    if (b == 3) {
      slot = coop_inc(&co.cnt[co.parity]);
      if (slot < co.cap) {
        for (int k = 0; k < 16; ++k) co.q[k * co.cap + slot] = a[k];
        for (int k = 0; k < 4; ++k) co.q[(16 + k) * co.cap + slot] = alpha[k];
        co.q[20 * co.cap + slot] = m;
      } else {           // queue full: solve in place, as gs_softfinger_begin does
        double newf[4];
        softfinger_sliding(a, alpha, m, e, newf, &status);
        for (int k = 0; k < 4; ++k) { d[k] = newf[k] - ff[k]; ff[k] = newf[k]; }
      }
    }
    coop_solve_sliding(co, e);
    if (b == 3 && slot < co.cap) {
      for (int k = 0; k < 4; ++k) {
        const double nf = co.r[k * co.cap + slot];
        d[k] = nf - ff[k];
        ff[k] = nf;
      }
      status |= co.rs[slot];
    }
  } else {
    const unsigned slmask = mode == 1 ? __ballot_sync(0xffffffffu, b == 3) : 0u;
    if (b == 3) {
      double newf[4];
      softfinger_sliding(a, alpha, m, e, newf, &status, slmask);
      for (int k = 0; k < 4; ++k) { d[k] = newf[k] - ff[k]; ff[k] = newf[k]; }
    }
  }
  if (!valid) return;
  for (int k = 0; k < 4; ++k) { EL(f, k) = ff[k]; EL(df, k) = d[k]; }
  EL(br, 0) = b;
  EL(st, 0) = status;
}

// sliding_root_structured; coop = 1: every lane of the warp calls with the full mask (the staged form)
__global__ void __launch_bounds__(DT_THREADS) k_sliding_root(int N, int coop, const double* A, const double* alpha,
                                                             const double* mu, double* s, int* found, int* ok) {
  const int64_t gi = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  const bool valid = gi < N;
  const int64_t i = valid ? gi : N - 1;
  double a[16], al[4];
  for (int k = 0; k < 16; ++k) a[k] = EL(A, k);
  for (int k = 0; k < 4; ++k) al[k] = EL(alpha, k);
  double so = 0.;
  bool fo = false;
  const bool r = sliding_root_structured(a, al, EL(mu, 0), &so, &fo, coop ? 0xffffffffu : 0u);
  if (!valid) return;
  EL(s, 0) = so;
  EL(found, 0) = fo ? 1 : 0;
  EL(ok, 0) = r ? 1 : 0;
}

// the sextic routines on one monic polynomial p[0..5] per thread, and poly6_certify at x
__global__ void __launch_bounds__(DT_THREADS) k_poly6(int N, const double* p, const double* x, int* fast_ok,
                                                      double* fast_root, int* positive, int* slow_n, double* slow_root,
                                                      int* certify) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double c[7], q[6];
  for (int k = 0; k < 6; ++k) q[k] = c[k] = EL(p, k);
  c[6] = 1.;
  double r = 0.;
  EL(fast_ok, 0) = poly6_largest_root_fast(c, &r);
  EL(fast_root, 0) = r;
  EL(positive, 0) = poly6_positive_on_halfline(q) ? 1 : 0;
  double T = 0.;
  for (int k = 0; k < 6; ++k) T = fmax(T, fabs(q[k]));
  T += 1.;
  double roots[6];
  const int nr = poly6_roots_slow(c, T, roots);
  EL(slow_n, 0) = nr;
  EL(slow_root, 0) = nr ? roots[nr - 1] : 0.;
  EL(certify, 0) = poly6_certify(q, EL(x, 0)) ? 1 : 0;
}

__global__ void __launch_bounds__(DT_THREADS) k_eig6(int N, const double* A, double* wr, double* wi, int* ok) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double a[36], r[6], im[6];
  for (int k = 0; k < 36; ++k) a[k] = EL(A, k);
  EL(ok, 0) = eig_real_general6(a, r, im) ? 1 : 0;
  for (int k = 0; k < 6; ++k) { EL(wr, k) = r[k]; EL(wi, k) = im[k]; }
}

template <int M>
__global__ void __launch_bounds__(DT_THREADS) k_pinv(int N, const double* A, double* out) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double a[M * M], o[M * M];
  for (int k = 0; k < M * M; ++k) a[k] = EL(A, k);
  pinv_small<M>(a, o);
  for (int k = 0; k < M * M; ++k) EL(out, k) = o[k];
}

__global__ void __launch_bounds__(DT_THREADS) k_inv_cond4(int N, const double* A, double* out, double* cond) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double a[16], o[16];
  for (int k = 0; k < 16; ++k) a[k] = EL(A, k);
  EL(cond, 0) = inv_small_cond<4>(a, o);
  for (int k = 0; k < 16; ++k) EL(out, k) = o[k];
}

__global__ void __launch_bounds__(DT_THREADS) k_solve4(int N, const double* A, const double* b, double* x, int* ok) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double a[16], bb[4], xx[4];
  for (int k = 0; k < 16; ++k) a[k] = EL(A, k);
  for (int k = 0; k < 4; ++k) bb[k] = EL(b, k);
  EL(ok, 0) = solve_small<4>(a, bb, xx) ? 1 : 0;
  for (int k = 0; k < 4; ++k) EL(x, k) = xx[k];
}

__global__ void __launch_bounds__(DT_THREADS) k_se3_exp(int N, const double* tw, double* out) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double t[6];
  for (int k = 0; k < 6; ++k) t[k] = EL(tw, k);
  Se3 h;
  se3_exp(t, h);
  for (int k = 0; k < 9; ++k) EL(out, k) = h.R[k];
  for (int k = 0; k < 3; ++k) EL(out, 9 + k) = h.p[k];
}

__global__ void __launch_bounds__(DT_THREADS) k_zaligned(int N, const double* z, double* R, int* idx) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double zz[3], r[9];
  int ix[3];
  for (int k = 0; k < 3; ++k) zz[k] = EL(z, k);
  zaligned(zz, r, ix);
  for (int k = 0; k < 9; ++k) EL(R, k) = r[k];
  for (int k = 0; k < 3; ++k) EL(idx, k) = ix[k];
}

// contact_collide: frames as 12 doubles (R row-major, p); cd holds ARB_CONS_NDBL doubles per problem
__global__ void __launch_bounds__(DT_THREADS) k_collide(int N, const int* pair, const double* cd, const double* H0,
                                                        const double* H1, double* sdist, double* Hc0, double* Hc1,
                                                        int* zidx) {
  const int64_t i = blockIdx.x * (int64_t)DT_THREADS + threadIdx.x;
  if (i >= N) return;
  double c[ARB_CONS_NDBL];
  for (int k = 0; k < ARB_CONS_NDBL; ++k) c[k] = EL(cd, k);
  Se3 g0, g1, c0, c1;
  for (int k = 0; k < 9; ++k) { g0.R[k] = EL(H0, k); g1.R[k] = EL(H1, k); }
  for (int k = 0; k < 3; ++k) { g0.p[k] = EL(H0, 9 + k); g1.p[k] = EL(H1, 9 + k); }
  int zi[3];
  EL(sdist, 0) = contact_collide(EL(pair, 0), c, g0, g1, c0, c1, zi);
  for (int k = 0; k < 9; ++k) { EL(Hc0, k) = c0.R[k]; EL(Hc1, k) = c1.R[k]; }
  for (int k = 0; k < 3; ++k) { EL(Hc0, 9 + k) = c0.p[k]; EL(Hc1, 9 + k) = c1.p[k]; EL(zidx, k) = zi[k]; }
}

extern "C" {
int dt_softfinger_solve(int N, const double* v, const double* A, const double* P, const double* sdist, const double* mu,
                        const double* eps, double dt, double* f, double* df, int* br, int* st) {
  k_softfinger_solve<<<dt_blocks(N), DT_THREADS>>>(N, v, A, P, sdist, mu, eps, dt, f, df, br, st);
  return dt_err();
}
int dt_softfinger_fused(int N, int mode, const double* v, const double* A, const double* P, const double* aux,
                        const double* mu, const double* eps, double dt, double* f, double* df, int* br, int* st) {
  k_softfinger_fused<<<dt_blocks(N), DT_THREADS>>>(N, mode, v, A, P, aux, mu, eps, dt, f, df, br, st);
  return dt_err();
}
int dt_sliding_root(int N, int coop, const double* A, const double* alpha, const double* mu, double* s, int* found,
                    int* ok) {
  k_sliding_root<<<dt_blocks(N), DT_THREADS>>>(N, coop, A, alpha, mu, s, found, ok);
  return dt_err();
}
int dt_poly6(int N, const double* p, const double* x, int* fast_ok, double* fast_root, int* positive, int* slow_n,
             double* slow_root, int* certify) {
  k_poly6<<<dt_blocks(N), DT_THREADS>>>(N, p, x, fast_ok, fast_root, positive, slow_n, slow_root, certify);
  return dt_err();
}
int dt_eig6(int N, const double* A, double* wr, double* wi, int* ok) {
  k_eig6<<<dt_blocks(N), DT_THREADS>>>(N, A, wr, wi, ok);
  return dt_err();
}
int dt_pinv(int N, int n, const double* A, double* out) {
  if (n == 1) k_pinv<1><<<dt_blocks(N), DT_THREADS>>>(N, A, out);
  else if (n == 3) k_pinv<3><<<dt_blocks(N), DT_THREADS>>>(N, A, out);
  else if (n == 4) k_pinv<4><<<dt_blocks(N), DT_THREADS>>>(N, A, out);
  else return -1;
  return dt_err();
}
int dt_inv_cond4(int N, const double* A, double* out, double* cond) {
  k_inv_cond4<<<dt_blocks(N), DT_THREADS>>>(N, A, out, cond);
  return dt_err();
}
int dt_solve4(int N, const double* A, const double* b, double* x, int* ok) {
  k_solve4<<<dt_blocks(N), DT_THREADS>>>(N, A, b, x, ok);
  return dt_err();
}
int dt_se3_exp(int N, const double* tw, double* out) {
  k_se3_exp<<<dt_blocks(N), DT_THREADS>>>(N, tw, out);
  return dt_err();
}
int dt_zaligned(int N, const double* z, double* R, int* idx) {
  k_zaligned<<<dt_blocks(N), DT_THREADS>>>(N, z, R, idx);
  return dt_err();
}
int dt_collide(int N, const int* pair, const double* cd, const double* H0, const double* H1, double* sdist, double* Hc0,
               double* Hc1, int* zidx) {
  k_collide<<<dt_blocks(N), DT_THREADS>>>(N, pair, cd, H0, H1, sdist, Hc0, Hc1, zidx);
  return dt_err();
}
}

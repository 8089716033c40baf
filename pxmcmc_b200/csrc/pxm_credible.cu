// Streaming credible intervals (pxmcmc/uncertainty.py:7-16 computes them from the stored chain): numpy's linear
// quantiles at alpha/2 and 1 - alpha/2 of N pooled samples read two adjacent order statistics each, x(lo) and
// x(min(lo + 1, N - 1)).  Those of the lower quantile are among the K_lo = min(lo_a + 2, N) smallest samples, those of
// the upper one among the K_hi = N - lo_b largest, so two bounded heaps per (element, component) give numpy's answer
// bit for bit without storing the chain (DESIGN.md 7b).  The K smallest values of a multiset do not depend on the order
// in which they arrive: the result is the same whatever the chain order, the acceptance pattern or a checkpoint split.
//
// State (doubles, T = ncomp n columns, ncomp = 2 in mode 1, else 1; column t = component t / n, element t % n):
//   lower heap  K_lo slots per column: a max-heap of the K_lo smallest values offered so far;
//   upper heap  K_hi slots per column: a max-heap of the negated K_hi largest;
//   NaN flag    one row [T]: nonzero once a NaN was offered (both quantiles are then NaN, as in numpy; a comparison
//               would silently drop it).
// Heap slot s of column t lives at t K + s ([column][slot]: a sift-down walks one column's heap, whose top levels share
// cache lines; measured 8-24 % less push time per run than [slot][column], DESIGN.md 5).  -DPXM_CREDIBLE_SLOT_MAJOR
// builds the [slot][column] layout (s T + t) instead, for that comparison (scripts/credible_overhead.py).
#include <math.h>
#include <math_constants.h>

#include <algorithm>

#include "pxm_common.cuh"
#include "pxm_plan.h"

namespace {

typedef double2 cplx;

constexpr int CR_THREADS = 256;
constexpr int CR_BATCH = 8;  // chains whose samples are loaded before any of them is offered (loads in flight)

__device__ __forceinline__ size_t hslot(size_t t, long long s, size_t T, long long K) {
#ifdef PXM_CREDIBLE_SLOT_MAJOR
  (void)K;
  return (size_t)s * T + t;
#else
  (void)T;
  return t * (size_t)K + (size_t)s;
#endif
}

// offer `key` as the pos-th value (0-based) to the max-heap of the K smallest values of column t; `root` holds h[0]
__device__ __forceinline__ void heap_offer(double* __restrict__ h, size_t t, size_t T, long long K, long long pos,
                                           double key, double& root) {
  if (pos < K) {  // filling: insert and sift up
    long long s = pos;
    while (s > 0) {
      const long long p = (s - 1) >> 1;
      const double pv = h[hslot(t, p, T, K)];
      if (!(pv < key)) break;
      h[hslot(t, s, T, K)] = pv;
      s = p;
    }
    h[hslot(t, s, T, K)] = key;
    if (s == 0) root = key;
    return;
  }
  if (!(key < root)) return;  // full: only a value below the K-th smallest enters, replacing the root
  long long s = 0;
  for (;;) {
    long long c = 2 * s + 1;
    if (c >= K) break;
    double cv = h[hslot(t, c, T, K)];
    if (c + 1 < K) {
      const double rv = h[hslot(t, c + 1, T, K)];
      if (rv > cv) {
        cv = rv;
        ++c;
      }
    }
    if (!(cv > key)) break;
    h[hslot(t, s, T, K)] = cv;
    if (s == 0) root = cv;
    s = c;
  }
  h[hslot(t, s, T, K)] = key;
  if (s == 0) root = key;
}

// one thread per column; the chains (and in mode 2 both packed parts, real first) in order.  Value number k offered
// by this push takes position count + k: count is the pooled number of samples before the push.
__global__ void __launch_bounds__(CR_THREADS) k_credible_push(double* __restrict__ st, const cplx* __restrict__ x,
                                                              size_t n, size_t T, int mode, int nchains, long long klo,
                                                              long long khi, long long count,
                                                              const long long* __restrict__ d_j) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (t >= T) return;
  const size_t e = t % n;
  const bool imag_part = mode == 1 && t >= n;
  double* lo = st;
  double* hi = st + (size_t)klo * T;
  double rlo = lo[hslot(t, 0, T, klo)], rhi = hi[hslot(t, 0, T, khi)];
  bool nan = false;
  long long pos = count;
  for (int c0 = 0; c0 < nchains; c0 += CR_BATCH) {
    cplx v[CR_BATCH];
    bool act[CR_BATCH];
#pragma unroll
    for (int k = 0; k < CR_BATCH; ++k) {
      const int c = c0 + k;
      act[k] = c < nchains && (d_j == nullptr || __ldg(d_j + c) >= 0);
      if (act[k]) v[k] = x[(size_t)c * n + e];
    }
#pragma unroll
    for (int k = 0; k < CR_BATCH; ++k) {
      if (!act[k]) continue;
      const int nv = mode == 2 ? 2 : 1;
      for (int q = 0; q < nv; ++q) {
        const double y = (q == 1 || imag_part) ? v[k].y : v[k].x;
        if (isnan(y)) {
          nan = true;
        } else {
          heap_offer(lo, t, T, klo, pos, y, rlo);
          heap_offer(hi, t, T, khi, pos, -y, rhi);
        }
        ++pos;
      }
    }
  }
  if (nan) st[(size_t)(klo + khi) * T + t] = 1.0;
}

// x(lo) and x(hi), hi = min(lo + 1, N - 1), of both quantiles from the roots and larger children, then numpy's _lerp
__global__ void k_credible_finalize(const double* __restrict__ st, size_t T, long long npooled, long long klo,
                                    long long khi, long long lo_a, double g_a, long long lo_b, double g_b,
                                    double* __restrict__ out_lo, double* __restrict__ out_hi) {
  const double* lo = st;
  const double* hi = st + (size_t)klo * T;
  const double* flag = st + (size_t)(klo + khi) * T;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < T; t += (size_t)gridDim.x * blockDim.x) {
    if (flag[t] != 0.0) {
      out_lo[t] = CUDART_NAN;
      out_hi[t] = CUDART_NAN;
      continue;
    }
    // lower heap: root = x(K_lo - 1) = x(hi_a); larger child = x(K_lo - 2), which is x(lo_a) unless lo_a = N - 1
    const long long hi_a = min(lo_a + 1, npooled - 1);
    const double ra = lo[hslot(t, 0, T, klo)];
    double xa = ra;
    if (lo_a != hi_a) {
      xa = lo[hslot(t, 1, T, klo)];
      if (klo > 2) xa = fmax(xa, lo[hslot(t, 2, T, klo)]);
    }
    out_lo[t] = pxm_lerp_np(xa, ra, g_a);
    // upper heap (negated): root = -x(lo_b); larger child = -x(lo_b + 1) unless lo_b = N - 1
    const long long hi_b = min(lo_b + 1, npooled - 1);
    const double rb = -hi[hslot(t, 0, T, khi)];
    double xb = rb;
    if (hi_b != lo_b) {
      double c = hi[hslot(t, 1, T, khi)];
      if (khi > 2) c = fmax(c, hi[hslot(t, 2, T, khi)]);
      xb = -c;
    }
    out_hi[t] = pxm_lerp_np(rb, xb, g_b);
  }
}

}  // namespace

int pxm_credible_tails(long long npooled, long long lo_a, long long lo_b, long long* klo, long long* khi) {
  if (npooled < 1 || lo_a < 0 || lo_a >= npooled || lo_b < 0 || lo_b >= npooled) return PXM_ERR_ARG;
  *klo = std::min(lo_a + 2, npooled);
  *khi = npooled - lo_b;
  return PXM_OK;
}

int pxm_launch_credible_push(double* st, const void* x, size_t n, size_t nchains, int mode, long long klo,
                             long long khi, long long count, const long long* d_j, cudaStream_t s) {
  const size_t T = (mode == 1 ? 2 : 1) * n;
  const unsigned grid = (unsigned)((T + CR_THREADS - 1) / CR_THREADS);
  k_credible_push<<<grid, CR_THREADS, 0, s>>>(st, (const cplx*)x, n, T, mode, (int)nchains, klo, khi, count, d_j);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_credible_finalize(const double* st, size_t n, int mode, long long npooled, long long klo, long long khi,
                                 long long lo_a, double g_a, long long lo_b, double g_b, double* out_lo,
                                 double* out_hi, cudaStream_t s) {
  const size_t T = (mode == 1 ? 2 : 1) * n;
  const unsigned grid = (unsigned)std::min<size_t>((T + 255) / 256, 148 * 32);
  k_credible_finalize<<<grid, 256, 0, s>>>(st, T, npooled, klo, khi, lo_a, g_a, lo_b, g_b, out_lo, out_hi);
  PXM_LAUNCHED();
  return PXM_OK;
}

// Streaming posterior summaries (no counterpart in the reference): per-element running moments of the chains on the
// tracking grid, from which the pooled mean / variance, split-R-hat and a batch-means effective sample size follow
// without storing a single sample (DESIGN.md 7b).
//
// A "slot" is one scalar component of one logical chain: mode 0 (real part) slot = c; mode 1 (re + im) slot = 2c + part;
// mode 2 (packed real chain pairs) slot = 2c + part = the logical (unpacked) chain.  The accumulator holds 8 fields,
// each [nslots][n] doubles (structure of arrays: every field is one contiguous, coalesced stream):
//   0 mean of half A   1 M2 of half A   2 middle sample (odd n)   3 mean of half B   4 M2 of half B
//   5 open batch sum   6 mean of the batch means   7 M2 of the batch means
// With h = n/2, b = max(1, floor(sqrt n)), a = n/b: sample j goes into half A (j < h), half B (j >= n - h) or is the
// middle sample (j == h, odd n); into batch j/b when j < a b.  The first write of every accumulator overwrites it, so
// nothing left in the buffer (not even NaN) reaches a statistic.
#include <math.h>
#include <math_constants.h>

#include <algorithm>

#include "pxm_common.cuh"
#include "pxm_plan.h"

namespace {

typedef double2 cplx;

constexpr int NREC = 10;
constexpr int ACC_THREADS = 256;

struct ChainStep {
  int active;    // this chain takes a sample
  int half;      // 0 half A, 1 middle sample, 2 half B
  int hfirst;    // first sample of its half
  int inbatch;   // sample lies in a batch
  int bfirst;    // first sample of its batch
  int fold;      // last sample of its batch: fold the batch mean
  int bmfirst;   // first batch of the chain
  double rh;     // 1 / (samples in the half so far, this one included)
  double rb;     // 1 / b
  double rbm;    // 1 / (batches folded so far, this one included)
};

__device__ __forceinline__ void welford(double* __restrict__ mean, double* __restrict__ m2, size_t k, double x, int first,
                                        double r) {
  if (first) {
    mean[k] = x;
    m2[k] = 0.0;
    return;
  }
  const double mu = mean[k];
  const double d = x - mu;
  const double mu1 = mu + d * r;
  mean[k] = mu1;
  m2[k] = m2[k] + d * (x - mu1);
}

__device__ __forceinline__ void push_one(double* __restrict__ acc, size_t S, size_t k, double x, const ChainStep& cs) {
  if (cs.half == 0)
    welford(acc, acc + S, k, x, cs.hfirst, cs.rh);
  else if (cs.half == 2)
    welford(acc + 3 * S, acc + 4 * S, k, x, cs.hfirst, cs.rh);
  else
    acc[2 * S + k] = x;
  if (!cs.inbatch) return;
  double* bsum = acc + 5 * S;
  const double s = cs.bfirst ? x : bsum[k] + x;
  if (cs.fold) welford(acc + 6 * S, acc + 7 * S, k, s * cs.rb, cs.bmfirst, cs.rbm);
  else bsum[k] = s;
}

// grid (ceil(n / 256), nchains): one block row per chain, so that the per-chain Welford coefficients are computed once
// (no division per element)
__global__ void __launch_bounds__(ACC_THREADS) k_stats_accumulate(double* __restrict__ acc, const cplx* __restrict__ x,
                                                                  size_t n, size_t S, int mode, long long nsamples,
                                                                  long long j_host, const long long* __restrict__ d_j) {
  __shared__ ChainStep cs;
  const size_t c = blockIdx.y;
  if (threadIdx.x == 0) {
    const long long j = d_j ? d_j[c] : j_host;
    ChainStep t{};
    t.active = j >= 0 && j < nsamples;
    if (t.active) {
      const long long h = nsamples / 2;
      long long b = (long long)floor(sqrt((double)nsamples));
      while (b * b > nsamples) --b;
      while ((b + 1) * (b + 1) <= nsamples) ++b;
      b = b < 1 ? 1 : b;
      const long long a = nsamples / b;
      long long kh = 0;
      if (j < h) {
        t.half = 0;
        kh = j;
      } else if (j >= nsamples - h) {
        t.half = 2;
        kh = j - (nsamples - h);
      } else {
        t.half = 1;
      }
      t.hfirst = kh == 0;
      t.rh = 1.0 / (double)(kh + 1);
      t.inbatch = j < a * b;
      t.bfirst = j % b == 0;
      t.fold = t.inbatch && (j + 1) % b == 0;
      t.bmfirst = j / b == 0;
      t.rb = 1.0 / (double)b;
      t.rbm = 1.0 / (double)(j / b + 1);
    }
    cs = t;
  }
  __syncthreads();
  if (!cs.active) return;
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= n) return;
  const cplx v = x[c * n + e];
  if (mode == 0) {
    push_one(acc, S, c * n + e, v.x, cs);
  } else {  // modes 1 and 2: the two parts are slots 2c and 2c + 1
    push_one(acc, S, (2 * c) * n + e, v.x, cs);
    push_one(acc, S, (2 * c + 1) * n + e, v.y, cs);
  }
}

// Chan's combination of (na, ma, M2a) with (nb, mb, M2b) into the first
__device__ __forceinline__ void chan(double& na, double& ma, double& m2a, double nb, double mb, double m2b) {
  if (nb == 0.0) return;
  if (na == 0.0) {
    na = nb;
    ma = mb;
    m2a = m2b;
    return;
  }
  const double nn = na + nb;
  const double d = mb - ma;
  ma = ma + d * (nb / nn);
  m2a = m2a + m2b + d * d * (na * nb / nn);
  na = nn;
}

// one thread per (component, element); chains in order: deterministic
__global__ void k_stats_partials(const double* __restrict__ acc, size_t n, size_t S, int ncomp, int mlog,
                                 long long nsamples, double* __restrict__ rec, double* __restrict__ cmean,
                                 double* __restrict__ cvar) {
  const size_t total = (size_t)ncomp * n;
  const long long h = nsamples / 2;
  long long b = (long long)floor(sqrt((double)nsamples));
  while (b * b > nsamples) --b;
  while ((b + 1) * (b + 1) <= nsamples) ++b;
  b = b < 1 ? 1 : b;
  const double a = (double)(nsamples / b);
  const double hd = (double)h;
  const bool odd = nsamples & 1;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t comp = t / n, e = t % n;
    double hk = 0.0, hm = 0.0, hm2 = 0.0, ssum = 0.0;  // half-chain means (Welford), sum of half variances
    double pn = 0.0, pm = 0.0, pm2 = 0.0;               // pooled samples
    double bn = 0.0, bm = 0.0, bm2 = 0.0;               // batch means
    for (int q = 0; q < mlog; ++q) {
      const size_t k = ((size_t)q * ncomp + comp) * n + e;
      double cn = 0.0, cm = 0.0, cm2 = 0.0;
      if (h > 0) {
        const double mA = acc[k], m2A = acc[S + k], mB = acc[3 * S + k], m2B = acc[4 * S + k];
        cn = hd;
        cm = mA;
        cm2 = m2A;
        chan(cn, cm, cm2, hd, mB, m2B);
        hk += 1.0;
        double d = mA - hm;
        hm += d / hk;
        hm2 += d * (mA - hm);
        hk += 1.0;
        d = mB - hm;
        hm += d / hk;
        hm2 += d * (mB - hm);
        if (h >= 2) ssum += m2A / (hd - 1.0) + m2B / (hd - 1.0);
      }
      if (odd) chan(cn, cm, cm2, 1.0, acc[2 * S + k], 0.0);
      if (cmean) cmean[k] = cm;
      if (cvar) cvar[k] = nsamples > 1 ? cm2 / (cn - 1.0) : CUDART_NAN;
      chan(pn, pm, pm2, cn, cm, cm2);
      chan(bn, bm, bm2, a, acc[6 * S + k], acc[7 * S + k]);
    }
    const double r[NREC] = {hk, hm, hm2, ssum, pn, pm, pm2, bn, bm, bm2};
    for (int f = 0; f < NREC; ++f) rec[(size_t)f * total + t] = r[f];
  }
}

}  // namespace

long long pxm_stats_slots(int mode, long long nchains) { return mode == 0 ? nchains : 2 * nchains; }

int pxm_launch_stats_accumulate(double* acc, const void* x, size_t n, size_t nchains, int mode, long long nsamples,
                                long long j, const long long* d_j, cudaStream_t st) {
  const size_t S = (size_t)pxm_stats_slots(mode, (long long)nchains) * n;
  dim3 grid((unsigned)((n + ACC_THREADS - 1) / ACC_THREADS), (unsigned)nchains);
  k_stats_accumulate<<<grid, ACC_THREADS, 0, st>>>(acc, (const cplx*)x, n, S, mode, nsamples, j, d_j);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_stats_partials(const double* acc, size_t n, size_t nchains, int mode, long long nsamples, double* rec,
                              double* cmean, double* cvar, cudaStream_t st) {
  const size_t S = (size_t)pxm_stats_slots(mode, (long long)nchains) * n;
  const int ncomp = mode == 1 ? 2 : 1;
  const int mlog = (int)(mode == 2 ? 2 * nchains : nchains);
  const size_t total = (size_t)ncomp * n;
  const unsigned grid = (unsigned)std::min<size_t>((total + 255) / 256, 148 * 32);
  k_stats_partials<<<grid, 256, 0, st>>>(acc, n, S, ncomp, mlog, nsamples, rec, cmean, cvar);
  PXM_LAUNCHED();
  return PXM_OK;
}

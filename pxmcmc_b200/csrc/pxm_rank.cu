// Rank-normalised split-R-hat and bulk / tail ESS of stored multi-chain samples (Vehtari, Gelman, Simpson, Carpenter &
// Buerkner 2021, as ArviZ's rhat(method="rank") and ess(method="bulk" | "tail"); no counterpart in the reference).
// DESIGN.md 7b states the definition; oracle/rank_diagnostics_ref.py restates it in numpy.
//
// A column is one parameter: S = m n values x[c][i] stored at chain[(c n + i) ld + col].  Two kernels:
//  k_rank_transpose  copies a block of columns into column-contiguous scratch [ncols][S] (32 x 32 tiles: both the
//                    strided read of the stored layout and the write are coalesced);
//  k_rank_columns    one CTA per column.  The column is sorted in shared memory as (value, sample index) pairs with
//                    the bitonic network of k_quantile_columns; median, q05 and q95 are read off the sorted order; the
//                    average ranks over the split subset (the middle sample of odd n is flagged out) come from a
//                    CTA-wide prefix count over the flags and the tie-group boundaries; z = normcdfinv((r - 3/8) /
//                    (N + 1/4)) is written in split-series order.  R and the Geyer ESS then run on the series in shared
//                    memory (centered in place), the autocovariance as direct lag sums, RK_LAGS lags per CTA-wide
//                    reduction, stopping where Geyer's initial-positive sequence stops.  The folded series |x - med|
//                    repeats the sort; the indicators 1[x <= q] are formed from the column as it is reloaded.
// Every reduction runs in a fixed order: the outputs are deterministic.
#include <math.h>
#include <math_constants.h>
#include <stdint.h>

#include <climits>

#include "pxm_common.cuh"
#include "pxm_plan.h"

namespace {

constexpr int RK_THREADS = 512;
constexpr int RK_WARPS = RK_THREADS / 32;
constexpr int RK_LAGS = 8;       // autocovariance lags per CTA-wide reduction (pairs of Geyer's loop start at even lags)
constexpr int RK_ENC = 1 << 15;  // (position, prefix count) packed into one int: both are <= 16384

__global__ void k_rank_transpose(const double* __restrict__ x, long long S, long long ncols, long long ld,
                                 double* __restrict__ out) {
  __shared__ double tile[32][33];
  const long long c0 = (long long)blockIdx.x * 32, r0 = (long long)blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const long long r = r0 + k, c = c0 + threadIdx.x;
    if (r < S && c < ncols) tile[k][threadIdx.x] = x[r * ld + c];
  }
  __syncthreads();
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const long long c = c0 + k, r = r0 + threadIdx.x;
    if (r < S && c < ncols) out[c * S + r] = tile[threadIdx.x][k];
  }
}

// exclusive scan over the threads of the CTA (op commutative and associative, ident its identity); sh: RK_WARPS ints
template <class Op>
__device__ __forceinline__ int block_exscan(int v, int ident, int* sh, Op op) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int inc = v;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc = op(inc, y);
  }
  int ex = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) ex = ident;
  if (lane == 31) sh[w] = inc;
  __syncthreads();
  int carry = ident;
  for (int k = 0; k < w; ++k) carry = op(carry, sh[k]);
  __syncthreads();
  return op(carry, ex);
}

// sum of NV values over the CTA, the same on every thread: warps in order; red: RK_WARPS * NV doubles
template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int g = 0; g < NV; ++g) {
    for (int o = 16; o > 0; o >>= 1) v[g] += __shfl_down_sync(0xffffffffu, v[g], o);
    if (lane == 0) red[w * NV + g] = v[g];
  }
  __syncthreads();
#pragma unroll
  for (int g = 0; g < NV; ++g) {
    double s = 0.0;
    for (int k = 0; k < RK_WARPS; ++k) s += red[k * NV + g];
    v[g] = s;
  }
  __syncthreads();
}

__device__ __forceinline__ void block_minmax(double& lo, double& hi, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    lo = fmin(lo, __shfl_down_sync(0xffffffffu, lo, o));
    hi = fmax(hi, __shfl_down_sync(0xffffffffu, hi, o));
  }
  if (lane == 0) {
    red[2 * w] = lo;
    red[2 * w + 1] = hi;
  }
  __syncthreads();
  lo = red[0];
  hi = red[1];
  for (int k = 1; k < RK_WARPS; ++k) {
    lo = fmin(lo, red[2 * k]);
    hi = fmax(hi, red[2 * k + 1]);
  }
  __syncthreads();
}

// bitonic sort of npad (key, index) pairs in shared memory, ascending (the network of k_quantile_columns)
__device__ void sort_pairs(double* keys, uint16_t* idx, int npad) {
  const int half = npad >> 1;
  for (int size = 2; size <= npad; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < half; i += blockDim.x) {
        const int pos = 2 * i - (i & (stride - 1));
        const double a = keys[pos], b = keys[pos + stride];
        const bool up = (pos & size) == 0;
        if ((a > b) == up) {
          keys[pos] = b;
          keys[pos + stride] = a;
          const uint16_t t = idx[pos];
          idx[pos] = idx[pos + stride];
          idx[pos + stride] = t;
        }
      }
      __syncthreads();
    }
}

struct Split {
  int n, h, m;
  // series index of sample r = c n + i in split order (first halves of chains 0..m-1, then second halves), -1: the
  // middle sample of an odd n, in no series
  __device__ __forceinline__ int series_pos(int r) const {
    const int c = r / n, i = r - c * n;
    if (i < h) return c * h + i;
    if (i >= n - h) return (m + c) * h + (i - (n - h));
    return -1;
  }
};

// keys[0, npad) sorted ascending (values at positions >= S are +inf padding), idx the sample index of each position.
// Writes z = Phi^-1((r - 3/8) / (N + 1/4)) of every split sample, r its average rank among the N split samples, into
// keys[0, N) in split-series order.  rk: npad uint16 of scratch; chunk: RK_THREADS ints; isc: RK_WARPS ints.
__device__ void ranks_to_z(double* keys, const uint16_t* idx, uint16_t* rk, int npad, int S, int N, const Split& sp,
                           int* chunk, int* isc) {
  const int T = RK_THREADS, tid = threadIdx.x;
  const int K = npad >= T ? npad / T : 1;
  const int p0 = min(tid * K, npad), p1 = min(p0 + K, npad);
  // a tie group starts at a head: position 0, a change of value, or position S (first padding)
  auto head = [&](int p) { return p <= S && (p == 0 || keys[p] != keys[p - 1]); };
  auto flag = [&](int p) { return p < S && sp.series_pos(idx[p]) >= 0; };
  int cnt = 0, first_h = -1, first_c = 0, last_h = -1, last_c = 0;
  for (int p = p0; p < p1; ++p) {
    if (head(p)) {
      if (first_h < 0) {
        first_h = p;
        first_c = cnt;
      }
      last_h = p;
      last_c = cnt;
    }
    cnt += flag(p);
  }
  // P[p] = flagged positions before p; a group [a, b) of g flagged ranks P[a] + 1 .. P[b] has average (P[a] + P[b] + 1) / 2
  const int base = block_exscan(cnt, 0, isc, [](int a, int b) { return a + b; });
  const int last_enc = last_h >= 0 ? last_h * RK_ENC + base + last_c : -1;
  const int a_enc = block_exscan(last_enc, -1, isc, [](int a, int b) { return max(a, b); });  // last head before p0
  chunk[tid] = first_h >= 0 ? first_h * RK_ENC + base + first_c : INT_MAX;
  __syncthreads();
  // suffix minimum over the chunks after this one: scan the reversed chunk order
  const int rev = block_exscan(chunk[T - 1 - tid], INT_MAX, isc, [](int a, int b) { return min(a, b); });
  __syncthreads();
  chunk[T - 1 - tid] = rev;
  __syncthreads();
  int b_enc = chunk[tid] == INT_MAX ? S * RK_ENC + N : chunk[tid];  // first head after p1 (position S when S == npad)
  int c = cnt;
  for (int p = p1 - 1; p >= p0; --p) {
    const int f = flag(p);
    c -= f;
    if (f) rk[idx[p]] = (uint16_t)(b_enc % RK_ENC);
    if (head(p)) b_enc = p * RK_ENC + base + c;
  }
  int a = a_enc;
  for (int p = p0; p < p1; ++p) {
    if (head(p)) a = p * RK_ENC + base + c;
    const int f = flag(p);
    if (f) rk[idx[p]] = (uint16_t)(rk[idx[p]] + a % RK_ENC + 1);
    c += f;
  }
  __syncthreads();
  const double den = (double)N + 0.25;
  for (int r = tid; r < S; r += T) {
    const int s = sp.series_pos(r);
    if (s >= 0) keys[s] = normcdfinv(((double)rk[r] * 0.5 - 0.375) / den);
  }
  __syncthreads();
}

// R and (want_ess) the Geyer ESS of the M series of length h in buf[0, M h).  buf is centered in place; aux holds
// max(M, h) doubles of scratch.
__device__ void series_stats(double* buf, double* aux, int M, int h, bool want_ess, double* red, double* lagsum,
                             double& R, double& ess) {
  const int T = RK_THREADS, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int N = M * h;
  double lo = CUDART_INF, hi = -CUDART_INF;
  for (int s = tid; s < N; s += T) {
    lo = fmin(lo, buf[s]);
    hi = fmax(hi, buf[s]);
  }
  block_minmax(lo, hi, red);
  // per series (one warp each): mean, centering, sum of squares
  double ss[1] = {0.0};
  for (int k = w; k < M; k += RK_WARPS) {
    double* y = buf + (size_t)k * h;
    double sum = 0.0;
    for (int j = lane; j < h; j += 32) sum += y[j];
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const double mean = sum / h;
    double q = 0.0;
    for (int j = lane; j < h; j += 32) {
      const double d = y[j] - mean;
      y[j] = d;
      q += d * d;
    }
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    if (lane == 0) {
      aux[k] = mean;
      ss[0] += q;
    }
  }
  __syncthreads();
  double mm[1] = {0.0};
  for (int k = tid; k < M; k += T) mm[0] += aux[k];
  block_sum(mm, red);
  const double mbar = mm[0] / M;
  double dv[2] = {ss[0], 0.0};
  for (int k = tid; k < M; k += T) dv[1] += (aux[k] - mbar) * (aux[k] - mbar);
  block_sum(dv, red);  // also orders the reads of aux before it is reused below
  const double ssum = dv[0], varm = dv[1] / (M - 1);
  const double W = ssum / (h - 1.0) / M;
  R = sqrt((h * varm / W + h - 1.0) / h);
  if (!want_ess) return;
  const double Nd = (double)N;
  if (hi - lo < 1e-15) {  // np.finfo(float).resolution
    ess = Nd;
    return;
  }
  const double mean_var = ssum / Nd * h / (h - 1.0);
  const double var_plus = mean_var * (h - 1.0) / h + varm;
  double* rho = aux;  // rho_hat[0, T + 2)
  double ev = 1.0, od = 0.0;
  int t = 1;
  bool go = true;
  for (int L0 = 0; go; L0 += RK_LAGS) {
    double A[RK_LAGS];
#pragma unroll
    for (int g = 0; g < RK_LAGS; ++g) A[g] = 0.0;
    for (int s = tid; s < N; s += T) {
      const int j = s % h;
      const double v = buf[s];
#pragma unroll
      for (int g = 0; g < RK_LAGS; ++g)
        if (j + L0 + g < h) A[g] += v * buf[s + L0 + g];
    }
    block_sum(A, red);
    if (tid == 0)
      for (int g = 0; g < RK_LAGS; ++g) lagsum[g] = A[g];
    __syncthreads();
    auto rho_at = [&](int lag) { return 1.0 - (mean_var - lagsum[lag - L0] / Nd) / var_plus; };
    if (L0 == 0) {
      od = rho_at(1);
      if (tid == 0) {
        rho[0] = 1.0;
        rho[1] = od;
      }
    }
    // Geyer's initial positive sequence: pairs (t + 1, t + 2), t odd
    while (t + 2 < L0 + RK_LAGS) {
      if (!(t < h - 3 && ev + od > 0.0)) {
        go = false;
        break;
      }
      ev = rho_at(t + 1);
      od = rho_at(t + 2);
      const bool keep = ev + od >= 0.0;
      if (tid == 0) {
        rho[t + 1] = keep ? ev : 0.0;
        rho[t + 2] = keep ? od : 0.0;
      }
      t += 2;
    }
    if (go && !(t < h - 3 && ev + od > 0.0)) go = false;
  }
  if (tid == 0) {
    const int Tm = t - 2;
    if (ev > 0.0) rho[Tm + 1] = ev;
    // Geyer's initial monotone sequence
    for (int u = 1; u <= Tm - 2; u += 2)
      if (rho[u + 1] + rho[u + 2] > rho[u - 1] + rho[u]) {
        rho[u + 1] = (rho[u - 1] + rho[u]) / 2.0;
        rho[u + 2] = rho[u + 1];
      }
    double sum = 0.0;
    for (int u = 0; u <= Tm; ++u) sum += rho[u];
    const double tau = fmax(-1.0 + 2.0 * sum + rho[Tm + 1], 1.0 / log10(Nd));
    red[0] = Nd / tau;
  }
  __syncthreads();
  ess = red[0];
  __syncthreads();
}

__global__ void __launch_bounds__(RK_THREADS) k_rank_columns(const double* __restrict__ xs, int m, int n, int npad,
                                                             long long lo05, double g05, long long lo95, double g95,
                                                             double* __restrict__ out_rhat,
                                                             double* __restrict__ out_bulk,
                                                             double* __restrict__ out_tail) {
  extern __shared__ double keys[];  // npad doubles, then 2 npad uint16 (idx, rk) = npad / 2 doubles (aux)
  uint16_t* idx = reinterpret_cast<uint16_t*>(keys + npad);
  uint16_t* rk = idx + npad;
  double* aux = keys + npad;
  __shared__ double red[RK_WARPS * RK_LAGS];
  __shared__ double lagsum[RK_LAGS];
  __shared__ int chunk[RK_THREADS];
  __shared__ int isc[RK_WARPS];
  __shared__ double qv[3];  // median, q05, q95
  const long long col = blockIdx.x;
  const int S = m * n, h = n / 2, M = 2 * m, N = M * h, tid = threadIdx.x;
  const Split sp{n, h, m};
  const double* x = xs + col * (long long)S;

  int bad = n < 4;
  for (int p = tid; p < npad; p += RK_THREADS) {
    double v = CUDART_INF;  // padding sorts to the end
    if (p < S) {
      v = x[p];
      bad |= !isfinite(v);
    }
    keys[p] = v;
    idx[p] = (uint16_t)p;
  }
  if (__syncthreads_or(bad)) {
    if (tid == 0) out_rhat[col] = out_bulk[col] = out_tail[col] = CUDART_NAN;
    return;
  }
  sort_pairs(keys, idx, npad);
  if (tid == 0) {
    qv[0] = (S & 1) ? keys[S / 2] : (keys[S / 2 - 1] + keys[S / 2]) / 2.0;  // numpy's median
    qv[1] = pxm_lerp_np(keys[lo05], keys[min(lo05 + 1, (long long)S - 1)], g05);
    qv[2] = pxm_lerp_np(keys[lo95], keys[min(lo95 + 1, (long long)S - 1)], g95);
  }
  __syncthreads();
  const double med = qv[0], q05 = qv[1], q95 = qv[2];

  double Rb, Rf, eb, e05, e95, unused;
  ranks_to_z(keys, idx, rk, npad, S, N, sp, chunk, isc);
  series_stats(keys, aux, M, h, true, red, lagsum, Rb, eb);

  for (int p = tid; p < npad; p += RK_THREADS) {
    keys[p] = p < S ? fabs(x[p] - med) : CUDART_INF;
    idx[p] = (uint16_t)p;
  }
  __syncthreads();
  sort_pairs(keys, idx, npad);
  ranks_to_z(keys, idx, rk, npad, S, N, sp, chunk, isc);
  series_stats(keys, aux, M, h, false, red, lagsum, Rf, unused);

  for (int pass = 0; pass < 2; ++pass) {
    const double q = pass ? q95 : q05;
    for (int r = tid; r < S; r += RK_THREADS) {
      const int s = sp.series_pos(r);
      if (s >= 0) keys[s] = x[r] <= q ? 1.0 : 0.0;
    }
    __syncthreads();
    series_stats(keys, aux, M, h, true, red, lagsum, unused, pass ? e95 : e05);
  }
  if (tid == 0) {
    out_rhat[col] = (isnan(Rb) || isnan(Rf)) ? CUDART_NAN : fmax(Rb, Rf);
    out_bulk[col] = eb;
    out_tail[col] = fmin(e05, e95);
  }
}

// numpy's default "linear" quantile: lower order statistic and weight of the virtual index (S - 1) q
void virtual_index(long long S, double q, long long* lo, double* gamma) {
  const double v = (double)(S - 1) * q;
  const double f = floor(v);
  if (v >= (double)(S - 1)) {
    *lo = S - 1;
    *gamma = 0.0;
    return;
  }
  *lo = (long long)f;
  *gamma = v - f;
}

}  // namespace

int pxm_launch_rank_diagnostics(const double* chain, long long m, long long n, long long ncols, long long ld,
                                double* scratch, double* rhat, double* ess_bulk, double* ess_tail, cudaStream_t st) {
  if (ncols == 0) return PXM_OK;
  const long long S = m * n;
  int npad = 2;
  while (npad < S) npad <<= 1;
  const size_t smem = (size_t)npad * 12;
  static bool configured = false;
  if (!configured) {
    PXM_CUDA(cudaFuncSetAttribute(k_rank_columns, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured = true;
  }
  dim3 tgrid((unsigned)((ncols + 31) / 32), (unsigned)((S + 31) / 32));
  k_rank_transpose<<<tgrid, dim3(32, 8), 0, st>>>(chain, S, ncols, ld, scratch);
  PXM_LAUNCHED();
  long long lo05, lo95;
  double g05, g95;
  virtual_index(S, 0.05, &lo05, &g05);
  virtual_index(S, 0.95, &lo95, &g95);
  k_rank_columns<<<(unsigned)ncols, RK_THREADS, smem, st>>>(scratch, (int)m, (int)n, npad, lo05, g05, lo95, g95, rhat,
                                                            ess_bulk, ess_tail);
  PXM_LAUNCHED();
  return PXM_OK;
}

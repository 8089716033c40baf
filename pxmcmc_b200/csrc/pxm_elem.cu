// Fused elementwise / reduction / gather kernels of the proximal-Langevin step
// (HBM-bound, coalesced, grid-stride).  Each replaces a chain of numpy passes in
// the reference; file:line of what it follows is given per kernel.
//
// All per-chain arrays are [nchains][n] row-major; thresholds, data, inverse
// covariance and weights are shared by all chains and indexed by i.
#include <math_constants.h>

#include <algorithm>

#include "pxm_common.cuh"

namespace {

typedef double2 cplx;

// ---------------------------------------------------------------------------
// soft threshold, exactly the reference's operation order
// (/root/reference/pxmcmc/utils.py:55-67, _sign :84-88):
//   sign(x) * (|x| - T), 0 where |x| <= T (inclusive), sign(z) = z/|z| (0 at 0)
// ---------------------------------------------------------------------------
// |z| exactly as numpy's vectorised complex abs computes it
// (numpy/_core/src/umath/loops_unary_complex.dispatch.c.src, simd_cabs_f64):
//   larger * sqrt(fma(r, r, 1)),  r = smaller/larger
__device__ __forceinline__ double np_cabs(double re, double im) {
  re = fabs(re);
  im = fabs(im);
  const double larger = fmax(re, im), smaller = fmin(im, re);
  // (selects instead of early returns: the same values, no divergent regions around the division and the root)
  const double ratio = smaller / larger;
  const double h = sqrt(fma(ratio, ratio, 1.0)) * larger;
  return (larger == 0.0 || isinf(larger)) ? larger : h;
}

__device__ __forceinline__ cplx soft_c(cplx z, double T) {
  const double a = np_cabs(z.x, z.y);
  const double r = a - T;
  // numpy evaluates z/|z| through its complex division loop, i.e. as a product
  // with the reciprocal 1/|z| (loops.c.src, *_divide); replicate it bit for bit
  const double scl = 1.0 / a;
  const bool zero = a <= T;
  return make_double2(zero ? 0.0 : (z.x * scl) * r, zero ? 0.0 : (z.y * scl) * r);
}
// two REAL chains packed as the real and imaginary part of one complex chain (MYULA real_pairs): the threshold acts on
// each part, sign(x) (|x| - T) evaluated exactly
__device__ __forceinline__ double soft_part(double x, double T) {
  const double a = fabs(x);
  return a <= T ? 0.0 : copysign(a - T, x);
}
__device__ __forceinline__ cplx soft_parts(cplx z, double T) { return make_double2(soft_part(z.x, T), soft_part(z.y, T)); }
__device__ __forceinline__ double soft_r(double x, double T) {
  const double a = fabs(x);
  if (a <= T) return 0.0;
  return (x / a) * (a - T);
}

__global__ void k_soft_c(const cplx* __restrict__ x, const double* __restrict__ Tv, double Ts, cplx* __restrict__ out,
                         size_t n, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const double T = Tv ? Tv[i % n] : Ts;
    out[i] = soft_c(x[i], T);
  }
}
__global__ void k_soft_r(const double* __restrict__ x, const double* __restrict__ Tv, double Ts,
                         double* __restrict__ out, size_t n, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const double T = Tv ? Tv[i % n] : Ts;
    out[i] = soft_r(x[i], T);
  }
}

// ---------------------------------------------------------------------------
// Philox4x32-10 counter-based generator + Box-Muller (throughput mode noise)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
// two independent N(0,1) for (seed, stream, step, pair index)
__device__ __forceinline__ void philox_normal2(unsigned long long seed, unsigned int stream, unsigned long long step,
                                               unsigned long long pair, double* z0, double* z1) {
  uint32_t c[4] = {(uint32_t)pair, (uint32_t)(pair >> 32), (uint32_t)step, (uint32_t)(step >> 32) ^ (stream * 0x85EBCA6Bu)};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32) ^ stream);
  const unsigned long long a = ((unsigned long long)c[0] << 32) | c[1];
  const unsigned long long b = ((unsigned long long)c[2] << 32) | c[3];
  const double u1 = ((double)(a >> 11) + 0.5) * (1.0 / 9007199254740992.0);  // (0,1)
  const double u2 = ((double)(b >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  const double r = sqrt(-2.0 * log(u1));
  double sn, cs;
  sincospi(2.0 * u2, &sn, &cs);
  *z0 = r * cs;
  *z1 = r * sn;
}

// ---------------------------------------------------------------------------
// MYULA / PxMALA proposal (/root/reference/pxmcmc/mcmc.py:185-201), fused with
// the synthesis-setting prox (prior.py:49-50):
//   X' = (1 - d/l) X + (d/l) P - d g + sqrt(2 d) w
// P = soft(X, T) computed here (prox == nullptr) or given (analysis setting).
// Noise: w_re (and w_im if the sampler is `complex`) injected from the host RNG
// for parity, or Philox-generated (noise_mode 2).  Optionally also writes P.
// ---------------------------------------------------------------------------
struct MyulaArgs {
  const cplx* X;
  const cplx* prox;   // may be null -> soft(X,T)
  const cplx* gradg;
  const double* Tv;   // may be null -> Ts
  double Ts;
  const double* w_re;  // noise_mode 1
  const double* w_im;  // may be null
  cplx* Xout;
  cplx* prox_out;  // may be null
  size_t n, total;
  double a, b, delta, sq2d;
  int noise_mode;  // 0 none, 1 injected, 2 philox (real), 3 philox (complex); real chain pairs (chain 2c in the real,
                   // 2c+1 in the imaginary part, threshold per part): 4 philox (streams stream0 + 2c, + 2c + 1), 5 injected
  unsigned long long seed, step;
  const unsigned long long* step_ptr;  // may be null; otherwise the step is read from the device (CUDA-graph replays)
  const double* dpar;  // may be null; otherwise chain c reads {delta, 1 - delta/lmda, delta/lmda, sqrt(2 delta)} from
                       // dpar[16 c ..] (PxMALA tunes the step of every chain on the device)
  unsigned int stream0;
};
constexpr int PXM_STATE_DOUBLES = 16;  // per-chain state block of the device-resident PxMALA loop (k_pxmala_accept)
__device__ __forceinline__ void myula_device_params(MyulaArgs& p) {
  if (p.step_ptr) p.step = *p.step_ptr;
  if (p.dpar && p.step == 0) p.step = (unsigned long long)p.dpar[14];  // CUDA-graph replays: the step lives in the state block
}
__device__ __forceinline__ void myula_chain_params(const MyulaArgs& p, size_t chain, double* a, double* b, double* delta,
                                                   double* sq2d) {
  if (p.dpar) {
    const double* d = p.dpar + chain * PXM_STATE_DOUBLES;
    *delta = d[0];
    *a = d[1];
    *b = d[2];
    *sq2d = d[3];
  } else {
    *a = p.a;
    *b = p.b;
    *delta = p.delta;
    *sq2d = p.sq2d;
  }
}

__global__ void k_counter_add(unsigned long long* ctr, unsigned long long inc) { *ctr += inc; }

__global__ void k_myula_update(MyulaArgs p) {
  myula_device_params(p);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < p.total; i += (size_t)gridDim.x * blockDim.x) {
    const cplx x = p.X[i];
    cplx px;
    if (p.prox) {
      px = p.prox[i];
    } else {
      const double T = p.Tv ? p.Tv[i % p.n] : p.Ts;
      px = p.noise_mode >= 4 ? soft_parts(x, T) : soft_c(x, T);
    }
    if (p.prox_out) p.prox_out[i] = px;
    const cplx g = p.gradg[i];
    double wr = 0.0, wi = 0.0;
    if (p.noise_mode == 1 || p.noise_mode == 5) {
      wr = p.w_re[i];
      if (p.w_im) wi = p.w_im[i];
    } else if (p.noise_mode == 4) {
      const size_t chain = i / p.n, e = i % p.n;
      double z0, z1;
      philox_normal2(p.seed, p.stream0 + 2u * (unsigned int)chain, p.step, e >> 1, &z0, &z1);
      wr = (e & 1) ? z1 : z0;
      philox_normal2(p.seed, p.stream0 + 2u * (unsigned int)chain + 1u, p.step, e >> 1, &z0, &z1);
      wi = (e & 1) ? z1 : z0;
    } else if (p.noise_mode >= 2) {
      const size_t chain = i / p.n, e = i % p.n;
      double z0, z1;
      if (p.noise_mode == 3) {
        philox_normal2(p.seed, p.stream0 + (unsigned int)chain, p.step, e, &z0, &z1);
        wr = z0;
        wi = z1;
      } else {
        philox_normal2(p.seed, p.stream0 + (unsigned int)chain, p.step, e >> 1, &z0, &z1);
        wr = (e & 1) ? z1 : z0;
      }
    }
    // same association order as the reference expression
    double ca, cb, cd, cs;
    myula_chain_params(p, i / p.n, &ca, &cb, &cd, &cs);
    cplx o;
    o.x = ((ca * x.x + cb * px.x) - cd * g.x) + cs * wr;
    o.y = ((ca * x.y + cb * px.y) - cd * g.y) + cs * wi;
    p.Xout[i] = o;
  }
}

// Philox real-noise variant: one Box-Muller pair serves two consecutive coefficients, so a
// thread updates elements (2p, 2p+1) of one chain (halves the transcendental work; the noise
// stream is identical to the per-element kernel: element e uses normal (e&1) of pair e>>1)
// grid = (blocks per chain, chains in this launch); `chain0` = first chain of the launch (more than 65 535 chains are
// launched in slices): no 64-bit division per pair (ncu: 552 instructions per pair, issue slots 75 % busy, with it)
__global__ void k_myula_update_pair(MyulaArgs p, size_t chain0) {
  const size_t npairs = (p.n + 1) >> 1;
  myula_device_params(p);
  const size_t chain = chain0 + blockIdx.y;
  double ca, cb, cd, cs;
  myula_chain_params(p, chain, &ca, &cb, &cd, &cs);
  for (size_t pr = blockIdx.x * (size_t)blockDim.x + threadIdx.x; pr < npairs; pr += (size_t)gridDim.x * blockDim.x) {
    const size_t e0 = 2 * pr, i0 = chain * p.n + e0;
    const bool two = e0 + 1 < p.n;
    // every input of the pair is requested before any arithmetic: one exposed DRAM latency per iteration, not three
    cplx x[2], g[2], px[2];
    double T[2];
    x[0] = p.X[i0];
    g[0] = p.gradg[i0];
    x[1] = two ? p.X[i0 + 1] : make_double2(0.0, 0.0);
    g[1] = two ? p.gradg[i0 + 1] : make_double2(0.0, 0.0);
    if (p.prox) {
      px[0] = p.prox[i0];
      px[1] = two ? p.prox[i0 + 1] : make_double2(0.0, 0.0);
    } else {
      T[0] = p.Tv ? p.Tv[e0] : p.Ts;
      T[1] = (p.Tv && two) ? p.Tv[e0 + 1] : p.Ts;
    }
    double z[2];
    philox_normal2(p.seed, p.stream0 + (unsigned int)chain, p.step, pr, &z[0], &z[1]);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      const size_t i = i0 + h;
      if (!p.prox) px[h] = soft_c(x[h], T[h]);
      if (p.prox_out) p.prox_out[i] = px[h];
      cplx o;
      o.x = ((ca * x[h].x + cb * px[h].x) - cd * g[h].x) + cs * z[h];
      o.y = ((ca * x[h].y + cb * px[h].y) - cd * g[h].y) + cs * 0.0;
      p.Xout[i] = o;
    }
  }
}

// Real chain pairs with Philox noise (noise_mode 4): packed chain c holds real chain 2c in its real and 2c+1 in its
// imaginary part; each part is thresholded on its own and draws the normals the unpacked chain would draw (element e of
// real chain r: normal (e & 1) of pair e >> 1 of stream stream0 + r), so packing does not change the noise.
__global__ void k_myula_update_realpair(MyulaArgs p, size_t chain0) {
  const size_t npairs = (p.n + 1) >> 1;
  myula_device_params(p);
  const size_t chain = chain0 + blockIdx.y;
  double ca, cb, cd, cs;
  myula_chain_params(p, chain, &ca, &cb, &cd, &cs);
  const unsigned int sa = p.stream0 + 2u * (unsigned int)chain;
  for (size_t pr = blockIdx.x * (size_t)blockDim.x + threadIdx.x; pr < npairs; pr += (size_t)gridDim.x * blockDim.x) {
    const size_t e0 = 2 * pr, i0 = chain * p.n + e0;
    const bool two = e0 + 1 < p.n;
    cplx x[2], g[2], px[2];
    double T[2];
    x[0] = p.X[i0];
    g[0] = p.gradg[i0];
    x[1] = two ? p.X[i0 + 1] : make_double2(0.0, 0.0);
    g[1] = two ? p.gradg[i0 + 1] : make_double2(0.0, 0.0);
    if (p.prox) {
      px[0] = p.prox[i0];
      px[1] = two ? p.prox[i0 + 1] : make_double2(0.0, 0.0);
    } else {
      T[0] = p.Tv ? p.Tv[e0] : p.Ts;
      T[1] = (p.Tv && two) ? p.Tv[e0 + 1] : p.Ts;
    }
    double za[2], zb[2];
    philox_normal2(p.seed, sa, p.step, pr, &za[0], &za[1]);
    philox_normal2(p.seed, sa + 1u, p.step, pr, &zb[0], &zb[1]);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      const size_t i = i0 + h;
      if (!p.prox) px[h] = soft_parts(x[h], T[h]);
      if (p.prox_out) p.prox_out[i] = px[h];
      cplx o;
      o.x = ((ca * x[h].x + cb * px[h].x) - cd * g[h].x) + cs * za[h];
      o.y = ((ca * x[h].y + cb * px[h].y) - cd * g[h].y) + cs * zb[h];
      p.Xout[i] = o;
    }
  }
}

// ---------------------------------------------------------------------------
// data-fidelity residual (/root/reference/pxmcmc/forward.py:66-69):
//   r = invcov (.) (preds - data), invcov diagonal, possibly complex (:80-82)
// ---------------------------------------------------------------------------
__global__ void k_resid(const cplx* __restrict__ preds, const cplx* __restrict__ data, const cplx* __restrict__ ic,
                        cplx* __restrict__ out, size_t n, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t e = i % n;
    const cplx p = preds[i], d = data[e], c = ic[e];
    const double dx = p.x - d.x, dy = p.y - d.y;
    out[i] = make_double2(c.x * dx - c.y * dy, c.x * dy + c.y * dx);
  }
}

// Residual in ring-Fourier space (see pxm_wav_ring_resid): out = ic[t] * (scale * pred - data) on k4-interleaved ring
// arrays [slot][ring/4][col][ring%4], col = 4 chain + 2 (m < 0) + (im); the data array holds chain 0 only.
__global__ void k_ring_resid(const double* __restrict__ pred, const double* __restrict__ data, const cplx* __restrict__ ic,
                             double* __restrict__ out, int rings, int nld, int ncols, double scale,
                             unsigned long long slot_stride, unsigned long long total) {
  // one thread per (slot, row-group, column pair, ring%4); ring%4 fastest, then the column pair
  const unsigned int halfc = (unsigned int)ncols >> 1;
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < total;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned int r4 = (unsigned int)(i & 3);
    unsigned long long q = i >> 2;
    const unsigned int c2 = (unsigned int)(q % halfc);
    q /= halfc;
    const unsigned int rgs = (unsigned int)((rings + 3) >> 2);
    const unsigned int rg = (unsigned int)(q % rgs);
    const unsigned long long slot = q / rgs;
    const unsigned int t = rg * 4 + r4;
    if ((int)t >= rings) continue;
    const unsigned long long base = slot * slot_stride + ((unsigned long long)rg * nld) * 4 + r4;
    const unsigned long long ire = base + (unsigned long long)(2 * c2) * 4, iim = ire + 4;
    const unsigned long long dre = base + (unsigned long long)(2 * (c2 & 1)) * 4, dim_ = dre + 4;  // chain 0, same sign
    const double vx = scale * pred[ire] - data[dre], vy = scale * pred[iim] - data[dim_];
    const cplx c = ic[t];
    out[ire] = c.x * vx - c.y * vy;
    out[iim] = c.x * vy + c.y * vx;
  }
}

// ---------------------------------------------------------------------------
// per-chain reductions (deterministic two-stage)
//  kind 0: sum |w_i x_i|                         (prior.py:28-35, :83-84)   -> (re, 0)
//  kind 1: sum conj(d_i) ic_i d_i, d = data-preds (mcmc.py:78-79)           -> complex
//  kind 2: sum (X2 - X1 - (delta/2) glp)^2, glp = -(X1-P)/lmda - g (mcmc.py:285-289) -> complex
// ---------------------------------------------------------------------------
struct ReduceArgs {
  int kind;
  const cplx* a;   // kind0: x ; kind1: preds ; kind2: X1
  const cplx* b;   // kind1: data ; kind2: X2
  const cplx* c;   // kind1: invcov ; kind2: P (prox of X1)
  const cplx* d;   // kind2: gradg(X1)
  const double* w; // kind0 weights (may be null)
  double delta, lmda;
  const double* dpar;  // may be null; otherwise delta = dpar[0] (device-resident PxMALA step)
  size_t n;
  cplx* partial;  // [nchains][gridDim.x]
  cplx* out;      // [nchains]
};

__device__ __forceinline__ cplx block_sum(cplx v) {
  __shared__ cplx sh[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v.x += __shfl_down_sync(0xffffffffu, v.x, o);
    v.y += __shfl_down_sync(0xffffffffu, v.y, o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  if (w == 0) {
    v = (lane < (int)(blockDim.x >> 5)) ? sh[lane] : make_double2(0.0, 0.0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      v.x += __shfl_down_sync(0xffffffffu, v.x, o);
      v.y += __shfl_down_sync(0xffffffffu, v.y, o);
    }
  }
  return v;
}

__global__ void k_reduce_stage1(ReduceArgs p) {
  const size_t chain = blockIdx.y;
  if (p.dpar) p.delta = p.dpar[chain * PXM_STATE_DOUBLES];
  const size_t off = chain * p.n;
  cplx acc = make_double2(0.0, 0.0);
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < p.n; e += (size_t)gridDim.x * blockDim.x) {
    if (p.kind == 0) {
      cplx x = p.a[off + e];
      if (p.w) {
        x.x *= p.w[e];
        x.y *= p.w[e];
      }
      acc.x += np_cabs(x.x, x.y);
    } else if (p.kind == 1) {
      const cplx pr = p.a[off + e], da = p.b[e], ic = p.c[e];
      const double dx = da.x - pr.x, dy = da.y - pr.y;
      const double tx = ic.x * dx - ic.y * dy, ty = ic.x * dy + ic.y * dx;  // ic*d
      acc.x += dx * tx + dy * ty;                                          // conj(d)*(ic*d)
      acc.y += dx * ty - dy * tx;
    } else {
      const cplx x1 = p.a[off + e], x2 = p.b[off + e], px = p.c[off + e], g = p.d[off + e];
      const double gx = -((x1.x - px.x) / p.lmda) - g.x, gy = -((x1.y - px.y) / p.lmda) - g.y;
      const double vx = x2.x - x1.x - (p.delta / 2) * gx, vy = x2.y - x1.y - (p.delta / 2) * gy;
      acc.x += vx * vx - vy * vy;
      acc.y += 2.0 * vx * vy;
    }
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) p.partial[chain * gridDim.x + blockIdx.x] = acc;
}

__global__ void k_reduce_stage2(const cplx* __restrict__ partial, int nparts, cplx* __restrict__ out) {
  const size_t chain = blockIdx.x;
  cplx acc = make_double2(0.0, 0.0);
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
    const cplx v = partial[chain * nparts + i];
    acc.x += v.x;
    acc.y += v.y;
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) out[chain] = acc;
}

// ---------------------------------------------------------------------------
// grad log pi (/root/reference/pxmcmc/mcmc.py:84-89), same operation order:
//   out = -((X - P)/lmda) - gradg,  P = soft(X,T) (prox == nullptr) or given
// ---------------------------------------------------------------------------
__global__ void k_gradlogpi(const cplx* __restrict__ X, const cplx* __restrict__ prox, const double* __restrict__ Tv,
                            double Ts, const cplx* __restrict__ gradg, double lmda, cplx* __restrict__ out, size_t n,
                            size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const cplx x = X[i];
    const cplx px = prox ? prox[i] : soft_c(x, Tv ? Tv[i % n] : Ts);
    const cplx g = gradg[i];
    out[i] = make_double2(-((x.x - px.x) / lmda) - g.x, -((x.y - px.y) / lmda) - g.y);
  }
}

// ---------------------------------------------------------------------------
// generic complex linear combination with real coefficients (analysis-setting prox
// assembly; SKROCK's stages run k_skrock_stage):  out = c0 + sum_k a_k x_k  (+ cz * z, z real)
// (/root/reference/pxmcmc/mcmc.py:349-368, prior.py:52-53)
// ---------------------------------------------------------------------------
struct LinArgs {
  const cplx* x[4];
  double a[4];
  int nx;
  const double* z;  // real vector added to the real part (may be null)
  double cz;
  double c0;  // real constant added to the real part
  cplx* out;
  size_t total;
};
__global__ void k_lincomb(LinArgs p) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < p.total; i += (size_t)gridDim.x * blockDim.x) {
    double re = 0.0, im = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (k < p.nx) {
        const cplx v = p.x[k][i];
        re += p.a[k] * v.x;
        im += p.a[k] * v.y;
      }
    }
    if (p.z) re += p.cz * p.z[i];
    re += p.c0;
    p.out[i] = make_double2(re, im);
  }
}

// ---------------------------------------------------------------------------
// SKROCK stages (/root/reference/pxmcmc/mcmc.py:338-368 and the published scheme of Abdulle, Almuslimani & Vilmart
// 2018), one pass per stage instead of gradlogpi + lincomb (+ philox_normal + lincomb at stage 1):
//   shift:  Y = U + cs Z
//   stage:  out = a g + b U + c V + c0 (+ e Z),  g = -((P - prox(P))/lmda) - gradg,
//           P = U + cs Z when Z is present (stage 1: neither Y nor Z is read back), else P = U.
// Each sum is accumulated in the order of the lincomb terms it replaces (stage 1: U, g, Z; later stages: g, U, V),
// products rounded on their own (this file is compiled without FMA contraction, as k_lincomb and k_gradlogpi are), so
// the reference scheme reproduces the composed kernels bit for bit.
// Z: injected real (mode 1) or real and imaginary (mode 2) normals, or the Philox normals pxm_philox_normal draws at
// (seed, stream0 + chain, step), regenerated here: mode 3 real, mode 4 complex = one draw of 2n normals per chain, the
// first n the real and the last n the imaginary parts.
// grid = (blocks per chain, chains in this launch); a thread owns elements (2 pr, 2 pr + 1) of one chain, so one
// Box-Muller pair serves both real parts and no 64-bit division runs per element.
// ---------------------------------------------------------------------------
struct SkrockArgs {
  const cplx* U;
  const cplx* V;      // null at stage 1
  const cplx* gradg;  // stage only
  const cplx* prox;   // may be null -> soft(P, T)
  const double* Tv;   // may be null -> Ts
  double Ts, lmda;
  double a, b, c, c0, cs, e;
  const double* z_re;  // modes 1, 2
  const double* z_im;  // mode 2
  int noise_mode;      // 0 none, 1 injected real, 2 injected complex, 3 Philox real, 4 Philox complex
  unsigned long long seed, step;
  const unsigned long long* step_ptr;  // may be null; otherwise the step is read from the device (CUDA-graph replays)
  unsigned int stream0;
  cplx* out;
  size_t n;
};

// the normals of elements e0 and e0 + 1 (when `two`) of `chain`; i0 = chain * n + e0
__device__ __forceinline__ void skrock_noise(const SkrockArgs& p, size_t chain, size_t e0, size_t i0, bool two,
                                             double zr[2], double zi[2]) {
  zr[0] = zr[1] = zi[0] = zi[1] = 0.0;
  if (p.noise_mode == 1 || p.noise_mode == 2) {
    zr[0] = p.z_re[i0];
    if (two) zr[1] = p.z_re[i0 + 1];
    if (p.noise_mode == 2) {
      zi[0] = p.z_im[i0];
      if (two) zi[1] = p.z_im[i0 + 1];
    }
  } else if (p.noise_mode >= 3) {
    const unsigned int stream = p.stream0 + (unsigned int)chain;
    philox_normal2(p.seed, stream, p.step, e0 >> 1, &zr[0], &zr[1]);
    if (p.noise_mode == 4) {
      const size_t k = p.n + e0;  // index of the imaginary part of element e0 in the chain's 2n draw
      double z0, z1;
      philox_normal2(p.seed, stream, p.step, k >> 1, &z0, &z1);
      if (!(k & 1)) {
        zi[0] = z0;
        zi[1] = z1;
      } else {
        zi[0] = z1;
        if (two) philox_normal2(p.seed, stream, p.step, (k >> 1) + 1, &zi[1], &z1);
      }
    }
  }
}

__global__ void k_skrock_shift(SkrockArgs p, size_t chain0) {
  if (p.step_ptr) p.step = *p.step_ptr;
  const size_t npairs = (p.n + 1) >> 1, chain = chain0 + blockIdx.y;
  const bool cz = p.noise_mode == 2 || p.noise_mode == 4;
  for (size_t pr = blockIdx.x * (size_t)blockDim.x + threadIdx.x; pr < npairs; pr += (size_t)gridDim.x * blockDim.x) {
    const size_t e0 = 2 * pr, i0 = chain * p.n + e0;
    const bool two = e0 + 1 < p.n;
    cplx u[2];
    u[0] = p.U[i0];
    u[1] = two ? p.U[i0 + 1] : make_double2(0.0, 0.0);
    double zr[2], zi[2];
    skrock_noise(p, chain, e0, i0, two, zr, zi);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      // lincomb([(1, U)], z=Z, cz=cs) / lincomb([(1, U), (cs, Z_re + i Z_im)]): 0 + 1 U, + cs Z, + 0 (real part)
      double re = 0.0, im = 0.0;
      re += u[h].x;
      im += u[h].y;
      re += p.cs * zr[h];
      if (cz) im += p.cs * zi[h];
      re += 0.0;
      p.out[i0 + h] = make_double2(re, im);
    }
  }
}

__global__ void k_skrock_stage(SkrockArgs p, size_t chain0) {
  if (p.step_ptr) p.step = *p.step_ptr;
  const size_t npairs = (p.n + 1) >> 1, chain = chain0 + blockIdx.y;
  const bool noise = p.noise_mode != 0, cz = p.noise_mode == 2 || p.noise_mode == 4;
  for (size_t pr = blockIdx.x * (size_t)blockDim.x + threadIdx.x; pr < npairs; pr += (size_t)gridDim.x * blockDim.x) {
    const size_t e0 = 2 * pr, i0 = chain * p.n + e0;
    const bool two = e0 + 1 < p.n;
    // every input of the pair is requested before any arithmetic
    cplx u[2], g[2], v[2], px[2];
    double T[2];
    u[0] = p.U[i0];
    g[0] = p.gradg[i0];
    u[1] = two ? p.U[i0 + 1] : make_double2(0.0, 0.0);
    g[1] = two ? p.gradg[i0 + 1] : make_double2(0.0, 0.0);
    if (p.V) {
      v[0] = p.V[i0];
      v[1] = two ? p.V[i0 + 1] : make_double2(0.0, 0.0);
    }
    if (p.prox) {
      px[0] = p.prox[i0];
      px[1] = two ? p.prox[i0 + 1] : make_double2(0.0, 0.0);
    } else {
      T[0] = p.Tv ? p.Tv[e0] : p.Ts;
      T[1] = (p.Tv && two) ? p.Tv[e0 + 1] : p.Ts;
    }
    double zr[2], zi[2];
    skrock_noise(p, chain, e0, i0, two, zr, zi);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      cplx P = u[h];
      if (noise) {  // the shift's Y, recomputed in registers (same operations as k_skrock_shift)
        double re = 0.0, im = 0.0;
        re += u[h].x;
        im += u[h].y;
        re += p.cs * zr[h];
        if (cz) im += p.cs * zi[h];
        re += 0.0;
        P = make_double2(re, im);
      }
      if (!p.prox) px[h] = soft_c(P, T[h]);
      // k_gradlogpi
      const double gx = -((P.x - px[h].x) / p.lmda) - g[h].x, gy = -((P.y - px[h].y) / p.lmda) - g[h].y;
      // k_lincomb, terms in the order the stages list them
      double re = 0.0, im = 0.0;
      if (p.V) {
        re += p.a * gx;
        im += p.a * gy;
        re += p.b * u[h].x;
        im += p.b * u[h].y;
        re += p.c * v[h].x;
        im += p.c * v[h].y;
      } else {
        re += p.b * u[h].x;
        im += p.b * u[h].y;
        re += p.a * gx;
        im += p.a * gy;
      }
      if (noise) {
        re += p.e * zr[h];
        if (cz) im += p.e * zi[h];
      }
      re += p.c0;
      p.out[i0 + h] = make_double2(re, im);
    }
  }
}

// ---------------------------------------------------------------------------
// FISTA (Beck & Teboulle 2009) for the synthesis-setting MAP, nchains independent problems:
//   x_{k+1} = soft(y_k - t gradg(y_k), s T),   y_{k+1} = x_{k+1} + beta_k (x_{k+1} - x_k),
//   beta_k = (tau_k - 1) / tau_{k+1},  tau_{k+1} = (1 + sqrt(1 + 4 tau_k^2)) / 2,  tau_0 = 1.
// The iteration counter k and tau_k live in the device state block {k, tau_k}, so one captured block of iterations
// replays unchanged.  Stage 1 also writes, per block, the partial sums of |x_{k+1} - x_k|^2 and |x_{k+1}|^2 (partial
// [chain][PXM_REDUCE_PARTS], the scratch scheme of pxm_reduce); stage 2 sums them in a fixed order into history slot
// k mod cap and advances the state.  y and x are read before they are written: x_out / y_out may be x_k / y_k.
// ---------------------------------------------------------------------------
struct FistaArgs {
  const cplx* y;
  const cplx* gradg;
  const cplx* x;
  const double* Tv;  // may be null -> Ts
  double Ts, Tscale, t;
  const double* state;  // {k, tau_k}
  cplx* x_out;
  cplx* y_out;
  cplx* partial;  // [nchains][gridDim.x]: (sum |x_{k+1} - x_k|^2, sum |x_{k+1}|^2)
  size_t n;
};

__device__ __forceinline__ double fista_next_tau(double tau) { return (1.0 + sqrt(1.0 + 4.0 * tau * tau)) / 2.0; }

__global__ void k_fista_update(FistaArgs p) {
  const double tau = p.state[1], tau1 = fista_next_tau(tau);
  const double beta = (tau - 1.0) / tau1;
  const size_t chain = blockIdx.y, off = chain * p.n;
  cplx acc = make_double2(0.0, 0.0);
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < p.n; e += (size_t)gridDim.x * blockDim.x) {
    const size_t i = off + e;
    const cplx y = p.y[i], g = p.gradg[i], xk = p.x[i];
    const double T = (p.Tv ? p.Tv[e] : p.Ts) * p.Tscale;
    const cplx xn = soft_c(make_double2(y.x - p.t * g.x, y.y - p.t * g.y), T);
    const double dx = xn.x - xk.x, dy = xn.y - xk.y;
    p.x_out[i] = xn;
    p.y_out[i] = make_double2(xn.x + beta * dx, xn.y + beta * dy);
    acc.x += dx * dx + dy * dy;
    acc.y += xn.x * xn.x + xn.y * xn.y;
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) p.partial[chain * gridDim.x + blockIdx.x] = acc;
}

// one CTA: every chain's partials in order, then the state advances (after every read of it in this launch)
__global__ void k_fista_finish(const cplx* __restrict__ partial, int nparts, int nchains, double* state, double* hist,
                               long long cap) {
  const long long slot = (long long)state[0] % cap;
  for (int c = 0; c < nchains; ++c) {
    cplx acc = make_double2(0.0, 0.0);
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
      const cplx v = partial[(size_t)c * nparts + i];
      acc.x += v.x;
      acc.y += v.y;
    }
    acc = block_sum(acc);
    if (threadIdx.x == 0) {
      hist[(slot * nchains + c) * 2] = acc.x;
      hist[(slot * nchains + c) * 2 + 1] = acc.y;
    }
  }
  if (threadIdx.x == 0) {
    const double tau = state[1];
    state[0] += 1.0;
    state[1] = fista_next_tau(tau);
  }
}

// ---------------------------------------------------------------------------
// masked gather / scatter with covariance weighting (weak lensing,
// /root/reference/pxmcmc/measurements.py:242-304)
// ---------------------------------------------------------------------------
__global__ void k_gather_w(const cplx* __restrict__ x, const int* __restrict__ idx, const double* __restrict__ w,
                           cplx* __restrict__ out, size_t nsel, size_t nfull, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t chain = i / nsel, e = i % nsel;
    cplx v = x[chain * nfull + idx[e]];
    const double s = w ? w[e] : 1.0;
    out[i] = make_double2(v.x * s, v.y * s);
  }
}
__global__ void k_scatter_w(const cplx* __restrict__ y, const int* __restrict__ idx, const double* __restrict__ w,
                            cplx* __restrict__ out, size_t nsel, size_t nfull, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t chain = i / nsel, e = i % nsel;
    cplx v = y[i];
    const double s = w ? w[e] : 1.0;
    out[chain * nfull + idx[e]] = make_double2(v.x * s, v.y * s);
  }
}

// ---------------------------------------------------------------------------
// pyssht harmonic layout  flm[chain][l^2+l+m]  <->  internal per-m slots
// (k4-interleaved rows lambda = l-|m|), with an optional real multiplier g[l]
// (harmonic-space kernels: weak-lensing k_l, measurements.py:151-171).
// ---------------------------------------------------------------------------
struct LmArgs {
  cplx* flm;          // [nchains][L*L]
  double* H;          // internal
  const unsigned long long* slot_off;  // per slot
  const double* gl;   // may be null
  const unsigned char* own;  // may be null; per slot: does this rank own the azimuthal order (m-sharded plans)
  int L, paired, nld, nchains, to_internal;
};
__global__ void k_lm_convert(LmArgs p) {
  const size_t per = (size_t)p.L * p.L;
  const size_t total = per * p.nchains;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int chain = (int)(i / per);
    const int ind = (int)(i % per);
    int l = (int)sqrt((double)ind);
    while (l * l > ind) --l;
    while ((l + 1) * (l + 1) <= ind) ++l;
    const int m = ind - l * l - l;
    const int am = m < 0 ? -m : m;
    int slot, col;
    // harmonic-side arrays hold the TRUE f_lm for both signs of m; the (-1)^m of
    // Lambda^{-m} = (-1)^m Lambda^{m} lives on the ring side only (ring FFT kernel)
    const double sg = 1.0;
    if (p.paired) {
      slot = am;
      col = chain * 4 + (m < 0 ? 2 : 0);
    } else {
      slot = m + p.L - 1;
      col = chain * 2;
    }
    if (p.own && !p.own[slot]) {  // another rank's order: nothing to load, zero on the way out
      if (!p.to_internal) p.flm[i] = make_double2(0.0, 0.0);
      continue;
    }
    const size_t base = p.slot_off[slot] + pxm_il_index(l - am, col, p.nld);
    const double gl = p.gl ? p.gl[l] : 1.0;
    if (p.to_internal) {
      const cplx v = p.flm[i];
      p.H[base] = sg * gl * v.x;
      p.H[base + 4] = sg * gl * v.y;
    } else {
      p.flm[i] = make_double2(sg * gl * p.H[base], sg * gl * p.H[base + 4]);
    }
  }
}

// real -> complex widening copy (the reference's X.astype(complex))
__global__ void k_r2c(const double* __restrict__ x, cplx* __restrict__ out, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    out[i] = make_double2(x[i], 0.0);
}

// ---------------------------------------------------------------------------
// CSR SpMV, warp per row, real values x complex vectors
// (/root/reference/pxmcmc/measurements.py:75-83: path_matrix.dot / getH().dot)
// ---------------------------------------------------------------------------
__global__ void k_csr_spmv(const int* __restrict__ indptr, const int* __restrict__ indices,
                           const double* __restrict__ vals, const cplx* __restrict__ x, cplx* __restrict__ y,
                           int nrows, size_t ncols) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const size_t chain = blockIdx.y;
  if (row >= nrows) return;
  const cplx* xc = x + chain * ncols;
  double re = 0.0, im = 0.0;
  for (int j = indptr[row] + lane; j < indptr[row + 1]; j += 32) {
    const double v = vals[j];
    const cplx xv = xc[indices[j]];
    re += v * xv.x;
    im += v * xv.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    re += __shfl_down_sync(0xffffffffu, re, o);
    im += __shfl_down_sync(0xffffffffu, im, o);
  }
  if (lane == 0) y[chain * (size_t)nrows + row] = make_double2(re, im);
}

// several chains per warp: the row's values and column indices are read ONCE for CH chains (a batch of chains
// multiplies the same matrix; with one chain per grid.y slice the matrix was re-read per chain)
template <int CH>
__global__ void k_csr_spmv_multi(const int* __restrict__ indptr, const int* __restrict__ indices,
                                 const double* __restrict__ vals, const cplx* __restrict__ x, cplx* __restrict__ y,
                                 int nrows, size_t ncols, int nchains) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int c0 = blockIdx.y * CH;
  if (row >= nrows) return;
  double re[CH], im[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) re[c] = im[c] = 0.0;
  const int nc = min(CH, nchains - c0);
  for (int j = indptr[row] + lane; j < indptr[row + 1]; j += 32) {
    const double v = vals[j];
    const size_t col = (size_t)indices[j];
#pragma unroll
    for (int c = 0; c < CH; ++c)
      if (c < nc) {
        const cplx xv = x[(size_t)(c0 + c) * ncols + col];
        re[c] += v * xv.x;
        im[c] += v * xv.y;
      }
  }
#pragma unroll
  for (int c = 0; c < CH; ++c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      re[c] += __shfl_down_sync(0xffffffffu, re[c], o);
      im[c] += __shfl_down_sync(0xffffffffu, im[c], o);
    }
    if (lane == 0 && c < nc) y[(size_t)(c0 + c) * (size_t)nrows + row] = make_double2(re[c], im[c]);
  }
}

// ---------------------------------------------------------------------------
// Column quantiles of a stored chain [nsamples][ld] (np.quantile(chain, (q_a, q_b), axis=0), method
// "linear": /root/reference/pxmcmc/uncertainty.py:7-16).  A CTA keeps C adjacent columns in shared
// memory (rows arrive as C consecutive doubles: coalesced), sorts every column with a bitonic network
// and interpolates exactly like numpy's _lerp (pxm_lerp_np).
// ---------------------------------------------------------------------------
__global__ void k_quantile_columns(const double* __restrict__ chain, long long nsamples, long long ncols, long long ld,
                                   int npad, int C, long long lo_a, double g_a, long long lo_b, double g_b,
                                   double* __restrict__ out_a, double* __restrict__ out_b) {
  extern __shared__ double qs[];
  const long long col0 = (long long)blockIdx.x * C;
  const int cs = npad + 1;  // column stride: the transposing stores of a row land in distinct banks
  const int nc = (int)min((long long)C, ncols - col0);
  for (long long i = threadIdx.x; i < (long long)npad * C; i += blockDim.x) {
    const long long row = i / C;
    const int c = (int)(i - row * C);
    double v = CUDART_INF;  // padding sorts to the end
    if (row < nsamples && c < nc) v = chain[row * ld + col0 + c];
    qs[c * cs + row] = v;
  }
  __syncthreads();
  const int half = npad >> 1;
  for (int size = 2; size <= npad; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < half * nc; i += blockDim.x) {
        const int c = i / half, k = i - c * half;
        const int pos = 2 * k - (k & (stride - 1));
        double* col = qs + c * cs;
        const double x = col[pos], y = col[pos + stride];
        const bool up = (pos & size) == 0;
        if ((x > y) == up) {
          col[pos] = y;
          col[pos + stride] = x;
        }
      }
      __syncthreads();
    }
  for (int c = threadIdx.x; c < nc; c += blockDim.x) {
    const double* col = qs + c * cs;
    const long long hi_a = min(lo_a + 1, nsamples - 1), hi_b = min(lo_b + 1, nsamples - 1);
    out_a[col0 + c] = pxm_lerp_np(col[lo_a], col[hi_a], g_a);
    out_b[col0 + c] = pxm_lerp_np(col[lo_b], col[hi_b], g_b);
  }
}

// ---------------------------------------------------------------------------
// PxMALA accept / reject on the device (/root/reference/pxmcmc/mcmc.py:240-259, :277-289): one thread evaluates
// log alpha = log q(Xc|Xp) + log pi(Xp) - log q(Xp|Xc) - log pi(Xc) from the four reductions, draws the uniform
// from the Philox stream of the step, writes the decision, the traces and -- when tuning -- the new step size,
// so that an iteration needs no host round trip.  State block S (doubles):
//   0 delta | 1 1-delta/lmda | 2 delta/lmda | 3 sqrt(2 delta) | 4,5 log pi(Xc) | 6,7 L2(Xc) | 8 prior(Xc) | 9 accepted
//   10 log u | 11,12 log alpha | 13 iteration index | 14 Philox step  (13, 14: used -- and advanced -- when the
//   launch passes i < 0, the form a captured CUDA graph replays)
// ---------------------------------------------------------------------------
struct AcceptArgs {
  double* S;
  const cplx* s1;      // sum (Xp - Xc - (delta/2) grad log pi(Xc))^2
  const cplx* s2;      // sum (Xc - Xp - (delta/2) grad log pi(Xp))^2
  const cplx* L2p;
  const cplx* priorp;  // real part used
  double mu, lmda;
  int tune;
  long long i;         // iteration index
  unsigned long long seed, step;
  unsigned int stream;
  signed char* acc_trace;   // [nchains][trace_stride], entries 0..i
  double* delta_trace;      // [nchains][trace_stride + 1], entries 0..i+1; entry 0 = initial delta
  long long trace_stride;
  int nchains;
};
__global__ void k_pxmala_accept(AcceptArgs p) {
  const int chain = blockIdx.x * blockDim.x + threadIdx.x;  // one thread per chain
  if (chain >= p.nchains) return;
  double* S = p.S + (size_t)chain * PXM_STATE_DOUBLES;
  p.s1 += chain;
  p.s2 += chain;
  p.L2p += chain;
  p.priorp += chain;
  p.stream += (unsigned int)chain;
  p.acc_trace += (size_t)chain * p.trace_stride;
  p.delta_trace += (size_t)chain * (p.trace_stride + 1);
  const bool counters_on_device = p.i < 0;
  if (counters_on_device) {
    p.i = (long long)S[13];
    p.step = (unsigned long long)S[14];
  }
  const double delta = S[0];
  const double k = -(1.0 / 2 * delta);  // as coded in the reference: (1/2*delta) = delta/2
  const cplx a1 = p.s1[0], a2 = p.s2[0];
  const cplx q1 = make_double2(a1.x * a1.x - a1.y * a1.y, a1.x * a1.y + a1.y * a1.x);  // s1 ** 2
  const cplx q2 = make_double2(a2.x * a2.x - a2.y * a2.y, a2.x * a2.y + a2.y * a2.x);
  const cplx ltXcXp = make_double2(k * q1.x, k * q1.y), ltXpXc = make_double2(k * q2.x, k * q2.y);
  const cplx L2p = p.L2p[0];
  const double priorp = p.priorp[0].x;
  const cplx lpp = make_double2(-p.mu * priorp - L2p.x, -L2p.y);
  cplx la = make_double2(ltXpXc.x + lpp.x, ltXpXc.y + lpp.y);
  la = make_double2(la.x - ltXcXp.x, la.y - ltXcXp.y);
  la = make_double2(la.x - S[4], la.y - S[5]);
  // uniform of this step: the Philox block no coefficient pair can reach
  uint32_t c[4] = {0xFFFFFFFFu, 0xFFFFFFFFu, (uint32_t)p.step, (uint32_t)(p.step >> 32) ^ (p.stream * 0x85EBCA6Bu)};
  philox4x32_10(c, (uint32_t)p.seed, (uint32_t)(p.seed >> 32) ^ p.stream);
  const unsigned long long bits = ((unsigned long long)c[0] << 32) | c[1];
  const double lu = log(((double)(bits >> 11) + 0.5) * (1.0 / 9007199254740992.0));
  // numpy's ordering of complex numbers: real parts first, then imaginary parts (log u is real)
  const bool accept = (lu < la.x) || (lu == la.x && 0.0 < la.y);
  S[9] = accept ? 1.0 : 0.0;
  S[10] = lu;
  S[11] = la.x;
  S[12] = la.y;
  if (accept) {
    S[4] = lpp.x;
    S[5] = lpp.y;
    S[6] = L2p.x;
    S[7] = L2p.y;
    S[8] = priorp;
  }
  // the traces are rings of trace_stride slots: the host drains them every trace_stride iterations
  const long long slot = p.i % (long long)p.trace_stride;
  p.acc_trace[slot] = accept ? 1 : 0;
  if (p.tune) {
    double d = delta * (1 + ((accept ? 1.0 : 0.0) - 0.5) / pow((double)(p.i + 1), 0.75));
    d = fmin(fmax(d, p.lmda * 1e-8), p.lmda / 2);
    S[0] = d;
    S[1] = 1 - d / p.lmda;
    S[2] = d / p.lmda;
    S[3] = sqrt(2 * d);
    p.delta_trace[slot + 1] = d;
  }
  if (counters_on_device) {
    S[13] = (double)(p.i + 1);
    S[14] = (double)(p.step + 1);
  }
}
// the accepted proposal becomes the current state: up to four arrays copied when S[9] != 0
struct SelectArgs {
  const double* flag;   // chain c: flag[flag_stride c]
  size_t flag_stride;
  size_t nchains;
  cplx* dst[4];
  const cplx* src[4];
  size_t n[4];          // elements per chain
};
__global__ void k_select(SelectArgs p) {
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const size_t tot = p.n[a] * p.nchains;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < tot; i += (size_t)gridDim.x * blockDim.x)
      if (p.flag[(i / p.n[a]) * p.flag_stride] != 0.0) p.dst[a][i] = p.src[a][i];
  }
}

// standard normals from the Philox stream (seed, stream0 + chain, step): element e of a chain is normal (e & 1) of
// pair e >> 1 -- the same numbers the MYULA update kernel draws (SKROCK's Z, /root/reference/pxmcmc/mcmc.py:344)
__global__ void k_philox_normal(double* __restrict__ out, size_t n, size_t nchains, unsigned long long seed,
                                unsigned long long step, const unsigned long long* step_ptr, unsigned int stream0) {
  if (step_ptr) step = *step_ptr;
  const size_t npairs = (n + 1) >> 1, tot = npairs * nchains;
  for (size_t q = blockIdx.x * (size_t)blockDim.x + threadIdx.x; q < tot; q += (size_t)gridDim.x * blockDim.x) {
    const size_t chain = q / npairs, pr = q - chain * npairs;
    double z0, z1;
    philox_normal2(seed, stream0 + (unsigned int)chain, step, pr, &z0, &z1);
    out[chain * n + 2 * pr] = z0;
    if (2 * pr + 1 < n) out[chain * n + 2 * pr + 1] = z1;
  }
}

inline int grid_for(size_t total, int block = 256) {
  size_t g = (total + block - 1) / block;
  const size_t cap = 148 * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

// ------------------------------- launchers ---------------------------------
int pxm_launch_soft(int is_complex, const void* x, const double* Tv, double Ts, void* out, size_t n, size_t nchains,
                    cudaStream_t st) {
  const size_t total = n * nchains;
  if (!total) return PXM_OK;
  if (is_complex)
    k_soft_c<<<grid_for(total), 256, 0, st>>>((const cplx*)x, Tv, Ts, (cplx*)out, n, total);
  else
    k_soft_r<<<grid_for(total), 256, 0, st>>>((const double*)x, Tv, Ts, (double*)out, n, total);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_myula(const void* X, const void* prox, const void* gradg, const double* Tv, double Ts,
                     const double* w_re, const double* w_im, void* Xout, void* prox_out, size_t n, size_t nchains,
                     double delta, double lmda, int noise_mode, unsigned long long seed, unsigned long long step,
                     const unsigned long long* d_step, unsigned int stream0, cudaStream_t st, const double* d_par) {
  MyulaArgs p;
  p.step_ptr = d_step;
  p.dpar = d_par;
  p.X = (const cplx*)X;
  p.prox = (const cplx*)prox;
  p.gradg = (const cplx*)gradg;
  p.Tv = Tv;
  p.Ts = Ts;
  p.w_re = w_re;
  p.w_im = w_im;
  p.Xout = (cplx*)Xout;
  p.prox_out = (cplx*)prox_out;
  p.n = n;
  p.total = n * nchains;
  p.a = 1 - delta / lmda;  // same expressions as mcmc.py:197-200
  p.b = delta / lmda;
  p.delta = delta;
  p.sq2d = sqrt(2 * delta);
  p.noise_mode = noise_mode;
  p.seed = seed;
  p.step = step;
  p.stream0 = stream0;
  if (!p.total) return PXM_OK;
  if (noise_mode == 2 || noise_mode == 4) {
    const size_t npairs = (n + 1) / 2;
    for (size_t c0 = 0; c0 < nchains; c0 += 65535) {
      const size_t nc = std::min<size_t>(nchains - c0, 65535);
      const int per_chain = std::max(1, std::min(grid_for(npairs), (int)((148 * 16 + nc - 1) / nc)));
      if (noise_mode == 2)
        k_myula_update_pair<<<dim3(per_chain, (unsigned)nc), 256, 0, st>>>(p, c0);
      else
        k_myula_update_realpair<<<dim3(per_chain, (unsigned)nc), 256, 0, st>>>(p, c0);
    }
  } else
    k_myula_update<<<grid_for(p.total), 256, 0, st>>>(p);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_counter_add(unsigned long long* ctr, unsigned long long inc, cudaStream_t st) {
  k_counter_add<<<1, 1, 0, st>>>(ctr, inc);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_resid(const void* preds, const void* data, const void* ic, void* out, size_t n, size_t nchains,
                     cudaStream_t st) {
  const size_t total = n * nchains;
  if (!total) return PXM_OK;
  k_resid<<<grid_for(total), 256, 0, st>>>((const cplx*)preds, (const cplx*)data, (const cplx*)ic, (cplx*)out, n, total);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_ring_resid(const double* pred, const double* data, const void* ic, double* out, int nslots, int rings,
                          int nld, int ncols, double scale, unsigned long long slot_stride, cudaStream_t st) {
  const unsigned long long total = (unsigned long long)nslots * ((rings + 3) / 4) * (ncols / 2) * 4;
  if (!total) return PXM_OK;
  k_ring_resid<<<grid_for((size_t)total), 256, 0, st>>>(pred, data, (const cplx*)ic, out, rings, nld, ncols, scale, slot_stride, total);
  PXM_LAUNCHED();
  return PXM_OK;
}

constexpr int PXM_REDUCE_PARTS = 148;

int pxm_launch_reduce(int kind, const void* a, const void* b, const void* c, const void* d, const double* w,
                      double delta, double lmda, size_t n, size_t nchains, void* partial, void* out,
                      cudaStream_t st, const double* d_par) {
  ReduceArgs p;
  p.kind = kind;
  p.dpar = d_par;
  p.a = (const cplx*)a;
  p.b = (const cplx*)b;
  p.c = (const cplx*)c;
  p.d = (const cplx*)d;
  p.w = w;
  p.delta = delta;
  p.lmda = lmda;
  p.n = n;
  p.partial = (cplx*)partial;
  p.out = (cplx*)out;
  if (!nchains) return PXM_OK;
  dim3 grid(PXM_REDUCE_PARTS, (unsigned)nchains);
  k_reduce_stage1<<<grid, 256, 0, st>>>(p);
  PXM_LAUNCHED();
  k_reduce_stage2<<<(unsigned)nchains, 256, 0, st>>>((const cplx*)partial, PXM_REDUCE_PARTS, (cplx*)out);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_lincomb(int nx, const void* const* xs, const double* as, const double* z, double cz, double c0,
                       void* out, size_t total, cudaStream_t st) {
  LinArgs p;
  p.nx = nx;
  for (int k = 0; k < 4; ++k) {
    p.x[k] = k < nx ? (const cplx*)xs[k] : nullptr;
    p.a[k] = k < nx ? as[k] : 0.0;
  }
  p.z = z;
  p.cz = cz;
  p.c0 = c0;
  p.out = (cplx*)out;
  p.total = total;
  if (!total) return PXM_OK;
  k_lincomb<<<grid_for(total), 256, 0, st>>>(p);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_skrock(int stage, const void* U, const void* V, const void* gradg, const void* prox, const double* Tv,
                      double Ts, double lmda, double a, double b, double c, double c0, double cs, double e,
                      const double* z_re, const double* z_im, int noise_mode, unsigned long long seed,
                      unsigned long long step, const unsigned long long* d_step, unsigned int stream0, void* out, size_t n,
                      size_t nchains, cudaStream_t st) {
  SkrockArgs p;
  p.U = (const cplx*)U;
  p.V = (const cplx*)V;
  p.gradg = (const cplx*)gradg;
  p.prox = (const cplx*)prox;
  p.Tv = Tv;
  p.Ts = Ts;
  p.lmda = lmda;
  p.a = a;
  p.b = b;
  p.c = c;
  p.c0 = c0;
  p.cs = cs;
  p.e = e;
  p.z_re = z_re;
  p.z_im = z_im;
  p.noise_mode = noise_mode;
  p.seed = seed;
  p.step = step;
  p.step_ptr = d_step;
  p.stream0 = stream0;
  p.out = (cplx*)out;
  p.n = n;
  if (!n || !nchains) return PXM_OK;
  const size_t npairs = (n + 1) / 2;
  for (size_t c0c = 0; c0c < nchains; c0c += 65535) {
    const size_t nc = std::min<size_t>(nchains - c0c, 65535);
    const int per_chain = std::max(1, std::min(grid_for(npairs), (int)((148 * 16 + nc - 1) / nc)));
    if (stage)
      k_skrock_stage<<<dim3(per_chain, (unsigned)nc), 256, 0, st>>>(p, c0c);
    else
      k_skrock_shift<<<dim3(per_chain, (unsigned)nc), 256, 0, st>>>(p, c0c);
    PXM_LAUNCHED();
  }
  return PXM_OK;
}

int pxm_launch_fista(const void* y, const void* gradg, const void* x, const double* Tv, double Ts, double Tscale,
                     double t, double* state, void* x_out, void* y_out, double* hist, long long cap, size_t n,
                     size_t nchains, void* partial, cudaStream_t st) {
  FistaArgs p;
  p.y = (const cplx*)y;
  p.gradg = (const cplx*)gradg;
  p.x = (const cplx*)x;
  p.Tv = Tv;
  p.Ts = Ts;
  p.Tscale = Tscale;
  p.t = t;
  p.state = state;
  p.x_out = (cplx*)x_out;
  p.y_out = (cplx*)y_out;
  p.partial = (cplx*)partial;
  p.n = n;
  if (!nchains) return PXM_OK;
  k_fista_update<<<dim3(PXM_REDUCE_PARTS, (unsigned)nchains), 256, 0, st>>>(p);
  PXM_LAUNCHED();
  k_fista_finish<<<1, 256, 0, st>>>((const cplx*)partial, PXM_REDUCE_PARTS, (int)nchains, state, hist, cap);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_gather(int scatter, const void* in, const int* idx, const double* w, void* out, size_t nsel,
                      size_t nfull, size_t nchains, cudaStream_t st) {
  const size_t total = nsel * nchains;
  if (scatter) PXM_CUDA(cudaMemsetAsync(out, 0, nfull * nchains * sizeof(cplx), st));
  if (!total) return PXM_OK;
  if (scatter)
    k_scatter_w<<<grid_for(total), 256, 0, st>>>((const cplx*)in, idx, w, (cplx*)out, nsel, nfull, total);
  else
    k_gather_w<<<grid_for(total), 256, 0, st>>>((const cplx*)in, idx, w, (cplx*)out, nsel, nfull, total);
  PXM_LAUNCHED();
  return PXM_OK;
}

// force-load every kernel of this file (see pxm_legendre_preload)
int pxm_elem_preload() {
  cudaFuncAttributes a;
  PXM_CUDA(cudaFuncGetAttributes(&a, k_lm_convert));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_soft_c));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_soft_r));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_myula_update));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_myula_update_pair));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_myula_update_realpair));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_resid));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_ring_resid));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_reduce_stage1));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_reduce_stage2));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_gradlogpi));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_lincomb));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_skrock_shift));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_skrock_stage));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_fista_update));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_fista_finish));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_gather_w));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_scatter_w));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_r2c));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_csr_spmv));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_csr_spmv_multi<4>));
  PXM_CUDA(cudaFuncGetAttributes(&a, k_counter_add));
  return PXM_OK;
}

int pxm_launch_lm_convert(int to_internal, void* flm, double* H, const unsigned long long* d_slot_off,
                          const unsigned char* d_own, const double* d_gl, int L, int paired, int nld, int nchains,
                          cudaStream_t st) {
  LmArgs p;
  p.own = d_own;
  p.flm = (cplx*)flm;
  p.H = H;
  p.slot_off = d_slot_off;
  p.gl = d_gl;
  p.L = L;
  p.paired = paired;
  p.nld = nld;
  p.nchains = nchains;
  p.to_internal = to_internal;
  const size_t total = (size_t)L * L * nchains;
  if (!total) return PXM_OK;
  k_lm_convert<<<grid_for(total), 256, 0, st>>>(p);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_r2c(const double* x, void* out, size_t total, cudaStream_t st) {
  if (!total) return PXM_OK;
  k_r2c<<<grid_for(total), 256, 0, st>>>(x, (cplx*)out, total);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_csr_spmv(const int* indptr, const int* indices, const double* vals, const void* x, void* y, int nrows,
                        size_t ncols, size_t nchains, cudaStream_t st) {
  if (!nrows || !nchains) return PXM_OK;
  if (nchains == 1) {
    dim3 grid((unsigned)(((size_t)nrows * 32 + 255) / 256), 1);
    k_csr_spmv<<<grid, 256, 0, st>>>(indptr, indices, vals, (const cplx*)x, (cplx*)y, nrows, ncols);
  } else {
    constexpr int CH = 4;
    dim3 grid((unsigned)(((size_t)nrows * 32 + 255) / 256), (unsigned)((nchains + CH - 1) / CH));
    k_csr_spmv_multi<CH><<<grid, 256, 0, st>>>(indptr, indices, vals, (const cplx*)x, (cplx*)y, nrows, ncols, (int)nchains);
  }
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_gradlogpi(const void* X, const void* prox, const double* Tv, double Ts, const void* gradg, double lmda,
                         void* out, size_t n, size_t nchains, cudaStream_t st) {
  const size_t total = n * nchains;
  if (!total) return PXM_OK;
  k_gradlogpi<<<grid_for(total), 256, 0, st>>>((const cplx*)X, (const cplx*)prox, Tv, Ts, (const cplx*)gradg, lmda,
                                                (cplx*)out, n, total);
  PXM_LAUNCHED();
  return PXM_OK;
}

// largest chain length the in-shared-memory sort handles (one column of 2^14 doubles + padding)
int pxm_quantile_max_samples() { return 16384; }

int pxm_launch_quantile_columns(const double* chain, long long nsamples, long long ncols, long long ld, long long lo_a,
                                double g_a, long long lo_b, double g_b, double* out_a, double* out_b, cudaStream_t st) {
  if (nsamples <= 0 || ncols <= 0) return PXM_OK;
  if (nsamples > pxm_quantile_max_samples()) {
    pxm_set_error("quantile: more samples than the shared-memory sort holds (16384)");
    return PXM_ERR_UNSUPPORTED;
  }
  int npad = 2;
  while (npad < nsamples) npad <<= 1;
  const size_t budget = 200 * 1024;
  int C = (int)(budget / ((size_t)(npad + 1) * 8));
  if (C > 32) C = 32;
  if (C < 1) C = 1;
  const size_t smem = (size_t)C * (npad + 1) * 8;
  static bool configured = false;
  if (!configured) {
    PXM_CUDA(cudaFuncSetAttribute(k_quantile_columns, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    configured = true;
  }
  const long long grid = (ncols + C - 1) / C;
  k_quantile_columns<<<(unsigned)grid, 256, smem, st>>>(chain, nsamples, ncols, ld, npad, C, lo_a, g_a, lo_b, g_b, out_a, out_b);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_pxmala_accept(double* S, const void* s1, const void* s2, const void* L2p, const void* priorp, double mu,
                             double lmda, int tune, long long i, unsigned long long seed, unsigned long long step,
                             unsigned int stream_id, signed char* acc_trace, double* delta_trace, long long trace_stride,
                             int nchains, cudaStream_t st) {
  AcceptArgs p;
  p.trace_stride = trace_stride;
  p.nchains = nchains;
  p.S = S;
  p.s1 = (const cplx*)s1;
  p.s2 = (const cplx*)s2;
  p.L2p = (const cplx*)L2p;
  p.priorp = (const cplx*)priorp;
  p.mu = mu;
  p.lmda = lmda;
  p.tune = tune;
  p.i = i;
  p.seed = seed;
  p.step = step;
  p.stream = stream_id;
  p.acc_trace = acc_trace;
  p.delta_trace = delta_trace;
  k_pxmala_accept<<<(nchains + 63) / 64, 64, 0, st>>>(p);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_select(const double* flag, size_t flag_stride, size_t nchains, void* const* dst, const void* const* src,
                      const size_t* counts, int narrays, cudaStream_t st) {
  SelectArgs p;
  p.flag = flag;
  p.flag_stride = flag_stride;
  p.nchains = nchains;
  size_t mx = 0;
  for (int a = 0; a < 4; ++a) {
    p.dst[a] = a < narrays ? (cplx*)dst[a] : nullptr;
    p.src[a] = a < narrays ? (const cplx*)src[a] : nullptr;
    p.n[a] = a < narrays ? counts[a] : 0;
    mx = p.n[a] > mx ? p.n[a] : mx;
  }
  if (!mx) return PXM_OK;
  k_select<<<grid_for(mx * nchains), 256, 0, st>>>(p);
  PXM_LAUNCHED();
  return PXM_OK;
}

int pxm_launch_philox_normal(double* out, size_t n, size_t nchains, unsigned long long seed, unsigned long long step,
                             const unsigned long long* d_step, unsigned int stream0, cudaStream_t st) {
  if (!n || !nchains) return PXM_OK;
  k_philox_normal<<<grid_for(((n + 1) / 2) * nchains), 256, 0, st>>>(out, n, nchains, seed, step, d_step, stream0);
  PXM_LAUNCHED();
  return PXM_OK;
}

// Batched phi-direction DFT of MW rings (odd length n = 2l-1) for every
// bandlimit of a transform in ONE launch, fused with the transposition between
// the pixel layout [chain][ring t][phi p] and the per-m "k4-interleaved" layout
// the Legendre contraction consumes.
//
// Replaces the FFTW calls inside ssht (reference call sites:
// /root/reference/pxmcmc/transforms.py:95-98, pxmcmc/measurements.py:223-239).
// Odd, often prime lengths (511, 389, 259, 173, ...) => Bluestein chirp-z with a
// power-of-two length M >= 2n-1, entirely on-chip:
//   * in-place radix-16 passes (one leading radix-2/4/8 pass when log2 M is not a
//     multiple of 4); every thread holds its 16 points in registers, shared
//     memory is only the exchange medium between passes and is padded by one
//     element per 16 so that both the strided and the contiguous access patterns
//     are bank-conflict free;
//   * decimation in frequency forward, decimation in time inverse, so the
//     spectrum is only ever seen in the kernel's own digit-reversed order (the
//     filter spectrum is precomputed in that order: no reordering pass exists);
//   * the last forward pass, the product with the filter spectrum and the first
//     inverse pass act on the same 16 contiguous points and are fused in
//     registers.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstdint>
#include <map>
#include <mutex>
#include <tuple>

#include "pxm_common.cuh"
#include "pxm_dft.cuh"

namespace {

__device__ __forceinline__ int padi(int i) { return i + (i >> 4); }

// One in-place pass over 2^lgnr rings (padded stride MP): sub-transform length 2^lgLs,
// radix R, element stride S = Ls/R >= 16 (so the padded address is affine in k).
// Forward (DIF): butterfly then twiddle; inverse (DIT): conj-twiddle then butterfly.
template <int R, bool INV>
__device__ __forceinline__ void fft_pass(cplx* s, int lgnr, int lgM, int MP, int lgLs, const cplx* __restrict__ tw) {
  constexpr int lgR = R == 2 ? 1 : R == 4 ? 2 : R == 8 ? 3 : 4;
  const int lgS = lgLs - lgR, S = 1 << lgS, lgnbf = lgM - lgR, tstep = 1 << (lgM - lgLs);
  const int stride = S + (S >> 4);
  const int total = 1 << (lgnr + lgnbf);
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int r = idx >> lgnbf, b = idx & ((1 << lgnbf) - 1);
    const int blk = b >> lgS, j = b & (S - 1);
    cplx* p = s + r * MP + padi((blk << lgLs) + j);
    cplx x[R];
#pragma unroll
    for (int k = 0; k < R; ++k) x[k] = p[k * stride];
    // twiddles w^k, k < R, from ONE table load; the powers are formed on the fly in
    // two interleaved chains (even / odd exponents, <= 8 products deep => a few ulp),
    // which keeps the L1TEX pipe free for the shared-memory exchange
    if (INV) {
      cplx w1 = tw[j * tstep];
      w1.y = -w1.y;
      const cplx w2 = cmul(w1, w1);
      cplx wo = w1, we = w2;
#pragma unroll
      for (int k = 1; k < R; k += 2) {
        x[k] = cmul(x[k], wo);
        if (k + 1 < R) x[k + 1] = cmul(x[k + 1], we);
        wo = cmul(wo, w2);
        we = cmul(we, w2);
      }
      dftR<R, INV>(x);
    } else {
      dftR<R, INV>(x);
      const cplx w1 = tw[j * tstep];
      const cplx w2 = cmul(w1, w1);
      cplx wo = w1, we = w2;
#pragma unroll
      for (int k = 1; k < R; k += 2) {
        x[k] = cmul(x[k], wo);
        if (k + 1 < R) x[k + 1] = cmul(x[k + 1], we);
        wo = cmul(wo, w2);
        we = cmul(we, w2);
      }
    }
#pragma unroll
    for (int k = 0; k < R; ++k) p[k * stride] = x[k];
  }
  __syncthreads();
}

__device__ __forceinline__ int first_radix_log(int logM) { return logM & 3; }  // 0 -> only radix-16 passes

// forward passes except the last (Ls = 16) one
__device__ void fft_forward_head(cplx* s, int lgnr, int lgM, int MP, const cplx* __restrict__ tw) {
  int lgLs = lgM;
  const int f = first_radix_log(lgM);
  if (f == 1) {
    fft_pass<2, false>(s, lgnr, lgM, MP, lgLs, tw);
    lgLs -= 1;
  } else if (f == 2) {
    fft_pass<4, false>(s, lgnr, lgM, MP, lgLs, tw);
    lgLs -= 2;
  } else if (f == 3) {
    fft_pass<8, false>(s, lgnr, lgM, MP, lgLs, tw);
    lgLs -= 3;
  }
  for (; lgLs > 4; lgLs -= 4) fft_pass<16, false>(s, lgnr, lgM, MP, lgLs, tw);
}
// inverse passes except the first (Ls = 16) one
__device__ void fft_inverse_tail(cplx* s, int lgnr, int lgM, int MP, const cplx* __restrict__ tw) {
  const int f = first_radix_log(lgM);
  const int top16 = lgM - f;  // largest Ls handled by radix-16 passes
  for (int lgLs = 8; lgLs <= top16; lgLs += 4) fft_pass<16, true>(s, lgnr, lgM, MP, lgLs, tw);
  if (f == 1) fft_pass<2, true>(s, lgnr, lgM, MP, lgM, tw);
  if (f == 2) fft_pass<4, true>(s, lgnr, lgM, MP, lgM, tw);
  if (f == 3) fft_pass<8, true>(s, lgnr, lgM, MP, lgM, tw);
}
// middle: last forward pass (contiguous 16 points, no twiddles) x filter spectrum x first inverse
// pass; bhat == nullptr: plain last forward pass (used to build the filter spectrum itself)
__device__ void fft_middle(cplx* s, int lgnr, int lgM, int MP, const cplx* __restrict__ bhat) {
  const int lgnbf = lgM - 4, nbf = 1 << lgnbf;
  const int total = 1 << (lgnr + lgnbf);
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int r = idx >> lgnbf, b = idx & (nbf - 1);
    cplx* p = s + r * MP + b * 17;  // padi(16 b + k) = 17 b + k
    cplx x[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) x[k] = p[k];
    dft16<false>(x);
    if (bhat) {
      const cplx* bh = bhat + b;  // filter spectrum stored [k][b]: coalesced across the lanes
#pragma unroll
      for (int k = 0; k < 16; ++k) x[k] = cmul(x[k], bh[k << lgnbf]);
      dft16<true>(x);
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) p[k] = x[k];
  }
  __syncthreads();
}

// ---- table setup -------------------------------------------------------------
__global__ void fft_fill_tables_kernel(const PxmFftGroup* groups, int ngroups, cplx* arena) {
  const PxmFftGroup gr = groups[blockIdx.x];
  cplx* chirp = arena + gr.chirp_off;
  cplx* tw = arena + gr.tw_off;
  for (int j = threadIdx.x; j < gr.n; j += blockDim.x) {
    const long long r = ((long long)j * j) % (2LL * gr.n);
    double sn, cs;
    sincospi(-(double)r / (double)gr.n, &sn, &cs);
    chirp[j] = make_double2(cs, sn);
  }
  for (int k = threadIdx.x; k < gr.M; k += blockDim.x) {
    double sn, cs;
    sincospi(-2.0 * (double)k / (double)gr.M, &sn, &cs);
    tw[k] = make_double2(cs, sn);
  }
  if (gr.logM == 9 || gr.logM == 10) {  // twiddles of the persistent two-pass kernel, in both thread orders
    const int R2 = 32, R1 = gr.M / R2;
    cplx* tw2 = arena + gr.tw2_off;
    for (int i = threadIdx.x; i < gr.M; i += blockDim.x) {
      const int k1 = i / R2, j2 = i - k1 * R2;
      double sn, cs;
      sincospi(-2.0 * (double)((k1 * j2) % gr.M) / (double)gr.M, &sn, &cs);
      tw2[k1 * R2 + j2] = make_double2(cs, sn);
      tw2[gr.M + j2 * R1 + k1] = make_double2(cs, sn);
    }
  }
}

// filter spectrum in the digit-reversed order produced by the forward passes
__global__ void fft_fill_bhat_kernel(const PxmFftGroup* groups, int ngroups, cplx* arena) {
  extern __shared__ __align__(16) unsigned char fsm[];
  cplx* s = reinterpret_cast<cplx*>(fsm);
  const PxmFftGroup gr = groups[blockIdx.x];
  const int M = gr.M, MP = M + (M >> 4) + 2;
  const cplx* chirp = arena + gr.chirp_off;
  for (int i = threadIdx.x; i < MP; i += blockDim.x) s[i] = make_double2(0.0, 0.0);
  __syncthreads();
  for (int j = threadIdx.x; j < gr.n; j += blockDim.x) {
    const cplx c = chirp[j];
    const cplx b = make_double2(c.x, -c.y);
    s[padi(j)] = b;
    if (j > 0) s[padi(M - j)] = b;
  }
  __syncthreads();
  fft_forward_head(s, 0, gr.logM, MP, arena + gr.tw_off);
  fft_middle(s, 0, gr.logM, MP, nullptr);
  cplx* bhat = arena + gr.bhat_off;
  for (int i = threadIdx.x; i < M; i += blockDim.x) bhat[(i & 15) * (M >> 4) + (i >> 4)] = s[padi(i)];
}

// filter spectrum in NATURAL order for the two-pass kernel: Bhat[k] = sum_j b_j e^{-2 pi i j k / M},
// b_j = conj(c_|j|) for |j| < n (wrapped), by direct summation (plan creation only)
__global__ void fft_fill_bhat2_kernel(const PxmFftGroup* groups, int ngroups, cplx* arena) {
  const PxmFftGroup gr = groups[blockIdx.y];
  const int M = gr.M, n = gr.n;
  const cplx* chirp = arena + gr.chirp_off;
  cplx* out = arena + gr.bhat2_off;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < M; k += gridDim.x * blockDim.x) {
    double re = chirp[0].x, im = -chirp[0].y;
    for (int j = 1; j < n; ++j) {
      // b_j (e^{-i a} + e^{+i a}) with a = 2 pi j k / M : the +j and the wrapped -j entry
      const long long r = ((long long)j * k) % M;
      const double c = cospi(2.0 * (double)r / (double)M);
      re += 2.0 * c * chirp[j].x;
      im += 2.0 * c * (-chirp[j].y);
    }
    out[k] = make_double2(re, im);
  }
}

// ---- the ring transform ---------------------------------------------------------
// DIR 0: pixels -> ring coefficients  F_m[t] = scale * sum_p f[t,p] e^{-i m phi_p}
// DIR 1: ring coefficients -> pixels  f[t,p] = scale * sum_m F_m[t] e^{+i m phi_p}
// A CTA owns 2^lgr consecutive rings (a whole number of k4 row-groups when >= 4).
// m-sharded plans: a rank transforms only the rings [ring0, rings) it owns; its pixel vector holds those rows.
#ifndef PXM_FFT_MINB
#define PXM_FFT_MINB 3
#endif
template <int DIR>
__global__ void __launch_bounds__(256, PXM_FFT_MINB)
pxm_ring_fft_kernel(const PxmFftGroup* __restrict__ groups, int ngroups, cplx* __restrict__ pix,
                    size_t pix_chain_stride, double* __restrict__ F, int nld, const cplx* __restrict__ arena,
                    int min_logM) {
  extern __shared__ __align__(16) unsigned char fsm[];
  cplx* s = reinterpret_cast<cplx*>(fsm);
  int gi = 0;
  while (gi + 1 < ngroups && (int)blockIdx.x >= groups[gi + 1].cta_begin) ++gi;
  const PxmFftGroup gr = groups[gi];
  if (min_logM > 0 && gr.logM < min_logM) return;  // this group belongs to the two-pass kernels
  const int chain = blockIdx.y;
  const int lgr = gr.pad;  // log2(rings per CTA)
  const int t0 = gr.ring0 + (((int)blockIdx.x - gr.cta_begin) << lgr);  // global ring index
  const int n = gr.n, M = gr.M, ell = gr.ell, lgM = gr.logM, rings = gr.rings;
  const int MP = M + (M >> 4) + 2;  // +2: the rings of one row-group land in different banks
  const cplx* chirp = arena + gr.chirp_off;
  const cplx* bhat = arena + gr.bhat_off;
  const cplx* tw = arena + gr.tw_off;
  cplx* mypix = pix + (size_t)chain * pix_chain_stride + gr.pix_off;
  // gather / scatter of the k4-interleaved ring array: a thread keeps ONE ring (ring index fastest
  // across the lanes: the 4 rings of a row-group are adjacent doubles) and walks over m
  const int rr = threadIdx.x & ((1 << lgr) - 1);
  const int j0 = threadIdx.x >> lgr, jstep = blockDim.x >> lgr;
  const int tr = t0 + rr;
  const bool tvalid = tr < rings;
  const size_t frow = gr.f_off + ((size_t)(tr >> 2) * (size_t)nld + (size_t)(gr.paired ? chain * 4 : chain * 2)) * 4 +
                      (size_t)(tr & 3);
  const size_t sstride = gr.slot_stride;

  // 1. load, pre-multiply by the chirp, zero-pad
  if (DIR == 0) {
    const int total = 1 << (lgr + lgM);
#pragma unroll 4
    for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
      const int r = idx >> lgM, j = idx & (M - 1);
      cplx v = make_double2(0.0, 0.0);
      if (j < n && t0 + r < rings) v = cmul(mypix[(size_t)(t0 + r - gr.ring0) * n + j], chirp[j]);
      s[r * MP + padi(j)] = v;
    }
  } else {
    cplx* srow = s + rr * MP;
#pragma unroll 4
    for (int j = j0; j < M; j += jstep) {
      cplx v = make_double2(0.0, 0.0);
      if (j < n && tvalid) {
        const int m = (j < ell) ? j : j - n;
        size_t base;
        double sg = 1.0;
        if (gr.paired) {
          const int am = m < 0 ? -m : m;
          base = frow + (size_t)am * sstride + (m < 0 ? 8 : 0);
          if (m < 0 && (am & 1)) sg = -1.0;
        } else {
          base = frow + (size_t)(m + ell - 1) * sstride;
        }
        // conj on load: x_p = conj( DFT( conj(F) ) )
        v = cmul(make_double2(sg * F[base], -sg * F[base + 4]), chirp[j]);
      }
      srow[padi(j)] = v;
    }
  }
  __syncthreads();
  // 2. circular convolution with the chirp filter
  fft_forward_head(s, lgr, lgM, MP, tw);
  fft_middle(s, lgr, lgM, MP, bhat);
  fft_inverse_tail(s, lgr, lgM, MP, tw);
  // 3. post-multiply, scale, scatter
  const double sc = gr.scale / (double)M;
  if (DIR == 0) {
    if (tvalid) {
      const cplx* srow = s + rr * MP;
#pragma unroll 2
      for (int k = j0; k < n; k += jstep) {
        cplx v = cmul(srow[padi(k)], chirp[k]);
        v.x *= sc;
        v.y *= sc;
        const int m = (k < ell) ? k : k - n;
        size_t base;
        if (gr.paired) {
          const int am = m < 0 ? -m : m;
          base = frow + (size_t)am * sstride + (m < 0 ? 8 : 0);
          if (m < 0 && (am & 1)) {
            v.x = -v.x;
            v.y = -v.y;
          }
        } else {
          base = frow + (size_t)(m + ell - 1) * sstride;
        }
        F[base] = v.x;
        F[base + 4] = v.y;  // next column in the k4-interleaved layout
      }
    }
  } else {
    const int nr = min(1 << lgr, rings - t0);
    for (int r = 0; r < nr; ++r) {
      const cplx* srow = s + r * MP;
      cplx* prow = mypix + (size_t)(t0 + r - gr.ring0) * n;
#pragma unroll 2
      for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const cplx v = cmul(srow[padi(k)], chirp[k]);
        prow[k] = make_double2(v.x * sc, -v.y * sc);
      }
    }
  }
}


// =============================================================================================
// Two-pass variant for M = R1 x R2 <= 1024 (every ring grid up to L = 256): the whole Bluestein
// convolution crosses shared memory twice instead of six times.
//   pass 1  (thread = one j2, R1 points in registers, inputs straight from global memory):
//           A[k1][j2] = W_M^{j2 k1} sum_{j1} y[j1 R2 + j2] W_R1^{j1 k1}
//   middle  (thread = one k1, R2 points): Y[k2 R1 + k1] = sum_{j2} A[k1][j2] W_R2^{j2 k2};
//           Z = Y * Bhat (natural order);  B[k1][j2] = W_M^{-j2 k1} sum_{k2} Z[k2 R1 + k1] W_R2^{-j2 k2}
//   pass 3  (thread = one j2): z[j1 R2 + j2] = sum_{k1} B[k1][j2] W_R1^{-j1 k1}, straight to global memory
// Rows k1 are padded by one element (conflict-free strided access of the middle pass); the ring
// stride is = 2 (mod 8) elements so that the 4 rings x 2 columns a quarter-warp touches in the
// ring-coefficient gather/scatter phases fall into distinct banks.
// =============================================================================================
// x[k] *= w^k, k < R (two interleaved product chains: <= R/2 roundings deep)
template <int R>
__device__ __forceinline__ void twiddle_powers(cplx* x, cplx w1) {
  const cplx w2 = cmul(w1, w1);
  cplx wo = w1, we = w2;
#pragma unroll
  for (int k = 1; k < R; k += 2) {
    x[k] = cmul(x[k], wo);
    if (k + 1 < R) x[k + 1] = cmul(x[k + 1], we);
    if (k + 2 < R) {
      wo = cmul(wo, w2);
      we = cmul(we, w2);
    }
  }
}

// x[k] *= w^k, k < R, for R = 16 / 32 with a radix-4 power tree: w^(4a+b) = (w^4)^a w^b, every power at most six
// products deep (short dependency chains; the same 30 products as the linear chain at R = 32)
template <int R, bool CONJ>
__device__ __forceinline__ void twiddle_tree(cplx* x, cplx w1) {
  if (CONJ) w1.y = -w1.y;
  const cplx w2 = cmul(w1, w1), w3 = cmul(w2, w1), w4 = cmul(w2, w2);
  x[1] = cmul(x[1], w1);
  x[2] = cmul(x[2], w2);
  x[3] = cmul(x[3], w3);
  cplx b[R / 4];  // (w^4)^a
  b[1] = w4;
#pragma unroll
  for (int a = 2; a < R / 4; ++a) b[a] = (a & 1) ? cmul(b[a - 1], w4) : cmul(b[a / 2], b[a / 2]);
#pragma unroll
  for (int a = 1; a < R / 4; ++a) {
    x[4 * a] = cmul(x[4 * a], b[a]);
    x[4 * a + 1] = cmul(x[4 * a + 1], cmul(b[a], w1));
    x[4 * a + 2] = cmul(x[4 * a + 2], cmul(b[a], w2));
    x[4 * a + 3] = cmul(x[4 * a + 3], cmul(b[a], w3));
  }
}

// table loads (chirp, filter spectrum: L1/L2 hits) run PF elements ahead of their use, so their
// latencies overlap instead of adding up along the in-order instruction stream
template <int N, int PF, class Load, class Use>
__device__ __forceinline__ void prefetched(Load ld, Use use) {
  cplx buf[PF];
#pragma unroll
  for (int i = 0; i < PF && i < N; ++i) buf[i] = ld(i);
#pragma unroll
  for (int i = 0; i < N; ++i) {
    const cplx c = buf[i % PF];
    if (i + PF < N) buf[i % PF] = ld(i + PF);
    use(i, c);
  }
}

__device__ __forceinline__ int ring_stride2(int R1, int R2) {
  int rs = R1 * (R2 + 1);
  return rs + ((2 - (rs & 7)) + 8) % 8;
}

// address of ring coefficient (m(j), ring) in the k4-interleaved array and its sign on the ring side
__device__ __forceinline__ size_t f_address(const PxmFftGroup& gr, size_t frow, int j, double* sg) {
  const int m = (j < gr.ell) ? j : j - gr.n;
  *sg = 1.0;
  if (gr.paired) {
    const int am = m < 0 ? -m : m;
    if (m < 0 && (am & 1)) *sg = -1.0;
    return frow + (size_t)am * gr.slot_stride + (m < 0 ? 8 : 0);
  }
  return frow + (size_t)(m + gr.ell - 1) * gr.slot_stride;
}

template <int DIR, int R1, int R2>
__device__ __forceinline__ void ring_fft2_body(const PxmFftGroup& gr, cplx* __restrict__ s, cplx* __restrict__ mypix,
                                               double* __restrict__ F, int nld, int chain,
                                               const cplx* __restrict__ arena, int t0) {
  constexpr int M = R1 * R2;
  const int n = gr.n, rings = gr.rings;
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const cplx* __restrict__ chirp = arena + gr.chirp_off;
  const cplx* __restrict__ bhat = arena + gr.bhat2_off;
  const cplx* __restrict__ tw = arena + gr.tw_off;
  const size_t col0 = (size_t)(gr.paired ? chain * 4 : chain * 2);

  // ---------------- pass 1: load (x chirp), DFT over j1, twiddle, to shared ----------------
  for (int idx = threadIdx.x; idx < nr * R2; idx += blockDim.x) {
    int r, j2;
    if (DIR == 0) {
      r = idx / R2;
      j2 = idx - r * R2;
    } else {  // 4 rings of one row-group on adjacent lanes: one 32-byte sector per (m, re/im)
      const int rhi = idx / (4 * R2), rem = idx - rhi * 4 * R2;
      r = rhi * 4 + (rem & 3);
      j2 = rem >> 2;
    }
    const int t = t0 + r;
    const bool tvalid = t < rings;
    // all loads of the thread are issued back to back (raw values straight into x[]), the
    // arithmetic on them comes afterwards: one exposed memory latency per thread instead of R1
    cplx x[R1];
    if (DIR == 0) {
      const cplx* row = mypix + (size_t)(t - gr.ring0) * n;
#pragma unroll
      for (int j1 = 0; j1 < R1; ++j1) {
        const int j = j1 * R2 + j2;
        x[j1] = (tvalid && j < n) ? row[j] : make_double2(0.0, 0.0);
      }
      prefetched<R1, 4>([&](int j1) { const int j = j1 * R2 + j2; return chirp[j < n ? j : 0]; },
                        [&](int j1, cplx c) { x[j1] = cmul(x[j1], c); });  // padded entries are 0 anyway
    } else {
      const size_t frow = gr.f_off + ((size_t)(t >> 2) * (size_t)nld + col0) * 4 + (size_t)(t & 3);
#pragma unroll
      for (int j1 = 0; j1 < R1; ++j1) {
        const int j = j1 * R2 + j2;
        cplx v = make_double2(0.0, 0.0);
        if (tvalid && j < n) {
          double sg;
          const size_t base = f_address(gr, frow, j, &sg);
          v = make_double2(F[base], F[base + 4]);
        }
        x[j1] = v;
      }
      prefetched<R1, 4>([&](int j1) { const int j = j1 * R2 + j2; return chirp[j < n ? j : 0]; },
                        [&](int j1, cplx c) {
                          const int j = j1 * R2 + j2;
                          const int m = (j < gr.ell) ? j : j - n;
                          const double sg = (gr.paired && m < 0 && (m & 1)) ? -1.0 : 1.0;
                          x[j1] = cmul(make_double2(sg * x[j1].x, -sg * x[j1].y), c);  // conj on load
                        });
    }
    dftN<R1, false>(x);
    twiddle_powers<R1>(x, tw[j2 * (gr.M / M)]);  // gr.M == M
    cplx* dst = s + r * RS + j2;
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) dst[k1 * (R2 + 1)] = x[k1];
  }
  __syncthreads();
  // ---------------- middle: DFT over j2, filter, inverse DFT over k2, inverse twiddle ----------------
  for (int idx = threadIdx.x; idx < nr * R1; idx += blockDim.x) {
    const int r = idx / R1, k1 = idx - r * R1;
    cplx* row = s + r * RS + k1 * (R2 + 1);
    cplx x[R2];
#pragma unroll
    for (int j2 = 0; j2 < R2; ++j2) x[j2] = row[j2];
    dftN<R2, false>(x);
    prefetched<R2, 4>([&](int k2) { return bhat[k2 * R1 + k1]; }, [&](int k2, cplx b) { x[k2] = cmul(x[k2], b); });
    dftN<R2, true>(x);
    cplx w1 = tw[k1];
    w1.y = -w1.y;
    twiddle_powers<R2>(x, w1);
#pragma unroll
    for (int j2 = 0; j2 < R2; ++j2) row[j2] = x[j2];
  }
  __syncthreads();
  // ---------------- pass 3: inverse DFT over k1, x chirp, scale, store ----------------
  const double sc = gr.scale / (double)M;
  for (int idx = threadIdx.x; idx < nr * R2; idx += blockDim.x) {
    int r, j2;
    if (DIR == 1) {
      r = idx / R2;
      j2 = idx - r * R2;
    } else {
      const int rhi = idx / (4 * R2), rem = idx - rhi * 4 * R2;
      r = rhi * 4 + (rem & 3);
      j2 = rem >> 2;
    }
    const int t = t0 + r;
    if (t >= rings) continue;
    const cplx* src = s + r * RS + j2;
    cplx x[R1];
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) x[k1] = src[k1 * (R2 + 1)];
    dftN<R1, true>(x);
    if (DIR == 0) {
      const size_t frow = gr.f_off + ((size_t)(t >> 2) * (size_t)nld + col0) * 4 + (size_t)(t & 3);
      prefetched<R1, 4>([&](int j1) { const int j = j1 * R2 + j2; return chirp[j < n ? j : 0]; },
                        [&](int j1, cplx c) {
                          const int j = j1 * R2 + j2;
                          if (j < n) {
                            const cplx v = cmul(x[j1], c);
                            double sg;
                            const size_t base = f_address(gr, frow, j, &sg);
                            F[base] = sg * sc * v.x;
                            F[base + 4] = sg * sc * v.y;
                          }
                        });
    } else {
      cplx* row = mypix + (size_t)(t - gr.ring0) * n;
      prefetched<R1, 4>([&](int j1) { const int j = j1 * R2 + j2; return chirp[j < n ? j : 0]; },
                        [&](int j1, cplx c) {
                          const int j = j1 * R2 + j2;
                          if (j < n) {
                            const cplx v = cmul(x[j1], c);
                            row[j] = make_double2(v.x * sc, -v.y * sc);
                          }
                        });
    }
  }
}

// CLS 0: M <= 256 (radices <= 16), CLS 1: M = 512, 1024 (radix 32).  CTAs of groups that belong to
// another class (or to the multi-pass kernel, M > 1024) exit at once.
// The group descriptors travel as a kernel parameter (constant bank): finding a CTA's group and
// reading its descriptor costs no dependent global loads at the head of every CTA.
constexpr int PXM_FFT_MAX_GROUPS = 24;
struct PxmFftGroupTable {
  int ngroups;
  int pad;
  PxmFftGroup g[PXM_FFT_MAX_GROUPS];
};

// radix-32 class: 2 CTAs of 128 threads per SM (255 registers, no spills) measured faster than 3 (168, spills)
#ifndef PXM_FFT2_MINB1
#define PXM_FFT2_MINB1 2
#endif
// CTAs (within one chain) that a launch of one class actually has work for: a launch covers only those instead
// of starting -- and immediately retiring -- the CTAs of every other class (n = 0: identity, all CTAs)
constexpr int PXM_FFT2_MAX_REMAP = 254;
struct Fft2Remap {
  int n;
  unsigned short cta[PXM_FFT2_MAX_REMAP];
};

template <int DIR, int CLS>
__global__ void __launch_bounds__(CLS == 0 ? 256 : 128, CLS == 0 ? 2 : PXM_FFT2_MINB1)
pxm_ring_fft2_kernel(const __grid_constant__ PxmFftGroupTable tab, const __grid_constant__ Fft2Remap remap,
                     cplx* __restrict__ pix, size_t pix_chain_stride, double* __restrict__ F, int nld,
                     const cplx* __restrict__ arena) {
  extern __shared__ __align__(16) unsigned char fsm[];
  cplx* s = reinterpret_cast<cplx*>(fsm);
  const int cta = remap.n ? (int)remap.cta[blockIdx.x] : (int)blockIdx.x;
  int gi = 0;
  while (gi + 1 < tab.ngroups && cta >= tab.g[gi + 1].cta_begin) ++gi;
  const PxmFftGroup& gr = tab.g[gi];
  const int lgM = gr.logM;
  if (CLS == 0 ? (lgM > 8) : (lgM < 9 || lgM > 10)) return;
  const int chain = blockIdx.y;
  const int t0 = gr.ring0 + ((cta - gr.cta_begin) << gr.pad);
  cplx* mypix = pix + (size_t)chain * pix_chain_stride + gr.pix_off;
  if (CLS == 0) {
    switch (lgM) {
      case 4: ring_fft2_body<DIR, 4, 4>(gr, s, mypix, F, nld, chain, arena, t0); break;
      case 5: ring_fft2_body<DIR, 4, 8>(gr, s, mypix, F, nld, chain, arena, t0); break;
      case 6: ring_fft2_body<DIR, 8, 8>(gr, s, mypix, F, nld, chain, arena, t0); break;
      case 7: ring_fft2_body<DIR, 8, 16>(gr, s, mypix, F, nld, chain, arena, t0); break;
      default: ring_fft2_body<DIR, 16, 16>(gr, s, mypix, F, nld, chain, arena, t0); break;
    }
  } else {
    if (lgM == 9)
      ring_fft2_body<DIR, 16, 32>(gr, s, mypix, F, nld, chain, arena, t0);
    else
      ring_fft2_body<DIR, 32, 32>(gr, s, mypix, F, nld, chain, arena, t0);
  }
}


// =============================================================================================
// Persistent, staged variant of the two-pass transform for the radix-32 class (M = 512, 1024):
//   * grid = 2 CTAs per SM; a CTA walks over work items (ring block x chain, chain fastest) of
//     the launch, so the group tables stay hot and no CTA start-up cost is paid per ring block;
//   * the inputs of item i+1 (4 pixel rows = one contiguous 32 KB piece, or the 64/128-byte
//     (m, row-group, chain) pieces of the k4-interleaved ring array) travel global -> shared
//     with cp.async (LDGSTS, no registers) WHILE the middle pass and pass 3 of item i run: the
//     FP64 pipe never waits on DRAM (the non-staged kernel: 27 % of its warp samples);
//   * the zero-padded half of the Bluestein input and the unused half of its output are pruned
//     from the first / last radix-R1 DFT (x_j = 0 for j >= n and only z_j, j < n, is needed;
//     n <= M/2 always): a half-input DFT is two DFTs of half the size.
// Staging of the ring array: piece (slot, row-group) is copied in 16-byte granules to granule
// index G = slot * gpc + g with the XOR swizzle (G & 7) ^ ((G >> 3) & 7) inside every 128-byte
// line, so the quarter-warp reads of pass 1 (4 rings x 2 slots) are bank-conflict free.
// =============================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  const uint32_t addr = smem_u32(bar);
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
// 4-D tiled TMA copy global -> shared (tensor map in kernel-parameter space), completes on `bar`
__device__ __forceinline__ void tma_g2s_4d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                           uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// The ring array of a paired group as a 4-D tensor of doubles:
//   [16: (re, im) x (+m, -m) x 4 rings of a row-group][chain][row-group][order |m|]
// One copy with box (16, 1, 1, ell) and the 128-byte swizzle brings the 128-byte pieces of all orders of one
// (row-group, chain) to shared memory as rows of 128 bytes whose 16-byte chunks are XOR-ed with (row & 7):
// the 8 consecutive orders a warp of pass 1 reads fall on every bank exactly twice (the minimum for
// 64-bit loads).  One instruction per item instead of one 128-byte copy per order.
constexpr int PXM_FFT3_MAX_MAPS = 8;
struct Fft3Maps {
  CUtensorMap m[PXM_FFT3_MAX_MAPS];
};

// table loads of the persistent kernel run this many elements ahead of their use (pass 1 / middle pass)
#ifndef PXM_PF1
#define PXM_PF1 4
#endif
#ifndef PXM_PF2
#define PXM_PF2 4
#endif

struct Fft3Item {
  int gi;     // group
  int t0;     // first ring of the block
  int chain;
};

// ring blocks of the radix-32 class in processing order (longest transforms first), built by the launcher
constexpr int PXM_FFT3_MAX_BLOCKS = 1024;
constexpr int PXM_FFT_MAX_GROUPS_C = 24;  // = PXM_FFT_MAX_GROUPS
struct Fft3Blocks {
  unsigned char gi[PXM_FFT3_MAX_BLOCKS];   // group
  unsigned char blk[PXM_FFT3_MAX_BLOCKS];  // ring block inside the group
  unsigned char map_of_group[PXM_FFT_MAX_GROUPS_C];  // tensor map of a group's ring array
};
// item -> (group, ring block, chain), chain fastest
__device__ __forceinline__ void fft3_find(const PxmFftGroupTable& tab, const Fft3Blocks& blocks, int b, int chain,
                                          Fft3Item* out) {
  out->chain = chain;
  out->gi = blocks.gi[b];
  out->t0 = tab.g[out->gi].ring0 + ((int)blocks.blk[b] << tab.g[out->gi].pad);
}

template <int DIR>
__device__ __forceinline__ void fft3_stage_one(const PxmFftGroup& gr, const Fft3Item& it, unsigned char* stage,
                                               uint64_t* bar, const cplx* __restrict__ pix, size_t pix_chain_stride,
                                               const CUtensorMap* map);
// issue the TMA copies global -> shared of one item's inputs (one thread); they complete on `bar`
template <int DIR>
__device__ __forceinline__ void fft3_stage(const PxmFftGroup& gr, const Fft3Item& it, unsigned char* stage,
                                           uint64_t* bar, const cplx* __restrict__ pix, size_t pix_chain_stride,
                                           const CUtensorMap* map) {
  if (threadIdx.x != 0) return;
  fft3_stage_one<DIR>(gr, it, stage, bar, pix, pix_chain_stride, map);
}
// the same, called by the one thread that issues the copies
template <int DIR>
__device__ __forceinline__ void fft3_stage_one(const PxmFftGroup& gr, const Fft3Item& it, unsigned char* stage,
                                               uint64_t* bar, const cplx* __restrict__ pix, size_t pix_chain_stride,
                                               const CUtensorMap* map) {
  const int nr = 1 << gr.pad;
  if (DIR == 0) {  // the rows of a block are contiguous: one 1-D copy
    const int rows = min(nr, gr.rings - it.t0);
    const uint32_t bytes = (uint32_t)(rows * gr.n) * 16u;
    const cplx* src = pix + (size_t)it.chain * pix_chain_stride + gr.pix_off + (size_t)(it.t0 - gr.ring0) * gr.n;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(stage, src, bytes, bar);
  } else {
    const int ngrp = min((nr + 3) >> 2, (gr.rings - it.t0 + 3) >> 2);
    const int blk_bytes = (gr.ell * 128 + 1023) & ~1023;  // every row-group block keeps the swizzle phase
    mbar_expect_tx(bar, (uint32_t)(ngrp * gr.ell * 128));
    for (int g4 = 0; g4 < ngrp; ++g4) tma_g2s_4d(stage + g4 * blk_bytes, map, 0, it.chain, (it.t0 >> 2) + g4, 0, bar);
  }
}

__device__ __forceinline__ double flip_sign(double x, int mask_hi) {
  return __hiloint2double(__double2hiint(x) ^ mask_hi, __double2loint(x));
}

// chirp_s: this group's chirp times sqrt(scale / M) in shared memory (pass 1 and pass 3 each apply it once)
// NG: item groups per CTA (the threads of a group are blockDim.x / NG consecutive threads; tid: index within the group)
template <int DIR, int R1, int R2, int NG>
__device__ __forceinline__ void ring_fft3_pass1(const PxmFftGroup& gr, const Fft3Item& it, cplx* __restrict__ s,
                                                const unsigned char* __restrict__ stage,
                                                const cplx* __restrict__ chirp_s, const cplx* __restrict__ arena, int tid) {
  constexpr int H1 = R1 / 2;
  const int n = gr.n, rings = gr.rings, ell = gr.ell;
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const cplx* __restrict__ tw2 = arena + gr.tw2_off;  // [k1][j2]
  for (int idx = tid; idx < nr * R2; idx += blockDim.x / NG) {
    // 4 rings of a row-group on adjacent lanes, 8 values of j2 per warp: the chirp / twiddle reads are
    // broadcasts over the rings, the ring-array accesses are 32-byte sectors, the pixel rows 128-byte pieces
    const int rhi = idx / (4 * R2), rem = idx - rhi * 4 * R2;
    const int r = rhi * 4 + (rem & 3), j2 = rem >> 2;
    const int nj = (it.t0 + r < rings) ? n : 0;  // rows past the end of the grid are zeros
    cplx x[R1];
    if (DIR == 0) {
      const cplx* row = reinterpret_cast<const cplx*>(stage) + r * n;
#pragma unroll
      for (int j1 = 0; j1 < H1; ++j1) {
        const int j = j1 * R2 + j2;
        x[j1] = (j < nj) ? cmul(row[j], chirp_s[j]) : make_double2(0.0, 0.0);
      }
    } else {
      const unsigned char* grp = stage + (size_t)(r >> 2) * ((ell * 128 + 1023) & ~1023);
      const int rl = r & 3;
#pragma unroll
      for (int j1 = 0; j1 < H1; ++j1) {
        const int j = j1 * R2 + j2;
        cplx v = make_double2(0.0, 0.0);
        if (j < nj) {
          const bool minus = j >= ell;  // order m = j - n < 0: second half of the 128-byte row
          const int am = minus ? n - j : j;
          const int d = (minus ? 8 : 0) + rl;  // re at double d, im at d + 4 (two chunks further)
          const unsigned char* row = grp + am * 128 + (d & 1) * 8;
          const int sw = am & 7, ch = d >> 1;
          const double re = *reinterpret_cast<const double*>(row + ((ch ^ sw) << 4));
          const double im = *reinterpret_cast<const double*>(row + (((ch + 2) ^ sw) << 4));
          const int neg = (minus && (am & 1)) ? (int)0x80000000 : 0;
          // (-1)^m of the paired layout and the conjugation on load (x_p = conj(DFT(conj F))) are sign-bit flips
          v = cmul(make_double2(flip_sign(re, neg), flip_sign(im, neg ^ (int)0x80000000)), chirp_s[j]);
        }
        x[j1] = v;
      }
    }
#ifndef PXM_ABL_NODFT
    dft_half_in<R1>(x);
#endif
#ifdef PXM_ABL_NOTABLES
    prefetched<R1 - 1, PXM_PF1>([&](int i) { return tw2[0]; }, [&](int i, cplx w) { x[i + 1] = cmul(x[i + 1], w); });
#elif !defined(PXM_FFT3_TWTABLE)
    // W_M^(k1 j2), k1 < R1, from W_M^(j2): one table load instead of R1 - 1 (the loads, not the FP64 pipe, bound
    // the pass: 1.164 -> 1.132 ms per 64-chain step, gpurun_out/r2l_lf.log)
    twiddle_tree<R1, false>(x, tw2[R2 + j2]);
#else
    prefetched<R1 - 1, PXM_PF1>([&](int i) { return tw2[(i + 1) * R2 + j2]; }, [&](int i, cplx w) { x[i + 1] = cmul(x[i + 1], w); });
#endif
    cplx* dst = s + r * RS + j2;
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) dst[k1 * (R2 + 1)] = x[k1];
  }
}

// bhat: the group's filter spectrum in natural order [k2 R1 + k1], in global (two-CTA kernel) or shared memory
template <int R1, int R2, int NG>
__device__ __forceinline__ void ring_fft3_middle(const PxmFftGroup& gr, cplx* __restrict__ s, const cplx* __restrict__ bhat,
                                                 const cplx* __restrict__ arena, int tid) {
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const cplx* __restrict__ tw2t = arena + gr.tw2_off + R1 * R2;  // [j2][k1]
  for (int idx = tid; idx < nr * R1; idx += blockDim.x / NG) {
    // 4 rings on adjacent lanes, 8 values of k1 per warp: the filter-spectrum and twiddle loads are
    // broadcasts over the rings (a quarter of the L1 wavefronts), the row accesses stay conflict free
    const int rhi = idx / (4 * R1), rem = idx - rhi * 4 * R1;
    const int r = rhi * 4 + (rem & 3), k1 = rem >> 2;
    cplx* row = s + r * RS + k1 * (R2 + 1);
    cplx x[R2];
#pragma unroll
    for (int j2 = 0; j2 < R2; ++j2) x[j2] = row[j2];
#ifndef PXM_ABL_NODFT
    dftN<R2, false>(x);
#endif
#if defined(PXM_ABL_NOTABLES) || defined(PXM_ABL_NOBHAT)
    prefetched<R2, PXM_PF2>([&](int k2) { return bhat[0]; }, [&](int k2, cplx b) { x[k2] = cmul(x[k2], b); });
#else
    prefetched<R2, PXM_PF2>([&](int k2) { return bhat[k2 * R1 + k1]; }, [&](int k2, cplx b) { x[k2] = cmul(x[k2], b); });
#endif
#ifndef PXM_ABL_NODFT
    dftN<R2, true>(x);
#endif
#ifdef PXM_ABL_NOTABLES
    prefetched<R2 - 1, PXM_PF2>([&](int i) { return tw2t[0]; }, [&](int i, cplx w) { x[i + 1] = cmulc(x[i + 1], w); });
#elif !defined(PXM_FFT3_TWTABLE)
    twiddle_tree<R2, true>(x, tw2t[R1 + k1]);  // conj W_M^(j2 k1), j2 < R2, from W_M^(k1)
#else
    prefetched<R2 - 1, PXM_PF2>([&](int i) { return tw2t[(i + 1) * R1 + k1]; },
                          [&](int i, cplx w) { x[i + 1] = cmulc(x[i + 1], w); });
#endif
#pragma unroll
    for (int j2 = 0; j2 < R2; ++j2) row[j2] = x[j2];
  }
}

template <int DIR, int R1, int R2, int NG>
__device__ __forceinline__ void ring_fft3_pass3(const PxmFftGroup& gr, const Fft3Item& it, const cplx* __restrict__ s,
                                                const cplx* __restrict__ chirp_s, cplx* __restrict__ pix,
                                                size_t pix_chain_stride, double* __restrict__ F, int nld, int tid) {
  constexpr int H1 = R1 / 2;
  const int n = gr.n, rings = gr.rings, ell = gr.ell;
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const size_t col0 = (size_t)it.chain * 4;  // paired layout only (the launcher checks)
  for (int idx = tid; idx < nr * R2; idx += blockDim.x / NG) {
    // 4 rings of a row-group on adjacent lanes, 8 values of j2 per warp: the chirp / twiddle reads are
    // broadcasts over the rings, the ring-array accesses are 32-byte sectors, the pixel rows 128-byte pieces
    const int rhi = idx / (4 * R2), rem = idx - rhi * 4 * R2;
    const int r = rhi * 4 + (rem & 3), j2 = rem >> 2;
    const int t = it.t0 + r;
    if (t >= rings) continue;
    const cplx* src = s + r * RS + j2;
    cplx x[R1];
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) x[k1] = src[k1 * (R2 + 1)];
#ifndef PXM_ABL_NODFT
    dft_half_out<R1>(x);
#endif
    if (DIR == 0) {
      double* frow = F + gr.f_off + ((size_t)(t >> 2) * (size_t)nld + col0) * 4 + (size_t)(t & 3);
      const size_t ss = gr.slot_stride;
#pragma unroll
      for (int j1 = 0; j1 < H1; ++j1) {
        const int j = j1 * R2 + j2;
        if (j < n) {
          const cplx v = cmul(x[j1], chirp_s[j]);
          const bool minus = j >= ell;
          const int am = minus ? n - j : j;
          double* dst = frow + (size_t)am * ss + (minus ? 8 : 0);
          const int neg = (minus && (am & 1)) ? (int)0x80000000 : 0;
          dst[0] = flip_sign(v.x, neg);
          dst[4] = flip_sign(v.y, neg);  // next column of the k4-interleaved layout
        }
      }
    } else {
      cplx* row = pix + (size_t)it.chain * pix_chain_stride + gr.pix_off + (size_t)(t - gr.ring0) * n;
#pragma unroll
      for (int j1 = 0; j1 < H1; ++j1) {
        const int j = j1 * R2 + j2;
        if (j < n) {
          const cplx v = cmul(x[j1], chirp_s[j]);
          row[j] = make_double2(v.x, flip_sign(v.y, (int)0x80000000));
        }
      }
    }
  }
}

#ifdef PXM_FFT3_TIMING
__device__ unsigned long long g_fft3_clk[16];
#define FFT3_T(i)                                                        \
  do {                                                                   \
    const long long now_ = clock64();                                    \
    if (threadIdx.x == 0) atomicAdd(&g_fft3_clk[DIR * 8 + (i)], (unsigned long long)(now_ - tprev_)); \
    tprev_ = now_;                                                       \
  } while (0)
#else
#define FFT3_T(i)
#endif

constexpr int PXM_FFT3_WORK = 8 * (16 * 33 + 2) * 16;  // >= 4 * (32 * 33 + 2) * 16
constexpr int PXM_FFT3_STAGE = 32768;  // 4 rows x 511 x 16 bytes, or 256 orders x 128 bytes
constexpr int PXM_FFT3_CHIRP = 512 * 16;
constexpr int PXM_FFT3_SMEM = PXM_FFT3_STAGE + PXM_FFT3_WORK + PXM_FFT3_CHIRP + 16;

template <int DIR>
__global__ void __launch_bounds__(128, 2)
pxm_ring_fft3_kernel(const __grid_constant__ PxmFftGroupTable tab, const __grid_constant__ Fft3Blocks blocks,
                     const __grid_constant__ Fft3Maps maps, cplx* __restrict__ pix, size_t pix_chain_stride,
                     double* __restrict__ F, int nld, const cplx* __restrict__ arena, int nchains, long long nitems) {
  extern __shared__ __align__(1024) unsigned char fsm3[];
  unsigned char* stage = fsm3;  // 1024-byte aligned: the TMA swizzle phase is (row & 7)
  cplx* s = reinterpret_cast<cplx*>(fsm3 + PXM_FFT3_STAGE);
  cplx* chirp_s = reinterpret_cast<cplx*>(fsm3 + PXM_FFT3_STAGE + PXM_FFT3_WORK);
  uint64_t* bar = reinterpret_cast<uint64_t*>(fsm3 + PXM_FFT3_STAGE + PXM_FFT3_WORK + PXM_FFT3_CHIRP);
  long long item = blockIdx.x;
  if (item >= nitems) return;
  if (threadIdx.x == 0) {
    if (smem_u32(fsm3) & 1023) __trap();
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t phase = 0;
  Fft3Item cur, nxt;
  // (block, chain) of the item, advanced without divisions
  int ib = (int)(item / nchains), ic = (int)(item - (long long)ib * nchains);
  const int db = (int)gridDim.x / nchains, dc = (int)gridDim.x - db * nchains;
  fft3_find(tab, blocks, ib, ic, &cur);
  nxt = cur;
  fft3_stage<DIR>(tab.g[cur.gi], cur, stage, bar, pix, pix_chain_stride, &maps.m[blocks.map_of_group[cur.gi]]);
#ifdef PXM_FFT3_TIMING
  long long tprev_ = clock64();
#endif
  int chirp_group = -1;
  for (; item < nitems; item += gridDim.x) {
    const PxmFftGroup& gr = tab.g[cur.gi];
    const bool big = gr.logM == 10;
    if (cur.gi != chirp_group) {  // a few times per launch: the blocks of a group are consecutive items
      __syncthreads();            // pass 3 of the previous item has finished with the old chirp
      const cplx* __restrict__ chirp = arena + gr.chirp_off;
      const double rs = sqrt(gr.scale / (double)gr.M);
      for (int j = threadIdx.x; j < gr.n; j += blockDim.x) {
        const cplx c = chirp[j];
        chirp_s[j] = make_double2(c.x * rs, c.y * rs);
      }
      chirp_group = cur.gi;
    }
    __syncthreads();  // pass 3 of the previous item has left the work buffer
    mbar_wait(bar, phase);  // the staged inputs have landed
    phase ^= 1;
    FFT3_T(0);
    if (big)
      ring_fft3_pass1<DIR, 32, 32, 1>(gr, cur, s, stage, chirp_s, arena, threadIdx.x);
    else
      ring_fft3_pass1<DIR, 16, 32, 1>(gr, cur, s, stage, chirp_s, arena, threadIdx.x);
    FFT3_T(1);
    __syncthreads();
    FFT3_T(2);
    if (item + gridDim.x < nitems) {
      ib += db;
      ic += dc;
      if (ic >= nchains) {
        ic -= nchains;
        ++ib;
      }
      fft3_find(tab, blocks, ib, ic, &nxt);
      fft3_stage<DIR>(tab.g[nxt.gi], nxt, stage, bar, pix, pix_chain_stride, &maps.m[blocks.map_of_group[nxt.gi]]);
    }
    FFT3_T(3);
    if (big)
      ring_fft3_middle<32, 32, 1>(gr, s, arena + gr.bhat2_off, arena, threadIdx.x);
    else
      ring_fft3_middle<16, 32, 1>(gr, s, arena + gr.bhat2_off, arena, threadIdx.x);
    FFT3_T(4);
    __syncthreads();
    FFT3_T(5);
    if (big)
      ring_fft3_pass3<DIR, 32, 32, 1>(gr, cur, s, chirp_s, pix, pix_chain_stride, F, nld, threadIdx.x);
    else
      ring_fft3_pass3<DIR, 16, 32, 1>(gr, cur, s, chirp_s, pix, pix_chain_stride, F, nld, threadIdx.x);
    FFT3_T(6);
    cur = nxt;
  }
}

// =============================================================================================
// The persistent staged transform with ONE CTA of 256 threads per SM (pxm_ring_fft6_kernel, what the launcher
// picks for the radix-32 class): two groups of 4 warps, each running exactly the per-item code of
// pxm_ring_fft3_kernel -- its own TMA stage, mbarrier and work buffer, synchronised on its own named barrier --
// with no hand-over between the groups.  Items are dealt in chain pairs: group g takes chain 2k + g of a ring
// block, so both groups always work in the same Bluestein group and the CTA holds ONE copy of the chirp and ONE
// of the filter spectrum, in shared memory.  The middle pass then reads its 32 filter-spectrum values per thread
// and item from shared memory (broadcasts over the 4 rings of a quarter-warp) instead of from L2: next to the
// shared memory of two CTAs of the two-CTA kernel about 28 KB of L1 remained, with a 13 % load hit rate.
// The tables change a few times per launch (the blocks of a group are consecutive items), behind CTA barriers
// that both groups reach in the same iterations: they walk the same sequence of chain pairs.
// =============================================================================================
constexpr int PXM_FFT6_WORK0 = 2 * PXM_FFT3_STAGE;  // the two stages first: 1024-byte aligned for the TMA swizzle
constexpr int PXM_FFT6_CHIRP0 = PXM_FFT6_WORK0 + 2 * PXM_FFT3_WORK;
constexpr int PXM_FFT6_BHAT0 = PXM_FFT6_CHIRP0 + PXM_FFT3_CHIRP;
constexpr int PXM_FFT6_BAR0 = PXM_FFT6_BHAT0 + 1024 * 16;
constexpr int PXM_FFT6_SMEM = PXM_FFT6_BAR0 + 2 * 8;  // 225 808 bytes
static_assert(PXM_FFT6_SMEM <= 232448, "one CTA per SM: the opt-in shared memory of a block");

__device__ __forceinline__ void grp_sync(int g) { asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory"); }

template <int DIR>
__global__ void __launch_bounds__(256, 1)
pxm_ring_fft6_kernel(const __grid_constant__ PxmFftGroupTable tab, const __grid_constant__ Fft3Blocks blocks,
                     const __grid_constant__ Fft3Maps maps, cplx* __restrict__ pix, size_t pix_chain_stride,
                     double* __restrict__ F, int nld, const cplx* __restrict__ arena, int nchains, long long npairs) {
  extern __shared__ __align__(1024) unsigned char fsm6[];
  const int g = threadIdx.x >> 7, tid = threadIdx.x & 127;  // 256 threads: two groups of 128
  unsigned char* stage = fsm6 + g * PXM_FFT3_STAGE;
  cplx* s = reinterpret_cast<cplx*>(fsm6 + PXM_FFT6_WORK0 + g * PXM_FFT3_WORK);
  cplx* chirp_s = reinterpret_cast<cplx*>(fsm6 + PXM_FFT6_CHIRP0);
  cplx* bhat_s = reinterpret_cast<cplx*>(fsm6 + PXM_FFT6_BHAT0);
  uint64_t* bar = reinterpret_cast<uint64_t*>(fsm6 + PXM_FFT6_BAR0) + g;
  long long pair = blockIdx.x;
  if (pair >= npairs) return;
  if (tid == 0) {
    if (smem_u32(fsm6) & 1023) __trap();
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  // (block, chain pair) of the pair, advanced without divisions; with an odd chain count the last pair of a
  // block has no chain for group 1, which then skips the item
  const int npc = (nchains + 1) >> 1;
  int ib = (int)(pair / npc), ik = (int)(pair - (long long)ib * npc);
  const int db = (int)gridDim.x / npc, dk = (int)gridDim.x - db * npc;
  uint32_t phase = 0;
  Fft3Item cur, nxt;
  fft3_find(tab, blocks, ib, 2 * ik + g, &cur);
  bool have = cur.chain < nchains;
  if (have && tid == 0)
    fft3_stage_one<DIR>(tab.g[cur.gi], cur, stage, bar, pix, pix_chain_stride, &maps.m[blocks.map_of_group[cur.gi]]);
  nxt = cur;
  int table_group = -1;
  for (; pair < npairs; pair += gridDim.x) {
    const PxmFftGroup& gr = tab.g[cur.gi];
    const bool big = gr.logM == 10;
    if (cur.gi != table_group) {
      __syncthreads();  // both groups have finished with the old chirp (pass 3) and filter spectrum (middle pass)
      const cplx* __restrict__ chirp = arena + gr.chirp_off;
      const double rs = sqrt(gr.scale / (double)gr.M);
      for (int j = threadIdx.x; j < gr.n; j += blockDim.x) {
        const cplx c = chirp[j];
        chirp_s[j] = make_double2(c.x * rs, c.y * rs);
      }
#ifndef PXM_ABL_FFT6_GLOBAL_BHAT
      const cplx* __restrict__ bhat = arena + gr.bhat2_off;
      for (int k = threadIdx.x; k < gr.M; k += blockDim.x) bhat_s[k] = bhat[k];
#endif
      table_group = cur.gi;
      __syncthreads();
    }
#ifdef PXM_ABL_FFT6_GLOBAL_BHAT
    const cplx* bh = arena + gr.bhat2_off;
#else
    const cplx* bh = bhat_s;
#endif
    if (have) {
      grp_sync(g);            // pass 3 of the group's previous item has left the work buffer
      mbar_wait(bar, phase);  // the staged inputs have landed
      phase ^= 1;
      if (big)
        ring_fft3_pass1<DIR, 32, 32, 2>(gr, cur, s, stage, chirp_s, arena, tid);
      else
        ring_fft3_pass1<DIR, 16, 32, 2>(gr, cur, s, stage, chirp_s, arena, tid);
      grp_sync(g);
    }
    bool have_next = false;
    if (pair + gridDim.x < npairs) {
      ib += db;
      ik += dk;
      if (ik >= npc) {
        ik -= npc;
        ++ib;
      }
      fft3_find(tab, blocks, ib, 2 * ik + g, &nxt);
      have_next = nxt.chain < nchains;
      if (have_next && tid == 0)  // the stage is free: pass 1 has read it, or the group had no item
        fft3_stage_one<DIR>(tab.g[nxt.gi], nxt, stage, bar, pix, pix_chain_stride, &maps.m[blocks.map_of_group[nxt.gi]]);
    }
    if (have) {
      if (big)
        ring_fft3_middle<32, 32, 2>(gr, s, bh, arena, tid);
      else
        ring_fft3_middle<16, 32, 2>(gr, s, bh, arena, tid);
      grp_sync(g);
      if (big)
        ring_fft3_pass3<DIR, 32, 32, 2>(gr, cur, s, chirp_s, pix, pix_chain_stride, F, nld, tid);
      else
        ring_fft3_pass3<DIR, 16, 32, 2>(gr, cur, s, chirp_s, pix, pix_chain_stride, F, nld, tid);
    }
    cur = nxt;
    have = have_next;
  }
}

#ifdef PXM_FFT_PAIRSPLIT
// =============================================================================================
// DEVELOPMENT VARIANT, compiled only with -DPXM_FFT_PAIRSPLIT (correct -- it passes the ring-FFT parity tests -- but measured
// SLOWER: 1.57 vs 1.14 ms per 64-chain step; profiles/fft5_r2_metrics.txt: +49 % instructions from selects, shuffles, doubled
// twiddle generation and index arithmetic; FP64 pipe 48 % at 16 warps per SM).
// Pair-split variant of the persistent staged transform (pxm_ring_fft5_kernel): the same items, staging,
// work-buffer layout and three passes as pxm_ring_fft3_kernel, but every 32-point column / row DFT is shared
// by a PAIR of threads (adjacent lanes l and l ^ 4) that hold 16 points each and swap halves with warp
// shuffles.  Half the registers per thread (<= 128) => 256-thread CTAs, 2 per SM = 16 warps per SM instead
// of 8: the round-2 ablations showed the two-CTA kernel bound by exposed latency at 2 warps per scheduler,
// not by FP64 issue or shared-memory bandwidth (DESIGN.md 3).
//   pass 1  (pruned forward DFT over j1, inputs j1 >= R1/2 are zero):  thread h of a pair computes
//           X[2q + h] = DFT_{R1/2}(x_j W_R1^{h j})[q]  -- the same code for both threads, the input twiddle
//           selected by h; no exchange.
//   middle  (row DFT over j2, x filter, inverse DFT):  thread h transforms the inputs j2 = 2i + h (radix-2
//           decimation in time), the pair swaps 8 values and each finishes 8 of the 16 butterflies
//           (k = i + 8h: the extra twiddle W_32^{8h} = (-i)^h is a predicated rotation); the inverse runs the
//           mirror image (decimation in frequency, one swap) and leaves thread h with the outputs j2 = 2q + h.
//   pass 3  (pruned inverse DFT over k1, only outputs j1 < R1/2 needed): thread h transforms the inputs
//           k1 = 2q + h, one swap, thread h finishes the outputs j1 = i + (R1/4) h.
// Lane layout: lane = 8 (column & 3) + 4 h + (ring & 3): the 4 rings of a row-group stay on adjacent lanes
// (32-byte sectors of the k4-interleaved ring array), partners are 4 lanes apart, and every shared-memory
// access of a quarter-warp (4 rings x 2 halves) falls on 32 distinct banks.
// =============================================================================================
__device__ __forceinline__ cplx shfl_pair(cplx v) {
  return make_double2(__shfl_xor_sync(0xffffffffu, v.x, 4), __shfl_xor_sync(0xffffffffu, v.y, 4));
}
__device__ __forceinline__ cplx csel(bool p, cplx a, cplx b) { return make_double2(p ? a.x : b.x, p ? a.y : b.y); }

// x[q] *= f * w^q, q < N, where f is a per-thread factor and w a per-thread base (radix-4 power tree)
template <int N>
__device__ __forceinline__ void twiddle_tree_f(cplx* x, cplx f, cplx w) {
  const cplx w2 = cmul(w, w), w3 = cmul(w2, w), w4 = cmul(w2, w2);
  cplx b = f;  // f (w^4)^a
#pragma unroll
  for (int a = 0; a < N / 4; ++a) {
    x[4 * a] = cmul(x[4 * a], b);
    x[4 * a + 1] = cmul(x[4 * a + 1], cmul(b, w));
    x[4 * a + 2] = cmul(x[4 * a + 2], cmul(b, w2));
    x[4 * a + 3] = cmul(x[4 * a + 3], cmul(b, w3));
    if (a + 1 < N / 4) b = cmul(b, w4);
  }
}

template <int DIR, int R1, int R2>
__device__ __forceinline__ void ring_fft5_pass1(const PxmFftGroup& gr, const Fft3Item& it, cplx* __restrict__ s,
                                                const unsigned char* __restrict__ stage,
                                                const cplx* __restrict__ chirp_s, const cplx* __restrict__ arena) {
  constexpr int H1 = R1 / 2;       // nonzero inputs = outputs per thread
  constexpr int STEP = 32 / R1;    // W_R1 = W_32^STEP
  const int n = gr.n, rings = gr.rings, ell = gr.ell;
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const cplx* __restrict__ tw2 = arena + gr.tw2_off;  // [k1][j2]
  for (int idx = threadIdx.x; idx < nr * R2 * 2; idx += blockDim.x) {
    const int h = (idx >> 2) & 1, j2 = (idx >> 3) & (R2 - 1);
    const int r = ((idx >> 8) << 2) | (idx & 3);
    const int nj = (it.t0 + r < rings) ? n : 0;  // rows past the end of the grid are zeros
    cplx x[H1];
    if (DIR == 0) {
      const cplx* row = reinterpret_cast<const cplx*>(stage) + r * n;
#pragma unroll
      for (int j1 = 0; j1 < H1; ++j1) {
        const int j = j1 * R2 + j2;
        x[j1] = (j < nj) ? cmul(row[j], chirp_s[j]) : make_double2(0.0, 0.0);
      }
    } else {
      const unsigned char* grp = stage + (size_t)(r >> 2) * ((ell * 128 + 1023) & ~1023);
      const int rl = r & 3;
#pragma unroll
      for (int j1 = 0; j1 < H1; ++j1) {
        const int j = j1 * R2 + j2;
        cplx v = make_double2(0.0, 0.0);
        if (j < nj) {
          const bool minus = j >= ell;  // order m = j - n < 0: second half of the 128-byte row
          const int am = minus ? n - j : j;
          const int d = (minus ? 8 : 0) + rl;  // re at double d, im at d + 4 (two chunks further)
          const unsigned char* row = grp + am * 128 + (d & 1) * 8;
          const int sw = am & 7, ch = d >> 1;
          const double re = *reinterpret_cast<const double*>(row + ((ch ^ sw) << 4));
          const double im = *reinterpret_cast<const double*>(row + (((ch + 2) ^ sw) << 4));
          const int neg = (minus && (am & 1)) ? (int)0x80000000 : 0;
          v = cmul(make_double2(flip_sign(re, neg), flip_sign(im, neg ^ (int)0x80000000)), chirp_s[j]);
        }
        x[j1] = v;
      }
    }
    // input twiddle W_R1^{h j1}: identity for h = 0 (same instructions for both halves, constants by select)
#pragma unroll
    for (int j1 = 1; j1 < H1; ++j1) {
      double c, sn;
      w32(j1 * STEP, &c, &sn);
      x[j1] = twc<false>(x[j1], h ? c : 1.0, h ? sn : 0.0);
    }
    dftR<H1, false>(x);  // x[q] = X[2q + h]
    // inter-pass twiddle W_M^{(2q + h) j2} = (W^{j2})^h (W^{2 j2})^q
    {
      const cplx w1 = tw2[R2 + j2];
      const cplx f = h ? w1 : make_double2(1.0, 0.0);
      twiddle_tree_f<H1>(x, f, cmul(w1, w1));
    }
    cplx* dst = s + r * RS + j2 + h * (R2 + 1);
#pragma unroll
    for (int q = 0; q < H1; ++q) dst[2 * q * (R2 + 1)] = x[q];
  }
}

// middle pass, R2 = 32: 16 points per thread
template <int R1>
__device__ __forceinline__ void ring_fft5_middle(const PxmFftGroup& gr, cplx* __restrict__ s,
                                                 const cplx* __restrict__ arena) {
  constexpr int R2 = 32;
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const cplx* __restrict__ bhat = arena + gr.bhat2_off;
  const cplx* __restrict__ tw2t = arena + gr.tw2_off + R1 * R2;  // [j2][k1]
  for (int idx = threadIdx.x; idx < nr * R1 * 2; idx += blockDim.x) {
    const bool h = (idx >> 2) & 1;
    // columns k1: 3 + log2(R1) bits above the ring / half bits; R1 * 8 thread slots per group of 4 rings
    const int k1 = (idx >> 3) & (R1 - 1);
    const int r = ((idx / (8 * R1)) << 2) | (idx & 3);
    cplx* row = s + r * RS + k1 * (R2 + 1) + (h ? 1 : 0);
    cplx y[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) y[i] = row[2 * i];
    dft16<false>(y);  // h = 0: E[k], h = 1: O[k]
    cplx p[8], q[8];
    // swap: thread 0 keeps E[0..7] and receives O[0..7]; thread 1 keeps O[8..15] and receives E[8..15]
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const cplx got = shfl_pair(csel(h, y[i], y[8 + i]));
      p[i] = csel(h, got, y[i]);        // E[k], k = i + 8 h
      q[i] = csel(h, y[8 + i], got);    // O[k]
      if (h) q[i] = rot90<false>(q[i]); // W_32^{8} = -i
    }
    // X[k] = E[k] + W_32^k O[k], X[k + 16] = E[k] - W_32^k O[k]; times the filter spectrum
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      double c, sn;
      w32(i, &c, &sn);
      bfly_tw<false>(p[i], q[i], c, sn);
    }
    {
      const int k0 = h ? 8 : 0;
      prefetched<8, PXM_PF2>([&](int i) { return bhat[(k0 + i) * R1 + k1]; }, [&](int i, cplx b) { p[i] = cmul(p[i], b); });
      prefetched<8, PXM_PF2>([&](int i) { return bhat[(k0 + i + 16) * R1 + k1]; }, [&](int i, cplx b) { q[i] = cmul(q[i], b); });
    }
    // inverse, decimation in frequency: u[k] = X[k] + X[k+16], v[k] = (X[k] - X[k+16]) W_32^{-k}
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const cplx u = cadd(p[i], q[i]);
      cplx d = csub(p[i], q[i]);
      if (h) d = rot90<true>(d);  // W_32^{-8} = +i
      double c, sn;
      w32(i, &c, &sn);
      p[i] = u;
      q[i] = (i == 0) ? d : twc<true>(d, c, sn);
    }
    // swap: thread 0 collects u[0..15] (even outputs), thread 1 collects v[0..15] (odd outputs)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const cplx got = shfl_pair(csel(h, p[i], q[i]));  // thread 1 sends u[8 + i], thread 0 sends v[i]
      y[i] = csel(h, got, p[i]);
      y[8 + i] = csel(h, q[i], got);
    }
    dft16<true>(y);  // y[qq] = x[2 qq + h]
    // inverse inter-pass twiddle conj(W_M^{(2qq + h) k1})
    {
      cplx w1 = tw2t[R1 + k1];
      w1.y = -w1.y;
      const cplx f = h ? w1 : make_double2(1.0, 0.0);
      twiddle_tree_f<16>(y, f, cmul(w1, w1));
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) row[2 * i] = y[i];
  }
}

template <int DIR, int R1, int R2>
__device__ __forceinline__ void ring_fft5_pass3(const PxmFftGroup& gr, const Fft3Item& it, const cplx* __restrict__ s,
                                                const cplx* __restrict__ chirp_s, cplx* __restrict__ pix,
                                                size_t pix_chain_stride, double* __restrict__ F, int nld) {
  constexpr int H1 = R1 / 2;     // inputs per thread
  constexpr int Q1 = R1 / 4;     // outputs per thread
  constexpr int STEP = 32 / R1;
  const int n = gr.n, rings = gr.rings, ell = gr.ell;
  const int nr = 1 << gr.pad;
  const int RS = ring_stride2(R1, R2);
  const size_t col0 = (size_t)it.chain * 4;  // paired layout only (the launcher checks)
  for (int idx = threadIdx.x; idx < nr * R2 * 2; idx += blockDim.x) {
    const bool h = (idx >> 2) & 1;
    const int j2 = (idx >> 3) & (R2 - 1);
    const int r = ((idx >> 8) << 2) | (idx & 3);
    const int t = it.t0 + r;
    const cplx* src = s + r * RS + j2 + (h ? (R2 + 1) : 0);
    cplx x[H1];
#pragma unroll
    for (int q = 0; q < H1; ++q) x[q] = src[2 * q * (R2 + 1)];
    dftR<H1, true>(x);  // h = 0: E[j], h = 1: O[j], j < R1/2
    // z[j] = E[j] + W_R1^{-j} O[j], j < R1/2: thread h finishes j = i + (R1/4) h; W_R1^{-R1/4} = +i
    cplx z[Q1];
#pragma unroll
    for (int i = 0; i < Q1; ++i) {
      const cplx got = shfl_pair(csel(h, x[i], x[Q1 + i]));  // thread 1 sends O[i], thread 0 sends E[Q1 + i]
      const cplx e = csel(h, got, x[i]);
      cplx o = csel(h, x[Q1 + i], got);
      if (h) o = rot90<true>(o);
      double c, sn;
      w32(i * STEP, &c, &sn);
      z[i] = add_tw<true>(e, o, c, sn);
    }
    if (t >= rings) continue;
    const int j1base = h ? Q1 : 0;
    if (DIR == 0) {
      double* frow = F + gr.f_off + ((size_t)(t >> 2) * (size_t)nld + col0) * 4 + (size_t)(t & 3);
      const size_t ss = gr.slot_stride;
#pragma unroll
      for (int i = 0; i < Q1; ++i) {
        const int j = (j1base + i) * R2 + j2;
        if (j < n) {
          const cplx v = cmul(z[i], chirp_s[j]);
          const bool minus = j >= ell;
          const int am = minus ? n - j : j;
          double* dst = frow + (size_t)am * ss + (minus ? 8 : 0);
          const int neg = (minus && (am & 1)) ? (int)0x80000000 : 0;
          dst[0] = flip_sign(v.x, neg);
          dst[4] = flip_sign(v.y, neg);  // next column of the k4-interleaved layout
        }
      }
    } else {
      cplx* row = pix + (size_t)it.chain * pix_chain_stride + gr.pix_off + (size_t)(t - gr.ring0) * n;
#pragma unroll
      for (int i = 0; i < Q1; ++i) {
        const int j = (j1base + i) * R2 + j2;
        if (j < n) {
          const cplx v = cmul(z[i], chirp_s[j]);
          row[j] = make_double2(v.x, flip_sign(v.y, (int)0x80000000));
        }
      }
    }
  }
}

template <int DIR>
__global__ void __launch_bounds__(256, 2)
pxm_ring_fft5_kernel(const __grid_constant__ PxmFftGroupTable tab, const __grid_constant__ Fft3Blocks blocks,
                     const __grid_constant__ Fft3Maps maps, cplx* __restrict__ pix, size_t pix_chain_stride,
                     double* __restrict__ F, int nld, const cplx* __restrict__ arena, int nchains, long long nitems) {
  extern __shared__ __align__(1024) unsigned char fsm5[];
  unsigned char* stage = fsm5;  // 1024-byte aligned: the TMA swizzle phase is (row & 7)
  cplx* s = reinterpret_cast<cplx*>(fsm5 + PXM_FFT3_STAGE);
  cplx* chirp_s = reinterpret_cast<cplx*>(fsm5 + PXM_FFT3_STAGE + PXM_FFT3_WORK);
  uint64_t* bar = reinterpret_cast<uint64_t*>(fsm5 + PXM_FFT3_STAGE + PXM_FFT3_WORK + PXM_FFT3_CHIRP);
  long long item = blockIdx.x;
  if (item >= nitems) return;
  if (threadIdx.x == 0) {
    if (smem_u32(fsm5) & 1023) __trap();
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  uint32_t phase = 0;
  Fft3Item cur, nxt;
  int ib = (int)(item / nchains), ic = (int)(item - (long long)ib * nchains);
  const int db = (int)gridDim.x / nchains, dc = (int)gridDim.x - db * nchains;
  fft3_find(tab, blocks, ib, ic, &cur);
  nxt = cur;
  fft3_stage<DIR>(tab.g[cur.gi], cur, stage, bar, pix, pix_chain_stride, &maps.m[blocks.map_of_group[cur.gi]]);
  int chirp_group = -1;
  for (; item < nitems; item += gridDim.x) {
    const PxmFftGroup& gr = tab.g[cur.gi];
    const bool big = gr.logM == 10;
    if (cur.gi != chirp_group) {  // a few times per launch: the blocks of a group are consecutive items
      __syncthreads();            // pass 3 of the previous item has finished with the old chirp
      const cplx* __restrict__ chirp = arena + gr.chirp_off;
      const double rs = sqrt(gr.scale / (double)gr.M);
      for (int j = threadIdx.x; j < gr.n; j += blockDim.x) {
        const cplx c = chirp[j];
        chirp_s[j] = make_double2(c.x * rs, c.y * rs);
      }
      chirp_group = cur.gi;
    }
    __syncthreads();        // pass 3 of the previous item has left the work buffer
    mbar_wait(bar, phase);  // the staged inputs have landed
    phase ^= 1;
    if (big)
      ring_fft5_pass1<DIR, 32, 32>(gr, cur, s, stage, chirp_s, arena);
    else
      ring_fft5_pass1<DIR, 16, 32>(gr, cur, s, stage, chirp_s, arena);
    __syncthreads();
    if (item + gridDim.x < nitems) {
      ib += db;
      ic += dc;
      if (ic >= nchains) {
        ic -= nchains;
        ++ib;
      }
      fft3_find(tab, blocks, ib, ic, &nxt);
      fft3_stage<DIR>(tab.g[nxt.gi], nxt, stage, bar, pix, pix_chain_stride, &maps.m[blocks.map_of_group[nxt.gi]]);
    }
    if (big)
      ring_fft5_middle<32>(gr, s, arena);
    else
      ring_fft5_middle<16>(gr, s, arena);
    __syncthreads();
    if (big)
      ring_fft5_pass3<DIR, 32, 32>(gr, cur, s, chirp_s, pix, pix_chain_stride, F, nld);
    else
      ring_fft5_pass3<DIR, 16, 32>(gr, cur, s, chirp_s, pix, pix_chain_stride, F, nld);
    cur = nxt;
  }
}

#endif  // PXM_FFT_PAIRSPLIT


constexpr int PXM_FFT2_SMEM = (16 * (16 * 17 + 2)) * 16 > (4 * (32 * 33 + 2)) * 16 ? (16 * (16 * 17 + 2)) * 16
                                                                                  : (4 * (32 * 33 + 2)) * 16;

}  // namespace

// tensor map of one paired ring array (see Fft3Maps), cached per (address, layout)
static bool fft3_tensor_map(const double* base, int nld, unsigned long long slot_stride, int ell, CUtensorMap* out) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static std::mutex mu;
  static EncodeFn encode = nullptr;
  static bool tried = false;
  static std::map<std::tuple<const double*, int, unsigned long long, int>, CUtensorMap> cache;
  std::lock_guard<std::mutex> lock(mu);
  if (!tried) {
    tried = true;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      encode = (EncodeFn)fn;
  }
  if (!encode || ell > 256) return false;
  const auto key = std::make_tuple(base, nld, slot_stride, ell);
  auto it = cache.find(key);
  if (it == cache.end()) {
    CUtensorMap m;
    const cuuint64_t dims[4] = {16, (cuuint64_t)(nld / 4), (cuuint64_t)(slot_stride / (4ULL * nld)), (cuuint64_t)ell};
    const cuuint64_t strides[3] = {128, (cuuint64_t)nld * 32, (cuuint64_t)slot_stride * 8};  // bytes, dims 1..3
    const cuuint32_t box[4] = {16, 1, 1, (cuuint32_t)ell};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (encode(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return false;
    if (cache.size() > 4096) cache.clear();
    it = cache.emplace(key, m).first;
  }
  *out = it->second;
  return true;
}

int pxm_fft_choose_M(int n, int* logM) {
  int M = 16, lg = 4;
  while (M < 2 * n - 1) {
    M <<= 1;
    ++lg;
  }
  *logM = lg;
  return M;
}

// log2 of the rings one CTA transforms (4096 points per CTA, at most 16 rings)
int pxm_fft_rings_per_cta_log(int M) {
  int lg = 0;
  while ((M << (lg + 1)) <= 4096 && lg < 4) ++lg;
  return lg;
}

static int g_fft_legacy = 0;
static int g_fft_pair = 0;      // persistent class: the pair-split kernel (16 points per thread, 16 warps per SM)
static int g_fft_two_cta = 0;  // persistent class: the two-CTA kernel pxm_ring_fft3_kernel instead of pxm_ring_fft6_kernel
constexpr int PXM_FFT_SMEM = (4096 + 256 + 32) * 16;  // up to 4096 complex points (+1/16 padding) per CTA

int pxm_fft_setup_tables(const PxmFftGroup* d_groups, const PxmFftGroup* h_groups, int ngroups, void* d_arena,
                         cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    PXM_CUDA(cudaFuncSetAttribute(fft_fill_bhat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft2_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT2_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft2_kernel<0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT2_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft2_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT2_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft2_kernel<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT2_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft3_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT3_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft3_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT3_SMEM));
#ifdef PXM_FFT_PAIRSPLIT
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft5_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT3_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft5_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT3_SMEM));
#endif
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft6_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT6_SMEM));
    PXM_CUDA(cudaFuncSetAttribute(pxm_ring_fft6_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PXM_FFT6_SMEM));
    configured = true;
  }
  if (ngroups <= 0) return PXM_OK;  // a rank of an m-sharded plan that owns no ring
  for (int i = 0; i < ngroups; ++i) {
    if (h_groups[i].M > 4096) {
      pxm_set_error("ring FFT: bandlimit too large (Bluestein length > 4096, i.e. L > 1024)");
      return PXM_ERR_UNSUPPORTED;
    }
  }
  fft_fill_tables_kernel<<<ngroups, 256, 0, stream>>>(d_groups, ngroups, (cplx*)d_arena);
  PXM_LAUNCHED();
  fft_fill_bhat_kernel<<<ngroups, 256, PXM_FFT_SMEM, stream>>>(d_groups, ngroups, (cplx*)d_arena);
  PXM_LAUNCHED();
  fft_fill_bhat2_kernel<<<dim3(8, ngroups), 128, 0, stream>>>(d_groups, ngroups, (cplx*)d_arena);
  PXM_LAUNCHED();
  return PXM_OK;
}

// class of a Bluestein length: bit 0: M <= 256, bit 1: M = 512 / 1024 (two-pass kernels), bit 2: M > 1024
int pxm_fft_class_bit(int logM) { return logM <= 8 ? 1 : (logM <= 10 ? 2 : 4); }

// dir 0: pix -> F ; dir 1: F -> pix.  class_mask: which kernel classes the stage's groups need
int pxm_fft_launch(int dir, const PxmFftGroup* d_groups, const PxmFftGroup* h_groups, int ngroups, int ctas_per_chain,
                   void* pix, size_t pix_chain_stride, double* F, int nld, const void* d_arena, int nchains,
                   int class_mask, cudaStream_t stream) {
  if (nchains <= 0 || ctas_per_chain <= 0) return PXM_OK;
  dim3 grid(ctas_per_chain, nchains);
  cplx* px = (cplx*)pix;
  const cplx* ar = (const cplx*)d_arena;
  PxmFftGroupTable tab;
  tab.ngroups = ngroups;
  tab.pad = 0;
  if (ngroups <= PXM_FFT_MAX_GROUPS)
    for (int i = 0; i < ngroups; ++i) tab.g[i] = h_groups[i];
  // Few CTAs (single chain, m-sharded ranks): the launch is one wave whose duration is the latency of a
  // single CTA, and the multi-pass kernel spreads a ring over twice as many threads -> measured faster
  // there (L=256: 1 chain 0.099 vs 0.115 ms of ring FFT per iteration, 2 chains equal, 4 chains 0.187 vs 0.157:
  // gpurun_out/fft_dev_small.log); the persistent two-pass kernel wins on throughput.
  // (grids whose rings are all short, M <= 256, stay on the two-pass kernel: radices <= 16, fewer barriers)
  const bool small_grid = (long long)ctas_per_chain * nchains < 700 && (class_mask & 6) != 0;
  if (g_fft_legacy == 1 || (small_grid && g_fft_legacy == 0) || ngroups > PXM_FFT_MAX_GROUPS) {
    if (dir == 0)
      pxm_ring_fft_kernel<0><<<grid, 256, PXM_FFT_SMEM, stream>>>(d_groups, ngroups, px, pix_chain_stride, F, nld, ar, 0);
    else
      pxm_ring_fft_kernel<1><<<grid, 256, PXM_FFT_SMEM, stream>>>(d_groups, ngroups, px, pix_chain_stride, F, nld, ar, 0);
    PXM_LAUNCHED();
    return PXM_OK;
  }
  // CTA lists of the two-pass classes (class 0: M <= 256, class 1: M = 512 / 1024)
  Fft2Remap remap[2];
  for (int c = 0; c < 2; ++c) {
    remap[c].n = 0;
    bool fits = true;
    for (int i = 0; i < ngroups && fits; ++i) {
      const bool mine = c == 0 ? h_groups[i].logM <= 8 : (h_groups[i].logM == 9 || h_groups[i].logM == 10);
      if (!mine) continue;
      const int end = (i + 1 < ngroups) ? h_groups[i + 1].cta_begin : ctas_per_chain;
      for (int b = h_groups[i].cta_begin; b < end; ++b) {
        if (remap[c].n >= PXM_FFT2_MAX_REMAP || b > 65535) {
          fits = false;
          break;
        }
        remap[c].cta[remap[c].n++] = (unsigned short)b;
      }
    }
    if (!fits) remap[c].n = 0;  // identity: every CTA of the chain is started
  }
  const dim3 grid0(remap[0].n ? remap[0].n : ctas_per_chain, nchains), grid1(remap[1].n ? remap[1].n : ctas_per_chain, nchains);
  if (class_mask & 2) {
    // persistent staged kernel unless the two-pass one is forced or the ring array is not 16-byte granular
    Fft3Blocks blocks;
    Fft3Maps maps;
    int nmaps = 0;
    long long n1 = 0;
    bool ok3 = g_fft_legacy != 2 && (((uintptr_t)F) & 15) == 0 && (nld & 3) == 0;
    for (int lg = 10; lg >= 9 && ok3; --lg)
      for (int i = 0; i < ngroups && ok3; ++i) {
        const PxmFftGroup& g = h_groups[i];
        if (g.logM != lg) continue;
        const int end = (i + 1 < ngroups) ? h_groups[i + 1].cta_begin : ctas_per_chain;
        const int nb = end - g.cta_begin;
        // paired (+m, -m) layout only; TMA needs 16-byte granularity; the block and map tables have fixed sizes
        if (!g.paired || g.nslots != g.ell || (g.f_off & 1) || (g.slot_stride % (4ULL * nld)) != 0 ||
            n1 + nb > PXM_FFT3_MAX_BLOCKS || nb > 256 || nmaps >= PXM_FFT3_MAX_MAPS) {
          ok3 = false;
          break;
        }
        if (dir == 1 && !fft3_tensor_map(F + g.f_off, nld, g.slot_stride, g.ell, &maps.m[nmaps])) {
          ok3 = false;
          break;
        }
        blocks.map_of_group[i] = (unsigned char)nmaps++;
        for (int b = 0; b < nb; ++b) {
          blocks.gi[n1] = (unsigned char)i;
          blocks.blk[n1] = (unsigned char)b;
          ++n1;
        }
      }
    if (ok3) {
      static int nsm = 0;
      if (nsm == 0) {
        int devi = 0;
        PXM_CUDA(cudaGetDevice(&devi));
        PXM_CUDA(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, devi));
      }
      const long long nitems = n1 * nchains;
#ifdef PXM_FFT3_TIMING
      const int per_sm = getenv("PXM_FFT3_CTAS_PER_SM") ? atoi(getenv("PXM_FFT3_CTAS_PER_SM")) : 2;
      const int g3 = (int)std::min<long long>(nitems, (long long)per_sm * nsm);
#else
      const int g3 = (int)std::min<long long>(nitems, 2LL * nsm);  // 2 CTAs per SM (shared memory, 252 registers)
#endif
#ifdef PXM_FFT_PAIRSPLIT
      if (g_fft_pair) {
        // pair-split kernel: 256-thread CTAs, 16 points per thread, 2 CTAs per SM = 16 warps per SM
        if (dir == 0)
          pxm_ring_fft5_kernel<0><<<g3, 256, PXM_FFT3_SMEM, stream>>>(tab, blocks, maps, px, pix_chain_stride, F, nld, ar, nchains,
                                                                    nitems);
        else
          pxm_ring_fft5_kernel<1><<<g3, 256, PXM_FFT3_SMEM, stream>>>(tab, blocks, maps, px, pix_chain_stride, F, nld, ar, nchains,
                                                                    nitems);
      } else
#endif
      if (!g_fft_two_cta) {
        // one 256-thread CTA per SM: two groups of 4 warps on chain pairs, one shared chirp and filter spectrum
        const long long npairs = n1 * ((nchains + 1) / 2);
        const int g6 = (int)std::min<long long>(npairs, (long long)nsm);
        if (dir == 0)
          pxm_ring_fft6_kernel<0><<<g6, 256, PXM_FFT6_SMEM, stream>>>(tab, blocks, maps, px, pix_chain_stride, F, nld, ar, nchains,
                                                                    npairs);
        else
          pxm_ring_fft6_kernel<1><<<g6, 256, PXM_FFT6_SMEM, stream>>>(tab, blocks, maps, px, pix_chain_stride, F, nld, ar, nchains,
                                                                    npairs);
      } else if (dir == 0)
        pxm_ring_fft3_kernel<0><<<g3, 128, PXM_FFT3_SMEM, stream>>>(tab, blocks, maps, px, pix_chain_stride, F, nld, ar, nchains,
                                                                  nitems);
      else
        pxm_ring_fft3_kernel<1><<<g3, 128, PXM_FFT3_SMEM, stream>>>(tab, blocks, maps, px, pix_chain_stride, F, nld, ar, nchains,
                                                                  nitems);
    } else if (dir == 0)
      pxm_ring_fft2_kernel<0, 1><<<grid1, 128, PXM_FFT2_SMEM, stream>>>(tab, remap[1], px, pix_chain_stride, F, nld, ar);
    else
      pxm_ring_fft2_kernel<1, 1><<<grid1, 128, PXM_FFT2_SMEM, stream>>>(tab, remap[1], px, pix_chain_stride, F, nld, ar);
    PXM_LAUNCHED();
  }
  if (class_mask & 1) {
    if (dir == 0)
      pxm_ring_fft2_kernel<0, 0><<<grid0, 256, PXM_FFT2_SMEM, stream>>>(tab, remap[0], px, pix_chain_stride, F, nld, ar);
    else
      pxm_ring_fft2_kernel<1, 0><<<grid0, 256, PXM_FFT2_SMEM, stream>>>(tab, remap[0], px, pix_chain_stride, F, nld, ar);
    PXM_LAUNCHED();
  }
  if (class_mask & 4) {
    if (dir == 0)
      pxm_ring_fft_kernel<0><<<grid, 256, PXM_FFT_SMEM, stream>>>(d_groups, ngroups, px, pix_chain_stride, F, nld, ar, 11);
    else
      pxm_ring_fft_kernel<1><<<grid, 256, PXM_FFT_SMEM, stream>>>(d_groups, ngroups, px, pix_chain_stride, F, nld, ar, 11);
    PXM_LAUNCHED();
  }
  return PXM_OK;
}

// 0: choose by grid size, 1: always the multi-pass kernel, 2: always the two-pass kernel (where it applies),
// 3: two-pass, with the persistent staged kernel for the radix-32 class (what 0 picks for large grids)
// 4: like 3 but with the two-CTA persistent kernel pxm_ring_fft3_kernel instead of pxm_ring_fft6_kernel
// 5: like 3 with the pair-split persistent kernel, 6: like 3 with the 32-points-per-thread persistent kernel
void pxm_fft_set_legacy(int on) {
  g_fft_two_cta = on == 4;
  if (on == 5) g_fft_pair = 1;
  if (on == 6) g_fft_pair = 0;
  g_fft_legacy = (on >= 4) ? 3 : on;
}

#ifdef PXM_FFT3_TIMING
namespace {
// register-only radix-32 DFT pairs (what the middle pass does between its shared-memory accesses)
__global__ void __launch_bounds__(128, 2) dft32_ubench_kernel(cplx* out, int iters, double a) {
  cplx x[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) x[k] = make_double2(a * (k + threadIdx.x), a * (k - 3.0));
  for (int it = 0; it < iters; ++it) {
    dft32<false>(x);
#pragma unroll
    for (int k = 0; k < 32; ++k) x[k] = cmul(x[k], make_double2(a, 0.5 * a));
    dft32<true>(x);
  }
  cplx acc = make_double2(0.0, 0.0);
#pragma unroll
  for (int k = 0; k < 32; ++k) acc = cadd(acc, x[k]);
  out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}
}  // namespace
extern "C" int pxm_debug_dft_ubench(int ctas_per_sm, int iters, float* ms_out) {
  int nsm = 0;
  cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, 0);
  cplx* out = nullptr;
  cudaMalloc(&out, sizeof(cplx) * nsm * ctas_per_sm * 128);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  dft32_ubench_kernel<<<nsm * ctas_per_sm, 128>>>(out, 10, 0.001);
  cudaEventRecord(e0);
  dft32_ubench_kernel<<<nsm * ctas_per_sm, 128>>>(out, iters, 0.001);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  cudaEventElapsedTime(ms_out, e0, e1);
  cudaFree(out);
  return 0;
}
#endif

// development aid (built with -DPXM_FFT3_TIMING only): cycles thread 0 of every CTA of the persistent
// kernel spent in each phase since the last call
#ifdef PXM_FFT3_TIMING
extern "C" int pxm_debug_fft3_clocks(unsigned long long* out8) {
  unsigned long long z[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out8, g_fft3_clk, sizeof(z));
  cudaMemcpyToSymbol(g_fft3_clk, z, sizeof(z));
  return 0;
}
#endif

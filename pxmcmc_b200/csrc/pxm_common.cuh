// pxmcmc_b200: shared definitions for the sm_100a kernels and the host plans.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#ifndef PXM_HD
#define PXM_HD __host__ __device__ __forceinline__
#endif

// ---------------------------------------------------------------------------
// error handling (C ABI returns int codes; message kept per thread)
// ---------------------------------------------------------------------------
enum {
  PXM_OK = 0,
  PXM_ERR_CUDA = 1,
  PXM_ERR_ARG = 2,
  PXM_ERR_NODEVICE = 3,
  PXM_ERR_ALLOC = 4,
  PXM_ERR_UNSUPPORTED = 5,
};

void pxm_set_error(const std::string& msg);

#define PXM_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      pxm_set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " @" + __FILE__ + \
                    ":" + std::to_string(__LINE__));                                     \
      return PXM_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

// every kernel launch of the library goes through this (launch counter for bench.py's gpu_launches)
extern long long g_pxm_launches;
#define PXM_LAUNCHED()           \
  do {                           \
    ++g_pxm_launches;            \
    PXM_CUDA(cudaGetLastError()); \
  } while (0)

#define PXM_REQUIRE(cond, msg)                     \
  do {                                             \
    if (!(cond)) {                                 \
      pxm_set_error(std::string("bad argument: ") + (msg)); \
      return PXM_ERR_ARG;                          \
    }                                              \
  } while (0)

#define PXM_TRY(expr)          \
  do {                         \
    int _r = (expr);           \
    if (_r != PXM_OK) return _r; \
  } while (0)

// ---------------------------------------------------------------------------
// Data layouts (DESIGN.md "Data layout in HBM")
//
// 1. Legendre table tile: 32 ring rows (t) x 16 degree columns (l), 4 KB,
//    stored contiguously with a 16-byte-chunk XOR swizzle so that the FP64
//    mma.m8n8k4 A-fragment loads are shared-memory bank-conflict free in BOTH
//    contraction orientations (over l: synthesis-type; over t: analysis-type).
//    word index inside the tile for (r, c):
// ---------------------------------------------------------------------------
constexpr int PXM_TILE_T = 32;
constexpr int PXM_TILE_L = 16;
constexpr int PXM_TILE_DOUBLES = PXM_TILE_T * PXM_TILE_L;  // 512 doubles = 4 KB

PXM_HD int pxm_tile_word(int r, int c) { return r * PXM_TILE_L + (c ^ ((r & 3) << 2)); }

// 2. "k4-interleaved" matrices: every intermediate array that is the streamed
//    data operand of a Legendre contraction (ring-Fourier coefficients F_m(t),
//    harmonic coefficients f_lm) is stored per m-slot as [row/4][col][row%4]
//    doubles, `nld` columns.  One mma B fragment (4 k-rows x 8 columns) is then
//    32 consecutive doubles.
PXM_HD size_t pxm_il_index(int row, int col, int nld) {
  return ((size_t)(row >> 2) * (size_t)nld + (size_t)col) * 4 + (size_t)(row & 3);
}

// numpy's _lerp (quantile method "linear"): a + (b-a) t, or b - (b-a)(1-t) when t >= 0.5.  Explicitly rounded
// products, so that no translation unit contracts them into an FMA numpy does not evaluate.
__device__ __forceinline__ double pxm_lerp_np(double a, double b, double t) {
  const double d = b - a;
  return (t >= 0.5) ? __dsub_rn(b, __dmul_rn(d, 1.0 - t)) : __dadd_rn(a, __dmul_rn(d, t));
}

PXM_HD int pxm_round_up(int x, int m) { return (x + m - 1) / m * m; }
PXM_HD int pxm_ceil_div(int x, int m) { return (x + m - 1) / m; }

// descriptors of the grouped Legendre contraction -----------------------------
struct PxmLegSeg {
  unsigned long long a_off;  // doubles: first table tile of this (item, segment)
  unsigned long long b_off;  // doubles: row 0 of this segment's data operand (interleaved)
  int a_kstride;             // doubles between the tile groups of consecutive k-stages
  int a_mstride;             // doubles between consecutive M-direction tiles of one stage
  int mt0;                   // first M-direction tile present (others are implicit zeros)
  int nmt;                   // number of M-direction tiles present
  int nk;                    // number of k-stages
  int src;                   // rank whose workspace holds this segment's data operand (0 when not sharded)
};

struct PxmLegItem {
  unsigned long long c_off;  // doubles: first output row-group of the tile
  int seg_begin;
  int seg_count;
  int nmt_out;  // number of M-direction tiles to store
  int cost;     // k-stages x tiles, for ordering
  int dst;      // rank whose workspace receives the output tile (0 when not sharded)
  int pad;      // 1: also store (zero) rows beyond nmt_out up to the 64-row tile (outputs in harmonic buffers)
};

// optional epilogue of a contraction whose output is a harmonic array: out <- c (acc - b) on the complex numbers formed by
// adjacent (re, im) columns, b = chain 0 of an array in the output's own layout (b == nullptr: plain store).  The Gram
// form of the data-fidelity gradient, g = ic (G f - A^dagger d), in one launch (pxm_wav_gram_gradient)
struct PxmLegAffine {
  const double* b;  // same base convention as the output pointer (item.c_off applies)
  double re, im;
};

// Workspaces of the ranks of an m-sharded plan (peer-mapped device memory, NVLink):
// the contraction over l PUSHES its output tile into the ring buffer of the rank that
// owns those rings, the contraction over rings PULLS ring blocks from their owners with
// the same cp.async.bulk copies it uses locally.  Unsharded plans use p[0] only.
constexpr int PXM_MAX_PEERS = 8;
struct PxmPeers {
  double* p[PXM_MAX_PEERS];
};

// descriptors of the ring FFT ---------------------------------------------------
struct PxmFftGroup {
  int ell;          // bandlimit of this ring grid
  int n;            // 2*ell-1 samples per ring
  int M;            // power-of-two Bluestein length >= 2n-1
  int logM;
  int rings;        // end of this rank's ring range (ell when not sharded)
  int rings_per_cta;
  int cta_begin;    // first CTA (within one chain) of this group
  int nslots;       // ell (paired +-m, spin 0) or 2*ell-1
  int paired;       // 1: slot = |m|, 4 columns per chain; 0: slot = m+ell-1, 2 columns per chain
  int pad;          // log2(rings_per_cta)
  int ring0;        // first ring this rank transforms (`rings` is the end, exclusive); 0 when not sharded
  int pad2;
  double scale;     // applied to every output
  unsigned long long pix_off;       // complex elements: start of this map's LOCAL rows inside one chain's pixel vector
  unsigned long long f_off;         // doubles: start of this grid's ring-Fourier array
  unsigned long long slot_stride;   // doubles between m-slots
  unsigned long long chirp_off;     // complex elements into the twiddle arena: c_j = exp(-i pi j^2/n), n entries
  unsigned long long bhat_off;      // complex: FFT_M of the chirp filter, M entries, in the kernel's own permuted order
  unsigned long long tw_off;        // complex: exp(-2 pi i k/M), k < M
  unsigned long long bhat2_off;     // complex: FFT_M of the chirp filter in natural order (two-pass kernel)
  unsigned long long tw2_off;       // complex, M = 512 / 1024 only: W_M^{j2 k1} as [k1][j2], then as [j2][k1] (2 M entries)
};

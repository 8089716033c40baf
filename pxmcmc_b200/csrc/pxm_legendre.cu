// Grouped FP64 tensor-core (DMMA) Legendre contraction for sm_100a.
//
// This is the O(L^3) stage of every spherical harmonic / wavelet transform the
// reference performs through pyssht/pys2let (call sites:
// /root/reference/pxmcmc/transforms.py:95-98, pxmcmc/measurements.py:223-239).
// For every azimuthal order m it multiplies a precomputed REAL table
// T^m[t, l] (32x16 swizzled tiles, see pxm_common.cuh) with complex data stored
// as real columns (re/im x +-m x chains):
//
//   ORIENT 0 (synthesis-type):  C[t, n] = sum_l T^m[t, l] B[l, n]
//   ORIENT 1 (analysis-type) :  C[l, n] = sum_t T^m[t, l] B[t, n]   (sum may run
//                               over several segments = wavelet scales)
//
// One CTA = one 64-row output tile of one m (work item) x one block of BN
// columns.  Table tiles and data rows are staged by cp.async.bulk (1-D TMA
// bulk copies) into a STAGES-deep shared-memory ring guarded by mbarriers; 8
// warps issue mma.sync.m8n8k4.f64 (DMMA) from conflict-free fragment loads.
// tcgen05/TMEM has no FP64 kind, so DMMA is the FP64 tensor path on Blackwell.
#include "pxm_common.cuh"

namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// the same copy with an L2 eviction-priority hint: table tiles are read once per launch and, at 0.2-4 GB per
// transform, can never stay in the 126 MB L2 -- streamed evict-first they stop flushing the state vectors, the ring
// arrays and the FFT tables out of it between the launches of an iteration
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
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
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

#ifdef PXM_LEG_NO_L2_HINT
#define LEG_TABLE_COPY(dst, src, bytes, bar) bulk_g2s(dst, src, bytes, bar)
#else
#define LEG_TABLE_COPY(dst, src, bytes, bar) bulk_g2s_hint(dst, src, bytes, bar, pol)
#endif

constexpr int LEG_CONSUMER_WARPS = 8;
constexpr int LEG_THREADS = (LEG_CONSUMER_WARPS + 1) * 32;  // + one TMA producer warp

template <int ORIENT, int BN, int WARPS_M, int WARPS_N, int STAGES>
struct LegCfg {
  static constexpr int BM = 64;
  static constexpr int BK = 16;                             // k rows per pipeline stage
  static constexpr int TILE_ROWS = ORIENT == 0 ? 32 : 16;  // output rows covered by one table tile
  static constexpr int NT_M = BM / TILE_ROWS;              // 2 full tiles (S) or 4 half tiles (A) per stage
  static constexpr int A_PIECE = ORIENT == 0 ? PXM_TILE_DOUBLES : PXM_TILE_DOUBLES / 2;
  static constexpr int A_STAGE = NT_M * A_PIECE;            // 1024 doubles = 8 KB
  static constexpr int B_STAGE = BK * BN;
  static constexpr int WM = BM / WARPS_M;
  static constexpr int WN = BN / WARPS_N;
  static constexpr int MI = WM / 8;
  static constexpr int NI = WN / 8;
  static constexpr size_t SMEM = 128 + (size_t)STAGES * (A_STAGE + B_STAGE) * sizeof(double);
  static_assert(WARPS_M * WARPS_N == LEG_CONSUMER_WARPS, "8 consumer warps");
  static_assert(MI >= 1 && NI >= 1, "warp tile");
  static_assert(2 * STAGES * 8 <= 128, "barrier area");
};

// ORIENT 0: a k-stage is one 16-degree block: NT_M = 2 full 32x16 tiles (rows = rings).
// ORIENT 1: a k-stage is HALF a ring block (16 rings): 4 half tiles (rows = degrees); the
//           descriptor's nk counts ring blocks, i.e. two stages each.
template <int ORIENT, int BN, int WARPS_M, int WARPS_N, int STAGES>
__global__ void __launch_bounds__(LEG_THREADS, 2)
pxm_legendre_kernel(const double* __restrict__ tab, const __grid_constant__ PxmPeers bpeers,
                    const __grid_constant__ PxmPeers cpeers, const PxmLegItem* __restrict__ items,
                    const PxmLegSeg* __restrict__ segs, int nld, const PxmLegAffine aff) {
  using C = LegCfg<ORIENT, BN, WARPS_M, WARPS_N, STAGES>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* empty = full + STAGES;
  double* sA = reinterpret_cast<double*>(smem_raw + 128);
  double* sB = sA + STAGES * C::A_STAGE;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const PxmLegItem item = items[blockIdx.x];
  const int n0 = blockIdx.y * BN;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], LEG_CONSUMER_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp == LEG_CONSUMER_WARPS) {
    // ===================== TMA producer warp (one elected lane) =====================
    if (lane == 0) {
      int it = 0;
#ifndef PXM_LEG_NO_L2_HINT
      const uint64_t pol = l2_evict_first_policy();
#endif
      for (int s = 0; s < item.seg_count; ++s) {
        const PxmLegSeg sg = segs[item.seg_begin + s];
        const int nst = ORIENT == 0 ? sg.nk : 2 * sg.nk;
        const uint32_t bytes = (uint32_t)(sg.nmt * C::A_PIECE * 8 + C::BK * BN * 8);
        for (int k = 0; k < nst; ++k, ++it) {
          const int slot = it % STAGES;
          if (it >= STAGES) mbar_wait(&empty[slot], (uint32_t)(((it / STAGES) - 1) & 1));
          uint64_t* bar = &full[slot];
          mbar_expect_tx(bar, bytes);
          double* dstA = sA + slot * C::A_STAGE + sg.mt0 * C::A_PIECE;
          if (ORIENT == 0) {
            const double* srcA = tab + sg.a_off + (size_t)k * (size_t)sg.a_kstride;
            for (int j = 0; j < sg.nmt; ++j)
              LEG_TABLE_COPY(dstA + j * C::A_PIECE, srcA + (size_t)j * (size_t)sg.a_mstride, C::A_PIECE * 8, bar);
          } else {
            const double* srcA = tab + sg.a_off + (size_t)(k >> 1) * (size_t)sg.a_kstride + (k & 1) * C::A_PIECE;
            for (int j = 0; j < sg.nmt; ++j)
              LEG_TABLE_COPY(dstA + j * C::A_PIECE, srcA + (size_t)j * (size_t)sg.a_mstride, C::A_PIECE * 8, bar);
          }
          double* dstB = sB + slot * C::B_STAGE;
          // m-sharded plans: the ring block may live in a peer's workspace (pulled over NVLink)
          const double* srcB = bpeers.p[sg.src] + sg.b_off + ((size_t)k * (C::BK / 4) * (size_t)nld + (size_t)n0) * 4;
          if (BN == nld) {
            bulk_g2s(dstB, srcB, (uint32_t)(C::BK * BN * 8), bar);
          } else {
#pragma unroll
            for (int rg = 0; rg < C::BK / 4; ++rg)
              bulk_g2s(dstB + rg * BN * 4, srcB + (size_t)rg * (size_t)nld * 4, BN * 32, bar);
          }
        }
      }
    }
    return;
  }

  // ================================ consumer warps ================================
  const int g = lane >> 2, q = lane & 3;
  const int wm = warp / WARPS_N, wn = warp % WARPS_N;
  double acc[C::MI][C::NI][2];
#pragma unroll
  for (int mi = 0; mi < C::MI; ++mi)
#pragma unroll
    for (int ni = 0; ni < C::NI; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;

  int it = 0;
  for (int s = 0; s < item.seg_count; ++s) {
    const int seg_nst = (ORIENT == 0 ? 1 : 2) * segs[item.seg_begin + s].nk;
    const int seg_mt0 = segs[item.seg_begin + s].mt0;
    const int seg_mt1 = seg_mt0 + segs[item.seg_begin + s].nmt;
    bool mv[C::MI];
#pragma unroll
    for (int mi = 0; mi < C::MI; ++mi) {
      const int tl = (wm * C::WM + mi * 8) / C::TILE_ROWS;
      mv[mi] = (tl >= seg_mt0) && (tl < seg_mt1);
    }
    for (int k = 0; k < seg_nst; ++k, ++it) {
      const int slot = it % STAGES;
      mbar_wait(&full[slot], (uint32_t)((it / STAGES) & 1));
      const double* a_s = sA + slot * C::A_STAGE;
      const double* b_s = sB + slot * C::B_STAGE;
#pragma unroll
      for (int kk = 0; kk < C::BK / 4; ++kk) {
        double a[C::MI], b[C::NI];
#pragma unroll
        for (int mi = 0; mi < C::MI; ++mi) {
          const int row = wm * C::WM + mi * 8 + g;
          if (ORIENT == 0) {
            const int tl = row >> 5, r = row & 31;
            a[mi] = a_s[tl * C::A_PIECE + r * PXM_TILE_L + (((kk ^ (r & 3)) << 2) | q)];
          } else {
            const int tl = row >> 4, c = row & 15, r = kk * 4 + q;
            a[mi] = a_s[tl * C::A_PIECE + r * PXM_TILE_L + (c ^ (q << 2))];
          }
        }
#pragma unroll
        for (int ni = 0; ni < C::NI; ++ni) b[ni] = b_s[(kk * BN + wn * C::WN + ni * 8 + g) * 4 + q];
#pragma unroll
        for (int mi = 0; mi < C::MI; ++mi) {
          if (mv[mi]) {
#pragma unroll
            for (int ni = 0; ni < C::NI; ++ni) dmma(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[slot]);  // this warp is done with the slot
    }
  }

  // ---- epilogue: k4-interleaved store (into the owner of these rows: a peer when m-sharded) ----
  double* __restrict__ cmat = cpeers.p[item.dst];
#pragma unroll
  for (int mi = 0; mi < C::MI; ++mi) {
    const int row = wm * C::WM + mi * 8 + g;
    // rows past the last tile: skipped, or -- harmonic buffers, whose slots are padded to whole 64-row tiles -- written as the
    // zeros the accumulators still hold, so that a caller-provided output array needs no initialisation
    if (row / C::TILE_ROWS >= item.nmt_out && !item.pad) continue;
#pragma unroll
    for (int ni = 0; ni < C::NI; ++ni) {
      const int col = n0 + wn * C::WN + ni * 8 + 2 * q;  // even: the thread holds (re, im) of one complex number
      double vr = acc[mi][ni][0], vi = acc[mi][ni][1];
      if (aff.b != nullptr) {
        const double xr = vr - aff.b[item.c_off + pxm_il_index(row, col & 2, nld)];
        const double xi = vi - aff.b[item.c_off + pxm_il_index(row, (col & 2) + 1, nld)];
        vr = __dsub_rn(__dmul_rn(aff.re, xr), __dmul_rn(aff.im, xi));  // products rounded as in the elementwise kernels
        vi = __dadd_rn(__dmul_rn(aff.re, xi), __dmul_rn(aff.im, xr));
      }
      cmat[item.c_off + pxm_il_index(row, col, nld)] = vr;
      cmat[item.c_off + pxm_il_index(row, col + 1, nld)] = vi;
    }
  }
}

// Plain one-thread-per-output contraction over the same descriptors.  Debugging
// aid for the GPU tests (localises a fault to the tensor-core kernel or to the
// tables/descriptors); never selected by the product path.
template <int ORIENT>
__global__ void pxm_legendre_naive_kernel(const double* __restrict__ tab, const PxmPeers bpeers, const PxmPeers cpeers,
                                          const PxmLegItem* __restrict__ items, const PxmLegSeg* __restrict__ segs,
                                          int nld, const PxmLegAffine aff) {
  constexpr int BK = ORIENT == 0 ? 16 : 32;
  constexpr int TILE_ROWS = ORIENT == 0 ? 32 : 16;
  const PxmLegItem item = items[blockIdx.x];
  double* cmat = cpeers.p[item.dst];
  const int row = threadIdx.x & 63;
  for (int col = blockIdx.y * blockDim.x / 64 + (threadIdx.x >> 6); col < nld; col += gridDim.y * (blockDim.x / 64)) {
    const int tl = row / TILE_ROWS;
    if (tl >= item.nmt_out) {
      // padded rows of harmonic buffers: zeros, as the tensor-core kernel writes them (outputs need no initialisation)
      if (item.pad) cmat[item.c_off + pxm_il_index(row, col, nld)] = 0.0;
      continue;
    }
    double acc = 0.0;
    for (int s = 0; s < item.seg_count; ++s) {
      const PxmLegSeg sg = segs[item.seg_begin + s];
      const double* bmat = bpeers.p[sg.src];
      if (tl < sg.mt0 || tl >= sg.mt0 + sg.nmt) continue;
      for (int k = 0; k < sg.nk; ++k) {
        const double* tile = tab + sg.a_off + (size_t)k * sg.a_kstride + (size_t)(tl - sg.mt0) * sg.a_mstride;
        for (int kk = 0; kk < BK; ++kk) {
          double a;
          if (ORIENT == 0)
            a = tile[pxm_tile_word(row & 31, kk)];
          else
            a = tile[pxm_tile_word(kk, row & 15)];
          acc += a * bmat[sg.b_off + pxm_il_index(k * BK + kk, col, nld)];
        }
      }
    }
    if (aff.b != nullptr) {  // the partner (re or im) of this column is recomputed: keep the debugging kernel simple
      double oth = 0.0;
      const int pc = col ^ 1;
      for (int s = 0; s < item.seg_count; ++s) {
        const PxmLegSeg sg = segs[item.seg_begin + s];
        const double* bmat = bpeers.p[sg.src];
        if (tl < sg.mt0 || tl >= sg.mt0 + sg.nmt) continue;
        for (int k = 0; k < sg.nk; ++k) {
          const double* tile = tab + sg.a_off + (size_t)k * sg.a_kstride + (size_t)(tl - sg.mt0) * sg.a_mstride;
          for (int kk = 0; kk < BK; ++kk)
            oth += (ORIENT == 0 ? tile[pxm_tile_word(row & 31, kk)] : tile[pxm_tile_word(kk, row & 15)]) *
                   bmat[sg.b_off + pxm_il_index(k * BK + kk, pc, nld)];
        }
      }
      const double x0 = acc - aff.b[item.c_off + pxm_il_index(row, col & 3, nld)];
      const double x1 = oth - aff.b[item.c_off + pxm_il_index(row, pc & 3, nld)];
      acc = (col & 1) ? __dadd_rn(__dmul_rn(aff.re, x0), __dmul_rn(aff.im, x1))    // im: re * xi + im * xr
                      : __dsub_rn(__dmul_rn(aff.re, x0), __dmul_rn(aff.im, x1));   // re: re * xr - im * xi
    }
    cmat[item.c_off + pxm_il_index(row, col, nld)] = acc;
  }
}

template <int ORIENT, int BN, int WARPS_M, int WARPS_N, int STAGES>
int launch_cfg(const double* tab, const PxmPeers& b, const PxmPeers& c, const PxmLegItem* items, const PxmLegSeg* segs,
               int nitems, int nld, cudaStream_t stream, const PxmLegAffine& aff) {
  using C = LegCfg<ORIENT, BN, WARPS_M, WARPS_N, STAGES>;
  static bool configured = false;
  auto kern = pxm_legendre_kernel<ORIENT, BN, WARPS_M, WARPS_N, STAGES>;
  if (!configured) {
    PXM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    configured = true;
  }
  if (nitems == 0) return PXM_OK;  // preload only (pxm_legendre_preload)
  dim3 grid(nitems, nld / BN);
  kern<<<grid, LEG_THREADS, C::SMEM, stream>>>(tab, b, c, items, segs, nld, aff);
  PXM_LAUNCHED();
  return PXM_OK;
}

// warp layouts: contraction over l (ORIENT 0) splits rows x columns 2x4; contraction over rings
// (ORIENT 1) gives every warp all 64 degrees (1x8), so that segments whose l-support covers only
// part of the tile (wavelet scales) keep all eight warps equally busy
template <int ORIENT>
int launch_orient(const double* tab, const PxmPeers& b, const PxmPeers& c, const PxmLegItem* items,
                  const PxmLegSeg* segs, int nitems, int nld, cudaStream_t stream, const PxmLegAffine& aff) {
  // pipeline depth: few right-hand sides (single chain) make the kernel a pure table stream, so the
  // narrow variants keep 8 stages (~10 KB each) in flight per CTA; the wide ones are DMMA-bound
  constexpr int ST = 4, STN = 8;
  if (ORIENT == 0) {
    if (nld % 128 == 0) return launch_cfg<ORIENT, 128, 2, 4, ST>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 64) return launch_cfg<ORIENT, 64, 2, 4, ST>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 32) return launch_cfg<ORIENT, 32, 4, 2, STN>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 16) return launch_cfg<ORIENT, 16, 4, 2, STN>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 8) return launch_cfg<ORIENT, 8, 8, 1, STN>(tab, b, c, items, segs, nitems, nld, stream, aff);
  } else {
    if (nld % 128 == 0) return launch_cfg<ORIENT, 128, 1, 8, ST>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 64) return launch_cfg<ORIENT, 64, 1, 8, ST>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 32) return launch_cfg<ORIENT, 32, 2, 4, STN>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 16) return launch_cfg<ORIENT, 16, 4, 2, STN>(tab, b, c, items, segs, nitems, nld, stream, aff);
    if (nld == 8) return launch_cfg<ORIENT, 8, 8, 1, STN>(tab, b, c, items, segs, nitems, nld, stream, aff);
  }
  pxm_set_error("legendre: unsupported column count " + std::to_string(nld));
  return PXM_ERR_ARG;
}

}  // namespace

// valid leading dimensions: 8, 16, 32, 64 or a multiple of 128
int pxm_legendre_pad_columns(int ncols) {
  if (ncols <= 8) return 8;
  if (ncols <= 16) return 16;
  if (ncols <= 32) return 32;
  if (ncols <= 64) return 64;
  return pxm_round_up(ncols, 128);
}

int pxm_legendre_launch_peers(int orient, const double* tab, const PxmPeers& b, const PxmPeers& c,
                              const PxmLegItem* items, const PxmLegSeg* segs, int nitems, int nld,
                              cudaStream_t stream, int naive, const PxmLegAffine* affine);

int pxm_legendre_launch(int orient, const double* tab, const double* b, double* c, const PxmLegItem* items,
                        const PxmLegSeg* segs, int nitems, int nld, cudaStream_t stream, int naive) {
  PxmPeers bp = {}, cp = {};
  bp.p[0] = const_cast<double*>(b);
  cp.p[0] = c;
  return pxm_legendre_launch_peers(orient, tab, bp, cp, items, segs, nitems, nld, stream, naive, nullptr);
}

// Load and configure the kernels a plan with `nld` columns will launch (CUDA loads kernels
// lazily, and a first-use load may synchronise the device -- fatal while a peer barrier spins).
int pxm_legendre_preload(int nld) {
  PxmPeers z = {};
  const PxmLegAffine none = {nullptr, 0.0, 0.0};
  PXM_TRY(launch_orient<0>(nullptr, z, z, nullptr, nullptr, 0, nld, 0, none));
  PXM_TRY(launch_orient<1>(nullptr, z, z, nullptr, nullptr, 0, nld, 0, none));
  cudaFuncAttributes a;
  PXM_CUDA(cudaFuncGetAttributes(&a, pxm_legendre_naive_kernel<0>));
  PXM_CUDA(cudaFuncGetAttributes(&a, pxm_legendre_naive_kernel<1>));
  return PXM_OK;
}

int pxm_legendre_launch_peers(int orient, const double* tab, const PxmPeers& b, const PxmPeers& c,
                              const PxmLegItem* items, const PxmLegSeg* segs, int nitems, int nld,
                              cudaStream_t stream, int naive, const PxmLegAffine* affine) {
  if (nitems <= 0) return PXM_OK;
  const PxmLegAffine aff = affine ? *affine : PxmLegAffine{nullptr, 0.0, 0.0};
  if (naive) {
    dim3 grid(nitems, 4);
    if (orient == 0)
      pxm_legendre_naive_kernel<0><<<grid, 256, 0, stream>>>(tab, b, c, items, segs, nld, aff);
    else
      pxm_legendre_naive_kernel<1><<<grid, 256, 0, stream>>>(tab, b, c, items, segs, nld, aff);
    PXM_LAUNCHED();
    return PXM_OK;
  }
  if (orient == 0) return launch_orient<0>(tab, b, c, items, segs, nitems, nld, stream, aff);
  return launch_orient<1>(tab, b, c, items, segs, nitems, nld, stream, aff);
}

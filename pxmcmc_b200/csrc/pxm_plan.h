// Host-side plan structures shared by the table generator and the plans.
#pragma once
#include <vector>

#include "pxm_common.cuh"

struct PxmWigSlot {
  int m;
  int lb0;
  int nlb;
  int pad;
  unsigned long long tile_off;
};

template <class T>
struct PxmDevVec {
  T* d = nullptr;
  size_t n = 0;
  int upload(const std::vector<T>& h) {
    release();
    n = h.size();
    if (n == 0) return PXM_OK;
    PXM_CUDA(cudaMalloc(&d, n * sizeof(T)));
    PXM_CUDA(cudaMemcpy(d, h.data(), n * sizeof(T), cudaMemcpyHostToDevice));
    return PXM_OK;
  }
  void release() {
    if (d) cudaFree(d);
    d = nullptr;
    n = 0;
  }
};

// One set of per-m Legendre tables (see pxm_tables.cu)
struct PxmTableLayout {
  int grid_L = 0, rings = 0, lmax = 0, spin = 0;
  bool paired = true;
  int l_lo = 0, l_hi = 0;
  int nslots = 0, ntb = 0;
  std::vector<int> slot_m, lb0, nlb;
  std::vector<unsigned long long> tile_off;  // doubles, relative to the arena the layout was made for
  size_t doubles = 0;
  // device array [rings][2] of (sin, cos) of theta/2 for ring grids that are not MW (HEALPix);
  // nullptr: MW ring t of bandlimit grid_L
  const double* d_half_angles = nullptr;
};

// m-sharding (SURVEY.md 8e-2): azimuthal orders are dealt to the ranks in a snake so that the
// triangular work (L - |m|) balances; +m and -m always share an owner.
inline int pxm_owner_of_m(int am, int world) {
  if (world <= 1) return 0;
  const int k = am % (2 * world);
  return k < world ? k : 2 * world - 1 - k;
}
// theta-sharding: rings are owned in blocks of 64 (one output tile of the contraction over l).
// Grids with fewer blocks than ranks are spread with a stride and rotated by `rot` (the scale
// index) so that the small wavelet scales do not all land on rank 0.
inline int pxm_owner_of_ring_block(int ell, int blk, int rot, int world) {
  if (world <= 1) return 0;
  const int nb = (ell + 63) / 64;
  if (nb >= world) return (int)(((long long)blk * world) / nb);
  return (blk * (world / nb) + rot) % world;
}
inline void pxm_ring_range(int ell, int rot, int rank, int world, int* t0, int* t1) {
  const int nb = (ell + 63) / 64;
  int first = -1, last = -1;
  for (int b = 0; b < nb; ++b)
    if (pxm_owner_of_ring_block(ell, b, rot, world) == rank) {
      if (first < 0) first = b;
      last = b;
    }
  if (first < 0) {
    *t0 = *t1 = 0;
    return;
  }
  *t0 = 64 * first;
  *t1 = 64 * (last + 1) < ell ? 64 * (last + 1) : ell;
}

// slots whose |m| is owned by another rank get no tiles (rank = 0, world = 1: everything)
void pxm_make_table_layout(PxmTableLayout& T, int grid_L, int rings, int lmax, int spin, int l_lo, int l_hi,
                           unsigned long long base_off, int rank = 0, int world = 1);
int pxm_generate_lambda(const PxmTableLayout& T, double* d_tab, const double* d_g, cudaStream_t st);
int pxm_generate_w(const PxmTableLayout& T, double* d_tab, const double* d_g, cudaStream_t st);
int pxm_generate_gram(const PxmTableLayout& Tl, const double* d_lam_tab, const PxmTableLayout& Tg, double* d_g_tab, double scale,
                      cudaStream_t st, const double* d_ring_weights = nullptr);

// kernels' launchers -------------------------------------------------------------
int pxm_legendre_pad_columns(int ncols);
int pxm_legendre_launch(int orient, const double* tab, const double* b, double* c, const PxmLegItem* items,
                        const PxmLegSeg* segs, int nitems, int nld, cudaStream_t stream, int naive);
int pxm_legendre_launch_peers(int orient, const double* tab, const PxmPeers& b, const PxmPeers& c,
                              const PxmLegItem* items, const PxmLegSeg* segs, int nitems, int nld,
                              cudaStream_t stream, int naive, const PxmLegAffine* affine = nullptr);
int pxm_legendre_preload(int nld);
int pxm_elem_preload();
int pxm_hpx_ring_dft_launch(int dir, int nside, int L, const void* map, double* F, unsigned long long f_off,
                            unsigned long long slot_stride, int nld, cudaStream_t stream);
int pxm_fft_choose_M(int n, int* logM);
int pxm_fft_rings_per_cta_log(int M);
int pxm_fft_setup_tables(const PxmFftGroup* d_groups, const PxmFftGroup* h_groups, int ngroups, void* d_arena,
                         cudaStream_t stream);
int pxm_fft_class_bit(int logM);
void pxm_fft_set_legacy(int on);
int pxm_fft_launch(int dir, const PxmFftGroup* d_groups, const PxmFftGroup* h_groups, int ngroups, int ctas_per_chain,
                   void* pix, size_t pix_chain_stride, double* F, int nld, const void* d_arena, int nchains,
                   int class_mask, cudaStream_t stream);

int pxm_launch_soft(int is_complex, const void* x, const double* Tv, double Ts, void* out, size_t n, size_t nchains,
                    cudaStream_t st);
int pxm_launch_myula(const void* X, const void* prox, const void* gradg, const double* Tv, double Ts,
                     const double* w_re, const double* w_im, void* Xout, void* prox_out, size_t n, size_t nchains,
                     double delta, double lmda, int noise_mode, unsigned long long seed, unsigned long long step,
                     const unsigned long long* d_step, unsigned int stream0, cudaStream_t st,
                     const double* d_par = nullptr);
int pxm_launch_counter_add(unsigned long long* ctr, unsigned long long inc, cudaStream_t st);
int pxm_launch_resid(const void* preds, const void* data, const void* ic, void* out, size_t n, size_t nchains,
                     cudaStream_t st);
int pxm_launch_ring_resid(const double* pred, const double* data, const void* ic, double* out, int nslots, int rings,
                          int nld, int ncols, double scale, unsigned long long slot_stride, cudaStream_t st);
int pxm_launch_reduce(int kind, const void* a, const void* b, const void* c, const void* d, const double* w,
                      double delta, double lmda, size_t n, size_t nchains, void* partial, void* out, cudaStream_t st,
                      const double* d_par = nullptr);
int pxm_launch_pxmala_accept(double* S, const void* s1, const void* s2, const void* L2p, const void* priorp, double mu,
                             double lmda, int tune, long long i, unsigned long long seed, unsigned long long step,
                             unsigned int stream_id, signed char* acc_trace, double* delta_trace, long long trace_stride,
                             int nchains, cudaStream_t st);
int pxm_launch_philox_normal(double* out, size_t n, size_t nchains, unsigned long long seed, unsigned long long step,
                             const unsigned long long* d_step, unsigned int stream0, cudaStream_t st);
int pxm_launch_select(const double* flag, size_t flag_stride, size_t nchains, void* const* dst, const void* const* src,
                      const size_t* counts, int narrays, cudaStream_t st);
int pxm_launch_lincomb(int nx, const void* const* xs, const double* as, const double* z, double cz, double c0,
                       void* out, size_t total, cudaStream_t st);
int pxm_launch_gradlogpi(const void* X, const void* prox, const double* Tv, double Ts, const void* gradg, double lmda,
                         void* out, size_t n, size_t nchains, cudaStream_t st);
int pxm_launch_skrock(int stage, const void* U, const void* V, const void* gradg, const void* prox, const double* Tv,
                      double Ts, double lmda, double a, double b, double c, double c0, double cs, double e,
                      const double* z_re, const double* z_im, int noise_mode, unsigned long long seed,
                      unsigned long long step, const unsigned long long* d_step, unsigned int stream0, void* out, size_t n,
                      size_t nchains, cudaStream_t st);
int pxm_launch_fista(const void* y, const void* gradg, const void* x, const double* Tv, double Ts, double Tscale,
                     double t, double* state, void* x_out, void* y_out, double* hist, long long cap, size_t n,
                     size_t nchains, void* partial, cudaStream_t st);
int pxm_launch_gather(int scatter, const void* in, const int* idx, const double* w, void* out, size_t nsel,
                      size_t nfull, size_t nchains, cudaStream_t st);
int pxm_launch_lm_convert(int to_internal, void* flm, double* H, const unsigned long long* d_slot_off,
                          const unsigned char* d_own, const double* d_gl, int L, int paired, int nld, int nchains,
                          cudaStream_t st);
int pxm_launch_r2c(const double* x, void* out, size_t total, cudaStream_t st);
int pxm_launch_csr_spmv(const int* indptr, const int* indices, const double* vals, const void* x, void* y, int nrows,
                        size_t ncols, size_t nchains, cudaStream_t st);

int pxm_quantile_max_samples();
int pxm_launch_quantile_columns(const double* chain, long long nsamples, long long ncols, long long ld, long long lo_a,
                                double g_a, long long lo_b, double g_b, double* out_a, double* out_b, cudaStream_t st);

long long pxm_stats_slots(int mode, long long nchains);
int pxm_launch_stats_accumulate(double* acc, const void* x, size_t n, size_t nchains, int mode, long long nsamples,
                                long long j, const long long* d_j, cudaStream_t st);
int pxm_launch_stats_partials(const double* acc, size_t n, size_t nchains, int mode, long long nsamples, double* rec,
                              double* cmean, double* cvar, cudaStream_t st);

int pxm_launch_rank_diagnostics(const double* chain, long long m, long long n, long long ncols, long long ld,
                                double* scratch, double* rhat, double* ess_bulk, double* ess_tail, cudaStream_t st);

int pxm_credible_tails(long long npooled, long long lo_a, long long lo_b, long long* klo, long long* khi);
int pxm_launch_credible_push(double* st, const void* x, size_t n, size_t nchains, int mode, long long klo,
                             long long khi, long long count, const long long* d_j, cudaStream_t s);
int pxm_launch_credible_finalize(const double* st, size_t n, int mode, long long npooled, long long klo, long long khi,
                                 long long lo_a, double g_a, long long lo_b, double g_b, double* out_lo,
                                 double* out_hi, cudaStream_t s);

int pxm_debug_naive();

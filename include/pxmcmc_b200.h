/* pxmcmc_b200 -- C ABI of the B200 (sm_100a) implementation of pxmcmc's
 * per-iteration proximal-Langevin hot path.
 *
 * The reference (auggiemarignier/pxmcmc) is pure Python; the arithmetic of its
 * hot path lives in C libraries reached through Cython (pyssht, pys2let) and in
 * numpy/scipy.  Each entry point below names the reference call it replaces
 * (paths relative to the reference repository root).
 *
 * Conventions
 *  - every d_* pointer is a DEVICE pointer; complex arrays are interleaved
 *    (re, im) float64 (numpy complex128); batched arrays are [nchains][n]
 *    row-major; the caller owns all buffers.
 *  - `stream` is a cudaStream_t passed as void* (0 = default stream).
 *  - return value 0 = success; otherwise pxm_last_error() describes the
 *    failure (thread-local).  There is NO CPU fallback: pxm_init fails when no
 *    sm_100-class device is visible.
 *  - a plan is immutable after creation and may be used from one stream at a
 *    time (it owns the workspace of its operators).
 */
#ifndef PXMCMC_B200_H
#define PXMCMC_B200_H
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pxm_sht_plan pxm_sht_plan;
typedef struct pxm_wav_plan pxm_wav_plan;
typedef struct pxm_hpx_plan pxm_hpx_plan;

const char* pxm_last_error(void);
int pxm_init(int device);

/* ---- spin spherical harmonic transforms on MW sampling --------------------
 * pyssht.inverse / forward / inverse_adjoint / forward_adjoint (Method="MW",
 * Reality=False): pxmcmc/measurements.py:223,225,237,239.
 * f: [nbatch][L][2L-1] complex, flm: [nbatch][L*L] complex (index l*l+l+m).
 * d_gl (may be NULL): real per-degree multiplier g[l], l<L, applied to the
 * harmonic side of the call (fuses WeakLensingHarmonic.harmonic_mapping,
 * pxmcmc/measurements.py:162-171). */
int pxm_sht_plan_create(int L, int spin, int max_batch, pxm_sht_plan** out);
int pxm_sht_plan_destroy(pxm_sht_plan* plan);
size_t pxm_sht_plan_table_bytes(const pxm_sht_plan* plan);
int pxm_sht_inverse(pxm_sht_plan* plan, const void* d_flm, void* d_f, int nbatch, const double* d_gl, void* stream);
int pxm_sht_forward(pxm_sht_plan* plan, const void* d_f, void* d_flm, int nbatch, const double* d_gl, void* stream);
int pxm_sht_inverse_adjoint(pxm_sht_plan* plan, const void* d_f, void* d_flm, int nbatch, const double* d_gl,
                            void* stream);
int pxm_sht_forward_adjoint(pxm_sht_plan* plan, const void* d_flm, void* d_f, int nbatch, const double* d_gl,
                            void* stream);

/* ---- scale-discretised wavelet transform (N=1, spin 0, multiresolution) ----
 * pys2let.synthesis_wav2px / synthesis_adjoint_px2wav / analysis_px2wav /
 * analysis_adjoint_wav2px as wrapped by SphericalWaveletTransform.inverse /
 * inverse_adjoint / forward / forward_adjoint: pxmcmc/transforms.py:95-154.
 * coef: [nbatch][ncoefs] complex = [scaling map, wavelet maps j=J_min..J]
 * (utils.flatten_mlm, pxmcmc/utils.py:11-22); pix: [nbatch][L(2L-1)] complex. */
int pxm_wav_plan_create(int L, double B, int J_min, int max_batch, pxm_wav_plan** out);
int pxm_wav_plan_destroy(pxm_wav_plan* plan);
int pxm_wav_plan_info(const pxm_wav_plan* plan, int* nscales_total, long long* ncoefs, long long* nscal, int* J_max,
                      long long* table_bytes);
int pxm_wav_plan_bandlimits(const pxm_wav_plan* plan, int* out, int cap);
/* bytes of this rank's Legendre tables by family: synthesis {Lambda_L, W_j kappa_j}, analysis {W_L, Lambda_j kappa_j} */
int pxm_wav_plan_table_bytes_by_family(const pxm_wav_plan* plan, long long* out4);
/* bytes of the Gram table G^m = (2L-1) Lambda^T Lambda behind pxm_wav_gram_gradient (0 until its first call builds it) */
int pxm_wav_plan_gram_bytes(const pxm_wav_plan* plan, long long* out);
/* per-ring weights w_t of the Gram table, G^m = (2L-1) Lambda^T diag(w) Lambda: the Gram form for a noise level that is
 * constant along every ring (pxmcmc/forward.py:74-88 with the per-ring sigma of experiments/earthtopography/main.py:92-94);
 * pxm_wav_gram_gradient then takes d_b = pxm_wav_pix_to_harm_adjoint(w . data).  h_w: L host doubles, NULL: w = 1. */
int pxm_wav_set_gram_weights(pxm_wav_plan* plan, const double* h_w, int n);
int pxm_wav_synthesis(pxm_wav_plan* plan, const void* d_coef, void* d_pix, int nbatch, void* stream);
int pxm_wav_synthesis_adjoint(pxm_wav_plan* plan, const void* d_pix, void* d_coef, int nbatch, void* stream);
int pxm_wav_analysis(pxm_wav_plan* plan, const void* d_pix, void* d_coef, int nbatch, void* stream);
int pxm_wav_analysis_adjoint(pxm_wav_plan* plan, const void* d_coef, void* d_pix, int nbatch, void* stream);
/* Harmonic-space ends of the synthesis pair: synthesis without its last A_inv(L,0) (output f_lm, [nbatch][L^2],
 * index l^2+l+m) and synthesis_adjoint without its first A_inv^dagger (input f_lm).  A measurement that starts with
 * A_fwd(L,0) (WeakLensing, pxmcmc/measurements.py:223,239) composes with them exactly (A_fwd o A_inv = I on f_lm). */
int pxm_wav_synthesis_harmonic(pxm_wav_plan* plan, const void* d_coef, void* d_flm, int nbatch, void* stream);
int pxm_wav_synthesis_adjoint_harmonic(pxm_wav_plan* plan, const void* d_flm, void* d_coef, int nbatch, void* stream);
/* Ring-Fourier form of the predictions: ForwardOperator with an Identity measurement behind a wavelet synthesis
 * (pxmcmc/forward.py:60-72, pxmcmc/measurements.py:43-56).  Psi ends with the ring FFT F_m(theta_t) -> pixels and the next
 * gradient starts with the ring FFT pixels -> F_m(theta_t); the DFT of length n = 2L-1 is invertible, so for an inverse
 * covariance that is constant along every ring the pair cancels:  FFT_in(ic (FFT_out(F) - data)) = ic_t (n F - FFT_in(data)).
 * Ring array = the plan's layout [slot |m| < L][ring/4][col][ring%4] doubles, col = 4 chain + 2 (m<0) + (im);
 * pxm_wav_ring_doubles: its size (all chains of the plan).  _to_ring: synthesis without its last stage; _from_ring:
 * synthesis_adjoint without its first stage; ring_to_pix / pix_to_ring: those stages alone; ring_resid:
 * out = ic[t] ((2L-1) pred - data), data = pix_to_ring(data) with nbatch = 1, d_ic = L complex values (one per ring).
 * Not available on m-sharded plans. */
long long pxm_wav_ring_doubles(const pxm_wav_plan* plan);
int pxm_wav_synthesis_to_ring(pxm_wav_plan* plan, const void* d_coef, double* d_ring, int nbatch, void* stream);
int pxm_wav_synthesis_adjoint_from_ring(pxm_wav_plan* plan, const double* d_ring, void* d_coef, int nbatch, void* stream);
int pxm_wav_ring_to_pix(pxm_wav_plan* plan, const double* d_ring, void* d_pix, int nbatch, void* stream);
int pxm_wav_pix_to_ring(pxm_wav_plan* plan, const void* d_pix, double* d_ring, int nbatch, void* stream);
int pxm_wav_ring_resid(pxm_wav_plan* plan, const double* d_ring_pred, const double* d_ring_data, const void* d_ic,
                       double* d_ring_out, int nbatch, void* stream);
/* Harmonic form of the same predictions, for an inverse covariance that is ONE (complex) constant over the sphere: per order m
 * the ring-space composition is g = ic Lambda^T ((2L-1) Lambda f - D) = ic (G f - b) with the Gram matrix
 * G^m = (2L-1) Lambda^T Lambda ((L-|m|)^2 entries, generated once per plan) and b = A_inv^dagger(data): one contraction
 * with a third fewer entries replaces the two full-L contractions of pxm_wav_synthesis_to_ring + _from_ring, and the
 * predictions are carried as f_lm.  Harmonic arrays: the plan's layout, concatenated slots |m| < L of [rows/4][col][rows%4]
 * doubles, rows = l - |m| padded to 64, col = 4 chain + 2 (m<0) + (im); pxm_wav_harm_doubles = its size.
 * _to_harm: synthesis stopped at f_lm; gram_gradient: coefficients of Psi^dagger ic (Psi X - data) from f = _to_harm(X) and
 * d_b = pxm_wav_pix_to_harm_adjoint(data, nbatch = 1); harm_to_pix: the pixels of f.  Not on m-sharded plans. */
long long pxm_wav_harm_doubles(const pxm_wav_plan* plan);
int pxm_wav_synthesis_to_harm(pxm_wav_plan* plan, const void* d_coef, double* d_harm, int nbatch, void* stream);
int pxm_wav_gram_gradient(pxm_wav_plan* plan, const double* d_harm, const double* d_b, double ic_re, double ic_im, void* d_coef,
                          int nbatch, void* stream);
int pxm_wav_harm_to_pix(pxm_wav_plan* plan, const double* d_harm, void* d_pix, int nbatch, void* stream);
int pxm_wav_pix_to_harm_adjoint(pxm_wav_plan* plan, const void* d_pix, double* d_harm, int nbatch, void* stream);
/* host-only: kappa0[L], kappa[(J-J_min+1)][L] of pys2let.wavelet_tiling
 * (pxmcmc/utils.py:117, pxmcmc/prior.py:121,132) */
int pxm_wavelet_tiling(int L, double B, int J_min, double* kappa0, double* kappa, int* J_out);

/* ---- HEALPix RING maps <-> harmonic coefficients (data preparation, once per run) ---
 * healpy.alm2map / healpy.map2alm as wrapped by utils.alm2map / utils.map2alm
 * (pxmcmc/utils.py:106-113; experiments/earthtopography/main.py:80-82,
 * experiments/weaklensing/main.py:31-37).  L = lmax + 1; flm: [L*L] complex with the
 * ssht index l*l+l+m (pys2let.lm_hp2lm converts from healpy's m >= 0 storage);
 * map: [12 nside^2] complex (a real map has zero imaginary part).
 * pxm_hpx_alm2map:          map[p] = sum_lm flm Y_lm(p)
 * pxm_hpx_map2alm_adjoint:  flm    = sum_p  conj(Y_lm(p)) map[p]     (no weights)
 * healpy.map2alm(iter=k) = (4 pi / npix) x adjoint, then k Jacobi refinements
 * alm += (4 pi / npix) adjoint(map - alm2map(alm)), assembled by the host layer. */
int pxm_hpx_plan_create(int nside, int L, pxm_hpx_plan** out);
int pxm_hpx_plan_destroy(pxm_hpx_plan* plan);
int pxm_hpx_alm2map(pxm_hpx_plan* plan, const void* d_flm, void* d_map, void* stream);
int pxm_hpx_map2alm_adjoint(pxm_hpx_plan* plan, const void* d_map, void* d_flm, void* stream);

/* ---- m-sharded plans: one chain, bandlimit too large or too slow for one GPU ---
 * (no counterpart in the reference, which is single-process; SURVEY.md 8e-2.)
 * One process per GPU, `world` <= 8 ranks on one NVLink/NVSwitch node.  Rank r
 * owns the azimuthal orders |m| with pxm_shard_owner_of_m(|m|) == r (harmonic
 * space, Legendre tables: 1/world of the memory) and, of every ring grid, the
 * rows [t0, t1) of pxm_*_plan_local_rows (pixel / coefficient space: every
 * pixel-side pointer of the transform calls then addresses those LOCAL rows
 * only, scale maps concatenated in the usual order).  flm arrays keep their
 * full length; a rank reads and writes only the orders it owns (others: 0).
 * The theta<->m transposition is fused into the Legendre contractions: the
 * contraction over l stores each 64-ring output tile straight into the ring
 * buffer of the rank owning those rings, the contraction over rings pulls ring
 * blocks from their owners with the same bulk copies it uses locally; a
 * flag-based peer barrier separates the local and the peer-access phases.
 * Set-up: create -> exchange pxm_*_plan_workspace addresses (same process:
 * directly; other processes: pxm_ipc_export / pxm_ipc_open) -> attach.  All
 * ranks must issue the same sequence of transform calls. */
int pxm_sht_plan_create_sharded(int L, int spin, int max_batch, int rank, int world, pxm_sht_plan** out);
int pxm_wav_plan_create_sharded(int L, double B, int J_min, int max_batch, int rank, int world, pxm_wav_plan** out);
int pxm_sht_plan_prepare(pxm_sht_plan* plan); /* build all tables now (mandatory before a sharded plan is used) */
int pxm_wav_plan_prepare(pxm_wav_plan* plan);
void* pxm_sht_plan_workspace(pxm_sht_plan* plan, size_t* bytes);
void* pxm_wav_plan_workspace(pxm_wav_plan* plan, size_t* bytes);
int pxm_sht_plan_attach(pxm_sht_plan* plan, void* const* peer_workspaces /* [world]; own entry ignored */);
int pxm_wav_plan_attach(pxm_wav_plan* plan, void* const* peer_workspaces);
int pxm_sht_plan_local_rows(const pxm_sht_plan* plan, int* t0, int* t1);
int pxm_wav_plan_local_rows(const pxm_wav_plan* plan, int* t0, int* t1 /* [nscales_total + 1], last = pixel map */,
                            long long* ncoefs_local, long long* npix_local);
int pxm_sht_plan_barrier_status(pxm_sht_plan* plan, long long* failed_epoch /* 0 = no time-out */);
int pxm_wav_plan_barrier_status(pxm_wav_plan* plan, long long* failed_epoch);
int pxm_shard_owner_of_m(int abs_m, int world);                                        /* host only */
int pxm_shard_ring_range(int ell, int rot, int rank, int world, int* t0, int* t1);      /* host only */
int pxm_ipc_export(const void* d_ptr, void* handle64);
int pxm_ipc_open(const void* handle64, void** d_ptr);
int pxm_ipc_close(void* d_ptr);

/* ---- fused elementwise passes ---------------------------------------------
 * pxm_soft: utils.soft (pxmcmc/utils.py:55-67); T vector (d_T, length n) or scalar. */
int pxm_soft(int is_complex, const void* d_x, const double* d_T, double T_scalar, void* d_out, long long n,
             long long nchains, void* stream);
/* pxm_myula_update: MYULA.chain_step (pxmcmc/mcmc.py:185-201) fused with the
 * synthesis prox (pxmcmc/prior.py:49-50) when d_prox == NULL.
 * noise_mode 0: none; 1: injected d_w_re (+ d_w_im); 2/3: Philox4x32-10 real/complex.
 * Real chain pairs (two real-valued chains packed as the real and imaginary part of one complex chain; every linear
 * operator of the path is complex-linear and maps real fields to real fields, so the parts never mix; the threshold
 * acts on each part): 4: Philox, packed chain c draws streams stream0 + 2c (real part) and stream0 + 2c + 1; 5: injected
 * d_w_re / d_w_im = the two chains' noise. */
int pxm_myula_update(const void* d_X, const void* d_prox, const void* d_gradg, const double* d_T, double T_scalar,
                     const double* d_w_re, const double* d_w_im, void* d_Xout, void* d_prox_out, long long n,
                     long long nchains, double delta, double lmda, int noise_mode, unsigned long long seed,
                     unsigned long long step, unsigned int stream0, void* stream);
/* CUDA-graph friendly variant: the Philox step is read from *d_step (device), so one captured
 * iteration can be replayed; pxm_counter_add advances it from inside the graph. */
int pxm_myula_update_dstep(const void* d_X, const void* d_prox, const void* d_gradg, const double* d_T, double T_scalar,
                           void* d_Xout, void* d_prox_out, long long n, long long nchains, double delta, double lmda,
                           int noise_mode, unsigned long long seed, const unsigned long long* d_step,
                           unsigned int stream0, void* stream);
int pxm_counter_add(unsigned long long* d_counter, unsigned long long inc, void* stream);
/* d_out[chain][n] <- N(0,1) from the Philox stream (seed, stream0 + chain, step); d_step != NULL: the step is read from
 * the device (CUDA-graph replays).  The numbers the update kernel draws in its real-noise mode (SKROCK's Z, mcmc.py:344). */
int pxm_philox_normal(double* d_out, long long n, long long nchains, unsigned long long seed, unsigned long long step,
                      const unsigned long long* d_step, unsigned int stream0, void* stream);
/* PxMALA (pxmcmc/mcmc.py:218-289) without a host round trip per iteration.  d_state: 16 doubles PER CHAIN
 *   {delta, 1-delta/lmda, delta/lmda, sqrt(2 delta), log pi(Xc) re, im, L2(Xc) re, im, prior(Xc), accepted, log u,
 *    log alpha re, im, iteration, Philox step, -}
 * (every chain tunes its own step size; chain c draws its uniform from the Philox stream stream_id + c).
 * pxm_myula_update_dpar / pxm_reduce_dpar: the proposal and the kind-2 reduction with the step size read from
 * d_state; pxm_pxmala_accept: log alpha from the four reductions, uniform from the step's Philox stream, decision,
 * traces (acceptances int8[i], deltas[i+1]) and -- tune != 0 -- the new step size, all written on the device;
 * pxm_select_if: dst_k <- src_k (complex arrays) when *d_flag != 0 (the accepted proposal becomes the state).
 * CUDA-graph form: step = 0 (update) and i < 0 (accept) make the kernels take the Philox step and the iteration index
 * from d_state[14] and d_state[13]; pxm_pxmala_accept then advances both. */
int pxm_myula_update_dpar(const void* d_X, const void* d_prox, const void* d_gradg, const double* d_T, double T_scalar,
                          void* d_Xout, void* d_prox_out, long long n, long long nchains, const double* d_par,
                          int noise_mode, unsigned long long seed, unsigned long long step, unsigned int stream0,
                          void* stream);
int pxm_reduce_dpar(int kind, const void* a, const void* b, const void* c, const void* d, const double* w,
                    const double* d_par, double lmda, long long n, long long nchains, void* d_partial, void* d_out,
                    void* stream);
int pxm_pxmala_accept(double* d_state, const void* d_s1, const void* d_s2, const void* d_L2p, const void* d_priorp,
                      double mu, double lmda, int tune, long long i, unsigned long long seed, unsigned long long step,
                      unsigned int stream_id, signed char* d_acc_trace /* [nchains][trace_stride] */,
                      double* d_delta_trace /* [nchains][trace_stride + 1] */, long long trace_stride, int nchains,
                      void* stream);
int pxm_select_if(const double* d_flag /* chain c: d_flag[flag_stride c] */, long long flag_stride, long long nchains,
                  void* const* d_dst, const void* const* d_src, const long long* counts /* elements per chain */,
                  int narrays, void* stream);
/* pxm_resid_invcov: invcov @ (preds - data) of ForwardOperator._gradg_analysis
 * (pxmcmc/forward.py:66-69) for a diagonal, possibly complex, inverse covariance. */
int pxm_resid_invcov(const void* d_preds, const void* d_data, const void* d_invcov, void* d_out, long long n,
                     long long nchains, void* stream);
/* pxm_reduce: per-chain deterministic reductions -> d_out[nchains] complex.
 *  kind 0: sum |w x|        (L1.prior, pxmcmc/prior.py:28-35,83-84)   a=x, w=weights or NULL
 *  kind 1: vdot(d, ic*d), d=data-preds (PxMCMC.logpi, pxmcmc/mcmc.py:78-79)   a=preds b=data c=invcov
 *  kind 2: sum (X2-X1-(delta/2) glp)^2 (PxMALA.calc_logtransition, pxmcmc/mcmc.py:285-289) a=X1 b=X2 c=prox d=gradg
 * d_partial: scratch of nchains*pxm_reduce_scratch_elems() complex. */
int pxm_reduce_scratch_elems(void);
int pxm_reduce(int kind, const void* a, const void* b, const void* c, const void* d, const double* w, double delta,
               double lmda, long long n, long long nchains, void* d_partial, void* d_out, void* stream);
/* pxm_lincomb: out = c0 + sum_k coef_k x_k (+ cz*z, z real): the analysis prox assembly (pxmcmc/prior.py:52-53);
 * SKROCK's stages run pxm_skrock_stage. */
int pxm_lincomb(int nx, const void* const* d_xs, const double* coefs, const double* d_z, double cz, double c0,
                void* d_out, long long total, void* stream);
/* pxm_gradlogpi: PxMCMC._gradlogpi (pxmcmc/mcmc.py:84-89): -((X - P)/lmda) - gradg with
 * P = soft(X, T) when d_prox == NULL. */
int pxm_gradlogpi(const void* d_X, const void* d_prox, const double* d_T, double T_scalar, const void* d_gradg,
                  double lmda, void* d_out, long long n, long long nchains, void* stream);
/* SKROCK stages (pxmcmc/mcmc.py:338-368; Abdulle, Almuslimani & Vilmart 2018), one kernel each.
 * pxm_skrock_shift: Y = X + c Z.
 * pxm_skrock_stage: out = a g + b U + c V + c0 (+ e Z), g = -((P - prox(P))/lmda) - gradg, prox = soft(P, T) when
 *   d_prox == NULL (T: d_T of length n, or T_scalar).  With noise (noise_mode != 0) P = U + c_shift Z is recomputed in
 *   registers (stage 1: U = X, d_V = NULL, gradg of Y; Y and Z are not read back), else P = U (stage j >= 2: U = K_{j-1},
 *   V = K_{j-2}).  The sum runs in the order of the reference's stage expressions, every product rounded: U, g, Z when
 *   d_V == NULL, else g, U, V; then c0 (added to the real part).  The reference scheme (b = nu_j, c = -1, c0 = k_j)
 *   equals pxm_gradlogpi + pxm_lincomb bit for bit.  d_out may be d_U or d_V.
 * Z: noise_mode 1 injected real d_z_re; 2 injected d_z_re + i d_z_im; 3 the Philox normals pxm_philox_normal draws at
 *   (seed, stream0 + chain, step); 4 complex Philox: one draw of 2n normals per chain, the first n the real and the
 *   last n the imaginary parts.  d_step != NULL: the step is read from the device (CUDA-graph replays).
 * All arrays [nchains][n]; the chain comes from the launch grid. */
int pxm_skrock_shift(const void* d_X, double c, const double* d_z_re, const double* d_z_im, int noise_mode,
                     unsigned long long seed, unsigned long long step, const unsigned long long* d_step,
                     unsigned int stream0, void* d_Y, long long n, long long nchains, void* stream);
int pxm_skrock_stage(const void* d_U, const void* d_V, const void* d_gradg, const void* d_prox, const double* d_T,
                     double T_scalar, double lmda, double a, double b, double c, double c0, double c_shift, double e,
                     const double* d_z_re, const double* d_z_im, int noise_mode, unsigned long long seed,
                     unsigned long long step, const unsigned long long* d_step, unsigned int stream0, void* d_out,
                     long long n, long long nchains, void* stream);
/* pxm_fista_update: one FISTA iteration (Beck & Teboulle 2009) of the synthesis-setting MAP for every chain:
 *   x_{k+1} = soft(y_k - t gradg, T_scale T),  y_{k+1} = x_{k+1} + beta_k (x_{k+1} - x_k),
 *   beta_k = (tau_k - 1)/tau_{k+1},  tau_{k+1} = (1 + sqrt(1 + 4 tau_k^2))/2
 * with gradg the data-fidelity gradient at y_k (T: d_T of length n, or T_scalar).  d_state = {k, tau_k} (doubles;
 * start from {0, 1}) is read on the device and advanced by the call, so a captured block of iterations replays
 * unchanged.  d_hist[cap][nchains][2] receives, in slot k mod cap, |x_{k+1} - x_k|^2 and |x_{k+1}|^2 of every chain
 * (deterministic two-level sums).  d_x_out / d_y_out may be d_x / d_y.  d_partial: scratch of
 * nchains*pxm_reduce_scratch_elems() complex.  All vectors [nchains][n], nchains <= 65535. */
int pxm_fista_update(const void* d_y, const void* d_gradg, const void* d_x, const double* d_T, double T_scalar,
                     double T_scale, double t, double* d_state, void* d_x_out, void* d_y_out, double* d_hist,
                     long long cap, long long n, long long nchains, void* d_partial, void* stream);
/* masked gather / zero-filled scatter with optional per-datum weight:
 * WeakLensing.mask_forward/mask_adjoint/cov_weight (pxmcmc/measurements.py:242-304). */
int pxm_masked_gather(const void* d_full, const int* d_idx, const double* d_w, void* d_sel, long long nsel,
                      long long nfull, long long nchains, void* stream);
int pxm_masked_scatter(const void* d_sel, const int* d_idx, const double* d_w, void* d_full, long long nsel,
                       long long nfull, long long nchains, void* stream);
int pxm_real_to_complex(const double* d_x, void* d_out, long long total, void* stream);

/* ---- sparse path operator ---------------------------------------------------
 * PathIntegral.forward / adjoint (pxmcmc/measurements.py:75-83): CSR with real
 * float64 values times complex vectors; pass the CSR of A^T for the adjoint. */
int pxm_csr_spmv(const int* d_indptr, const int* d_indices, const double* d_vals, const void* d_x, void* d_y,
                 int nrows, long long ncols, long long nchains, void* stream);

/* ---- great-circle path matrix (data preparation of the phase-velocity experiment) ----------
 * Replaces greatcirclepaths.GreatCirclePath(start, stop, "MW", L=L, weighting="average", latlon=True)
 * .get_points(points_per_rad).fill() of experiments/phasevel/main.py:40-47.  d_start / d_stop: [npaths][2]
 * (latitude, longitude) in degrees.  pxm_gc_count_points: points per path = max(2, ceil(points_per_rad *
 * distance)).  pxm_gc_rasterise: one CTA per path; row r of d_cols / d_w ([npaths][cap], cap a power of two >=
 * every point count) receives the sorted distinct MW pixels t (2L-1) + p the path visits and their share of the
 * path's points (a row sums to one), padded with -1; d_nnz[r] = number of pixels.  pxm_gc_compact packs the
 * padded rows into CSR arrays given the exclusive prefix sum d_indptr[npaths + 1] of d_nnz. */
int pxm_gc_count_points(const double* d_start, const double* d_stop, long long npaths, double points_per_rad,
                        int* d_npoints, void* stream);
int pxm_gc_rasterise(const double* d_start, const double* d_stop, long long npaths, int L, double points_per_rad,
                     int cap, int* d_cols, double* d_w, int* d_nnz, void* stream);
int pxm_gc_compact(const long long* d_indptr, const int* d_cols, const double* d_w, int cap, long long npaths,
                   int* d_indices, double* d_data, void* stream);

/* ---- uncertainty quantification ---------------------------------------------
 * credible_interval_range (pxmcmc/uncertainty.py:7-16): two quantiles of every column of a stored
 * chain [nsamples][ld] of doubles, numpy's default "linear" method.  The caller passes, for each
 * quantile q, the lower order statistic lo = floor(v) and the weight gamma = v - lo of the virtual
 * index v = (n - 1) q (numpy's own expression, evaluated on the host); out = lerp(x[lo],
 * x[lo+1], gamma) evaluated as numpy's _lerp does.  nsamples <= pxm_quantile_columns_max_samples(). */
int pxm_quantile_columns(const double* d_chain, long long nsamples, long long ncols, long long ld, long long lo_a,
                         double gamma_a, long long lo_b, double gamma_b, double* d_out_a, double* d_out_b, void* stream);
int pxm_quantile_columns_max_samples(void);

/* ---- streaming posterior summaries --------------------------------------------
 * (no counterpart in the reference, which stores every tracked sample.)  Per-element running moments of a batch of
 * chains on the tracking grid, from which the pooled mean and variance, split-R-hat and a batch-means ESS follow
 * without storing samples (DESIGN.md 7b).  d_x: the chains' state or predictions, complex [nchains][n].
 * mode 0: the real part of every chain; 1: real and imaginary part as two components; 2: packed real chain pairs
 * (real part = logical chain 2c, imaginary part = 2c + 1).  A slot is one component of one logical chain:
 * mode 0 slot = c, modes 1 and 2 slot = 2c + part; nslots = nchains (mode 0) or 2 nchains.
 * Accumulator: 8 fields, each [nslots][n] doubles, in this order: mean and M2 of half A (samples [0, h)), middle
 * sample (j = h when nsamples is odd), mean and M2 of half B ([nsamples - h, nsamples)), open batch sum, mean and M2
 * of the batch means; h = nsamples / 2, batch size b = max(1, floor(sqrt nsamples)), a = nsamples / b batches.
 * pxm_stats_accumulator_doubles: its size (-1 on a bad argument).  pxm_stats_reset: zero it.
 * pxm_stats_accumulate: push sample j of every chain (d_j == NULL) or sample d_j[c] of chain c (< 0: chain c takes no
 * sample now); 0 <= j < nsamples.  Every sample index of a chain is pushed once, in increasing order.
 * pxm_stats_partials: the partial record, 10 fields each [ncomp][n] doubles (ncomp = 2 in mode 1, else 1), over the
 * logical chains in order: half-chain count, mean and M2 of the half-chain means, sum of the half-chain variances
 * (ddof 1); sample count, pooled mean, pooled M2; batch count, mean and M2 of the batch means.  Records of disjoint
 * chain groups combine with Chan's rule.  d_chain_mean / d_chain_var (may be NULL): [nslots][n] per-chain mean and
 * variance (ddof 1). */
long long pxm_stats_accumulator_doubles(long long n, long long nchains, int mode);
int pxm_stats_reset(double* d_acc, long long n, long long nchains, int mode, void* stream);
int pxm_stats_accumulate(double* d_acc, const void* d_x, long long n, long long nchains, int mode, long long nsamples,
                         long long j, const long long* d_j, void* stream);
int pxm_stats_partials(const double* d_acc, long long n, long long nchains, int mode, long long nsamples,
                       double* d_partial, double* d_chain_mean, double* d_chain_var, void* stream);

/* ---- streaming credible intervals ----------------------------------------------
 * (pxmcmc/uncertainty.py:7-16 takes them from the stored chain.)  numpy's linear quantiles at q_a and q_b of the
 * npooled = N samples that the logical chains push over a run, per element and component, without storing them
 * (DESIGN.md 7b).  lo_a, gamma_a, lo_b, gamma_b: numpy's virtual indices of q_a and q_b for N values (0 <= lo < N).
 * d_x, modes 0 / 1 / 2 and d_j as in pxm_stats_accumulate.  The state keeps the K_lo = min(lo_a + 2, N) smallest and
 * the K_hi = N - lo_b largest values of every column t < T (T = 2 n in mode 1, column t = part t / n of element
 * t % n; T = n otherwise): the lower heaps [T][K_lo], the upper heaps [T][K_hi], then a NaN flag row [T] (doubles).
 * pxm_credible_state_doubles: its size (-1 on a bad argument).  pxm_credible_reset: zero it.
 * pxm_credible_push: offer one sample of every chain (d_j == NULL) or of the chains with d_j[c] >= 0 (the value of
 * d_j[c] is not read otherwise); `count` = samples pooled per column before this push (the chains' logical parts
 * included: 2 per active chain in mode 2).  Pushes come in order and no more than N samples are pooled.
 * pxm_credible_finalize: after exactly N pooled samples, d_lower / d_upper [T] = numpy's quantiles at q_a / q_b,
 * lerp(x(lo), x(min(lo + 1, N - 1)), gamma) evaluated as numpy's _lerp does; NaN where a NaN was pushed. */
long long pxm_credible_state_doubles(long long n, int mode, long long npooled, long long lo_a, long long lo_b);
int pxm_credible_reset(double* d_state, long long n, int mode, long long npooled, long long lo_a, long long lo_b,
                       void* stream);
int pxm_credible_push(double* d_state, const void* d_x, long long n, long long nchains, int mode, long long npooled,
                      long long lo_a, long long lo_b, long long count, const long long* d_j, void* stream);
int pxm_credible_finalize(const double* d_state, long long n, int mode, long long npooled, long long lo_a,
                          double gamma_a, long long lo_b, double gamma_b, double* d_lower, double* d_upper,
                          void* stream);

/* ---- rank-normalised convergence diagnostics of stored chains ---------------------
 * (no counterpart in the reference.)  Column col < ncols of d_chain holds the S = m n samples of m chains, x[c][i] =
 * d_chain[(c n + i) ld + col] (the layout of a tracked [nchains][nsamples][nparams] array).  Per column, as defined in
 * DESIGN.md 7b (Vehtari et al. 2021; ArviZ rhat(method="rank"), ess(method="bulk" | "tail")):
 *   d_rhat[col]      rank-normalised split-R-hat, the larger of the bulk and the folded (|x - median|) R; NaN when
 *                    either is NaN;
 *   d_ess_bulk[col]  ESS of the rank-normalised split chains;
 *   d_ess_tail[col]  the smaller ESS of the split indicators 1[x <= q05] and 1[x <= q95] (numpy's linear quantiles
 *                    over all S samples).
 * All three are NaN for a column with a non-finite sample, and for every column when n < 4.  S <=
 * pxm_quantile_columns_max_samples().  d_scratch: pxm_rank_diagnostics_scratch_doubles(m, n, ncols) doubles (the
 * columns, transposed); the query returns -1 on a bad argument. */
long long pxm_rank_diagnostics_scratch_doubles(long long m, long long n, long long ncols);
int pxm_rank_diagnostics(const double* d_chain, long long m, long long n, long long ncols, long long ld,
                         double* d_scratch, double* d_rhat, double* d_ess_bulk, double* d_ess_tail, void* stream);

/* ---- measurement aids (bench.py) ---------------------------------------------
 * pxm_profile_begin/end bracket a region in which every library call records a
 * CUDA-event pair on its launching stream; end() returns the summed device time
 * and the number of timed calls per kernel class: 0 Legendre contraction,
 * 1 ring FFT, 2 elementwise/reduction/sparse.  pxm_launch_count: kernels
 * launched by the library since load. */
int pxm_profile_begin(int max_events);
int pxm_profile_end(double* ms_by_kind, long long* count_by_kind);
long long pxm_launch_count(void);

/* ---- debugging aids (tests only) ---------------------------------------------- */
int pxm_debug_set_naive(int on); /* route Legendre contractions through the plain kernel */
int pxm_debug_set_fft_multipass(int mode); /* ring FFT kernel choice: 0 by grid size (default), 1 always the multi-pass kernel, 2 always the two-pass kernel (Bluestein lengths <= 1024), 3 two-pass with the persistent TMA-staged kernel for lengths 512 / 1024 whatever the grid size (the one-CTA-per-SM kernel pxm_ring_fft6_kernel, as mode 0 picks for large grids); 4 as 3 with the two-CTA kernel pxm_ring_fft3_kernel it replaced */
int pxm_debug_wigner_row_host(int grid_L, int ring, int m, int spin, int lmax, double* out); /* host, no GPU */

#ifdef __cplusplus
}
#endif
#endif

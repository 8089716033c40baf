// Host-side plans and the C ABI (include/pxmcmc_b200.h).
//
// A plan owns: the Legendre table arena, the ring-FFT twiddle arena, a
// zero-initialised workspace (ring-Fourier and harmonic buffers in the
// k4-interleaved layout) and the work-item descriptors of every operator.
// Every transform is the same four-stage pipeline
//     [ring FFT in] -> [DMMA contraction over rings] -> [DMMA contraction over l] -> [ring FFT out]
// with stages dropped at the harmonic-space boundary of the pyssht-level calls.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/pxmcmc_b200.h"
#include "pxm_plan.h"

// ------------------------------------------------------------------ errors
static thread_local std::string g_err;
void pxm_set_error(const std::string& msg) { g_err = msg; }
static int g_naive = 0;
int pxm_debug_naive() { return g_naive; }
long long g_pxm_launches = 0;

// ---- optional per-kernel-class device timing (CUDA events on the launching stream) ----
// kinds: 0 Legendre contraction, 1 ring FFT, 2 elementwise/reduction/sparse
namespace {
struct ProfEv {
  cudaEvent_t e0, e1;
  int kind;
};
bool g_prof_on = false;
std::vector<ProfEv> g_prof_pool;
size_t g_prof_used = 0;
struct ProfScope {
  cudaStream_t st;
  ProfEv* ev = nullptr;
  ProfScope(int kind, cudaStream_t s) : st(s) {
    if (!g_prof_on || g_prof_used >= g_prof_pool.size()) return;
    ev = &g_prof_pool[g_prof_used++];
    ev->kind = kind;
    cudaEventRecord(ev->e0, st);
  }
  ~ProfScope() {
    if (ev) cudaEventRecord(ev->e1, st);
  }
};
}  // namespace

namespace {

typedef unsigned long long ull;

// first doubles of every workspace: barrier flags of an m-sharded plan (one 64-bit epoch per
// peer) and, at word PXM_WS_ERR, the barrier's time-out flag
constexpr ull PXM_WS_RESERVED = 512;
constexpr int PXM_WS_ERR = 64;
constexpr int PXM_WS_EPOCH = 65;  // this rank's barrier count (device-resident: barriers replay inside CUDA graphs)

struct Shard {
  int rank = 0, world = 1;
};

struct RingBuf {
  int ell = 0;
  bool paired = true;
  int nslots = 0;
  int rows = 0;         // rings of the grid (= ell on MW sampling; 4 nside - 1 on HEALPix)
  int rot = 0;          // rotation of the ring-block ownership (scale index)
  int t0 = 0, t1 = 0;   // rings owned by this rank
  ull off = 0;          // doubles into the workspace
  ull slot_stride = 0;  // doubles
  int slot_of(int m) const { return paired ? std::abs(m) : m + ell - 1; }
  ull doubles() const { return (ull)nslots * slot_stride; }
};

struct HarmBuf {
  int L = 0;
  bool paired = true;
  std::vector<ull> slot_off;  // absolute doubles into the workspace
  PxmDevVec<ull> d_slot_off;
  ull total = 0;
  int slot_of(int m) const { return paired ? std::abs(m) : m + L - 1; }
};

void make_ring(RingBuf& R, int ell, bool paired, int nld, ull& cursor, const Shard& sh = Shard(), int rot = 0) {
  R.ell = ell;
  R.rows = ell;
  R.paired = paired;
  R.rot = rot;
  pxm_ring_range(ell, rot, sh.rank, sh.world, &R.t0, &R.t1);
  R.nslots = paired ? ell : 2 * ell - 1;
  R.slot_stride = (ull)pxm_round_up(ell, 32) * nld;
  R.off = cursor;
  cursor += R.doubles();
}

void make_harm(HarmBuf& H, int L, bool paired, int nld, ull& cursor) {
  H.L = L;
  H.paired = paired;
  const int ns = paired ? L : 2 * L - 1;
  H.slot_off.resize(ns);
  ull c = cursor;
  for (int s = 0; s < ns; ++s) {
    const int am = paired ? s : std::abs(s - (L - 1));
    H.slot_off[s] = c;
    c += (ull)pxm_round_up(L - am, 64) * nld;
  }
  H.total = c - cursor;
  cursor = c;
}

struct TableRef {
  PxmTableLayout T;
  ull base = 0;  // doubles into the plan's table arena (T.tile_off are relative to 0 with base folded in)
  int family = 0;  // 0 lambda, 1 W
  std::vector<double> g;
  bool built = false;
};

struct Stage {
  std::vector<PxmLegItem> items;
  std::vector<PxmLegSeg> segs;
  PxmDevVec<PxmLegItem> d_items;
  PxmDevVec<PxmLegSeg> d_segs;
  int orient = 0;
  int upload() {
    // heaviest items first: the hardware block scheduler then balances the triangular workload
    std::vector<int> order(items.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return items[a].cost > items[b].cost; });
    std::vector<PxmLegItem> sorted;
    for (int i : order) sorted.push_back(items[i]);
    items.swap(sorted);
    PXM_TRY(d_items.upload(items));
    PXM_TRY(d_segs.upload(segs));
    return PXM_OK;
  }
  void release() {
    d_items.release();
    d_segs.release();
  }
};

struct FftStage {
  std::vector<PxmFftGroup> groups;
  PxmDevVec<PxmFftGroup> d_groups;
  int ctas = 0;
  int class_mask = 0;  // kernel classes the groups need (pxm_fft_class_bit)
  void release() { d_groups.release(); }
};

// ring-FFT twiddle bookkeeping: one (chirp, bhat, tw) triple per distinct ring length
struct FftTables {
  std::map<int, PxmFftGroup> by_n;
  ull cursor = 0;  // complex elements
  void* d_arena = nullptr;
  PxmFftGroup get(int ell) {
    const int n = 2 * ell - 1;
    auto it = by_n.find(n);
    if (it != by_n.end()) return it->second;
    PxmFftGroup g = {};
    g.ell = ell;
    g.n = n;
    g.M = pxm_fft_choose_M(n, &g.logM);
    g.chirp_off = cursor;
    cursor += (ull)pxm_round_up(n, 2);
    g.bhat_off = cursor;
    cursor += g.M;
    g.tw_off = cursor;
    cursor += g.M;
    g.bhat2_off = cursor;
    cursor += g.M;
    g.tw2_off = cursor;
    if (g.logM == 9 || g.logM == 10) cursor += 2ULL * g.M;
    by_n[n] = g;
    return g;
  }
  int finalize(cudaStream_t st) {
    std::vector<PxmFftGroup> hs;
    for (auto& kv : by_n) hs.push_back(kv.second);
    PXM_CUDA(cudaMalloc(&d_arena, std::max<ull>(cursor, 1) * 16));
    PxmDevVec<PxmFftGroup> dg;
    PXM_TRY(dg.upload(hs));
    PXM_TRY(pxm_fft_setup_tables(dg.d, hs.data(), (int)hs.size(), d_arena, st));
    PXM_CUDA(cudaStreamSynchronize(st));
    dg.release();
    return PXM_OK;
  }
  void release() {
    if (d_arena) cudaFree(d_arena);
    d_arena = nullptr;
  }
};

void add_fft_group(FftStage& S, FftTables& tabs, const RingBuf& R, ull pix_off, double scale) {
  if (R.t1 <= R.t0) return;  // this rank owns no ring of the grid
  PxmFftGroup g = tabs.get(R.ell);
  g.rings = R.t1;
  g.ring0 = R.t0;
  g.pad = pxm_fft_rings_per_cta_log(g.M);  // log2(rings per CTA)
  g.rings_per_cta = 1 << g.pad;
  g.cta_begin = S.ctas;
  g.nslots = R.nslots;
  g.paired = R.paired ? 1 : 0;
  g.scale = scale;
  g.pix_off = pix_off;
  g.f_off = R.off;
  g.slot_stride = R.slot_stride;
  S.ctas += pxm_ceil_div(R.t1 - R.t0, g.rings_per_cta);
  S.class_mask |= pxm_fft_class_bit(g.logM);
  S.groups.push_back(g);
}

int slot_index(const PxmTableLayout& T, int m) { return T.paired ? std::abs(m) : m + T.lmax - 1; }

// contraction over l:  ring buffer R  <-  table T  x  harmonic buffer H
void build_s_items(Stage& S, const TableRef& tr, const HarmBuf& H, const RingBuf& R, int nld,
                   const Shard& sh = Shard()) {
  const PxmTableLayout& T = tr.T;
  S.orient = 0;
  for (int s = 0; s < T.nslots; ++s) {
    if (T.nlb[s] == 0) continue;
    const int m = T.slot_m[s];
    const int hs = H.slot_of(m), rs = R.slot_of(m);
    for (int i = 0; 2 * i < T.ntb; ++i) {
      PxmLegSeg sg = {};
      sg.a_off = T.tile_off[s] + (ull)(2 * i) * T.nlb[s] * PXM_TILE_DOUBLES;
      sg.a_kstride = PXM_TILE_DOUBLES;
      sg.a_mstride = T.nlb[s] * PXM_TILE_DOUBLES;
      sg.mt0 = 0;
      sg.nmt = std::min(2, T.ntb - 2 * i);
      sg.nk = T.nlb[s];
      sg.b_off = H.slot_off[hs] + (ull)T.lb0[s] * PXM_TILE_L * nld;
      sg.src = sh.rank;  // harmonic coefficients of an owned order are local
      PxmLegItem it = {};
      it.c_off = R.off + (ull)rs * R.slot_stride + (ull)(64 * i) * nld;
      it.seg_begin = (int)S.segs.size();
      it.seg_count = 1;
      it.nmt_out = sg.nmt;
      it.cost = sg.nk * sg.nmt;
      it.dst = pxm_owner_of_ring_block(R.rows, i, R.rot, sh.world);  // pushed to the owner of these 64 rings
      S.segs.push_back(sg);
      S.items.push_back(it);
    }
  }
}

// Gram contraction:  harmonic buffer (same layout)  <-  G^m x harmonic buffer   (rows and columns of G relative to |m|)
void build_g_items(Stage& S, const PxmTableLayout& T, const HarmBuf& H, int nld) {
  S.orient = 0;
  for (int s = 0; s < T.nslots; ++s) {
    if (T.nlb[s] == 0) continue;
    const int m = T.slot_m[s];
    const int hs = H.slot_of(m);
    const int nrow = H.L - std::abs(m);
    for (int i = 0; 64 * i < nrow; ++i) {
      PxmLegSeg sg = {};
      sg.a_off = T.tile_off[s] + (ull)(2 * i) * T.nlb[s] * PXM_TILE_DOUBLES;
      sg.a_kstride = PXM_TILE_DOUBLES;
      sg.a_mstride = T.nlb[s] * PXM_TILE_DOUBLES;
      sg.mt0 = 0;
      sg.nmt = std::min(2, pxm_ceil_div(nrow - 64 * i, PXM_TILE_T));
      sg.nk = T.nlb[s];
      sg.b_off = H.slot_off[hs];
      sg.src = 0;
      PxmLegItem it = {};
      it.c_off = H.slot_off[hs] + (ull)(64 * i) * nld;
      it.seg_begin = (int)S.segs.size();
      it.seg_count = 1;
      it.nmt_out = sg.nmt;
      it.pad = 1;
      it.cost = sg.nk * sg.nmt;
      it.dst = 0;
      S.segs.push_back(sg);
      S.items.push_back(it);
    }
  }
}

struct ASource {
  const TableRef* tr;
  const RingBuf* R;
};

// contraction over rings:  harmonic buffer H  <-  sum over sources  table^T x ring buffer
void build_a_items(Stage& S, const std::vector<ASource>& srcs, const HarmBuf& H, int nld,
                   const Shard& sh = Shard()) {
  S.orient = 1;
  const int ns = (int)H.slot_off.size();
  for (int hs = 0; hs < ns; ++hs) {
    const int m = H.paired ? hs : hs - (H.L - 1);
    const int am = std::abs(m);
    if (pxm_owner_of_m(am, sh.world) != sh.rank) continue;
    const int nlbH = pxm_ceil_div(H.L - am, PXM_TILE_L);
    for (int lt = 0; 4 * lt < nlbH; ++lt) {
      PxmLegItem it = {};
      it.seg_begin = (int)S.segs.size();
      it.cost = 0;
      for (const ASource& src : srcs) {
        const PxmTableLayout& T = src.tr->T;
        if (am >= T.lmax) continue;
        const int s = slot_index(T, m);
        if (T.nlb[s] == 0) continue;
        const int lbA = std::max(4 * lt, T.lb0[s]), lbB = std::min(4 * lt + 4, T.lb0[s] + T.nlb[s]);
        if (lbA >= lbB) continue;
        // one segment per rank that owns part of the source rings (pulled from that rank's workspace)
        for (int q = 0; q < sh.world; ++q) {
          int qt0, qt1;
          pxm_ring_range(src.R->rows, src.R->rot, q, sh.world, &qt0, &qt1);
          if (qt1 <= qt0) continue;
          const int tb0 = qt0 / PXM_TILE_T, tb1 = pxm_ceil_div(qt1, PXM_TILE_T);
          PxmLegSeg sg = {};
          sg.a_kstride = T.nlb[s] * PXM_TILE_DOUBLES;
          sg.a_off = T.tile_off[s] + (ull)(lbA - T.lb0[s]) * PXM_TILE_DOUBLES + (ull)tb0 * sg.a_kstride;
          sg.a_mstride = PXM_TILE_DOUBLES;
          sg.mt0 = lbA - 4 * lt;
          sg.nmt = lbB - lbA;
          sg.nk = tb1 - tb0;
          sg.b_off = src.R->off + (ull)src.R->slot_of(m) * src.R->slot_stride + (ull)tb0 * PXM_TILE_T * nld;
          sg.src = q;
          it.cost += sg.nk * sg.nmt;
          S.segs.push_back(sg);
        }
      }
      it.seg_count = (int)S.segs.size() - it.seg_begin;
      it.dst = sh.rank;  // harmonic coefficients of an owned order stay local
      it.c_off = H.slot_off[hs] + (ull)(64 * lt) * nld;
      it.nmt_out = std::min(4, nlbH - 4 * lt);
      it.pad = 1;  // harmonic slots hold whole 64-row tiles: the padding rows are written (as zeros)
      S.items.push_back(it);
    }
  }
}

// ---------------------------------------------------------------- tiling
// Scale-discretised wavelet tiling (axisymmetric), restating s2let's
// s2let_tiling_axisym / phi2_s2dw that the reference reaches through
// pys2let.wavelet_tiling (/root/reference/pxmcmc/utils.py:117, prior.py:121,132).
double f_s2dw(double k, double B) {
  const double t = (k - (1.0 / B)) * (2.0 * B / (B - 1.0)) - 1.0;
  return std::exp(-2.0 / (1.0 - t * t)) / k;
}
double quadtrap(double a, double b, int n, double B) {
  if (a == b) return 0.0;
  const double h = (b - a) / n;
  double sum = 0.0;
  for (int i = 0; i < n; ++i) {
    const double f1 = f_s2dw(a + i * h, B), f2 = f_s2dw(a + (i + 1) * h, B);
    if (std::isfinite(f1) && std::isfinite(f2)) sum += ((f1 + f2) * h) / 2.0;
  }
  return sum;
}
int j_max(int L, double B) { return (int)std::ceil(std::log((double)L) / std::log(B)); }

struct Tiling {
  int J = 0;
  std::vector<int> bandlimits;                // scaling first, then j = J_min..J
  std::vector<std::vector<double>> kernels;   // kappa0, kappa_j  (length L each)
};

Tiling make_tiling(int L, double B, int J_min) {
  Tiling t;
  t.J = j_max(L, B);
  const int J = t.J, n = 300;
  const double norm = quadtrap(1.0 / B, 1.0, n, B);
  std::vector<std::vector<double>> phi2(J + 2, std::vector<double>(L, 0.0));
  for (int j = 0; j <= J + 1; ++j)
    for (int l = 0; l < L; ++l) {
      if (l < std::pow(B, j - 1))
        phi2[j][l] = 1.0;
      else if (l > std::pow(B, j))
        phi2[j][l] = 0.0;
      else
        phi2[j][l] = quadtrap((double)l / std::pow(B, j), 1.0, n, B) / norm;
    }
  t.bandlimits.push_back(std::min((int)std::ceil(std::pow(B, J_min)), L));
  std::vector<double> k0(L);
  for (int l = 0; l < L; ++l) k0[l] = std::sqrt(phi2[J_min][l]);
  t.kernels.push_back(k0);
  for (int j = J_min; j <= J; ++j) {
    std::vector<double> k(L);
    for (int l = 0; l < L; ++l) {
      const double d = phi2[j + 1][l] - phi2[j][l];
      k[l] = d > 0.0 ? std::sqrt(d) : 0.0;
    }
    t.bandlimits.push_back(std::min((int)std::ceil(std::pow(B, j + 1)), L));
    t.kernels.push_back(k);
  }
  return t;
}

}  // namespace

// ---------------------------------------------------------------- peer barrier
// All ranks of an m-sharded plan meet here between a phase that touches only local memory (ring
// FFTs, elementwise) and a phase that pushes to / pulls from peer workspaces (the contractions).
// One 64-bit epoch per (rank, peer) in the reserved head of every workspace; release/acquire at
// system scope over NVLink.  A time-out (a peer that never arrives) sets the error word instead
// of hanging the GPU.
__global__ void k_peer_barrier(PxmPeers peers, int rank, int world) {
  const int q = threadIdx.x;  // one warp; lane q < world talks to peer q
  ull* local = reinterpret_cast<ull*>(peers.p[rank]);
  const ull epoch = local[PXM_WS_EPOCH] + 1;
  __syncwarp();
  if (q < world) {
    ull* remote = reinterpret_cast<ull*>(peers.p[q]) + rank;
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(remote), "l"(epoch) : "memory");
    const ull* mine = local + q;
    const long long t_start = clock64();
    for (;;) {
      ull v;
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(mine) : "memory");
      if (v >= epoch) break;
      if (clock64() - t_start > 20000000000LL) {  // ~10 s
        local[PXM_WS_ERR] = epoch;
        break;
      }
      __nanosleep(100);
    }
  }
  __syncwarp();
  if (q == 0) local[PXM_WS_EPOCH] = epoch;
}

struct PeerSet {
  Shard sh;
  PxmPeers peers = {};
  bool attached = false;
  int barrier(cudaStream_t st) {
    if (sh.world <= 1) return PXM_OK;
    if (!attached) {
      pxm_set_error("m-sharded plan used before pxm_*_plan_attach");
      return PXM_ERR_ARG;
    }
    k_peer_barrier<<<1, 32, 0, st>>>(peers, sh.rank, sh.world);
    PXM_LAUNCHED();
    return PXM_OK;
  }
  int attach(double* own, void* const* ws) {
    for (int q = 0; q < sh.world; ++q) peers.p[q] = (q == sh.rank) ? own : static_cast<double*>(ws[q]);
    for (int q = 0; q < sh.world; ++q)
      if (!peers.p[q]) {
        pxm_set_error("attach: null peer workspace");
        return PXM_ERR_ARG;
      }
    attached = true;
    return PXM_OK;
  }
  int status(long long* failed_epoch) const {
    ull v = 0;
    PXM_CUDA(cudaMemcpy(&v, reinterpret_cast<const ull*>(peers.p[sh.rank]) + PXM_WS_ERR, 8, cudaMemcpyDeviceToHost));
    *failed_epoch = (long long)v;
    return PXM_OK;
  }
};

int check_shard(int rank, int world) {
  PXM_REQUIRE(world >= 1 && world <= PXM_MAX_PEERS, "world size must be in [1, 8]");
  PXM_REQUIRE(rank >= 0 && rank < world, "rank out of range");
  return PXM_OK;
}

// =========================================================================
//                               SHT plan
// =========================================================================
struct pxm_sht_plan {
  int L = 0, spin = 0, nb = 0, nld = 0;
  bool paired = true;
  PeerSet ps;
  size_t ws_bytes = 0;
  PxmDevVec<unsigned char> d_own;  // per harmonic slot: 1 when this rank owns the azimuthal order
  TableRef lam, w;
  double* d_tab = nullptr;
  double* d_ws = nullptr;
  RingBuf R;
  HarmBuf H;
  FftTables ffttab;
  FftStage fft_in_unit, fft_in_norm, fft_out_unit, fft_out_norm;
  Stage s_lam, a_lam, s_w, a_w;
  cudaStream_t setup_stream = 0;

  int ensure(TableRef& tr) {
    if (tr.built) return PXM_OK;
    if (tr.family == 0)
      PXM_TRY(pxm_generate_lambda(tr.T, d_tab, nullptr, setup_stream));
    else
      PXM_TRY(pxm_generate_w(tr.T, d_tab, nullptr, setup_stream));
    tr.built = true;
    return PXM_OK;
  }
};

extern "C" {

const char* pxm_last_error(void) { return g_err.c_str(); }

int pxm_profile_begin(int max_events) {
  for (auto& e : g_prof_pool) {
    cudaEventDestroy(e.e0);
    cudaEventDestroy(e.e1);
  }
  g_prof_pool.assign((size_t)std::max(max_events, 0), ProfEv());
  for (auto& e : g_prof_pool) {
    PXM_CUDA(cudaEventCreate(&e.e0));
    PXM_CUDA(cudaEventCreate(&e.e1));
  }
  g_prof_used = 0;
  g_prof_on = true;
  return PXM_OK;
}

int pxm_profile_end(double* ms_by_kind, long long* count_by_kind) {
  g_prof_on = false;
  PXM_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < 3; ++k) {
    ms_by_kind[k] = 0.0;
    count_by_kind[k] = 0;
  }
  for (size_t i = 0; i < g_prof_used; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_prof_pool[i].e0, g_prof_pool[i].e1) == cudaSuccess) {
      ms_by_kind[g_prof_pool[i].kind] += ms;
      count_by_kind[g_prof_pool[i].kind] += 1;
    }
  }
  g_prof_used = 0;
  return PXM_OK;
}

long long pxm_launch_count(void) { return g_pxm_launches; }

int pxm_debug_set_naive(int on) {
  g_naive = on;
  return PXM_OK;
}

int pxm_debug_set_fft_multipass(int on) {
  pxm_fft_set_legacy(on);
  return PXM_OK;
}

int pxm_init(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    pxm_set_error("no CUDA device visible: pxmcmc_b200 has no CPU fallback");
    return PXM_ERR_NODEVICE;
  }
  PXM_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  PXM_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) {
    pxm_set_error(std::string("device ") + prop.name + " is not sm_100a (Blackwell); kernels are built for sm_100a only");
    return PXM_ERR_UNSUPPORTED;
  }
  return PXM_OK;
}

int pxm_sht_plan_create(int L, int spin, int max_batch, pxm_sht_plan** out) {
  return pxm_sht_plan_create_sharded(L, spin, max_batch, 0, 1, out);
}

int pxm_sht_plan_create_sharded(int L, int spin, int max_batch, int rank, int world, pxm_sht_plan** out) {
  PXM_TRY(check_shard(rank, world));
  PXM_REQUIRE(L >= 1 && L <= 1024, "L must be in [1, 1024]");
  PXM_REQUIRE(std::abs(spin) < L || L == 1, "|spin| must be < L");
  PXM_REQUIRE(max_batch >= 1, "max_batch >= 1");
  std::unique_ptr<pxm_sht_plan> p(new pxm_sht_plan);
  p->L = L;
  p->spin = spin;
  p->nb = max_batch;
  p->paired = (spin == 0);
  p->nld = pxm_legendre_pad_columns((p->paired ? 4 : 2) * max_batch);
  p->ps.sh.rank = rank;
  p->ps.sh.world = world;
  const Shard& sh = p->ps.sh;
  ull tcur = 0;
  pxm_make_table_layout(p->lam.T, L, L, L, spin, 0, L, tcur, rank, world);
  tcur += p->lam.T.doubles;
  p->lam.family = 0;
  pxm_make_table_layout(p->w.T, L, L, L, spin, 0, L, tcur, rank, world);
  tcur += p->w.T.doubles;
  p->w.family = 1;
  PXM_CUDA(cudaMalloc(&p->d_tab, std::max<ull>(tcur, 1) * 8));
  PXM_CUDA(cudaMemset(p->d_tab, 0, std::max<ull>(tcur, 1) * 8));
  ull wcur = PXM_WS_RESERVED;
  make_ring(p->R, L, p->paired, p->nld, wcur, sh, 0);
  make_harm(p->H, L, p->paired, p->nld, wcur);
  PXM_CUDA(cudaMalloc(&p->d_ws, wcur * 8));
  PXM_CUDA(cudaMemset(p->d_ws, 0, wcur * 8));
  p->ws_bytes = wcur * 8;
  p->ps.peers.p[0] = p->d_ws;
  if (world == 1) p->ps.attached = true;
  PXM_TRY(p->H.d_slot_off.upload(p->H.slot_off));
  {
    std::vector<unsigned char> own(p->H.slot_off.size());
    for (size_t s = 0; s < own.size(); ++s) {
      const int am = p->paired ? (int)s : std::abs((int)s - (L - 1));
      own[s] = pxm_owner_of_m(am, world) == rank;
    }
    PXM_TRY(p->d_own.upload(own));
  }
  const double inv_n = 1.0 / (2 * L - 1);
  add_fft_group(p->fft_in_unit, p->ffttab, p->R, 0, 1.0);
  add_fft_group(p->fft_in_norm, p->ffttab, p->R, 0, inv_n);
  add_fft_group(p->fft_out_unit, p->ffttab, p->R, 0, 1.0);
  add_fft_group(p->fft_out_norm, p->ffttab, p->R, 0, inv_n);
  PXM_TRY(p->ffttab.finalize(0));
  for (FftStage* f : {&p->fft_in_unit, &p->fft_in_norm, &p->fft_out_unit, &p->fft_out_norm})
    PXM_TRY(f->d_groups.upload(f->groups));
  build_s_items(p->s_lam, p->lam, p->H, p->R, p->nld, sh);
  build_s_items(p->s_w, p->w, p->H, p->R, p->nld, sh);
  build_a_items(p->a_lam, {{&p->lam, &p->R}}, p->H, p->nld, sh);
  build_a_items(p->a_w, {{&p->w, &p->R}}, p->H, p->nld, sh);
  for (Stage* s : {&p->s_lam, &p->s_w, &p->a_lam, &p->a_w}) PXM_TRY(s->upload());
  *out = p.release();
  return PXM_OK;
}

int pxm_sht_plan_destroy(pxm_sht_plan* p) {
  if (!p) return PXM_OK;
  for (Stage* s : {&p->s_lam, &p->s_w, &p->a_lam, &p->a_w}) s->release();
  for (FftStage* f : {&p->fft_in_unit, &p->fft_in_norm, &p->fft_out_unit, &p->fft_out_norm}) f->release();
  p->ffttab.release();
  p->H.d_slot_off.release();
  p->d_own.release();
  if (p->d_tab) cudaFree(p->d_tab);
  if (p->d_ws) cudaFree(p->d_ws);
  delete p;
  return PXM_OK;
}

size_t pxm_sht_plan_table_bytes(const pxm_sht_plan* p) { return (p->lam.T.doubles + p->w.T.doubles) * 8; }

// which: 0 inverse, 1 forward, 2 inverse_adjoint, 3 forward_adjoint
static int sht_run(pxm_sht_plan* p, int which, void* d_flm, void* d_f, int nb, const double* d_gl, void* stream) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_REQUIRE(nb >= 1 && nb <= p->nb, "nbatch exceeds the plan's max_batch");
  cudaStream_t st = (cudaStream_t)stream;
  // pixel vectors hold the rows of the rings this rank owns (all of them when not sharded)
  const size_t npix = (size_t)(p->R.t1 - p->R.t0) * (2 * p->L - 1);
  TableRef& tr = (which == 0 || which == 2) ? p->lam : p->w;
  PXM_TRY(p->ensure(tr));
  const int naive = pxm_debug_naive();
  const PxmPeers& pe = p->ps.peers;
  const unsigned char* own = p->ps.sh.world > 1 ? p->d_own.d : nullptr;
  if (which == 0 || which == 3) {  // harmonic -> pixel
    PXM_TRY(pxm_launch_lm_convert(1, d_flm, p->d_ws, p->H.d_slot_off.d, own, d_gl, p->L, p->paired, p->nld, nb, st));
    Stage& S = which == 0 ? p->s_lam : p->s_w;
    PXM_TRY(p->ps.barrier(st));  // peers are done reading the ring buffers this stage overwrites
    { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, pe, pe, S.d_items.d, S.d_segs.d, (int)S.items.size(), p->nld,
                                st, naive)); }
    PXM_TRY(p->ps.barrier(st));  // every rank's tiles have landed
    FftStage& F = which == 0 ? p->fft_out_unit : p->fft_out_norm;
    { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, F.d_groups.d, F.groups.data(), (int)F.groups.size(), F.ctas, d_f, npix, p->d_ws, p->nld,
                           p->ffttab.d_arena, nb, F.class_mask, st)); }
  } else {  // pixel -> harmonic
    FftStage& F = which == 2 ? p->fft_in_unit : p->fft_in_norm;
    { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, F.d_groups.d, F.groups.data(), (int)F.groups.size(), F.ctas, d_f, npix, p->d_ws, p->nld,
                           p->ffttab.d_arena, nb, F.class_mask, st)); }
    Stage& S = which == 2 ? p->a_lam : p->a_w;
    PXM_TRY(p->ps.barrier(st));  // every rank's ring coefficients are in place
    { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, pe, S.d_items.d, S.d_segs.d, (int)S.items.size(), p->nld,
                                st, naive)); }
    PXM_TRY(p->ps.barrier(st));  // peers are done pulling from this rank's ring buffer
    PXM_TRY(pxm_launch_lm_convert(0, d_flm, p->d_ws, p->H.d_slot_off.d, own, d_gl, p->L, p->paired, p->nld, nb, st));
  }
  return PXM_OK;
}

int pxm_sht_inverse(pxm_sht_plan* p, const void* d_flm, void* d_f, int nbatch, const double* d_gl, void* stream) {
  return sht_run(p, 0, const_cast<void*>(d_flm), d_f, nbatch, d_gl, stream);
}
int pxm_sht_forward(pxm_sht_plan* p, const void* d_f, void* d_flm, int nbatch, const double* d_gl, void* stream) {
  return sht_run(p, 1, d_flm, const_cast<void*>(d_f), nbatch, d_gl, stream);
}
int pxm_sht_inverse_adjoint(pxm_sht_plan* p, const void* d_f, void* d_flm, int nbatch, const double* d_gl,
                            void* stream) {
  return sht_run(p, 2, d_flm, const_cast<void*>(d_f), nbatch, d_gl, stream);
}
int pxm_sht_forward_adjoint(pxm_sht_plan* p, const void* d_flm, void* d_f, int nbatch, const double* d_gl,
                            void* stream) {
  return sht_run(p, 3, const_cast<void*>(d_flm), d_f, nbatch, d_gl, stream);
}

}  // extern "C"

// =========================================================================
//                             wavelet plan
// =========================================================================
struct WavDirection {  // tables + stages of one transform pair
  TableRef full;                 // bandlimit-L table (lambda for synthesis pair, W for analysis pair)
  std::vector<TableRef> scales;  // per-scale tables premultiplied by the harmonic kernels
  Stage a_multi;                 // scale rings  -> harmonic (sum over scales)
  Stage s_full;                  // harmonic     -> full-L rings
  Stage a_full;                  // full-L rings -> harmonic
  Stage s_multi;                 // harmonic     -> scale rings
  FftStage fft_scales_in, fft_full_out, fft_full_in, fft_scales_out;
  PxmDevVec<double> d_g;         // concatenated kernels
  bool built = false;
};

struct pxm_wav_plan {
  int L = 0, J_min = 0, nb = 0, nld = 0, nscales_total = 0;
  double B = 0;
  Tiling til;
  PeerSet ps;
  size_t ws_bytes = 0;
  std::vector<ull> coef_off;  // complex offset of every scale map's LOCAL rows inside the local coefficient vector
  ull ncoefs = 0, nscal = 0;  // global sizes
  ull ncoefs_local = 0, npix_local = 0;
  double* d_tab = nullptr;
  double* d_ws = nullptr;
  ull tab_doubles = 0;
  RingBuf Rfull;
  std::vector<RingBuf> Rsc;
  HarmBuf H;
  PxmDevVec<unsigned char> d_own;  // per harmonic slot: 1 when this rank owns the azimuthal order
  FftTables ffttab;
  WavDirection syn, ana;  // syn: synthesis + synthesis_adjoint ; ana: analysis + analysis_adjoint
  // Gram form of the pixel side (pxm_wav_gram_gradient): G^m = (2L-1) Lambda_L^T Lambda_L, a second harmonic buffer
  PxmTableLayout gramT;
  Stage g_full;
  double* d_gram = nullptr;
  double* d_h2 = nullptr;
  double* d_gram_w = nullptr;  // per-ring weights of the Gram table (pxm_wav_set_gram_weights), nullptr: all one
  bool gram_built = false;     // the table holds the Gram matrices of the current weights
  bool gram_alloc = false;

  int ensure_gram() {
    if (gram_built) return PXM_OK;
    PXM_TRY(ensure(syn));
    if (!gram_alloc) {
      pxm_make_table_layout(gramT, L, L, L, 0, 0, L, 0, 0, 1);
      PXM_CUDA(cudaMalloc(&d_gram, std::max<size_t>(gramT.doubles, 1) * 8));
      PXM_CUDA(cudaMalloc(&d_h2, std::max<ull>(H.total, 1) * 8));
      PXM_CUDA(cudaMemset(d_h2, 0, std::max<ull>(H.total, 1) * 8));
      build_g_items(g_full, gramT, H, nld);
      PXM_TRY(g_full.upload());
      gram_alloc = true;
    }
    PXM_CUDA(cudaMemset(d_gram, 0, std::max<size_t>(gramT.doubles, 1) * 8));
    PXM_TRY(pxm_generate_gram(syn.full.T, d_tab, gramT, d_gram, (double)(2 * L - 1), 0, d_gram_w));
    gram_built = true;
    return PXM_OK;
  }

  int ensure(WavDirection& D) {
    if (D.built) return PXM_OK;
    // per-scale kernels live contiguously on the device
    std::vector<double> allg;
    std::vector<size_t> goff;
    for (auto& tr : D.scales) {
      goff.push_back(allg.size());
      allg.insert(allg.end(), tr.g.begin(), tr.g.end());
    }
    PXM_TRY(D.d_g.upload(allg));
    if (D.full.family == 0)
      PXM_TRY(pxm_generate_lambda(D.full.T, d_tab, nullptr, 0));
    else
      PXM_TRY(pxm_generate_w(D.full.T, d_tab, nullptr, 0));
    for (size_t i = 0; i < D.scales.size(); ++i) {
      if (D.scales[i].family == 0)
        PXM_TRY(pxm_generate_lambda(D.scales[i].T, d_tab, D.d_g.d + goff[i], 0));
      else
        PXM_TRY(pxm_generate_w(D.scales[i].T, d_tab, D.d_g.d + goff[i], 0));
    }
    D.built = true;
    return PXM_OK;
  }
};

extern "C" {

int pxm_wav_plan_create(int L, double B, int J_min, int max_batch, pxm_wav_plan** out) {
  return pxm_wav_plan_create_sharded(L, B, J_min, max_batch, 0, 1, out);
}

int pxm_wav_plan_create_sharded(int L, double B, int J_min, int max_batch, int rank, int world, pxm_wav_plan** out) {
  PXM_TRY(check_shard(rank, world));
  PXM_REQUIRE(L >= 2 && L <= 1024, "L must be in [2, 1024]");
  PXM_REQUIRE(B > 1.0, "B must be > 1");
  PXM_REQUIRE(J_min >= 0, "J_min >= 0");
  PXM_REQUIRE(max_batch >= 1, "max_batch >= 1");
  std::unique_ptr<pxm_wav_plan> p(new pxm_wav_plan);
  p->L = L;
  p->B = B;
  p->J_min = J_min;
  p->nb = max_batch;
  p->nld = pxm_legendre_pad_columns(4 * max_batch);
  p->til = make_tiling(L, B, J_min);
  PXM_REQUIRE(p->til.J >= J_min, "J_min larger than J_max");
  const int S = (int)p->til.bandlimits.size();
  p->nscales_total = S;
  p->ps.sh.rank = rank;
  p->ps.sh.world = world;
  const Shard& sh = p->ps.sh;
  ull c = 0, cl = 0;
  for (int i = 0; i < S; ++i) {
    p->coef_off.push_back(cl);
    const ull Lj = p->til.bandlimits[i];
    c += Lj * (2 * Lj - 1);
    int t0, t1;
    pxm_ring_range((int)Lj, i + 1, rank, world, &t0, &t1);
    cl += (ull)(t1 - t0) * (2 * Lj - 1);
  }
  p->ncoefs = c;
  p->ncoefs_local = cl;
  p->nscal = (ull)p->til.bandlimits[0] * (2 * p->til.bandlimits[0] - 1);

  // ---- table layouts ----------------------------------------------------------
  const double SQ2PI = std::sqrt(2.0 * 3.14159265358979323846);
  ull tcur = 0;
  auto add_table = [&](TableRef& tr, int fam, int ell, int lo, int hi, const std::vector<double>& g) {
    tr.family = fam;
    tr.g = g;
    pxm_make_table_layout(tr.T, ell, ell, ell, 0, lo, hi, tcur, rank, world);
    tcur += tr.T.doubles;
  };
  std::vector<double> ones;
  add_table(p->syn.full, 0, L, 0, L, ones);
  add_table(p->ana.full, 1, L, 0, L, ones);
  p->syn.scales.resize(S);
  p->ana.scales.resize(S);
  for (int i = 0; i < S; ++i) {
    const int Lj = p->til.bandlimits[i];
    std::vector<double> gs(Lj), ga(Lj);
    int lo = Lj, hi = 0;
    for (int l = 0; l < Lj; ++l) {
      const double k = p->til.kernels[i][l];
      // (2 pi)^(+-1/2): so3's N=1 normalisation split between analysis and synthesis (SURVEY.md A.5)
      gs[l] = (i == 0) ? k : k * SQ2PI;
      ga[l] = (i == 0) ? k : k / SQ2PI;
      if (k != 0.0) {
        lo = std::min(lo, l);
        hi = std::max(hi, l + 1);
      }
    }
    if (hi <= lo) {
      lo = 0;
      hi = Lj;
    }
    add_table(p->syn.scales[i], 1, Lj, lo, hi, gs);
    add_table(p->ana.scales[i], 0, Lj, lo, hi, ga);
  }
  p->tab_doubles = tcur;
  PXM_CUDA(cudaMalloc(&p->d_tab, std::max<ull>(tcur, 1) * 8));
  PXM_CUDA(cudaMemset(p->d_tab, 0, std::max<ull>(tcur, 1) * 8));

  // ---- workspace ------------------------------------------------------------------
  ull wcur = PXM_WS_RESERVED;
  make_ring(p->Rfull, L, true, p->nld, wcur, sh, 0);
  p->Rsc.resize(S);
  for (int i = 0; i < S; ++i) make_ring(p->Rsc[i], p->til.bandlimits[i], true, p->nld, wcur, sh, i + 1);
  make_harm(p->H, L, true, p->nld, wcur);
  PXM_TRY(p->H.d_slot_off.upload(p->H.slot_off));  // for the harmonic-space entry points
  {
    std::vector<unsigned char> own(p->H.slot_off.size());
    for (size_t sl = 0; sl < own.size(); ++sl) own[sl] = pxm_owner_of_m((int)sl, world) == rank;
    PXM_TRY(p->d_own.upload(own));
  }
  PXM_CUDA(cudaMalloc(&p->d_ws, wcur * 8));
  PXM_CUDA(cudaMemset(p->d_ws, 0, wcur * 8));
  p->ws_bytes = wcur * 8;
  p->ps.peers.p[0] = p->d_ws;
  if (world == 1) p->ps.attached = true;
  p->npix_local = (ull)(p->Rfull.t1 - p->Rfull.t0) * (2 * L - 1);

  // ---- stages -----------------------------------------------------------------------
  const double inv_nL = 1.0 / (2 * L - 1);
  for (WavDirection* D : {&p->syn, &p->ana}) {
    const bool is_syn = (D == &p->syn);
    // pixel-side normalisations: the 1/(2l-1) belongs to the W (quadrature) side
    for (int i = 0; i < S; ++i) {
      const double inv_n = 1.0 / (2 * p->til.bandlimits[i] - 1);
      add_fft_group(D->fft_scales_in, p->ffttab, p->Rsc[i], p->coef_off[i], is_syn ? inv_n : 1.0);
      add_fft_group(D->fft_scales_out, p->ffttab, p->Rsc[i], p->coef_off[i], is_syn ? inv_n : 1.0);
    }
    add_fft_group(D->fft_full_in, p->ffttab, p->Rfull, 0, is_syn ? 1.0 : inv_nL);
    add_fft_group(D->fft_full_out, p->ffttab, p->Rfull, 0, is_syn ? 1.0 : inv_nL);
    std::vector<ASource> srcs;
    for (int i = 0; i < S; ++i) srcs.push_back({&D->scales[i], &p->Rsc[i]});
    build_a_items(D->a_multi, srcs, p->H, p->nld, sh);
    build_s_items(D->s_full, D->full, p->H, p->Rfull, p->nld, sh);
    build_a_items(D->a_full, {{&D->full, &p->Rfull}}, p->H, p->nld, sh);
    for (int i = 0; i < S; ++i) build_s_items(D->s_multi, D->scales[i], p->H, p->Rsc[i], p->nld, sh);
    for (Stage* s : {&D->a_multi, &D->s_full, &D->a_full, &D->s_multi}) PXM_TRY(s->upload());
  }
  PXM_TRY(p->ffttab.finalize(0));
  for (WavDirection* D : {&p->syn, &p->ana})
    for (FftStage* f : {&D->fft_scales_in, &D->fft_scales_out, &D->fft_full_in, &D->fft_full_out})
      PXM_TRY(f->d_groups.upload(f->groups));
  *out = p.release();
  return PXM_OK;
}

int pxm_wav_plan_destroy(pxm_wav_plan* p) {
  if (!p) return PXM_OK;
  for (WavDirection* D : {&p->syn, &p->ana}) {
    for (Stage* s : {&D->a_multi, &D->s_full, &D->a_full, &D->s_multi}) s->release();
    for (FftStage* f : {&D->fft_scales_in, &D->fft_scales_out, &D->fft_full_in, &D->fft_full_out}) f->release();
    D->d_g.release();
  }
  p->ffttab.release();
  p->H.d_slot_off.release();
  p->d_own.release();
  p->g_full.release();
  if (p->d_gram) cudaFree(p->d_gram);
  if (p->d_h2) cudaFree(p->d_h2);
  if (p->d_gram_w) cudaFree(p->d_gram_w);
  if (p->d_tab) cudaFree(p->d_tab);
  if (p->d_ws) cudaFree(p->d_ws);
  delete p;
  return PXM_OK;
}

int pxm_wav_plan_info(const pxm_wav_plan* p, int* nscales_total, long long* ncoefs, long long* nscal, int* J_max,
                      long long* table_bytes) {
  PXM_REQUIRE(p != nullptr, "null plan");
  if (nscales_total) *nscales_total = p->nscales_total;
  if (ncoefs) *ncoefs = (long long)p->ncoefs;
  if (nscal) *nscal = (long long)p->nscal;
  if (J_max) *J_max = p->til.J;
  if (table_bytes) *table_bytes = (long long)p->tab_doubles * 8;
  return PXM_OK;
}

int pxm_wav_plan_bandlimits(const pxm_wav_plan* p, int* out, int cap) {
  PXM_REQUIRE(p != nullptr && cap >= p->nscales_total, "bandlimits: buffer too small");
  for (int i = 0; i < p->nscales_total; ++i) out[i] = p->til.bandlimits[i];
  return PXM_OK;
}

// bytes of the four table families of this rank: {synthesis Lambda_L, synthesis W_j kappa_j, analysis W_L, analysis Lambda_j kappa_j}
int pxm_wav_plan_table_bytes_by_family(const pxm_wav_plan* p, long long* out4) {
  PXM_REQUIRE(p != nullptr && out4 != nullptr, "null argument");
  const WavDirection* dirs[2] = {&p->syn, &p->ana};
  for (int d = 0; d < 2; ++d) {
    out4[2 * d] = (long long)dirs[d]->full.T.doubles * 8;
    long long sc = 0;
    for (const TableRef& tr : dirs[d]->scales) sc += (long long)tr.T.doubles * 8;
    out4[2 * d + 1] = sc;
  }
  return PXM_OK;
}

// Per-ring weights w_t of the Gram table: G^m = (2L-1) Lambda^T diag(w) Lambda -- the data-fidelity gradient of a noise
// level that is constant along every ring (pxm_wav_gram_gradient then takes b = A_inv^dagger(w d)).  h_w: L host
// doubles, or NULL for w = 1.  The table is regenerated on the next pxm_wav_gram_gradient (about 1 ms at L = 256).
int pxm_wav_set_gram_weights(pxm_wav_plan* p, const double* h_w, int n) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_REQUIRE(p->ps.sh.world == 1, "gram form: unsharded plans only");
  PXM_REQUIRE(h_w == nullptr || n == p->L, "gram weights: one weight per ring");
  PXM_CUDA(cudaDeviceSynchronize());  // the table may be in use by launches in flight
  if (h_w == nullptr) {
    if (p->d_gram_w) cudaFree(p->d_gram_w);
    p->d_gram_w = nullptr;
  } else {
    if (!p->d_gram_w) PXM_CUDA(cudaMalloc(&p->d_gram_w, (size_t)p->L * 8));
    PXM_CUDA(cudaMemcpy(p->d_gram_w, h_w, (size_t)p->L * 8, cudaMemcpyHostToDevice));
  }
  p->gram_built = false;
  return PXM_OK;
}

int pxm_wav_plan_gram_bytes(const pxm_wav_plan* p, long long* out) {
  PXM_REQUIRE(p != nullptr && out != nullptr, "null argument");
  *out = p->gram_built ? (long long)p->gramT.doubles * 8 : 0;
  return PXM_OK;
}

// host-only: harmonic kernels kappa0 / kappa_j (what pys2let.wavelet_tiling exposes)
int pxm_wavelet_tiling(int L, double B, int J_min, double* kappa0, double* kappa, int* J_out) {
  PXM_REQUIRE(L >= 1 && B > 1.0 && J_min >= 0, "tiling arguments");
  Tiling t = make_tiling(L, B, J_min);
  if (J_out) *J_out = t.J;
  for (int l = 0; l < L; ++l) kappa0[l] = t.kernels[0][l];
  for (size_t j = 1; j < t.kernels.size(); ++j)
    for (int l = 0; l < L; ++l) kappa[(j - 1) * L + l] = t.kernels[j][l];
  return PXM_OK;
}

// which: 0 synthesis (coef->pix), 1 synthesis_adjoint (pix->coef), 2 analysis (pix->coef), 3 analysis_adjoint (coef->pix)
static int wav_run(pxm_wav_plan* p, int which, void* d_coef, void* d_pix, int nb, void* stream) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_REQUIRE(nb >= 1 && nb <= p->nb, "nbatch exceeds the plan's max_batch");
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = (which < 2) ? p->syn : p->ana;
  PXM_TRY(p->ensure(D));
  const int naive = pxm_debug_naive();
  // local sizes: the rows of the rings this rank owns (everything when not sharded)
  const size_t npix = (size_t)p->npix_local, ncoef = (size_t)p->ncoefs_local;
  const PxmPeers& pe = p->ps.peers;
  const bool coef_to_pix = (which == 0 || which == 3);
  // m-sharded: [local ring FFTs] | barrier | [pull rings -> own m's ; push own m's -> ring owners] | barrier | [local ring FFTs]
  if (coef_to_pix) {
    { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, D.fft_scales_in.d_groups.d, D.fft_scales_in.groups.data(), (int)D.fft_scales_in.groups.size(), D.fft_scales_in.ctas,
                           d_coef, ncoef, p->d_ws, p->nld, p->ffttab.d_arena, nb, D.fft_scales_in.class_mask, st)); }
    PXM_TRY(p->ps.barrier(st));
    { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, pe, D.a_multi.d_items.d, D.a_multi.d_segs.d,
                                (int)D.a_multi.items.size(), p->nld, st, naive)); }
    { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, pe, pe, D.s_full.d_items.d, D.s_full.d_segs.d,
                                (int)D.s_full.items.size(), p->nld, st, naive)); }
    PXM_TRY(p->ps.barrier(st));
    { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, D.fft_full_out.d_groups.d, D.fft_full_out.groups.data(), (int)D.fft_full_out.groups.size(), D.fft_full_out.ctas,
                           d_pix, npix, p->d_ws, p->nld, p->ffttab.d_arena, nb, D.fft_full_out.class_mask, st)); }
  } else {
    { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, D.fft_full_in.d_groups.d, D.fft_full_in.groups.data(), (int)D.fft_full_in.groups.size(), D.fft_full_in.ctas, d_pix,
                           npix, p->d_ws, p->nld, p->ffttab.d_arena, nb, D.fft_full_in.class_mask, st)); }
    PXM_TRY(p->ps.barrier(st));
    { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, pe, D.a_full.d_items.d, D.a_full.d_segs.d,
                                (int)D.a_full.items.size(), p->nld, st, naive)); }
    { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, pe, pe, D.s_multi.d_items.d, D.s_multi.d_segs.d,
                                (int)D.s_multi.items.size(), p->nld, st, naive)); }
    PXM_TRY(p->ps.barrier(st));
    { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, D.fft_scales_out.d_groups.d, D.fft_scales_out.groups.data(), (int)D.fft_scales_out.groups.size(),
                           D.fft_scales_out.ctas, d_coef, ncoef, p->d_ws, p->nld, p->ffttab.d_arena, nb, D.fft_scales_out.class_mask, st)); }
  }
  return PXM_OK;
}

int pxm_wav_synthesis(pxm_wav_plan* p, const void* d_coef, void* d_pix, int nbatch, void* stream) {
  return wav_run(p, 0, const_cast<void*>(d_coef), d_pix, nbatch, stream);
}
int pxm_wav_synthesis_adjoint(pxm_wav_plan* p, const void* d_pix, void* d_coef, int nbatch, void* stream) {
  return wav_run(p, 1, d_coef, const_cast<void*>(d_pix), nbatch, stream);
}
int pxm_wav_analysis(pxm_wav_plan* p, const void* d_pix, void* d_coef, int nbatch, void* stream) {
  return wav_run(p, 2, d_coef, const_cast<void*>(d_pix), nbatch, stream);
}
int pxm_wav_analysis_adjoint(pxm_wav_plan* p, const void* d_coef, void* d_pix, int nbatch, void* stream) {
  return wav_run(p, 3, const_cast<void*>(d_coef), d_pix, nbatch, stream);
}

// Harmonic-space ends of the synthesis pair.  Psi = A_inv(L,0) o [sum_j kappa_j A_fwd(L_j,0)]: a measurement that
// starts with A_fwd(L,0) (WeakLensing, /root/reference/pxmcmc/measurements.py:223) meets A_fwd o A_inv = I on f_lm
// (MW sampling is exact), and its adjoint ends with A_fwd^dagger against Psi^dagger's leading A_inv^dagger: the two full-L
// transforms of each direction are skipped (SURVEY.md 3.5).  d_flm: [nbatch][L^2] complex, index l^2 + l + m; on an
// m-sharded plan only the orders this rank owns are written / read.
int pxm_wav_synthesis_harmonic(pxm_wav_plan* p, const void* d_coef, void* d_flm, int nb, void* stream) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_REQUIRE(nb >= 1 && nb <= p->nb, "nbatch exceeds the plan's max_batch");
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  const unsigned char* own = p->ps.sh.world > 1 ? p->d_own.d : nullptr;
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, D.fft_scales_in.d_groups.d, D.fft_scales_in.groups.data(), (int)D.fft_scales_in.groups.size(),
                         D.fft_scales_in.ctas, const_cast<void*>(d_coef), (size_t)p->ncoefs_local, p->d_ws, p->nld, p->ffttab.d_arena, nb,
                         D.fft_scales_in.class_mask, st)); }
  PXM_TRY(p->ps.barrier(st));  // every rank's ring coefficients are in place
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, pe, D.a_multi.d_items.d, D.a_multi.d_segs.d,
                              (int)D.a_multi.items.size(), p->nld, st, pxm_debug_naive())); }
  PXM_TRY(p->ps.barrier(st));  // peers are done pulling from this rank's ring buffers
  { ProfScope _ps(2, st); PXM_TRY(pxm_launch_lm_convert(0, d_flm, p->d_ws, p->H.d_slot_off.d, own, nullptr, p->L, 1, p->nld, nb, st)); }
  return PXM_OK;
}
int pxm_wav_synthesis_adjoint_harmonic(pxm_wav_plan* p, const void* d_flm, void* d_coef, int nb, void* stream) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_REQUIRE(nb >= 1 && nb <= p->nb, "nbatch exceeds the plan's max_batch");
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  const unsigned char* own = p->ps.sh.world > 1 ? p->d_own.d : nullptr;
  { ProfScope _ps(2, st); PXM_TRY(pxm_launch_lm_convert(1, const_cast<void*>(d_flm), p->d_ws, p->H.d_slot_off.d, own, nullptr, p->L, 1, p->nld, nb, st)); }
  PXM_TRY(p->ps.barrier(st));  // peers are done reading the ring buffers this stage overwrites
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, pe, pe, D.s_multi.d_items.d, D.s_multi.d_segs.d,
                              (int)D.s_multi.items.size(), p->nld, st, pxm_debug_naive())); }
  PXM_TRY(p->ps.barrier(st));  // every rank's tiles have landed
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, D.fft_scales_out.d_groups.d, D.fft_scales_out.groups.data(), (int)D.fft_scales_out.groups.size(),
                         D.fft_scales_out.ctas, d_coef, (size_t)p->ncoefs_local, p->d_ws, p->nld, p->ffttab.d_arena, nb,
                         D.fft_scales_out.class_mask, st)); }
  return PXM_OK;
}

// Ring-Fourier form of the predictions (Identity measurement behind a wavelet synthesis).  Psi ends with the ring FFT
// F_m(theta_t) -> pixels and the next gradient evaluation starts with the ring FFT pixels -> F_m(theta_t)
// (pxmcmc/forward.py:60-72 with an Identity measurement); the DFT of length n = 2L - 1 is invertible, so for an inverse
// covariance that is constant along every ring the pair cancels:
//     FFT_in( ic (FFT_out(F) - data) ) = ic_t ( n F - FFT_in(data) ).
// The ring array is the plan's own layout [slot |m| < L][ring/4][col][ring%4] (doubles), col = 4 chain + 2 (m < 0) + (im),
// `nld` columns, rings padded to a multiple of 32; pxm_wav_ring_doubles gives its size for all chains of the plan.
// Not available on m-sharded plans.
static int ring_check(const pxm_wav_plan* p, int nb) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_REQUIRE(nb >= 1 && nb <= p->nb, "nbatch exceeds the plan's max_batch");
  PXM_REQUIRE(p->ps.sh.world == 1, "ring-space predictions are not available on m-sharded plans");
  return PXM_OK;
}
long long pxm_wav_ring_doubles(const pxm_wav_plan* p) { return p ? (long long)p->Rfull.doubles() : 0; }

int pxm_wav_synthesis_to_ring(pxm_wav_plan* p, const void* d_coef, double* d_ring, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  PxmPeers out = pe;
  out.p[0] = d_ring - p->Rfull.off;  // the last contraction stores its tiles straight into the caller's ring array
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, D.fft_scales_in.d_groups.d, D.fft_scales_in.groups.data(), (int)D.fft_scales_in.groups.size(),
                         D.fft_scales_in.ctas, const_cast<void*>(d_coef), (size_t)p->ncoefs_local, p->d_ws, p->nld, p->ffttab.d_arena, nb,
                         D.fft_scales_in.class_mask, st)); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, pe, D.a_multi.d_items.d, D.a_multi.d_segs.d,
                              (int)D.a_multi.items.size(), p->nld, st, pxm_debug_naive())); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, pe, out, D.s_full.d_items.d, D.s_full.d_segs.d,
                              (int)D.s_full.items.size(), p->nld, st, pxm_debug_naive())); }
  return PXM_OK;
}

int pxm_wav_synthesis_adjoint_from_ring(pxm_wav_plan* p, const double* d_ring, void* d_coef, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  PxmPeers in = pe;
  in.p[0] = const_cast<double*>(d_ring) - p->Rfull.off;  // the first contraction pulls its ring blocks from the caller's array
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, in, pe, D.a_full.d_items.d, D.a_full.d_segs.d,
                              (int)D.a_full.items.size(), p->nld, st, pxm_debug_naive())); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, pe, pe, D.s_multi.d_items.d, D.s_multi.d_segs.d,
                              (int)D.s_multi.items.size(), p->nld, st, pxm_debug_naive())); }
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, D.fft_scales_out.d_groups.d, D.fft_scales_out.groups.data(), (int)D.fft_scales_out.groups.size(),
                         D.fft_scales_out.ctas, d_coef, (size_t)p->ncoefs_local, p->d_ws, p->nld, p->ffttab.d_arena, nb,
                         D.fft_scales_out.class_mask, st)); }
  return PXM_OK;
}

int pxm_wav_ring_to_pix(pxm_wav_plan* p, const double* d_ring, void* d_pix, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  ProfScope _ps(1, st);
  return pxm_fft_launch(1, D.fft_full_out.d_groups.d, D.fft_full_out.groups.data(), (int)D.fft_full_out.groups.size(), D.fft_full_out.ctas,
                        d_pix, (size_t)p->npix_local, const_cast<double*>(d_ring) - p->Rfull.off, p->nld, p->ffttab.d_arena, nb,
                        D.fft_full_out.class_mask, st);
}

int pxm_wav_pix_to_ring(pxm_wav_plan* p, const void* d_pix, double* d_ring, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  ProfScope _ps(1, st);
  return pxm_fft_launch(0, D.fft_full_in.d_groups.d, D.fft_full_in.groups.data(), (int)D.fft_full_in.groups.size(), D.fft_full_in.ctas,
                        const_cast<void*>(d_pix), (size_t)p->npix_local, d_ring - p->Rfull.off, p->nld, p->ffttab.d_arena, nb,
                        D.fft_full_in.class_mask, st);
}

// d_ring_out = ic[t] * ((2L - 1) d_ring_pred - d_ring_data); d_ring_data = pxm_wav_pix_to_ring of the data (chain 0 of a ring
// array); d_ic: L complex values, the inverse covariance of every ring.  d_ring_out may be d_ring_pred.
int pxm_wav_ring_resid(pxm_wav_plan* p, const double* d_ring_pred, const double* d_ring_data, const void* d_ic, double* d_ring_out,
                       int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_ring_resid(d_ring_pred, d_ring_data, d_ic, d_ring_out, p->Rfull.nslots, p->Rfull.rows, p->nld, 4 * nb,
                               (double)(2 * p->L - 1), p->Rfull.slot_stride, (cudaStream_t)stream);
}

// Harmonic form of the predictions, for an inverse covariance that is one (complex) constant over the sphere: the ring-space
// composition above is  g = ic Lambda^T ((2L-1) Lambda f - D)  per order m, i.e.  g = ic (G f - b)  with the Gram matrix
// G^m = (2L-1) Lambda^T Lambda ((L-|m|)^2 entries per order, generated once per plan from the Lambda_L tiles) and
// b = Lambda^T D = A_inv^dagger(data): ONE contraction with a third fewer entries replaces the two full-L contractions, and
// the predictions are carried as f_lm.  Harmonic arrays use the plan's layout: concatenated slots |m| < L of
// [rows/4][col][rows%4] doubles, rows = l - |m| padded to 64, col = 4 chain + 2 (m<0) + (im); pxm_wav_harm_doubles = size.
long long pxm_wav_harm_doubles(const pxm_wav_plan* p) { return p ? (long long)p->H.total : 0; }

static PxmPeers harm_peers(const pxm_wav_plan* p, const double* harm) {
  PxmPeers q = p->ps.peers;
  q.p[0] = const_cast<double*>(harm) - p->H.slot_off[0];
  return q;
}

int pxm_wav_synthesis_to_harm(pxm_wav_plan* p, const void* d_coef, double* d_harm, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, D.fft_scales_in.d_groups.d, D.fft_scales_in.groups.data(), (int)D.fft_scales_in.groups.size(),
                         D.fft_scales_in.ctas, const_cast<void*>(d_coef), (size_t)p->ncoefs_local, p->d_ws, p->nld, p->ffttab.d_arena, nb,
                         D.fft_scales_in.class_mask, st)); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, harm_peers(p, d_harm), D.a_multi.d_items.d, D.a_multi.d_segs.d,
                              (int)D.a_multi.items.size(), p->nld, st, pxm_debug_naive())); }
  return PXM_OK;
}

// coefficients of  Psi^dagger ic (Psi X - data)  from f = pxm_wav_synthesis_to_harm(X): d_b = pxm_wav_pix_to_harm_adjoint(data)
int pxm_wav_gram_gradient(pxm_wav_plan* p, const double* d_harm, const double* d_b, double ic_re, double ic_im, void* d_coef, int nb,
                          void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure_gram());
  const PxmPeers& pe = p->ps.peers;
  const PxmPeers h2 = harm_peers(p, p->d_h2);
  // g = ic (G f - b): the affine part rides on the epilogue of the Gram contraction
  const PxmLegAffine aff = {d_b - p->H.slot_off[0], ic_re, ic_im};
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_gram, harm_peers(p, d_harm), h2, p->g_full.d_items.d, p->g_full.d_segs.d,
                              (int)p->g_full.items.size(), p->nld, st, pxm_debug_naive(), &aff)); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, h2, pe, D.s_multi.d_items.d, D.s_multi.d_segs.d,
                              (int)D.s_multi.items.size(), p->nld, st, pxm_debug_naive())); }
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, D.fft_scales_out.d_groups.d, D.fft_scales_out.groups.data(), (int)D.fft_scales_out.groups.size(),
                         D.fft_scales_out.ctas, d_coef, (size_t)p->ncoefs_local, p->d_ws, p->nld, p->ffttab.d_arena, nb,
                         D.fft_scales_out.class_mask, st)); }
  return PXM_OK;
}

int pxm_wav_harm_to_pix(pxm_wav_plan* p, const double* d_harm, void* d_pix, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(0, p->d_tab, harm_peers(p, d_harm), pe, D.s_full.d_items.d, D.s_full.d_segs.d,
                              (int)D.s_full.items.size(), p->nld, st, pxm_debug_naive())); }
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(1, D.fft_full_out.d_groups.d, D.fft_full_out.groups.data(), (int)D.fft_full_out.groups.size(),
                         D.fft_full_out.ctas, d_pix, (size_t)p->npix_local, p->d_ws, p->nld, p->ffttab.d_arena, nb, D.fft_full_out.class_mask, st)); }
  return PXM_OK;
}

// A_inv^dagger of a pixel map into a harmonic array (the constant b of pxm_wav_gram_gradient: pass the data, nbatch = 1)
int pxm_wav_pix_to_harm_adjoint(pxm_wav_plan* p, const void* d_pix, double* d_harm, int nb, void* stream) {
  PXM_TRY(ring_check(p, nb));
  cudaStream_t st = (cudaStream_t)stream;
  WavDirection& D = p->syn;
  PXM_TRY(p->ensure(D));
  const PxmPeers& pe = p->ps.peers;
  { ProfScope _ps(1, st); PXM_TRY(pxm_fft_launch(0, D.fft_full_in.d_groups.d, D.fft_full_in.groups.data(), (int)D.fft_full_in.groups.size(), D.fft_full_in.ctas,
                         const_cast<void*>(d_pix), (size_t)p->npix_local, p->d_ws, p->nld, p->ffttab.d_arena, nb, D.fft_full_in.class_mask, st)); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch_peers(1, p->d_tab, pe, harm_peers(p, d_harm), D.a_full.d_items.d, D.a_full.d_segs.d,
                              (int)D.a_full.items.size(), p->nld, st, pxm_debug_naive())); }
  return PXM_OK;
}

// =========================================================================
//        HEALPix plan (healpy.alm2map / map2alm: data preparation, once per run)
// =========================================================================
}  // extern "C"

void pxm_hpx_half_angles(int nside, double* out);

struct pxm_hpx_plan {
  int nside = 0, L = 0, nrings = 0, nld = 0;
  TableRef lam;
  PxmDevVec<double> d_half;
  double* d_tab = nullptr;
  double* d_ws = nullptr;
  RingBuf R;
  HarmBuf H;
  Stage s_lam, a_lam;
};

extern "C" {

int pxm_hpx_plan_create(int nside, int L, pxm_hpx_plan** out) {
  PXM_REQUIRE(nside >= 1 && nside <= 8192 && (nside & (nside - 1)) == 0, "nside must be a power of two in [1, 8192]");
  PXM_REQUIRE(L >= 1 && L <= 1024, "L (= lmax + 1) must be in [1, 1024]");
  std::unique_ptr<pxm_hpx_plan> p(new pxm_hpx_plan);
  p->nside = nside;
  p->L = L;
  p->nrings = 4 * nside - 1;
  p->nld = pxm_legendre_pad_columns(4);
  std::vector<double> half(2 * (size_t)p->nrings);
  pxm_hpx_half_angles(nside, half.data());
  PXM_TRY(p->d_half.upload(half));
  pxm_make_table_layout(p->lam.T, L, p->nrings, L, 0, 0, L, 0);
  p->lam.T.d_half_angles = p->d_half.d;
  p->lam.family = 0;
  const ull tdoubles = std::max<ull>(p->lam.T.doubles, 1);
  PXM_CUDA(cudaMalloc(&p->d_tab, tdoubles * 8));
  PXM_CUDA(cudaMemset(p->d_tab, 0, tdoubles * 8));
  PXM_TRY(pxm_generate_lambda(p->lam.T, p->d_tab, nullptr, 0));
  ull wcur = PXM_WS_RESERVED;
  p->R.ell = L;
  p->R.rows = p->nrings;
  p->R.paired = true;
  p->R.nslots = L;
  p->R.t0 = 0;
  p->R.t1 = p->nrings;
  p->R.slot_stride = (ull)pxm_round_up(p->nrings, 64) * p->nld;
  p->R.off = wcur;
  wcur += p->R.doubles();
  make_harm(p->H, L, true, p->nld, wcur);
  PXM_CUDA(cudaMalloc(&p->d_ws, wcur * 8));
  PXM_CUDA(cudaMemset(p->d_ws, 0, wcur * 8));
  PXM_TRY(p->H.d_slot_off.upload(p->H.slot_off));
  build_s_items(p->s_lam, p->lam, p->H, p->R, p->nld);
  build_a_items(p->a_lam, {{&p->lam, &p->R}}, p->H, p->nld);
  PXM_TRY(p->s_lam.upload());
  PXM_TRY(p->a_lam.upload());
  *out = p.release();
  return PXM_OK;
}

int pxm_hpx_plan_destroy(pxm_hpx_plan* p) {
  if (!p) return PXM_OK;
  p->s_lam.release();
  p->a_lam.release();
  p->H.d_slot_off.release();
  p->d_half.release();
  if (p->d_tab) cudaFree(p->d_tab);
  if (p->d_ws) cudaFree(p->d_ws);
  delete p;
  return PXM_OK;
}

// map[p] = sum_lm flm Y_lm(theta_p, phi_p)   (complex field; flm index l*l+l+m)
int pxm_hpx_alm2map(pxm_hpx_plan* p, const void* d_flm, void* d_map, void* stream) {
  PXM_REQUIRE(p != nullptr, "null plan");
  cudaStream_t st = (cudaStream_t)stream;
  PXM_TRY(pxm_launch_lm_convert(1, const_cast<void*>(d_flm), p->d_ws, p->H.d_slot_off.d, nullptr, nullptr, p->L, 1,
                                p->nld, 1, st));
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch(0, p->d_tab, p->d_ws, p->d_ws, p->s_lam.d_items.d, p->s_lam.d_segs.d,
                              (int)p->s_lam.items.size(), p->nld, st, pxm_debug_naive())); }
  { ProfScope _ps(1, st); PXM_TRY(pxm_hpx_ring_dft_launch(1, p->nside, p->L, d_map, p->d_ws, p->R.off, p->R.slot_stride, p->nld, st)); }
  return PXM_OK;
}

// flm = sum_p conj(Y_lm(theta_p, phi_p)) map[p]   (no quadrature weight: the Euclidean adjoint of alm2map;
// healpy.map2alm = (4 pi / npix) x this, plus Jacobi iterations built from the two calls)
int pxm_hpx_map2alm_adjoint(pxm_hpx_plan* p, const void* d_map, void* d_flm, void* stream) {
  PXM_REQUIRE(p != nullptr, "null plan");
  cudaStream_t st = (cudaStream_t)stream;
  { ProfScope _ps(1, st); PXM_TRY(pxm_hpx_ring_dft_launch(0, p->nside, p->L, d_map, p->d_ws, p->R.off, p->R.slot_stride, p->nld, st)); }
  { ProfScope _ps(0, st); PXM_TRY(pxm_legendre_launch(1, p->d_tab, p->d_ws, p->d_ws, p->a_lam.d_items.d, p->a_lam.d_segs.d,
                              (int)p->a_lam.items.size(), p->nld, st, pxm_debug_naive())); }
  PXM_TRY(pxm_launch_lm_convert(0, d_flm, p->d_ws, p->H.d_slot_off.d, nullptr, nullptr, p->L, 1, p->nld, 1, st));
  return PXM_OK;
}

// =========================================================================
//          m-sharded plans: workspace exchange, local layout, IPC
// =========================================================================
void* pxm_sht_plan_workspace(pxm_sht_plan* p, size_t* bytes) {
  if (bytes) *bytes = p->ws_bytes;
  return p->d_ws;
}
void* pxm_wav_plan_workspace(pxm_wav_plan* p, size_t* bytes) {
  if (bytes) *bytes = p->ws_bytes;
  return p->d_ws;
}
// Build every Legendre table now instead of on first use.  Required for m-sharded plans (the
// table generator allocates/frees scratch memory, which synchronises the device and must not
// happen while a peer barrier is spinning); optional otherwise.
static int preload_kernels(int nld) {
  cudaFuncAttributes a;
  PXM_CUDA(cudaFuncGetAttributes(&a, k_peer_barrier));
  PXM_TRY(pxm_legendre_preload(nld));
  PXM_TRY(pxm_elem_preload());
  return PXM_OK;
}
int pxm_sht_plan_prepare(pxm_sht_plan* p) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_TRY(preload_kernels(p->nld));
  PXM_TRY(p->ensure(p->lam));
  PXM_TRY(p->ensure(p->w));
  PXM_CUDA(cudaDeviceSynchronize());
  return PXM_OK;
}
int pxm_wav_plan_prepare(pxm_wav_plan* p) {
  PXM_REQUIRE(p != nullptr, "null plan");
  PXM_TRY(preload_kernels(p->nld));
  PXM_TRY(p->ensure(p->syn));
  PXM_TRY(p->ensure(p->ana));
  PXM_CUDA(cudaDeviceSynchronize());
  return PXM_OK;
}
int pxm_sht_plan_attach(pxm_sht_plan* p, void* const* peer_ws) {
  PXM_REQUIRE(p && peer_ws, "attach: null argument");
  return p->ps.attach(p->d_ws, peer_ws);
}
int pxm_wav_plan_attach(pxm_wav_plan* p, void* const* peer_ws) {
  PXM_REQUIRE(p && peer_ws, "attach: null argument");
  return p->ps.attach(p->d_ws, peer_ws);
}
int pxm_sht_plan_barrier_status(pxm_sht_plan* p, long long* failed_epoch) { return p->ps.status(failed_epoch); }
int pxm_wav_plan_barrier_status(pxm_wav_plan* p, long long* failed_epoch) { return p->ps.status(failed_epoch); }

int pxm_sht_plan_local_rows(const pxm_sht_plan* p, int* t0, int* t1) {
  PXM_REQUIRE(p != nullptr, "null plan");
  *t0 = p->R.t0;
  *t1 = p->R.t1;
  return PXM_OK;
}
// t0/t1[i], i < nscales_total: rows of scale map i; t0/t1[nscales_total]: rows of the pixel map
int pxm_wav_plan_local_rows(const pxm_wav_plan* p, int* t0, int* t1, long long* ncoefs_local, long long* npix_local) {
  PXM_REQUIRE(p != nullptr, "null plan");
  for (int i = 0; i < p->nscales_total; ++i) {
    t0[i] = p->Rsc[i].t0;
    t1[i] = p->Rsc[i].t1;
  }
  t0[p->nscales_total] = p->Rfull.t0;
  t1[p->nscales_total] = p->Rfull.t1;
  if (ncoefs_local) *ncoefs_local = (long long)p->ncoefs_local;
  if (npix_local) *npix_local = (long long)p->npix_local;
  return PXM_OK;
}

// host-only views of the partition (what tests/test_host_cpu.py checks without a GPU)
int pxm_shard_owner_of_m(int abs_m, int world) { return pxm_owner_of_m(abs_m, world); }
int pxm_shard_ring_range(int ell, int rot, int rank, int world, int* t0, int* t1) {
  PXM_REQUIRE(world >= 1 && world <= PXM_MAX_PEERS && rank >= 0 && rank < world && ell >= 1, "shard arguments");
  pxm_ring_range(ell, rot, rank, world, t0, t1);
  return PXM_OK;
}

// CUDA IPC: how the ranks (one process per GPU) learn each other's workspace addresses
int pxm_ipc_export(const void* d_ptr, void* handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  cudaIpcMemHandle_t h;
  PXM_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(d_ptr)));
  memcpy(handle64, &h, 64);
  return PXM_OK;
}
int pxm_ipc_open(const void* handle64, void** d_ptr) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  PXM_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return PXM_OK;
}
int pxm_ipc_close(void* d_ptr) {
  PXM_CUDA(cudaIpcCloseMemHandle(d_ptr));
  return PXM_OK;
}

// =========================================================================
//                 elementwise / reductions / sparse entry points
// =========================================================================
int pxm_soft(int is_complex, const void* d_x, const double* d_T, double T_scalar, void* d_out, long long n,
             long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_soft(is_complex, d_x, d_T, T_scalar, d_out, (size_t)n, (size_t)nchains, (cudaStream_t)stream);
}

int pxm_myula_update(const void* d_X, const void* d_prox, const void* d_gradg, const double* d_T, double T_scalar,
                     const double* d_w_re, const double* d_w_im, void* d_Xout, void* d_prox_out, long long n,
                     long long nchains, double delta, double lmda, int noise_mode, unsigned long long seed,
                     unsigned long long step, unsigned int stream0, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_myula(d_X, d_prox, d_gradg, d_T, T_scalar, d_w_re, d_w_im, d_Xout, d_prox_out, (size_t)n,
                          (size_t)nchains, delta, lmda, noise_mode, seed, step, nullptr, stream0, (cudaStream_t)stream);
}

// same, with the Philox step read from device memory: a captured CUDA graph of the iteration can be
// replayed without re-recording (pxm_counter_add advances the counter inside the graph)
int pxm_myula_update_dstep(const void* d_X, const void* d_prox, const void* d_gradg, const double* d_T, double T_scalar,
                           void* d_Xout, void* d_prox_out, long long n, long long nchains, double delta, double lmda,
                           int noise_mode, unsigned long long seed, const unsigned long long* d_step,
                           unsigned int stream0, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_step != nullptr && (noise_mode == 2 || noise_mode == 3 || noise_mode == 4),
              "dstep update needs a device counter and Philox noise");
  return pxm_launch_myula(d_X, d_prox, d_gradg, d_T, T_scalar, nullptr, nullptr, d_Xout, d_prox_out, (size_t)n,
                          (size_t)nchains, delta, lmda, noise_mode, seed, 0, d_step, stream0, (cudaStream_t)stream);
}

// PxMALA without a host round trip per iteration: the tuned step size lives in a device state block
// (layout: pxm_elem.cu, k_pxmala_accept), the accept test and the state hand-over run on the device
int pxm_myula_update_dpar(const void* d_X, const void* d_prox, const void* d_gradg, const double* d_T, double T_scalar,
                          void* d_Xout, void* d_prox_out, long long n, long long nchains, const double* d_par,
                          int noise_mode, unsigned long long seed, unsigned long long step, unsigned int stream0,
                          void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_par != nullptr && (noise_mode == 2 || noise_mode == 3), "dpar update needs a device state block and Philox noise");
  return pxm_launch_myula(d_X, d_prox, d_gradg, d_T, T_scalar, nullptr, nullptr, d_Xout, d_prox_out, (size_t)n,
                          (size_t)nchains, 0.0, 1.0, noise_mode, seed, step, nullptr, stream0, (cudaStream_t)stream, d_par);
}
int pxm_reduce_dpar(int kind, const void* a, const void* b, const void* c, const void* d, const double* w,
                    const double* d_par, double lmda, long long n, long long nchains, void* d_partial, void* d_out,
                    void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(kind == 2 && d_par != nullptr, "reduce_dpar: kind 2 with a device state block");
  return pxm_launch_reduce(kind, a, b, c, d, w, 0.0, lmda, (size_t)n, (size_t)nchains, d_partial, d_out,
                           (cudaStream_t)stream, d_par);
}
int pxm_pxmala_accept(double* d_state, const void* d_s1, const void* d_s2, const void* d_L2p, const void* d_priorp,
                      double mu, double lmda, int tune, long long i, unsigned long long seed, unsigned long long step,
                      unsigned int stream_id, signed char* d_acc_trace, double* d_delta_trace, long long trace_stride,
                      int nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_state && d_s1 && d_s2 && d_L2p && d_priorp && d_acc_trace && d_delta_trace && nchains >= 1 && trace_stride >= 1,
              "pxmala_accept: bad argument");
  return pxm_launch_pxmala_accept(d_state, d_s1, d_s2, d_L2p, d_priorp, mu, lmda, tune, i, seed, step, stream_id,
                                  d_acc_trace, d_delta_trace, trace_stride, nchains, (cudaStream_t)stream);
}
int pxm_select_if(const double* d_flag, long long flag_stride, long long nchains, void* const* d_dst,
                  const void* const* d_src, const long long* counts, int narrays, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_flag != nullptr && narrays >= 1 && narrays <= 4 && nchains >= 1 && flag_stride >= 0, "select_if: 1 to 4 arrays");
  size_t n[4] = {0, 0, 0, 0};
  for (int a = 0; a < narrays; ++a) n[a] = (size_t)counts[a];
  return pxm_launch_select(d_flag, (size_t)flag_stride, (size_t)nchains, d_dst, d_src, n, narrays, (cudaStream_t)stream);
}

int pxm_philox_normal(double* d_out, long long n, long long nchains, unsigned long long seed, unsigned long long step,
                      const unsigned long long* d_step, unsigned int stream0, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_out != nullptr && n >= 0 && nchains >= 0, "philox_normal: bad argument");
  return pxm_launch_philox_normal(d_out, (size_t)n, (size_t)nchains, seed, step, d_step, stream0, (cudaStream_t)stream);
}

int pxm_counter_add(unsigned long long* d_counter, unsigned long long inc, void* stream) {
  PXM_REQUIRE(d_counter != nullptr, "null counter");
  return pxm_launch_counter_add(d_counter, inc, (cudaStream_t)stream);
}

int pxm_resid_invcov(const void* d_preds, const void* d_data, const void* d_invcov, void* d_out, long long n,
                     long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_resid(d_preds, d_data, d_invcov, d_out, (size_t)n, (size_t)nchains, (cudaStream_t)stream);
}

int pxm_reduce_scratch_elems(void) { return 148; }

int pxm_reduce(int kind, const void* a, const void* b, const void* c, const void* d, const double* w, double delta,
               double lmda, long long n, long long nchains, void* d_partial, void* d_out, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(kind >= 0 && kind <= 2, "reduce kind");
  return pxm_launch_reduce(kind, a, b, c, d, w, delta, lmda, (size_t)n, (size_t)nchains, d_partial, d_out,
                           (cudaStream_t)stream);
}

int pxm_lincomb(int nx, const void* const* d_xs, const double* coefs, const double* d_z, double cz, double c0,
                void* d_out, long long total, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(nx >= 0 && nx <= 4, "lincomb supports up to 4 terms");
  return pxm_launch_lincomb(nx, d_xs, coefs, d_z, cz, c0, d_out, (size_t)total, (cudaStream_t)stream);
}

int pxm_gradlogpi(const void* d_X, const void* d_prox, const double* d_T, double T_scalar, const void* d_gradg,
                  double lmda, void* d_out, long long n, long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_gradlogpi(d_X, d_prox, d_T, T_scalar, d_gradg, lmda, d_out, (size_t)n, (size_t)nchains,
                              (cudaStream_t)stream);
}

static bool skrock_noise_ok(int noise_mode, const double* d_z_re, const double* d_z_im) {
  return noise_mode >= 0 && noise_mode <= 4 && (noise_mode < 1 || noise_mode > 2 || d_z_re != nullptr) &&
         (noise_mode != 2 || d_z_im != nullptr);
}

int pxm_skrock_shift(const void* d_X, double c, const double* d_z_re, const double* d_z_im, int noise_mode,
                     unsigned long long seed, unsigned long long step, const unsigned long long* d_step,
                     unsigned int stream0, void* d_Y, long long n, long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_X != nullptr && d_Y != nullptr && n >= 0 && nchains >= 0, "skrock_shift: bad argument");
  PXM_REQUIRE(noise_mode >= 1 && skrock_noise_ok(noise_mode, d_z_re, d_z_im), "skrock_shift: noise_mode 1..4 with its arrays");
  return pxm_launch_skrock(0, d_X, nullptr, nullptr, nullptr, nullptr, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, c, 0.0, d_z_re,
                           d_z_im, noise_mode, seed, step, d_step, stream0, d_Y, (size_t)n, (size_t)nchains,
                           (cudaStream_t)stream);
}

int pxm_skrock_stage(const void* d_U, const void* d_V, const void* d_gradg, const void* d_prox, const double* d_T,
                     double T_scalar, double lmda, double a, double b, double c, double c0, double c_shift, double e,
                     const double* d_z_re, const double* d_z_im, int noise_mode, unsigned long long seed,
                     unsigned long long step, const unsigned long long* d_step, unsigned int stream0, void* d_out,
                     long long n, long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_U != nullptr && d_gradg != nullptr && d_out != nullptr && n >= 0 && nchains >= 0,
              "skrock_stage: bad argument");
  PXM_REQUIRE(skrock_noise_ok(noise_mode, d_z_re, d_z_im), "skrock_stage: noise_mode 0..4 with its arrays");
  return pxm_launch_skrock(1, d_U, d_V, d_gradg, d_prox, d_T, T_scalar, lmda, a, b, c, c0, c_shift, e, d_z_re, d_z_im,
                           noise_mode, seed, step, d_step, stream0, d_out, (size_t)n, (size_t)nchains,
                           (cudaStream_t)stream);
}

int pxm_fista_update(const void* d_y, const void* d_gradg, const void* d_x, const double* d_T, double T_scalar,
                     double T_scale, double t, double* d_state, void* d_x_out, void* d_y_out, double* d_hist,
                     long long cap, long long n, long long nchains, void* d_partial, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  PXM_REQUIRE(d_y && d_gradg && d_x && d_state && d_x_out && d_y_out && d_hist && d_partial && n >= 0 && cap >= 1 &&
                  nchains >= 0 && nchains <= 65535,
              "fista_update: bad argument");
  return pxm_launch_fista(d_y, d_gradg, d_x, d_T, T_scalar, T_scale, t, d_state, d_x_out, d_y_out, d_hist, cap,
                          (size_t)n, (size_t)nchains, d_partial, (cudaStream_t)stream);
}

int pxm_masked_gather(const void* d_full, const int* d_idx, const double* d_w, void* d_sel, long long nsel,
                      long long nfull, long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_gather(0, d_full, d_idx, d_w, d_sel, (size_t)nsel, (size_t)nfull, (size_t)nchains,
                           (cudaStream_t)stream);
}
int pxm_masked_scatter(const void* d_sel, const int* d_idx, const double* d_w, void* d_full, long long nsel,
                       long long nfull, long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_gather(1, d_sel, d_idx, d_w, d_full, (size_t)nsel, (size_t)nfull, (size_t)nchains,
                           (cudaStream_t)stream);
}

int pxm_real_to_complex(const double* d_x, void* d_out, long long total, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_r2c(d_x, d_out, (size_t)total, (cudaStream_t)stream);
}

int pxm_quantile_columns(const double* d_chain, long long nsamples, long long ncols, long long ld, long long lo_a,
                         double gamma_a, long long lo_b, double gamma_b, double* d_out_a, double* d_out_b, void* stream) {
  PXM_REQUIRE(ld >= ncols && lo_a >= 0 && lo_b >= 0 && lo_a < nsamples && lo_b < nsamples, "quantile: bad index or stride");
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_quantile_columns(d_chain, nsamples, ncols, ld, lo_a, gamma_a, lo_b, gamma_b, d_out_a, d_out_b,
                                     (cudaStream_t)stream);
}
int pxm_quantile_columns_max_samples(void) { return pxm_quantile_max_samples(); }

long long pxm_stats_accumulator_doubles(long long n, long long nchains, int mode) {
  if (n < 1 || nchains < 1 || mode < 0 || mode > 2) {
    pxm_set_error("bad argument: stats_accumulator_doubles: n >= 1, nchains >= 1, mode 0, 1 or 2");
    return -1;
  }
  return 8 * pxm_stats_slots(mode, nchains) * n;
}

int pxm_stats_reset(double* d_acc, long long n, long long nchains, int mode, void* stream) {
  const long long nd = pxm_stats_accumulator_doubles(n, nchains, mode);
  PXM_REQUIRE(nd > 0 && d_acc != nullptr, "stats_reset: null accumulator, n >= 1, nchains >= 1, mode 0, 1 or 2");
  PXM_CUDA(cudaMemsetAsync(d_acc, 0, (size_t)nd * sizeof(double), (cudaStream_t)stream));
  return PXM_OK;
}

int pxm_stats_accumulate(double* d_acc, const void* d_x, long long n, long long nchains, int mode, long long nsamples,
                         long long j, const long long* d_j, void* stream) {
  PXM_REQUIRE(d_acc != nullptr && d_x != nullptr, "stats_accumulate: null pointer");
  PXM_REQUIRE(n >= 1 && nchains >= 1 && nchains <= 65535, "stats_accumulate: n >= 1, 1 <= nchains <= 65535");
  PXM_REQUIRE(mode >= 0 && mode <= 2, "stats_accumulate: mode 0 (real part), 1 (re + im) or 2 (packed real pairs)");
  PXM_REQUIRE(nsamples >= 1, "stats_accumulate: nsamples >= 1");
  PXM_REQUIRE(d_j != nullptr || (j >= 0 && j < nsamples), "stats_accumulate: sample index j outside [0, nsamples)");
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_stats_accumulate(d_acc, d_x, (size_t)n, (size_t)nchains, mode, nsamples, j, d_j, (cudaStream_t)stream);
}

int pxm_stats_partials(const double* d_acc, long long n, long long nchains, int mode, long long nsamples,
                       double* d_partial, double* d_chain_mean, double* d_chain_var, void* stream) {
  PXM_REQUIRE(d_acc != nullptr && d_partial != nullptr, "stats_partials: null pointer");
  PXM_REQUIRE(n >= 1 && nchains >= 1, "stats_partials: n >= 1, nchains >= 1");
  PXM_REQUIRE(mode >= 0 && mode <= 2, "stats_partials: mode 0 (real part), 1 (re + im) or 2 (packed real pairs)");
  PXM_REQUIRE(nsamples >= 1, "stats_partials: nsamples >= 1");
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_stats_partials(d_acc, (size_t)n, (size_t)nchains, mode, nsamples, d_partial, d_chain_mean,
                                   d_chain_var, (cudaStream_t)stream);
}

long long pxm_rank_diagnostics_scratch_doubles(long long m, long long n, long long ncols) {
  if (m < 1 || n < 1 || ncols < 0 || m * n > pxm_quantile_max_samples() || ncols > INT_MAX) {
    pxm_set_error("bad argument: rank_diagnostics: m >= 1, n >= 1, m n <= 16384 samples per column, 0 <= ncols < 2^31");
    return -1;
  }
  return m * n * ncols;
}

int pxm_rank_diagnostics(const double* d_chain, long long m, long long n, long long ncols, long long ld,
                         double* d_scratch, double* d_rhat, double* d_ess_bulk, double* d_ess_tail, void* stream) {
  PXM_REQUIRE(pxm_rank_diagnostics_scratch_doubles(m, n, ncols) >= 0,
              "rank_diagnostics: m >= 1, n >= 1, m n <= 16384 samples per column, 0 <= ncols < 2^31");
  PXM_REQUIRE(ld >= ncols && ld >= 1, "rank_diagnostics: leading dimension ld >= ncols");
  PXM_REQUIRE(ncols == 0 || (d_chain && d_scratch && d_rhat && d_ess_bulk && d_ess_tail), "rank_diagnostics: null pointer");
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_rank_diagnostics(d_chain, m, n, ncols, ld, d_scratch, d_rhat, d_ess_bulk, d_ess_tail,
                                     (cudaStream_t)stream);
}

long long pxm_credible_state_doubles(long long n, int mode, long long npooled, long long lo_a, long long lo_b) {
  long long klo = 0, khi = 0;
  const long long T = (mode == 1 ? 2 : 1) * n;
  if (n < 1 || n > INT_MAX || mode < 0 || mode > 2 || pxm_credible_tails(npooled, lo_a, lo_b, &klo, &khi) != PXM_OK ||
      klo + khi + 1 > LLONG_MAX / T) {
    pxm_set_error("bad argument: credible_state_doubles: 1 <= n < 2^31, mode 0, 1 or 2, npooled >= 1, "
                  "0 <= lo_a, lo_b < npooled");
    return -1;
  }
  return (klo + khi + 1) * T;
}

int pxm_credible_reset(double* d_state, long long n, int mode, long long npooled, long long lo_a, long long lo_b,
                       void* stream) {
  const long long nd = pxm_credible_state_doubles(n, mode, npooled, lo_a, lo_b);
  PXM_REQUIRE(nd > 0 && d_state != nullptr, "credible_reset: null state or bad size arguments");
  PXM_CUDA(cudaMemsetAsync(d_state, 0, (size_t)nd * sizeof(double), (cudaStream_t)stream));
  return PXM_OK;
}

int pxm_credible_push(double* d_state, const void* d_x, long long n, long long nchains, int mode, long long npooled,
                      long long lo_a, long long lo_b, long long count, const long long* d_j, void* stream) {
  long long klo = 0, khi = 0;
  PXM_REQUIRE(d_state != nullptr && d_x != nullptr, "credible_push: null pointer");
  PXM_REQUIRE(pxm_credible_state_doubles(n, mode, npooled, lo_a, lo_b) > 0,
              "credible_push: 1 <= n < 2^31, mode 0, 1 or 2, npooled >= 1, 0 <= lo_a, lo_b < npooled");
  PXM_REQUIRE(nchains >= 1 && nchains <= INT_MAX, "credible_push: 1 <= nchains < 2^31");
  PXM_REQUIRE(count >= 0 && count <= npooled, "credible_push: 0 <= count <= npooled");
  pxm_credible_tails(npooled, lo_a, lo_b, &klo, &khi);
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_credible_push(d_state, d_x, (size_t)n, (size_t)nchains, mode, klo, khi, count, d_j,
                                  (cudaStream_t)stream);
}

int pxm_credible_finalize(const double* d_state, long long n, int mode, long long npooled, long long lo_a,
                          double gamma_a, long long lo_b, double gamma_b, double* d_lower, double* d_upper,
                          void* stream) {
  long long klo = 0, khi = 0;
  PXM_REQUIRE(d_state != nullptr && d_lower != nullptr && d_upper != nullptr, "credible_finalize: null pointer");
  PXM_REQUIRE(pxm_credible_state_doubles(n, mode, npooled, lo_a, lo_b) > 0,
              "credible_finalize: 1 <= n < 2^31, mode 0, 1 or 2, npooled >= 1, 0 <= lo_a, lo_b < npooled");
  pxm_credible_tails(npooled, lo_a, lo_b, &klo, &khi);
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_credible_finalize(d_state, (size_t)n, mode, npooled, klo, khi, lo_a, gamma_a, lo_b, gamma_b,
                                      d_lower, d_upper, (cudaStream_t)stream);
}

int pxm_csr_spmv(const int* d_indptr, const int* d_indices, const double* d_vals, const void* d_x, void* d_y,
                 int nrows, long long ncols, long long nchains, void* stream) {
  ProfScope _ps(2, (cudaStream_t)stream);
  return pxm_launch_csr_spmv(d_indptr, d_indices, d_vals, d_x, d_y, nrows, (size_t)ncols, (size_t)nchains,
                             (cudaStream_t)stream);
}

}  // extern "C"

// b200pde: host side of the B200-native Navier2D spectral hot path + its C ABI.
//
// Mirrors the reference's Space / Field / Solve / Integrate surface (see include/b200pde.h for
// the file:line of every interface replaced).  Everything numeric runs in lane_kernel.cuh;
// this file only (a) builds the small per-axis coefficient vectors on the host exactly as
// src/field.rs:195-249 + src/solver/*.rs define them, (b) strings lane programs together and
// (c) owns device memory.  There is NO CPU fallback: every entry point needs a CUDA device.
#include "lane_kernel.cuh"
#include "gemm_f64.cuh"
#include "../../include/b200pde.h"

#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include <algorithm>

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(B2_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
  } while (0)
#define RET(call)                    \
  do {                               \
    int r_ = (call);                 \
    if (r_ != B2_OK) return r_;      \
  } while (0)

static inline int roundup(int a, int b) { return (a + b - 1) / b * b; }
#ifdef B2_EMU
#define B2_SPIN_PAUSE() std::this_thread::sleep_for(std::chrono::microseconds(20))   // emulated ranks are OS processes sharing a few cores
#else
#define B2_SPIN_PAUSE()
#endif

// ------------------------------------------------------------------------------------------------
// structures
// ------------------------------------------------------------------------------------------------
struct b2_ctx {
  int device = 0, rank = 0, nranks = 1;
  cudaStream_t stream = nullptr;      // origin stream: everything is ordered on it
  cudaStream_t side[2] = {nullptr, nullptr};   // side streams: independent passes of a step run as parallel graph branches
  cudaStream_t cur = nullptr;         // stream the next pass is launched on (origin or a side stream)
  cudaEvent_t evp[16] = {nullptr};    // fork / join events
  int evn = 0;
  long long launches = 0;  // lane-kernel + helper launches (counted, for bench.py's gpu_launches)
  double* stage = nullptr; size_t stage_bytes = 0;   // host<->device staging (plain layout)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;          // b2_ctx_timer_*
  bool profile = false;                              // time the GEMM launches separately
  std::vector<cudaEvent_t> gemm_events;
  // symmetric heap for nranks > 1: every rank allocates the same arrays in the same order, so an
  // array has the same offset on every GPU and a peer's copy is peer_base[r] + offset
  char* heap = nullptr;
  size_t heap_bytes = 0, heap_used = 0;
  std::vector<std::pair<size_t, size_t>> heap_free;   // (offset, bytes) blocks returned by ctx_free: every rank frees in the same order, so the heaps stay symmetric
  std::map<void*, size_t> heap_live;                  // live blocks: pointer -> bytes
  double** d_peers = nullptr;  // device table of peer heap bases
  void* peer_base[B2_MAXPEERS] = {nullptr};
  bool attached = false;
  long long barriers = 0;
  unsigned long long* d_prof = nullptr;   // per-op cycle counters (debug/profiling)
  int* d_differs = nullptr;               // result word of k_same_value (collective allocator)
  double* d_acc = nullptr;                // accumulator of the norm reductions (integrate() asks for |div| after every step)
};
static const size_t B2_HEAP_RESERVED = 4096;  // flags[0..nranks) + epoch counter live at the start of the heap

static int ctx_alloc(b2_ctx* c, size_t bytes, double** out) {
  if (c->nranks == 1) { CK(cudaMalloc(out, bytes)); return B2_OK; }
  const size_t need = (bytes + 255) / 256 * 256;
  // exact-size reuse (arrays of a problem share one padded size); the LOWEST free block of that size, so that the choice depends
  // on the set of free blocks only, not on the order in which a rank's host code happened to release them
  size_t best = c->heap_free.size();
  for (size_t i = 0; i < c->heap_free.size(); i++)
    if (c->heap_free[i].second == need && (best == c->heap_free.size() || c->heap_free[i].first < c->heap_free[best].first)) best = i;
  if (best < c->heap_free.size()) {
    *out = reinterpret_cast<double*>(c->heap + c->heap_free[best].first);
    c->heap_free.erase(c->heap_free.begin() + best);
    c->heap_live[*out] = need;
    return B2_OK;
  }
  if (c->heap_used + need > c->heap_bytes) return fail(B2_ERR_ARG, "symmetric heap exhausted: pass a larger heap_bytes to b2_ctx_create");
  *out = reinterpret_cast<double*>(c->heap + c->heap_used);
  c->heap_used += need;
  c->heap_live[*out] = need;
  return B2_OK;
}
static void ctx_free(b2_ctx* c, void* p) {
  if (!p) return;
  if (c->nranks == 1) { cudaFree(p); return; }
  auto it = c->heap_live.find(p);
  if (it == c->heap_live.end()) return;
  c->heap_free.emplace_back((size_t)(static_cast<char*>(p) - c->heap), it->second);
  c->heap_live.erase(it);
}

// all-ranks barrier on the stream: signal every peer's flag slot, then wait for every peer's signal
// `slot`: independent barrier lanes (one per stream / graph branch), 16 words each: flags[0..8) + the epoch counter
__global__ void k_barrier(unsigned long long* const* peers_, int rank, int nranks, int slot) {
  __shared__ unsigned long long* peers[B2_MAXPEERS];
  if ((int)threadIdx.x < nranks) peers[threadIdx.x] = peers_[threadIdx.x] + 16 * slot;
  __syncthreads();
  unsigned long long* mine = peers[rank];
  __shared__ unsigned long long epoch;
  if (threadIdx.x == 0) epoch = mine[B2_MAXPEERS] + 1;
  __syncthreads();
  const unsigned long long e = epoch;
  __threadfence_system();
  if ((int)threadIdx.x < nranks) {
    *reinterpret_cast<volatile unsigned long long*>(peers[threadIdx.x] + rank) = e;
    __threadfence_system();
    while (*reinterpret_cast<volatile unsigned long long*>(mine + threadIdx.x) < e) { B2_SPIN_PAUSE(); }
  }
  __syncthreads();
  if (threadIdx.x == 0) mine[B2_MAXPEERS] = e;
}
// sum of one double over the ranks, on the stream: every rank writes its term into every peer's slot, the flag exchange
// of barrier lane 3 orders the writes, then everyone adds the nranks terms in rank order (same result on every rank).
// Two value buffers alternate with the epoch so that a fast rank's next all-reduce cannot overwrite unread terms.
__global__ void k_allreduce(unsigned long long* const* peers_, int rank, int nranks, const double* in, double* out) {
  __shared__ unsigned long long* peers[B2_MAXPEERS];
  if ((int)threadIdx.x < nranks) peers[threadIdx.x] = peers_[threadIdx.x] + 16 * 3;
  __syncthreads();
  unsigned long long* mine = peers[rank];
  __shared__ unsigned long long epoch;
  if (threadIdx.x == 0) epoch = mine[B2_MAXPEERS] + 1;
  __syncthreads();
  const unsigned long long e = epoch;
  const int buf = (int)(e & 1ull) * B2_MAXPEERS;
  if ((int)threadIdx.x < nranks) {
    volatile double* dst = reinterpret_cast<volatile double*>(peers_[threadIdx.x]) + 256 + buf + rank;
    *dst = *in;
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(peers[threadIdx.x] + rank) = e;
    __threadfence_system();
    while (*reinterpret_cast<volatile unsigned long long*>(mine + threadIdx.x) < e) { B2_SPIN_PAUSE(); }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const volatile double* v = reinterpret_cast<const volatile double*>(peers_[rank]) + 256 + buf;
    double s = 0;
    for (int r = 0; r < nranks; r++) s += v[r];
    *out = s;
    mine[B2_MAXPEERS] = e;
  }
}
// Barrier + agreement check on the stream: every rank publishes one word to every peer (flag exchange of barrier lane 3, value
// buffers alternating with the epoch like k_allreduce) and reports whether any rank's word differs from its own.  Used by the
// collective allocator: an array must have the same heap offset on every rank, or peer stores land in somebody else's array.
__global__ void k_same_value(unsigned long long* const* peers_, int rank, int nranks, unsigned long long value, int* differs) {
  __shared__ unsigned long long* peers[B2_MAXPEERS];
  if ((int)threadIdx.x < nranks) peers[threadIdx.x] = peers_[threadIdx.x] + 16 * 3;
  __syncthreads();
  unsigned long long* mine = peers[rank];
  __shared__ unsigned long long epoch;
  if (threadIdx.x == 0) epoch = mine[B2_MAXPEERS] + 1;
  __syncthreads();
  const unsigned long long e = epoch;
  const int buf = (int)(e & 1ull) * B2_MAXPEERS;
  if ((int)threadIdx.x < nranks) {
    *reinterpret_cast<volatile unsigned long long*>(peers_[threadIdx.x] + 320 + buf + rank) = value;
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(peers[threadIdx.x] + rank) = e;
    __threadfence_system();
    while (*reinterpret_cast<volatile unsigned long long*>(mine + threadIdx.x) < e) { B2_SPIN_PAUSE(); }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const volatile unsigned long long* v = peers_[rank] + 320 + buf;
    int d = 0;
    for (int r = 0; r < nranks; r++) d |= (v[r] != value);
    *differs = d;
    mine[B2_MAXPEERS] = e;
  }
}
static int ctx_barrier(b2_ctx* c) {
  if (c->nranks == 1) return B2_OK;
  if (!c->attached) return fail(B2_ERR_ARG, "b2_ctx_attach_peers has not been called");
  const int slot = c->cur == c->side[0] ? 1 : (c->cur == c->side[1] ? 2 : 0);   // every stream has its own flags and epoch
  B2_LAUNCH(k_barrier, 1, 32, 0, c->cur ? c->cur : c->stream, reinterpret_cast<unsigned long long* const*>(c->d_peers), c->rank, c->nranks, slot);
  CK(cudaGetLastError());
  c->barriers++;
  return B2_OK;
}

struct DVecD {  // device vector of doubles
  double* d = nullptr;
  size_t n = 0;
  int upload(const std::vector<double>& h) {
    n = h.size();
    if (n == 0) return B2_OK;
    CK(cudaMalloc(&d, n * sizeof(double)));
    CK(cudaMemcpy(d, h.data(), n * sizeof(double), cudaMemcpyHostToDevice));
    return B2_OK;
  }
  void release() { if (d) cudaFree(d); d = nullptr; }
};

// unsweeped 4-diagonal matrix, as Fdma::from_matrix_raw (src/solver/fdma.rs:44-54)
struct Diags {
  int m = 0;
  std::vector<double> low, dia, up1, up2;  // all length m (tails unused / zero)
  explicit Diags(int m_ = 0) : m(m_), low(m_, 0.0), dia(m_, 0.0), up1(m_, 0.0), up2(m_, 0.0) {}
};
// LU vectors in the form the kernel wants: fl[i] = low[i-2], id[i] = 1/dia[i], u1, u2 (zero tails)
struct LuVecs { std::vector<double> fl, id, u1, u2; };

// Fdma::sweep, src/solver/fdma.rs:73-82, then repack
static LuVecs sweep(const Diags& a) {
  const int n = a.m;
  std::vector<double> low = a.low, dia = a.dia, up1 = a.up1, up2 = a.up2;
  for (int i = 2; i < n; i++) {
    low[i - 2] /= dia[i - 2];
    dia[i] -= low[i - 2] * up1[i - 2];
    if (i < n - 2) up1[i] -= low[i - 2] * up2[i - 2];
  }
  LuVecs r;
  r.fl.assign(n, 0.0); r.id.assign(n, 0.0); r.u1.assign(n, 0.0); r.u2.assign(n, 0.0);
  for (int i = 0; i < n; i++) {
    if (i >= 2) r.fl[i] = low[i - 2];
    r.id[i] = 1.0 / dia[i];
    if (i < n - 2) r.u1[i] = up1[i];
    if (i < n - 4) r.u2[i] = up2[i];
  }
  return r;
}

// PdmaPlus2::from_matrix (src/solver/pdma_plus2.rs:45-121): LU sweep of a matrix with diagonals at offsets -2..+4, packed for
// OP_PDMA as [l2 shifted | ka | 1/mu | al | be | ga | de], each L doubles (zero tails).  d[k] = diagonal at offset k - 2,
// indexed by the row for k >= 2 and by the column for the two sub-diagonals (ndarray `diag`).
static std::vector<double> pdma_sweep(int n, const std::vector<double> (&d)[7], int L) {
  const std::vector<double>&l2 = d[0], &l1 = d[1], &d0 = d[2], &u1 = d[3], &u2 = d[4], &u3 = d[5], &u4 = d[6];
  std::vector<double> al(n, 0.0), be(n, 0.0), ga(n, 0.0), de(n, 0.0), ka(n, 0.0), mu(n, 0.0);
  for (int i = 0; i < n; i++) {
    const double l2i = i >= 2 ? l2[i - 2] : 0.0;
    ka[i] = (i >= 1 ? l1[i - 1] : 0.0) - (i >= 2 ? al[i - 2] * l2i : 0.0);
    mu[i] = d0[i] - (i >= 2 ? be[i - 2] * l2i : 0.0) - (i >= 1 ? al[i - 1] * ka[i] : 0.0);
    if (i + 1 < n) al[i] = (u1[i] - (i >= 2 ? ga[i - 2] * l2i : 0.0) - (i >= 1 ? be[i - 1] * ka[i] : 0.0)) / mu[i];
    if (i + 2 < n) be[i] = (u2[i] - (i >= 2 ? de[i - 2] * l2i : 0.0) - (i >= 1 ? ga[i - 1] * ka[i] : 0.0)) / mu[i];
    if (i + 3 < n) ga[i] = (u3[i] - (i >= 1 ? de[i - 1] * ka[i] : 0.0)) / mu[i];
    if (i + 4 < n) de[i] = u4[i] / mu[i];
  }
  std::vector<double> out((size_t)7 * L, 0.0);
  for (int i = 0; i < n; i++) {
    out[i] = i >= 2 ? l2[i - 2] : 0.0; out[(size_t)L + i] = ka[i]; out[(size_t)2 * L + i] = 1.0 / mu[i];
    out[(size_t)3 * L + i] = al[i]; out[(size_t)4 * L + i] = be[i]; out[(size_t)5 * L + i] = ga[i]; out[(size_t)6 * L + i] = de[i];
  }
  return out;
}

// natural-order band coefficient vector -> its scan-layout copy (same chunking as the LU coefficients of that axis)
static std::map<const void*, const void*>& scan_of() { static std::map<const void*, const void*> m; return m; }

struct Base1 {
  int kind = 0, n = 0, m = 0;
  bool cheb = false, composite = false;   // composite: ChebDirichlet / ChebNeumann (stencil at even offsets: pair-structured lane operators)
  bool cdn = false;                        // ChebDirichletNeumann (bc = "hc"): three-term stencil, PdmaPlus2 solves
  bool c2c = false;                        // FourierC2c: complex physical values, n modes in FFT order (k = 0 .. n/2-1, -n/2 .. -1)
  int rows_phys = 0, rows_spec = 0, rows_ortho = 0;  // real rows along this axis (complex => 2 per mode)
  int N = 0;                                          // transform size (n-1 Chebyshev, n Fourier)
  std::vector<double> s2;                             // stencil: ortho_k = c_k + s2[k-2] c_{k-2}
  DVecD d_sten2, d_sten2s, d_s2, d_tfl, d_tid, d_tu1, d_bd, d_bu1, d_bu2, d_tw, d_tw2, d_isin;
  std::vector<double> ca, cb;                         // cdn stencil: ortho_k = c_k + ca[k-1] c_{k-1} + cb[k-2] c_{k-2}
  DVecD d_dfwd, d_dbwd; bool dense_tr = false;       // transform sizes the FFT core does not handle: dense matrices (OP_DENSE)
  DVecD d_ca, d_cb, d_pent; int pent_L = 0;            // cdn: stencil vectors, packed PdmaPlus2 LU of S^T S (from_ortho)
  DVecD d_s2_sc, d_bd_sc, d_bu1_sc, d_bu2_sc, d_sten2s_sc;   // scan-layout copies for band ops folded into an LU solve (see run_pass)

  // B2 = laplace_inv (SURVEY 8a row G); pv(i, off) = (laplace_inv_eye . laplace_inv)[i, i+off]
  double pv(int i, int off) const {
    const int r = i + 2;
    if (off == 0) return r == 2 ? 0.25 : 1.0 / (4.0 * r * (r - 1.0));
    if (off == 2) return (r < n - 2) ? -1.0 / (2.0 * ((double)r * r - 1.0)) : 0.0;
    if (off == 4) return (r < n - 4) ? 1.0 / (4.0 * r * (r + 1.0)) : 0.0;
    return 0.0;
  }
  // mat_a = pinv . S and mat_b = peye . S of src/field.rs:204-208 (composite bases)
  Diags mat_a() const {
    Diags a(m);
    for (int i = 0; i < m; i++) {
      if (i >= 2) a.low[i - 2] = pv(i, 0) * s2[i - 2];
      a.dia[i] = pv(i, 0) + pv(i, 2) * s2[i];
      if (i + 2 < m) a.up1[i] = pv(i, 2) + pv(i, 4) * s2[i + 2];
      if (i + 4 < m) a.up2[i] = pv(i, 4);
    }
    return a;
  }
  Diags mat_b() const {
    Diags b(m);
    for (int i = 0; i < m; i++) {
      b.dia[i] = s2[i];
      if (i + 2 < m) b.up1[i] = 1.0;
    }
    return b;
  }
  // cdn: the seven diagonals (offsets -2..+4) of mat_a - c * mat_b = (pinv - c * peye) . S of src/field.rs:204-208,
  // S[k][k] = 1, S[k+1][k] = ca[k], S[k+2][k] = cb[k]
  void cdn_hholtz_diags(double c, std::vector<double> (&d)[7]) const {
    auto S = [&](int r, int j) -> double { if (j < 0 || j >= m) return 0.0; return r == j ? 1.0 : (r == j + 1 ? ca[j] : (r == j + 2 ? cb[j] : 0.0)); };
    for (int k = 0; k < 7; k++) d[k].assign(m, 0.0);
    for (int i = 0; i < m; i++)
      for (int off = -2; off <= 4; off++) {
        const int j = i + off;
        if (j < 0 || j >= m) continue;
        const double a = pv(i, 0) * S(i, j) + pv(i, 2) * S(i + 2, j) + pv(i, 4) * S(i + 4, j);
        const double v = a - c * S(i + 2, j);
        d[off + 2][off >= 0 ? i : j] = v;
      }
  }
  int init_host(int kind_, int n_);
  int init(int C, int TPL);   // device vectors; (C, TPL) = chunking of the passes whose lanes run along this axis
  int lay_C = 1, lay_TPL = 1;
  // pair/scan order of a coefficient vector: double2 slot [t*TPL + q] = (v[2p], v[2p+1]), p = q*CP + t
  std::vector<double> scan_layout(const std::vector<double>& v) const {
    std::vector<double> o((size_t)2 * lay_C * lay_TPL, 0.0);
    for (int q = 0; q < lay_TPL; q++)
      for (int t = 0; t < lay_C; t++) {
        const size_t p = (size_t)q * lay_C + t, k = (size_t)t * lay_TPL + q;
        if (2 * p < v.size()) o[2 * k] = v[2 * p];
        if (2 * p + 1 < v.size()) o[2 * k + 1] = v[2 * p + 1];
      }
    return o;
  }
  void release() {
    const void* keys[] = {d_bd.d, d_bu1.d, d_bu2.d, d_s2.d, d_sten2s.d};
    for (auto k : keys) if (k) scan_of().erase(k);
    DVecD* all[] = {&d_sten2, &d_sten2s, &d_s2, &d_tfl, &d_tid, &d_tu1, &d_bd, &d_bu1, &d_bu2, &d_tw, &d_tw2, &d_isin, &d_s2_sc, &d_bd_sc, &d_bu1_sc, &d_bu2_sc, &d_sten2s_sc, &d_ca, &d_cb, &d_pent, &d_dfwd, &d_dbwd};
    for (auto* v : all) v->release();
  }
};

static bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }

int Base1::init_host(int kind_, int n_) {
  kind = kind_; n = n_;
  cheb = (kind <= B2_CHEB_DIRICHLET_NEUMANN);
  composite = (kind == B2_CHEB_DIRICHLET || kind == B2_CHEB_NEUMANN);
  cdn = (kind == B2_CHEB_DIRICHLET_NEUMANN);
  c2c = (kind == B2_FOURIER_C2C);
  if (kind < 0 || kind > B2_FOURIER_C2C) return fail(B2_ERR_ARG, "bad base kind");
  if (n < 5) return fail(B2_ERR_ARG, "n too small");
  if (cheb) {
    m = (composite || cdn) ? n - 2 : n;
    rows_phys = n; rows_spec = m; rows_ortho = n; N = n - 1;
  } else if (c2c) {
    // complex in, complex out (bases.rs:15): no Navier2D configuration uses it, so it runs the dense-matrix transform only
    // (2n x 2n real matrix per lane, OP_DENSE) -- N = 0 keeps it off the FFT thread layouts
    if (n > 1024) return fail(B2_ERR_UNSUPPORTED, "fourier_c2c: n <= 1024 (dense-matrix transform)");
    m = n;
    rows_phys = 2 * n; rows_spec = 2 * n; rows_ortho = 2 * n; N = 0;
  } else {
    if (n % 2) return fail(B2_ERR_UNSUPPORTED, "fourier_r2c needs even n");
    m = n / 2 + 1;
    rows_phys = n; rows_spec = 2 * m; rows_ortho = 2 * m; N = n;
  }
  if (cdn) {   // SURVEY A.2: a_k = ((k+2)^2 - k^2) / ((k+1)^2 + (k+2)^2), b_k = a_k - 1
    ca.assign(m, 0.0); cb.assign(m, 0.0);
    for (int k = 0; k < m; k++) { const double kd = k; ca[k] = ((kd + 2) * (kd + 2) - kd * kd) / ((kd + 1) * (kd + 1) + (kd + 2) * (kd + 2)); cb[k] = ca[k] - 1.0; }
  }
  if (composite) {
    s2.assign(m, 0.0);
    for (int k = 0; k < m; k++) s2[k] = (kind == B2_CHEB_DIRICHLET) ? -1.0 : -((double)k / (k + 2.0)) * ((double)k / (k + 2.0));
  }
  return B2_OK;
}

int Base1::init(int C, int TPL) {
  lay_C = C; lay_TPL = TPL;
  const int L = roundup(std::max(rows_phys, rows_ortho) + 8, 4) + 64;  // generous coefficient-vector length
  if (composite) {
    std::vector<double> sten2(L, 0.0), s2v(L, 0.0);
    for (int i = 2; i < n; i++) sten2[i] = s2[i - 2];
    for (int k = 0; k < m; k++) s2v[k] = s2[k];
    RET(d_sten2.upload(sten2)); RET(d_sten2s.upload(sten2)); RET(d_s2.upload(s2v));   // banded mat-vec coefficients: natural order
    // from_ortho: (S^T S) c = S^T o, tridiagonal at offsets (-2,0,2) (SURVEY A.2)
    Diags t(m);
    for (int k = 0; k < m; k++) {
      t.dia[k] = 1.0 + s2[k] * s2[k];
      if (k + 2 < m) { t.low[k] = s2[k]; t.up1[k] = s2[k]; }
    }
    LuVecs lu = sweep(t);
    lu.fl.resize(L, 0.0); lu.id.resize(L, 0.0); lu.u1.resize(L, 0.0);
    RET(d_tfl.upload(scan_layout(lu.fl))); RET(d_tid.upload(scan_layout(lu.id))); RET(d_tu1.upload(scan_layout(lu.u1)));
    // MatVecFdma of the preconditioner pinv (src/solver/matvec.rs:177-203)
    std::vector<double> bd(L, 0.0), bu1(L, 0.0), bu2(L, 0.0);
    for (int i = 0; i < m; i++) {
      bd[i] = pv(i, 0);
      if (i < m - 2) bu1[i] = pv(i, 2);
      if (i < m - 4) bu2[i] = pv(i, 4);
    }
    RET(d_bd.upload(bd)); RET(d_bu1.upload(bu1)); RET(d_bu2.upload(bu2));
    RET(d_bd_sc.upload(scan_layout(bd))); RET(d_bu1_sc.upload(scan_layout(bu1))); RET(d_bu2_sc.upload(scan_layout(bu2))); RET(d_s2_sc.upload(scan_layout(s2v)));
    scan_of()[d_bd.d] = d_bd_sc.d; scan_of()[d_bu1.d] = d_bu1_sc.d; scan_of()[d_bu2.d] = d_bu2_sc.d; scan_of()[d_s2.d] = d_s2_sc.d;
    RET(d_sten2s_sc.upload(scan_layout(sten2))); scan_of()[d_sten2s.d] = d_sten2s_sc.d;
  }
  if (cdn) {
    std::vector<double> a(L, 0.0), b(L, 0.0);
    for (int k = 0; k < m; k++) { a[k] = ca[k]; b[k] = cb[k]; }
    RET(d_ca.upload(a)); RET(d_cb.upload(b));
    // from_ortho: (S^T S) c = S^T o, pentadiagonal (funspace); solved with the PdmaPlus2 recurrences (outer diagonals zero)
    std::vector<double> d[7];
    for (int k = 0; k < 7; k++) d[k].assign(m, 0.0);
    for (int j = 0; j < m; j++) {
      d[2][j] = 1.0 + ca[j] * ca[j] + cb[j] * cb[j];
      if (j + 1 < m) { d[3][j] = ca[j] + cb[j] * ca[j + 1]; d[1][j] = d[3][j]; }
      if (j + 2 < m) { d[4][j] = cb[j]; d[0][j] = cb[j]; }
    }
    pent_L = L;
    RET(d_pent.upload(pdma_sweep(m, d, L)));
    // MatVecFdma of the preconditioner pinv (the same for every composite base)
    std::vector<double> bd(L, 0.0), bu1(L, 0.0), bu2(L, 0.0);
    for (int i = 0; i < m; i++) {
      bd[i] = pv(i, 0);
      if (i < m - 2) bu1[i] = pv(i, 2);
      if (i < m - 4) bu2[i] = pv(i, 4);
    }
    RET(d_bd.upload(bd)); RET(d_bu1.upload(bu1)); RET(d_bu2.upload(bu2));
    RET(d_bd_sc.upload(scan_layout(bd))); RET(d_bu1_sc.upload(scan_layout(bu1))); RET(d_bu2_sc.upload(scan_layout(bu2)));
    scan_of()[d_bd.d] = d_bd_sc.d; scan_of()[d_bu1.d] = d_bu1_sc.d; scan_of()[d_bu2.d] = d_bu2_sc.d;
  }
  // transform tables (only when the size is one the FFT core handles)
  if (is_pow2(N) && N >= 64) {
    const int M = N / 2;
    const long double PI = 3.14159265358979323846264338327950288L;
    std::vector<double> tw(2 * M), tw2(2 * (M + 1)), isin(M, 0.0);
    for (int t = 0; t < M; t++) { tw[2 * t] = (double)cosl(2 * PI * t / M); tw[2 * t + 1] = (double)(-sinl(2 * PI * t / M)); }
    for (int j = 0; j <= M; j++) { tw2[2 * j] = (double)cosl(2 * PI * j / N); tw2[2 * j + 1] = (double)(-sinl(2 * PI * j / N)); }
    for (int k = 1; k < M; k++) isin[k] = (double)(1.0L / (4.0L * sinl(PI * k / N)));
    RET(d_tw.upload(tw)); RET(d_tw2.upload(tw2)); RET(d_isin.upload(isin));
  } else if (n <= 2049) {
    // any other size: the transforms as dense matrices (SURVEY A.1 / A.4), applied per lane by OP_DENSE -- O(n^2) per lane, meant
    // for small grids such as the reference's criterion sizes (128, 264, 265, 512)
    const long double PI = 3.14159265358979323846264338327950288L;
    if (c2c) {    // c_k = sum_j v_j e^{-2 pi i j k / n} (unnormalised), v_j = 1/n sum_k c_k e^{+2 pi i j k / n}; rows 2k, 2k+1 = Re, Im
      std::vector<double> F((size_t)4 * n * n), B((size_t)4 * n * n);
      const size_t w = (size_t)2 * n;
      for (int k = 0; k < n; k++)
        for (int j = 0; j < n; j++) {
          const long double a = 2 * PI * (long double)((long long)j * k % n) / n;
          const double ca_ = (double)cosl(a), sa_ = (double)sinl(a), cn_ = (double)(cosl(a) / n), sn_ = (double)(sinl(a) / n);
          F[(size_t)(2 * k) * w + 2 * j] = ca_;      F[(size_t)(2 * k) * w + 2 * j + 1] = sa_;
          F[(size_t)(2 * k + 1) * w + 2 * j] = -sa_; F[(size_t)(2 * k + 1) * w + 2 * j + 1] = ca_;
          B[(size_t)(2 * j) * w + 2 * k] = cn_;      B[(size_t)(2 * j) * w + 2 * k + 1] = -sn_;
          B[(size_t)(2 * j + 1) * w + 2 * k] = sn_;  B[(size_t)(2 * j + 1) * w + 2 * k + 1] = cn_;
        }
      RET(d_dfwd.upload(F)); RET(d_dbwd.upload(B));
    } else if (cheb) {   // c = F v: c_k = f_k (-1)^k / (n-1) sum_j g_j v_j cos(pi j k / (n-1));  v = B c: v_j = sum_k (-1)^k c_k cos(pi j k / (n-1))
      std::vector<double> F((size_t)n * n), B((size_t)n * n);
      for (int k = 0; k < n; k++)
        for (int j = 0; j < n; j++) {
          const long double c = cosl(PI * (long double)((long long)j * k % (2 * (n - 1))) / (n - 1));
          const long double fk = (k == 0 || k == n - 1) ? 0.5L : 1.0L, gj = (j == 0 || j == n - 1) ? 1.0L : 2.0L, sg = (k & 1) ? -1.0L : 1.0L;
          F[(size_t)k * n + j] = (double)(fk * sg * gj * c / (n - 1));
          B[(size_t)j * n + k] = (double)(sg * c);
        }
      RET(d_dfwd.upload(F)); RET(d_dbwd.upload(B));
    } else {      // r2c (unnormalised) / c2r (1/n): rows 2k, 2k+1 = Re, Im of mode k
      std::vector<double> F((size_t)2 * m * n), B((size_t)n * 2 * m);
      for (int k = 0; k < m; k++)
        for (int j = 0; j < n; j++) {
          const long double a = 2 * PI * (long double)((long long)j * k % n) / n, wk = (k == 0 || 2 * k == n) ? 1.0L : 2.0L;
          F[(size_t)(2 * k) * n + j] = (double)cosl(a); F[(size_t)(2 * k + 1) * n + j] = (double)(-sinl(a));
          B[(size_t)j * 2 * m + 2 * k] = (double)(wk * cosl(a) / n); B[(size_t)j * 2 * m + 2 * k + 1] = (double)(-wk * sinl(a) / n);
        }
      RET(d_dfwd.upload(F)); RET(d_dbwd.upload(B));
    }
    dense_tr = true;
  }
  return B2_OK;
}

struct PassCfg {
  int in_tiles, out_tiles, LP, TPL, C, E, groups, LN;
  bool fast;   // transform-sized lane: N = 2*E*TPL and LP >= N + 4 (lane_fast.cuh)
  int NT, CHW, nsc, wslot_bytes, CHD, nchd, w_off, st_off;   // copy-pipeline geometry (lane_kernel.cuh)
  size_t smem;
};

struct b2_space {
  b2_ctx* ctx = nullptr;
  Base1 b[2];
  int P[2] = {0, 0};   // padded real rows along axis 0 / axis 1
  PassCfg cfg[2];      // [0]: lanes along axis 1 (arrays stored P0 x P1); [1]: lanes along axis 0
  bool transforms_ok = false;
  size_t elems() const { return (size_t)P[0] * P[1] / ctx->nranks; }   // local slab
  double* tmp[6] = {nullptr};  // scratch arrays
  int refs = 0;
};

struct b2_array {
  b2_space* sp;
  double* d;
  int shape_kind;
};

struct b2_field {
  b2_space* sp;
  b2_array* v;
  b2_array* vhat;
};

// One product of gemm_f64.cuh: the packed operand(s) and the launch geometry (B / C are bound at run time).
struct GemmPlan {
  DVecD A[2];
  GemmParams p;
  int grid = 0;
};

struct b2_solver {
  b2_space* sp = nullptr;
  int type = 0;  // 0 hholtz_adi, 1 poisson
  // per axis: banded LU (Chebyshev) or reciprocal diagonal (Fourier)
  DVecD fl[2], id[2], u1[2], u2[2], sd[2], pd[2];   // pd: packed PdmaPlus2 LU (ChebDirichletNeumann axis)
  int pd_L[2] = {0, 0};
  // poisson
  bool dense = false;
  int m0 = 0;
  DVecD pfl, pid, pu1, pu2; // per-lane LU in scan layout
  // parity blocks: the eigenvectors couple indices of equal parity only, so with the modes grouped by parity class both
  // GEMMs split into two half-size GEMMs (half the flops)
  bool blocks = false;
  int ce = 0, co = 0;       // even / odd indices (= modes of the even / odd class)
  DVecD qfl, qid, qu1, qu2; // per-lane LU for the parity-grouped mode order
  // own FP64 GEMM on the tiled arrays (gemm_f64.cuh): forward (x -> eigenmodes) and backward products
  GemmPlan gf, gb;
  bool own_gemm = false;
};

// ------------------------------------------------------------------------------------------------
// helper kernels
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ size_t tiled_index(int r, int c, int tiles) {
  return ((size_t)(r >> 2) * tiles + (c >> 2)) * 16 + (r & 3) * 4 + (c & 3);
}
// host layout (row-major real, or complex interleaved) <-> tiled real rows (complex => rows 2k / 2k+1)
__global__ void k_host_layout(double* tiled, double* plain, int rows, int cols, int tiles, int cplx, int to_tiled) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)rows * cols;
  if (idx >= total) return;
  int r = (int)(idx / cols), c = (int)(idx % cols);
  size_t p = cplx ? (((size_t)(r >> 1) * cols + c) * 2 + (r & 1)) : idx;
  size_t t = tiled_index(r, c, tiles);
  if (to_tiled) tiled[t] = plain[p]; else plain[p] = tiled[t];
}
__global__ void k_axpby(size_t n, double* __restrict__ y, double a, const double* __restrict__ x, double b) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) y[i] = a * x[i] + b * y[i];
}
// out = (acc ? out : 0) + u * p
__global__ void k_muladd(size_t n, double* __restrict__ out, const double* __restrict__ u, const double* __restrict__ p, int acc) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) out[i] = (acc ? out[i] : 0.0) + u[i] * p[i];
}
__global__ void k_sumsq(size_t n, const double* __restrict__ x, double* out) {
  __shared__ double sh[32];
  double s = 0;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) s += x[i] * x[i];
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (threadIdx.x == 0) atomicAdd(out, s);
  }
}

// dst = alpha * a * b (op 0), alpha * sqrt(a^2 + b^2) (op 1), dst + alpha * a * b (op 2): pointwise on arrays of one layout
__global__ void k_combine(size_t n, double* __restrict__ dst, const double* __restrict__ a, const double* __restrict__ b, int op, double alpha) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    const double x = a[i], y = b[i];
    dst[i] = op == 0 ? alpha * x * y : (op == 1 ? alpha * sqrt(x * x + y * y) : dst[i] + alpha * x * y);
  }
}
// dx-weighted sums of a tiled real array slab (src/field/average.rs:26-59): thread per column j,
//   out[j] = sum_i w0[i] a[i][j]  (mode 1)   or   out[0] += w1[j] * that  (mode 0)
__global__ void k_weighted_sum(const double* __restrict__ a, int rows, int cols, int tiles, const double* __restrict__ w0,
                               const double* __restrict__ w1, int mode, double* out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  double s = 0.0;
  if (j < cols)
    for (int i = 0; i < rows; i++) s += w0[i] * a[tiled_index(i, j, tiles)];
  if (mode == 1) { if (j < cols) out[j] = s; return; }
  s *= (j < cols) ? w1[j] : 0.0;
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, s);
}
// mode 2: thread per local row i, out[i] = sum_j w1[j] a[i][j]  (average_axis(1): one value per x row of this rank's slab)
__global__ void k_weighted_rowsum(const double* __restrict__ a, int rows, int cols, int tiles, const double* __restrict__ w1, double* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  double s = 0.0;
  for (int j = 0; j < cols; j++) s += w1[j] * a[tiled_index(i, j, tiles)];
  out[i] = s;
}

static int ew_grid(size_t n) { return (int)std::min<size_t>((n + 255) / 256, 148 * 8); }

// ------------------------------------------------------------------------------------------------
// program builder / launcher
// ------------------------------------------------------------------------------------------------
static int pack_offs(int o0, int o1, int o2) { return (o0 & 0xff) | ((o1 & 0xff) << 8) | ((o2 & 0xff) << 16); }

struct Prog {
  LaneProg p;
  int err = B2_OK;
  Prog() { memset(&p, 0, sizeof(p)); }
  LaneOp* add(int code) {
    if (p.nops >= B2_MAXOPS) { err = fail(B2_ERR_ARG, "lane program too long"); return &p.ops[B2_MAXOPS - 1]; }
    LaneOp* o = &p.ops[p.nops++];
    memset(o, 0, sizeof(*o));
    o->code = code; o->a = 1.0;
    return o;
  }
  void load(const double* src, int len, double a = 1.0, int flags = 0, int i1 = 0) { LaneOp* o = add(OP_LOAD); o->p0 = src; o->i0 = len; o->a = a; o->i2 = flags; o->i1 = i1; }
  void store(double* dst, int len, int flags, double a = 1.0, int i1 = 0) { LaneOp* o = add(OP_STORE); o->p0 = dst; o->i0 = len; o->a = a; o->i2 = flags; o->i1 = i1; }
  void band(int len_out, int len_in, int o0, const double* c0, int o1, const double* c1, int o2 = 127, const double* c2 = nullptr) {
    LaneOp* o = add(OP_BAND); o->i0 = len_out; o->i2 = len_in; o->i1 = pack_offs(o0, o1, o2); o->p0 = c0; o->p1 = c1; o->p2 = c2;
  }
  void deriv(int n, int times, double scale) { LaneOp* o = add(OP_DERIV); o->i0 = n; o->i1 = times; o->a = scale; }
  void fdma(int len, const double* fl, const double* id, const double* u1, const double* u2, int flags) {
    LaneOp* o = add(OP_FDMA); o->i0 = len; o->i2 = flags; o->p0 = fl; o->p1 = id; o->p2 = u1; o->p3 = u2;
  }
  void dense(int n_out, int n_in, const double* M) { LaneOp* o = add(OP_DENSE); o->i0 = n_out; o->i1 = n_in; o->p0 = M; }
  void dct(const Base1& b, int mode) {
    if (b.dense_tr) { dense(b.n, b.n, mode == 0 ? b.d_dfwd.d : b.d_dbwd.d); return; }
    LaneOp* o = add(OP_DCT); o->i0 = b.n; o->i1 = mode; o->p0 = b.d_tw.d; o->p1 = b.d_tw2.d; o->p2 = b.d_isin.d; }
  void rfft(const Base1& b, int mode) {
    if (b.dense_tr) { if (mode == 0) dense(b.rows_ortho, b.rows_phys, b.d_dfwd.d); else dense(b.rows_phys, b.rows_ortho, b.d_dbwd.d); return; }
    LaneOp* o = add(OP_RFFT); o->i0 = b.n; o->i1 = mode; o->p0 = b.d_tw.d; o->p1 = b.d_tw2.d; }
  void fdiff(int modes, int d, double scale, int wrap = 0) { LaneOp* o = add(OP_FDIFF); o->i0 = modes; o->i1 = d; o->a = scale; o->i2 = wrap; }
  void scalevec(int len, const double* v, int shift) { LaneOp* o = add(OP_SCALEVEC); o->i0 = len; o->i1 = shift; o->p0 = v; }
  void zerotail(int from) { LaneOp* o = add(OP_ZEROTAIL); o->i0 = from; }
  void lanemask(int from) { LaneOp* o = add(OP_LANEMASK); o->i0 = from; }
  void zeroelem(int lane, int pos) { LaneOp* o = add(OP_ZEROELEM); o->i0 = lane; o->i1 = pos; }
  void scale(double a) { LaneOp* o = add(OP_SCALE); o->a = a; }

  // ---- per-axis operator chains (funspace semantics, SURVEY Appendix A) ----
  // returns the new valid length along the lane
  void sten3(int len_out, int mode, const Base1& b) { LaneOp* o = add(OP_STEN3); o->i0 = len_out; o->i1 = mode; o->p0 = b.d_ca.d; o->p1 = b.d_cb.d; }
  void pdma(int n, const double* packed, int L) { LaneOp* o = add(OP_PDMA); o->i0 = n; o->i1 = L; o->p0 = packed; }
  int to_ortho(const Base1& b) {
    if (b.composite) { band(b.n, b.m, 0, nullptr, -2, b.d_sten2s.d); return b.n; }
    if (b.cdn) { sten3(b.n, 0, b); return b.n; }
    return b.rows_ortho;
  }
  int from_ortho(const Base1& b) {
    if (b.cdn) { sten3(b.m, 1, b); pdma(b.m, b.d_pent.d, b.pent_L); return b.m; }
    if (b.composite) {
      band(b.m, b.n, 0, nullptr, 2, b.d_s2.d);
      fdma(b.m, b.d_tfl.d, b.d_tid.d, b.d_tu1.d, nullptr, FD_NOU2);
      return b.m;
    }
    return b.rows_spec;
  }
  int deriv_axis(const Base1& b, int d, double sc) {  // on ortho coefficients; sc = 1/scale^d
    if (d == 0) { if (sc != 1.0) scale(sc); return b.rows_ortho; }
    if (b.cheb) deriv(b.n, d, sc); else fdiff(b.m, d, sc, b.c2c ? b.n : 0);
    return b.rows_ortho;
  }
  int backward_ortho(const Base1& b) {  // ortho coefficients -> physical values
    if (b.cheb) dct(b, 1); else rfft(b, 1);
    return b.rows_phys;
  }
  int forward_ortho(const Base1& b) {   // physical values -> ortho coefficients
    if (b.cheb) dct(b, 0); else rfft(b, 0);
    return b.rows_ortho;
  }
  void load_stencil(const double* src, const Base1& b, double a, bool acc) {  // W [+]= a * to_ortho(src) along the lane
    LaneOp* o = add(OP_LOAD); o->p0 = src; o->a = a;
    o->i0 = b.rows_ortho;
    if (b.cdn) err = fail(B2_ERR_UNSUPPORTED, "stencil-on-load is pair-structured (ChebDirichletNeumann uses OP_STEN3)");
    o->i2 = (acc ? LD_ACC : 0) | (b.composite ? LD_STENCIL : 0);
    o->p1 = b.d_sten2.d;
  }
  int matvec(const Base1& b) {          // MatVecFdma with pinv (Chebyshev axes only)
    if (b.composite || b.cdn) { band(b.m, b.n, 0, b.d_bd.d, 2, b.d_bu1.d, 4, b.d_bu2.d); return b.m; }
    return b.rows_spec;
  }
};

template <int E, int LN, int TPLC> static int launch_ELT(b2_ctx* ctx, const PassCfg& c, const LaneProg& p) {
  static size_t set_smem[64] = {0};   // per device: the attribute belongs to the (function, device) pair
  size_t& have = set_smem[ctx->device & 63];
  if (c.smem > have) {
    CK(cudaFuncSetAttribute(lane_kernel<E, LN, TPLC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem));
    have = c.smem;
  }
  B2_LAUNCH((lane_kernel<E, LN, TPLC>), (c.groups / ctx->nranks) * (4 / c.LN), c.NT, c.smem, ctx->cur, p);
  CK(cudaGetLastError());
  return B2_OK;
}
// Kernel instances: transform-sized lanes (c.fast) get the compile-time-geometry instance of their (E, LN, TPL);
// every other geometry runs the generic instance of its (E, LN).
static int launch_pass(b2_ctx* ctx, const PassCfg& c, const LaneProg& p) {
#define B2_INST(e, ln, tpl) if (c.fast && c.E == e && c.LN == ln && c.TPL == tpl) return launch_ELT<e, ln, tpl>(ctx, c, p);
  B2_INST(16, 4, 128) B2_INST(16, 4, 64) B2_INST(16, 4, 32) B2_INST(16, 4, 16) B2_INST(16, 4, 8)
  B2_INST(16, 2, 256) B2_INST(16, 2, 128)
  B2_INST(8, 4, 64) B2_INST(8, 4, 32) B2_INST(8, 4, 16) B2_INST(8, 4, 8) B2_INST(4, 4, 8) B2_INST(4, 4, 16) B2_INST(4, 4, 32)
#undef B2_INST
  // the launcher has already rewritten band ops into OP_BANDC / OP_PREBAND, which the generic instances do not implement:
  // a fast layout that has_fast_instance accepts but the list above lacks would otherwise give wrong results without an error
  if (c.fast) return fail(B2_ERR_ARG, "internal: fast layout E/LN/TPL without a compiled instance");
  if (c.LN == 4) {
    if (c.E == 16) return launch_ELT<16, 4, 0>(ctx, c, p);
    if (c.E == 8) return launch_ELT<8, 4, 0>(ctx, c, p);
    return launch_ELT<4, 4, 0>(ctx, c, p);
  }
  if (c.E == 16) return launch_ELT<16, 2, 0>(ctx, c, p);
  if (c.E == 8) return launch_ELT<8, 2, 0>(ctx, c, p);
  return launch_ELT<4, 2, 0>(ctx, c, p);
}

static bool g_use_tma = getenv("B2_NOTMA") == nullptr;     // B2_NOTMA=1: every load/store on the per-thread LDG/STG path (A/B measurements)
static bool g_use_ring = getenv("B2_LDTHREADS") == nullptr;  // combining loads (accumulate / multiply / stencil / scaled) stream through the warps' own
                                                             // copy pipelines (load_warps); B2_LDTHREADS=1: per-thread 16-byte loads instead

// orient 0: lanes along axis 1; orient 1: lanes along axis 0
static int run_pass(b2_space* sp, int orient, Prog& pr) {
  if (pr.err != B2_OK) return pr.err;
  const PassCfg& c = sp->cfg[orient];
  LaneProg& p = pr.p;
  b2_ctx* ctx = sp->ctx;
  p.LP = c.LP; p.in_tiles = c.in_tiles; p.out_tiles = c.out_tiles; p.TPL = c.TPL; p.C = c.C;
  p.group0 = ctx->rank * (c.groups / ctx->nranks); p.groups_per_rank = c.in_tiles / ctx->nranks; p.rank = ctx->rank;
  p.prof = ctx->d_prof; p.LN = c.LN;
  p.NT = c.NT; p.CHW = c.CHW; p.nsc = c.nsc; p.wslot_bytes = c.wslot_bytes; p.CHD = c.CHD; p.nchd = c.nchd;
  p.w_off = c.w_off; p.st_off = c.st_off;
  p.bulk1d = c.LN == 4 ? 1 : 0;   // a whole lane group is one contiguous slab: 1-D bulk copies, no tensor map
  bool exchange = false;
  int npst = 0;
  if (ctx->nranks > 1) {   // a transposing store is the pencil transpose: tiles go straight into the owner's slab
    for (int i = 0; i < p.nops; i++)
      if (p.ops[i].code == OP_STORE && (p.ops[i].i2 & ST_TRANS)) { p.ops[i].i2 |= ST_PEER; p.ops[i].p1 = ctx->d_peers; exchange = true; }
      else if (p.ops[i].code == OP_STORE && (p.ops[i].i2 & ST_COLSPLIT)) { p.ops[i].p1 = ctx->d_peers; exchange = true; }
  } else {
    for (int i = 0; i < p.nops; i++) if (p.ops[i].code == OP_STORE) p.ops[i].i2 &= ~ST_COLSPLIT;   // one GPU: a plain same-orientation store
  }
  // Generic geometry: a tiled load followed by the composite -> orthonormal stencil (to_ortho: y_j = x_j + s_j x_{j-2}) becomes
  // ONE load that applies the stencil on the fly (LD_STENCIL).  Transform-sized lanes keep the zero-copy load and run the
  // stencil as a chunk-streaming band op instead (measured on C4: stencil-on-load through the staging slots 20-22k cycles
  // per lane group, zero-copy load + band_chunk 5.7k + 9.8k; profiles/r02/sweep_*.log).
  for (int i = 0; !c.fast && i + 1 < p.nops; i++) {
    LaneOp& lo = p.ops[i]; LaneOp& bo = p.ops[i + 1];
    if (lo.code != OP_LOAD || (lo.i2 & (LD_PLAIN | LD_STENCIL | LD_ACC | LD_MUL)) || bo.code != OP_BAND) continue;
    const int h0 = (int)(signed char)(bo.i1 & 0xff), h1 = (int)(signed char)((bo.i1 >> 8) & 0xff), h2 = (int)(signed char)((bo.i1 >> 16) & 0xff);
    if (h0 != 0 || bo.p0 != nullptr || h1 != -2 || bo.p1 == nullptr || h2 != 127 || bo.i2 != lo.i0) continue;   // not to_ortho of what was loaded
    lo.i2 |= LD_STENCIL; lo.p1 = bo.p1; lo.i0 = bo.i0;
    bo.code = OP_PREBAND;   // no-op
  }
  // Fold a banded mat-vec into the LU solve that consumes it (forward offsets only, same output length; shared
  // coefficient vectors): the solve forms its right-hand side on the fly (lane_fast.cuh, fdma_fast_body<PREBAND>).
  // Measured: +1.5 % on C2 (E = 8), -2 % on C4 (E = 16, where the extra coefficient streams cost more than the saved
  // pass), so it is applied to the short-lane instances only.
  if (c.fast && c.E <= 8) {
    for (int i = 0; i + 1 < p.nops; i++) {
      LaneOp& bo = p.ops[i]; LaneOp& fo = p.ops[i + 1];
      if (bo.code != OP_BAND || fo.code != OP_FDMA || (fo.i2 & FD_PERLANE) || bo.i0 != fo.i0) continue;
      bool ok = true;
      const void* sc[3] = {nullptr, nullptr, nullptr};
      const void* nat[3] = {bo.p0, bo.p1, bo.p2};
      for (int m = 0; m < 3; m++) {
        const int h = (int)(signed char)((bo.i1 >> (8 * m)) & 0xff);
        if (h == 127) continue;
        if (h != 0 && h != 2 && h != 4) ok = false;
        if (nat[m]) { auto it = scan_of().find(nat[m]); if (it == scan_of().end()) ok = false; else sc[m] = it->second; }
      }
      if (!ok) continue;
      bo.code = OP_PREBAND; bo.p0 = sc[0]; bo.p1 = sc[1]; bo.p2 = sc[2]; fo.i2 |= FD_PREBAND;
    }
  }
  // Remaining banded mat-vecs on transform-sized lanes run in chunk-streaming form (band_chunk: one read and one write
  // traversal of the lane group): pair offsets {0, +1, +2} or {0, -1}, vector coefficients through their scan-layout copies.
  if (c.fast) {
    for (int i = 0; i < p.nops; i++) {
      LaneOp& bo = p.ops[i];
      if (bo.code != OP_BAND) continue;
      const void* nat[3] = {bo.p0, bo.p1, bo.p2};
      const void* slot[3] = {nullptr, nullptr, nullptr};
      int flag[3] = {0, 0, 0};
      bool ok = true, anyvec = false, fwd = false, bwd = false;
      for (int m = 0; m < 3 && ok; m++) {
        const int h = (int)(signed char)((bo.i1 >> (8 * m)) & 0xff);
        if (h == 127) continue;
        int k;
        if (h == 0) k = 0; else if (h == 2) { k = 1; fwd = true; } else if (h == 4) { k = 2; fwd = true; } else if (h == -2) { k = 1; bwd = true; } else { ok = false; break; }
        if (flag[k]) { ok = false; break; }
        if (nat[m]) { auto it = scan_of().find(nat[m]); if (it == scan_of().end()) { ok = false; break; } slot[k] = it->second; flag[k] = 2; anyvec = true; }
        else flag[k] = 1;
      }
      if (!ok || !anyvec || (fwd && bwd)) continue;
      bo.code = OP_BANDC; bo.p0 = slot[0]; bo.p1 = slot[1]; bo.p2 = slot[2];
      bo.i1 = (bwd ? 1 : 0) | (flag[0] << 2) | (flag[1] << 4) | (flag[2] << 6);
    }
  }
  // TMA views.  Arrays are 4x4-tiled: tile (I, J) at ((I * tiles_per_row) + J) * 128 bytes, element [i][j] inside.
  //   slab view (loads, same-orientation stores): [16 doubles of a tile][tile J of the lane group][lane group]
  //   transposed view (transposing stores): tile (J, g) of the destination holds [jl][lane]:
  //                   [lane 0..3][jl 0..3][g : tile column][J : tile row]
  const int groups_local = c.groups / ctx->nranks;
  for (int i = 0; i < p.nops && g_use_tma; i++) {
    LaneOp& op = p.ops[i];
    B2TMapDesc d; memset(&d, 0, sizeof(d));
    if (op.code == OP_LOAD && !(op.i2 & LD_PLAIN)) {
      const bool direct = !(op.i2 & (LD_ACC | LD_MUL | LD_STENCIL)) && op.a == 1.0;
      for (int k = 0; k < i; k++)   // re-reading an array this program stored: the bulk stores have to be complete first
        if (p.ops[k].code == OP_STORE && p.ops[k].p0 == op.p0) op.i2 |= LD_AFTER_STORE;
      if (!direct && !g_use_ring) continue;   // per-thread path (B2_LDTHREADS=1)
      d.base = const_cast<void*>(op.p0); d.rank = 3;
      d.dim[0] = 16; d.dim[1] = (uint64_t)c.in_tiles; d.dim[2] = (uint64_t)groups_local;
      d.stride[1] = 128; d.stride[2] = (uint64_t)c.in_tiles * 128;
      d.box[0] = 4 * c.LN; d.box[1] = direct ? c.CHD : c.CHW + 1; d.box[2] = 1;
      op.i2 |= direct ? LD_DIRECT : LD_TMA;
    } else if (op.code == OP_STORE && (op.i2 & ST_PEER) && !(op.i2 & ST_PLAIN)) {
      // one transposed view per owner: rows = the tiles of the destination that live in that rank's slab
      static const bool peer_threads = getenv("B2_PEER_THREADS") != nullptr;   // debugging: per-thread peer stores instead of tensor stores
      if (npst >= B2_MAXPST || peer_threads) continue;   // (more peer views than the program has room for: per-thread peer stores)
      const int gpr = c.in_tiles / ctx->nranks;
      for (int o = 0; o < ctx->nranks; o++) {
        B2TMapDesc dd; memset(&dd, 0, sizeof(dd));
        dd.base = static_cast<char*>(ctx->peer_base[o]) + (static_cast<const char*>(op.p0) - static_cast<const char*>(ctx->peer_base[ctx->rank]));
        if (c.LN == 4) {   // whole tiles: [16 doubles of a tile][tile column g][tile row J]
          dd.rank = 3;
          dd.dim[0] = 16; dd.dim[1] = (uint64_t)c.out_tiles; dd.dim[2] = (uint64_t)gpr;
          dd.stride[1] = 128; dd.stride[2] = (uint64_t)c.out_tiles * 128;
          dd.box[0] = 16; dd.box[1] = 1; dd.box[2] = c.CHW;
        } else {
          dd.rank = 4;
          dd.dim[0] = 4; dd.dim[1] = 4; dd.dim[2] = (uint64_t)c.out_tiles; dd.dim[3] = (uint64_t)gpr;
          dd.stride[1] = 32; dd.stride[2] = 128; dd.stride[3] = (uint64_t)c.out_tiles * 128;
          dd.box[0] = c.LN; dd.box[1] = 4; dd.box[2] = 1; dd.box[3] = c.CHW;
        }
        const int er = b2_encode_tmap(dd, &p.tmp[npst][o]);
        if (er) return fail(B2_ERR_CUDA, "cuTensorMapEncodeTiled failed for a peer view (" + std::to_string(er) + ")");
      }
      op.i1 = npst++;
      op.i2 |= ST_TMA;
      continue;
    } else if (op.code == OP_STORE && !(op.i2 & (ST_PLAIN | ST_PEER))) {
      d.base = const_cast<void*>(op.p0);
      if (op.i2 & ST_TRANS) {
        if (c.LN == 4) {   // whole tiles: [16 doubles of a tile][tile column g][tile row J], 128-byte rows
          d.rank = 3;
          d.dim[0] = 16; d.dim[1] = (uint64_t)c.out_tiles; d.dim[2] = (uint64_t)c.in_tiles;
          d.stride[1] = 128; d.stride[2] = (uint64_t)c.out_tiles * 128;
          d.box[0] = 16; d.box[1] = 1; d.box[2] = c.CHW;
        } else {
          d.rank = 4;
          d.dim[0] = 4; d.dim[1] = 4; d.dim[2] = (uint64_t)c.out_tiles; d.dim[3] = (uint64_t)c.in_tiles;
          d.stride[1] = 32; d.stride[2] = 128; d.stride[3] = (uint64_t)c.out_tiles * 128;
          d.box[0] = c.LN; d.box[1] = 4; d.box[2] = 1; d.box[3] = c.CHW;
        }
        op.i2 |= ST_TMA;
      } else {
        const bool direct = !(op.i2 & ST_ACC) && op.a == 1.0;
        if (op.i2 & ST_COLSPLIT) {   // zero-copy runs per owner (contiguous slabs only), else per-thread peer stores
          if (direct && p.bulk1d) op.i2 |= ST_DIRECT;
          continue;
        }
        d.rank = 3;
        d.dim[0] = 16; d.dim[1] = (uint64_t)c.in_tiles; d.dim[2] = (uint64_t)groups_local;
        d.stride[1] = 128; d.stride[2] = (uint64_t)c.in_tiles * 128;
        d.box[0] = 4 * c.LN; d.box[1] = direct ? c.CHD : c.CHW; d.box[2] = 1;
        op.i2 |= direct ? ST_DIRECT : ST_TMA;
      }
    } else continue;
    const int er = b2_encode_tmap(d, &p.tm[i]);
    if (er) return fail(B2_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string(er) + ")");
  }
  ctx->launches++;
  const int r = launch_pass(ctx, c, p);
  if (r != B2_OK) return r;
  static const bool dbg_sync = getenv("B2_DEBUG_SYNC") != nullptr;   // debugging: name the pass a device fault belongs to
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (dbg_sync) cudaStreamIsCapturing(ctx->cur, &cap);
  if (dbg_sync && cap == cudaStreamCaptureStatusNone) {
    cudaError_t e = cudaStreamSynchronize(ctx->cur);
    if (e != cudaSuccess) {
      std::string ops;
      for (int i = 0; i < p.nops; i++) ops += std::to_string(p.ops[i].code) + ":" + std::to_string(p.ops[i].i2) + " ";
      return fail(B2_ERR_CUDA, std::string("pass failed (") + cudaGetErrorString(e) + "), orient " + std::to_string(orient) + ", ops code:flags = " + ops);
    }
  }
  return exchange ? ctx_barrier(ctx) : B2_OK;
}

// ------------------------------------------------------------------------------------------------
// context / space / arrays
// ------------------------------------------------------------------------------------------------
// the (E, LN, TPL) combinations that have a compile-time-geometry kernel instance (launch_pass): only those may run the
// launcher's fast-geometry rewrites (OP_BANDC, OP_PREBAND) -- the generic instances do not implement them
static bool has_fast_instance(int E, int LN, int TPL) {
  if (LN == 2) return E == 16 && (TPL == 256 || TPL == 128);
  if (E == 16) return TPL == 128 || TPL == 64 || TPL == 32 || TPL == 16 || TPL == 8;
  if (E == 8) return TPL == 64 || TPL == 32 || TPL == 16 || TPL == 8;
  if (E == 4) return TPL == 8 || TPL == 16 || TPL == 32;
  return false;
}
static int make_cfg(const Base1& lane_base, int Pl, int Pc, PassCfg* c, int nranks) {
  c->in_tiles = Pl / 4; c->out_tiles = Pc / 4; c->groups = Pc / 4; c->LP = Pl;
  const int N = lane_base.N;
  // E = FFT points per thread; a thread also owns CP = E+1 element pairs of the lane for the banded ops,
  // so the lane (LP doubles) must fit in 2*CP*TPL.  LN = lanes per CTA (4 = whole lane group, 2 = half).
  int ln_want = 4;
  if (const char* e = getenv("B2_LN")) { if (atoi(e) == 2) ln_want = 2; }
  auto pick = [&](int LN, int want) -> bool {
    const int Nc = N / 2;
    for (int e = want; e >= 4; e /= 2) {
      const int tpl = Nc / e;
      if (tpl >= 8 && (tpl * LN) % 32 == 0 && tpl * LN <= 512 && tpl <= 256 && 2 * (e + 1) * tpl >= Pl) { c->E = e; c->TPL = tpl; c->LN = LN; return true; }
    }
    return false;
  };
  if (is_pow2(N) && N >= 64) {
    const int Nc = N / 2;
    int want = Nc >= 1024 ? 16 : (Nc >= 64 ? 8 : 4);   // short lanes: fewer points per thread = more threads per lane
    if (const char* e = getenv("B2_E")) {   // tuning knob
      int ev = atoi(e);
      if (ev == 4 || ev == 8 || ev == 16) want = ev;
    }
    c->E = 0;
    const size_t smem4 = ((size_t)4 * Pl + 32 * 12) * sizeof(double);
    bool ok = false;
    if (ln_want == 4 && smem4 <= 227 * 1024) ok = pick(4, want) || pick(4, 16);
    if (!ok) ok = pick(2, want) || pick(2, 16);
    if (!ok && smem4 <= 227 * 1024) ok = pick(4, want) || pick(4, 16);
    if (!ok) return fail(B2_ERR_UNSUPPORTED, "lane of " + std::to_string(Pl) + " points: no supported thread layout");
  } else {  // no transform along this axis: banded ops only
    c->E = 16; c->LN = 4;
    int t = 8;
    while (2 * 17 * t < Pl) t *= 2;
    c->TPL = t;
    if (t > 128) return fail(B2_ERR_UNSUPPORTED, "lane too long");
  }
  c->C = c->E + 1;
  c->NT = c->LN * c->TPL;
  c->fast = is_pow2(N) && N >= 64 && N == 2 * c->E * c->TPL && Pl >= N + 4 && has_fast_instance(c->E, c->LN, c->TPL) && getenv("B2_NOFAST") == nullptr;
  if (c->NT % 32) return fail(B2_ERR_UNSUPPORTED, "compute threads must fill whole warps");
  // shared memory: [mbarriers][program copy][scratch][W][per warp: 2 staging slots of CHW + 1 tiles]
  const int tile_bytes = c->LN * 32;
  c->nchd = (c->in_tiles + 255) / 256;                     // direct copies: boxes of <= 256 tiles straight into / out of W
  c->CHD = roundup((c->in_tiles + c->nchd - 1) / c->nchd, 4 / c->LN);   // box bytes multiple of 128: TMA shared-memory alignment
  const size_t budget = 227 * 1024, fixed = B2_BARBYTES + B2_PROGCOPY + B2_SCRATCH;
  const size_t wbytes = (size_t)roundup(c->nchd * c->CHD * tile_bytes, 128);   // the last direct box may overhang the lane by < nchd tiles
  if (fixed + wbytes > budget) return fail(B2_ERR_UNSUPPORTED, "lane group does not fit in shared memory");
  // short lanes: keep the CTA near 72 KB so that three fit on an SM; long lanes: one CTA owns the SM
  size_t room = budget - fixed - wbytes;
  if (wbytes <= 40 * 1024) room = std::min(room, std::max((size_t)8192, (size_t)72 * 1024 - std::min((size_t)72 * 1024, fixed + wbytes)));
  if (const char* e = getenv("B2_SMEMCAP")) {   // tuning knob: total dynamic shared memory per CTA in KB (e.g. 113 = two CTAs per SM)
    const size_t cap = (size_t)atoi(e) * 1024;
    if (cap > fixed + wbytes + 4096) room = std::min(room, cap - fixed - wbytes);
  }
  const int nwarps = c->NT / 32;
  int chw = (int)(room / ((size_t)nwarps * 2) / tile_bytes) - 1;   // one halo tile in front of every slot
  if (const char* e = getenv("B2_CHW")) { int v = atoi(e); if (v >= 2) chw = std::min(chw, v); }
  chw = std::max(2, std::min(chw, std::min(64, c->in_tiles)));
  if (wbytes > 100 * 1024) chw = std::min(chw, 12);   // long lanes: 12-tile sub-chunks pipeline better than the largest that fit (C4: lane time 8.50 -> 8.27 ms)
  if (nranks > 1) chw = std::max(2, std::min(chw, c->in_tiles / nranks));   // a sub-chunk's tensor-store box never exceeds one owner's rows of the transposed view
  if (c->LN == 2 && (chw % 2 == 0)) chw--;                 // (CHW + 1) tiles of 64 bytes: a multiple of 128
  c->CHW = chw;
  c->nsc = (c->in_tiles + chw - 1) / chw;
  c->wslot_bytes = roundup((chw + 1) * tile_bytes, 128);
  c->w_off = (int)fixed; c->st_off = c->w_off + (int)wbytes;
  c->smem = (size_t)c->st_off + (size_t)nwarps * 2 * c->wslot_bytes;
  if (c->smem > budget) return fail(B2_ERR_UNSUPPORTED, "lane group does not fit in shared memory");
  return B2_OK;
}

static int alloc_zero(b2_space* sp, double** out) {
  RET(ctx_alloc(sp->ctx, sp->elems() * sizeof(double), out));
  CK(cudaMemsetAsync(*out, 0, sp->elems() * sizeof(double), sp->ctx->stream));
  // several GPUs: a peer may store into this array as soon as ITS allocation returns -- not before every rank has cleared its copy
  // (allocation is collective on the symmetric heap: every rank allocates the same arrays in the same order)
  // The same exchange checks that the heaps are still symmetric (host code that releases arrays at different moments on different
  // ranks -- e.g. garbage collection -- would otherwise corrupt other arrays silently).
  b2_ctx* c = sp->ctx;
  if (c->nranks > 1 && c->attached) {
    if (!c->d_differs) CK(cudaMalloc(&c->d_differs, sizeof(int)));
    const unsigned long long off = (unsigned long long)(reinterpret_cast<char*>(*out) - c->heap);
    B2_LAUNCH(k_same_value, 1, 32, 0, c->stream, reinterpret_cast<unsigned long long* const*>(c->d_peers), c->rank, c->nranks, off, c->d_differs);
    CK(cudaGetLastError());
    c->barriers++;
    int differs = 0;
    CK(cudaMemcpyAsync(&differs, c->d_differs, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (differs) return fail(B2_ERR_ARG, "symmetric heap diverged: the ranks did not create / release their arrays in the same order (offset " + std::to_string(off) + " on rank " + std::to_string(c->rank) + ")");
  }
  return B2_OK;
}

static int shape_of(const b2_space* sp, int shape_kind, int* rows, int* cols) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  switch (shape_kind) {
    case B2_SHAPE_PHYSICAL: *rows = b0.rows_phys; *cols = b1.rows_phys; return B2_OK;
    case B2_SHAPE_SPECTRAL: *rows = b0.rows_spec; *cols = b1.rows_spec; return B2_OK;
    case B2_SHAPE_ORTHO: *rows = b0.rows_ortho; *cols = b1.rows_ortho; return B2_OK;
  }
  return fail(B2_ERR_ARG, "bad shape kind");
}
static bool shape_complex(const b2_space* sp, int shape_kind) { return !sp->b[0].cheb && (shape_kind != B2_SHAPE_PHYSICAL || sp->b[0].c2c); }

// ------------------------------------------------------------------------------------------------
// field operators (2 passes each: along y, transpose, along x, transpose back)
// ------------------------------------------------------------------------------------------------
static int op_forward(b2_space* sp, const double* v, double* vhat) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  if (!sp->transforms_ok) return fail(B2_ERR_UNSUPPORTED, "transform size: n-1 (Chebyshev) / n (Fourier) = 2^k >= 64 runs the FFT core, other sizes up to 2049 a dense matrix; larger non-power-of-two sizes are not supported");
  Prog y; y.load(v, b1.rows_phys); y.forward_ortho(b1); int l = y.from_ortho(b1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_phys); x.forward_ortho(b0); l = x.from_ortho(b0); x.store(vhat, l, ST_TRANS);
  return run_pass(sp, 1, x);
}
static int op_backward(b2_space* sp, const double* vhat, double* v) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  if (!sp->transforms_ok) return fail(B2_ERR_UNSUPPORTED, "transform size: n-1 (Chebyshev) / n (Fourier) = 2^k >= 64 runs the FFT core, other sizes up to 2049 a dense matrix; larger non-power-of-two sizes are not supported");
  Prog y; y.load(vhat, b1.rows_spec); y.to_ortho(b1); int l = y.backward_ortho(b1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_spec); x.to_ortho(b0); l = x.backward_ortho(b0); x.store(v, l, ST_TRANS);
  return run_pass(sp, 1, x);
}
static int op_to_ortho(b2_space* sp, const double* vhat, double* out, double alpha = 1.0, bool acc = false) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  Prog y; y.load(vhat, b1.rows_spec); int l = y.to_ortho(b1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_spec); l = x.to_ortho(b0); x.store(out, l, ST_TRANS | (acc ? ST_ACC : 0), alpha);
  return run_pass(sp, 1, x);
}
static int op_from_ortho(b2_space* sp, const double* in, double* vhat, double alpha = 1.0, bool acc = false) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  Prog y; y.load(in, b1.rows_ortho); int l = y.from_ortho(b1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_ortho); l = x.from_ortho(b0); x.store(vhat, l, ST_TRANS | (acc ? ST_ACC : 0), alpha);
  return run_pass(sp, 1, x);
}
static int op_gradient(b2_space* sp, const double* vhat, int d0, int d1, const double* scale, double* out, double alpha = 1.0, bool acc = false) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  double s0 = 1.0, s1 = 1.0;
  if (scale) { s0 = 1.0 / std::pow(scale[0], d0); s1 = 1.0 / std::pow(scale[1], d1); }
  Prog y; y.load(vhat, b1.rows_spec); y.to_ortho(b1); int l = y.deriv_axis(b1, d1, s1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_spec); x.to_ortho(b0); l = x.deriv_axis(b0, d0, s0); x.store(out, l, ST_TRANS | (acc ? ST_ACC : 0), alpha);
  return run_pass(sp, 1, x);
}
// transforms of an orthonormal ("field" = ch x ch or r2c x ch) array, funspace backward_par / forward
static int op_backward_ortho(b2_space* sp, const double* ortho, double* phys) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  if (!sp->transforms_ok) return fail(B2_ERR_UNSUPPORTED, "transform size");
  Prog y; y.load(ortho, b1.rows_ortho); int l = y.backward_ortho(b1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_ortho); l = x.backward_ortho(b0); x.store(phys, l, ST_TRANS);
  return run_pass(sp, 1, x);
}
// forward + dealias (src/navier_stokes/functions.rs:72-82), result scaled by alpha
static int op_forward_ortho_dealias(b2_space* sp, const double* phys, double* ortho, bool dealias, double alpha = 1.0, bool acc = false) {
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  if (!sp->transforms_ok) return fail(B2_ERR_UNSUPPORTED, "transform size");
  // bit-exact index rule: n_x = shape0*2/3, n_y = shape1*2/3 with integer division on the spectral shape
  const int shape0 = b0.cheb ? b0.n : b0.m, shape1 = b1.cheb ? b1.n : b1.m;
  const int cut0 = (shape0 * 2 / 3) * (b0.cheb ? 1 : 2), cut1 = (shape1 * 2 / 3) * (b1.cheb ? 1 : 2);
  Prog y; y.load(phys, b1.rows_phys); int l = y.forward_ortho(b1); if (dealias) y.zerotail(cut1); y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_phys); l = x.forward_ortho(b0); if (dealias) x.zerotail(cut0);
  x.store(ortho, l, ST_TRANS | (acc ? ST_ACC : 0), alpha);
  return run_pass(sp, 1, x);
}

// ------------------------------------------------------------------------------------------------
// solvers
// ------------------------------------------------------------------------------------------------
static int upload_lu(const LuVecs& lu, const Base1& b, DVecD* fl, DVecD* id, DVecD* u1, DVecD* u2) {
  RET(fl->upload(b.scan_layout(lu.fl))); RET(id->upload(b.scan_layout(lu.id)));
  RET(u1->upload(b.scan_layout(lu.u1))); RET(u2->upload(b.scan_layout(lu.u2)));
  return B2_OK;
}

static int hholtz_create(b2_space* sp, double c0, double c1, b2_solver** out) {
  b2_solver* s = new b2_solver();
  s->sp = sp; s->type = 0;
  const double c[2] = {c0, c1};
  for (int ax = 0; ax < 2; ax++) {
    const Base1& b = sp->b[ax];
    const int L = sp->P[ax] + 64;
    if (b.composite) {  // mat = mat_a - mat_b * c, src/solver/hholtz_adi.rs:57-63
      Diags a = b.mat_a(), bm = b.mat_b(), mat(b.m);
      for (int i = 0; i < b.m; i++) {
        mat.low[i] = a.low[i] - bm.low[i] * c[ax];
        mat.dia[i] = a.dia[i] - bm.dia[i] * c[ax];
        mat.up1[i] = a.up1[i] - bm.up1[i] * c[ax];
        mat.up2[i] = a.up2[i] - bm.up2[i] * c[ax];
      }
      RET(upload_lu(sweep(mat), b, &s->fl[ax], &s->id[ax], &s->u1[ax], &s->u2[ax]));
    } else if (b.cdn) {  // PdmaPlus2::from_matrix(mat), src/solver/hholtz_adi.rs:64
      std::vector<double> d[7];
      b.cdn_hholtz_diags(c[ax], d);
      s->pd_L[ax] = L;
      RET(s->pd[ax].upload(pdma_sweep(b.m, d, L)));
    } else if (!b.cheb) {  // Sdma: dia = 1 - c * (-k^2), src/solver/sdma.rs:37-46
      std::vector<double> sd(L, 0.0);
      for (int k = 0; k < b.m; k++) {
        const double kk = (b.c2c && 2 * k >= b.n) ? k - b.n : k;   // FourierC2c: modes in FFT order
        sd[k] = 1.0 / (1.0 - (-kk * kk) * c[ax]);
      }
      RET(s->sd[ax].upload(sd));
    } else {
      delete s;
      return fail(B2_ERR_UNSUPPORTED, "HholtzAdi on an orthonormal Chebyshev axis is not on the Navier2D path");
    }
  }
  *out = s;
  return B2_OK;
}

static void emit_hh_axis(Prog& p, const b2_solver* s, int ax);
// HholtzAdi::solve_par, src/solver/hholtz_adi.rs:149-169 (axis operators commute; y first here)
static int hholtz_solve(b2_solver* s, const double* in, double* out) {
  b2_space* sp = s->sp;
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  Prog y; y.load(in, b1.rows_ortho); emit_hh_axis(y, s, 1);
  y.store(sp->tmp[0], b1.rows_spec, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_ortho); emit_hh_axis(x, s, 0);
  x.store(out, b0.rows_spec, ST_TRANS);
  return run_pass(sp, 1, x);
}

// laplacian / mass of axis ax as in Poisson::new (src/solver/poisson.rs:65-74)
// ------------------------------------------------------------------------------------------------
// FP64 GEMM on the tiled arrays (gemm_f64.cuh): host side
// ------------------------------------------------------------------------------------------------
// A (row-major, M x K, leading dimension ld) -> fragment order [slice mt][k stage][k4 step][8-row fragment][lane]:
// slice mt holds the global rows mt * mstep + row0 + [0, 64); zero outside M x K.
static std::vector<double> pack_gemm_a(const double* A, int M, int K, int ld, int nmt, int nks, int mstep, int row0) {
  std::vector<double> out((size_t)nmt * nks * G_ACHUNK, 0.0);
  for (int mt = 0; mt < nmt; mt++)
    for (int ks = 0; ks < nks; ks++)
      for (int kk = 0; kk < G_KK; kk++)
        for (int mf = 0; mf < 8; mf++)
          for (int lane = 0; lane < 32; lane++) {
            const int m = mt * mstep + row0 + 8 * mf + (lane >> 2), k = 4 * G_KK * ks + 4 * kk + (lane & 3);
            if (m < M && k < K) out[((((size_t)mt * nks + ks) * G_KK + kk) * 8 + mf) * 32 + lane] = A[(size_t)m * ld + k];
          }
  return out;
}
// Parity-block product: blocks (Ae: Me x Ke, Ao: Mo x Ko); dense product (Ao == nullptr): one M x K matrix run as two
// 64-row halves of 128-row slices over the same rows of B.
static int gemm_plan_create(b2_space* sp, GemmPlan* g, const double* Ae, int Me, int Ke, const double* Ao, int Mo, int Ko,
                            bool b_interleaved, bool c_interleaved) {
  GemmParams& p = g->p;
  memset(&p, 0, sizeof(p));
  const int Kmax = std::max(Ke, Ko);
  p.nks = (Kmax + 4 * G_KK - 1) / (4 * G_KK);
  if (Ao) {
    p.mstep = 64; p.bshift = 0; p.nmt = (std::max(Me, Mo) + 63) / 64;
    p.Mb[0] = Me; p.Mb[1] = Mo;
    RET(g->A[0].upload(pack_gemm_a(Ae, Me, Ke, Ke, p.nmt, p.nks, 64, 0)));
    RET(g->A[1].upload(pack_gemm_a(Ao, Mo, Ko, Ko, p.nmt, p.nks, 64, 0)));
    if (b_interleaved) { p.offB[0] = 0; p.offB[1] = 1; p.strB = 2; } else { p.offB[0] = 0; p.offB[1] = Ke; p.strB = 1; }
    if (c_interleaved) { p.offC[0] = 0; p.offC[1] = 1; p.strC = 2; } else { p.offC[0] = 0; p.offC[1] = Me; p.strC = 1; }
    if ((!b_interleaved && Ke % 4) || (!c_interleaved && Me % 4)) return fail(B2_ERR_UNSUPPORTED, "parity-block GEMM: the odd block must start on a tile row");
  } else {
    p.mstep = 128; p.bshift = 64; p.nmt = (Me + 127) / 128;
    p.Mb[0] = Me; p.Mb[1] = Me;
    RET(g->A[0].upload(pack_gemm_a(Ae, Me, Ke, Ke, p.nmt, p.nks, 128, 0)));
    RET(g->A[1].upload(pack_gemm_a(Ae, Me, Ke, Ke, p.nmt, p.nks, 128, 64)));
    p.offB[0] = p.offB[1] = 0; p.strB = 1; p.offC[0] = p.offC[1] = 0; p.strC = 1;
  }
  p.A[0] = g->A[0].d; p.A[1] = g->A[1].d;
  // B = this rank's [all rows][local columns] array, C = rows distributed over the ranks, all columns (one GPU: the same thing)
  const int nr = sp->ctx->nranks;
  p.TJc = sp->P[1] / 4; p.TJb = p.TJc / nr; p.rowsB = sp->P[0] / 4; p.jc0 = sp->ctx->rank * p.TJb;
  p.ncb = (p.TJb + 31) / 32;
  p.rows_per_rank = sp->P[0] / nr;
  p.peers = nr > 1 ? reinterpret_cast<double* const*>(sp->ctx->d_peers) : nullptr; p.c_off = 0;
  g->grid = p.nmt * p.ncb;
  return B2_OK;
}
static int gemm_run(b2_ctx* ctx, const GemmPlan& g, const double* B, double* C) {
  static bool attr_set[64] = {false};
  static const int dbg = getenv("B2_GEMM_DBG") ? atoi(getenv("B2_GEMM_DBG")) : 0;   // measurement only (tools/sweep.py): see gemm_pb_kernel
  if (!attr_set[ctx->device & 63]) {
    CK(cudaFuncSetAttribute(gemm_pb_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_SMEM_BYTES));
    CK(cudaFuncSetAttribute(gemm_pb_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_SMEM_BYTES));
    CK(cudaFuncSetAttribute(gemm_pb_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_SMEM_BYTES));
    attr_set[ctx->device & 63] = true;
  }
  GemmParams p = g.p;
  p.B = B; p.C = C;
  static const int gate = getenv("B2_GEMM_GATE") ? std::max(1, std::min(G_NSTAGE - 1, atoi(getenv("B2_GEMM_GATE")))) : 2;   // measurement knob
  p.gate = gate;
  if (ctx->nranks > 1) p.c_off = reinterpret_cast<const char*>(C) - static_cast<const char*>(ctx->peer_base[ctx->rank]);
  if (dbg == 1) B2_LAUNCH(gemm_pb_kernel<1>, g.grid, G_THREADS, (size_t)G_SMEM_BYTES, ctx->cur, p);
  else if (dbg == 2) B2_LAUNCH(gemm_pb_kernel<2>, g.grid, G_THREADS, (size_t)G_SMEM_BYTES, ctx->cur, p);
  else B2_LAUNCH(gemm_pb_kernel<0>, g.grid, G_THREADS, (size_t)G_SMEM_BYTES, ctx->cur, p);
  CK(cudaGetLastError());
  ctx->launches++;
  return ctx->nranks > 1 ? ctx_barrier(ctx) : B2_OK;   // the epilogue wrote into the peers' slabs
}

static void poisson_axis(const Base1& b, double c, Diags* lap, Diags* mass) {
  Diags a = b.mat_a(), bm = b.mat_b();
  *mass = a;
  *lap = Diags(b.m);
  for (int i = 0; i < b.m; i++) { lap->low[i] = bm.low[i] * c; lap->dia[i] = bm.dia[i] * c; lap->up1[i] = bm.up1[i] * c; lap->up2[i] = bm.up2[i] * c; }
}

// hholtz = true: Hholtz::new (src/solver/hholtz.rs:66-101) -- the same FdmaTensor with laplacian = -c * mat_b, alpha = 1 and
// no singularity shift: (I - c D2) vhat = A f
static int poisson_create(b2_space* sp, double c0, double c1, const double* lam_in, const double* fwd, const double* bwd, b2_solver** out, bool hholtz = false) {
  const double alpha = hholtz ? 1.0 : 0.0;
  if (hholtz) { c0 = -c0; c1 = -c1; }
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  if (!b1.composite) return fail(B2_ERR_UNSUPPORTED, "Poisson needs a composite Chebyshev axis 1");
  b2_solver* s = new b2_solver();
  s->sp = sp; s->type = 1;
  std::vector<double> lam;  // one eigenvalue per real row of the axis-0-transformed array
  int lanes;
  if (b0.composite) {
    if (!lam_in || !fwd || !bwd) { delete s; return fail(B2_ERR_ARG, "Poisson on a Chebyshev axis 0 needs lam/fwd/bwd (host LAPACK eig)"); }
    s->dense = true; s->m0 = b0.m;
    lam.assign(lam_in, lam_in + b0.m);
    lanes = b0.m;
  } else if (!b0.cheb) {
    // Fourier axis 0: lam = diag(laplacian) = -k^2 c0 (fdma_tensor.rs:118-121), singularity shift poisson.rs:84-86
    lanes = 2 * b0.m;
    lam.resize(lanes);
    for (int k = 0; k < b0.m; k++) {
      const double kk = (b0.c2c && 2 * k >= b0.n) ? k - b0.n : k;   // FourierC2c: modes in FFT order
      lam[2 * k] = lam[2 * k + 1] = -kk * kk * c0;
    }
    if (!hholtz && std::fabs(lam[0]) < 1e-10) for (auto& v : lam) v -= 1e-10;
  } else { delete s; return fail(B2_ERR_UNSUPPORTED, "Poisson axis-0 base"); }
  for (auto& v : lam) v += alpha;   // FdmaTensor::solve: (A1 + (lam_i + alpha) C1), src/solver/fdma_tensor.rs:277
  // per-lane LU of (lap1 + lam_i mass1), src/solver/poisson.rs:222-229, in scan layout [group][t][q][lane]
  Diags lap1, mass1;
  poisson_axis(b1, c1, &lap1, &mass1);
  const PassCfg& c = sp->cfg[0];
  const int nr = sp->ctx->nranks, lane0 = sp->ctx->rank * (c.groups / nr) * 4, lane1 = lane0 + (c.groups / nr) * 4;
  const size_t total = (size_t)(c.groups / nr) * c.C * 4 * c.TPL * 2;
  const int m1 = b1.m;
  auto build_lanes = [&](const std::vector<double>& lamv, DVecD* dfl, DVecD* did, DVecD* du1, DVecD* du2) -> int {
    std::vector<double> pfl(total, 0.0), pid(total, 0.0), pu1(total, 0.0), pu2(total, 0.0);
    Diags mat(m1);
    for (int lane = lane0; lane < std::min(lanes, lane1); lane++) {
      const double lm = lamv[lane];
      for (int i = 0; i < m1; i++) {
        mat.low[i] = lap1.low[i] + mass1.low[i] * lm;
        mat.dia[i] = lap1.dia[i] + mass1.dia[i] * lm;
        mat.up1[i] = lap1.up1[i] + mass1.up1[i] * lm;
        mat.up2[i] = lap1.up2[i] + mass1.up2[i] * lm;
      }
      LuVecs lu = sweep(mat);
      const int g = (lane - lane0) / 4, l = lane % 4;
      for (int i = 0; i < m1; i++) {
        const int pr = i / 2, q = pr / c.C, t = pr % c.C;
        const size_t k = ((((size_t)g * c.C + t) * c.TPL + q) * 4 + l) * 2 + (i & 1);
        pfl[k] = lu.fl[i]; pid[k] = lu.id[i]; pu1[k] = lu.u1[i]; pu2[k] = lu.u2[i];
      }
    }
    RET(dfl->upload(pfl)); RET(did->upload(pid)); RET(du1->upload(pu1)); RET(du2->upload(pu2));
    return B2_OK;
  };
  RET(build_lanes(lam, &s->pfl, &s->pid, &s->pu1, &s->pu2));
  if (s->dense) {
    // parity classes of the modes: row r of fwd (= mode r) touches even columns only, or odd columns only
    const int m0 = s->m0, ce = (m0 + 1) / 2, co = m0 / 2;
    std::vector<int> cls(m0, 0), perm;
    bool ok = true;
    for (int r = 0; r < m0 && ok; r++) {
      bool ev = false, od = false;
      for (int i = 0; i < m0; i++) {
        if (fwd[(size_t)r * m0 + i] != 0.0) ((i & 1) ? od : ev) = true;
        if (bwd[(size_t)i * m0 + r] != 0.0) ((i & 1) ? od : ev) = true;
      }
      if (ev && od) ok = false;
      cls[r] = od ? 1 : 0;
    }
    for (int k = 0; k < 2 && ok; k++) for (int r = 0; r < m0; r++) if (cls[r] == k) perm.push_back(r);
    int ne = 0; for (int r = 0; r < m0; r++) ne += (cls[r] == 0);
    if (ok && ne == ce && ce % 4 == 0) {   // the odd block starts on a tile row of the grouped array (gemm_f64.cuh)
      std::vector<double> fe((size_t)ce * ce), fo((size_t)co * co), be((size_t)ce * ce), bo((size_t)co * co), lam2(lam.size());
      for (int r = 0; r < ce; r++) for (int k = 0; k < ce; k++) { fe[(size_t)r * ce + k] = fwd[(size_t)perm[r] * m0 + 2 * k]; be[(size_t)k * ce + r] = bwd[(size_t)(2 * k) * m0 + perm[r]]; }
      for (int r = 0; r < co; r++) for (int k = 0; k < co; k++) { fo[(size_t)r * co + k] = fwd[(size_t)perm[ce + r] * m0 + 2 * k + 1]; bo[(size_t)k * co + r] = bwd[(size_t)(2 * k + 1) * m0 + perm[ce + r]]; }
      for (int r = 0; r < m0; r++) lam2[r] = lam[perm[r]];
      RET(build_lanes(lam2, &s->qfl, &s->qid, &s->qu1, &s->qu2));
      s->blocks = true; s->ce = ce; s->co = co;
      RET(gemm_plan_create(sp, &s->gf, fe.data(), ce, ce, fo.data(), co, co, true, false));   // forward: natural x rows -> modes grouped by class
      RET(gemm_plan_create(sp, &s->gb, be.data(), ce, ce, bo.data(), co, co, false, true));   // backward: the reverse
      s->own_gemm = true;
    }
  }
  if (s->dense && !s->own_gemm) {   // a decomposition without the parity structure: full products, natural mode order
    RET(gemm_plan_create(sp, &s->gf, fwd, s->m0, s->m0, nullptr, 0, 0, false, false));
    RET(gemm_plan_create(sp, &s->gb, bwd, s->m0, s->m0, nullptr, 0, 0, false, false));
    s->own_gemm = true; s->blocks = false;
  }
  *out = s;
  return B2_OK;
}

static int gemm_mark(b2_ctx* ctx) {
  if (!ctx->profile) return B2_OK;
  cudaEvent_t e;
  CK(cudaEventCreate(&e));
  CK(cudaEventRecord(e, ctx->stream));
  ctx->gemm_events.push_back(e);
  return B2_OK;
}

// Eigen-transform core of the confined Poisson solve (src/solver/poisson.rs:213-235) on the tiled arrays, shared by the
// fused step and Poisson::solve.  src: right-hand side in the y-lane orientation (rows = x index), already multiplied by the
// x-axis preconditioner; matvec_y: apply the y-axis one here.  gx: [all x rows][local y columns] scratch (the GEMM operand:
// the contraction runs over x; with several GPUs the lane passes scatter their column blocks to the owners -- ST_COLSPLIT --
// and the GEMM epilogue scatters its row blocks back, so both exchanges ride on a kernel that runs anyway), y1: slab scratch.
static int poisson_core(b2_solver* s, b2_space* rs, const double* src, bool matvec_y, double* gx, double* y1, double* out, bool zero00) {
  b2_ctx* ctx = rs->ctx;
  const Base1& b1 = s->sp->b[1];
  Prog y; y.load(src, matvec_y ? b1.rows_ortho : b1.m);
  if (matvec_y) y.matvec(b1);
  y.store(gx, b1.m, ST_COLSPLIT);
  RET(run_pass(rs, 0, y));
  RET(gemm_mark(ctx));
  RET(gemm_run(ctx, s->gf, gx, y1));   // forward: x index -> eigenmodes (parity blocks: modes grouped by class, the order of q*)
  RET(gemm_mark(ctx));
  Prog y2; y2.load(y1, b1.m);
  if (s->blocks) y2.fdma(b1.m, s->qfl.d, s->qid.d, s->qu1.d, s->qu2.d, FD_PERLANE);
  else y2.fdma(b1.m, s->pfl.d, s->pid.d, s->pu1.d, s->pu2.d, FD_PERLANE);
  y2.store(gx, b1.m, ST_COLSPLIT);
  RET(run_pass(rs, 0, y2));
  RET(gemm_mark(ctx));
  RET(gemm_run(ctx, s->gb, gx, out));  // backward: eigenmodes -> x index (natural order)
  RET(gemm_mark(ctx));
  if (zero00 && ctx->rank == 0) CK(cudaMemsetAsync(out, 0, sizeof(double), ctx->cur));   // element (0, 0) of tile (0, 0) (navier_eq.rs:161)
  return B2_OK;
}

// Poisson::solve_par, src/solver/poisson.rs:195-236
static int poisson_solve(b2_solver* s, const double* in, double* out, bool zero00) {
  b2_space* sp = s->sp;
  b2_ctx* ctx = sp->ctx;
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  const int P0 = sp->P[0], P1 = sp->P[1];
  if (s->dense) {
    // matvec along y and x (two transposing passes: back in the y-lane orientation, rows = x index), then the core
    Prog y; y.load(in, b1.rows_ortho); int l = y.matvec(b1); y.store(sp->tmp[0], l, ST_TRANS);
    RET(run_pass(sp, 0, y));
    Prog x; x.load(sp->tmp[0], b0.rows_ortho); l = x.matvec(b0); x.store(sp->tmp[1], l, ST_TRANS);
    RET(run_pass(sp, 1, x));
    return poisson_core(s, sp, sp->tmp[1], false, sp->tmp[0], sp->tmp[2], out, zero00);
  }
  Prog y; y.load(in, b1.rows_ortho); int l = y.matvec(b1);
  y.fdma(b1.m, s->pfl.d, s->pid.d, s->pu1.d, s->pu2.d, FD_PERLANE);
  y.store(sp->tmp[0], l, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_spec);
  if (zero00) { x.zeroelem(0, 0); x.zeroelem(0, 1); }
  x.store(out, b0.rows_spec, ST_TRANS);
  return run_pass(sp, 1, x);
}

// one axis of HholtzAdi: precondition (MatVecFdma) + banded / diagonal solve
static void emit_hh_axis(Prog& p, const b2_solver* s, int ax) {
  const Base1& b = s->sp->b[ax];
  p.matvec(b);
  if (b.composite) p.fdma(b.m, s->fl[ax].d, s->id[ax].d, s->u1[ax].d, s->u2[ax].d, 0);
  else if (b.cdn) p.pdma(b.m, s->pd[ax].d, s->pd_L[ax]);   // hholtz_adi.rs:64
  else p.scalevec(b.rows_spec, s->sd[ax].d, 1);
}

// ------------------------------------------------------------------------------------------------
// Navier2D
// ------------------------------------------------------------------------------------------------
struct b2_navier {
  b2_ctx* ctx = nullptr;
  int nx = 0, ny = 0, periodic = 0;
  double ra = 0, pr = 0, dt = 0, nu = 0, ka = 0, time = 0, scale[2] = {1, 1};
  // spaces: [0] velocity (cd x cd), [1] temp (cn x cd), [2] ortho "field"/pres (ch x ch), [3] pseu (cn x cn)
  b2_space* sp_vel = nullptr; b2_space* sp_temp = nullptr; b2_space* sp_ortho = nullptr; b2_space* sp_pseu = nullptr;
  b2_field *temp = nullptr, *velx = nullptr, *vely = nullptr, *pres = nullptr, *pseu = nullptr, *tempbc = nullptr;
  b2_solver* hh[3] = {nullptr, nullptr, nullptr};
  b2_solver* pois = nullptr;
  // work arrays (ortho-sized, tiled)
  double *that = nullptr, *tbc_ortho = nullptr, *tbc_diff = nullptr, *rhs = nullptr, *g1 = nullptr, *g2 = nullptr, *conv = nullptr, *div = nullptr, *ux = nullptr, *uy = nullptr;
  double* d_scalar = nullptr;
  // fused schedule: intermediates (suffix T = stored in the transposed orientation)
  double *Pf[3] = {nullptr}, *Qf[3] = {nullptr}, *V1[3] = {nullptr}, *Cx[3] = {nullptr}, *Zf[3] = {nullptr}, *Of[3] = {nullptr};
  double *VTv = nullptr, *uxT = nullptr, *uyT = nullptr, *cv[3] = {nullptr}, *PH = nullptr, *PHy = nullptr, *F1 = nullptr, *F2 = nullptr, *R0 = nullptr;
  double *G0 = nullptr, *G1 = nullptr, *U1 = nullptr, *U2 = nullptr, *U3 = nullptr;
  double *GxT = nullptr, *GyT = nullptr, *KbT = nullptr, *KTT = nullptr;   // constants of the step
  int fused = 1;
  int branches = 1;   // run independent passes of the fused step as parallel graph branches
  long long launches_per_step = 0;
#ifndef B2_EMU
  cudaGraphExec_t graph = nullptr;
#endif
  int use_graph = 1, warm_steps = 0;
};

#ifndef B2_EMU
static int b2_heap_malloc(void** p, size_t bytes) { CK(cudaMalloc(p, bytes)); return B2_OK; }
#endif

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

const char* b2_last_error(void) { return g_err.c_str(); }
int b2_version(void) { return 1; }

int b2_ctx_create(int device, int rank, int nranks, size_t heap_bytes, b2_ctx** out) {
  if (!out || nranks < 1 || nranks > B2_MAXPEERS || rank < 0 || rank >= nranks) return fail(B2_ERR_ARG, "b2_ctx_create: bad arguments");
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (ndev == 0) return fail(B2_ERR_CUDA, "no CUDA device: b200pde has no CPU fallback");
  CK(cudaSetDevice(device));
  b2_ctx* c = new b2_ctx();
  c->device = device; c->rank = rank; c->nranks = nranks;
  CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->cur = c->stream;
  for (int i = 0; i < 2; i++) CK(cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking));
  for (int i = 0; i < 16; i++) CK(cudaEventCreateWithFlags(&c->evp[i], cudaEventDisableTiming));
  if (nranks > 1) {
    if (heap_bytes < (1u << 20)) return fail(B2_ERR_ARG, "nranks > 1 needs a symmetric heap (heap_bytes)");
    c->heap_bytes = heap_bytes;
    RET(b2_heap_malloc(reinterpret_cast<void**>(&c->heap), heap_bytes));
    CK(cudaMemset(c->heap, 0, heap_bytes));
    c->heap_used = B2_HEAP_RESERVED;
    c->peer_base[rank] = c->heap;
  }
  *out = c;
  return B2_OK;
}
int b2_ctx_destroy(b2_ctx* c) {
  if (!c) return B2_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (auto& st : c->side) if (st) cudaStreamSynchronize(st);
  for (auto e : c->gemm_events) cudaEventDestroy(e);
  for (auto& e : c->evp) if (e) cudaEventDestroy(e);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  for (auto& st : c->side) if (st) cudaStreamDestroy(st);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->stage) cudaFree(c->stage);
  if (c->d_prof) cudaFree(c->d_prof);
  if (c->d_differs) cudaFree(c->d_differs);
  if (c->d_acc) cudaFree(c->d_acc);
  if (c->d_peers) cudaFree(c->d_peers);
#ifndef B2_EMU
  for (int r = 0; r < c->nranks; r++) if (r != c->rank && c->peer_base[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
  if (c->heap) cudaFree(c->heap);
#endif
  delete c;
  return B2_OK;
}
int b2_ctx_sync(b2_ctx* c) { CK(cudaStreamSynchronize(c->stream)); return B2_OK; }
int b2_ctx_timer_start(b2_ctx* c) {
  if (!c->ev0) { CK(cudaEventCreate(&c->ev0)); CK(cudaEventCreate(&c->ev1)); }
  CK(cudaStreamSynchronize(c->stream));
  CK(cudaEventRecord(c->ev0, c->stream));
  return B2_OK;
}
int b2_ctx_timer_stop(b2_ctx* c, double* ms) {
  CK(cudaEventRecord(c->ev1, c->stream));
  CK(cudaEventSynchronize(c->ev1));
  float f = 0;
  CK(cudaEventElapsedTime(&f, c->ev0, c->ev1));
  *ms = f;
  return B2_OK;
}
int b2_ctx_launch_count(const b2_ctx* c, long long* n) { *n = c->launches; return B2_OK; }
// per-op cycle counters of the lane kernel (thread 0 of every CTA): out[code] = cycles, out[32+code] = count
int b2_ctx_opprof(b2_ctx* c, int on, unsigned long long* out64) {
  CK(cudaStreamSynchronize(c->stream));
  if (c->d_prof && out64) CK(cudaMemcpy(out64, c->d_prof, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if (on && !c->d_prof) CK(cudaMalloc(&c->d_prof, 64 * sizeof(unsigned long long)));
  if (c->d_prof) CK(cudaMemset(c->d_prof, 0, 64 * sizeof(unsigned long long)));
  if (!on && c->d_prof) { CK(cudaFree(c->d_prof)); c->d_prof = nullptr; }
  return B2_OK;
}
int b2_ctx_profile(b2_ctx* c, int on, double* gemm_ms) {
  CK(cudaStreamSynchronize(c->stream));
  double tot = 0;
  for (size_t i = 0; i + 1 < c->gemm_events.size(); i += 2) {
    float f = 0;
    CK(cudaEventElapsedTime(&f, c->gemm_events[i], c->gemm_events[i + 1]));
    tot += f;
  }
  for (auto e : c->gemm_events) cudaEventDestroy(e);
  c->gemm_events.clear();
  if (gemm_ms) *gemm_ms = tot;
  c->profile = on != 0;
  return B2_OK;
}
// Memory-pipeline probe (tools/copyprobe.py): `reps` passes of { load a slab, optional DCT, store it (transposed or not) }
// over a full array of the space, timed with CUDA events.  mode bit 0: transposing store; bit 1: add a backward DCT;
// bit 2: scale by 2 on load (forces the ring path); bit 3: scale on store (forces the staged path).
int b2_debug_copy(b2_space* sp, int mode, int reps, double* ms) {
  double *a = nullptr, *b = nullptr;
  RET(alloc_zero(sp, &a)); RET(alloc_zero(sp, &b));
  b2_ctx* ctx = sp->ctx;
  const Base1& by = sp->b[1];
  auto pass = [&]() -> int {
    Prog y; y.load(a, by.rows_ortho, (mode & 4) ? 2.0 : 1.0);
    if (mode & 2) y.dct(by, 1);
    y.store(b, by.rows_ortho, (mode & 1) ? ST_TRANS : 0, (mode & 8) ? 2.0 : 1.0);
    return run_pass(sp, 0, y);
  };
  RET(pass());
  if (!ctx->ev0) { CK(cudaEventCreate(&ctx->ev0)); CK(cudaEventCreate(&ctx->ev1)); }
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  for (int r = 0; r < reps; r++) RET(pass());
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->ev1));
  float t = 0; CK(cudaEventElapsedTime(&t, ctx->ev0, ctx->ev1));
  *ms = t / reps;
  ctx_free(ctx, a); ctx_free(ctx, b);
  return B2_OK;
}
int b2_ctx_nranks(const b2_ctx* c) { return c->nranks; }
int b2_ctx_heap_handle(b2_ctx* c, void* handle64) {
  if (c->nranks == 1) return fail(B2_ERR_ARG, "single-rank context has no heap");
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, c->heap));
  static_assert(sizeof(h) == 64, "IPC handle size");
  memcpy(handle64, &h, 64);
  return B2_OK;
}
int b2_ctx_attach_peers(b2_ctx* c, const void* handles) {
  if (c->nranks == 1) return B2_OK;
  CK(cudaSetDevice(c->device));
  for (int r = 0; r < c->nranks; r++) {
    if (r == c->rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(handles) + 64 * r, 64);
    CK(cudaIpcOpenMemHandle(&c->peer_base[r], h, cudaIpcMemLazyEnablePeerAccess));
  }
  CK(cudaMalloc(&c->d_peers, B2_MAXPEERS * sizeof(double*)));
  CK(cudaMemcpy(c->d_peers, c->peer_base, B2_MAXPEERS * sizeof(double*), cudaMemcpyHostToDevice));
  c->attached = true;
  return B2_OK;
}
int b2_ctx_barrier(b2_ctx* c) { return ctx_barrier(c); }

int b2_space2_create(b2_ctx* ctx, int kind0, int n0, int kind1, int n1, b2_space** out) {
  if (!ctx || !out) return fail(B2_ERR_ARG, "b2_space2_create: null");
  CK(cudaSetDevice(ctx->device));
  b2_space* sp = new b2_space();
  sp->ctx = ctx;
  int r = sp->b[0].init_host(kind0, n0);
  if (r == B2_OK) r = sp->b[1].init_host(kind1, n1);
  if (r == B2_OK && !sp->b[1].cheb) r = fail(B2_ERR_UNSUPPORTED, "axis 1 must be a Chebyshev base (Navier2D spaces)");
  if (r != B2_OK) { delete sp; return r; }
  // padded so that the 4-row lane groups split evenly over the ranks (slab decomposition)
  for (int ax = 0; ax < 2; ax++) sp->P[ax] = roundup(std::max(sp->b[ax].rows_phys, sp->b[ax].rows_ortho), 4 * ctx->nranks);
  r = make_cfg(sp->b[1], sp->P[1], sp->P[0], &sp->cfg[0], ctx->nranks);
  if (r == B2_OK) r = make_cfg(sp->b[0], sp->P[0], sp->P[1], &sp->cfg[1], ctx->nranks);
  if (r == B2_OK) r = sp->b[1].init(sp->cfg[0].C, sp->cfg[0].TPL);   // cfg[0]: lanes along axis 1
  if (r == B2_OK) r = sp->b[0].init(sp->cfg[1].C, sp->cfg[1].TPL);
  if (r != B2_OK) { delete sp; return r; }
  sp->transforms_ok = (sp->b[0].d_tw.d || sp->b[0].dense_tr) && (sp->b[1].d_tw.d || sp->b[1].dense_tr);
  for (int i = 0; i < 3; i++) RET(alloc_zero(sp, &sp->tmp[i]));
  *out = sp;
  return B2_OK;
}
int b2_space_destroy(b2_space* sp) {
  if (!sp) return B2_OK;
  for (auto& t : sp->tmp) ctx_free(sp->ctx, t);
  sp->b[0].release(); sp->b[1].release();
  delete sp;
  return B2_OK;
}
int b2_space_shape(const b2_space* sp, int shape_kind, int* rows, int* cols, int* is_complex) {
  int r, c;
  RET(shape_of(sp, shape_kind, &r, &c));
  bool cx = shape_complex(sp, shape_kind);
  if (rows) *rows = cx ? r / 2 : r;
  if (cols) *cols = c;
  if (is_complex) *is_complex = cx;
  return B2_OK;
}
int b2_space_coords(const b2_space* sp, int axis, double* x) {
  if (axis < 0 || axis > 1) return fail(B2_ERR_ARG, "axis");
  const Base1& b = sp->b[axis];
  const double PI = 3.14159265358979323846;
  for (int j = 0; j < b.n; j++) x[j] = b.cheb ? -std::cos(PI * j / (b.n - 1)) : 2.0 * PI * j / b.n;
  return B2_OK;
}
int b2_space_lane_layout(const b2_space* sp, int orient, int* out8) {
  if (!sp || !out8) return fail(B2_ERR_ARG, "b2_space_lane_layout: null");
  if (orient < 0 || orient > 1) return fail(B2_ERR_ARG, "orient");
  const PassCfg& c = sp->cfg[orient];
  const int v[8] = {c.E, c.LN, c.TPL, c.fast ? 1 : 0, c.CHW, c.nsc, c.NT, (int)c.smem};
  for (int i = 0; i < 8; i++) out8[i] = v[i];
  return B2_OK;
}

int b2_array_create(b2_space* sp, int shape_kind, b2_array** out) {
  int r, c;
  RET(shape_of(sp, shape_kind, &r, &c));
  CK(cudaSetDevice(sp->ctx->device));
  b2_array* a = new b2_array{sp, nullptr, shape_kind};
  RET(alloc_zero(sp, &a->d));
  *out = a;
  return B2_OK;
}
int b2_array_destroy(b2_array* a) { if (a) { ctx_free(a->sp->ctx, a->d); delete a; } return B2_OK; }

// rows of the logical (real-row) array that live on this rank: [row0, row0 + count)
static void local_rows(const b2_space* sp, int rows_total, int* row0, int* count) {
  const int per = sp->P[0] / sp->ctx->nranks;
  *row0 = sp->ctx->rank * per;
  *count = std::max(0, std::min(per, rows_total - *row0));
}

static int array_copy(const b2_array* a, void* buf, size_t bytes, int to_device) {
  b2_space* sp = a->sp;
  int r, c;
  RET(shape_of(sp, a->shape_kind, &r, &c));
  { int row0; local_rows(sp, r, &row0, &r); }   // multi-rank: the host buffer is this rank's slab of rows
  if (r == 0) return bytes == 0 ? B2_OK : fail(B2_ERR_SHAPE, "this rank owns no rows of the array");
  const size_t need = (size_t)r * c * sizeof(double);
  if (bytes != need) return fail(B2_ERR_SHAPE, "host buffer has " + std::to_string(bytes) + " bytes, array needs " + std::to_string(need));
  CK(cudaSetDevice(sp->ctx->device));
  b2_ctx* ctx = sp->ctx;
  if (ctx->stage_bytes < need) {
    if (ctx->stage) CK(cudaFree(ctx->stage));
    CK(cudaMalloc(&ctx->stage, need));
    ctx->stage_bytes = need;
  }
  double* stage = ctx->stage;
  cudaStream_t st = sp->ctx->stream;
  const int cx = shape_complex(sp, a->shape_kind);
  const size_t total = (size_t)r * c;
  const int grid = (int)((total + 255) / 256);
  if (to_device) {
    CK(cudaMemcpyAsync(stage, buf, need, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(a->d, 0, sp->elems() * sizeof(double), st));
    B2_LAUNCH(k_host_layout, grid, 256, 0, st, a->d, stage, r, c, sp->P[1] / 4, cx, 1);
  } else {
    B2_LAUNCH(k_host_layout, grid, 256, 0, st, a->d, stage, r, c, sp->P[1] / 4, cx, 0);
    CK(cudaMemcpyAsync(buf, stage, need, cudaMemcpyDeviceToHost, st));
  }
  CK(cudaGetLastError());
  ctx->launches++;
  CK(cudaStreamSynchronize(st));
  return B2_OK;
}
int b2_array_local_rows(const b2_array* a, int* row_start, int* row_count) {
  int r, c, row0, cnt;
  RET(shape_of(a->sp, a->shape_kind, &r, &c));
  local_rows(a->sp, r, &row0, &cnt);
  const int div = shape_complex(a->sp, a->shape_kind) ? 2 : 1;
  if (row_start) *row_start = row0 / div;
  if (row_count) *row_count = cnt / div;
  return B2_OK;
}
int b2_array_set_host(b2_array* a, const void* buf, size_t bytes) { return array_copy(a, const_cast<void*>(buf), bytes, 1); }
int b2_array_get_host(const b2_array* a, void* buf, size_t bytes) { return array_copy(a, buf, bytes, 0); }
int b2_array_axpy(b2_array* y, double alpha, const b2_array* x) {
  int yr, yc, xr, xc;
  RET(shape_of(y->sp, y->shape_kind, &yr, &yc)); RET(shape_of(x->sp, x->shape_kind, &xr, &xc));
  if (y->sp->elems() != x->sp->elems() || yr != xr || yc != xc || shape_complex(y->sp, y->shape_kind) != shape_complex(x->sp, x->shape_kind))
    return fail(B2_ERR_SHAPE, "axpy: different shapes");
  const size_t n = y->sp->elems();
  B2_LAUNCH(k_axpby, ew_grid(n), 256, 0, y->sp->ctx->stream, n, y->d, alpha, x->d, 1.0);
  CK(cudaGetLastError());
  y->sp->ctx->launches++;
  return B2_OK;
}
int b2_field_array(b2_field* f, int which, b2_array** out) {
  if (!f || !out) return fail(B2_ERR_ARG, "b2_field_array: null argument");
  if (which < 0 || which > 1) return fail(B2_ERR_ARG, "which: 0 = v, 1 = vhat");
  *out = which == 0 ? f->v : f->vhat;   // borrowed: owned by the field
  return B2_OK;
}
int b2_array_copy(b2_array* dst, const b2_array* src) {
  if (!dst || !src) return fail(B2_ERR_ARG, "b2_array_copy: null array");
  if (dst->sp->elems() != src->sp->elems() || dst->sp->P[0] != src->sp->P[0] || dst->sp->P[1] != src->sp->P[1]) return fail(B2_ERR_SHAPE, "copy: different padded shapes");
  CK(cudaMemcpyAsync(dst->d, src->d, dst->sp->elems() * sizeof(double), cudaMemcpyDeviceToDevice, dst->sp->ctx->stream));
  return B2_OK;
}
int b2_array_combine(b2_array* dst, const b2_array* a, const b2_array* b, int op, double alpha) {
  if (!dst || !a || !b) return fail(B2_ERR_ARG, "b2_array_combine: null array");
  if (op < 0 || op > 2) return fail(B2_ERR_ARG, "combine op");
  const size_t n = dst->sp->elems();
  if (a->sp->elems() != n || b->sp->elems() != n || a->sp->P[1] != dst->sp->P[1] || b->sp->P[1] != dst->sp->P[1]) return fail(B2_ERR_SHAPE, "combine: different padded shapes");
  B2_LAUNCH(k_combine, ew_grid(n), 256, 0, dst->sp->ctx->stream, n, dst->d, a->d, b->d, op, alpha);
  CK(cudaGetLastError());
  dst->sp->ctx->launches++;
  return B2_OK;
}
// scratch device buffer of one call: released on every return path
struct ScratchBuf {
  double* p = nullptr;
  ~ScratchBuf() { if (p) cudaFree(p); }
};
int b2_array_weighted_sum(const b2_array* a, const double* w0_local, const double* w1, int mode, double* out) {
  if (!a || !w0_local || !w1 || !out || mode < 0 || mode > 2) return fail(B2_ERR_ARG, "b2_array_weighted_sum: null argument or mode not 0 / 1 / 2");
  b2_space* sp = a->sp;
  if (shape_complex(sp, a->shape_kind)) return fail(B2_ERR_UNSUPPORTED, "weighted sums are defined on real (physical) arrays");
  int rows, cols, row0, cnt;
  RET(shape_of(sp, a->shape_kind, &rows, &cols));
  local_rows(sp, rows, &row0, &cnt);
  const int nout = mode == 1 ? cols : mode == 2 ? cnt : 1;
  ScratchBuf buf;
  CK(cudaMalloc(&buf.p, (size_t)(cnt + cols + nout + 1) * sizeof(double)));
  double* dw0 = buf.p; double* dw1 = buf.p + cnt; double* dout = dw1 + cols;
  if (cnt) CK(cudaMemcpyAsync(dw0, w0_local, (size_t)cnt * sizeof(double), cudaMemcpyHostToDevice, sp->ctx->stream));
  CK(cudaMemcpyAsync(dw1, w1, (size_t)cols * sizeof(double), cudaMemcpyHostToDevice, sp->ctx->stream));
  CK(cudaMemsetAsync(dout, 0, (size_t)nout * sizeof(double), sp->ctx->stream));
  if (mode == 2) {
    if (cnt) B2_LAUNCH(k_weighted_rowsum, (cnt + 127) / 128, 128, 0, sp->ctx->stream, a->d, cnt, cols, sp->P[1] / 4, dw1, dout);
  } else {
    B2_LAUNCH(k_weighted_sum, (cols + 127) / 128, 128, 0, sp->ctx->stream, a->d, cnt, cols, sp->P[1] / 4, dw0, dw1, mode, dout);
  }
  CK(cudaGetLastError());
  sp->ctx->launches++;
  if (nout) CK(cudaMemcpyAsync(out, dout, (size_t)nout * sizeof(double), cudaMemcpyDeviceToHost, sp->ctx->stream));
  CK(cudaStreamSynchronize(sp->ctx->stream));
  return B2_OK;
}
static int norm2_dev(b2_space* sp, const double* d, double* out, bool global) {
  if (!sp->ctx->d_acc) CK(cudaMalloc(&sp->ctx->d_acc, sizeof(double)));   // once per context, released by b2_ctx_destroy
  double* acc = sp->ctx->d_acc;
  CK(cudaMemsetAsync(acc, 0, sizeof(double), sp->ctx->stream));
  const size_t n = sp->elems();
  B2_LAUNCH(k_sumsq, ew_grid(n), 256, 0, sp->ctx->stream, n, d, acc);
  CK(cudaGetLastError());
  if (global && sp->ctx->nranks > 1) {
    if (!sp->ctx->attached) return fail(B2_ERR_ARG, "b2_ctx_attach_peers has not been called");
    B2_LAUNCH(k_allreduce, 1, 32, 0, sp->ctx->stream, reinterpret_cast<unsigned long long* const*>(sp->ctx->d_peers), sp->ctx->rank, sp->ctx->nranks, acc, acc);
    CK(cudaGetLastError());
  }
  double h = 0;
  CK(cudaMemcpyAsync(&h, acc, sizeof(double), cudaMemcpyDeviceToHost, sp->ctx->stream));
  CK(cudaStreamSynchronize(sp->ctx->stream));
  *out = h;
  return B2_OK;
}
// sum |a|^2 over this rank's slab; with one rank b2_array_norm2 = sqrt of it (functions.rs:24-35)
int b2_array_sumsq_local(const b2_array* a, double* out) { return norm2_dev(a->sp, a->d, out, false); }
int b2_array_norm2(const b2_array* a, double* out) {
  RET(norm2_dev(a->sp, a->d, out, true));   // all ranks: the norm of the global array (collective call)
  *out = std::sqrt(*out);
  return B2_OK;
}

int b2_field_create(b2_space* sp, b2_field** out) {
  b2_field* f = new b2_field{sp, nullptr, nullptr};
  RET(b2_array_create(sp, B2_SHAPE_PHYSICAL, &f->v));
  RET(b2_array_create(sp, B2_SHAPE_SPECTRAL, &f->vhat));
  *out = f;
  return B2_OK;
}
int b2_field_destroy(b2_field* f) { if (f) { b2_array_destroy(f->v); b2_array_destroy(f->vhat); delete f; } return B2_OK; }
int b2_field_set_v_host(b2_field* f, const void* buf, size_t bytes) { return b2_array_set_host(f->v, buf, bytes); }
int b2_field_get_v_host(const b2_field* f, void* buf, size_t bytes) { return b2_array_get_host(f->v, buf, bytes); }
int b2_field_set_vhat_host(b2_field* f, const void* buf, size_t bytes) { return b2_array_set_host(f->vhat, buf, bytes); }
int b2_field_get_vhat_host(const b2_field* f, void* buf, size_t bytes) { return b2_array_get_host(f->vhat, buf, bytes); }
int b2_field_local_rows(const b2_field* f, int shape_kind, int* row_start, int* row_count) {
  return b2_array_local_rows(shape_kind == B2_SHAPE_PHYSICAL ? f->v : f->vhat, row_start, row_count);
}
int b2_forward(b2_field* f) { return op_forward(f->sp, f->v->d, f->vhat->d); }
int b2_backward(b2_field* f) { return op_backward(f->sp, f->vhat->d, f->v->d); }
static int need_kind(const b2_array* a, int kind, const char* what) {
  if (a->shape_kind != kind) return fail(B2_ERR_SHAPE, std::string(what) + ": array has the wrong shape kind");
  return B2_OK;
}
int b2_to_ortho(const b2_field* f, b2_array* out) {
  RET(need_kind(out, B2_SHAPE_ORTHO, "to_ortho"));
  return op_to_ortho(f->sp, f->vhat->d, out->d);
}
int b2_from_ortho(b2_field* f, const b2_array* in) {
  RET(need_kind(in, B2_SHAPE_ORTHO, "from_ortho"));
  return op_from_ortho(f->sp, in->d, f->vhat->d);
}
int b2_gradient(const b2_field* f, int d0, int d1, const double* scale, b2_array* out) {
  RET(need_kind(out, B2_SHAPE_ORTHO, "gradient"));
  if (d0 < 0 || d1 < 0 || d0 > 3 || d1 > 3) return fail(B2_ERR_ARG, "gradient: derivative order");
  return op_gradient(f->sp, f->vhat->d, d0, d1, scale, out->d);
}

// dealias(&mut field), src/navier_stokes/functions.rs:72-82: vhat[n_x.., ..] = 0 and vhat[.., n_y..] = 0 with
// n = shape * 2 / 3 in integer arithmetic on the spectral shape (modes, not real rows)
int b2_field_dealias(b2_field* f) {
  b2_space* sp = f->sp;
  const Base1& b0 = sp->b[0]; const Base1& b1 = sp->b[1];
  if (b0.c2c) return fail(B2_ERR_UNSUPPORTED, "dealias: the 2/3 tail rule of functions.rs:72-82 is written for r2c / Chebyshev mode order");
  const int cut0 = (b0.m * 2 / 3) * (b0.cheb ? 1 : 2), cut1 = b1.m * 2 / 3;
  Prog y; y.load(f->vhat->d, b1.rows_spec); y.zerotail(cut1); y.store(sp->tmp[0], b1.rows_spec, ST_TRANS);
  RET(run_pass(sp, 0, y));
  Prog x; x.load(sp->tmp[0], b0.rows_spec); x.zerotail(cut0); x.store(f->vhat->d, b0.rows_spec, ST_TRANS);
  return run_pass(sp, 1, x);
}

int b2_hholtz_adi_create(const b2_field* f, double c0, double c1, b2_solver** out) { return hholtz_create(f->sp, c0, c1, out); }
int b2_poisson_create(const b2_field* f, double c0, double c1, const double* lam, const double* fwd, const double* bwd, b2_solver** out) {
  return poisson_create(f->sp, c0, c1, lam, fwd, bwd, out);
}
int b2_hholtz_create(const b2_field* f, double c0, double c1, const double* lam, const double* fwd, const double* bwd, b2_solver** out) {
  return poisson_create(f->sp, c0, c1, lam, fwd, bwd, out, true);
}
int b2_solver_destroy(b2_solver* s) {
  if (!s) return B2_OK;
  for (int ax = 0; ax < 2; ax++) { s->fl[ax].release(); s->id[ax].release(); s->u1[ax].release(); s->u2[ax].release(); s->sd[ax].release(); s->pd[ax].release(); }
  s->pfl.release(); s->pid.release(); s->pu1.release(); s->pu2.release();
  s->qfl.release(); s->qid.release(); s->qu1.release(); s->qu2.release();
  for (GemmPlan* g : {&s->gf, &s->gb}) { g->A[0].release(); g->A[1].release(); }
  delete s;
  return B2_OK;
}
int b2_solve(b2_solver* s, const b2_array* in, b2_array* out) {
  // shape checks replace the reference's assert!/panic! (src/solver/fdma_tensor.rs:256-263)
  RET(need_kind(in, B2_SHAPE_ORTHO, "solve input"));
  RET(need_kind(out, B2_SHAPE_SPECTRAL, "solve output"));
  if (in->sp != s->sp || out->sp != s->sp) return fail(B2_ERR_SHAPE, "solve: arrays belong to a different space");
  return s->type == 0 ? hholtz_solve(s, in->d, out->d) : poisson_solve(s, in->d, out->d, false);
}

static void dense_from_diags(const Diags& d, double* out) {
  const int m = d.m;
  std::fill(out, out + (size_t)m * m, 0.0);
  for (int i = 0; i < m; i++) {
    out[(size_t)i * m + i] = d.dia[i];
    if (i + 2 < m) { out[(size_t)(i + 2) * m + i] = d.low[i]; out[(size_t)i * m + i + 2] = d.up1[i]; }
    if (i + 4 < m) out[(size_t)i * m + i + 4] = d.up2[i];
  }
}
int b2_host_poisson_matrices(int kind0, int n0, double c0, double* a0, double* cmat0) {
  Base1 b0;
  RET(b0.init_host(kind0, n0));
  if (!b0.composite) return fail(B2_ERR_ARG, "axis 0 is not a composite Chebyshev base");
  Diags lap, mass;
  poisson_axis(b0, c0, &lap, &mass);
  dense_from_diags(lap, a0);
  dense_from_diags(mass, cmat0);
  return B2_OK;
}
int b2_poisson_axis0_matrices(const b2_field* f, double c0, double* a0, double* cmat0) {
  return b2_host_poisson_matrices(f->sp->b[0].kind, f->sp->b[0].n, c0, a0, cmat0);
}

// ---------------------------------------------------------------------------------------------
// Navier2D
// ---------------------------------------------------------------------------------------------
static int nav_alloc(b2_space* sp, double** p) { return alloc_zero(sp, p); }

int b2_navier2d_create(b2_ctx* ctx, int nx, int ny, double ra, double pr, double dt, double aspect, const char* bc,
                       int periodic, const double* lam, const double* fwd, const double* bwd, b2_navier** out) {
  if (!bc || (std::string(bc) != "rbc" && std::string(bc) != "hc")) return fail(B2_ERR_ARG, "Boundary condition type not recognized (\"rbc\" or \"hc\", navier.rs:238-252)");
  const bool hc = std::string(bc) == "hc";
  b2_navier* nv = new b2_navier();
  nv->ctx = ctx; nv->nx = nx; nv->ny = ny; nv->periodic = periodic;
  nv->ra = ra; nv->pr = pr; nv->dt = dt; nv->scale[0] = aspect; nv->scale[1] = 1.0;
  const double height = nv->scale[1] * 2.0;  // functions.rs:12-21
  nv->nu = std::sqrt(pr / (ra / std::pow(height, 3.0)));
  nv->ka = std::sqrt(1.0 / ((ra / std::pow(height, 3.0)) * pr));
  const int kx_vel = periodic ? B2_FOURIER_R2C : B2_CHEB_DIRICHLET;
  const int kx_temp = periodic ? B2_FOURIER_R2C : B2_CHEB_NEUMANN;
  const int kx_ortho = periodic ? B2_FOURIER_R2C : B2_CHEBYSHEV;
  const int kx_pseu = periodic ? B2_FOURIER_R2C : B2_CHEB_NEUMANN;
  RET(b2_space2_create(ctx, kx_vel, nx, B2_CHEB_DIRICHLET, ny, &nv->sp_vel));     // navier.rs:235-236 / 356-357
  RET(b2_space2_create(ctx, kx_temp, nx, hc ? B2_CHEB_DIRICHLET_NEUMANN : B2_CHEB_DIRICHLET, ny, &nv->sp_temp));   // :240,246-247 / :361,367
  RET(b2_space2_create(ctx, kx_ortho, nx, B2_CHEBYSHEV, ny, &nv->sp_ortho));      // :254,256 / :375,377
  RET(b2_space2_create(ctx, kx_pseu, nx, B2_CHEB_NEUMANN, ny, &nv->sp_pseu));     // :255 / :376
  RET(b2_field_create(nv->sp_vel, &nv->velx)); RET(b2_field_create(nv->sp_vel, &nv->vely));
  RET(b2_field_create(nv->sp_temp, &nv->temp)); RET(b2_field_create(nv->sp_ortho, &nv->pres));
  RET(b2_field_create(nv->sp_pseu, &nv->pseu)); RET(b2_field_create(nv->sp_ortho, &nv->tempbc));
  const double sx2 = nv->scale[0] * nv->scale[0], sy2 = nv->scale[1] * nv->scale[1];
  RET(hholtz_create(nv->sp_vel, dt * nv->nu / sx2, dt * nv->nu / sy2, &nv->hh[0]));   // navier.rs:263-274
  RET(hholtz_create(nv->sp_vel, dt * nv->nu / sx2, dt * nv->nu / sy2, &nv->hh[1]));
  RET(hholtz_create(nv->sp_temp, dt * nv->ka / sx2, dt * nv->ka / sy2, &nv->hh[2]));
  RET(poisson_create(nv->sp_pseu, 1.0 / sx2, 1.0 / sy2, lam, fwd, bwd, &nv->pois)); // navier.rs:275
  b2_space* so = nv->sp_ortho;
  double** work[] = {&nv->that, &nv->tbc_ortho, &nv->tbc_diff, &nv->rhs, &nv->g1, &nv->g2, &nv->conv, &nv->div, &nv->ux, &nv->uy};
  for (auto w : work) RET(nav_alloc(so, w));
  CK(cudaMalloc(&nv->d_scalar, sizeof(double)));
  // tempbc, src/navier_stokes/boundary_conditions.rs:18-36 / :143-161: v[i, :] = m y + n, forward, backward
  {
    std::vector<double> y(ny), v((size_t)nx * ny);
    RET(b2_space_coords(so, 1, y.data()));
    const double x1 = y[0], x2 = y[ny - 1], y1 = 0.5, y2 = -0.5;
    const double m = (y2 - y1) / (x2 - x1), n = (y1 * x2 - y2 * x1) / (x2 - x1);
    int row0 = 0, cnt = nx;
    RET(b2_field_local_rows(nv->tempbc, B2_SHAPE_PHYSICAL, &row0, &cnt));
    if (!hc) {   // every row is the same profile
      for (int i = 0; i < nx; i++) for (int j = 0; j < ny; j++) v[(size_t)i * ny + j] = m * y[j] + n;
    } else {     // bc_hc / bc_hc_periodic (boundary_conditions.rs:103-135 / :165-195): -0.5 cos(2 pi (x - x0) / L) at the bottom,
                 // T = T' = 0 at the top: a parabola in y with its vertex at the top wall; L = x[last] - x[0] in both variants
      std::vector<double> x(nx);
      RET(b2_space_coords(so, 0, x.data()));
      const double len = x[nx - 1] - x[0], pi = 3.14159265358979323846;
      for (int i = 0; i < cnt; i++) {
        const double fx = -0.5 * std::cos(2.0 * pi * (x[row0 + i] - x[0]) / len), a = fx / ((x1 - x2) * (x1 - x2));
        for (int j = 0; j < ny; j++) v[(size_t)i * ny + j] = a * (y[j] - x2) * (y[j] - x2);
      }
    }
    RET(b2_field_set_v_host(nv->tempbc, v.data(), (size_t)cnt * ny * sizeof(double)));
    RET(b2_forward(nv->tempbc));
    RET(b2_backward(nv->tempbc));
    // constants of the step: to_ortho(tempbc) and dt*ka*(d2/dx2 + d2/dy2) tempbc (navier_eq.rs:214-218)
    RET(op_to_ortho(so, nv->tempbc->vhat->d, nv->tbc_ortho));
    RET(op_gradient(so, nv->tempbc->vhat->d, 2, 0, nv->scale, nv->tbc_diff, dt * nv->ka, false));
    RET(op_gradient(so, nv->tempbc->vhat->d, 0, 2, nv->scale, nv->tbc_diff, dt * nv->ka, true));
  }
  // ---- fused schedule: work arrays and the constants that never change during a run ----
  {
    double** fw[] = {&nv->VTv, &nv->uxT, &nv->uyT, &nv->cv[0], &nv->cv[1], &nv->cv[2], &nv->PH, &nv->PHy, &nv->F1, &nv->F2, &nv->R0, &nv->G0, &nv->G1,
                     &nv->U1, &nv->U2, &nv->U3, &nv->GxT, &nv->GyT, &nv->KbT, &nv->KTT};
    for (auto w : fw) RET(nav_alloc(so, w));
    for (int i = 0; i < 3; i++) { RET(nav_alloc(so, &nv->Pf[i])); RET(nav_alloc(so, &nv->Qf[i])); RET(nav_alloc(so, &nv->V1[i])); RET(nav_alloc(so, &nv->Cx[i])); RET(nav_alloc(so, &nv->Zf[i])); RET(nav_alloc(so, &nv->Of[i])); }
    const Base1& bxo = so->b[0]; const Base1& byo = so->b[1];
    // GxT / GyT = backward(d/dx tempbc), backward(d/dy tempbc): physical values, kept in x-lane orientation
    for (int d = 0; d < 2; d++) {
      RET(op_gradient(so, nv->tempbc->vhat->d, d == 0, d == 1, nv->scale, nv->g1));
      Prog y; y.load(nv->g1, byo.rows_ortho); int l = y.backward_ortho(byo); y.store(so->tmp[0], l, ST_TRANS);
      RET(run_pass(so, 0, y));
      Prog x; x.load(so->tmp[0], bxo.rows_ortho); l = x.backward_ortho(bxo); x.store(d == 0 ? nv->GxT : nv->GyT, l, 0);
      RET(run_pass(so, 1, x));
    }
    // KbT = dt * Hholtz_vely(to_ortho(tempbc)); KTT = Hholtz_temp(dt ka lap tempbc); both transposed
    RET(hholtz_solve(nv->hh[1], nv->tbc_ortho, nv->g1));
    { Prog y; y.load(nv->g1, so->P[1], dt); y.store(nv->KbT, so->P[1], ST_TRANS); RET(run_pass(so, 0, y)); }
    RET(hholtz_solve(nv->hh[2], nv->tbc_diff, nv->g1));
    { Prog y; y.load(nv->g1, so->P[1]); y.store(nv->KTT, so->P[1], ST_TRANS); RET(run_pass(so, 0, y)); }
  }
  CK(cudaStreamSynchronize(ctx->stream));
  *out = nv;
  return B2_OK;
}

int b2_navier_destroy(b2_navier* nv) {
  if (!nv) return B2_OK;
  double* work[] = {nv->that, nv->tbc_ortho, nv->tbc_diff, nv->rhs, nv->g1, nv->g2, nv->conv, nv->div, nv->ux, nv->uy};
  for (auto w : work) ctx_free(nv->ctx, w);
  if (nv->d_scalar) cudaFree(nv->d_scalar);
  double* fw[] = {nv->VTv, nv->uxT, nv->uyT, nv->cv[0], nv->cv[1], nv->cv[2], nv->PH, nv->PHy, nv->F1, nv->F2, nv->R0, nv->G0, nv->G1, nv->U1, nv->U2, nv->U3,
                  nv->GxT, nv->GyT, nv->KbT, nv->KTT};
  for (auto w : fw) ctx_free(nv->ctx, w);
  for (int i = 0; i < 3; i++) { ctx_free(nv->ctx, nv->Pf[i]); ctx_free(nv->ctx, nv->Qf[i]); ctx_free(nv->ctx, nv->V1[i]); ctx_free(nv->ctx, nv->Cx[i]); ctx_free(nv->ctx, nv->Zf[i]); ctx_free(nv->ctx, nv->Of[i]); }
  b2_field* fs[] = {nv->temp, nv->velx, nv->vely, nv->pres, nv->pseu, nv->tempbc};
  for (auto f : fs) b2_field_destroy(f);
#ifndef B2_EMU
  if (nv->graph) cudaGraphExecDestroy(nv->graph);
#endif
  for (auto s : nv->hh) b2_solver_destroy(s);
  b2_solver_destroy(nv->pois);
  b2_space* sps[] = {nv->sp_vel, nv->sp_temp, nv->sp_ortho, nv->sp_pseu};
  for (auto s : sps) b2_space_destroy(s);
  delete nv;
  return B2_OK;
}

int b2_navier_field(b2_navier* nv, int which, b2_field** out) {
  b2_field* fs[] = {nv->temp, nv->velx, nv->vely, nv->pres, nv->pseu, nv->tempbc};
  if (which < 0 || which > 5) return fail(B2_ERR_ARG, "field index");
  *out = fs[which];
  return B2_OK;
}

static int ew_axpby(b2_navier* nv, double* y, double a, const double* x, double b) {
  const size_t n = nv->sp_ortho->elems();
  B2_LAUNCH(k_axpby, ew_grid(n), 256, 0, nv->ctx->stream, n, y, a, x, b);
  nv->ctx->launches++;
  CK(cudaGetLastError());
  return B2_OK;
}
static int ew_muladd(b2_navier* nv, double* out, const double* u, const double* p, int acc) {
  const size_t n = nv->sp_ortho->elems();
  B2_LAUNCH(k_muladd, ew_grid(n), 256, 0, nv->ctx->stream, n, out, u, p, acc);
  nv->ctx->launches++;
  CK(cudaGetLastError());
  return B2_OK;
}

// conv_term x2 (+ bc terms), forward, dealias: navier_eq.rs:60-101 + functions.rs:56-82.  rhs -= dt * conv
static int nav_conv_into_rhs(b2_navier* nv, b2_field* f, bool with_bc) {
  b2_space* so = nv->sp_ortho;
  RET(op_gradient(f->sp, f->vhat->d, 1, 0, nv->scale, nv->g1));
  if (with_bc) RET(op_gradient(so, nv->tempbc->vhat->d, 1, 0, nv->scale, nv->g1, 1.0, true));  // linear: u * B(g_T) + u * B(g_bc)
  RET(op_backward_ortho(so, nv->g1, nv->g2));
  RET(ew_muladd(nv, nv->conv, nv->ux, nv->g2, 0));
  RET(op_gradient(f->sp, f->vhat->d, 0, 1, nv->scale, nv->g1));
  if (with_bc) RET(op_gradient(so, nv->tempbc->vhat->d, 0, 1, nv->scale, nv->g1, 1.0, true));
  RET(op_backward_ortho(so, nv->g1, nv->g2));
  RET(ew_muladd(nv, nv->conv, nv->uy, nv->g2, 1));
  return op_forward_ortho_dealias(so, nv->conv, nv->rhs, true, -nv->dt, true);
}

// one reference call = one pass pair ("unfused" mode; mirrors navier.rs:438-466 line by line)
static int nav_update_unfused(b2_navier* nv) {
  b2_space* so = nv->sp_ortho;
  const double dt = nv->dt;
  // that = temp.to_ortho() + tempbc.to_ortho()
  RET(op_to_ortho(nv->sp_temp, nv->temp->vhat->d, nv->that));
  RET(ew_axpby(nv, nv->that, 1.0, nv->tbc_ortho, 1.0));
  // convection velocity
  RET(op_backward(nv->sp_vel, nv->velx->vhat->d, nv->ux));
  RET(op_backward(nv->sp_vel, nv->vely->vhat->d, nv->uy));
  // solve_velx (navier_eq.rs:176-187)
  RET(op_to_ortho(nv->sp_vel, nv->velx->vhat->d, nv->rhs));
  RET(op_gradient(so, nv->pres->vhat->d, 1, 0, nv->scale, nv->rhs, -dt, true));
  RET(nav_conv_into_rhs(nv, nv->velx, false));
  RET(hholtz_solve(nv->hh[0], nv->rhs, nv->velx->vhat->d));
  // solve_vely (navier_eq.rs:190-203)
  RET(op_to_ortho(nv->sp_vel, nv->vely->vhat->d, nv->rhs));
  RET(op_gradient(so, nv->pres->vhat->d, 0, 1, nv->scale, nv->rhs, -dt, true));
  RET(ew_axpby(nv, nv->rhs, dt, nv->that, 1.0));
  RET(nav_conv_into_rhs(nv, nv->vely, false));
  RET(hholtz_solve(nv->hh[1], nv->rhs, nv->vely->vhat->d));
  // div (navier_eq.rs:19-24)
  RET(op_gradient(nv->sp_vel, nv->velx->vhat->d, 1, 0, nv->scale, nv->div));
  RET(op_gradient(nv->sp_vel, nv->vely->vhat->d, 0, 1, nv->scale, nv->div, 1.0, true));
  // solve_pres + remove singularity (navier_eq.rs:158-162)
  RET(poisson_solve(nv->pois, nv->div, nv->pseu->vhat->d, true));
  // correct_velocity(1.0) (navier_eq.rs:117-125)
  RET(op_gradient(nv->sp_pseu, nv->pseu->vhat->d, 1, 0, nv->scale, nv->g1, -1.0));
  RET(op_from_ortho(nv->sp_vel, nv->g1, nv->velx->vhat->d, 1.0, true));
  RET(op_gradient(nv->sp_pseu, nv->pseu->vhat->d, 0, 1, nv->scale, nv->g1, -1.0));
  RET(op_from_ortho(nv->sp_vel, nv->g1, nv->vely->vhat->d, 1.0, true));
  // update_pres (navier_eq.rs:137-143)
  RET(ew_axpby(nv, nv->pres->vhat->d, -nv->nu, nv->div, 1.0));
  RET(op_to_ortho(nv->sp_pseu, nv->pseu->vhat->d, nv->pres->vhat->d, 1.0 / dt, true));
  // solve_temp (navier_eq.rs:209-224)
  RET(op_to_ortho(nv->sp_temp, nv->temp->vhat->d, nv->rhs));
  RET(ew_axpby(nv, nv->rhs, 1.0, nv->tbc_diff, 1.0));
  RET(nav_conv_into_rhs(nv, nv->temp, true));
  RET(hholtz_solve(nv->hh[2], nv->rhs, nv->temp->vhat->d));
  nv->time += dt;
  return B2_OK;
}

// Parallel branches: stream k (0 = origin, 1/2 = side streams).  "after(k, j)": whatever is launched on stream k
// next also waits for everything launched on stream j so far.  Under stream capture these become graph edges.
static cudaStream_t nav_stream(b2_ctx* c, int k) { return k == 0 ? c->stream : c->side[k - 1]; }
static int nav_after(b2_ctx* c, int k, int j) {
  if (k == j) return B2_OK;
  cudaEvent_t e = c->evp[c->evn++ & 15];
  CK(cudaEventRecord(e, nav_stream(c, j)));
  CK(cudaStreamWaitEvent(nav_stream(c, k), e, 0));
  return B2_OK;
}

// Fused schedule: the same algebra as navier.rs:438-466 (all operators are tensor products, so the
// per-axis factors can be regrouped freely), organised as 23 lane passes + 2 GEMMs per step with
// ~91 array touches (SURVEY 8d work model) instead of one pass pair per reference call.
static int nav_update_fused(b2_navier* nv) {
  b2_space* so = nv->sp_ortho;
  b2_ctx* ctx = nv->ctx;
  const double dt = nv->dt, sx = 1.0 / nv->scale[0], sy = 1.0 / nv->scale[1];
  const Base1& bxo = so->b[0]; const Base1& byo = so->b[1];
  const Base1& bxp = nv->sp_pseu->b[0]; const Base1& byp = nv->sp_pseu->b[1];
  b2_field* fld[3] = {nv->velx, nv->vely, nv->temp};
  // dealias cuts, functions.rs:72-82 (integer division on the spectral shape of `field`)
  const int shape0 = bxo.cheb ? bxo.n : bxo.m, shape1 = byo.n;
  const int cut0 = (shape0 * 2 / 3) * (bxo.cheb ? 1 : 2), cut1 = shape1 * 2 / 3;
  const int P0 = so->P[0], P1 = so->P[1];

  // Independent passes run as parallel branches (three streams = three branches of the captured graph): a pass
  // has ~P/4 CTAs, which fills the GPU only for the largest grids.  With several GPUs every stream has its own
  // barrier flags and epoch (ctx_barrier), so the branches stay independent across the exchange barriers too.
  const bool par = nv->branches;   // (every stream has its own barrier flags)
  auto on = [&](int k) { ctx->cur = par ? nav_stream(ctx, k) : ctx->stream; };
  auto after = [&](int k, int j) -> int { return par ? nav_after(ctx, k, j) : B2_OK; };
  RET(after(1, 0)); RET(after(2, 0));   // fork
  {  // branch 2 first: pressure gradient terms, Helmholtz-y of pres and of d/dy pres
    on(2);
    Prog y;
    // (the factor -dt of the pressure-gradient terms rides on the transposing stores: the consumers' loads stay zero-copy)
    y.load(nv->pres->vhat->d, byo.rows_ortho); emit_hh_axis(y, nv->hh[0], 1); y.store(nv->PH, nv->sp_vel->b[1].m, ST_TRANS, -dt);
    y.load(nv->pres->vhat->d, byo.rows_ortho); y.deriv_axis(byo, 1, sy); emit_hh_axis(y, nv->hh[1], 1); y.store(nv->PHy, nv->sp_vel->b[1].m, ST_TRANS, -dt);
    RET(run_pass(so, 0, y));
  }
  // ---- A: along y on the three advected fields: values, d/dy values, Helmholtz-y of the old field ----
  for (int i = 0; i < 3; i++) {
    on(i);
    const b2_field* f = fld[i];
    const Base1& by = f->sp->b[1];
    const double* src = f->vhat->d;
    Prog y;
    // the orthonormal image of the lanes is needed three (four) times: project once, keep a copy (a zero-copy slab store and
    // zero-copy reloads) instead of repeating the stencil pass after every reload of the composite coefficients
    y.load(src, by.rows_spec); int lo = y.to_ortho(by); y.store(nv->Of[i], lo, 0);
    int l = y.backward_ortho(by); y.store(nv->Pf[i], l, ST_TRANS);
    y.load(nv->Of[i], lo); y.deriv_axis(by, 1, sy); l = y.backward_ortho(by); y.store(nv->Qf[i], l, ST_TRANS);
    y.load(nv->Of[i], lo); emit_hh_axis(y, nv->hh[i], 1); y.store(nv->V1[i], by.m, ST_TRANS);
    if (i == 2) { y.load(nv->Of[i], lo); emit_hh_axis(y, nv->hh[1], 1); y.store(nv->VTv, by.m, ST_TRANS); }
    RET(run_pass(so, 0, y));
  }
  // ---- A-x: convection velocities ux, uy (physical, x-lane orientation) ----
  for (int i = 0; i < 2; i++) {
    on(i);
    const Base1& bx = fld[i]->sp->b[0];
    Prog x; x.load(nv->Pf[i], bx.rows_spec); x.to_ortho(bx); int l = x.backward_ortho(bx); x.store(i == 0 ? nv->uxT : nv->uyT, l, 0);
    RET(run_pass(so, 1, x));
  }
  RET(after(1, 0)); RET(after(0, 1)); RET(after(2, 0)); RET(after(2, 1));   // every branch needs ux and uy
  // ---- B: u . grad f in physical space, forward transform along x, dealias rows ----
  for (int i = 0; i < 3; i++) {
    on(i);
    const Base1& bx = fld[i]->sp->b[0];
    Prog x;
    x.load(nv->Pf[i], bx.rows_spec); x.to_ortho(bx); x.deriv_axis(bx, 1, sx); int l = x.backward_ortho(bx);
    if (i == 2) x.load(nv->GxT, l, 1.0, LD_ACC);
    x.load(nv->uxT, l, 1.0, LD_MUL);
    x.store(nv->cv[i], l, 0);
    x.load(nv->Qf[i], bx.rows_spec); x.to_ortho(bx); l = x.backward_ortho(bx);
    if (i == 2) x.load(nv->GyT, l, 1.0, LD_ACC);
    x.load(nv->uyT, l, 1.0, LD_MUL);
    x.load(nv->cv[i], l, 1.0, LD_ACC);
    l = x.forward_ortho(bxo); x.zerotail(cut0);
    x.store(nv->Cx[i], l, ST_TRANS, -dt);   // rhs -= dt * conv: the factor rides on the store
    RET(run_pass(so, 1, x));
  }
  // ---- C-y: forward along y, dealias columns, -dt, Helmholtz-y ----
  for (int i = 0; i < 3; i++) {
    on(i);
    Prog y; y.load(nv->Cx[i], byo.rows_phys); y.forward_ortho(byo); y.zerotail(cut1);
    emit_hh_axis(y, nv->hh[i], 1); y.store(nv->Zf[i], fld[i]->sp->b[1].m, ST_TRANS);
    RET(run_pass(so, 0, y));
  }
  // ---- C-x: assemble rhs along x and finish the three Helmholtz solves ----
  RET(after(0, 2)); RET(after(1, 2));   // PH, PHy, VTv come from branch 2
  {
    const Base1& bxv = nv->sp_vel->b[0]; const Base1& bxT = nv->sp_temp->b[0];
    on(0);
    Prog x;  // velx
    x.load(nv->PH, bxo.rows_ortho); x.deriv_axis(bxo, 1, sx);
    x.load(nv->Zf[0], bxo.rows_ortho, 1.0, LD_ACC);
    x.load_stencil(nv->V1[0], bxv, 1.0, true);
    emit_hh_axis(x, nv->hh[0], 0);
    x.store(nv->velx->vhat->d, bxv.rows_spec, ST_TRANS);
    RET(run_pass(so, 1, x));
    on(1);
    Prog v;  // vely (+ buoyancy dt * (to_ortho(temp) + to_ortho(tempbc)))
    v.load(nv->PHy, bxo.rows_ortho);
    v.load(nv->Zf[1], bxo.rows_ortho, 1.0, LD_ACC);
    v.load_stencil(nv->V1[1], bxv, 1.0, true);
    v.load_stencil(nv->VTv, bxT, dt, true);
    emit_hh_axis(v, nv->hh[1], 0);
    v.load(nv->KbT, bxv.rows_spec, 1.0, LD_ACC);
    v.store(nv->vely->vhat->d, bxv.rows_spec, ST_TRANS);
    RET(run_pass(so, 1, v));
  }
  // temperature Helmholtz (branch 2: it only needs the old fields and its own convection term)
  {
    on(2);
    const Base1& bxT = nv->sp_temp->b[0];
    Prog t;
    t.load(nv->Zf[2], bxo.rows_ortho);
    t.load_stencil(nv->V1[2], bxT, 1.0, true);
    emit_hh_axis(t, nv->hh[2], 0);
    t.load(nv->KTT, bxT.rows_spec, 1.0, LD_ACC);
    t.store(nv->temp->vhat->d, bxT.rows_spec, ST_TRANS);
    RET(run_pass(so, 1, t));
  }
  RET(after(0, 1));
  on(0);
  // ---- D: divergence of the intermediate velocity, pressure update part 1, Poisson rhs ----
  {
    const Base1& byv = nv->sp_vel->b[1]; const Base1& bxv = nv->sp_vel->b[0];
    Prog y;
    y.load(nv->velx->vhat->d, byv.rows_spec); int l = y.to_ortho(byv); y.store(nv->F1, l, ST_TRANS);
    y.load(nv->vely->vhat->d, byv.rows_spec); y.to_ortho(byv); l = y.deriv_axis(byv, 1, sy); y.store(nv->F2, l, ST_TRANS);
    RET(run_pass(so, 0, y));
    Prog x;
    x.load(nv->F1, bxv.rows_spec); x.to_ortho(bxv); x.deriv_axis(bxv, 1, sx);
    x.load_stencil(nv->F2, bxv, 1.0, true);
    x.store(nv->pres->vhat->d, bxo.rows_ortho, ST_TRANS | ST_ACC, -nv->nu);   // pres += -nu div (navier_eq.rs:137-143)
    x.matvec(bxp);
    x.store(nv->R0, bxp.rows_spec, ST_TRANS);
    RET(run_pass(so, 1, x));
  }
  // ---- Poisson (src/solver/poisson.rs:195-236) ----
  b2_solver* ps = nv->pois;
  if (ps->dense) {
    // own FP64 GEMMs on the tiled arrays (gemm_f64.cuh): no row-major copies, every load / store of the lane passes
    // around them is a zero-copy slab copy; with several GPUs the exchanges ride on those stores and on the GEMM epilogue
    RET(poisson_core(ps, so, nv->R0, true, nv->G0, nv->G1, nv->pseu->vhat->d, true));
  } else {
    Prog y; y.load(nv->R0, byo.rows_ortho); y.matvec(byp);
    y.fdma(byp.m, ps->pfl.d, ps->pid.d, ps->pu1.d, ps->pu2.d, FD_PERLANE);
    y.zeroelem(0, 0); y.zeroelem(1, 0);
    y.store(nv->pseu->vhat->d, byp.m, 0);
    RET(run_pass(so, 0, y));
  }
  // ---- E: velocity correction and pressure update part 2 (navier_eq.rs:117-143) ----
  {
    const Base1& byv = nv->sp_vel->b[1]; const Base1& bxv = nv->sp_vel->b[0];
    Prog y;
    for (int k = 0; k < 3; k++) {
      if (k == 0) { y.load(nv->pseu->vhat->d, byp.m); const int lo = y.to_ortho(byp); y.store(nv->G0, lo, 0); }   // (G0 is free again: one projection, two zero-copy reloads)
      else y.load(nv->G0, byo.rows_ortho);
      if (k == 1) y.deriv_axis(byo, 1, sy);
      int l = byo.rows_ortho;
      if (k < 2) l = y.from_ortho(byv);
      y.store(k == 0 ? nv->U1 : (k == 1 ? nv->U2 : nv->U3), l, ST_TRANS);
    }
    RET(run_pass(so, 0, y));
    RET(after(1, 0)); RET(after(2, 0));
    on(0);
    Prog x1; x1.load(nv->U1, bxp.rows_spec); x1.to_ortho(bxp); x1.deriv_axis(bxo, 1, sx); int l = x1.from_ortho(bxv);
    x1.store(nv->velx->vhat->d, l, ST_TRANS | ST_ACC, -1.0);
    RET(run_pass(so, 1, x1));
    on(1);
    Prog x2; x2.load(nv->U2, bxp.rows_spec); x2.to_ortho(bxp); l = x2.from_ortho(bxv);
    x2.store(nv->vely->vhat->d, l, ST_TRANS | ST_ACC, -1.0);
    RET(run_pass(so, 1, x2));
    on(2);
    Prog x3; x3.load(nv->U3, bxp.rows_spec); l = x3.to_ortho(bxp);
    x3.store(nv->pres->vhat->d, l, ST_TRANS | ST_ACC, 1.0 / dt);
    RET(run_pass(so, 1, x3));
  }
  RET(after(0, 1)); RET(after(0, 2));   // join
  on(0);
  nv->time += dt;
  return B2_OK;
}

int b2_navier_update(b2_navier* nv, int nsteps) {
  CK(cudaSetDevice(nv->ctx->device));
  b2_ctx* ctx = nv->ctx;
  for (int s = 0; s < nsteps; s++) {
#ifndef B2_EMU
    // the fused step is a fixed launch sequence: capture it once into a CUDA graph and replay it
    if (nv->fused && nv->use_graph && !ctx->profile && !ctx->d_prof && nv->warm_steps >= 1) {
      if (!nv->graph) {
        cudaGraph_t g = nullptr;
        const long long l0 = ctx->launches;
        const double t0 = nv->time;
        CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        int r = nav_update_fused(nv);
        cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
        ctx->launches = l0; nv->time = t0;
        if (r != B2_OK) return r;
        CK(e);
        CK(cudaGraphInstantiate(&nv->graph, g, 0));
        CK(cudaGraphDestroy(g));
      }
      CK(cudaGraphLaunch(nv->graph, ctx->stream));
      ctx->launches += nv->launches_per_step;
      nv->time += nv->dt;
      continue;
    }
#endif
    long long l0 = ctx->launches;
    RET(nv->fused ? nav_update_fused(nv) : nav_update_unfused(nv));
    nv->launches_per_step = ctx->launches - l0;
    nv->warm_steps++;
  }
  return B2_OK;
}
int b2_navier_div_norm(b2_navier* nv, double* out) {
  RET(op_gradient(nv->sp_vel, nv->velx->vhat->d, 1, 0, nv->scale, nv->g1));
  RET(op_gradient(nv->sp_vel, nv->vely->vhat->d, 0, 1, nv->scale, nv->g1, 1.0, true));
  RET(norm2_dev(nv->sp_ortho, nv->g1, out, true));   // multi-rank: summed over the ranks on the device (peer heap)
  *out = std::sqrt(*out);
  return B2_OK;
}
int b2_navier_get_time(const b2_navier* nv, double* t) { *t = nv->time; return B2_OK; }
int b2_navier_set_time(b2_navier* nv, double t) {
  if (!nv) return fail(B2_ERR_ARG, "b2_navier_set_time: null handle");
  nv->time = t;
  return B2_OK;
}
int b2_navier_set_mode(b2_navier* nv, int mode) {
  // bit 0: fused schedule; bit 1: disable CUDA-graph replay; bit 2: disable parallel branches
  nv->fused = mode & 1; nv->use_graph = !(mode & 2); nv->branches = !(mode & 4); nv->warm_steps = 0;
#ifndef B2_EMU
  if (nv->graph) { cudaGraphExecDestroy(nv->graph); nv->graph = nullptr; }
#endif
  return B2_OK;
}
// out[0..7] = {parity-block GEMMs active, P0, P1, m0, ce, co, parallel branches active, lane passes per step}
int b2_navier_info(const b2_navier* nv, long long* out) {
  const b2_solver* ps = nv->pois;
  out[0] = ps && ps->blocks; out[1] = nv->sp_ortho->P[0]; out[2] = nv->sp_ortho->P[1];
  out[3] = ps ? ps->m0 : 0; out[4] = ps ? ps->ce : 0; out[5] = ps ? ps->co : 0;
  out[6] = nv->branches; out[7] = nv->launches_per_step;
  return B2_OK;
}
int b2_navier_launch_count(const b2_navier* nv, long long* k) { *k = nv->launches_per_step; return B2_OK; }
int b2_navier_poisson_matrices(b2_navier* nv, double* a0, double* cmat0, int* m0) {
  if (m0) *m0 = nv->sp_pseu->b[0].m;
  if (!a0 || !cmat0) return B2_OK;
  return b2_poisson_axis0_matrices(nv->pseu, 1.0 / (nv->scale[0] * nv->scale[0]), a0, cmat0);
}

}  // extern "C"

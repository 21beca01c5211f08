// Host orchestration of the right-to-left Gram sweep (dense TT-SVD), the TT rounding sweeps and
// the two-factor split.  Each routine is written once over an arena type so that the very same
// sequence of `take` calls sizes the workspace (ArenaSizer) and carves it (Arena).
//
// Dense TT-SVD (tn.Tensor(data, ranks_tt=r): tensor.py:401-408 -> round_tt tensor.py:2008-2083):
//   C <- T viewed (rows x I_{N-1});  for mu = N-1 .. 1:
//     G = C^T C (or C C^T when rows < cols)      Gram, fp64 accumulation   [replaces QR tensor.py:1816 + SVD round.py:96]
//     (lambda, V) = leading eigenpairs of G       Jacobi / Chebyshev subspace iteration
//     rank by the tail-energy rule                round.py:147-158
//     core_mu = V_r^T, C <- C V_r                 round.py:166-172 + tensor.py:2078-2083
//   core_0 = C.
// This is algebraically the reference's result (same subspaces, same gauge: cores 1..N-1 have
// orthonormal right unfoldings, core 0 carries the norm) without the identity-flanked full-rank TT.
#pragma once
#include "common.cuh"
#include "eig.cuh"
#include "gemm_generic.cuh"
#include "jacobi.cuh"
#include "jacobi2.cuh"
#include "small_kernels.cuh"
#include "gram_tc.cuh"
#include "gram_tc2.cuh"
#include "project.cuh"
#include "project_tc.cuh"
#include "chfsi_dev.cuh"

namespace tnb {

// C (rows x r) = A (rows x n) * V (n x r) in the data precision: streaming FFMA kernel for fp32 when the
// shape allows, generic tiled GEMM otherwise.
constexpr int64_t PROJ_TC_MIN_ROWS = 16384;
inline bool project_use_tc(int64_t rows, int64_t n, int64_t r, const void* A, const void* C) {
  return rows >= PROJ_TC_MIN_ROWS && project_tc_shape_ok(rows, n, r, A, C);
}
template <typename T>
inline int project_any(const T* A, int64_t rows, int64_t n, const T* V, int64_t r, T* C, cudaStream_t st,
                       void* tc_ws = nullptr, size_t tc_ws_bytes = 0) {
  if (std::is_same<T, float>::value && tc_ws && tc_path_available() && project_use_tc(rows, n, r, A, C))
    return project_tc_f32(reinterpret_cast<const float*>(A), rows, n, reinterpret_cast<const float*>(V), (int)r,
                          reinterpret_cast<float*>(C), tc_ws, tc_ws_bytes, st);
  if (std::is_same<T, float>::value && project_f32_fast_ok(rows, n, r, A, C))
    return project_f32_fast(reinterpret_cast<const float*>(A), rows, n, reinterpret_cast<const float*>(V), (int)r,
                            reinterpret_cast<float*>(C), st);
  return gemm_direct<T, T, T, T>(rows, r, n, A, n, true, V, r, false, C, r, (T)1, nullptr, 0, (T)0, nullptr, 0, (T)0, st);
}

// The project_tc workspace of a (rows x n) -> (rows x kcap) projection, when that kernel may run for it.
template <typename T, class ArenaT>
inline void project_tc_carve(ArenaT& ar, bool allow_tc, int64_t rows, int64_t n, int64_t kcap, void** ws, size_t* bytes) {
  *ws = nullptr;
  *bytes = 0;
  if (allow_tc && std::is_same<T, float>::value && rows >= n && rows >= PROJ_TC_MIN_ROWS && kcap <= PT_MAX_N && n % 4 == 0 &&
      n >= 32) {
    *bytes = project_tc_workspace_bytes(n, kcap);
    *ws = ar.template take<char>(*bytes);
  }
}

// Tensor cores are used unless the caller opted out; the sizing pass (dry) cannot ask the device and sizes for them.
inline bool tc_allowed(uint32_t flags, bool dry) { return !(flags & TNB_FLAG_NO_TENSORCORE) && (dry || tc_path_available()); }

// Squared tail-energy budget of one truncation step: the relative error eps is split evenly over the N - 1 bonds
// (tensor.py:2039-2051).
inline double eps_budget2(double eps, int N) {
  const double epsN = eps / std::max(1.0, std::sqrt((double)(N - 1)));
  return epsN * epsN;
}

constexpr int64_t TC_MIN_ROWS = 2048;  // below this the generic fp64-accumulating Gram is used

struct SweepDims {
  int N = 0;
  std::vector<int64_t> shape;
  std::vector<int64_t> rows;   // rows[mu] = prod_{j<mu} shape[j]
  std::vector<int64_t> rcap;   // rcap[k], k=0..N : max possible rank at bond k
  std::vector<int64_t> slot;   // element offset of core k in the cores buffer
  int64_t capacity = 0;
};

inline int make_dims(int ndim, const int64_t* shape, const int32_t* rmax, SweepDims& d) {
  if (ndim < 1 || ndim > 62) return fail(TNB_ERR_INVALID, "ndim=%d out of range", ndim);
  d.N = ndim;
  d.shape.assign(shape, shape + ndim);
  for (int k = 0; k < ndim; ++k)
    if (shape[k] < 1) return fail(TNB_ERR_INVALID, "shape[%d]=%lld must be >= 1", k, (long long)shape[k]);
  d.rows.assign(ndim + 1, 1);
  for (int k = 0; k < ndim; ++k) {
    if (d.rows[k] > (int64_t)1 << 56) return fail(TNB_ERR_INVALID, "tensor too large");
    d.rows[k + 1] = d.rows[k] * shape[k];
  }
  d.rcap.assign(ndim + 1, 1);
  for (int mu = ndim - 1; mu >= 1; --mu) {
    int64_t c = shape[mu] * d.rcap[mu + 1];
    if (d.rows[mu] < c) c = d.rows[mu];
    if (rmax && rmax[mu - 1] > 0 && rmax[mu - 1] < c) c = rmax[mu - 1];
    d.rcap[mu] = c;
  }
  d.slot.assign(ndim, 0);
  int64_t off = 0;
  for (int k = 0; k < ndim; ++k) {
    d.slot[k] = off;
    off += d.rcap[k] * shape[k] * d.rcap[k + 1];
    off = (off + 63) / 64 * 64;  // keep every core 256-byte aligned for fp32
  }
  d.capacity = off;
  return TNB_OK;
}

// Ping-pong carries of the right-to-left sweep (step t writes carry[t & 1] and reads the other), sized by the rank caps.
template <typename T, class ArenaT>
inline void carry_carve(ArenaT& ar, const SweepDims& d, T* carry[2]) {
  size_t carry_elems[2] = {0, 0};
  for (int mu = d.N - 1, t = 0; mu >= 1; --mu, ++t) {
    const size_t e = (size_t)d.rows[mu] * (size_t)d.rcap[mu];
    if (e > carry_elems[t & 1]) carry_elems[t & 1] = e;
  }
  carry[0] = ar.template take<T>(carry_elems[0]);
  carry[1] = ar.template take<T>(carry_elems[1]);
}

// ---------------------------------------------------------------------------------------------
// Gram of a (rows x n) row-major matrix on whichever side is smaller, into fp64 G (L x L).
// ---------------------------------------------------------------------------------------------
template <typename T>
struct GramWork {
  double* partial = nullptr;
  size_t partial_elems = 0;
  void* tc_ws = nullptr;
  size_t tc_bytes = 0;
};

template <typename T, class ArenaT>
inline void gram_carve(ArenaT& ar, int64_t rows, int64_t n, bool allow_tc, GramWork<T>& w) {
  const bool tall = rows >= n;
  const int64_t L = tall ? n : rows;
  const int64_t K = tall ? rows : n;
  GemmPlan pl = plan_gemm(L, L, K, true);
  w.partial_elems = pl.partial_elems;
  w.partial = ar.template take<double>(pl.partial_elems);
  w.tc_bytes = 0;
  w.tc_ws = nullptr;
  if (allow_tc && std::is_same<T, float>::value && tall && rows >= TC_MIN_ROWS && gram_tc_shape_ok(rows, n)) {
    w.tc_bytes = std::max(gram_tc_workspace_bytes(rows, n), gram_tc2_shape_ok(rows, n) ? gram_tc2_workspace_bytes(rows, n) : 0);
    w.tc_ws = ar.template take<char>(w.tc_bytes);
  }
}

template <typename T>
inline int gram_small_side(const T* C, int64_t rows, int64_t n, double* G, float* Gf, GramWork<T>& w, bool use_tc,
                           int* used_tc, cudaStream_t st) {
  const bool tall = rows >= n;
  if (used_tc) *used_tc = 0;
  if (tall) {
    if (use_tc && w.tc_ws && std::is_same<T, float>::value) {
      if (used_tc) *used_tc = 1;
      if (gram_tc2_shape_ok(rows, n))  // wide Gram: 256 x 256 tiles on CTA pairs
        return gram_tc2_f32(reinterpret_cast<const float*>(C), rows, n, G, Gf, w.tc_ws, w.tc_bytes, st);
      return gram_tc_f32(reinterpret_cast<const float*>(C), rows, n, G, Gf, w.tc_ws, w.tc_bytes, st);
    }
    GemmPlan pl = plan_gemm(n, n, rows, true);
    return gemm_splitk<T, T, double, double, float>(pl, n, n, rows, C, n, false, C, n, false, w.partial, G, n, 1.0,
                                                    nullptr, 0, 0.0, nullptr, 0, 0.0, true, Gf, n, st);
  }
  GemmPlan pl = plan_gemm(rows, rows, n, true);
  return gemm_splitk<T, T, double, double, float>(pl, rows, rows, n, C, n, true, C, n, true, w.partial, G, rows, 1.0,
                                                  nullptr, 0, 0.0, nullptr, 0, 0.0, true, Gf, rows, st);
}

// ---------------------------------------------------------------------------------------------
// Eigen stage: all eigenpairs (Jacobi) when L <= JACOBI_MAX_N, else k leading pairs (ChFSI).
// Outputs: w (>= L or b doubles, descending), V (L x ldv doubles, columns = vectors).
// ---------------------------------------------------------------------------------------------
template <typename TBk>
struct EigWork {
  double* w = nullptr;
  double* V = nullptr;
  int ldv = 0;
  double* jscratch = nullptr;
  int* jinfo = nullptr;
  bool chfsi = false;
  bool adaptive = false;  // eps-only: k grows until the rank rule is decided
  int k = 0, b = 0;       // capacity (carved); k_run / b_run are what the last solve used
  int k_run = 0, b_run = 0;
  TBk* Gb = nullptr;  // G in block precision (ChFSI only)
  ChfsiWork<TBk> cw;
};

template <typename TBk, class ArenaT>
inline int eig_carve(ArenaT& ar, int64_t L, int64_t rcap, bool have_rmax, EigWork<TBk>& e) {
  if (L <= JACOBI_MAX_N) {
    e.chfsi = false;
    e.w = ar.template take<double>(L);
    e.V = ar.template take<double>((size_t)L * L);
    e.ldv = (int)L;
    e.jscratch = ar.template take<double>(jacobi_scratch_doubles((int)L));
    e.jinfo = ar.template take<int>(4);
    return TNB_OK;
  }
  // eps-only truncation (no rank cap) of a large Gram matrix: the leading values are computed in growing blocks
  // (k = 32, 64, 128, 240) until the tail-energy rule is decided; ranks above 240 are out of reach of the subspace
  // eigensolver and raise.
  e.adaptive = !have_rmax;
  if (have_rmax && rcap + 16 > JACOBI_MAX_N)
    return fail(TNB_ERR_UNSUPPORTED, "target rank %lld too large for the subspace eigensolver (limit %d) at Gram size %lld",
                (long long)rcap, JACOBI_MAX_N - 16, (long long)L);
  if (!have_rmax || rcap + 16 > JACOBI_MAX_N) rcap = JACOBI_MAX_N - 16;
  if (L > 46000) return fail(TNB_ERR_UNSUPPORTED, "Gram size %lld too large", (long long)L);
  e.chfsi = true;
  e.k = (int)rcap;
  e.b = chfsi_default_block((int)L, e.k);
  e.w = ar.template take<double>(e.b);
  e.V = ar.template take<double>((size_t)L * e.b);
  e.ldv = e.b;
  if (!std::is_same<TBk, double>::value) e.Gb = ar.template take<TBk>((size_t)L * L);
  chfsi_carve<TBk>(ar, (int)L, e.b, e.cw);
  return TNB_OK;
}

template <typename TBk>
inline int eig_run(const double* G, const TBk* Gb_in, int64_t L, EigWork<TBk>& e, const double* d_trace,
                   ChfsiStats* stats, cudaStream_t st, bool allow_tc = false, bool shared_gpu = false, int k_try = 0,
                   double tol = 1e-6) {
  if (!e.chfsi) return jacobi2_eigh(G, (int)L, (int)L, e.w, e.V, e.jscratch, e.jinfo, st);
  e.cw.use_tc = allow_tc;
  e.cw.shared_gpu = shared_gpu;
  e.k_run = (k_try > 0 && k_try < e.k) ? k_try : e.k;
  e.b_run = chfsi_default_block((int)L, e.k_run);
  if (e.b_run > e.b) e.b_run = e.b;
  e.ldv = e.b_run;
  const TBk* Gb = Gb_in;
  if (std::is_same<TBk, double>::value) Gb = reinterpret_cast<const TBk*>(G);
  return eig_topk_chfsi<TBk>(Gb, (int)L, e.k_run, e.b_run, d_trace, tol, e.cw, e.w, e.V, stats, st);
}

// Eigen stage + rank rule + host read-back of the step scalars (one sync, which the caller needs anyway for the rank).
// eps-only truncation of a large Gram matrix (EigWork::adaptive) repeats the subspace solve with k = 32, 64, 128, 240
// leading values until the tail-energy rule is decided, with a stopping rule fine enough to resolve delta^2.
template <typename TBk>
inline int eig_solve_and_rank(const double* G, const TBk* Gb, int64_t L, EigWork<TBk>& ew, SweepScalars* sc, int* h_sc,
                              int32_t rm, int batch_mode, ChfsiStats* total, int* solves, cudaStream_t st, bool allow_tc,
                              bool shared_gpu, int used_tf32 = 0) {
  const SweepScalars* hs = reinterpret_cast<const SweepScalars*>(h_sc);
  const bool adaptive = ew.chfsi && ew.adaptive;
  int k_try = adaptive ? 32 : 0;
  double tol = 1e-6;
  if (adaptive) {
    TNB_CUDA(cudaMemcpyAsync(h_sc, sc, sizeof(SweepScalars), cudaMemcpyDeviceToHost, st));
    TNB_CUDA(cudaStreamSynchronize(st));
    const double floor_tol = std::is_same<TBk, float>::value ? 1e-7 : 1e-12;  // what fp32 / fp64 Ritz sums can resolve
    if (hs->trace > 0.0) tol = std::min(1e-6, std::max(floor_tol, 0.05 * hs->delta2 / hs->trace));
  }
  for (;;) {
    ChfsiStats cs;
    TNB_TRY(eig_run<TBk>(G, Gb, L, ew, &sc->trace, &cs, st, allow_tc, shared_gpu, k_try, tol));
    if (total)
      total->products += cs.products, total->fused_filters += cs.fused_filters, total->outer += cs.outer,
          total->rr_sweeps += cs.rr_sweeps;
    if (solves) *solves += 1;
    rank_rule_kernel<<<1, 32, 0, st>>>(ew.w, (int)L, ew.chfsi ? ew.k_run : (int)L, rm, ew.chfsi ? 1 : 0, batch_mode, sc,
                                       used_tf32, ew.chfsi ? ew.b_run : (int)L);
    TNB_LAUNCH_CHECK();
    TNB_CUDA(cudaMemcpyAsync(h_sc, sc, sizeof(SweepScalars), cudaMemcpyDeviceToHost, st));
    TNB_CUDA(cudaStreamSynchronize(st));
    if (!adaptive || !hs->undecided || hs->zero_flag) return TNB_OK;
    if (ew.k_run >= ew.k)
      return fail(TNB_ERR_UNSUPPORTED,
                  "eps-only truncation of a %lld x %lld Gram matrix needs a rank above %d; pass rmax / ranks_tt "
                  "(the direct eigensolver stops at %d)", (long long)L, (long long)L, ew.k, JACOBI_MAX_N);
    k_try = 2 * ew.k_run > 128 ? ew.k : 2 * ew.k_run;
  }
}

// ---------------------------------------------------------------------------------------------
// One truncation step, shared by the dense sweep and by phase B of TT rounding.
//   C (rows x n, row-major)  ->  core (rank x n, orthonormal rows)  and  Cn (rows x rank) with
//   C ~= Cn * core, exactly what tn.truncated_svd(M, left_ortho=False) returns (round.py:166-172,181)
//   for M = the right unfolding the reference holds at tensor.py:2054.
// ---------------------------------------------------------------------------------------------
struct SweepInfo {
  double norm = 0;
  int eig_solves = 0;
  int chfsi_products = 0;
  int fused_filters = 0;  // Chebyshev filters run as one resident kernel (cheb_filter.cuh)
  int rr_sweeps = 0, rr_solves = 0;  // Jacobi sweeps / solves of the Rayleigh-Ritz steps (diagnostic)
  int tc_grams = 0;
  int speculative = 0;  // 1: the sync-free sweep was accepted (one host synchronisation in total)
  int spec_flags = 0;   // why a speculative sweep was repeated on the host-driven path (spec_check_kernel bits)
  // TNB_FLAG_PROFILE: CUDA-event timings (ms) on the launching stream, per step (t = 0 is the first Gram)
  int nsteps = 0;
  double gram_ms[8] = {0}, eig_ms[8] = {0}, factor_ms[8] = {0};
};

// Event-based phase profiler (only active under TNB_FLAG_PROFILE; events are recorded on the stream the
// kernels are launched on, and read after the per-step synchronisation the sweep performs anyway).
struct Prof {
  bool on = false;
  std::vector<cudaEvent_t> ev;
  int used = 0;
  cudaEvent_t next() {
    if (used == (int)ev.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev.push_back(e);
    }
    return ev[used++];
  }
  void mark(cudaStream_t st) {
    if (on) cudaEventRecord(next(), st);
  }
  // after the synchronisation that ends the sweep; 4 events per step: start, after Gram, after eigen+rank, after
  // factor/projection
  void report(SweepInfo* info) const {
    const int steps = used / 4;
    info->nsteps = steps;
    for (int t = 0; t < steps && t < 8; ++t) {
      float a = 0, b = 0, c = 0;
      cudaEventElapsedTime(&a, ev[4 * t], ev[4 * t + 1]);
      cudaEventElapsedTime(&b, ev[4 * t + 1], ev[4 * t + 2]);
      cudaEventElapsedTime(&c, ev[4 * t + 2], ev[4 * t + 3]);
      info->gram_ms[t] = a;
      info->eig_ms[t] = b;
      info->factor_ms[t] = c;
    }
  }
  static Prof& get() {
    static thread_local Prof p;
    return p;
  }
};

struct StepCtx {
  SweepScalars* sc = nullptr;   // device
  int* h_sc = nullptr;          // pinned host mirror
  uint32_t flags = 0;
  bool allow_tc = false;
  double eps_scaled2 = 0;       // (eps / max(1, sqrt(N-1)))^2
  SweepInfo* info = nullptr;
  cudaStream_t st = 0;
  bool exact_gram = false;      // a TF32 Gram was rejected for this tensor: take the exact-product Gram throughout
  // speculative (sync-free) sweep
  int* d_flags = nullptr;       // device flags raised by spec_check_kernel / cd_finish_kernel
  int32_t* d_ranks = nullptr;   // the ranks the rule chose, [N + 1] (written by spec_check_kernel, not read back)

  StepCtx() = default;
  // Carves the device scalars of an N-mode sweep, and for a speculative one its device flags and ranks.
  template <class ArenaT>
  StepCtx(ArenaT& ar, int N, double eps, uint32_t flags_, bool allow_tc_, SweepInfo* info_, cudaStream_t st_, bool speculative)
      : flags(flags_), allow_tc(allow_tc_), eps_scaled2(eps_budget2(eps, N)), info(info_), st(st_) {
    sc = ar.template take<SweepScalars>(1);
    if (speculative) {
      d_flags = ar.template take<int>(4);
      d_ranks = ar.template take<int32_t>(N + 1);
    }
  }
};

// The two factors of a truncation step from the leading eigenpairs (w, V) of the Gram matrix on the smaller side of C:
// core (rank x n) and Cn (rows x rank) with C ~= Cn * core.  fac is (L x rank) scratch.
template <typename T>
inline int split_factors(const T* C, int64_t rows, int64_t n, const double* w, const double* V, int ldv, int64_t rank, T* fac,
                         void* ptc_ws, size_t ptc_bytes, bool concurrent, T* core, T* Cn, cudaStream_t st) {
  if (rows >= n) {
    // core = V_r^T (rank x n);  Cn = C V_r
    scale_extract_kernel<T><<<grid_for(n * rank), 256, 0, st>>>(V, ldv, (int)n, (int)rank, w, core, 0, 1);
    TNB_LAUNCH_CHECK();
    scale_extract_kernel<T><<<grid_for(n * rank), 256, 0, st>>>(V, ldv, (int)n, (int)rank, w, fac, 0, 0);
    TNB_LAUNCH_CHECK();
    BigKernelGate gate(st, concurrent && rows >= PROJ_TC_MIN_ROWS);
    return project_any<T>(C, rows, n, fac, rank, Cn, st, ptc_ws, ptc_bytes);
  }
  // core = diag(1/s) U_r^T C (rank x n);  Cn = U_r diag(s)
  scale_extract_kernel<T><<<grid_for(rows * rank), 256, 0, st>>>(V, ldv, (int)rows, (int)rank, w, fac, 1, 0);
  TNB_LAUNCH_CHECK();
  TNB_TRY((gemm_direct<T, T, T, T>(rank, n, rows, fac, rank, false, C, n, false, core, n, (T)1, nullptr, 0, (T)0, nullptr, 0,
                                   (T)0, st)));
  scale_extract_kernel<T><<<grid_for(rows * rank), 256, 0, st>>>(V, ldv, (int)rows, (int)rank, w, Cn, 2, 0);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

template <typename T, class ArenaT>
inline int truncate_step(ArenaT& ar, bool dry, const StepCtx& cx, const T* C, int64_t rows, int64_t n, int64_t rank_cap,
                         bool have_rmax, int32_t rm, bool first_step, T* core, T* Cn, int64_t* rank_out) {
  typedef T TBk;  // block precision of the subspace eigensolver follows the data
  const bool tall = rows >= n;
  const int64_t L = tall ? n : rows;
  const int batch_mode = (cx.flags & TNB_FLAG_BATCH_MODE) ? 1 : 0;
  cudaStream_t st = cx.st;
  GramWork<T> gw;
  EigWork<TBk> ew;
  // The TF32 Gram equals (1 - c) * G, c ~ 7e-4 (operand truncation shrinks every product alike: harmless, the rank
  // rule works on ratios) plus noise of ~1.6e-6 * ||G|| (measured, tests/test_model.py) — a floor under the tail
  // energies the rank rule can resolve.  An eps budget between "inactive" and 1e-4 of the trace needs finer
  // resolution than that: those sweeps take the exact-product fp64-accumulating Gram instead.
  const bool tc_gram = cx.allow_tc && !cx.exact_gram && (dry || cx.eps_scaled2 < 1e-20 || cx.eps_scaled2 >= 1e-4);
  gram_carve<T>(ar, rows, n, tc_gram, gw);
  double* G = ar.template take<double>((size_t)L * L);
  float* Gf = nullptr;
  const int64_t kcap = std::min<int64_t>(rank_cap, L);
  TNB_TRY(eig_carve<TBk>(ar, L, kcap, have_rmax, ew));
  if (ew.chfsi && std::is_same<TBk, float>::value) Gf = reinterpret_cast<float*>(ew.Gb);
  T* fac = ar.template take<T>((size_t)L * (size_t)kcap);  // V_r or U_r/s
  void* ptc_ws;
  size_t ptc_bytes;
  project_tc_carve<T>(ar, cx.allow_tc, rows, n, kcap, &ptc_ws, &ptc_bytes);
  if (dry) return TNB_OK;
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "workspace too small (need > %zu bytes)", ar.off);
  Prof& prof = Prof::get();
  prof.mark(st);
  int used_tc = 0;
  const bool concurrent = (cx.flags & TNB_FLAG_CONCURRENT) != 0;
  {
    BigKernelGate gate(st, concurrent && gw.tc_ws != nullptr);
    TNB_TRY(gram_small_side<T>(C, rows, n, G, Gf, gw, tc_gram, &used_tc, st));
  }
  if (cx.info) cx.info->tc_grams += used_tc;
  trace_kernel<<<1, 256, 0, st>>>(G, (int)L, (int)L, cx.sc, first_step ? 1 : 0, cx.eps_scaled2);
  TNB_LAUNCH_CHECK();
  prof.mark(st);
  ChfsiStats cs;
  int solves = 0;
  TNB_TRY(eig_solve_and_rank<TBk>(G, reinterpret_cast<const TBk*>(Gf), L, ew, cx.sc, cx.h_sc, rm, batch_mode, &cs, &solves, st,
                                  cx.allow_tc, concurrent, used_tc));
  if (used_tc && reinterpret_cast<const SweepScalars*>(cx.h_sc)->tf32_reject) {
    // the spectrum is too steep for the TF32 noise floor (small_kernels.cuh::tf32_gram_rejected): same step again on
    // the exact-product, fp64-accumulated Gram
    if (cx.info) cx.info->tc_grams -= 1;
    used_tc = 0;
    TNB_TRY(gram_small_side<T>(C, rows, n, G, Gf, gw, false, nullptr, st));
    trace_kernel<<<1, 256, 0, st>>>(G, (int)L, (int)L, cx.sc, first_step ? 1 : 0, cx.eps_scaled2);
    TNB_LAUNCH_CHECK();
    TNB_TRY(eig_solve_and_rank<TBk>(G, reinterpret_cast<const TBk*>(Gf), L, ew, cx.sc, cx.h_sc, rm, batch_mode, &cs, &solves,
                                    st, cx.allow_tc, concurrent, 0));
  }
  if (cx.info) cx.info->eig_solves += solves, cx.info->chfsi_products += cs.products, cx.info->fused_filters += cs.fused_filters,
        cx.info->rr_sweeps += cs.rr_sweeps, cx.info->rr_solves += cs.outer;
  prof.mark(st);
  const SweepScalars* hs = reinterpret_cast<const SweepScalars*>(cx.h_sc);
  if (first_step && cx.info) cx.info->norm = std::sqrt(hs->norm2 > 0 ? hs->norm2 : 0.0);
  int64_t rank = hs->rank;
  if (rank > kcap) rank = kcap;
  if (hs->zero_flag) {  // round.py:137-145: rank-1 zero factors
    rank = 1;
    fill_kernel<T><<<grid_for(n), 256, 0, st>>>(core, n, (T)0);
    TNB_LAUNCH_CHECK();
    fill_kernel<T><<<grid_for(rows), 256, 0, st>>>(Cn, rows, (T)0);
    TNB_LAUNCH_CHECK();
  } else {
    TNB_TRY(split_factors<T>(C, rows, n, ew.w, ew.V, ew.ldv, rank, fac, ptc_ws, ptc_bytes, concurrent, core, Cn, st));
  }
  prof.mark(st);
  *rank_out = rank;
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// The same truncation step, SPECULATIVE: enqueued without any host round trip, assuming the rank rule will return the
// cap (rank_cap) — which it does whenever a rank cap decides (ranks_tt= with an inactive eps budget, the benchmark's
// and the common case).  The rule still runs on the device; spec_check_kernel records what it chose and raises a flag
// if it differs (rank-deficient data, zero unfolding), if the TF32 Gram is not accurate enough for this spectrum, or if
// the sync-free subspace solver failed; the caller looks at the flags ONCE, after the whole sweep, and repeats the
// decomposition on the host-driven path when any is set.  Eligibility is decided up front by spec_eligible().
// ---------------------------------------------------------------------------------------------
template <typename T>
inline bool spec_step_ok(int64_t rows, int64_t n, int64_t rank_cap, bool allow_tc) {
  const int64_t L = rows >= n ? n : rows;
  if (L <= JACOBI_MAX_N) return true;
  if (!std::is_same<T, float>::value || !allow_tc) return false;
  const int64_t k = std::min<int64_t>(rank_cap, L);
  if (k + 16 > JACOBI_MAX_N) return false;
  return chfsi_dev_ok((int)L, chfsi_dev_block((int)L, (int)k));
}

// The step is split in enqueue phases (Gram; the eigen stages one by one; rank rule + projection) so that a batch of
// tensors can be interleaved phase by phase (ttsvd_batch_impl): the whole-GPU kernels of the batch then run back to back
// while the latency-bound eigen chains of the other tensors run beside them on their own streams.
template <typename T>
struct SpecStep {
  GramWork<T> gw;
  double *G = nullptr, *w = nullptr, *V = nullptr, *jscratch = nullptr;
  int* jinfo = nullptr;
  float* Gf = nullptr;
  CdWork<float> cw;
  T* fac = nullptr;
  void* ptc_ws = nullptr;
  size_t ptc_bytes = 0;
  int ldv = 0, b = 0, used_tc = 0;
  bool chfsi = false, tc_gram = false;
  int64_t L = 0, kcap = 0;
  CdRun cd;  // the subspace solve of this step, enqueued stage by stage
};

template <typename T, class ArenaT>
inline void spec_step_carve(ArenaT& ar, const StepCtx& cx, int64_t rows, int64_t n, int64_t rank_cap, SpecStep<T>& s) {
  const bool tall = rows >= n;
  s.L = tall ? n : rows;
  const int64_t L = s.L;
  s.tc_gram = cx.allow_tc && !cx.exact_gram;
  gram_carve<T>(ar, rows, n, s.tc_gram, s.gw);
  s.G = ar.template take<double>((size_t)L * L);
  s.kcap = std::min<int64_t>(rank_cap, L);
  s.chfsi = L > JACOBI_MAX_N;
  s.ldv = (int)L;
  s.b = 0;
  s.Gf = nullptr;
  if (!s.chfsi) {
    s.w = ar.template take<double>(L);
    s.V = ar.template take<double>((size_t)L * L);
    s.jscratch = ar.template take<double>(jacobi_scratch_doubles((int)L));
    s.jinfo = ar.template take<int>(4);
  } else {
    s.b = chfsi_dev_block((int)L, (int)s.kcap);
    s.w = ar.template take<double>(s.b);
    s.V = ar.template take<double>((size_t)L * s.b);
    s.ldv = s.b;
    s.Gf = ar.template take<float>((size_t)L * L);
    chfsi_dev_carve<float>(ar, (int)L, s.b, s.cw);
  }
  s.fac = ar.template take<T>((size_t)L * (size_t)s.kcap);
  project_tc_carve<T>(ar, cx.allow_tc, rows, n, s.kcap, &s.ptc_ws, &s.ptc_bytes);
}

// phase 1: Gram + trace
template <typename T>
inline int spec_step_gram(const StepCtx& cx, const T* C, int64_t rows, int64_t n, bool first_step, SpecStep<T>& s, bool prof_on) {
  cudaStream_t st = cx.st;
  Prof& prof = Prof::get();
  if (prof_on) prof.mark(st);
  const bool concurrent = (cx.flags & TNB_FLAG_CONCURRENT) != 0;
  {
    BigKernelGate gate(st, concurrent && s.gw.tc_ws != nullptr);
    TNB_TRY(gram_small_side<T>(C, rows, n, s.G, s.Gf, s.gw, s.tc_gram, &s.used_tc, st));
  }
  if (cx.info) cx.info->tc_grams += s.used_tc;
  trace_kernel<<<1, 256, 0, st>>>(s.G, (int)s.L, (int)s.L, cx.sc, first_step ? 1 : 0, cx.eps_scaled2);
  TNB_LAUNCH_CHECK();
  if (prof_on) prof.mark(st);
  return TNB_OK;
}

// phase 2a: start the eigen stage — a small Gram matrix is solved right here (one Jacobi kernel), a large one begins its
// subspace solve, whose stages are enqueued one at a time by spec_step_eig_stage so that a batch can interleave them
template <typename T>
inline int spec_step_eig_begin(const StepCtx& cx, SpecStep<T>& s) {
  const int64_t L = s.L;
  cudaStream_t st = cx.st;
  if (!s.chfsi) {
    // a TF32 Gram is accurate to ~2e-6 ||G||: rotating it in fp32 (backward error ~1e-6 ||G||, covered by the accept rule's
    // noise allowance) is consistent with it and 3-4x cheaper than fp64 on this machine (~16 fp64 FMAs / clk / SM);
    // eigenvalues still come out as fp64 Rayleigh quotients and the vectors are re-orthonormalised (jacobi2.cuh).
    // The same holds for fp32 DATA whatever Gram kernel produced G, as long as the accept rule — which then guards the
    // fp32 solve instead of the TF32 Gram, same noise allowance — finds the spectrum benign; a rejected step is repeated
    // on the host-driven path with fp64 rotations.
    const bool single = std::is_same<T, float>::value && (cx.allow_tc && !cx.exact_gram) && jacobi2_ok((int)L, true);
    s.used_tc = (s.used_tc || single) ? 1 : 0;
    return jacobi2_eigh(s.G, (int)L, (int)L, s.w, s.V, s.jscratch, s.jinfo, st, single, single ? 2e-6 : 0.0);
  }
  if (cx.info) cx.info->eig_solves += 1;
  return cd_begin(s.cd, s.Gf, (int)L, (int)s.kcap, s.b, &cx.sc->trace, 1e-6, s.cw, s.w, s.V, cx.d_flags, st);
}
template <typename T>
inline int spec_step_eig_stage(SpecStep<T>& s, int stage) {
  return s.chfsi ? cd_stage(s.cd, stage) : TNB_OK;
}

// phase 2b: end of the eigen stage, rank rule + speculation check, factor extraction, projection
template <typename T>
inline int spec_step_rest(const StepCtx& cx, const T* C, int64_t rows, int64_t n, int32_t rm, T* core, T* Cn, int mu,
                          SpecStep<T>& s, bool prof_on) {
  const int64_t L = s.L;
  const int batch_mode = (cx.flags & TNB_FLAG_BATCH_MODE) ? 1 : 0;
  cudaStream_t st = cx.st;
  Prof& prof = Prof::get();
  const bool concurrent = (cx.flags & TNB_FLAG_CONCURRENT) != 0;
  if (!s.chfsi) {
    rank_rule_kernel<<<1, 32, 0, st>>>(s.w, (int)L, (int)L, rm, 0, batch_mode, cx.sc, s.used_tc, (int)L);
  } else {
    TNB_TRY(cd_end(s.cd));
    rank_rule_kernel<<<1, 32, 0, st>>>(s.w, (int)L, (int)s.kcap, rm, 1, batch_mode, cx.sc, s.used_tc, s.b);
  }
  TNB_LAUNCH_CHECK();
  spec_check_kernel<<<1, 32, 0, st>>>(cx.sc, (int)s.kcap, cx.d_ranks + mu, cx.d_flags);
  TNB_LAUNCH_CHECK();
  if (prof_on) prof.mark(st);
  TNB_TRY(split_factors<T>(C, rows, n, s.w, s.V, s.ldv, s.kcap, s.fac, s.ptc_ws, s.ptc_bytes, concurrent, core, Cn, st));
  if (prof_on) prof.mark(st);
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// Dense TT-SVD
// ---------------------------------------------------------------------------------------------
template <typename T, class ArenaT>
inline int ttsvd_sync_impl(ArenaT& ar, bool dry, const T* data, const SweepDims& d, const int32_t* rmax, double eps,
                           uint32_t flags, T* cores, int32_t* ranks_host, SweepInfo* info, cudaStream_t st,
                           bool exact_gram = false) {
  const int N = d.N;
  StepCtx cx(ar, N, eps, flags, tc_allowed(flags, dry), info, st, false);
  cx.exact_gram = exact_gram;
  Prof& prof = Prof::get();
  prof.on = !dry && (flags & TNB_FLAG_PROFILE);
  prof.used = 0;
  if (!dry) {
    cx.h_sc = static_cast<int*>(pinned_scratch(sizeof(SweepScalars)));
    if (!cx.h_sc) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
    ranks_host[0] = 1;
    ranks_host[N] = 1;
  }
  if (N == 1) {
    if (!dry) {
      TNB_CUDA(cudaMemcpyAsync(cores + d.slot[0], data, sizeof(T) * d.shape[0], cudaMemcpyDeviceToDevice, st));
      TNB_CUDA(cudaStreamSynchronize(st));
      if (info) info->norm = 0;
    }
    return TNB_OK;
  }
  T* carry[2];
  carry_carve<T>(ar, d, carry);
  const T* C = data;
  int64_t r_next = 1;
  size_t peak = ar.off;
  for (int mu = N - 1, t = 0; mu >= 1; --mu, ++t) {
    const int64_t rows = d.rows[mu];
    const int64_t n = dry ? d.shape[mu] * d.rcap[mu + 1] : d.shape[mu] * r_next;
    const bool have_rmax = rmax && rmax[mu - 1] > 0;
    const size_t mark = ar.off;
    int64_t rank = d.rcap[mu];
    TNB_TRY((truncate_step<T>(ar, dry, cx, C, rows, n, d.rcap[mu], have_rmax, have_rmax ? rmax[mu - 1] : 0, t == 0,
                              dry ? nullptr : cores + d.slot[mu], carry[t & 1], &rank)));
    if (!dry) {
      ranks_host[mu] = (int32_t)rank;
      r_next = rank;
      C = carry[t & 1];
    }
    if (ar.off > peak) peak = ar.off;  // the sizing pass reports the largest step
    ar.off = mark;                     // release the step scratch
  }
  if (dry) ar.off = peak;
  if (!dry) {
    TNB_CUDA(cudaMemcpyAsync(cores + d.slot[0], C, sizeof(T) * (size_t)d.shape[0] * (size_t)r_next,
                             cudaMemcpyDeviceToDevice, st));
    TNB_CUDA(cudaStreamSynchronize(st));
    if (prof.on && info) prof.report(info);
    prof.on = false;
  }
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// Speculative dense TT-SVD: the whole right-to-left sweep enqueued in one go, ONE synchronisation at the end.
// ---------------------------------------------------------------------------------------------
// A rank cap on every bond of an N-mode train: the condition under which the sizing pass sizes a speculative path.
inline bool caps_on_every_bond(const int32_t* rmax, int N) {
  if (N < 2 || !rmax) return false;
  for (int k = 0; k < N - 1; ++k)
    if (rmax[k] <= 0) return false;
  return true;
}
// The speculative paths assume every rank is its cap: the caller did not opt out, a cap decides every bond, and no
// active eps budget decides ranks instead.
inline bool caps_decide(const int32_t* rmax, int N, double eps, uint32_t flags) {
  return !(flags & TNB_FLAG_NO_SPECULATE) && eps_budget2(eps, N) < 1e-20 && caps_on_every_bond(rmax, N);
}

template <typename T>
inline bool spec_eligible(const SweepDims& d, const int32_t* rmax, double eps, uint32_t flags, bool allow_tc) {
  if (!caps_decide(rmax, d.N, eps, flags)) return false;
  for (int mu = d.N - 1; mu >= 1; --mu)
    if (!spec_step_ok<T>(d.rows[mu], d.shape[mu] * d.rcap[mu + 1], d.rcap[mu], allow_tc)) return false;
  return true;
}

struct SpecHostBack {  // pinned read-back of one speculative sweep
  SweepScalars sc;
  int flags[4];
};

// The ranks of an accepted speculation: every bond took its cap.
inline void ranks_from_caps(const std::vector<int64_t>& rcap, int32_t* ranks_host) {
  const int N = (int)rcap.size() - 1;
  ranks_host[0] = 1;
  ranks_host[N] = 1;
  for (int mu = 1; mu < N; ++mu) ranks_host[mu] = (int32_t)rcap[mu];
}

// One tensor of a speculative sweep (or of a batch of them): its arena, device scalars, carries and position.
template <typename T, class ArenaT>
struct SpecRun {
  ArenaT* ar = nullptr;
  StepCtx cx;
  const T* C = nullptr;
  T* carry[2] = {nullptr, nullptr};
  T* cores = nullptr;
  SpecStep<T> step;
  size_t mark = 0, peak = 0;
};

template <typename T, class ArenaT>
inline int spec_begin(SpecRun<T, ArenaT>& r, ArenaT& ar, bool dry, const T* data, const SweepDims& d, double eps,
                      uint32_t flags, T* cores, SweepInfo* info, cudaStream_t st) {
  r.ar = &ar;
  r.cx = StepCtx(ar, d.N, eps, flags, tc_allowed(flags, dry), info, st, true);
  carry_carve<T>(ar, d, r.carry);
  r.C = data;
  r.cores = cores;
  r.peak = ar.off;
  if (!dry) TNB_CUDA(cudaMemsetAsync(r.cx.d_flags, 0, 4 * sizeof(int), st));
  return TNB_OK;
}

// the step scratch of step t+1 reuses that of step t: the kernels of one stream run in order, and every kernel of
// step t+1 that writes scratch is enqueued after every kernel of step t that reads it
template <typename T, class ArenaT>
inline int spec_phase1(SpecRun<T, ArenaT>& r, bool dry, const SweepDims& d, int mu, int t, bool prof_on) {
  ArenaT& ar = *r.ar;
  r.mark = ar.off;
  spec_step_carve<T>(ar, r.cx, d.rows[mu], d.shape[mu] * d.rcap[mu + 1], d.rcap[mu], r.step);
  if (ar.off > r.peak) r.peak = ar.off;
  if (dry) return TNB_OK;
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "workspace too small (need > %zu bytes)", ar.off);
  return spec_step_gram<T>(r.cx, r.C, d.rows[mu], d.shape[mu] * d.rcap[mu + 1], t == 0, r.step, prof_on);
}
template <typename T, class ArenaT>
inline int spec_phase2a(SpecRun<T, ArenaT>& r, bool dry) {
  return dry ? TNB_OK : spec_step_eig_begin<T>(r.cx, r.step);
}
template <typename T, class ArenaT>
inline int spec_phase2s(SpecRun<T, ArenaT>& r, bool dry, int stage) {
  return dry ? TNB_OK : spec_step_eig_stage<T>(r.step, stage);
}
template <typename T, class ArenaT>
inline int spec_phase2b(SpecRun<T, ArenaT>& r, bool dry, const SweepDims& d, const int32_t* rmax, int mu, int t, bool prof_on) {
  ArenaT& ar = *r.ar;
  if (!dry) {
    TNB_TRY(spec_step_rest<T>(r.cx, r.C, d.rows[mu], d.shape[mu] * d.rcap[mu + 1], rmax[mu - 1], r.cores + d.slot[mu],
                              r.carry[t & 1], mu, r.step, prof_on));
    r.C = r.carry[t & 1];
  }
  ar.off = r.mark;
  return TNB_OK;
}
// the whole phase 2 of one tensor
template <typename T, class ArenaT>
inline int spec_phase2(SpecRun<T, ArenaT>& r, bool dry, const SweepDims& d, const int32_t* rmax, int mu, int t, bool prof_on) {
  TNB_TRY((spec_phase2a<T, ArenaT>(r, dry)));
  for (int stage = 0; stage <= CD_MAX_STAGES; ++stage) TNB_TRY((spec_phase2s<T, ArenaT>(r, dry, stage)));
  return spec_phase2b<T, ArenaT>(r, dry, d, rmax, mu, t, prof_on);
}
template <typename T, class ArenaT>
inline int spec_end(SpecRun<T, ArenaT>& r, const SweepDims& d, SpecHostBack* hb) {
  cudaStream_t st = r.cx.st;
  TNB_CUDA(cudaMemcpyAsync(r.cores + d.slot[0], r.C, sizeof(T) * (size_t)d.shape[0] * (size_t)d.rcap[1],
                           cudaMemcpyDeviceToDevice, st));
  TNB_CUDA(cudaMemcpyAsync(&hb->sc, r.cx.sc, sizeof(SweepScalars), cudaMemcpyDeviceToHost, st));
  TNB_CUDA(cudaMemcpyAsync(hb->flags, r.cx.d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
  return TNB_OK;
}
// An accepted sweep, after the stream has been synchronised: ranks = caps, the scalars from the read-back.
inline void spec_accept(const SpecHostBack& hb, const SweepDims& d, int32_t* ranks_host, SweepInfo* info) {
  ranks_from_caps(d.rcap, ranks_host);
  if (info) {
    info->norm = std::sqrt(hb.sc.norm2 > 0 ? hb.sc.norm2 : 0.0);
    info->chfsi_products += hb.flags[1];
    info->rr_solves += hb.flags[2];
    info->rr_sweeps += hb.flags[3];
    info->fused_filters += hb.flags[2] - info->eig_solves;  // every Rayleigh-Ritz step but the first of a solve follows a filter
  }
}

// A real run enqueues the sweep, synchronises once and returns the device flags; the result stands when they are 0.
template <typename T, class ArenaT>
inline int ttsvd_spec_impl(ArenaT& ar, bool dry, const T* data, const SweepDims& d, const int32_t* rmax, double eps,
                           uint32_t flags, T* cores, int32_t* ranks_host, SweepInfo* info, cudaStream_t st,
                           int* spec_flags) {
  const int N = d.N;
  Prof& prof = Prof::get();
  prof.on = !dry && (flags & TNB_FLAG_PROFILE);
  prof.used = 0;
  const bool prof_on = prof.on;
  SpecHostBack* hb = nullptr;
  if (!dry) {
    hb = static_cast<SpecHostBack*>(pinned_scratch(sizeof(SpecHostBack)));
    if (!hb) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
  }
  SpecRun<T, ArenaT> r;
  TNB_TRY((spec_begin<T, ArenaT>(r, ar, dry, data, d, eps, flags, cores, info, st)));
  for (int mu = N - 1, t = 0; mu >= 1; --mu, ++t) {
    int rc = spec_phase1<T, ArenaT>(r, dry, d, mu, t, prof_on);
    if (rc == TNB_OK) rc = spec_phase2<T, ArenaT>(r, dry, d, rmax, mu, t, prof_on);
    if (rc != TNB_OK) {
      if (!dry) cudaStreamSynchronize(st);  // part of the sweep is enqueued: drain it before the host-driven path
      prof.on = false;
      return rc;
    }
  }
  if (dry) {
    ar.off = r.peak;
    return TNB_OK;
  }
  TNB_TRY((spec_end<T, ArenaT>(r, d, hb)));
  TNB_CUDA(cudaStreamSynchronize(st));
  *spec_flags = hb->flags[0];
  if (*spec_flags == 0) spec_accept(*hb, d, ranks_host, info);
  if (prof_on && info) prof.report(info);
  prof.on = false;
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// Speculate, then fall back: the policy of dense TT-SVD (ttsvd_impl) and TT rounding (tt_round_any).
//   spec(dry, &flags): a real run enqueues the speculative path, synchronises once, returns the device flags and, when
//                      they are 0, writes the result
//   sync(dry, flags):  the host-driven path, given the flags of the rejected speculation (0 when none ran)
// The sizing pass cannot ask the device what it supports: there `try_spec` is the caller's precondition instead of its
// eligibility test, and the workspace fits the larger path.  A flag, TNB_ERR_UNSUPPORTED or TNB_ERR_NOCONV restores
// the caller's info and arena and runs the host-driven path; any other error is returned.
// ---------------------------------------------------------------------------------------------
template <class ArenaT, class Spec, class Sync>
inline int speculate_or_fall_back(ArenaT& ar, bool dry, bool try_spec, SweepInfo* info, Spec spec, Sync sync) {
  const size_t base = ar.off;
  if (dry) {
    size_t need_spec = 0;
    if (try_spec) {
      int flags = 0;
      if (spec(true, &flags) == TNB_OK) need_spec = ar.off - base;
      ar.off = base;
    }
    const int rc = sync(true, 0);
    if (rc == TNB_OK && need_spec > ar.off - base) ar.off = base + need_spec;
    return rc;
  }
  if (!try_spec) return sync(false, 0);
  SweepInfo saved;
  if (info) saved = *info;
  int flags = 0;
  const int rc = spec(false, &flags);
  if (rc == TNB_OK && flags == 0) {
    if (info) info->speculative = 1;
    return TNB_OK;
  }
  if (rc != TNB_OK && rc != TNB_ERR_UNSUPPORTED && rc != TNB_ERR_NOCONV) return rc;
  if (info) {
    *info = saved;
    info->spec_flags = flags;
  }
  ar.off = base;
  ar.ok = true;
  return sync(false, flags);
}

template <typename T, class ArenaT>
inline int ttsvd_impl(ArenaT& ar, bool dry, const T* data, const SweepDims& d, const int32_t* rmax, double eps,
                      uint32_t flags, T* cores, int32_t* ranks_host, SweepInfo* info, cudaStream_t st) {
  const bool try_spec = dry ? caps_on_every_bond(rmax, d.N) : spec_eligible<T>(d, rmax, eps, flags, tc_allowed(flags, false));
  return speculate_or_fall_back(
      ar, dry, try_spec, info,
      [&](bool dr, int* spec_flags) {
        return ttsvd_spec_impl<T>(ar, dr, data, d, rmax, eps, flags, cores, ranks_host, info, st, spec_flags);
      },
      // flag bit 0: the TF32 Gram is too coarse for this spectrum, so the repeat takes exact-product Gram matrices
      [&](bool dr, int spec_flags) {
        return ttsvd_sync_impl<T>(ar, dr, data, d, rmax, eps, flags, cores, ranks_host, info, st, (spec_flags & 1) != 0);
      });
}

// ---------------------------------------------------------------------------------------------
// A batch of independent dense tensors of one shape (the reference's `batch=True` constructor, tensor.py:401-408 with
// a leading batch dimension; north_star: "batched decompositions").  Up to `inflight` speculative sweeps are enqueued
// from ONE host thread, interleaved phase by phase on internal streams, and synchronised once; tensors whose
// speculation the device rejected are then repeated one by one on the host-driven path.
// ---------------------------------------------------------------------------------------------
constexpr int TNB_BATCH_MAX_INFLIGHT = 8;

struct StreamPool {
  cudaStream_t st[TNB_BATCH_MAX_INFLIGHT] = {};
  cudaEvent_t ev[TNB_BATCH_MAX_INFLIGHT + 1] = {};
  bool ready = false;
  std::mutex mu;
  int ensure() {
    if (ready) return TNB_OK;
    for (int i = 0; i < TNB_BATCH_MAX_INFLIGHT; ++i) TNB_CUDA(cudaStreamCreateWithFlags(&st[i], cudaStreamNonBlocking));
    for (int i = 0; i <= TNB_BATCH_MAX_INFLIGHT; ++i) TNB_CUDA(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    ready = true;
    return TNB_OK;
  }
  static StreamPool& get() {
    static StreamPool pools[TNB_MAX_DEVICES];
    return pools[current_device_index()];
  }
};

// The batch form of speculate_or_fall_back over workspace slices of `per_tensor_bytes`.  Without speculation, or with
// fewer than two tensors or slices, tensor i goes through one(ar, i, info).  Otherwise enqueue(streams, n, hbs) puts the
// speculative work of every tensor on n internal streams forked from `st` (tensor i reads back into hbs[i]), the streams
// are joined back and the host synchronises once; then tensor i is accepted, accept(i, hbs[i]), or repeated host-driven
// on `st`, repeat(ar, i, flags).  spec_host[i] (may be null) says which.
template <class One, class Enqueue, class Accept, class Repeat>
inline int spec_batch(void* workspace, size_t per_tensor_bytes, int inflight, int batch, bool spec, int32_t* spec_host,
                      cudaStream_t st, One one, Enqueue enqueue, Accept accept, Repeat repeat) {
  if (!spec || inflight < 2 || batch < 2) {
    for (int i = 0; i < batch; ++i) {
      Arena ar(workspace, per_tensor_bytes);
      SweepInfo info;
      TNB_TRY(one(ar, i, &info));
      if (spec_host) spec_host[i] = info.speculative;
    }
    return TNB_OK;
  }
  if (inflight > TNB_BATCH_MAX_INFLIGHT) inflight = TNB_BATCH_MAX_INFLIGHT;
  if (inflight > batch) inflight = batch;
  StreamPool& pool = StreamPool::get();
  std::lock_guard<std::mutex> lk(pool.mu);  // one batch at a time per device uses the internal streams
  TNB_TRY(pool.ensure());
  SpecHostBack* hbs = static_cast<SpecHostBack*>(pinned_scratch((size_t)batch * sizeof(SpecHostBack)));
  if (!hbs) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
  // fork: the internal streams start after whatever the caller enqueued on `st`
  TNB_CUDA(cudaEventRecord(pool.ev[TNB_BATCH_MAX_INFLIGHT], st));
  for (int s = 0; s < inflight; ++s) TNB_CUDA(cudaStreamWaitEvent(pool.st[s], pool.ev[TNB_BATCH_MAX_INFLIGHT], 0));
  const int rc = enqueue(pool.st, inflight, hbs);
  // join: the caller's stream continues after every internal stream; then the one host synchronisation
  for (int s = 0; s < inflight; ++s) {
    cudaEventRecord(pool.ev[s], pool.st[s]);
    cudaStreamWaitEvent(st, pool.ev[s], 0);
  }
  TNB_CUDA(cudaStreamSynchronize(st));
  if (rc != TNB_OK && rc != TNB_ERR_UNSUPPORTED && rc != TNB_ERR_NOCONV) return rc;
  // read every outcome out of the pinned block first: the host-driven repeats below reuse that scratch
  std::vector<int> flags(batch, 0);
  for (int i = 0; i < batch && rc == TNB_OK; ++i) {
    flags[i] = hbs[i].flags[0];
    if (flags[i] == 0) accept(i, hbs[i]);
  }
  for (int i = 0; i < batch; ++i) {
    const bool accepted = rc == TNB_OK && flags[i] == 0;
    if (!accepted) {
      Arena ar(workspace, per_tensor_bytes);
      TNB_TRY(repeat(ar, i, flags[i]));
    }
    if (spec_host) spec_host[i] = accepted ? 1 : 0;
  }
  return TNB_OK;
}

template <typename T>
inline int ttsvd_batch_impl(void* workspace, size_t per_tensor_bytes, int inflight, const T* const* data, int batch,
                            const SweepDims& d, const int32_t* rmax, double eps, uint32_t flags, T* const* cores,
                            int32_t* ranks_host, double* norms_host, int32_t* spec_host, cudaStream_t st) {
  const int N = d.N;
  char* ws = static_cast<char*>(workspace);
  auto ranks = [&](int i) { return ranks_host + (size_t)i * (N + 1); };
  auto one = [&](Arena& ar, int i, SweepInfo* info) {
    TNB_TRY((ttsvd_impl<T, Arena>(ar, false, data[i], d, rmax, eps, flags, cores[i], ranks(i), info, st)));
    if (norms_host) norms_host[i] = info->norm;
    return TNB_OK;
  };
  auto enqueue = [&](cudaStream_t* streams, int inflight, SpecHostBack* hbs) {
    const uint32_t bflags = (flags | TNB_FLAG_CONCURRENT) & ~TNB_FLAG_PROFILE;
    int rc = TNB_OK;
    for (int g0 = 0; g0 < batch && rc == TNB_OK; g0 += inflight) {
      const int g = std::min(inflight, batch - g0);
      std::vector<Arena> arenas;
      arenas.reserve(g);
      std::vector<SpecRun<T, Arena>> runs(g);
      for (int s = 0; s < g; ++s) arenas.emplace_back(ws + (size_t)s * per_tensor_bytes, per_tensor_bytes);
      for (int s = 0; s < g && rc == TNB_OK; ++s)
        rc = spec_begin<T, Arena>(runs[s], arenas[s], false, data[g0 + s], d, eps, bflags, cores[g0 + s], nullptr, streams[s]);
      // Enqueued step by step: all Gram kernels of a step, then the eigen stages of all tensors interleaved stage by
      // stage, then every tensor's rank rule + projection.  The resident filter kernels are chained across the streams
      // (cheb_filter.cuh), so this order keeps tensor A's Rayleigh-Ritz step in flight while tensor B's filter runs; it
      // measured faster than enqueuing each tensor's whole eigen chain at once or a diagonal wavefront over the steps
      // (profiles/r02_batch_schedule.md).
      for (int mu = N - 1, t = 0; mu >= 1 && rc == TNB_OK; --mu, ++t) {
        for (int s = 0; s < g && rc == TNB_OK; ++s) rc = spec_phase1<T, Arena>(runs[s], false, d, mu, t, false);
        for (int s = 0; s < g && rc == TNB_OK; ++s) rc = spec_phase2a<T, Arena>(runs[s], false);
        for (int stage = 0; stage <= CD_MAX_STAGES && rc == TNB_OK; ++stage)
          for (int s = 0; s < g && rc == TNB_OK; ++s) rc = spec_phase2s<T, Arena>(runs[s], false, stage);
        for (int s = 0; s < g && rc == TNB_OK; ++s) rc = spec_phase2b<T, Arena>(runs[s], false, d, rmax, mu, t, false);
      }
      for (int s = 0; s < g && rc == TNB_OK; ++s) rc = spec_end<T, Arena>(runs[s], d, hbs + g0 + s);
    }
    return rc;
  };
  auto accept = [&](int i, const SpecHostBack& hb) {
    SweepInfo info;
    spec_accept(hb, d, ranks(i), &info);
    if (norms_host) norms_host[i] = info.norm;
  };
  // exact Gram matrices when the TF32 one was rejected (flag bit 0)
  auto repeat = [&](Arena& ar, int i, int spec_flags) {
    SweepInfo info;
    TNB_TRY((ttsvd_sync_impl<T, Arena>(ar, false, data[i], d, rmax, eps, flags & ~TNB_FLAG_PROFILE, cores[i], ranks(i), &info,
                                       st, (spec_flags & 1) != 0)));
    if (norms_host) norms_host[i] = info.norm;
    return TNB_OK;
  };
  const bool spec = batch > 0 && spec_eligible<T>(d, rmax, eps, flags, tc_allowed(flags, false));
  return spec_batch(workspace, per_tensor_bytes, inflight, batch, spec, spec_host, st, one, enqueue, accept, repeat);
}

}  // namespace tnb

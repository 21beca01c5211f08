// TT rounding of an existing tensor train, the two-factor split, and the reconstruction-error check.
#pragma once
#include "sweep.cuh"

namespace tnb {

// rank = #{ j : w_j > tau * w_0 } (at least 1): numerical rank of a Gram matrix for the
// orthogonalisation sweep (the reference's QR keeps min(rows, cols) columns; directions whose
// energy is below the fp64 noise floor of the Gram matrix are exactly the ones QR would have
// produced from rank deficiency).
__global__ void rank_thresh_kernel(const double* __restrict__ w, int L, double tau, int cap, SweepScalars* sc) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double w0 = w[0] > 0.0 ? w[0] : 0.0;
  int r = 0;
  for (int j = 0; j < L; ++j)
    if (w[j] > tau * w0 && w[j] > 0.0) ++r;
  if (r > cap) r = cap;
  if (r < 1) r = 1;
  sc->rank = r;
  sc->zero_flag = (w0 <= 0.0) ? 1 : 0;
}

struct RoundDims {
  int N;
  std::vector<int64_t> shape;
  std::vector<int64_t> rin;    // input ranks r_0..r_N
  std::vector<int64_t> ra;     // rank caps after orthogonalisation
  std::vector<int64_t> rcap;   // rank caps after truncation
  std::vector<int64_t> slot;
  int64_t capacity;
};

inline int make_round_dims(int ndim, const int64_t* shape, const int32_t* ranks_in, const int32_t* rmax, RoundDims& d) {
  if (ndim < 1 || ndim > 62) return fail(TNB_ERR_INVALID, "ndim=%d out of range", ndim);
  d.N = ndim;
  d.shape.assign(shape, shape + ndim);
  d.rin.resize(ndim + 1);
  for (int k = 0; k <= ndim; ++k) d.rin[k] = ranks_in[k];
  if (d.rin[0] != 1 || d.rin[ndim] != 1) return fail(TNB_ERR_INVALID, "boundary TT ranks must be 1");
  for (int k = 0; k <= ndim; ++k)
    if (d.rin[k] < 1) return fail(TNB_ERR_INVALID, "rank[%d] < 1", k);
  // after the left-to-right orthogonalisation: ra[k+1] = min(ra[k]*I_k, rin[k+1])
  d.ra.assign(ndim + 1, 1);
  for (int k = 0; k < ndim - 1; ++k) d.ra[k + 1] = std::min<int64_t>(d.ra[k] * shape[k], d.rin[k + 1]);
  d.rcap.assign(ndim + 1, 1);
  for (int mu = ndim - 1; mu >= 1; --mu) {
    int64_t c = std::min<int64_t>(d.ra[mu], shape[mu] * d.rcap[mu + 1]);
    if (rmax && rmax[mu - 1] > 0 && rmax[mu - 1] < c) c = rmax[mu - 1];
    d.rcap[mu] = c;
  }
  d.slot.assign(ndim, 0);
  int64_t off = 0;
  for (int k = 0; k < ndim; ++k) {
    d.slot[k] = off;
    // a core is first written at its orthogonalised size, then (k>=1) at its truncated size
    off += d.ra[k] * shape[k] * std::max<int64_t>(d.ra[k + 1], d.rcap[k + 1]);
    off = (off + 63) / 64 * 64;
  }
  d.capacity = off;
  return TNB_OK;
}

// Work buffers of both sweeps: `cur` / `nxt` hold the core being orthogonalised (R absorbed) and the next one; Q[k] is
// core k orthogonalised (phase A output), r_a[k] x I_k x r_a[k+1].
template <typename T, class ArenaT>
inline void round_carve(ArenaT& ar, const RoundDims& d, T** cur, T** nxt, std::vector<T*>& Q) {
  size_t maxcore = 0;
  for (int k = 0; k < d.N; ++k) maxcore = std::max<size_t>(maxcore, (size_t)d.ra[k] * d.shape[k] * d.rin[k + 1]);
  *cur = ar.template take<T>(maxcore);
  *nxt = ar.template take<T>(maxcore);
  Q.assign(d.N, nullptr);
  for (int k = 0; k < d.N; ++k) Q[k] = ar.template take<T>((size_t)d.ra[k] * d.shape[k] * std::max<int64_t>(d.ra[k + 1], 1));
}

// The two products that follow the orthogonalisation of A = core k (rowsA x cols) into fac (cols x q) and
// Rf (q x cols, A = (A fac) Rf): Q_k = A fac (rowsA x q), and next = Rf core_{k+1} (q x ncols) carries R on.
template <typename T>
inline int orth_products(const T* A, int64_t rowsA, int64_t cols, const T* fac, const T* Rf, int64_t q, const T* core_next,
                         int64_t ncols, T* Qk, T* next, cudaStream_t st) {
  TNB_TRY((gemm_direct<T, T, T, T>(rowsA, q, cols, A, cols, true, fac, q, false, Qk, q, (T)1, nullptr, 0, (T)0, nullptr, 0,
                                   (T)0, st)));
  return gemm_direct<T, T, T, T>(q, ncols, cols, Rf, cols, true, core_next, ncols, false, next, ncols, (T)1, nullptr, 0, (T)0,
                                 nullptr, 0, (T)0, st);
}

// Phase A + phase B of Tensor.round_tt (tensor.py:2008-2083) on device-resident cores.
template <typename T, class ArenaT>
inline int tt_round_impl(ArenaT& ar, bool dry, const T* const* cores_in, const RoundDims& d, const int32_t* rmax,
                         double eps, uint32_t flags, T* cores_out, int32_t* ranks_host, cudaStream_t st) {
  const int N = d.N;
  // TT cores are small: the generic fp64-accumulating kernels are used throughout
  StepCtx cx(ar, N, eps, flags, false, nullptr, st, false);
  if (!dry) {
    cx.h_sc = static_cast<int*>(pinned_scratch(sizeof(SweepScalars)));
    if (!cx.h_sc) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
    ranks_host[0] = 1;
    ranks_host[N] = 1;
  }
  if (N == 1) {
    if (!dry) {
      TNB_CUDA(cudaMemcpyAsync(cores_out + d.slot[0], cores_in[0], sizeof(T) * d.shape[0], cudaMemcpyDeviceToDevice, st));
      TNB_CUDA(cudaStreamSynchronize(st));
    }
    return TNB_OK;
  }
  T *cur, *nxt;
  std::vector<T*> Q;
  round_carve<T>(ar, d, &cur, &nxt, Q);
  std::vector<int64_t> r(N + 1, 1);        // actual ranks after phase A
  size_t peak = ar.off;

  // ---------------- phase A: left-to-right orthogonalisation (tensor.py:1800-1833) ----------------
  if (!dry) {
    TNB_CUDA(cudaMemcpyAsync(cur, cores_in[0], sizeof(T) * (size_t)d.shape[0] * d.rin[1], cudaMemcpyDeviceToDevice, st));
  }
  for (int k = 0; k < N - 1; ++k) {
    const size_t mark = ar.off;
    const int64_t rowsA = (dry ? d.ra[k] : r[k]) * d.shape[k];
    const int64_t cols = d.rin[k + 1];
    if (cols > JACOBI_MAX_N)
      return fail(TNB_ERR_UNSUPPORTED, "tt_round: input TT rank %lld exceeds the direct eigensolver limit %d",
                  (long long)cols, JACOBI_MAX_N);
    GemmPlan pl = plan_gemm(cols, cols, rowsA, true);
    double* partial = ar.template take<double>(pl.partial_elems);
    double* G = ar.template take<double>((size_t)cols * cols);
    double* w = ar.template take<double>(cols);
    double* V = ar.template take<double>((size_t)cols * cols);
    double* js = ar.template take<double>(jacobi_scratch_doubles((int)cols));
    int* jinfo = ar.template take<int>(4);
    T* fac = ar.template take<T>((size_t)cols * cols);   // V_q / sqrt(lambda)  (cols x q)
    T* Rf = ar.template take<T>((size_t)cols * cols);    // sqrt(lambda) V_q^T   (q x cols)
    if (!dry) {
      if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tt_round: workspace too small (need > %zu bytes)", ar.off);
      // G = A^T A with A = cur viewed (rowsA x cols)
      TNB_TRY((gemm_splitk<T, T, double, double, float>(pl, cols, cols, rowsA, cur, cols, false, cur, cols, false, partial,
                                                        G, cols, 1.0, nullptr, 0, 0.0, nullptr, 0, 0.0, true,
                                                        (float*)nullptr, 0, st)));
      // fast path: Cholesky-QR in fp64 (A = Q R with R = L^T from G = L L^T); a breakdown pivot (rank-deficient
      // or short core) raises the flag and the eigen-decomposition path below takes over for this core
      bool chol_ok = false;
      if (rowsA >= cols) {
        TNB_CUDA(cudaMemsetAsync(jinfo, 0, 4 * sizeof(int), st));
        TNB_TRY(chol_orth<T>(G, (int)cols, js, fac, jinfo + 1, Rf, st));
        TNB_CUDA(cudaMemcpyAsync(cx.h_sc, jinfo, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
        TNB_CUDA(cudaStreamSynchronize(st));
        chol_ok = (cx.h_sc[1] == 0);
      }
      int64_t q = cols;
      if (!chol_ok) {
        TNB_TRY(jacobi2_eigh(G, (int)cols, (int)cols, w, V, js, jinfo, st));
        const int64_t cap = std::min<int64_t>(rowsA, cols);
        rank_thresh_kernel<<<1, 32, 0, st>>>(w, (int)cols, 64.0 * 2.220446049250313e-16, (int)cap, cx.sc);
        TNB_LAUNCH_CHECK();
        TNB_CUDA(cudaMemcpyAsync(cx.h_sc, cx.sc, sizeof(SweepScalars), cudaMemcpyDeviceToHost, st));
        TNB_CUDA(cudaStreamSynchronize(st));
        q = reinterpret_cast<const SweepScalars*>(cx.h_sc)->rank;
        // fac = V_q lambda^-1/2 (cols x q);  Rf = lambda^1/2 V_q^T (q x cols)
        scale_extract_kernel<T><<<grid_for(cols * q), 256, 0, st>>>(V, (int)cols, (int)cols, (int)q, w, fac, 1, 0);
        TNB_LAUNCH_CHECK();
        scale_extract_kernel<T><<<grid_for(cols * q), 256, 0, st>>>(V, (int)cols, (int)cols, (int)q, w, Rf, 2, 1);
        TNB_LAUNCH_CHECK();
      }
      r[k + 1] = q;
      TNB_TRY(orth_products<T>(cur, rowsA, cols, fac, Rf, q, cores_in[k + 1], d.shape[k + 1] * d.rin[k + 2], Q[k], nxt, st));
      std::swap(cur, nxt);
    }
    if (ar.off > peak) peak = ar.off;
    ar.off = mark;
  }

  // ---------------- phase B: right-to-left truncation (tensor.py:2053-2083) ----------------
  // cur = last core (r[N-1] x I_{N-1} x 1), carries the whole norm.
  const T* M = cur;
  int64_t r_next = 1;
  T* left = nxt;  // rows x rank factor to absorb into the previous core
  for (int mu = N - 1, t = 0; mu >= 1; --mu, ++t) {
    const size_t mark = ar.off;
    const int64_t rows = dry ? d.ra[mu] : r[mu];
    const int64_t n = d.shape[mu] * (dry ? d.rcap[mu + 1] : r_next);
    const bool have_rmax = rmax && rmax[mu - 1] > 0;
    int64_t rank = d.rcap[mu];
    TNB_TRY((truncate_step<T>(ar, dry, cx, M, rows, n, d.rcap[mu], have_rmax, have_rmax ? rmax[mu - 1] : 0, t == 0,
                              dry ? nullptr : cores_out + d.slot[mu], left, &rank)));
    if (!dry) {
      ranks_host[mu] = (int32_t)rank;
      // cores[mu-1] <- cores[mu-1] * left     (tensor.py:2081-2083).  The step's input M (= cur) is dead
      // by now and the product only reads Q[mu-1] and `left`, so `cur` is reused for the result.
      const int64_t rowsP = r[mu - 1] * d.shape[mu - 1];
      T* dst = (mu - 1 == 0) ? cores_out + d.slot[0] : cur;
      TNB_TRY((gemm_direct<T, T, T, T>(rowsP, rank, rows, Q[mu - 1], rows, true, left, rank, false, dst, rank, (T)1,
                                       nullptr, 0, (T)0, nullptr, 0, (T)0, st)));
      M = dst;
      r_next = rank;
    }
    if (ar.off > peak) peak = ar.off;
    ar.off = mark;
  }
  if (dry) ar.off = peak;
  if (!dry) TNB_CUDA(cudaStreamSynchronize(st));
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// Speculative TT rounding: both sweeps of Tensor.round_tt enqueued without a host round trip.
//   phase A assumes every left unfolding is safely full-rank, i.e. the Cholesky-QR succeeds and keeps all rin[k+1]
//   columns (the flag of chol_orth_kernel says otherwise); phase B assumes every rank rule returns its cap (rank caps
//   on every bond, inactive eps budget) — spec_step_* of sweep.cuh.  ONE synchronisation at the end; a raised flag
//   sends the tensor to the host-driven tt_round_impl.  With no host in the loop a batch of TT tensors is simply
//   enqueued on several streams (tnb_tt_round_batch): the one-CTA Cholesky / Jacobi kernels of different tensors then
//   run side by side on different SMs — the batched-throughput form of BASELINE.json config 3.
// ---------------------------------------------------------------------------------------------
__global__ void or_flag_kernel(const int* src, int* flags, int bit) {
  if (threadIdx.x == 0 && blockIdx.x == 0 && *src) atomicOr(flags, bit);
}

// Largest input rank the speculative phase A takes: the Cholesky factors L, L^-1 then stay in shared memory.
constexpr int64_t ROUND_SPEC_MAX_RIN = 104;

// A rank cap on every bond and input ranks the speculative phase A takes: the sizing pass sizes the speculative path.
inline bool tt_round_spec_sizable(const RoundDims& d, const int32_t* rmax) {
  if (!caps_on_every_bond(rmax, d.N)) return false;
  for (int k = 0; k < d.N - 1; ++k)
    if (d.rin[k + 1] > ROUND_SPEC_MAX_RIN) return false;
  return true;
}

template <typename T>
inline bool tt_round_spec_eligible(const RoundDims& d, const int32_t* rmax, double eps, uint32_t flags) {
  if (!caps_decide(rmax, d.N, eps, flags) || !tt_round_spec_sizable(d, rmax)) return false;
  for (int k = 0; k < d.N - 1; ++k)
    if (d.ra[k + 1] != d.rin[k + 1] || d.ra[k] * d.shape[k] < d.rin[k + 1]) return false;  // Cholesky-QR keeps every column
  for (int mu = d.N - 1; mu >= 1; --mu)
    if (!spec_step_ok<T>(d.ra[mu], d.shape[mu] * d.rcap[mu + 1], d.rcap[mu], false)) return false;
  return true;
}

template <typename T, class ArenaT>
inline int tt_round_spec_enqueue(ArenaT& ar, bool dry, const T* const* cores_in, const RoundDims& d, const int32_t* rmax,
                                 double eps, uint32_t flags, T* cores_out, SpecHostBack* hb, cudaStream_t st) {
  const int N = d.N;
  StepCtx cx(ar, N, eps, flags, false, nullptr, st, true);
  int* d_chol = ar.template take<int>(4);
  T *cur, *nxt;
  std::vector<T*> Q;
  round_carve<T>(ar, d, &cur, &nxt, Q);
  size_t peak = ar.off;
  if (!dry) {
    TNB_CUDA(cudaMemsetAsync(cx.d_flags, 0, 4 * sizeof(int), st));
    TNB_CUDA(cudaMemsetAsync(d_chol, 0, 4 * sizeof(int), st));
    TNB_CUDA(cudaMemcpyAsync(cur, cores_in[0], sizeof(T) * (size_t)d.shape[0] * d.rin[1], cudaMemcpyDeviceToDevice, st));
  }
  // ---------------- phase A ----------------
  for (int k = 0; k < N - 1; ++k) {
    const size_t mark = ar.off;
    const int64_t rowsA = d.ra[k] * d.shape[k];
    const int64_t cols = d.rin[k + 1];
    GemmPlan pl = plan_gemm(cols, cols, rowsA, true);
    double* partial = ar.template take<double>(pl.partial_elems);
    double* G = ar.template take<double>((size_t)cols * cols);
    double* js = ar.template take<double>((size_t)2 * cols * (cols | 1));
    T* fac = ar.template take<T>((size_t)cols * cols);
    T* Rf = ar.template take<T>((size_t)cols * cols);
    if (ar.off > peak) peak = ar.off;
    if (!dry) {
      if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tt_round: workspace too small (need > %zu bytes)", ar.off);
      TNB_TRY((gemm_splitk<T, T, double, double, float>(pl, cols, cols, rowsA, cur, cols, false, cur, cols, false, partial, G,
                                                        cols, 1.0, nullptr, 0, 0.0, nullptr, 0, 0.0, true, (float*)nullptr, 0,
                                                        st)));
      TNB_TRY(chol_orth<T>(G, (int)cols, js, fac, d_chol, Rf, st));  // L, L^-1 in shared memory: cols <= ROUND_SPEC_MAX_RIN
      TNB_TRY(orth_products<T>(cur, rowsA, cols, fac, Rf, cols, cores_in[k + 1], d.shape[k + 1] * d.rin[k + 2], Q[k], nxt, st));
      std::swap(cur, nxt);
    }
    ar.off = mark;
  }
  if (!dry) {
    or_flag_kernel<<<1, 32, 0, st>>>(d_chol, cx.d_flags, 64);
    TNB_LAUNCH_CHECK();
  }
  // ---------------- phase B ----------------
  const T* M = cur;
  T* left = nxt;
  SpecStep<T> step;
  for (int mu = N - 1, t = 0; mu >= 1; --mu, ++t) {
    const size_t mark = ar.off;
    const int64_t rows = d.ra[mu];
    const int64_t n = d.shape[mu] * d.rcap[mu + 1];
    spec_step_carve<T>(ar, cx, rows, n, d.rcap[mu], step);
    if (ar.off > peak) peak = ar.off;
    if (!dry) {
      if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tt_round: workspace too small (need > %zu bytes)", ar.off);
      TNB_TRY(spec_step_gram<T>(cx, M, rows, n, t == 0, step, false));
      TNB_TRY(spec_step_eig_begin<T>(cx, step));
      for (int stage = 0; stage <= CD_MAX_STAGES; ++stage) TNB_TRY(spec_step_eig_stage<T>(step, stage));
      TNB_TRY(spec_step_rest<T>(cx, M, rows, n, rmax[mu - 1], cores_out + d.slot[mu], left, mu, step, false));
      const int64_t rank = d.rcap[mu];
      const int64_t rowsP = d.ra[mu - 1] * d.shape[mu - 1];
      T* dst = (mu - 1 == 0) ? cores_out + d.slot[0] : cur;
      TNB_TRY((gemm_direct<T, T, T, T>(rowsP, rank, rows, Q[mu - 1], rows, true, left, rank, false, dst, rank, (T)1, nullptr,
                                       0, (T)0, nullptr, 0, (T)0, st)));
      M = dst;
    }
    ar.off = mark;
  }
  if (dry) {
    ar.off = peak;
    return TNB_OK;
  }
  TNB_CUDA(cudaMemcpyAsync(&hb->sc, cx.sc, sizeof(SweepScalars), cudaMemcpyDeviceToHost, st));
  TNB_CUDA(cudaMemcpyAsync(hb->flags, cx.d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
  return TNB_OK;
}

// The speculative rounding never returns TNB_ERR_NOCONV: its steps are eligible only for the direct eigensolver
// (allow_tc is false), whose solve is enqueued and cannot report non-convergence.
template <typename T, class ArenaT>
inline int tt_round_any(ArenaT& ar, bool dry, const T* const* cores_in, const RoundDims& d, const int32_t* rmax, double eps,
                        uint32_t flags, T* cores_out, int32_t* ranks_host, cudaStream_t st, SweepInfo* info = nullptr) {
  const bool try_spec = dry ? tt_round_spec_sizable(d, rmax) : tt_round_spec_eligible<T>(d, rmax, eps, flags);
  return speculate_or_fall_back(
      ar, dry, try_spec, info,
      [&](bool dr, int* spec_flags) {
        if (dr) return tt_round_spec_enqueue<T>(ar, true, cores_in, d, rmax, eps, flags, cores_out, nullptr, st);
        SpecHostBack* hb = static_cast<SpecHostBack*>(pinned_scratch(sizeof(SpecHostBack)));
        if (!hb) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
        const int rc = tt_round_spec_enqueue<T>(ar, false, cores_in, d, rmax, eps, flags, cores_out, hb, st);
        TNB_CUDA(cudaStreamSynchronize(st));
        if (rc != TNB_OK) return rc;
        *spec_flags = hb->flags[0];
        if (*spec_flags == 0) ranks_from_caps(d.rcap, ranks_host);
        return TNB_OK;
      },
      [&](bool dr, int) { return tt_round_impl<T>(ar, dr, cores_in, d, rmax, eps, flags, cores_out, ranks_host, st); });
}

// A batch of TT tensors with one rank profile: every tensor's two sweeps on its own internal stream, one synchronisation.
template <typename T>
inline int tt_round_batch_impl(void* workspace, size_t per_tensor_bytes, int inflight, const T* const* cores_in /* [B][N] */,
                               int batch, const RoundDims& d, const int32_t* rmax, double eps, uint32_t flags,
                               T* const* cores_out, int32_t* ranks_host, int32_t* spec_host, cudaStream_t st) {
  const int N = d.N;
  char* ws = static_cast<char*>(workspace);
  auto in = [&](int i) { return cores_in + (size_t)i * N; };
  auto ranks = [&](int i) { return ranks_host + (size_t)i * (N + 1); };
  auto one = [&](Arena& ar, int i, SweepInfo* info) {
    return tt_round_any<T, Arena>(ar, false, in(i), d, rmax, eps, flags, cores_out[i], ranks(i), st, info);
  };
  auto enqueue = [&](cudaStream_t* streams, int inflight, SpecHostBack* hbs) {
    int rc = TNB_OK;
    for (int i = 0; i < batch && rc == TNB_OK; ++i) {
      const int s = i % inflight;  // tensor i + inflight reuses workspace slice s on the same stream: ordered
      Arena ar(ws + (size_t)s * per_tensor_bytes, per_tensor_bytes);
      rc = tt_round_spec_enqueue<T>(ar, false, in(i), d, rmax, eps, flags, cores_out[i], hbs + i, streams[s]);
    }
    return rc;
  };
  auto accept = [&](int i, const SpecHostBack&) { ranks_from_caps(d.rcap, ranks(i)); };
  auto repeat = [&](Arena& ar, int i, int) {
    return tt_round_impl<T, Arena>(ar, false, in(i), d, rmax, eps, flags, cores_out[i], ranks(i), st);
  };
  const bool spec = tt_round_spec_eligible<T>(d, rmax, eps, flags);
  return spec_batch(workspace, per_tensor_bytes, inflight, batch, spec, spec_host, st, one, enqueue, accept, repeat);
}

// ---------------------------------------------------------------------------------------------
// sum_k alpha_k T_k in TT format: block cores (tensor.py:445-520, Tensor.__add__ for TT operands — first core: blocks side
// by side, last core: blocks stacked, interior cores: block diagonal), assembled by ONE kernel per core straight into the
// buffer the rounding sweep reads, so that the `tn.round(a + b)` of tools.reduce (tools.py:460-512) is a single library call
// with no intermediate tensors on the host side.
// ---------------------------------------------------------------------------------------------
template <typename T>
struct SumSrc {
  const T* core[16];
  int r0[16], r1[16];
  int o0[16], o1[16];  // block offsets along the two rank axes
  double alpha[16];
  int K;
};
template <typename T>
__global__ void tt_sum_assemble_kernel(const SumSrc<T> src, int I, int R0, int R1, int first, int last, T* __restrict__ out) {
  const int64_t total = (int64_t)R0 * I * R1;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % R1);
    const int i = (int)((idx / R1) % I);
    const int a = (int)(idx / ((int64_t)R1 * I));
    T v = (T)0;
    if (first && last) {  // a 1-mode "tensor": plain weighted sum of vectors
      for (int k = 0; k < src.K; ++k) v += (T)(src.alpha[k] * (double)src.core[k][i]);
    } else {
      for (int k = 0; k < src.K; ++k) {
        const int aa = first ? a : a - src.o0[k];  // first core: one row, the blocks sit side by side
        const int cc = last ? c : c - src.o1[k];   // last core: one column, the blocks are stacked
        if (aa >= 0 && aa < src.r0[k] && cc >= 0 && cc < src.r1[k]) {
          const T x = src.core[k][((size_t)aa * I + i) * src.r1[k] + cc];
          v = first ? (T)(src.alpha[k] * (double)x) : x;  // the scalar goes into the first core (tensor.py: t * scalar)
          break;                                           // blocks do not overlap
        }
      }
    }
    out[idx] = v;
  }
}

// Elementwise (Hadamard) product of two TT tensors: Kronecker cores out[(a1 a2), i, (b1 b2)] = A[a1, i, b1] B[a2, i, b2]
// (tensor.py:560-640, Tensor.__mul__ for TT operands).
template <typename T>
__global__ void tt_hadamard_core_kernel(const T* __restrict__ A, const T* __restrict__ Bc, int ra0, int ra1, int rb0, int rb1,
                                        int I, T* __restrict__ out) {
  const int R1 = ra1 * rb1;
  const int64_t total = (int64_t)ra0 * rb0 * I * R1;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % R1);
    const int i = (int)((idx / R1) % I);
    const int a = (int)(idx / ((int64_t)R1 * I));
    const int a1 = a / rb0, a2 = a - a1 * rb0, b1 = c / rb1, b2 = c - b1 * rb1;
    out[idx] = A[((size_t)a1 * I + i) * ra1 + b1] * Bc[((size_t)a2 * I + i) * rb1 + b2];
  }
}

struct SumDims {
  int N = 0, K = 0;
  std::vector<int64_t> shape;
  std::vector<int32_t> rsum;               // N + 1 summed ranks
  std::vector<std::vector<int32_t>> rin;   // K x (N + 1)
  std::vector<int64_t> slot;               // element offset of assembled core n
  int64_t capacity = 0;
};
inline int make_sum_dims(int K, int ndim, const int64_t* shape, const int32_t* ranks_in, SumDims& d) {
  if (K < 1 || K > 16) return fail(TNB_ERR_INVALID, "tt_sum: between 1 and 16 operands per call, got %d", K);
  if (ndim < 1 || ndim > 62) return fail(TNB_ERR_INVALID, "ndim=%d out of range", ndim);
  d.N = ndim;
  d.K = K;
  d.shape.assign(shape, shape + ndim);
  d.rin.assign(K, std::vector<int32_t>(ndim + 1));
  d.rsum.assign(ndim + 1, 0);
  for (int k = 0; k < K; ++k)
    for (int n = 0; n <= ndim; ++n) {
      d.rin[k][n] = ranks_in[(size_t)k * (ndim + 1) + n];
      if (d.rin[k][n] < 1) return fail(TNB_ERR_INVALID, "tt_sum: rank < 1");
      d.rsum[n] += d.rin[k][n];
    }
  for (int k = 0; k < K; ++k)
    if (d.rin[k][0] != 1 || d.rin[k][ndim] != 1) return fail(TNB_ERR_INVALID, "boundary TT ranks must be 1");
  d.rsum[0] = 1;
  d.rsum[ndim] = 1;
  d.slot.assign(ndim, 0);
  int64_t off = 0;
  for (int n = 0; n < ndim; ++n) {
    d.slot[n] = off;
    off += (int64_t)d.rsum[n] * shape[n] * d.rsum[n + 1];
    off = (off + 63) / 64 * 64;
  }
  d.capacity = off;
  return TNB_OK;
}

template <typename T>
inline int tt_sum_assemble(const T* const* cores_in /* [K][N] */, const double* alpha, const SumDims& d, T* out, cudaStream_t st) {
  for (int n = 0; n < d.N; ++n) {
    SumSrc<T> src;
    src.K = d.K;
    int o0 = 0, o1 = 0;
    for (int k = 0; k < d.K; ++k) {
      src.core[k] = cores_in[(size_t)k * d.N + n];
      src.r0[k] = d.rin[k][n];
      src.r1[k] = d.rin[k][n + 1];
      src.o0[k] = o0;
      src.o1[k] = o1;
      src.alpha[k] = alpha ? alpha[k] : 1.0;
      o0 += d.rin[k][n];
      o1 += d.rin[k][n + 1];
    }
    const int64_t total = (int64_t)d.rsum[n] * d.shape[n] * d.rsum[n + 1];
    tt_sum_assemble_kernel<T><<<grid_for(total), 256, 0, st>>>(src, (int)d.shape[n], d.rsum[n], d.rsum[n + 1], n == 0 ? 1 : 0,
                                                                n == d.N - 1 ? 1 : 0, out + d.slot[n]);
    TNB_LAUNCH_CHECK();
  }
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// tn.truncated_svd (round.py:52-187), non-batch
// ---------------------------------------------------------------------------------------------
template <typename T, class ArenaT>
inline int truncated_svd_impl(ArenaT& ar, bool dry, const T* M, int64_t m, int64_t n, double delta, double eps,
                              int32_t rmax, int left_ortho_flags, T* left, T* right, int32_t* rank_host,
                              cudaStream_t st) {
  typedef T TBk;
  const int left_ortho = left_ortho_flags & 1;
  const int batch_mode = (left_ortho_flags & 2) ? 1 : 0;  // round.py:149-150: rank = min(rmax, len(S)), no eps, no zero branch
  const bool use_left = m <= n;  // round.py:102-107
  const int64_t L = use_left ? m : n;
  const int64_t K = use_left ? n : m;
  SweepScalars* sc = ar.template take<SweepScalars>(1);
  GemmPlan pl = plan_gemm(L, L, K, true);
  double* partial = ar.template take<double>(pl.partial_elems);
  double* G = ar.template take<double>((size_t)L * L);
  EigWork<TBk> ew;
  const bool have_rmax = rmax > 0;
  const int64_t kcap = have_rmax ? std::min<int64_t>(rmax, L) : L;
  TNB_TRY(eig_carve<TBk>(ar, L, kcap, have_rmax, ew));
  float* Gf = (ew.chfsi && std::is_same<TBk, float>::value) ? reinterpret_cast<float*>(ew.Gb) : nullptr;
  // the factor scratch holds what the eigen stage can return: all L vectors from the direct solver, at most ew.k
  // from the subspace solver (an eps/delta-only request and the sizing pass then carve the same amount)
  const int64_t fcap = ew.chfsi ? std::min<int64_t>(L, ew.k) : L;
  T* fac = ar.template take<T>((size_t)L * (size_t)fcap);
  if (dry) return TNB_OK;
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "truncated_svd: workspace too small (need > %zu bytes)", ar.off);
  int* h_sc = static_cast<int*>(pinned_scratch(sizeof(SweepScalars)));
  if (!h_sc) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
  if (use_left)
    TNB_TRY((gemm_splitk<T, T, double, double, float>(pl, m, m, n, M, n, true, M, n, true, partial, G, m, 1.0, nullptr, 0,
                                                      0.0, nullptr, 0, 0.0, true, Gf, m, st)));
  else
    TNB_TRY((gemm_splitk<T, T, double, double, float>(pl, n, n, m, M, n, false, M, n, false, partial, G, n, 1.0, nullptr,
                                                      0, 0.0, nullptr, 0, 0.0, true, Gf, n, st)));
  trace_kernel<<<1, 256, 0, st>>>(G, (int)L, (int)L, sc, 0, 0.0);
  TNB_LAUNCH_CHECK();
  set_delta2_kernel<<<1, 32, 0, st>>>(sc, delta, eps);
  TNB_LAUNCH_CHECK();
  TNB_TRY(eig_solve_and_rank<TBk>(G, reinterpret_cast<const TBk*>(Gf), L, ew, sc, h_sc, rmax, batch_mode, nullptr, nullptr,
                                  st, false, false));
  const SweepScalars* hs = reinterpret_cast<const SweepScalars*>(h_sc);
  int64_t r = std::min<int64_t>(hs->rank, std::min<int64_t>(kcap, fcap));
  if (hs->zero_flag && !batch_mode) {  // round.py:137-145
    *rank_host = 1;
    fill_kernel<T><<<grid_for(m), 256, 0, st>>>(left, m, (T)0);
    TNB_LAUNCH_CHECK();
    fill_kernel<T><<<grid_for(n), 256, 0, st>>>(right, n, (T)0);
    TNB_LAUNCH_CHECK();
    TNB_CUDA(cudaStreamSynchronize(st));
    return TNB_OK;
  }
  // batch mode: a zero sample keeps rank = min(rmax, len(S)) (its factors come out as zeros); the sign tells the
  // caller, which returns rank-1 zeros only when EVERY sample of the batch is zero (round.py:138-142)
  *rank_host = (batch_mode && hs->zero_flag) ? -(int32_t)r : (int32_t)r;
  if (use_left) {
    if (left_ortho) {  // left = U_r ; right = U_r^T M
      scale_extract_kernel<T><<<grid_for(m * r), 256, 0, st>>>(ew.V, ew.ldv, (int)m, (int)r, ew.w, left, 0, 0);
      TNB_LAUNCH_CHECK();
      TNB_TRY((gemm_direct<T, T, T, T>(r, n, m, left, r, false, M, n, false, right, n, (T)1, nullptr, 0, (T)0, nullptr, 0,
                                       (T)0, st)));
    } else {  // right = diag(1/s) U_r^T M ; left = U_r diag(s)     (round.py:170-172)
      scale_extract_kernel<T><<<grid_for(m * r), 256, 0, st>>>(ew.V, ew.ldv, (int)m, (int)r, ew.w, fac, 1, 0);
      TNB_LAUNCH_CHECK();
      TNB_TRY((gemm_direct<T, T, T, T>(r, n, m, fac, r, false, M, n, false, right, n, (T)1, nullptr, 0, (T)0, nullptr, 0,
                                       (T)0, st)));
      scale_extract_kernel<T><<<grid_for(m * r), 256, 0, st>>>(ew.V, ew.ldv, (int)m, (int)r, ew.w, left, 2, 0);
      TNB_LAUNCH_CHECK();
    }
  } else {
    if (left_ortho) {  // left = M (V_r / s) ; right = diag(s) V_r^T     (round.py:175-179)
      scale_extract_kernel<T><<<grid_for(n * r), 256, 0, st>>>(ew.V, ew.ldv, (int)n, (int)r, ew.w, fac, 1, 0);
      TNB_LAUNCH_CHECK();
      TNB_TRY((gemm_direct<T, T, T, T>(m, r, n, M, n, true, fac, r, false, left, r, (T)1, nullptr, 0, (T)0, nullptr, 0,
                                       (T)0, st)));
      scale_extract_kernel<T><<<grid_for(n * r), 256, 0, st>>>(ew.V, ew.ldv, (int)n, (int)r, ew.w, right, 2, 1);
      TNB_LAUNCH_CHECK();
    } else {  // left = M V_r ; right = V_r^T     (round.py:180-183)
      scale_extract_kernel<T><<<grid_for(n * r), 256, 0, st>>>(ew.V, ew.ldv, (int)n, (int)r, ew.w, fac, 0, 0);
      TNB_LAUNCH_CHECK();
      TNB_TRY((gemm_direct<T, T, T, T>(m, r, n, M, n, true, fac, r, false, left, r, (T)1, nullptr, 0, (T)0, nullptr, 0,
                                       (T)0, st)));
      scale_extract_kernel<T><<<grid_for(n * r), 256, 0, st>>>(ew.V, ew.ldv, (int)n, (int)r, ew.w, right, 0, 1);
      TNB_LAUNCH_CHECK();
    }
  }
  TNB_CUDA(cudaStreamSynchronize(st));
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// || T - TT(cores) ||_F / || T ||_F  with the last contraction fused with the difference and the
// two squared norms (fp64 accumulation).  Tensor.torch() tensor.py:1639-1687 + metrics.py:135-151.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) recon_diff_kernel(const T* __restrict__ F, int64_t rows, int r,
                                                         const T* __restrict__ core, int ncols,
                                                         const T* __restrict__ data, double* __restrict__ acc) {
  // each block handles a strip of rows; thread computes dot(F[row,:], core[:,col]) for its (row, col)
  __shared__ double red[32];
  double d2 = 0.0, t2 = 0.0;
  const int64_t total = rows * ncols;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = idx / ncols;
    const int col = (int)(idx % ncols);
    double s = 0.0;
    for (int k = 0; k < r; ++k) s += (double)F[row * r + k] * (double)core[(size_t)k * ncols + col];
    const double t = (double)data[idx];
    const double diff = t - (double)(T)s;  // reconstruct in the data precision, like the reference
    d2 += diff * diff;
    t2 += t * t;
  }
  d2 = block_reduce_sum(d2, red);
  t2 = block_reduce_sum(t2, red);
  if (threadIdx.x == 0) {
    atomicAdd(&acc[0], d2);
    atomicAdd(&acc[1], t2);
  }
}

template <typename T, class ArenaT>
inline int tt_relative_error_impl(ArenaT& ar, bool dry, const T* data, const T* const* cores, int N,
                                  const int64_t* shape, const int32_t* ranks, double* result_host, cudaStream_t st) {
  if (N < 2) return fail(TNB_ERR_UNSUPPORTED, "tt_relative_error: needs at least 2 modes");
  double* acc = ar.template take<double>(2);
  // F_k : (prod_{j<=k} I_j) x r_{k+1}; ping-pong buffers up to k = N-2
  size_t felems[2] = {1, 1};
  int64_t rows = 1;
  for (int k = 0; k < N - 1; ++k) {
    rows *= shape[k];
    const size_t e = (size_t)rows * ranks[k + 1];
    if (e > felems[k & 1]) felems[k & 1] = e;
  }
  T* F[2] = {ar.template take<T>(felems[0]), ar.template take<T>(felems[1])};
  if (dry) return TNB_OK;
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tt_relative_error: workspace too small (need > %zu bytes)", ar.off);
  TNB_CUDA(cudaMemsetAsync(acc, 0, 2 * sizeof(double), st));
  const T* Fc = cores[0];  // (I_0 x r_1)
  rows = shape[0];
  for (int k = 1; k < N - 1; ++k) {
    // F_k (rows*I_k x r_{k+1}) = F_{k-1} (rows x r_k) * core_k (r_k x I_k r_{k+1})
    const int64_t ncols = shape[k] * ranks[k + 1];
    TNB_TRY((gemm_direct<T, T, T, T>(rows, ncols, ranks[k], Fc, ranks[k], true, cores[k], ncols, false, F[k & 1], ncols,
                                     (T)1, nullptr, 0, (T)0, nullptr, 0, (T)0, st)));
    Fc = F[k & 1];
    rows *= shape[k];
  }
  const int ncols = (int)shape[N - 1];
  recon_diff_kernel<T><<<grid_for(rows * ncols, 256, 1184), 256, 0, st>>>(Fc, rows, ranks[N - 1], cores[N - 1], ncols,
                                                                         data, acc);
  TNB_LAUNCH_CHECK();
  double* h = static_cast<double*>(pinned_scratch(2 * sizeof(double)));
  TNB_CUDA(cudaMemcpyAsync(h, acc, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
  TNB_CUDA(cudaStreamSynchronize(st));
  *result_host = std::sqrt(h[0]) / std::sqrt(h[1]);
  return TNB_OK;
}

}  // namespace tnb

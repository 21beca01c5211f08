// Leading eigenpairs of a large PSD Gram matrix (n > JACOBI_MAX_N) without a full eigensolve:
// Chebyshev-filtered subspace iteration.  The TT-SVD step only needs the dominant r-dimensional
// invariant subspace of G = C^T C and the energy it captures (SURVEY.md §7 step 3); the stopping
// rule is therefore on captured energy sum_{i<r} theta_i, the quantity the relative error depends on.
// Algorithm validated in NumPy: tests/sweep_model.py::chfsi_topk.
//
// All heavy work is GEMM-shaped (G*X with a fused three-term epilogue, X^T X, X^T W, X*Q) and runs
// through gemm_generic.cuh; the small b x b problems go to the one-CTA Jacobi kernel.
#pragma once
#include "common.cuh"
#include "gemm_generic.cuh"
#include "gram_tc.cuh"
#include "cheb_filter.cuh"
#include "jacobi.cuh"
#include "jacobi2.cuh"
#include "small_kernels.cuh"

namespace tnb {

struct ChfsiStats {
  int fused_filters = 0;  // filters that ran as one resident kernel (cheb_filter.cuh)
  int rr_sweeps = 0;      // Jacobi sweeps summed over the Rayleigh-Ritz solves (diagnostic)
  int products = 0;  // number of G*X block products
  int outer = 0;
  int converged = 0;
};

inline int chfsi_default_block(int n, int k) {
  int b = 2 * k > k + 16 ? 2 * k : k + 16;
  if (b > JACOBI_MAX_N) b = JACOBI_MAX_N;
  if (b > n) b = n;
  return b;
}

template <typename TB>
struct ChfsiWork {
  TB *X, *Y, *Z, *W;        // n x b blocks
  TB* Tm;                   // b x b
  void* partial;            // split-K scratch, partial_bytes
  size_t partial_bytes;
  bool use_tc = false;      // filter products on the tcgen05 kernel (fp32 blocks only)
  bool shared_gpu = false;  // TNB_FLAG_CONCURRENT: other decompositions run beside this one: no resident 128-SM filter kernel
  double *S, *lam, *Q, *d;  // b*b, b, b*b, b
  double* jscratch;         // jacobi_scratch_doubles(b)
  int* jinfo;
};

template <typename TB, class ArenaT>
inline void chfsi_carve(ArenaT& ar, int n, int b, ChfsiWork<TB>& w) {
  const size_t nb = (size_t)n * b;
  w.X = ar.template take<TB>(nb);
  w.Y = ar.template take<TB>(nb);
  w.Z = ar.template take<TB>(nb);
  w.W = ar.template take<TB>(nb);
  w.Tm = ar.template take<TB>((size_t)b * b);
  // largest split-K scratch among the products used below
  GemmPlan p1 = plan_gemm(n, b, n, false);
  GemmPlan p2 = plan_gemm(b, b, n, false);
  size_t e1 = p1.partial_elems * sizeof(TB), e2 = p2.partial_elems * sizeof(double);
  w.partial_bytes = e1 > e2 ? e1 : e2;
  if (std::is_same<TB, float>::value && atb_tc_shape_ok(n, n, b)) {
    const size_t e3 = atb_tc_workspace_bytes(n, n, b);
    if (e3 > w.partial_bytes) w.partial_bytes = e3;
    if (cheb_filter_shape_ok(n, b) && cheb_filter_workspace_bytes(n, b) > w.partial_bytes)
      w.partial_bytes = cheb_filter_workspace_bytes(n, b);
  }
  w.partial = ar.template take<char>(w.partial_bytes);
  w.S = ar.template take<double>((size_t)b * b);
  w.lam = ar.template take<double>(b);
  w.Q = ar.template take<double>((size_t)b * b);
  w.d = ar.template take<double>(b);
  w.jscratch = ar.template take<double>(jacobi_scratch_doubles(b));
  w.jinfo = ar.template take<int>(4);  // [0] Jacobi sweeps, [1] Cholesky breakdown flag
}

// Y <- a * G*Yin + bc * Yin + g * Xin      (G symmetric, stored n x n in TB)
// tensorcore = true routes the product through the tcgen05 kernel (TF32 operands): used for the Chebyshev
// FILTER only, where operator accuracy merely affects the convergence rate; the Rayleigh-Ritz product stays
// fp32 FFMA so that the projected matrix, and with it the captured energy, is exact to fp32.
template <typename TB>
inline int chfsi_apply(const TB* G, int n, int b, const TB* Yin, const TB* Xin, TB* Yout, double a, double bc, double g,
                       ChfsiWork<TB>& w, cudaStream_t st, bool tensorcore = false) {
  if (tensorcore && w.use_tc && std::is_same<TB, float>::value)
    return atb_tc_f32(reinterpret_cast<const float*>(G), n, n, reinterpret_cast<const float*>(Yin), b,
                      reinterpret_cast<float*>(Yout), b, (float)a, (bc != 0.0 ? reinterpret_cast<const float*>(Yin) : nullptr),
                      b, (float)bc, (g != 0.0 ? reinterpret_cast<const float*>(Xin) : nullptr), b, (float)g, w.partial,
                      w.partial_bytes, st);
  GemmPlan pl = plan_gemm(n, b, n, false);
  return gemm_splitk<TB, TB, TB, TB, TB>(pl, n, b, n, G, n, /*a_kmaj (symmetric: either)*/ false, Yin, b, false,
                                         reinterpret_cast<TB*>(w.partial), Yout, b, (TB)a, (bc != 0.0 ? Yin : nullptr), b,
                                         (TB)bc, (g != 0.0 ? Xin : nullptr), b, (TB)g,
                                         false, (TB*)nullptr, 0, st);
}

// X <- orthonormal basis of span(X); result left in *Xio, *Xtmp is scratch.
//   use_chol = false: two SVQB passes (eigen-decomposition of the scaled Gram matrix; tolerates a
//                     numerically rank-deficient block — used while the block is still far from converged)
//   use_chol = true : one Cholesky-QR pass in fp64 (the filtered Ritz vectors are close to orthogonal after
//                     column scaling; the kernel raises w.jinfo[1] if a pivot says otherwise)
template <typename TB>
inline int chfsi_orthonormalize(int n, int b, TB** Xio, TB** Xtmp, ChfsiWork<TB>& w, cudaStream_t st,
                                bool use_chol = false) {
  if (use_chol) {
    GemmPlan pl = plan_gemm(b, b, n, false);
    TNB_TRY((gemm_splitk<TB, TB, double, double, double>(pl, b, b, n, *Xio, b, false, *Xio, b, false,
                                                         reinterpret_cast<double*>(w.partial), w.S, b, 1.0, nullptr, 0,
                                                         0.0, nullptr, 0, 0.0, false, (double*)nullptr, 0, st)));
    TNB_TRY(chol_orth<TB>(w.S, b, w.jscratch, w.Tm, w.jinfo + 1, nullptr, st));
    TNB_TRY((gemm_direct<TB, TB, TB, TB>(n, b, b, *Xio, b, true, w.Tm, b, false, *Xtmp, b, (TB)1, nullptr, 0, (TB)0,
                                         nullptr, 0, (TB)0, st)));
    TB* t = *Xio; *Xio = *Xtmp; *Xtmp = t;
    return TNB_OK;
  }
  for (int pass = 0; pass < 2; ++pass) {
    GemmPlan pl = plan_gemm(b, b, n, false);
    TNB_TRY((gemm_splitk<TB, TB, double, double, double>(pl, b, b, n, *Xio, b, false, *Xio, b, false,
                                                         reinterpret_cast<double*>(w.partial), w.S, b, 1.0, nullptr, 0,
                                                         0.0, nullptr, 0, 0.0, false, (double*)nullptr, 0, st)));
    svqb_prep_kernel<<<1, 1024, 0, st>>>(w.S, b, w.d);
    TNB_LAUNCH_CHECK();
    TNB_TRY(jacobi2_eigh(w.S, b, b, w.lam, w.Q, w.jscratch, w.jinfo, st, std::is_same<TB, float>::value));
    svqb_finish_kernel<TB><<<grid_for((int64_t)b * b), 256, 0, st>>>(w.Q, w.lam, w.d, b,
                                                                     std::is_same<TB, float>::value ? 1e-6 : 1e-13, w.Tm);
    TNB_LAUNCH_CHECK();
    TNB_TRY((gemm_direct<TB, TB, TB, TB>(n, b, b, *Xio, b, true, w.Tm, b, false, *Xtmp, b, (TB)1, nullptr, 0, (TB)0,
                                         nullptr, 0, (TB)0, st)));
    TB* t = *Xio; *Xio = *Xtmp; *Xtmp = t;
  }
  return TNB_OK;
}

// Rayleigh-Ritz on span(X): theta (descending, in w.lam) and X <- X * Q.  Uses W as scratch for G*X.
template <typename TB>
inline int chfsi_rayleigh_ritz(const TB* G, int n, int b, TB** Xio, TB** Xtmp, ChfsiWork<TB>& w, cudaStream_t st) {
  TNB_TRY(chfsi_apply<TB>(G, n, b, *Xio, nullptr, w.W, 1.0, 0.0, 0.0, w, st));
  GemmPlan pl = plan_gemm(b, b, n, false);
  TNB_TRY((gemm_splitk<TB, TB, double, double, double>(pl, b, b, n, *Xio, b, false, w.W, b, false,
                                                       reinterpret_cast<double*>(w.partial), w.S, b, 1.0, nullptr, 0,
                                                       0.0, nullptr, 0, 0.0, false, (double*)nullptr, 0, st)));
  // fp32 blocks: rotations in fp32 and a loose stop (the Ritz vectors are re-filtered anyway and stored in fp32);
  // fp64 blocks: full accuracy, so that U = M V S^-1 built from the Ritz vectors is orthonormal to working precision
  TNB_TRY(jacobi2_eigh(w.S, b, b, w.lam, w.Q, w.jscratch, w.jinfo, st, std::is_same<TB, float>::value,
                      std::is_same<TB, float>::value ? 2e-5 : 0.0));
  convert_kernel<double, TB><<<grid_for((int64_t)b * b), 256, 0, st>>>(w.Q, w.Tm, (int64_t)b * b);
  TNB_LAUNCH_CHECK();
  TNB_TRY((gemm_direct<TB, TB, TB, TB>(n, b, b, *Xio, b, true, w.Tm, b, false, *Xtmp, b, (TB)1, nullptr, 0, (TB)0,
                                       nullptr, 0, (TB)0, st)));
  TB* t = *Xio; *Xio = *Xtmp; *Xtmp = t;
  return TNB_OK;
}

// k leading eigenpairs of PSD G (n x n, type TB).  On return theta_out (b doubles, descending Ritz
// values, device) and X_out (n x b doubles, device).  tol: stop when the captured energy of the k
// leading Ritz values grows by less than tol * trace(G) between outer iterations.
template <typename TB>
inline int eig_topk_chfsi(const TB* G, int n, int k, int b, const double* d_trace, double tol, ChfsiWork<TB>& w,
                          double* theta_out, double* X_out, ChfsiStats* stats, cudaStream_t st) {
  if (b < k || b > JACOBI_MAX_N || b > n)
    return fail(TNB_ERR_UNSUPPORTED, "eig_topk: block %d invalid for k=%d n=%d (max %d)", b, k, n, JACOBI_MAX_N);
  double* h_theta = static_cast<double*>(pinned_scratch((size_t)(b + 4) * sizeof(double)));
  if (!h_theta) return fail(TNB_ERR_CUDA, "pinned scratch allocation failed");
  const int max_outer = 40, mmax = 40;
  const double spread = 1e4;
  w.use_tc = w.use_tc && std::is_same<TB, float>::value && tc_path_available() && atb_tc_shape_ok(n, n, b) &&
             (reinterpret_cast<uintptr_t>(G) & 15u) == 0;

  random_fill_kernel<TB><<<grid_for((int64_t)n * b), 256, 0, st>>>(w.X, (int64_t)n * b, 0x1234567u);
  TNB_LAUNCH_CHECK();
  TNB_CUDA(cudaMemsetAsync(w.jinfo, 0, 4 * sizeof(int), st));
  int* h_flag = reinterpret_cast<int*>(h_theta + b + 1);
  bool use_chol = true;   // Cholesky-QR; the eigen-decomposition based SVQB only after a flagged breakdown
  TB* X = w.X;
  TB* Xt = w.Z;  // scratch partner for orthonormalize / RR
  TNB_TRY(chfsi_orthonormalize<TB>(n, b, &X, &Xt, w, st, true));  // a random block is well conditioned
  TNB_TRY(chfsi_rayleigh_ritz<TB>(G, n, b, &X, &Xt, w, st));
  if (stats) stats->products += 1;
  TNB_CUDA(cudaMemcpyAsync(h_theta, w.lam, (size_t)b * sizeof(double), cudaMemcpyDeviceToHost, st));
  h_theta[b] = 0.0;
  if (d_trace) TNB_CUDA(cudaMemcpyAsync(h_theta + b, d_trace, sizeof(double), cudaMemcpyDeviceToHost, st));
  TNB_CUDA(cudaStreamSynchronize(st));
  double trace = h_theta[b];
  if (!(trace > 0.0)) {  // fall back to the Ritz sum as the scale
    trace = 0.0;
    for (int i = 0; i < b; ++i) trace += h_theta[i] > 0 ? h_theta[i] : 0;
  }
  double prev = 0.0;
  for (int i = 0; i < k; ++i) prev += h_theta[i];
  bool converged = false;
  int outer = 0;
  for (; outer < max_outer; ++outer) {
    const double top = h_theta[0];
    if (!(top > 0.0)) {  // numerically zero matrix: nothing to iterate on
      converged = true;
      break;
    }
    double cut = h_theta[b - 1] > 0.0 ? h_theta[b - 1] : 0.0;
    double hi = cut;
    const double tiny = 1e-30 * top + 1e-300;
    if (hi < tiny) hi = tiny;
    const double e = 0.5 * hi, c = 0.5 * hi;
    double x1 = (top - c) / e;
    if (x1 < 1.0) x1 = 1.0;
    double ac = acosh(x1);
    if (ac < 1e-12) ac = 1e-12;
    int m = (int)floor(log(2.0 * spread) / ac);
    if (m < 1) m = 1;
    if (m > mmax) m = mmax;
    // scaled Chebyshev recurrence: p_i(t) = T_i((t-c)/e) / T_i((top-c)/e)
    const double sigma1 = e / (top - c);
    double sigma = sigma1;
    // three rotating buffers: Xprev, Ycur, Ynew
    TB* bufs[3];
    {
      TB* all3[3] = {w.X, w.Y, w.Z};
      int c3 = 1;
      bufs[0] = X;
      for (int q = 0; q < 3; ++q)
        if (all3[q] != X) bufs[c3++] = all3[q];
    }
    bool fused = false;
    if (w.use_tc && !w.shared_gpu && std::is_same<TB, float>::value && m <= CF_MAX_STEPS) {
      // the whole filter as one resident kernel (cheb_filter.cuh); same recurrence, coefficients precomputed
      float fa[CF_MAX_STEPS], fb[CF_MAX_STEPS], fg[CF_MAX_STEPS];
      double sg = sigma1;
      fa[0] = (float)(sigma1 / e); fb[0] = (float)(-c * sigma1 / e); fg[0] = 0.f;
      for (int i = 2; i <= m; ++i) {
        const double sigma2 = 1.0 / (2.0 / sigma1 - sg);
        fa[i - 1] = (float)(2.0 * sigma2 / e); fb[i - 1] = (float)(-2.0 * sigma2 * c / e); fg[i - 1] = (float)(-sg * sigma2);
        sg = sigma2;
      }
      float* fbufs[3] = {reinterpret_cast<float*>(bufs[0]), reinterpret_cast<float*>(bufs[1]), reinterpret_cast<float*>(bufs[2])};
      const int rc = cheb_filter_f32(reinterpret_cast<const float*>(G), n, b, fbufs, m, fa, fb, fg, w.partial,
                                     w.partial_bytes, st);
      if (rc == TNB_OK) fused = true;
      else if (rc != TNB_ERR_UNSUPPORTED) return rc;
    }
    int icur = m % 3, inew = (m + 1) % 3;
    if (fused) {
      if (stats) stats->fused_filters += 1;
    } else {
      // Y = (G X - c X) * sigma1/e
      TNB_TRY(chfsi_apply<TB>(G, n, b, bufs[0], nullptr, bufs[1], sigma1 / e, -c * sigma1 / e, 0.0, w, st, true));
      int iprev = 0;
      icur = 1; inew = 2;
      for (int i = 2; i <= m; ++i) {
        const double sigma2 = 1.0 / (2.0 / sigma1 - sigma);
        // Ynew = 2 sigma2/e (G Y - c Y) - sigma sigma2 Xprev
        TNB_TRY(chfsi_apply<TB>(G, n, b, bufs[icur], bufs[iprev], bufs[inew], 2.0 * sigma2 / e, -2.0 * sigma2 * c / e,
                                -sigma * sigma2, w, st, true));
        const int t = iprev; iprev = icur; icur = inew; inew = t;
        sigma = sigma2;
      }
    }
    if (stats) stats->products += m + 1;
    X = bufs[icur];
    Xt = bufs[inew];
    TNB_TRY(chfsi_orthonormalize<TB>(n, b, &X, &Xt, w, st, use_chol));
    TNB_TRY(chfsi_rayleigh_ritz<TB>(G, n, b, &X, &Xt, w, st));
    TNB_CUDA(cudaMemcpyAsync(h_theta, w.lam, (size_t)b * sizeof(double), cudaMemcpyDeviceToHost, st));
    TNB_CUDA(cudaMemcpyAsync(h_flag, w.jinfo, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
    TNB_CUDA(cudaStreamSynchronize(st));
    double cap = 0.0;
    for (int i = 0; i < k; ++i) cap += h_theta[i];
    if (stats) stats->rr_sweeps += h_flag[0] < 0 ? -h_flag[0] : h_flag[0];
    if (h_flag[1] != 0) {
      // Cholesky saw numerically dependent columns: this iteration's basis is unreliable; go back to the
      // eigen-decomposition based transform for the rest of the solve and do not test convergence now
      use_chol = false;
      TNB_CUDA(cudaMemsetAsync(w.jinfo, 0, 4 * sizeof(int), st));
      prev = cap < prev ? cap : prev;
      continue;
    }
    if (outer >= 1 && cap - prev <= tol * trace) {
      converged = true;
      ++outer;
      break;
    }
    prev = cap;
  }
  if (stats) {
    stats->outer += outer;
    stats->converged = converged ? 1 : 0;
  }
  if (!use_chol) {
    // a Cholesky breakdown was seen (numerically rank-deficient block): the eigen-decomposition based transform
    // clamps the lost directions, which leaves the block orthonormal only approximately.  One Cholesky-QR pass in
    // column order (= Gram-Schmidt: clamped trailing pivots do not touch the leading vectors) restores it.
    TNB_TRY(chfsi_orthonormalize<TB>(n, b, &X, &Xt, w, st, true));
  }
  TNB_CUDA(cudaMemcpyAsync(theta_out, w.lam, (size_t)b * sizeof(double), cudaMemcpyDeviceToDevice, st));
  convert_kernel<TB, double><<<grid_for((int64_t)n * b), 256, 0, st>>>(X, X_out, (int64_t)n * b);
  TNB_LAUNCH_CHECK();
  if (!converged) return fail(TNB_ERR_NOCONV, "eig_topk: no convergence in %d outer iterations (n=%d k=%d b=%d)", max_outer, n, k, b);
  return TNB_OK;
}

}  // namespace tnb

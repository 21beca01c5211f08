// Glue kernels around the GEMM / eigen kernels: rank rule, factor extraction, traces, fills.
#pragma once
#include "common.cuh"
#include "jacobi.cuh"

namespace tnb {

// Device-side scalars shared by the steps of one sweep.
struct SweepScalars {
  double norm2;      // ||T||_F^2  (trace of the first Gram)
  double delta2;     // absolute tail-energy budget delta^2 (round.py:151)
  double trace;      // trace of the current Gram
  double spare[5];
  int rank;          // chosen rank of the current step
  int zero_flag;     // 1 when the current unfolding is numerically zero (round.py:137-145)
  int jacobi_info;   // sweeps used by the last Jacobi solve (negative: not converged)
  int undecided;     // leading-values rule only: 1 when the tail behind the kk known values is still above delta^2
  int tf32_reject;   // the Gram matrix of this step came from the TF32 tensor-core kernel and its noise floor could move
                     // the relative error by more than the parity bar: the step must be redone with the exact Gram
  int spare_i[3];
};

// Is a TF32 tensor-core Gram good enough for THIS spectrum?  G_tf32 = (1 - c) G + E with ||E|| ~ 2e-6 ||G||
// (tests/test_model.py).  The uniform shrink is harmless; E costs captured energy: at most 2 r ||E|| (Ky Fan), and when
// the kept and discarded parts are separated by gap = lambda_{r-1} - lambda_r, at most lambda_0 r (||E|| / gap)^2
// (Davis-Kahan).  The step is accepted when that loss moves the relative error sqrt(tail / trace) by less than 5e-6
// (half the 1e-5 parity bar), with the tail taken at the low end of what the noisy values resolve.  A flat spectrum
// (random data: lambda_0 << trace, tail ~ trace) passes on the first bound; signal + noise with a clear gap passes on the
// second; a tensor whose discarded tail is below ~1e-4 of its norm does not, and takes the exact Gram.
__device__ inline int tf32_gram_rejected(const double* w, int nvals, int L, int rank, double trace) {
  if (rank >= L) return 0;  // nothing discarded
  const double lam0 = w[0] > 0.0 ? w[0] : 0.0;
  if (!(trace > 0.0) || !(lam0 > 0.0)) return 0;
  const double normE = 4e-6 * lam0;  // twice the measured 2e-6
  double head = 0.0;
  for (int i = 0; i < rank && i < nvals; ++i) head += w[i] > 0.0 ? w[i] : 0.0;
  const double first = 2.0 * rank * normE;
  const double tail_lo = trace - head - first;
  if (!(tail_lo > 0.0)) return 1;
  double loss = first;
  if (rank < nvals) {
    const double next = w[rank] > 0.0 ? w[rank] : 0.0;
    const double gap = w[rank - 1] - next;
    if (gap > 4.0 * normE) {
      const double q = normE / gap;
      const double second = lam0 * rank * q * q;
      if (second < loss) loss = second;
    }
  }
  return loss > 1e-5 * sqrt(tail_lo * trace) ? 1 : 0;
}

__global__ void trace_kernel(const double* __restrict__ G, int n, int ld, SweepScalars* sc, int set_norm,
                             double eps_scaled /* (eps/max(1,sqrt(N-1)))^2, used when set_norm */) {
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += G[(size_t)i * ld + i];
  s = block_reduce_sum(s, red);
  if (threadIdx.x == 0) {
    sc->trace = s;
    if (set_norm) {
      sc->norm2 = s;
      sc->delta2 = eps_scaled * s;
    }
  }
}

__global__ void set_delta2_kernel(SweepScalars* sc, double delta_abs, double eps_rel) {
  // truncated_svd semantics (round.py:79-82): delta given, or eps * ||M||, or 0
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (delta_abs >= 0.0) sc->delta2 = delta_abs * delta_abs;
    else if (eps_rel >= 0.0) sc->delta2 = eps_rel * eps_rel * sc->trace;
    else sc->delta2 = 0.0;
  }
}

// round.py:137-158 on descending eigenvalues w (= squared singular values).
//   full spectrum (topk == 0): w holds all L values.
//   leading values only (topk == 1): w holds kk >= min(rmax, L) leading Ritz values; the tail energy
//   behind index k is trace - sum_{i<=k} w_i.
__global__ void rank_rule_kernel(const double* __restrict__ w, int L, int kk, int rmax, int topk, int batch_mode,
                                 SweepScalars* sc, int used_tf32 = 0, int nvals = 0) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  sc->tf32_reject = 0;
  const double w0 = w[0] > 0.0 ? w[0] : 0.0;
  sc->zero_flag = (sqrt(w0) < 1e-13) ? 1 : 0;
  sc->undecided = 0;
  int cap = L;
  if (rmax > 0 && rmax < cap) cap = rmax;
  int rank;
  if (batch_mode) {
    rank = cap;
  } else if (!topk) {
    double cum = 0.0;
    int count_true = 0;
    for (int i = L - 1; i >= 0; --i) {
      const double v = w[i] > 0.0 ? w[i] : 0.0;
      cum += v;
      if (cum <= sc->delta2) ++count_true; else break;
    }
    rank = L - count_true;
    if (rank > cap) rank = cap;
  } else {
    // rank = min(cap, L - count_true); only ranks <= cap matter, and tail_k for k < cap is computable
    double head = 0.0;
    rank = cap;
    sc->undecided = (cap > kk) ? 1 : 0;  // cleared when a rank within the known values meets the budget
    for (int k = 0; k < cap && k < kk; ++k) {
      head += (w[k] > 0.0 ? w[k] : 0.0);
      const double tail = sc->trace - head;  // energy discarded if the rank were k+1
      if (tail <= sc->delta2) {
        rank = k + 1;
        sc->undecided = 0;
        break;
      }
    }
  }
  if (rank < 1) rank = 1;
  sc->rank = rank;
  if (used_tf32 && !sc->zero_flag && !sc->undecided) sc->tf32_reject = tf32_gram_rejected(w, nvals > 0 ? nvals : (topk ? kk : L), L, rank, sc->trace);
}

// Speculative sweep (sweep.cuh): the step was enqueued assuming rank == expect; record the rank the rule chose and raise
// the flags the host checks at its single final synchronisation.
//   bit 0: TF32 Gram rejected   bits 1-3: subspace solver (chfsi_dev.cuh)   bit 4: rank differs   bit 5: zero unfolding
__global__ void spec_check_kernel(const SweepScalars* sc, int expect, int32_t* rank_out, int* flags) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  *rank_out = sc->rank;
  int f = 0;
  if (sc->tf32_reject) f |= 1;
  if (sc->rank != expect) f |= 16;
  if (sc->zero_flag) f |= 32;
  if (f) atomicOr(flags, f);
}

// out[i][j] (or out[j][i] when transpose) = V[i][j] * f(w_j) for j < rank, i < rows.
//   mode 0: f = 1        mode 1: f = 1/sqrt(w_j)        mode 2: f = sqrt(w_j)
template <typename TOut>
__global__ void scale_extract_kernel(const double* __restrict__ V, int ldv, int rows, int rank,
                                     const double* __restrict__ w, TOut* __restrict__ out, int mode, int transpose) {
  const int64_t total = (int64_t)rows * rank;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int i, j;
    if (transpose) {  // idx enumerates out[j][i]
      j = (int)(idx / rows);
      i = (int)(idx % rows);
    } else {
      i = (int)(idx / rank);
      j = (int)(idx % rank);
    }
    double f = 1.0;
    if (mode != 0) {
      const double wj = w[j] > 0.0 ? w[j] : 0.0;
      const double s = sqrt(wj);
      f = (mode == 1) ? (s > 0.0 ? 1.0 / s : 0.0) : s;
    }
    out[idx] = (TOut)(V[(size_t)i * ldv + j] * f);
  }
}

template <typename T>
__global__ void fill_kernel(T* p, int64_t n, T v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

template <typename TIn, typename TOut>
__global__ void convert_kernel(const TIn* __restrict__ in, TOut* __restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (TOut)in[i];
}

__device__ __forceinline__ uint32_t hash_u32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
  return x;
}
// deterministic pseudo-random block in (-1, 1)
template <typename T>
__global__ void random_fill_kernel(T* p, int64_t n, uint32_t seed) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t h = hash_u32((uint32_t)i * 2654435761U + seed) ^ hash_u32((uint32_t)(i >> 32) + 0x9e3779b9U * seed);
    p[i] = (T)(((double)(h >> 8) + 0.5) * (2.0 / 16777216.0) - 1.0);
  }
}

// SVQB step 1: d_i = 1/sqrt(S_ii), S_ij <- d_i S_ij d_j   (one CTA, b <= 256)
__global__ void svqb_prep_kernel(double* __restrict__ S, int b, double* __restrict__ d) {
  __shared__ double sd[JACOBI_MAX_N];
  for (int i = threadIdx.x; i < b; i += blockDim.x) {
    const double v = S[(size_t)i * b + i];
    const double di = v > 1e-300 ? 1.0 / sqrt(v) : 0.0;
    sd[i] = di;
    d[i] = di;
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < b * b; idx += blockDim.x) {
    const int i = idx / b, j = idx % b;
    S[idx] *= sd[i] * sd[j];
  }
}
// SVQB step 2: T_ij = d_i Q_ij / sqrt(max(lam_j, lam_0 * floor))
template <typename TB>
__global__ void svqb_finish_kernel(const double* __restrict__ Q, const double* __restrict__ lam,
                                   const double* __restrict__ d, int b, double floor_rel, TB* __restrict__ T) {
  const double lmax = lam[0] > 0.0 ? lam[0] : 0.0;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < b * b; idx += gridDim.x * blockDim.x) {
    const int i = idx / b, j = idx % b;
    double lj = lam[j];
    const double fl = lmax * floor_rel;
    if (lj < fl) lj = fl;
    T[idx] = (TB)(lj > 0.0 ? d[i] * Q[idx] / sqrt(lj) : 0.0);
  }
}

// Cholesky-QR transform for a block whose (column-scaled) Gram matrix S is safely positive definite:
//   d_i = 1/sqrt(S_ii),  D S D = L L^T,  T = D L^{-T}   =>   (Y T)^T (Y T) = I.
// One CTA, fp64; b <= 256.  scratch holds L and L^{-1} (2*b*b doubles) when they do not fit shared memory.
// A pivot below 1e-11 (numerically dependent columns) raises *flag and is clamped: the caller then
// falls back to the eigen-decomposition based SVQB transform.
template <typename TB>
__device__ __forceinline__ void chol_orth_device(const double* __restrict__ S, int b, double* scratch,
                                                 TB* __restrict__ T, int* flag, int use_smem, TB* __restrict__ Rout,
                                                 unsigned char* chol_smem_raw) {
  __shared__ double s_d[JACOBI_MAX_N];
  __shared__ double s_piv[JACOBI_MAX_N];
  const int ld = b | 1;  // odd leading dimension: column walks (stride ld) spread over the banks
  double* L = use_smem ? reinterpret_cast<double*>(chol_smem_raw) : scratch;
  double* Li = L + (size_t)b * ld;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < b; i += nt) {
    const double v = S[(size_t)i * b + i];
    s_d[i] = v > 1e-300 ? rsqrt(v) : 0.0;
  }
  __syncthreads();
  for (int idx = tid; idx < b * b; idx += nt) {
    const int i = idx / b, j = idx % b;
    L[(size_t)i * ld + j] = (j <= i) ? S[idx] * s_d[i] * s_d[j] : 0.0;
    Li[(size_t)i * ld + j] = 0.0;
  }
  __syncthreads();
  // right-looking Cholesky with ONE barrier per column: the trailing update uses the unscaled column k and
  // 1/pivot; column k is final after step k, so its scaling by 1/sqrt(pivot) is deferred to a single pass.
  for (int k = 0; k < b; ++k) {
    double piv = L[(size_t)k * ld + k];  // broadcast read
    if (!(piv > 1e-11)) {
      if (tid == 0) *flag = 1;
      piv = 1e-11;
    }
    if (tid == 0) s_piv[k] = piv;
    const double ipiv = 1.0 / piv;
    const int rem = b - k - 1;
    // rows i > k are dealt round-robin to the warps, the lanes walk j = k+1..i
    for (int i = k + 1 + (tid >> 5); i < b; i += (nt >> 5)) {
      const double lik = L[(size_t)i * ld + k] * ipiv;
      for (int j = k + 1 + (tid & 31); j <= i; j += 32) L[(size_t)i * ld + j] -= lik * L[(size_t)j * ld + k];
    }
    (void)rem;
    __syncthreads();
  }
  for (int idx = tid; idx < b * b; idx += nt) {
    const int i = idx / b, k = idx % b;
    if (k < i) L[(size_t)i * ld + k] *= rsqrt(s_piv[k]);
    else if (k == i) L[(size_t)i * ld + k] = sqrt(s_piv[k]);
  }
  __syncthreads();
  // L^{-1}: one warp per column j (forward substitution, the inner sum split over the lanes)
  {
    const int lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    for (int j = warp; j < b; j += nwarps) {
      if (lane == 0) Li[(size_t)j * ld + j] = 1.0 / L[(size_t)j * ld + j];
      __syncwarp();
      for (int i = j + 1; i < b; ++i) {
        double acc = 0.0;
        for (int k = j + lane; k < i; k += 32) acc = fma(L[(size_t)i * ld + k], Li[(size_t)k * ld + j], acc);
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) Li[(size_t)i * ld + j] = -acc / L[(size_t)i * ld + i];
        __syncwarp();
      }
    }
  }
  __syncthreads();
  for (int idx = tid; idx < b * b; idx += nt) {
    const int i = idx / b, j = idx % b;
    T[idx] = (TB)((j >= i) ? s_d[i] * Li[(size_t)j * ld + i] : 0.0);
    // the matching triangular factor R = L^T D^-1 (A = (A T) R): R[i][j] = L[j][i] / d_j
    if (Rout) Rout[idx] = (TB)((j >= i && s_d[j] > 0.0) ? L[(size_t)j * ld + i] / s_d[j] : 0.0);
  }
}

template <typename TB>
__global__ void __launch_bounds__(1024) chol_orth_kernel(const double* __restrict__ S, int b, double* scratch,
                                                         TB* __restrict__ T, int* flag, int use_smem,
                                                         TB* __restrict__ Rout = nullptr) {
  extern __shared__ __align__(16) unsigned char chol_smem_dyn[];
  chol_orth_device<TB>(S, b, scratch, T, flag, use_smem, Rout, chol_smem_dyn);
}

// chol_orth_kernel on `st`: L and L^-1 in shared memory when they fit its 180 KB, in `scratch` otherwise.
template <typename TB>
inline int chol_orth(const double* S, int b, double* scratch, TB* T, int* flag, TB* Rout, cudaStream_t st) {
  const size_t smem = (size_t)2 * b * (b | 1) * sizeof(double);
  const bool fits = smem <= (size_t)180 * 1024;
  static PerDeviceFlag attr_done;
  TNB_CUDA(ensure_dyn_smem(attr_done, chol_orth_kernel<TB>, 180 * 1024));
  chol_orth_kernel<TB><<<1, 1024, fits ? smem : 0, st>>>(S, b, scratch, T, flag, fits ? 1 : 0, Rout);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

inline int grid_for(int64_t n, int block = 256, int cap = 4096) {
  int64_t g = ceil_div<int64_t>(n, block);
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

}  // namespace tnb

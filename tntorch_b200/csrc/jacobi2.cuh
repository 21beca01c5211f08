// CUDA side of the two-sided Jacobi eigensolver (jacobi2_core.h): a block-level solve usable inside larger one-CTA
// kernels (the fused Rayleigh-Ritz step of chfsi_dev.cuh) and a stand-alone kernel with the interface of
// jacobi_eigh_kernel (jacobi.cuh).  Everything lives in shared memory; one __syncthreads after each of the two phases
// of a round.  n <= 80 in fp64, n <= 112 in fp32 (four n x (n+1) matrices must fit); larger problems stay on jacobi.cuh.
#pragma once
#include "common.cuh"
#include "jacobi.cuh"
#include "jacobi2_core.h"

namespace tnb {

constexpr int JAC2_MAX_N_F64 = 80;
constexpr int JAC2_MAX_N_F32 = 112;

template <typename R>
__host__ __device__ inline size_t jac2_smem_bytes(int n) {
  const int np = n + (n & 1), m = np / 2, lds = np + 2;
  size_t b = (size_t)4 * np * lds * sizeof(R);       // S[2], V[2]
  b += (size_t)(4 * m + 4) * sizeof(R);              // cs[2]
  b = (b + 15) / 16 * 16;
  b += 4 * sizeof(int);
  return (b + 15) / 16 * 16;
}

// Carve the solver state out of a shared-memory region of jac2_smem_bytes<R>(n) bytes (16-byte aligned).
template <typename R>
__device__ inline void jac2_carve(unsigned char* smem, int n, R tol, Jac2<R>& J) {
  const int np = n + (n & 1), m = np / 2, lds = np + 2;  // even row stride: the 2-element reads are aligned
  R* p = reinterpret_cast<R*>(smem);
  J.S[0] = p; p += (size_t)np * lds;
  J.S[1] = p; p += (size_t)np * lds;
  J.V[0] = p; p += (size_t)np * lds;
  J.V[1] = p; p += (size_t)np * lds;
  J.cs[0] = p; p += 2 * m + 2;
  J.cs[1] = p;
  size_t off = ((size_t)4 * np * lds + 4 * m + 4) * sizeof(R);
  off = (off + 15) / 16 * 16;
  J.flag = reinterpret_cast<int*>(smem + off);
  J.np = np;
  J.m = m;
  J.lds = lds;
  J.tol2 = tol * tol;
  J.big2 = tol;
  J.floor_abs = sizeof(R) == 8 ? (R)2.3e-16 : (R)1.2e-7;
}

// Block-level solve.  On entry S[0] holds the (scaled) matrix in canonical upper storage — element (i, j), i <= j, at
// [i * lds + j]; the strict lower triangle is never read — and V[0] the identity.  On return buffer `cur` (the return
// value) holds the rotated matrix (diagonal = eigenvalues, unsorted) and the eigenvectors in the columns of V[cur].
// Every thread of the block must call it.  Thread roles: the first ceil(m/32) warps are "pair threads" (thread k forms
// the next round's pair k and its rotation), the others are workers with up to JAC2_ITEMS static work items each in
// registers (when the block is too small for that, the items are regenerated every round: correct, slower).
template <typename R>
__device__ inline int jac2_solve(const Jac2<R>& Jin, int max_sweeps, int* sweeps_out) {
  const Jac2<R> J = Jin;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int m = J.m;
  const int pw = (m + 31) / 32 * 32;
  const int workers = nt - pw;
  const int total = jac2_total_items(J);
  const bool in_regs = total <= workers * JAC2_ITEMS;
  const int per = (total + workers - 1) / workers;
  const bool is_pair = tid < m, is_worker = tid >= pw;
  const int wid = tid - pw;
  Jac2Item it0, it1, it2;
  Jac2Pair pp;
  it0.kind = it1.kind = it2.kind = 0;
  if (is_worker && in_regs) {
    jac2_make_item(J, wid, it0);
    jac2_make_item(J, wid + workers, it1);
    jac2_make_item(J, wid + 2 * workers, it2);
  }
  if (is_pair) jac2_make_pair(J, tid, pp);
  if (tid == 0) { J.flag[0] = 0; J.flag[1] = 0; }
  __syncthreads();
  if (is_pair) jac2_first_pair(J, 0, 0, tid, &J.flag[0]);
  __syncthreads();
  const int rounds = J.np > 2 ? J.np - 1 : 1;
  // explicit buffer pointers swapped in registers (no dynamically indexed arrays in the round loop)
  R *Sr = J.S[0], *Sw = J.S[1], *Vr = J.V[0], *Vw = J.V[1], *cr = J.cs[0], *cw = J.cs[1];
  int cur = 0, sweep = 0;
  bool conv = false;
  for (; sweep < max_sweeps && !conv; ++sweep) {
    int* fl = &J.flag[sweep & 1];
    if (tid == 0) J.flag[(sweep + 1) & 1] = 0;  // nobody touches the other flag during this sweep
    for (int r = 0; r < rounds; ++r) {
      Jac2<R> Jc = J;  // read side at index 0, write side at index 1
      Jc.S[0] = Sr; Jc.S[1] = Sw; Jc.V[0] = Vr; Jc.V[1] = Vw; Jc.cs[0] = cr; Jc.cs[1] = cw;
      if (is_worker) {
        if (in_regs) {
          jac2_do_item(Jc, 0, 0, it0);
          jac2_do_item(Jc, 0, 0, it1);
          jac2_do_item(Jc, 0, 0, it2);
        } else {
          for (int q = 0; q < per; ++q) {
            Jac2Item it;
            jac2_make_item(J, wid + q * workers, it);
            jac2_do_item(Jc, 0, 0, it);
          }
        }
      } else if (is_pair) {
        jac2_do_pair(Jc, 0, 0, tid, pp, fl);
      }
      __syncthreads();
      cur ^= 1;
      { R* t = Sr; Sr = Sw; Sw = t; }
      { R* t = Vr; Vr = Vw; Vw = t; }
      { R* t = cr; cr = cw; cw = t; }
    }
    conv = (*fl == 0);
  }
  __syncthreads();
  if (sweeps_out) *sweeps_out = conv ? sweep : -sweep;
  return cur;
}

// Stand-alone eigensolver with the contract of jacobi_eigh_kernel: Gin n x n fp64 (ld ldg), w_out descending,
// V_out n x n row-major (column j = eigenvector of w_out[j]), info[0] = sweeps (negative: max_sweeps hit).
// Eigenvalues are Rayleigh quotients v^T G v in fp64 against the input matrix (so the fp32 variant returns values as
// accurate as its vectors allow, not the rounding-accumulated diagonal).
template <typename R>
__global__ void __launch_bounds__(1024) jacobi2_eigh_kernel(const double* __restrict__ Gin, int n, int ldg,
                                                            double* __restrict__ w_out, double* __restrict__ V_out,
                                                            int max_sweeps, R tol, int* __restrict__ info) {
  extern __shared__ __align__(16) unsigned char jac2_smem[];
  __shared__ double s_w[JAC2_MAX_N + 2];
  __shared__ int s_rank[JAC2_MAX_N + 2];
  __shared__ double s_gmax;
  __shared__ int s_sweeps;
  Jac2<R> J;
  jac2_carve<R>(jac2_smem, n, tol, J);
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
  const int np = J.np, lds = J.lds;
  double dmax = 0.0;
  for (int i = tid; i < n; i += nt) dmax = fmax(dmax, fabs(Gin[(size_t)i * ldg + i]));
  for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
  if (tid == 0) s_gmax = 0.0;
  __syncthreads();
  if (lane == 0) atomicMax(reinterpret_cast<unsigned long long*>(&s_gmax), (unsigned long long)__double_as_longlong(dmax));
  __syncthreads();
  const double gscale = s_gmax > 0.0 ? s_gmax : 1.0;
  const double ginv = 1.0 / gscale;
  for (int idx = tid; idx < np * np; idx += nt) {
    const int r = idx / np, c = idx - r * np;
    double v = 0.0;
    if (r < n && c < n) v = 0.5 * (Gin[(size_t)r * ldg + c] + Gin[(size_t)c * ldg + r]) * ginv;
    if (c >= r) J.S[0][r * lds + c] = (R)v;  // canonical upper storage
    J.V[0][r * lds + c] = (r == c) ? (R)1 : (R)0;
  }
  __syncthreads();
  const int cur = jac2_solve(J, max_sweeps, &s_sweeps);
  const R* V = J.V[cur];
  if (sizeof(R) == 4) {
    // ~500 fp32 rotations per column leave V orthogonal to ~1e-5; one Newton-Schulz step V <- V (1.5 I - 0.5 V^T V)
    // in fp32 brings that to ~1e-7, the level of the fp32 factors extracted from it
    R* E = J.S[0];
    R* Vn = J.V[cur ^ 1];
    for (int idx = tid; idx < np * np; idx += nt) {
      const int i = idx / np, j = idx - i * np;
      R acc = (R)0;
      for (int c = 0; c < np; ++c) acc = fma(V[c * lds + i], V[c * lds + j], acc);
      E[i * lds + j] = (i == j ? (R)1.5 : (R)0) - (R)0.5 * acc;
    }
    __syncthreads();
    for (int idx = tid; idx < np * np; idx += nt) {
      const int i = idx / np, j = idx - i * np;
      R acc = (R)0;
      for (int c = 0; c < np; ++c) acc = fma(V[i * lds + c], E[c * lds + j], acc);
      Vn[i * lds + j] = acc;
    }
    __syncthreads();
    V = Vn;
  }
  // Rayleigh quotients against the input (fp64), one warp per column; the pad column (odd n) is the one that still
  // carries the unit entry of the pad row and is ranked last
  for (int j = warp; j < np; j += nwarps) {
    double acc = 0.0;
    for (int r = lane; r < n; r += 32) {
      double t = 0.0;
      for (int c = 0; c < n; ++c) t = fma(Gin[(size_t)c * ldg + r], (double)V[c * lds + j], t);  // G symmetric: coalesced side
      acc = fma((double)V[r * lds + j], t, acc);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const bool pad = (np != n) && fabs((double)V[n * lds + j]) > 0.5;
      s_w[j] = pad ? -1e300 : acc;
    }
  }
  __syncthreads();
  for (int i = tid; i < np; i += nt) {
    const double wi = s_w[i];
    int r = 0;
    for (int j = 0; j < np; ++j) {
      const double wj = s_w[j];
      r += (wj > wi) || (wj == wi && j < i);
    }
    s_rank[i] = r;
    if (r < n) w_out[r] = wi;
  }
  __syncthreads();
  for (int idx = tid; idx < n * np; idx += nt) {
    const int k = idx / np, i = idx - k * np;
    const int r = s_rank[i];
    if (r < n) V_out[(size_t)k * n + r] = (double)V[k * lds + i];
  }
  if (tid == 0 && info) info[0] = s_sweeps;
}

// fp64 results at mostly fp32 cost.  The B200 issues ~16 fp64 FMAs per clock and SM against 128 fp32 ones, and a 64 x 64
// fp64 Jacobi solve is bound by exactly that (measured 0.88 ms, nine sweeps).  Here the sweeps that do the real work run
// in fp32; their basis V is promoted, re-orthonormalised in fp64 (one Newton-Schulz step: 1e-7 -> 1e-14), the matrix is
// taken into that basis in fp64, S2 = V^T G V — now diagonal up to ~1e-6 — and fp64 sweeps finish from there: two of them
// by quadratic convergence (1e-6 -> 1e-12 -> below the threshold).  Same contract and accuracy as the all-fp64 kernel.
constexpr int JAC2_MIXED_MAX_N = 64;

__global__ void __launch_bounds__(1024) jacobi2_mixed_kernel(const double* __restrict__ Gin, int n, int ldg,
                                                             double* __restrict__ w_out, double* __restrict__ V_out,
                                                             int max_sweeps, double tol, int* __restrict__ info) {
  extern __shared__ __align__(16) unsigned char jac2m_smem[];
  __shared__ double s_w[JAC2_MAX_N + 2];
  __shared__ int s_rank[JAC2_MAX_N + 2];
  __shared__ double s_gmax;
  __shared__ int s_sweeps32, s_sweeps64;
  Jac2<double> J;
  Jac2<float> F;
  jac2_carve<double>(jac2m_smem, n, tol, J);
  jac2_carve<float>(jac2m_smem + jac2_smem_bytes<double>(n), n, 2e-6f, F);
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
  const int np = J.np, lds = J.lds;
  double dmax = 0.0;
  for (int i = tid; i < n; i += nt) dmax = fmax(dmax, fabs(Gin[(size_t)i * ldg + i]));
  for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
  if (tid == 0) s_gmax = 0.0;
  __syncthreads();
  if (lane == 0) atomicMax(reinterpret_cast<unsigned long long*>(&s_gmax), (unsigned long long)__double_as_longlong(dmax));
  __syncthreads();
  const double gscale = s_gmax > 0.0 ? s_gmax : 1.0;
  const double ginv = 1.0 / gscale;
  // ---- fp32 solve ----
  for (int idx = tid; idx < np * np; idx += nt) {
    const int r = idx / np, c = idx - r * np;
    double v = 0.0;
    if (r < n && c < n) v = 0.5 * (Gin[(size_t)r * ldg + c] + Gin[(size_t)c * ldg + r]) * ginv;
    if (c >= r) F.S[0][r * lds + c] = (float)v;
    F.V[0][r * lds + c] = (r == c) ? 1.f : 0.f;
    J.S[1][r * lds + c] = v;  // the scaled symmetric matrix in fp64 (full storage), read by the congruence below
  }
  __syncthreads();
  const int c32 = jac2_solve(F, max_sweeps, &s_sweeps32);
  const float* V32 = F.V[c32];
  {
    // ~500 fp32 rotations per column leave V32 orthogonal to ~1e-5: a first Newton-Schulz step in fp32 (cheap) brings
    // that to ~1e-7, the fp64 step below then to ~1e-14 (one fp64 step from 1e-5 would only reach ~1e-10 and the
    // eigenvalues of the congruence V^T G V would be off by as much)
    float* E32 = F.S[0];
    float* Vn32 = F.V[c32 ^ 1];
    for (int idx = tid; idx < np * np; idx += nt) {
      const int i = idx / np, j = idx - i * np;
      float acc = 0.f;
      for (int c = 0; c < np; ++c) acc = fmaf(V32[c * lds + i], V32[c * lds + j], acc);
      E32[i * lds + j] = (i == j ? 1.5f : 0.f) - 0.5f * acc;
    }
    __syncthreads();
    for (int idx = tid; idx < np * np; idx += nt) {
      const int i = idx / np, j = idx - i * np;
      float acc = 0.f;
      for (int c = 0; c < np; ++c) acc = fmaf(V32[i * lds + c], E32[c * lds + j], acc);
      Vn32[i * lds + j] = acc;
    }
    __syncthreads();
    V32 = Vn32;
  }
  // ---- promote, re-orthonormalise (fp64 Newton-Schulz), congruence ----
  double* Vp = J.V[1];   // promoted basis
  double* E = J.S[0];    // 1.5 I - 0.5 V^T V (full storage), later overwritten by S2
  double* Vn = J.V[0];   // orthonormal basis the fp64 sweeps start from
  for (int idx = tid; idx < np * np; idx += nt) {
    const int r = idx / np, c = idx - r * np;
    Vp[r * lds + c] = (double)V32[r * lds + c];
  }
  __syncthreads();
  for (int idx = tid; idx < np * np; idx += nt) {
    const int i = idx / np, j = idx - i * np;
    double acc = 0.0;
    for (int c = 0; c < np; ++c) acc = fma(Vp[c * lds + i], Vp[c * lds + j], acc);
    E[i * lds + j] = (i == j ? 1.5 : 0.0) - 0.5 * acc;
  }
  __syncthreads();
  for (int idx = tid; idx < np * np; idx += nt) {
    const int i = idx / np, j = idx - i * np;
    double acc = 0.0;
    for (int c = 0; c < np; ++c) acc = fma(Vp[i * lds + c], E[c * lds + j], acc);
    Vn[i * lds + j] = acc;
  }
  __syncthreads();
  // W = G Vn into Vp (the promoted copy is dead), then S2 = Vn^T W (upper triangle) into S[0]
  const double* Gs = J.S[1];
  for (int idx = tid; idx < np * np; idx += nt) {
    const int i = idx / np, j = idx - i * np;
    double acc = 0.0;
    for (int c = 0; c < np; ++c) acc = fma(Gs[i * lds + c], Vn[c * lds + j], acc);
    Vp[i * lds + j] = acc;
  }
  __syncthreads();
  for (int idx = tid; idx < np * np; idx += nt) {
    const int i = idx / np, j = idx - i * np;
    if (j < i) continue;
    double acc = 0.0;
    for (int c = 0; c < np; ++c) acc = fma(Vn[c * lds + i], Vp[c * lds + j], acc);
    E[i * lds + j] = acc;  // E == J.S[0]
  }
  __syncthreads();
  // ---- fp64 finish (V[0] = Vn is the starting basis) ----
  const int cur = jac2_solve(J, max_sweeps, &s_sweeps64);
  const double* V = J.V[cur];
  const double* S = J.S[cur];
  for (int j = tid; j < np; j += nt) {
    const bool pad = (np != n) && fabs(V[n * lds + j]) > 0.5;
    s_w[j] = pad ? -1e300 : S[j * lds + j] * gscale;
  }
  __syncthreads();
  for (int i = tid; i < np; i += nt) {
    const double wi = s_w[i];
    int r = 0;
    for (int j = 0; j < np; ++j) {
      const double wj = s_w[j];
      r += (wj > wi) || (wj == wi && j < i);
    }
    s_rank[i] = r;
    if (r < n) w_out[r] = wi;
  }
  __syncthreads();
  for (int idx = tid; idx < n * np; idx += nt) {
    const int k = idx / np, i = idx - k * np;
    const int r = s_rank[i];
    if (r < n) V_out[(size_t)k * n + r] = V[k * lds + i];
  }
  if (tid == 0 && info) {
    const int a = s_sweeps32 < 0 ? -s_sweeps32 : s_sweeps32, b = s_sweeps64 < 0 ? -s_sweeps64 : s_sweeps64;
    info[0] = (s_sweeps32 < 0 || s_sweeps64 < 0) ? -(a + b) : (a + b);
  }
}

inline bool jacobi2_ok(int n, bool single_precision) {
  return n >= 1 && n <= (single_precision ? JAC2_MAX_N_F32 : JAC2_MAX_N_F64);
}
// pair warps + enough workers for JAC2_ITEMS items each (rounded to warps)
inline int jacobi2_threads(int n) {
  const int np = n + (n & 1), m = np / 2;
  const int pw = (m + 31) / 32 * 32;
  const int total = m * (m + 1) / 2 + np * m;
  int w = (total + JAC2_ITEMS - 1) / JAC2_ITEMS;
  w = (w + 31) / 32 * 32;
  int t = pw + w;
  if (t < 64) t = 64;
  return t > 1024 ? 1024 : t;
}

// Same contract as jacobi_eigh (jacobi.cuh); falls back to it outside the shared-memory envelope.
inline int jacobi2_eigh(const double* G, int n, int ldg, double* w, double* V, double* scratch, int* info, cudaStream_t st,
                        bool single_precision = false, double loose_tol = 0.0) {
  if (!jacobi2_ok(n, single_precision)) return jacobi_eigh(G, n, ldg, w, V, scratch, info, st, single_precision, loose_tol);
  const int max_sweeps = 30;
  static PerDeviceFlag attr_done[3];
  if (!single_precision && n <= JAC2_MIXED_MAX_N && n >= 8) {
    const double tol = loose_tol > 0.0 ? loose_tol : 1e-14;
    const size_t smem = jac2_smem_bytes<double>(n) + jac2_smem_bytes<float>(n);
    TNB_CUDA(ensure_dyn_smem(attr_done[2], jacobi2_mixed_kernel,
                             (int)(jac2_smem_bytes<double>(JAC2_MIXED_MAX_N) + jac2_smem_bytes<float>(JAC2_MIXED_MAX_N))));
    jacobi2_mixed_kernel<<<1, jacobi2_threads(n), smem, st>>>(G, n, ldg, w, V, max_sweeps, tol, info);
    TNB_LAUNCH_CHECK();
    return TNB_OK;
  }
  if (single_precision) {
    const float tol = loose_tol > 0.0 ? (float)loose_tol : 2e-6f;
    TNB_CUDA(ensure_dyn_smem(attr_done[0], jacobi2_eigh_kernel<float>, (int)jac2_smem_bytes<float>(JAC2_MAX_N_F32)));
    jacobi2_eigh_kernel<float><<<1, jacobi2_threads(n), jac2_smem_bytes<float>(n), st>>>(G, n, ldg, w, V, max_sweeps, tol, info);
  } else {
    const double tol = loose_tol > 0.0 ? loose_tol : 1e-14;
    TNB_CUDA(ensure_dyn_smem(attr_done[1], jacobi2_eigh_kernel<double>, (int)jac2_smem_bytes<double>(JAC2_MAX_N_F64)));
    jacobi2_eigh_kernel<double><<<1, jacobi2_threads(n), jac2_smem_bytes<double>(n), st>>>(G, n, ldg, w, V, max_sweeps, tol, info);
  }
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

}  // namespace tnb

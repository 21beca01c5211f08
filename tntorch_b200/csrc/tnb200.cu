// tnb200 — single translation unit: C-ABI entry points declared in include/tnb200.h.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (see build.py)
#include "common.cuh"
#include "gemm_generic.cuh"
#include "jacobi.cuh"
#include "small_kernels.cuh"
#include "eig.cuh"
#include "gram_tc.cuh"
#include "gram_tc2.cuh"
#include "sweep.cuh"
#include "round_impl.cuh"
#include "cp_als.cuh"
#include "maxvol.cuh"
#include "qr.cuh"
#include "cross_kernels.cuh"
#include "peak_tf32.cuh"

using namespace tnb;

namespace {
inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline int check_dtype(int dtype) {
  if (dtype != TNB_F32 && dtype != TNB_F64) return fail(TNB_ERR_INVALID, "dtype must be TNB_F32 or TNB_F64, got %d", dtype);
  return TNB_OK;
}
inline int require_device() {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || !device_info().valid) {
    cudaGetLastError();
    return fail(TNB_ERR_CUDA, "no CUDA device available: tnb200 has no CPU fallback");
  }
  return TNB_OK;
}
// headroom for rank-dependent re-planning between the sizing pass (rank caps) and the run (actual ranks)
inline size_t with_slack(size_t bytes) { return bytes + bytes / 8 + (size_t)(4 << 20); }

// Workspace of a batch call: one slice of `one` bytes per tensor in flight, up to TNB_BATCH_MAX_INFLIGHT
// (measured on B200: 4 -> 171, 6 -> 172, 8 -> 175 GElements/s).
inline size_t batch_workspace_bytes(size_t one, int batch, size_t* per_tensor_bytes) {
  if (per_tensor_bytes) *per_tensor_bytes = one;
  if (one == 0 || batch < 1) return 0;
  return one * (size_t)std::min(batch, TNB_BATCH_MAX_INFLIGHT);
}

// Checks shared by the batch entry points once their dims are known (cores buffers of `need` elements, a workspace
// slice of `one` bytes per tensor, 0 for an unsupported shape), and how many tensors the workspace holds in flight.
inline int batch_inflight(const char* fn, int64_t cores_capacity, int64_t need, size_t one, size_t workspace_bytes,
                          int* inflight) {
  if (cores_capacity < need)
    return fail(TNB_ERR_WORKSPACE, "%s: cores buffers hold %lld elements, need %lld", fn, (long long)cores_capacity,
                (long long)need);
  if (one == 0) return fail(TNB_ERR_UNSUPPORTED, "%s: unsupported shape", fn);
  if (workspace_bytes < one) return fail(TNB_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, one);
  *inflight = (int)std::min<size_t>(workspace_bytes / one, (size_t)TNB_BATCH_MAX_INFLIGHT);
  return TNB_OK;
}
}  // namespace

extern "C" {

int tnb_version(void) { return 100; }
const char* tnb_last_error(void) { return last_error_ref().c_str(); }
uint64_t tnb_launch_count(void) { return launch_counter().load(); }
int tnb_has_tensorcore_path(void) { return tc_path_available() ? 1 : 0; }
void tnb_set_reserved_sms(int32_t n) { reserved_sms_ref().store(n); }

// ------------------------------------------------------------------ dense TT-SVD
int64_t tnb_ttsvd_cores_capacity(int ndim, const int64_t* shape, const int32_t* rmax, int64_t* core_offsets_host) {
  SweepDims d;
  if (make_dims(ndim, shape, rmax, d) != TNB_OK) return -1;
  if (core_offsets_host)
    for (int k = 0; k < ndim; ++k) core_offsets_host[k] = d.slot[k];
  return d.capacity;
}

size_t tnb_ttsvd_workspace_bytes(int dtype, int ndim, const int64_t* shape, const int32_t* rmax, uint32_t flags) {
  SweepDims d;
  if (check_dtype(dtype) != TNB_OK || make_dims(ndim, shape, rmax, d) != TNB_OK) return 0;
  ArenaSizer ar;
  int rc;
  if (dtype == TNB_F32)
    rc = ttsvd_impl<float>(ar, true, nullptr, d, rmax, 0.0, flags, nullptr, nullptr, nullptr, 0);
  else
    rc = ttsvd_impl<double>(ar, true, nullptr, d, rmax, 0.0, flags, nullptr, nullptr, nullptr, 0);
  if (rc != TNB_OK) return 0;
  return with_slack(ar.off);
}

int tnb_ttsvd(int dtype, const void* data, int ndim, const int64_t* shape, const int32_t* rmax, double eps,
              uint32_t flags, void* workspace, size_t workspace_bytes, void* cores, int64_t cores_capacity,
              int32_t* ranks_host, double* info_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!data || !shape || !cores || !ranks_host || !workspace) return fail(TNB_ERR_INVALID, "tnb_ttsvd: null argument");
  if (rmax)
    for (int k = 0; k < ndim - 1; ++k)
      if (rmax[k] < 0) return fail(TNB_ERR_INVALID, "rmax[%d] must be >= 1 (or 0 for none)", k);
  SweepDims d;
  TNB_TRY(make_dims(ndim, shape, rmax, d));
  if (cores_capacity < d.capacity)
    return fail(TNB_ERR_WORKSPACE, "tnb_ttsvd: cores buffer holds %lld elements, need %lld", (long long)cores_capacity,
                (long long)d.capacity);
  Arena ar(workspace, workspace_bytes);
  SweepInfo info;
  int rc;
  if (dtype == TNB_F32)
    rc = ttsvd_impl<float>(ar, false, static_cast<const float*>(data), d, rmax, eps, flags, static_cast<float*>(cores),
                           ranks_host, &info, as_stream(stream));
  else
    rc = ttsvd_impl<double>(ar, false, static_cast<const double*>(data), d, rmax, eps, flags,
                            static_cast<double*>(cores), ranks_host, &info, as_stream(stream));
  if (info_host) {
    for (int i = 0; i < 32; ++i) info_host[i] = 0.0;
    info_host[0] = info.norm;
    info_host[1] = info.eig_solves;
    info_host[2] = info.chfsi_products;
    info_host[3] = info.tc_grams;
    info_host[7] = info.nsteps;
    info_host[31] = info.fused_filters;
    info_host[29] = info.rr_sweeps;
    info_host[30] = info.rr_solves;
    info_host[26] = info.speculative;
    info_host[27] = info.spec_flags;
    for (int t = 0; t < info.nsteps && t < 6; ++t) {
      info_host[4] += info.gram_ms[t];
      info_host[5] += info.eig_ms[t];
      info_host[6] += info.factor_ms[t];
      info_host[8 + 3 * t] = info.gram_ms[t];
      info_host[9 + 3 * t] = info.eig_ms[t];
      info_host[10 + 3 * t] = info.factor_ms[t];
    }
  }
  return rc;
}

size_t tnb_ttsvd_batch_workspace_bytes(int dtype, int batch, int ndim, const int64_t* shape, const int32_t* rmax,
                                       uint32_t flags, size_t* per_tensor_bytes) {
  return batch_workspace_bytes(tnb_ttsvd_workspace_bytes(dtype, ndim, shape, rmax, flags), batch, per_tensor_bytes);
}

int tnb_ttsvd_batch(int dtype, const void* const* data, int batch, int ndim, const int64_t* shape, const int32_t* rmax,
                    double eps, uint32_t flags, void* workspace, size_t workspace_bytes, void* const* cores,
                    int64_t cores_capacity, int32_t* ranks_host, double* norms_host, int32_t* speculative_host,
                    void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (batch < 0 || (batch > 0 && (!data || !cores)) || !shape || !ranks_host || !workspace)
    return fail(TNB_ERR_INVALID, "tnb_ttsvd_batch: null argument");
  if (rmax)
    for (int k = 0; k < ndim - 1; ++k)
      if (rmax[k] < 0) return fail(TNB_ERR_INVALID, "rmax[%d] must be >= 1 (or 0 for none)", k);
  SweepDims d;
  TNB_TRY(make_dims(ndim, shape, rmax, d));
  for (int i = 0; i < batch; ++i)
    if (!data[i] || !cores[i]) return fail(TNB_ERR_INVALID, "tnb_ttsvd_batch: null tensor %d", i);
  const size_t one = tnb_ttsvd_workspace_bytes(dtype, ndim, shape, rmax, flags);
  int inflight;
  TNB_TRY(batch_inflight("tnb_ttsvd_batch", cores_capacity, d.capacity, one, workspace_bytes, &inflight));
  if (dtype == TNB_F32)
    return ttsvd_batch_impl<float>(workspace, one, inflight, reinterpret_cast<const float* const*>(data), batch, d, rmax, eps,
                                   flags, reinterpret_cast<float* const*>(cores), ranks_host, norms_host, speculative_host,
                                   as_stream(stream));
  return ttsvd_batch_impl<double>(workspace, one, inflight, reinterpret_cast<const double* const*>(data), batch, d, rmax, eps,
                                  flags, reinterpret_cast<double* const*>(cores), ranks_host, norms_host, speculative_host,
                                  as_stream(stream));
}

int tnb_ttsvd_host(int dtype, const void* data_host, int ndim, const int64_t* shape, const int32_t* rmax, double eps,
                   uint32_t flags, void* device_buffer, void* workspace, size_t workspace_bytes, void* cores_dev,
                   int64_t cores_capacity, void* cores_host, int32_t* ranks_host, double* info_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!data_host || !device_buffer || !cores_host) return fail(TNB_ERR_INVALID, "tnb_ttsvd_host: null argument");
  SweepDims d;
  TNB_TRY(make_dims(ndim, shape, rmax, d));
  const size_t esz = dtype == TNB_F32 ? 4 : 8;
  const size_t total = (size_t)d.rows[ndim] * esz;
  cudaStream_t st = as_stream(stream);
  // chunked so that a pageable source still overlaps its staging copies with the DMA
  const size_t chunk = (size_t)256 << 20;
  for (size_t off = 0; off < total; off += chunk) {
    const size_t nb = total - off < chunk ? total - off : chunk;
    TNB_CUDA(cudaMemcpyAsync(static_cast<char*>(device_buffer) + off, static_cast<const char*>(data_host) + off, nb,
                             cudaMemcpyHostToDevice, st));
  }
  TNB_TRY(tnb_ttsvd(dtype, device_buffer, ndim, shape, rmax, eps, flags, workspace, workspace_bytes, cores_dev,
                    cores_capacity, ranks_host, info_host, stream));
  TNB_CUDA(cudaMemcpyAsync(cores_host, cores_dev, (size_t)d.capacity * esz, cudaMemcpyDeviceToHost, st));
  TNB_CUDA(cudaStreamSynchronize(st));
  return TNB_OK;
}

// ------------------------------------------------------------------ TT rounding
int64_t tnb_tt_round_cores_capacity(int ndim, const int64_t* shape, const int32_t* ranks_in, const int32_t* rmax,
                                    int64_t* core_offsets_host) {
  RoundDims d;
  if (make_round_dims(ndim, shape, ranks_in, rmax, d) != TNB_OK) return -1;
  if (core_offsets_host)
    for (int k = 0; k < ndim; ++k) core_offsets_host[k] = d.slot[k];
  return d.capacity;
}

size_t tnb_tt_round_workspace_bytes(int dtype, int ndim, const int64_t* shape, const int32_t* ranks_in,
                                    const int32_t* rmax) {
  RoundDims d;
  if (check_dtype(dtype) != TNB_OK || make_round_dims(ndim, shape, ranks_in, rmax, d) != TNB_OK) return 0;
  ArenaSizer ar;
  int rc;
  if (dtype == TNB_F32)
    rc = tt_round_any<float>(ar, true, nullptr, d, rmax, 0.0, 0, nullptr, nullptr, 0);
  else
    rc = tt_round_any<double>(ar, true, nullptr, d, rmax, 0.0, 0, nullptr, nullptr, 0);
  if (rc != TNB_OK) return 0;
  return with_slack(ar.off);
}

int tnb_tt_round(int dtype, const void* const* cores_in, int ndim, const int64_t* shape, const int32_t* ranks_in,
                 const int32_t* rmax, double eps, uint32_t flags, void* workspace, size_t workspace_bytes,
                 void* cores_out, int64_t cores_capacity, int32_t* ranks_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!cores_in || !shape || !ranks_in || !cores_out || !ranks_host || !workspace)
    return fail(TNB_ERR_INVALID, "tnb_tt_round: null argument");
  RoundDims d;
  TNB_TRY(make_round_dims(ndim, shape, ranks_in, rmax, d));
  if (cores_capacity < d.capacity)
    return fail(TNB_ERR_WORKSPACE, "tnb_tt_round: cores buffer holds %lld elements, need %lld",
                (long long)cores_capacity, (long long)d.capacity);
  Arena ar(workspace, workspace_bytes);
  if (dtype == TNB_F32)
    return tt_round_any<float>(ar, false, reinterpret_cast<const float* const*>(cores_in), d, rmax, eps, flags,
                               static_cast<float*>(cores_out), ranks_host, as_stream(stream));
  return tt_round_any<double>(ar, false, reinterpret_cast<const double* const*>(cores_in), d, rmax, eps, flags,
                              static_cast<double*>(cores_out), ranks_host, as_stream(stream));
}

size_t tnb_tt_round_batch_workspace_bytes(int dtype, int batch, int ndim, const int64_t* shape, const int32_t* ranks_in,
                                          const int32_t* rmax, size_t* per_tensor_bytes) {
  return batch_workspace_bytes(tnb_tt_round_workspace_bytes(dtype, ndim, shape, ranks_in, rmax), batch, per_tensor_bytes);
}

int tnb_tt_round_batch(int dtype, const void* const* cores_in, int batch, int ndim, const int64_t* shape,
                       const int32_t* ranks_in, const int32_t* rmax, double eps, uint32_t flags, void* workspace,
                       size_t workspace_bytes, void* const* cores_out, int64_t cores_capacity, int32_t* ranks_host,
                       int32_t* speculative_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (batch < 0 || (batch > 0 && (!cores_in || !cores_out)) || !shape || !ranks_in || !ranks_host || !workspace)
    return fail(TNB_ERR_INVALID, "tnb_tt_round_batch: null argument");
  RoundDims d;
  TNB_TRY(make_round_dims(ndim, shape, ranks_in, rmax, d));
  const size_t one = tnb_tt_round_workspace_bytes(dtype, ndim, shape, ranks_in, rmax);
  int inflight;
  TNB_TRY(batch_inflight("tnb_tt_round_batch", cores_capacity, d.capacity, one, workspace_bytes, &inflight));
  if (dtype == TNB_F32)
    return tt_round_batch_impl<float>(workspace, one, inflight, reinterpret_cast<const float* const*>(cores_in), batch, d, rmax,
                                      eps, flags, reinterpret_cast<float* const*>(cores_out), ranks_host, speculative_host,
                                      as_stream(stream));
  return tt_round_batch_impl<double>(workspace, one, inflight, reinterpret_cast<const double* const*>(cores_in), batch, d, rmax,
                                     eps, flags, reinterpret_cast<double* const*>(cores_out), ranks_host, speculative_host,
                                     as_stream(stream));
}

// ------------------------------------------------------------------ sums of TT tensors (+ fused rounding)
int64_t tnb_tt_sum_cores_capacity(int noperands, int ndim, const int64_t* shape, const int32_t* ranks_in,
                                  int32_t* ranks_sum_host, int64_t* core_offsets_host) {
  SumDims d;
  if (!shape || !ranks_in || make_sum_dims(noperands, ndim, shape, ranks_in, d) != TNB_OK) return -1;
  if (ranks_sum_host)
    for (int n = 0; n <= ndim; ++n) ranks_sum_host[n] = d.rsum[n];
  if (core_offsets_host)
    for (int n = 0; n < ndim; ++n) core_offsets_host[n] = d.slot[n];
  return d.capacity;
}

int tnb_tt_sum(int dtype, const void* const* cores_in, int noperands, const double* alpha, int ndim, const int64_t* shape,
               const int32_t* ranks_in, void* cores_out, int64_t cores_capacity, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!cores_in || !shape || !ranks_in || !cores_out) return fail(TNB_ERR_INVALID, "tnb_tt_sum: null argument");
  SumDims d;
  TNB_TRY(make_sum_dims(noperands, ndim, shape, ranks_in, d));
  if (cores_capacity < d.capacity) return fail(TNB_ERR_WORKSPACE, "tnb_tt_sum: cores buffer too small");
  if (dtype == TNB_F32)
    return tt_sum_assemble<float>(reinterpret_cast<const float* const*>(cores_in), alpha, d, static_cast<float*>(cores_out), as_stream(stream));
  return tt_sum_assemble<double>(reinterpret_cast<const double* const*>(cores_in), alpha, d, static_cast<double*>(cores_out), as_stream(stream));
}

static int sum_round_dims(int noperands, int ndim, const int64_t* shape, const int32_t* ranks_in, const int32_t* rmax, SumDims& sd,
                          RoundDims& rd) {
  TNB_TRY(make_sum_dims(noperands, ndim, shape, ranks_in, sd));
  return make_round_dims(ndim, shape, sd.rsum.data(), rmax, rd);
}

int64_t tnb_tt_sum_round_cores_capacity(int noperands, int ndim, const int64_t* shape, const int32_t* ranks_in,
                                        const int32_t* rmax, int64_t* core_offsets_host) {
  SumDims sd;
  RoundDims rd;
  if (!shape || !ranks_in || sum_round_dims(noperands, ndim, shape, ranks_in, rmax, sd, rd) != TNB_OK) return -1;
  if (core_offsets_host)
    for (int k = 0; k < ndim; ++k) core_offsets_host[k] = rd.slot[k];
  return rd.capacity;
}

size_t tnb_tt_sum_round_workspace_bytes(int dtype, int noperands, int ndim, const int64_t* shape, const int32_t* ranks_in,
                                        const int32_t* rmax) {
  SumDims sd;
  RoundDims rd;
  if (check_dtype(dtype) != TNB_OK || !shape || !ranks_in || sum_round_dims(noperands, ndim, shape, ranks_in, rmax, sd, rd) != TNB_OK)
    return 0;
  const size_t inner = tnb_tt_round_workspace_bytes(dtype, ndim, shape, sd.rsum.data(), rmax);
  if (inner == 0) return 0;
  return inner + align_up((size_t)sd.capacity * (dtype == TNB_F32 ? 4 : 8)) + 256;
}

int tnb_tt_sum_round(int dtype, const void* const* cores_in, int noperands, const double* alpha, int ndim, const int64_t* shape,
                     const int32_t* ranks_in, const int32_t* rmax, double eps, uint32_t flags, void* workspace,
                     size_t workspace_bytes, void* cores_out, int64_t cores_capacity, int32_t* ranks_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!cores_in || !shape || !ranks_in || !cores_out || !ranks_host || !workspace)
    return fail(TNB_ERR_INVALID, "tnb_tt_sum_round: null argument");
  SumDims sd;
  RoundDims rd;
  TNB_TRY(sum_round_dims(noperands, ndim, shape, ranks_in, rmax, sd, rd));
  if (cores_capacity < rd.capacity) return fail(TNB_ERR_WORKSPACE, "tnb_tt_sum_round: cores buffer too small");
  const size_t esz = dtype == TNB_F32 ? 4 : 8;
  const size_t abytes = align_up((size_t)sd.capacity * esz);
  if (workspace_bytes < abytes) return fail(TNB_ERR_WORKSPACE, "tnb_tt_sum_round: workspace too small");
  char* base = static_cast<char*>(workspace);
  std::vector<const void*> ptrs(ndim);
  cudaStream_t st = as_stream(stream);
  if (dtype == TNB_F32) {
    TNB_TRY(tt_sum_assemble<float>(reinterpret_cast<const float* const*>(cores_in), alpha, sd, reinterpret_cast<float*>(base), st));
    for (int n = 0; n < ndim; ++n) ptrs[n] = reinterpret_cast<float*>(base) + sd.slot[n];
  } else {
    TNB_TRY(tt_sum_assemble<double>(reinterpret_cast<const double* const*>(cores_in), alpha, sd, reinterpret_cast<double*>(base), st));
    for (int n = 0; n < ndim; ++n) ptrs[n] = reinterpret_cast<double*>(base) + sd.slot[n];
  }
  return tnb_tt_round(dtype, ptrs.data(), ndim, shape, sd.rsum.data(), rmax, eps, flags, base + abytes, workspace_bytes - abytes,
                      cores_out, cores_capacity, ranks_host, stream);
}

int tnb_tt_hadamard(int dtype, const void* const* cores_a, const void* const* cores_b, int ndim, const int64_t* shape,
                    const int32_t* ranks_a, const int32_t* ranks_b, void* const* cores_out, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!cores_a || !cores_b || !shape || !ranks_a || !ranks_b || !cores_out || ndim < 1)
    return fail(TNB_ERR_INVALID, "tnb_tt_hadamard: null argument");
  cudaStream_t st = as_stream(stream);
  for (int n = 0; n < ndim; ++n) {
    const int ra0 = ranks_a[n], ra1 = ranks_a[n + 1], rb0 = ranks_b[n], rb1 = ranks_b[n + 1];
    if (ra0 < 1 || ra1 < 1 || rb0 < 1 || rb1 < 1 || shape[n] < 1 || !cores_a[n] || !cores_b[n] || !cores_out[n])
      return fail(TNB_ERR_INVALID, "tnb_tt_hadamard: bad core %d", n);
    const int64_t total = (int64_t)ra0 * rb0 * shape[n] * ra1 * rb1;
    if (dtype == TNB_F32)
      tt_hadamard_core_kernel<float><<<grid_for(total), 256, 0, st>>>(static_cast<const float*>(cores_a[n]), static_cast<const float*>(cores_b[n]),
                                                                      ra0, ra1, rb0, rb1, (int)shape[n], static_cast<float*>(cores_out[n]));
    else
      tt_hadamard_core_kernel<double><<<grid_for(total), 256, 0, st>>>(static_cast<const double*>(cores_a[n]), static_cast<const double*>(cores_b[n]),
                                                                       ra0, ra1, rb0, rb1, (int)shape[n], static_cast<double*>(cores_out[n]));
    TNB_LAUNCH_CHECK();
  }
  return TNB_OK;
}

// ------------------------------------------------------------------ truncated_svd
size_t tnb_truncated_svd_workspace_bytes(int dtype, int64_t m, int64_t n) {
  if (check_dtype(dtype) != TNB_OK || m < 1 || n < 1) return 0;
  ArenaSizer ar;
  int rc;
  // sized for the worst admissible request (rmax up to the subspace-solver limit)
  const int32_t rmax_cap = JACOBI_MAX_N - 16;
  if (dtype == TNB_F32)
    rc = truncated_svd_impl<float>(ar, true, nullptr, m, n, -1, -1, rmax_cap, 1, nullptr, nullptr, nullptr, 0);
  else
    rc = truncated_svd_impl<double>(ar, true, nullptr, m, n, -1, -1, rmax_cap, 1, nullptr, nullptr, nullptr, 0);
  if (rc != TNB_OK) return 0;
  return with_slack(ar.off);
}

int tnb_truncated_svd(int dtype, const void* M, int64_t m, int64_t n, double delta, double eps, int32_t rmax,
                      int left_ortho, void* workspace, size_t workspace_bytes, void* left, void* right,
                      int32_t* rank_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!M || !left || !right || !rank_host || !workspace) return fail(TNB_ERR_INVALID, "tnb_truncated_svd: null argument");
  if (m < 1 || n < 1) return fail(TNB_ERR_INVALID, "tnb_truncated_svd: empty matrix");
  if (delta >= 0 && eps >= 0) return fail(TNB_ERR_INVALID, "Provide either `delta` or `eps`");  // round.py:77-78
  if (rmax < 0) return fail(TNB_ERR_INVALID, "rmax must be >= 1");                               // round.py:85
  Arena ar(workspace, workspace_bytes);
  if (dtype == TNB_F32)
    return truncated_svd_impl<float>(ar, false, static_cast<const float*>(M), m, n, delta, eps, rmax, left_ortho,
                                     static_cast<float*>(left), static_cast<float*>(right), rank_host, as_stream(stream));
  return truncated_svd_impl<double>(ar, false, static_cast<const double*>(M), m, n, delta, eps, rmax, left_ortho,
                                    static_cast<double*>(left), static_cast<double*>(right), rank_host,
                                    as_stream(stream));
}

// ------------------------------------------------------------------ CP-ALS
int64_t tnb_cp_als_factors_capacity(int ndim, const int64_t* shape, int32_t R, int64_t* factor_offsets_host) {
  CpDims d;
  if (make_cp_dims(ndim, shape, R, d) != TNB_OK) return -1;
  if (factor_offsets_host)
    for (int n = 0; n < ndim; ++n) factor_offsets_host[n] = d.foff[n];
  return d.ftotal;
}

size_t tnb_cp_als_workspace_bytes(int dtype, int ndim, const int64_t* shape, int32_t R) {
  CpDims d;
  if (check_dtype(dtype) != TNB_OK || make_cp_dims(ndim, shape, R, d) != TNB_OK) return 0;
  ArenaSizer ar;
  int rc;
  if (dtype == TNB_F32)
    rc = cp_als_impl<float>(ar, true, nullptr, d, R, 1, 0.0, nullptr, nullptr, nullptr, 0);
  else
    rc = cp_als_impl<double>(ar, true, nullptr, d, R, 1, 0.0, nullptr, nullptr, nullptr, 0);
  return rc == TNB_OK ? with_slack(ar.off) : 0;
}

int tnb_cp_als(int dtype, const void* data, int ndim, const int64_t* shape, int32_t R, int32_t max_iter, double tol,
               void* workspace, size_t workspace_bytes, void* factors, int64_t factors_capacity, double* errors_host,
               int32_t* iters_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!data || !shape || !workspace || !factors) return fail(TNB_ERR_INVALID, "tnb_cp_als: null argument");
  if (max_iter < 0) return fail(TNB_ERR_INVALID, "tnb_cp_als: max_iter < 0");
  CpDims d;
  TNB_TRY(make_cp_dims(ndim, shape, R, d));
  if (factors_capacity < d.ftotal) return fail(TNB_ERR_WORKSPACE, "tnb_cp_als: factor buffer too small");
  Arena ar(workspace, workspace_bytes);
  if (dtype == TNB_F32)
    return cp_als_impl<float>(ar, false, static_cast<const float*>(data), d, R, max_iter, tol,
                              static_cast<float*>(factors), errors_host, iters_host, as_stream(stream));
  return cp_als_impl<double>(ar, false, static_cast<const double*>(data), d, R, max_iter, tol,
                             static_cast<double*>(factors), errors_host, iters_host, as_stream(stream));
}

int tnb_cp_als_from(int dtype, const void* data, int ndim, const int64_t* shape, int32_t R, int32_t max_iter, double tol,
                    void* workspace, size_t workspace_bytes, void* factors, int64_t factors_capacity, double* errors_host,
                    int32_t* iters_host, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!data || !shape || !workspace || !factors) return fail(TNB_ERR_INVALID, "tnb_cp_als_from: null argument");
  if (max_iter < 0) return fail(TNB_ERR_INVALID, "tnb_cp_als_from: max_iter < 0");
  CpDims d;
  TNB_TRY(make_cp_dims(ndim, shape, R, d));
  if (factors_capacity < d.ftotal) return fail(TNB_ERR_WORKSPACE, "tnb_cp_als_from: factor buffer too small");
  Arena ar(workspace, workspace_bytes);
  if (dtype == TNB_F32)
    return cp_als_impl<float>(ar, false, static_cast<const float*>(data), d, R, max_iter, tol,
                              static_cast<float*>(factors), errors_host, iters_host, as_stream(stream), true);
  return cp_als_impl<double>(ar, false, static_cast<const double*>(data), d, R, max_iter, tol,
                             static_cast<double*>(factors), errors_host, iters_host, as_stream(stream), true);
}


// ------------------------------------------------------------------ maxvol
size_t tnb_maxvol_workspace_bytes(int32_t nbatch, int32_t N, int32_t r) {
  if (nbatch < 1 || N < 1 || r < 1) return 0;
  return maxvol_workspace_bytes(nbatch, N, r) + 256;
}

int tnb_maxvol(const double* A, int32_t nbatch, int32_t N, int32_t r, double tol, int32_t max_iters, void* workspace,
               size_t workspace_bytes, int32_t* index_dev, double* C_dev, int32_t* iters_host, void* stream) {
  TNB_TRY(require_device());
  if (!A || !workspace || !index_dev || !C_dev) return fail(TNB_ERR_INVALID, "tnb_maxvol: null argument");
  return maxvol_run(A, nbatch, N, r, tol, max_iters, workspace, workspace_bytes, index_dev, C_dev, iters_host,
                    as_stream(stream));
}

size_t tnb_rect_maxvol_workspace_bytes(int32_t nbatch, int32_t N, int32_t r, int32_t maxK) {
  if (nbatch < 1 || N < 1 || r < 1 || maxK < r) return 0;
  return rect_maxvol_workspace_bytes(nbatch, N, r, maxK) + 256;
}

int tnb_rect_maxvol(const double* A, int32_t nbatch, int32_t N, int32_t r, double tol, int32_t minK, int32_t maxK,
                    int32_t start_maxvol_iters, void* workspace, size_t workspace_bytes, int32_t* index_dev, double* C_dev,
                    int32_t* K_dev, void* stream) {
  TNB_TRY(require_device());
  if (!A || !workspace || !index_dev || !C_dev || !K_dev) return fail(TNB_ERR_INVALID, "tnb_rect_maxvol: null argument");
  return rect_maxvol_run(A, nbatch, N, r, tol, minK, maxK, start_maxvol_iters, workspace, workspace_bytes, index_dev, C_dev,
                         K_dev, as_stream(stream));
}

// ------------------------------------------------------------------ batched TT-cross plumbing
int tnb_cross_gather_coords(const int32_t* lsets, const int32_t* rsets, const double* grid, int32_t Imax, int32_t B,
                            int32_t N, int32_t j, int32_t Rl, int32_t I, int32_t Rr, double* X, void* stream) {
  TNB_TRY(require_device());
  if (!grid || !X || B < 1 || N < 1 || j < 0 || j >= N || Rl < 1 || I < 1 || Rr < 1 || (j > 0 && !lsets) || (j < N - 1 && !rsets))
    return fail(TNB_ERR_INVALID, "tnb_cross_gather_coords: bad argument");
  const int64_t total = (int64_t)B * Rl * I * Rr;
  cross_gather_coords_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(lsets, rsets, grid, Imax, B, N, j, Rl, I, Rr, X);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

int tnb_cross_update_lsets(const int32_t* lsets, const int32_t* local, int32_t B, int32_t j, int32_t Rl, int32_t I,
                           int32_t Rn, const int32_t* active, int32_t* lnext, void* stream) {
  TNB_TRY(require_device());
  if (!local || !lnext || B < 1 || j < 0 || Rl < 1 || I < 1 || Rn < 1 || (j > 0 && !lsets))
    return fail(TNB_ERR_INVALID, "tnb_cross_update_lsets: bad argument");
  cross_update_lsets_kernel<<<grid_for((int64_t)B * Rn), 256, 0, as_stream(stream)>>>(lsets, local, B, j, Rl, I, Rn, active, lnext);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

int tnb_cross_update_rsets(const int32_t* rsets, const int32_t* local, int32_t B, int32_t N, int32_t j, int32_t I,
                           int32_t Rr, int32_t Rp, const int32_t* active, int32_t* rprev, void* stream) {
  TNB_TRY(require_device());
  if (!local || !rprev || B < 1 || N < 1 || j < 1 || j >= N || I < 1 || Rr < 1 || Rp < 1 || (j < N - 1 && !rsets))
    return fail(TNB_ERR_INVALID, "tnb_cross_update_rsets: bad argument");
  cross_update_rsets_kernel<<<grid_for((int64_t)B * Rp), 256, 0, as_stream(stream)>>>(rsets, local, B, N, j, I, Rr, Rp, active, rprev);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

int tnb_cross_tt_eval(const double* const* cores, int32_t N, const int32_t* ranks, const int32_t* shape, const int32_t* idx,
                      int32_t B, int32_t P, int32_t per_problem, double* out, void* stream) {
  TNB_TRY(require_device());
  if (!cores || !ranks || !shape || !idx || !out || N < 1 || N > 32 || B < 1 || P < 1)
    return fail(TNB_ERR_INVALID, "tnb_cross_tt_eval: bad argument");
  CrossEvalArgs a;
  a.N = N;
  for (int n = 0; n < N; ++n) {
    if (!cores[n] || ranks[n] < 1 || ranks[n] > CROSS_EVAL_MAX_R || shape[n] < 1)
      return fail(TNB_ERR_UNSUPPORTED, "tnb_cross_tt_eval: rank %d outside [1, %d]", (int)ranks[n], CROSS_EVAL_MAX_R);
    a.cores[n] = cores[n];
    a.R[n] = ranks[n];
    a.I[n] = shape[n];
  }
  if (ranks[N] != 1 || ranks[0] != 1) return fail(TNB_ERR_INVALID, "tnb_cross_tt_eval: boundary ranks must be 1");
  a.R[N] = 1;
  cross_tt_eval_kernel<<<grid_for((int64_t)B * P, 128), 128, 0, as_stream(stream)>>>(a, idx, B, P, per_problem, out);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

int tnb_measure_tf32_peak(int32_t reps, int32_t per_commit, int32_t trials, double* tflops_host, double* ms_host, void* stream) {
  TNB_TRY(require_device());
  if (!tflops_host || reps < 1 || per_commit < 1 || trials < 1) return fail(TNB_ERR_INVALID, "tnb_measure_tf32_peak: bad argument");
  return measure_tf32_peak(reps, per_commit, trials, tflops_host, ms_host, as_stream(stream));
}

int tnb_matmul(int dtype, const void* A, const void* B, void* C, int64_t M, int64_t N, int64_t K, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!A || !B || !C || M < 1 || N < 1 || K < 1) return fail(TNB_ERR_INVALID, "tnb_matmul: bad argument");
  cudaStream_t st = as_stream(stream);
  if (dtype == TNB_F32)
    return gemm_direct<float, float, float, float>(M, N, K, static_cast<const float*>(A), K, true, static_cast<const float*>(B),
                                                   N, false, static_cast<float*>(C), N, 1.f, nullptr, 0, 0.f, nullptr, 0, 0.f, st);
  return gemm_direct<double, double, double, double>(M, N, K, static_cast<const double*>(A), K, true,
                                                     static_cast<const double*>(B), N, false, static_cast<double*>(C), N, 1.0,
                                                     nullptr, 0, 0.0, nullptr, 0, 0.0, st);
}

size_t tnb_qr_workspace_bytes(int32_t nbatch, int32_t rows, int32_t n) {
  if (nbatch < 1 || rows < 1 || n < 1) return 0;
  return householder_qr_workspace_bytes(nbatch, rows, n) + 256;
}

int tnb_qr_householder(const double* A, int32_t nbatch, int32_t rows, int32_t n, void* workspace, size_t workspace_bytes,
                       double* Q, double* R, void* stream) {
  TNB_TRY(require_device());
  if (!A || !workspace || !Q) return fail(TNB_ERR_INVALID, "tnb_qr_householder: null argument");
  return householder_qr_run(A, nbatch, rows, n, workspace, workspace_bytes, Q, R, as_stream(stream));
}

// ------------------------------------------------------------------ building blocks
size_t tnb_gram_workspace_bytes(int dtype, int64_t rows, int64_t n) {
  if (check_dtype(dtype) != TNB_OK || rows < 1 || n < 1) return 0;
  GemmPlan pl = plan_gemm(n, n, rows, true);
  return align_up(pl.partial_elems * sizeof(double)) + 256;
}

int tnb_gram(int dtype, const void* A, int64_t rows, int64_t n, double* G, void* workspace, size_t workspace_bytes,
             void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!A || !G || !workspace || rows < 1 || n < 1) return fail(TNB_ERR_INVALID, "tnb_gram: bad argument");
  GemmPlan pl = plan_gemm(n, n, rows, true);
  if (workspace_bytes < pl.partial_elems * sizeof(double)) return fail(TNB_ERR_WORKSPACE, "tnb_gram: workspace too small");
  double* partial = static_cast<double*>(workspace);
  cudaStream_t st = as_stream(stream);
  if (dtype == TNB_F32)
    return gemm_splitk<float, float, double, double, float>(pl, n, n, rows, static_cast<const float*>(A), n, false,
                                                            static_cast<const float*>(A), n, false, partial, G, n, 1.0,
                                                            nullptr, 0, 0.0, nullptr, 0, 0.0, true, (float*)nullptr, 0, st);
  return gemm_splitk<double, double, double, double, float>(pl, n, n, rows, static_cast<const double*>(A), n, false,
                                                            static_cast<const double*>(A), n, false, partial, G, n, 1.0,
                                                            nullptr, 0, 0.0, nullptr, 0, 0.0, true, (float*)nullptr, 0, st);
}

size_t tnb_gram_tc_workspace_bytes(int64_t rows, int64_t n) {
  if (!gram_tc_shape_ok(rows, n)) return 0;
  size_t b = gram_tc_workspace_bytes(rows, n);
  if (gram_tc2_shape_ok(rows, n)) b = std::max(b, gram_tc2_workspace_bytes(rows, n));
  return b + 256;
}

int tnb_gram_tc_f32(const float* A, int64_t rows, int64_t n, double* G, void* workspace, size_t workspace_bytes,
                    void* stream) {
  TNB_TRY(require_device());
  if (!A || !G || !workspace) return fail(TNB_ERR_INVALID, "tnb_gram_tc_f32: null argument");
  if (gram_tc2_shape_ok(rows, n)) return gram_tc2_f32(A, rows, n, G, nullptr, workspace, workspace_bytes, as_stream(stream));
  return gram_tc_f32(A, rows, n, G, nullptr, workspace, workspace_bytes, as_stream(stream));
}

size_t tnb_atb_tc_workspace_bytes(int64_t K, int64_t m, int64_t n) {
  if (!atb_tc_shape_ok(K, m, n)) return 0;
  return atb_tc_workspace_bytes(K, m, n) + 256;
}

int tnb_atb_tc_f32(const float* A, int64_t K, int64_t m, const float* B, int64_t n, float* C, float alpha,
                   const float* D, float beta, void* workspace, size_t workspace_bytes, void* stream) {
  TNB_TRY(require_device());
  if (!A || !B || !C || !workspace) return fail(TNB_ERR_INVALID, "tnb_atb_tc_f32: null argument");
  return atb_tc_f32(A, K, m, B, n, C, (int)n, alpha, D, (int)n, beta, nullptr, 0, 0.f, workspace, workspace_bytes,
                    as_stream(stream));
}

size_t tnb_cheb_filter_workspace_bytes(int32_t n, int32_t b) {
  if (n < 256 || n % 256 != 0 || b < 8 || b > 128) return 0;
  return cheb_filter_workspace_bytes(n, b);
}

int tnb_cheb_filter_f32(const float* G, int32_t n, int32_t b, float* buf0, float* buf1, float* buf2, int32_t steps,
                        const float* a_host, const float* bc_host, const float* g_host, void* workspace,
                        size_t workspace_bytes, void* stream) {
  TNB_TRY(require_device());
  if (!G || !buf0 || !buf1 || !buf2 || !a_host || !bc_host || !g_host || !workspace)
    return fail(TNB_ERR_INVALID, "tnb_cheb_filter_f32: null argument");
  float* bufs[3] = {buf0, buf1, buf2};
  const int rc = cheb_filter_f32(G, n, b, bufs, steps, a_host, bc_host, g_host, workspace, workspace_bytes,
                                 as_stream(stream));
  return rc;  // TNB_ERR_UNSUPPORTED carries the reason in tnb_last_error()
}

int tnb_project(int dtype, const void* A, int64_t rows, int64_t n, const void* V, int32_t r, void* C, void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!A || !V || !C || rows < 1 || n < 1 || r < 1) return fail(TNB_ERR_INVALID, "tnb_project: bad argument");
  cudaStream_t st = as_stream(stream);
  if (dtype == TNB_F32)
    return project_any<float>(static_cast<const float*>(A), rows, n, static_cast<const float*>(V), r,
                              static_cast<float*>(C), st);
  return project_any<double>(static_cast<const double*>(A), rows, n, static_cast<const double*>(V), r,
                             static_cast<double*>(C), st);
}

size_t tnb_project_tc_workspace_bytes(int64_t n, int32_t r) {
  if (n < 32 || n % 4 != 0 || r < 1 || r > PT_MAX_N) return 0;
  return project_tc_workspace_bytes(n, r) + 256;
}

int tnb_project_tc_f32(const float* A, int64_t rows, int64_t n, const float* V, int32_t r, float* C, void* workspace,
                       size_t workspace_bytes, void* stream) {
  TNB_TRY(require_device());
  if (!A || !V || !C || !workspace) return fail(TNB_ERR_INVALID, "tnb_project_tc_f32: null argument");
  return project_tc_f32(A, rows, n, V, r, C, workspace, workspace_bytes, as_stream(stream));
}

size_t tnb_eigh_workspace_bytes(int32_t n) {
  if (n < 1 || n > JACOBI_MAX_N) return 0;
  return align_up(jacobi_scratch_doubles(n) * sizeof(double)) + 256;
}

int tnb_eigh_jacobi(const double* G, int32_t n, double* w, double* V, void* workspace, size_t workspace_bytes,
                    void* stream) {
  TNB_TRY(require_device());
  if (!G || !w || !V || !workspace) return fail(TNB_ERR_INVALID, "tnb_eigh_jacobi: null argument");
  if (n < 1 || n > JACOBI_MAX_N) return fail(TNB_ERR_UNSUPPORTED, "tnb_eigh_jacobi: n=%d outside [1,%d]", n, JACOBI_MAX_N);
  Arena ar(workspace, workspace_bytes);
  double* js = ar.take<double>(jacobi_scratch_doubles(n));
  int* jinfo = ar.take<int>(4);
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tnb_eigh_jacobi: workspace too small");
  return jacobi2_eigh(G, n, n, w, V, js, jinfo, as_stream(stream));
}

size_t tnb_eig_topk_workspace_bytes(int32_t n, int32_t k, int32_t b) {
  if (n < 1 || k < 1) return 0;
  if (b <= 0) b = chfsi_default_block(n, k);
  ArenaSizer ar;
  ChfsiWork<double> w;
  chfsi_carve<double>(ar, n, b, w);
  return ar.off + 4096;
}

int tnb_eig_topk(const double* G, int32_t n, int32_t k, int32_t b, double tol, double* w, double* V, void* workspace,
                 size_t workspace_bytes, double* info_host, void* stream) {
  TNB_TRY(require_device());
  if (!G || !w || !V || !workspace) return fail(TNB_ERR_INVALID, "tnb_eig_topk: null argument");
  if (b <= 0) b = chfsi_default_block(n, k);
  if (k < 1 || k > b || b > n) return fail(TNB_ERR_INVALID, "tnb_eig_topk: need 1 <= k <= b <= n");
  Arena ar(workspace, workspace_bytes);
  ChfsiWork<double> cw;
  chfsi_carve<double>(ar, n, b, cw);
  double* d_trace = ar.take<double>(4);
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tnb_eig_topk: workspace too small");
  cudaStream_t st = as_stream(stream);
  SweepScalars* sc = reinterpret_cast<SweepScalars*>(ar.take<SweepScalars>(1));
  if (!ar.ok) return fail(TNB_ERR_WORKSPACE, "tnb_eig_topk: workspace too small");
  trace_kernel<<<1, 256, 0, st>>>(G, n, n, sc, 0, 0.0);
  TNB_LAUNCH_CHECK();
  (void)d_trace;
  ChfsiStats cs;
  int rc = eig_topk_chfsi<double>(G, n, k, b, &sc->trace, tol > 0 ? tol : 1e-6, cw, w, V, &cs, st);
  if (info_host) {
    info_host[0] = cs.products;
    info_host[1] = cs.outer;
    info_host[2] = cs.converged;
  }
  if (rc == TNB_OK) TNB_CUDA(cudaStreamSynchronize(st));
  return rc;
}

size_t tnb_tt_relative_error_workspace_bytes(int dtype, int ndim, const int64_t* shape, const int32_t* ranks) {
  if (check_dtype(dtype) != TNB_OK || ndim < 2) return 0;
  ArenaSizer ar;
  int rc;
  if (dtype == TNB_F32)
    rc = tt_relative_error_impl<float>(ar, true, nullptr, nullptr, ndim, shape, ranks, nullptr, 0);
  else
    rc = tt_relative_error_impl<double>(ar, true, nullptr, nullptr, ndim, shape, ranks, nullptr, 0);
  return rc == TNB_OK ? ar.off + 4096 : 0;
}

int tnb_tt_relative_error(int dtype, const void* data, const void* const* cores, int ndim, const int64_t* shape,
                          const int32_t* ranks, void* workspace, size_t workspace_bytes, double* result_host,
                          void* stream) {
  TNB_TRY(check_dtype(dtype));
  TNB_TRY(require_device());
  if (!data || !cores || !shape || !ranks || !workspace || !result_host)
    return fail(TNB_ERR_INVALID, "tnb_tt_relative_error: null argument");
  Arena ar(workspace, workspace_bytes);
  if (dtype == TNB_F32)
    return tt_relative_error_impl<float>(ar, false, static_cast<const float*>(data),
                                         reinterpret_cast<const float* const*>(cores), ndim, shape, ranks, result_host,
                                         as_stream(stream));
  return tt_relative_error_impl<double>(ar, false, static_cast<const double*>(data),
                                        reinterpret_cast<const double* const*>(cores), ndim, shape, ranks, result_host,
                                        as_stream(stream));
}

}  // extern "C"

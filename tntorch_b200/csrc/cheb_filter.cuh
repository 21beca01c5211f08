// Chebyshev filter of the subspace iteration (eig.cuh) as ONE resident kernel.
//
// The filter is m products Y_s = a_s * G*Y_{s-1} + b_s * Y_{s-1} + g_s * Y_{s-2} with the same symmetric G
// (n x n fp32, <= 16 MB).  Launched one product at a time it is latency-bound (15 us tensor-core kernel +
// 5 us split-K finalize per product, 60 products per eigensolve).  Here G is partitioned ONCE over the
// shared memories of the grid and stays there for all m products:
//
//   * a cluster of 8 CTAs owns a 128-row slab of the output; CTA q of the cluster holds the G block
//     (K-slice q: rows [q*n/8, (q+1)*n/8)) x (128 slab columns) — G is symmetric, so this block is the
//     MN-major A operand of the slab's product — loaded by TMA (128B swizzle, 32B atoms) before step 1;
//   * each step: TMA-load the matching K-slice of Y_{s-1} (n/8 x b, L2 resident), tcgen05.mma tf32
//     128 x b x n/8 into TMEM, drain TMEM -> shared memory, cluster barrier, every CTA sums 16 of the
//     slab's rows over the 8 partial tiles through distributed shared memory, applies the three-term
//     recurrence and writes its 16 rows of Y_s;
//   * a grid-wide barrier (all CTAs are co-resident: cooperative launch) separates the steps.
//
// A B200 schedules at most 15 clusters of 8 CTAs with this shared-memory footprint (one GPC has room for
// only one), so n = 2048 (16 slabs) cannot use the cluster form: there the 8 partial tiles of a slab go
// through L2 instead (row-major partial tiles, coalesced both ways) with a second grid barrier per step.
//
// Only the FILTER runs here (TF32 operands: operator accuracy affects the convergence rate only); the
// Rayleigh-Ritz product stays on the fp32 FFMA path (eig.cuh).
#pragma once
#include <mutex>

#include "common.cuh"
#include "gram_tc.cuh"
#include "gram_tc2.cuh"

namespace tnb {

constexpr int CF_KS = 8;          // cluster size = K-slices per slab
constexpr int CF_THREADS = 128;
constexpr int CF_MAX_STEPS = 48;
constexpr int CF_RED_LD = 129;    // odd column stride of the partial-tile buffer: conflict-free both ways

// Device-resident control block of the sync-free subspace eigensolver (chfsi_dev.cuh).  The first three ints are the
// skip words of common.cuh::tnb_skip.  The Rayleigh-Ritz kernel of stage s writes the degree, the coefficients and the
// ring position of the NEXT filter here; the filter kernel reads them (nothing about the filter passes through the host).
struct ChfsiCtrl {
  int done;        // 1 once the captured energy has converged
  int error;       // 0 ok, 1 Cholesky breakdown (numerically dependent block), 2 not converged, 3 non-finite values
  int conv_stage;  // stage at which `done` was raised
  int outer;       // Rayleigh-Ritz steps completed
  int products;    // filter products executed
  int steps;       // degree of the next filter
  int xin;         // ring buffer holding the input block of the next filter; its result lands in ring[0]
  int jac_sweeps;  // Jacobi sweeps summed over the Rayleigh-Ritz solves (diagnostic)
  double prev_cap, prev_delta, trace, cap;
  float a[48], bc[48], g[48];  // CF_MAX_STEPS
};

struct ChebFilterParams {
  int n, b;        // G is n x n, blocks are n x b (ld = b)
  int nbox;        // ceil(b / 32)
  int ksl;         // n / 8 rows of Y per CTA
  int steps;
  float a[CF_MAX_STEPS], bc[CF_MAX_STEPS], g[CF_MAX_STEPS];
  float* buf[3];   // rotating n x b blocks: step s reads buf[(s-1)%3] (and buf[(s-2)%3]), writes buf[s%3]
  unsigned* counter;  // zeroed grid-barrier counter
  int tmem_cols;
  int dsmem;          // 1: launched as clusters of 8, partial tiles reduced through distributed shared memory
  float* partial;     // dsmem == 0: [slab][q][128][nbox*32] partial tiles in global memory (L2 resident)
  const ChfsiCtrl* ctrl;  // non-null: steps / coefficients / ring rotation come from the device control block
  int stage;
};

inline size_t cheb_filter_smem_bytes(int n, int b) {
  const int nbox = (b + 31) / 32, ksl = n / CF_KS;
  return (size_t)ksl * 128 * 4 + (size_t)ksl * nbox * 128 + (size_t)nbox * 32 * CF_RED_LD * 4 + 1024 + 64;
}
inline bool cheb_filter_shape_ok(int n, int b) {
  if (n % 256 != 0 || n < 256 || b < 8 || b % 4 != 0 || b > 128) return false;
  if ((n / 128) * CF_KS > device_info().sm_count) return false;
  return cheb_filter_smem_bytes(n, b) <= (size_t)227 * 1024;
}

__device__ __forceinline__ void cf_grid_barrier(unsigned* ctr, unsigned target) {
  asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
  unsigned v;
  const long long t0 = clock64();
  for (;;) {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
    if (v >= target) break;
    if (clock64() - t0 > 4000000000LL) {
      printf("tnb200: filter grid barrier timed out (block %d, %u < %u)\n", blockIdx.x, v, target);
      __trap();
    }
  }
}

__global__ void __launch_bounds__(CF_THREADS, 1)
cheb_filter_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_y0,
                   const __grid_constant__ CUtensorMap tmap_y1, const __grid_constant__ CUtensorMap tmap_y2,
                   const ChebFilterParams p) {
  extern __shared__ unsigned char cf_smem_raw[];
  int nsteps = p.steps, rot = 0;
  if (p.ctrl) {  // speculative enqueue: the whole grid leaves at once when the solve has converged or failed
    if (tnb_skip(&p.ctrl->done, p.stage)) return;
    nsteps = __ldcg(&p.ctrl->steps);
    rot = __ldcg(&p.ctrl->xin);
    if (nsteps < 1 || nsteps > CF_MAX_STEPS) return;
  }
  const uint32_t raw_addr = smem_u32(cf_smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  unsigned char* g_sm = cf_smem_raw + pad;                                  // ksl/32 chunks x 4 boxes
  unsigned char* y_sm = g_sm + (size_t)p.ksl * 512;                         // ksl/32 chunks x nbox boxes
  float* red = reinterpret_cast<float*>(y_sm + (size_t)p.ksl * p.nbox * 128);  // [nbox*32][CF_RED_LD]
  uint64_t* bars = reinterpret_cast<uint64_t*>(red + (size_t)p.nbox * 32 * CF_RED_LD);
  uint64_t* g_bar = bars;
  uint64_t* y_bar = bars + 1;
  uint64_t* mma_bar = bars + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 3);

  const int tid = threadIdx.x, warp_idx = tid >> 5, lane = tid & 31;
  const uint32_t q = blockIdx.x % CF_KS;         // K-slice of this CTA (= its rank in the cluster, if any)
  const int slab = blockIdx.x / CF_KS;           // 128-row slab of the output
  const int m0 = slab * 128, k0 = (int)q * p.ksl;
  const int nchunk = p.ksl / 32;
  const int bn = p.nbox * 32;

  if (tid == 0) {
    mbar_init(g_bar, 1);
    mbar_init(y_bar, 1);
    mbar_init(mma_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp_idx == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                 "r"((uint32_t)p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (tid == 0) {
    // resident block of G: rows k0..k0+ksl, columns m0..m0+128
    mbar_expect_tx(g_bar, (uint32_t)p.ksl * 512u);
    for (int c = 0; c < nchunk; ++c)
      for (int j = 0; j < 4; ++j)
        tma_load_2d(g_sm + ((size_t)c * 4 + j) * TC_BOX_BYTES, &tmap_g, g_bar, m0 + 32 * j, k0 + 32 * c);
  }
  cluster_sync_all();  // every CTA of the cluster is running before any DSMEM access

  const uint32_t idesc = make_idesc_tf32_mn(128, bn);
  const uint32_t red_addr = smem_u32(red);
  const int row_base = m0 + 16 * (int)q;  // the 16 output rows this CTA reduces and writes

  for (int s = 1; s <= nsteps; ++s) {
    const uint32_t par = (uint32_t)(s - 1) & 1u;
    const int icur = (s - 1 + rot) % 3, iprev = (s + 1 + rot) % 3, iout = (s + rot) % 3;
    const float* ycur = p.buf[icur];   // written by other CTAs in earlier steps: read through L2 (__ldcg)
    const float* yprev = p.buf[iprev];
    float* yout = p.buf[iout];
    const float ca = p.ctrl ? __ldcg(&p.ctrl->a[s - 1]) : p.a[s - 1];
    const float cb = p.ctrl ? __ldcg(&p.ctrl->bc[s - 1]) : p.bc[s - 1];
    const float cg = p.ctrl ? __ldcg(&p.ctrl->g[s - 1]) : p.g[s - 1];
    if (tid == 0) {
      asm volatile("fence.proxy.async;" ::: "memory");  // Y_{s-1} was written with generic stores by other CTAs
      const CUtensorMap* tm = icur == 0 ? &tmap_y0 : (icur == 1 ? &tmap_y1 : &tmap_y2);
      mbar_expect_tx(y_bar, (uint32_t)p.ksl * (uint32_t)p.nbox * 128u);
      for (int c = 0; c < nchunk; ++c)
        for (int j = 0; j < p.nbox; ++j)
          tma_load_2d(y_sm + ((size_t)c * p.nbox + j) * TC_BOX_BYTES, tm, y_bar, 32 * j, k0 + 32 * c);
      if (s == 1) mbar_wait(g_bar, 0);
      mbar_wait(y_bar, par);
      tcgen05_fence_after();
      const uint32_t ga = smem_u32(g_sm), ya = smem_u32(y_sm);
      for (int c = 0; c < nchunk; ++c) {
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint64_t adesc = make_mn_major_desc(ga + (uint32_t)c * 4u * TC_BOX_BYTES + ks * 1024u, TC_BOX_BYTES, 512, 1);
          const uint64_t bdesc =
              make_mn_major_desc(ya + (uint32_t)c * (uint32_t)p.nbox * TC_BOX_BYTES + ks * 1024u, TC_BOX_BYTES, 512, 1);
          tcgen05_mma_tf32(tmem_base, adesc, bdesc, idesc, (c > 0 || ks > 0) ? 1u : 0u);
        }
      }
      tcgen05_commit(mma_bar);
    }
    // operands of the recurrence for this thread's share of the 16 x b output rows (independent of the MMA)
    float vc[16], vp[16];
#pragma unroll
    for (int cnt = 0; cnt < 16; ++cnt) {
      const int idx = tid + cnt * CF_THREADS;
      const int r = idx / bn, j = idx - r * bn;
      vc[cnt] = 0.f;
      vp[cnt] = 0.f;
      if (idx < 16 * bn && j < p.b) {
        const size_t off = (size_t)(row_base + r) * p.b + j;
        if (cb != 0.f) vc[cnt] = __ldcg(ycur + off);
        if (cg != 0.f) vp[cnt] = __ldcg(yprev + off);
      }
    }
    mbar_wait(mma_bar, par);
    __syncwarp();
    tcgen05_fence_after();
    if (p.dsmem) {
      const int row = warp_idx * 32 + lane;  // accumulator row = slab row
      for (int c0 = 0; c0 < bn; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(warp_idx * 32) << 16) + (uint32_t)c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) red[(size_t)(c0 + i) * CF_RED_LD + row] = __uint_as_float(v[i]);
      }
      tcgen05_fence_before();
      __syncwarp();
      cluster_sync_all();  // all 8 partial tiles of the slab are in shared memory
#pragma unroll
      for (int cnt = 0; cnt < 16; ++cnt) {
        const int idx = tid + cnt * CF_THREADS;
        if (idx >= 16 * bn) break;
        const int r = idx / bn, j = idx - r * bn;
        const uint32_t laddr = red_addr + (uint32_t)((j * CF_RED_LD + 16 * (int)q + r) * 4);
        float sum = 0.f;
#pragma unroll
        for (uint32_t peer = 0; peer < CF_KS; ++peer) {
          uint32_t raddr;
          float x;
          asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(laddr), "r"(peer));
          asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(x) : "r"(raddr) : "memory");
          sum += x;
        }
        if (j < p.b) yout[(size_t)(row_base + r) * p.b + j] = ca * sum + cb * vc[cnt] + cg * vp[cnt];
      }
    } else {
      const int row = warp_idx * 32 + lane;
      float* out = p.partial + (((size_t)slab * CF_KS + q) * 128 + row) * (size_t)bn;
      for (int c0 = 0; c0 < bn; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(warp_idx * 32) << 16) + (uint32_t)c0, v);
        tmem_ld_wait();
        float4* o4 = reinterpret_cast<float4*>(out + c0);
#pragma unroll
        for (int i = 0; i < 8; ++i)
          o4[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]),
                              __uint_as_float(v[4 * i + 3]));
      }
      tcgen05_fence_before();
      __threadfence();
      __syncthreads();
      if (tid == 0) cf_grid_barrier(p.counter, (unsigned)gridDim.x * (unsigned)(2 * s - 1));
      __syncthreads();
#pragma unroll
      for (int cnt = 0; cnt < 16; ++cnt) {
        const int idx = tid + cnt * CF_THREADS;
        if (idx >= 16 * bn) break;
        const int r = idx / bn, j = idx - r * bn;
        const float* src = p.partial + (((size_t)slab * CF_KS) * 128 + 16 * q + r) * (size_t)bn + j;
        float sum = 0.f;
#pragma unroll
        for (int peer = 0; peer < CF_KS; ++peer) sum += __ldcg(src + (size_t)peer * 128 * bn);
        if (j < p.b) yout[(size_t)(row_base + r) * p.b + j] = ca * sum + cb * vc[cnt] + cg * vp[cnt];
      }
    }
    __threadfence();
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncthreads();
    if (tid == 0) cf_grid_barrier(p.counter, (unsigned)gridDim.x * (unsigned)(p.dsmem ? s : 2 * s));
    __syncthreads();
  }

  tcgen05_fence_before();
  cluster_sync_all();
  if (warp_idx == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols)
                 : "memory");
  }
}

inline size_t cheb_filter_workspace_bytes(int n, int b) {
  return align_up((size_t)n * CF_KS * (size_t)((b + 31) / 32 * 32) * sizeof(float)) + 256;
}

// Runs `steps` filter products.  bufs[0] holds the input block; the result is left in bufs[steps % 3].
// ws: cheb_filter_workspace_bytes(n, b) of device scratch (grid-barrier counter + partial tiles).
// Returns TNB_ERR_UNSUPPORTED (without touching the blocks, reason in the last-error string) outside the
// envelope or when the driver refuses the cooperative launch, so that the caller can run the products one by one.
inline int cheb_filter_f32(const float* G, int n, int b, float* const bufs[3], int steps, const float* a,
                           const float* bc, const float* g, void* ws, size_t ws_bytes, cudaStream_t st,
                           const ChfsiCtrl* ctrl = nullptr, int stage = 0) {
  if (ctrl) steps = 1;  // the degree comes from the control block
  if (!tc_path_available() || !cheb_filter_shape_ok(n, b) || steps < 1 || steps > CF_MAX_STEPS ||
      ws_bytes < cheb_filter_workspace_bytes(n, b)) {
    last_error_ref() = "resident filter: shape outside the envelope or workspace too small";
    return TNB_ERR_UNSUPPORTED;
  }
  // everything remembered about the launch is per device: refused sizes, the chaining event, the cluster occupancy
  struct DevState {
    std::mutex mu;
    cudaEvent_t last = nullptr;
    int max_clusters = -1;  // co-resident clusters of 8 CTAs at the largest footprint
    unsigned refused = 0;   // sizes whose cooperative launch the driver refused once
  };
  static DevState states[TNB_MAX_DEVICES];
  DevState& ds = states[current_device_index()];
  if (ds.refused & (1u << (n / 256))) return TNB_ERR_UNSUPPORTED;
  ChebFilterParams p;
  p.n = n;
  p.b = b;
  p.nbox = (b + 31) / 32;
  p.ksl = n / CF_KS;
  p.steps = steps;
  p.ctrl = ctrl;
  p.stage = stage;
  for (int i = 0; i < steps && !ctrl; ++i) { p.a[i] = a[i]; p.bc[i] = bc[i]; p.g[i] = g[i]; }
  for (int i = 0; i < 3; ++i) p.buf[i] = bufs[i];
  p.counter = static_cast<unsigned*>(ws);
  p.partial = reinterpret_cast<float*>(static_cast<char*>(ws) + 256);
  int cols = 32;
  while (cols < p.nbox * 32) cols <<= 1;
  p.tmem_cols = cols;
  CUtensorMap tg, ty[3];
  TNB_TRY(encode_rowmajor_f32(&tg, G, n, n));
  for (int i = 0; i < 3; ++i) TNB_TRY(encode_rowmajor_f32(&ty[i], bufs[i], n, b));
  const size_t smem = cheb_filter_smem_bytes(n, b);
  std::lock_guard<std::mutex> lk(ds.mu);
  cudaEvent_t& last = ds.last;
  int& max_clusters = ds.max_clusters;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((n / 128) * CF_KS));
  cfg.blockDim = dim3(CF_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  // Speculatively enqueued stages (ctrl != nullptr) are NOT cooperative launches: a cooperative launch — even of a stage
  // that will return at once because the solve has converged — waits until all of its CTAs fit on the GPU at the same
  // time, i.e. for a gap between the whole-GPU kernels of the other in-flight tensors.  A plain launch lets the CTAs of a
  // skipped stage drain through whatever SMs are free.  Co-residency of a stage that does run is still guaranteed:
  // grid <= SM count with one CTA per SM (checked in cheb_filter_shape_ok), the filter kernels of all streams are
  // chained by the event below so two of them never hold SMs at the same time, and no other kernel of this library waits
  // on a filter while holding SMs; the grid barrier additionally times out instead of spinning for ever.
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeCooperative;
  attrs[0].val.cooperative = ctrl ? 0 : 1;
  attrs[1].id = cudaLaunchAttributeClusterDimension;
  attrs[1].val.clusterDim.x = CF_KS;
  attrs[1].val.clusterDim.y = 1;
  attrs[1].val.clusterDim.z = 1;
  cfg.attrs = attrs;
  if (max_clusters < 0) {
    TNB_CUDA(cudaFuncSetAttribute(cheb_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    TNB_CUDA(cudaEventCreateWithFlags(&last, cudaEventDisableTiming));
    cudaLaunchConfig_t probe = cfg;
    probe.dynamicSmemBytes = 227 * 1024 - 2048;
    probe.numAttrs = 2;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, cheb_filter_kernel, &probe) != cudaSuccess) nc = 0;
    cudaGetLastError();
    max_clusters = nc;
  }
  p.dsmem = (n / 128 <= max_clusters && !getenv("TNB_FILTER_NO_DSMEM")) ? 1 : 0;
  cfg.numAttrs = p.dsmem ? 2 : 1;
  TNB_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(unsigned), st));
  // two resident filter kernels that each hold part of the SMs would wait on each other for ever:
  // chain them across streams
  TNB_CUDA(cudaStreamWaitEvent(st, last, 0));
  cudaError_t e = cudaLaunchKernelEx(&cfg, cheb_filter_kernel, tg, ty[0], ty[1], ty[2], p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    fail(TNB_ERR_UNSUPPORTED, "resident filter launch refused: %s (n=%d b=%d smem=%zu dsmem=%d, max active clusters %d)",
         cudaGetErrorString(e), n, b, smem, p.dsmem, max_clusters);
    ds.refused |= 1u << (n / 256);
    return TNB_ERR_UNSUPPORTED;
  }
  TNB_CUDA(cudaEventRecord(last, st));
  return TNB_OK;
}

}  // namespace tnb

// Wide Gram matrices (n >= 256) on CTA PAIRS: tcgen05.mma.cta_group::2, 256 x 256 tf32 tiles.
//
// The 1-CTA kernel (gram_tc.cuh) feeds a 128 x 256 tile with 384 fp32 per contraction row — 21 MAC per
// byte staged — and ncu shows it at ~49 % tensor-pipe with the shared-memory fill as the limiter.  Here two
// CTAs of a cluster (one TPC) share one 256 x 256 accumulator: each CTA stages only ITS 128 A-columns and
// ITS 128 of the 256 B-columns (32 MAC per staged byte, 64 on diagonal tiles where the two coincide), the
// leader CTA issues the MMA for both, and each CTA keeps its 128 accumulator rows in its own TMEM.
//
//   * TMA loads are issued by both CTAs with .cta_group::2 and signal the LEADER's full barrier;
//   * tcgen05.commit multicasts the "stage free" / "accumulator ready" arrivals to both CTAs;
//   * TMEM is allocated with cta_group::2 by the same warp of both CTAs; cluster barriers frame the
//     barrier initialisation and the deallocation.
#pragma once
#include "gram_tc.cuh"

namespace tnb {

// KC rows of C per pipeline stage in 8 KB TMA boxes, 3 stages: 64 measured 21 % faster than 32-row boxes with 6 stages
// on the 262144 x 2048 Gram (half as many TMA instructions and barrier round trips per byte for the single producer /
// issuer threads; profiles/r02_gram_tc2_depth.md)
constexpr int TC2_KC = 64;
constexpr int TC2_BOX_BYTES = TC2_KC * 128;          // one TMA box: 32 fp32 columns x KC rows
constexpr int TC2_STAGE_BYTES = 8 * TC2_BOX_BYTES;   // A_r: 4 boxes, B_r: 4 boxes (64 KB)
constexpr int TC2_STAGES = 3;
constexpr int TC2_SMEM_BYTES = TC2_STAGES * TC2_STAGE_BYTES + 1024 + 256;

struct GramTc2Params {
  int64_t rows;
  int n;
  int nb;          // ceil(n / 256) tile blocks per side
  int num_tiles;   // nb (nb + 1) / 2 upper pair tiles
  int ksplit;
  int64_t iters_total, iters_per_split;
  float* partial;  // [ksplit][num_tiles][256][256]
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the barrier at the same offset in the LEADER CTA (rank 0)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
  const uint32_t mbar = smem_u32(bar) & 0xFEFFFFFFu;  // clear the peer bit of the shared::cluster address
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(mbar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tcgen05_commit_pair(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .b16 m;\n\tmov.b16 m, 3;\n\t"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], m;\n\t}"
      :
      : "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tcgen05_mma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                      uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
gram_tc2_kernel(const __grid_constant__ CUtensorMap tmap, const GramTc2Params p) {
  extern __shared__ unsigned char tc2_smem_raw[];
  const uint32_t raw_addr = smem_u32(tc2_smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  unsigned char* stage_base = tc2_smem_raw + pad;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stage_base + TC2_STAGES * TC2_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + TC2_STAGES;
  uint64_t* tmem_full_bar = empty_bar + TC2_STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp_idx = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const int tile_id = blockIdx.x >> 1, split = blockIdx.y;
  // flat upper-triangular tile id -> (bm, bn), bn >= bm
  int bm = 0, rem = tile_id;
  while (rem >= p.nb - bm) { rem -= p.nb - bm; ++bm; }
  const int bn = bm + rem;
  const bool diag = (bm == bn);

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC2_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp_idx == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                 "r"(256u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  cluster_sync_all();  // both CTAs' barriers are initialised before any cross-CTA arrival
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const int a_col0 = bm * 256 + (int)cta_rank * 128;   // this CTA's 128 accumulator rows
  const int b_col0 = bn * 256 + (int)cta_rank * 128;   // this CTA's half of the 256 B columns
  const int nbox = diag ? 4 : 8;
  const int64_t it_begin = (int64_t)split * p.iters_per_split;
  int64_t it_end = it_begin + p.iters_per_split;
  if (it_end > p.iters_total) it_end = p.iters_total;
  const int64_t iters = it_end > it_begin ? it_end - it_begin : 0;

  if (warp_idx == 0) {
    // ================= TMA producer (both CTAs) =================
    if (lane == 0 && iters > 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < iters; ++it) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        unsigned char* sb = stage_base + stage * TC2_STAGE_BYTES;
        if (cta_rank == 0) mbar_expect_tx(&full_bar[stage], 2u * (uint32_t)nbox * TC2_BOX_BYTES);  // bytes of BOTH CTAs
        const int row0 = (int)((it_begin + it) * TC2_KC);
        for (int j = 0; j < 4; ++j) tma_load_2d_pair(sb + j * TC2_BOX_BYTES, &tmap, &full_bar[stage], b_col0 + 32 * j, row0);
        if (!diag)
          for (int j = 0; j < 4; ++j)
            tma_load_2d_pair(sb + (4 + j) * TC2_BOX_BYTES, &tmap, &full_bar[stage], a_col0 + 32 * j, row0);
        if (++stage == TC2_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp_idx == 1) {
    // ================= MMA issuer (leader CTA only) =================
    if (cta_rank == 0 && lane == 0 && iters > 0) {
      const uint32_t idesc = make_idesc_tf32_mn(256, 256);
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        const uint32_t sb = smem_u32(stage_base + stage * TC2_STAGE_BYTES);
        const uint32_t b_addr = sb;
        const uint32_t a_addr = diag ? sb : sb + 4u * TC2_BOX_BYTES;
#pragma unroll
        for (int ks = 0; ks < TC2_KC / 8; ++ks) {
          const uint64_t adesc = make_mn_major_desc(a_addr + ks * 1024u, TC2_BOX_BYTES, 512u, 1u);
          const uint64_t bdesc = make_mn_major_desc(b_addr + ks * 1024u, TC2_BOX_BYTES, 512u, 1u);
          tcgen05_mma_tf32_pair(tmem_base, adesc, bdesc, idesc, (it > 0 || ks > 0) ? 1u : 0u);
        }
        tcgen05_commit_pair(&empty_bar[stage]);  // frees the stage in both CTAs
        if (++stage == TC2_STAGES) { stage = 0; phase ^= 1u; }
      }
      tcgen05_commit_pair(tmem_full_bar);
    }
  } else {
    // ================= epilogue (both CTAs): this CTA's 128 rows of the 256 x 256 tile =================
    const int lane_group = warp_idx & 3;
    const int row = (int)cta_rank * 128 + lane_group * 32 + lane;
    float* out = p.partial + (((size_t)split * p.num_tiles + tile_id) * 256 + row) * 256;
    if (iters > 0) {
      mbar_wait(tmem_full_bar, 0);
      tcgen05_fence_after();
      for (int c0 = 0; c0 < 256; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(tmem_base + ((uint32_t)(lane_group * 32) << 16) + (uint32_t)c0, v);
        tmem_ld_wait();
        float4* o4 = reinterpret_cast<float4*>(out + c0);
#pragma unroll
        for (int q = 0; q < 8; ++q)
          o4[q] = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                              __uint_as_float(v[4 * q + 3]));
      }
    } else {
      for (int c0 = 0; c0 < 256; c0 += 4) *reinterpret_cast<float4*>(out + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();  // the peer may still be reading smem / TMEM that this CTA's exit would release
  if (warp_idx == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
  }
}

__global__ void gram_tc2_finalize_kernel(const GramTc2Params p, double* __restrict__ G, float* __restrict__ Gf) {
  const int64_t total = (int64_t)p.n * p.n;
  const size_t split_stride = (size_t)p.num_tiles * 256 * 256;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / p.n), j = (int)(idx % p.n);
    const int ii = i <= j ? i : j, jj = i <= j ? j : i;
    const int bm = ii / 256, bn = jj / 256;
    const int tile = bm * p.nb - bm * (bm - 1) / 2 + (bn - bm);
    const size_t off = ((size_t)tile * 256 + (ii - bm * 256)) * 256 + (jj - bn * 256);
    double s = 0.0;
    for (int z = 0; z < p.ksplit; ++z) s += (double)p.partial[(size_t)z * split_stride + off];
    G[idx] = s;
    if (Gf) Gf[idx] = (float)s;
  }
}

inline bool gram_tc2_shape_ok(int64_t rows, int64_t n) { return n >= 512 && gram_tc_shape_ok(rows, n); }

inline void gram_tc2_plan(int64_t rows, int64_t n, GramTc2Params& p) {
  p.rows = rows;
  p.n = (int)n;
  p.nb = (int)((n + 255) / 256);
  p.num_tiles = p.nb * (p.nb + 1) / 2;
  p.iters_total = (rows + TC2_KC - 1) / TC2_KC;
  const int sms = usable_sms();
  int64_t ks = (sms / 2) / p.num_tiles;
  if (ks < 1) ks = 1;
  if (ks > p.iters_total) ks = p.iters_total;
  p.iters_per_split = (p.iters_total + ks - 1) / ks;
  p.ksplit = (int)((p.iters_total + p.iters_per_split - 1) / p.iters_per_split);
  p.partial = nullptr;
}
inline size_t gram_tc2_workspace_bytes(int64_t rows, int64_t n) {
  GramTc2Params p;
  gram_tc2_plan(rows, n, p);
  return align_up((size_t)p.ksplit * p.num_tiles * 256 * 256 * sizeof(float));
}

inline int gram_tc2_f32(const float* A, int64_t rows, int64_t n, double* G, float* Gf, void* ws, size_t ws_bytes,
                        cudaStream_t st) {
  if (!tc_path_available()) return fail(TNB_ERR_UNSUPPORTED, "gram_tc2: needs an sm_100 device");
  if (!gram_tc2_shape_ok(rows, n)) return fail(TNB_ERR_UNSUPPORTED, "gram_tc2: unsupported shape");
  if ((reinterpret_cast<uintptr_t>(A) & 15u) != 0) return fail(TNB_ERR_INVALID, "gram_tc2: input must be 16-byte aligned");
  GramTc2Params p;
  gram_tc2_plan(rows, n, p);
  const size_t need = (size_t)p.ksplit * p.num_tiles * 256 * 256 * sizeof(float);
  if (ws_bytes < need) return fail(TNB_ERR_WORKSPACE, "gram_tc2: workspace %zu < %zu", ws_bytes, need);
  p.partial = static_cast<float*>(ws);
  CUtensorMap tmap;
  TNB_TRY(encode_rowmajor_f32(&tmap, A, rows, n, TC2_KC));
  static PerDeviceFlag attr_done;
  TNB_CUDA(ensure_dyn_smem(attr_done, gram_tc2_kernel, TC2_SMEM_BYTES));
  dim3 grid((unsigned)(2 * p.num_tiles), (unsigned)p.ksplit);
  gram_tc2_kernel<<<grid, TC_THREADS, TC2_SMEM_BYTES, st>>>(tmap, p);
  TNB_LAUNCH_CHECK();
  const int64_t total = n * n;
  gram_tc2_finalize_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, 4096), 256, 0, st>>>(p, G, Gf);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

}  // namespace tnb

// Gram matrix G = C^T C of a tall row-major fp32 matrix C (rows x n) on the Blackwell tensor cores.
//
//   * row slabs of C are staged HBM -> shared memory by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle with 32-byte atoms,
//     out-of-bounds rows/columns zero-filled by the TMA unit), 4-stage mbarrier ring;
//   * the contraction runs over the ROW index of C, so both MMA operands are "MN-major" views of the
//     very same slab: tcgen05.mma.cta_group::1.kind::tf32, M = 128, N = TN <= 256, K = 8 per instruction,
//     fp32 accumulation in TMEM;
//   * G is symmetric: only tiles that touch the upper triangle are computed, and on diagonal tiles the
//     A operand is a sub-block of the B slab (loaded once);
//   * split-K over row ranges across CTAs; partial tiles are drained TMEM -> registers (tcgen05.ld)
//     -> global and summed in fp64 by a deterministic second kernel (no atomics).
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (TMEM lane group = warp_idx % 4).
//
// Replaces, for large fp32 unfoldings, the QR of tensor.py:1816 / the Gram of round.py:104-110.
#pragma once
#include <cuda.h>

#include <cstdlib>

#include "common.cuh"

namespace tnb {

constexpr int TC_KC = 32;                       // rows of C per pipeline stage
constexpr int TC_BOX_BYTES = TC_KC * 128;       // one TMA box: 32 fp32 columns x KC rows
constexpr int TC_STAGES = 4;
constexpr int TC_MAX_BOXES = 12;                // 4 (A) + 8 (B)
constexpr int TC_STAGE_BYTES = TC_MAX_BOXES * TC_BOX_BYTES;
constexpr int TC_THREADS = 192;
constexpr int TC_SMEM_BYTES = TC_STAGES * TC_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;

struct GramTcParams {
  int64_t rows;    // contraction length K (rows of both operands)
  int n;           // columns of B (= of A in the symmetric Gram case)
  int m;           // columns of A
  int symmetric;   // 1: A == B, only tiles touching the upper triangle; 0: general A^T B
  int tn;          // B tile width (multiple of 32, <= 256)
  int num_bm;      // ceil(m / 128)
  int num_bn;      // ceil(n / tn)
  int num_tiles;   // kept tiles
  int ksplit;
  int64_t iters_total;      // ceil(rows / KC)
  int64_t iters_per_split;
  float* partial;  // [ksplit][num_tiles][128][tn]
  int tmem_cols;
  // shared-memory operand descriptor fields (see make_mn_major_desc)
  uint32_t desc_layout;  // 1 = SWIZZLE_128B_BASE32B (the only MN-major layout tf32 operands accept)
  uint32_t desc_lbo;     // bytes between 32-column groups (one TMA box)
  uint32_t desc_sbo;     // bytes between K atoms (4 rows x 128 B)
  int fold;              // > 1: the matrix was viewed as (rows/fold) x (fold*n_orig); G = sum of the diagonal blocks
  int n_orig;
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a wrong descriptor or byte count must surface as an error, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;  // fast path: no clock read when the phase has already completed
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s
      printf("tnb200: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tcgen05_mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor of an MN-major fp32/tf32 operand (cute::UMMA::SmemDescriptor bit layout):
//   bits [0,14)  start address >> 4
//   bits [16,30) leading byte offset >> 4  = stride between 32-column (128-byte) groups along M/N
//   bits [32,46) stride byte offset >> 4   = stride between K atoms (4 rows of 128 B = 512 B)
//   bits [46,48) version = 1 (Blackwell)     bits [61,64) layout type
// tf32 MN-major operands only accept the "128-byte swizzle with 32-byte atoms" layout
// (UMMA::LayoutType::SWIZZLE_128B_BASE32B = 1; Swizzle<2,5,2>: the 32-byte chunk index is XORed with
// row % 4), which is what the TMA writes with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
__device__ __forceinline__ uint64_t make_mn_major_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                       uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(layout_type & 7u) << 61;
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accumulate, tf32 x tf32, both operands MN-major.
__host__ __device__ inline uint32_t make_idesc_tf32_mn(int M, int N) {
  uint32_t d = 0;
  d |= 1u << 4;                    // c_format = F32
  d |= 2u << 7;                    // a_format = TF32
  d |= 2u << 10;                   // b_format = TF32
  d |= 1u << 15;                   // a_major = MN
  d |= 1u << 16;                   // b_major = MN
  d |= (uint32_t)(N >> 3) << 17;   // n_dim
  d |= (uint32_t)(M >> 4) << 24;   // m_dim
  return d;
}

// ---------------------------------------------------------------------------------------------
// The kernel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TC_THREADS, 1)
gram_tc_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_b,
               const GramTcParams p) {
  extern __shared__ unsigned char tc_smem_raw[];
  // 1024-byte aligned stage buffers (SWIZZLE_128B atoms are 1024 B)
  const uint32_t raw_addr = smem_u32(tc_smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  unsigned char* stage_base = tc_smem_raw + pad;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stage_base + TC_STAGES * TC_STAGE_BYTES);
  uint64_t* empty_bar = full_bar + TC_STAGES;
  uint64_t* tmem_full_bar = empty_bar + TC_STAGES;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  int* tile_smem = reinterpret_cast<int*>(tmem_ptr_smem + 1);  // bm, bn

  const int warp_idx = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tile_id = blockIdx.x, split = blockIdx.y;

  if (threadIdx.x == 0) {
    // flat tile id -> (bm, bn) among the tiles that touch the upper triangle
    int cnt = 0, fbm = 0, fbn = 0;
    if (p.symmetric) {
      for (int bm = 0; bm < p.num_bm; ++bm)
        for (int bn = 0; bn < p.num_bn; ++bn)
          if ((bn + 1) * p.tn > bm * 128) {
            if (cnt == tile_id) { fbm = bm; fbn = bn; }
            ++cnt;
          }
    } else {
      fbm = tile_id / p.num_bn;
      fbn = tile_id % p.num_bn;
    }
    tile_smem[0] = fbm;
    tile_smem[1] = fbn;
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp_idx == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                 "r"((uint32_t)p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();

  const uint32_t tmem_base = *tmem_ptr_smem;
  const int bm = tile_smem[0], bn = tile_smem[1];
  const int a_col0 = bm * 128, b_col0 = bn * p.tn;
  const int nbox_b = p.tn / 32;
  const bool a_in_b = p.symmetric && (a_col0 >= b_col0) && (a_col0 + 128 <= b_col0 + p.tn);
  const int nbox_a = a_in_b ? 0 : 4;
  const int64_t it_begin = (int64_t)split * p.iters_per_split;
  int64_t it_end = it_begin + p.iters_per_split;
  if (it_end > p.iters_total) it_end = p.iters_total;
  const int64_t iters = it_end > it_begin ? it_end - it_begin : 0;

  if (warp_idx == 0) {
    // ================= TMA producer =================
    if (lane == 0 && iters > 0) {
      const uint32_t tx_bytes = (uint32_t)(nbox_a + nbox_b) * TC_BOX_BYTES;
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < iters; ++it) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        unsigned char* sb = stage_base + stage * TC_STAGE_BYTES;
        mbar_expect_tx(&full_bar[stage], tx_bytes);
        const int row0 = (int)((it_begin + it) * TC_KC);
        // B boxes first (slots 0..nbox_b), then A boxes (slots 8..11)
        for (int j = 0; j < nbox_b; ++j) tma_load_2d(sb + j * TC_BOX_BYTES, &tmap_b, &full_bar[stage], b_col0 + 32 * j, row0);
        for (int j = 0; j < nbox_a; ++j)
          tma_load_2d(sb + (8 + j) * TC_BOX_BYTES, &tmap, &full_bar[stage], a_col0 + 32 * j, row0);
        if (++stage == TC_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp_idx == 1) {
    // ================= MMA issuer =================
    if (lane == 0 && iters > 0) {
      const uint32_t idesc = make_idesc_tf32_mn(128, p.tn);
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < iters; ++it) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        const uint32_t sb = smem_u32(stage_base + stage * TC_STAGE_BYTES);
        const uint32_t b_addr = sb;
        const uint32_t a_addr = a_in_b ? sb + (uint32_t)((a_col0 - b_col0) / 32) * TC_BOX_BYTES : sb + 8u * TC_BOX_BYTES;
#pragma unroll
        for (int ks = 0; ks < TC_KC / 8; ++ks) {
          const uint64_t adesc = make_mn_major_desc(a_addr + ks * 1024u, p.desc_lbo, p.desc_sbo, p.desc_layout);
          const uint64_t bdesc = make_mn_major_desc(b_addr + ks * 1024u, p.desc_lbo, p.desc_sbo, p.desc_layout);
          tcgen05_mma_tf32(tmem_base, adesc, bdesc, idesc, (it > 0 || ks > 0) ? 1u : 0u);
        }
        tcgen05_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs have read it
        if (++stage == TC_STAGES) { stage = 0; phase ^= 1u; }
      }
      tcgen05_commit(tmem_full_bar);  // accumulator complete
    }
  } else {
    // ================= epilogue: TMEM -> registers -> global partial tile =================
    const int lane_group = warp_idx & 3;          // TMEM lanes [32*lane_group, +32)
    const int row = lane_group * 32 + lane;       // accumulator row = column (a_col0 + row) of C
    float* out = p.partial + (((size_t)split * p.num_tiles + tile_id) * 128 + row) * (size_t)p.tn;
    if (iters > 0) {
      mbar_wait(tmem_full_bar, 0);
      tcgen05_fence_after();
      for (int c0 = 0; c0 < p.tn; c0 += 32) {
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
      for (int c0 = 0; c0 < p.tn; c0 += 4) *reinterpret_cast<float4*>(out + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp_idx == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols)
                 : "memory");
  }
}

// Sum the split-K partial tiles in fp64 (fixed order), mirror to the lower triangle.
__global__ void gram_tc_finalize_kernel(const GramTcParams p, double* __restrict__ G, float* __restrict__ Gf) {
  if (p.fold > 1) {  // single 128 x 128 tile; fold the diagonal n_orig x n_orig blocks
    // one WARP per output element: the ksplit * fold terms (hundreds, strided) are dealt to the lanes and combined by a
    // shuffle tree in a fixed order — deterministic like the serial sum, without its 300-deep dependent chain per thread
    const int no = p.n_orig;
    const size_t split_stride = (size_t)p.num_tiles * 128 * p.tn;
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const int nterms = p.ksplit * p.fold;
    for (int idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; idx < no * no; idx += warps) {
      const int i = idx / no, j = idx % no;
      double s = 0.0;
      for (int t = lane; t < nterms; t += 32) {
        const int z = t / p.fold, a = t - z * p.fold;
        s += (double)p.partial[(size_t)z * split_stride + (size_t)(a * no + i) * p.tn + (a * no + j)];
      }
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) {
        G[idx] = s;
        if (Gf) Gf[idx] = (float)s;
      }
    }
    return;
  }
  const int64_t total = (int64_t)p.n * p.n;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / p.n), j = (int)(idx % p.n);
    const int ii = i <= j ? i : j, jj = i <= j ? j : i;
    const int bm = ii / 128, bn = jj / p.tn;
    // flat index of (bm, bn) among kept tiles: row a keeps the column tiles b >= first(a) = floor(a*128 / tn)
    int tile = 0;
    for (int a = 0; a < bm; ++a) tile += p.num_bn - (a * 128) / p.tn;
    tile += bn - (bm * 128) / p.tn;
    const size_t off = ((size_t)tile * 128 + (ii - bm * 128)) * (size_t)p.tn + (jj - bn * p.tn);
    const size_t split_stride = (size_t)p.num_tiles * 128 * p.tn;
    double s = 0.0;
    for (int z = 0; z < p.ksplit; ++z) s += (double)p.partial[(size_t)z * split_stride + off];
    G[idx] = s;
    if (Gf) Gf[idx] = (float)s;
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled load_encode_tiled() {
  void* f = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
      q == cudaDriverEntryPointSuccess)
    return reinterpret_cast<PFN_encodeTiled>(f);
  cudaGetLastError();
  return nullptr;
}
inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = load_encode_tiled();  // thread-safe one-time initialisation
  return fn;
}

inline bool tc_path_available() {
  const DeviceInfo& di = device_info();
  return di.valid && di.cc_major == 10 && get_encode_tiled() != nullptr;
}

inline bool gram_tc_shape_ok(int64_t rows, int64_t n) {
  return n >= 16 && n % 4 == 0 && n <= 16384 && rows >= 1 && rows < ((int64_t)1 << 31) - 64;
}

inline void gram_tc_plan(int64_t rows, int64_t n, GramTcParams& p, int64_t m_cols = -1) {
  p.rows = rows;
  p.n = (int)n;
  p.symmetric = m_cols < 0 ? 1 : 0;
  p.m = p.symmetric ? (int)n : (int)m_cols;
  int tn = n >= 256 ? 256 : (int)((n + 31) / 32 * 32);
  p.tn = tn;
  p.num_bm = (int)((p.m + 127) / 128);
  p.num_bn = (int)((n + tn - 1) / tn);
  int cnt = 0;
  if (p.symmetric) {
    for (int bm = 0; bm < p.num_bm; ++bm)
      for (int bn = 0; bn < p.num_bn; ++bn)
        if ((bn + 1) * tn > bm * 128) ++cnt;
  } else {
    cnt = p.num_bm * p.num_bn;
  }
  p.num_tiles = cnt;
  p.iters_total = (rows + TC_KC - 1) / TC_KC;
  int sms = usable_sms();
  int64_t ks = sms / cnt;
  if (ks < 1) ks = 1;
  if (ks > p.iters_total) ks = p.iters_total;
  p.iters_per_split = (p.iters_total + ks - 1) / ks;
  ks = (p.iters_total + p.iters_per_split - 1) / p.iters_per_split;
  p.ksplit = (int)ks;
  int cols = 32;
  while (cols < tn) cols <<= 1;
  p.tmem_cols = cols;
  p.partial = nullptr;
  p.desc_layout = 1;
  p.desc_lbo = TC_BOX_BYTES;
  p.desc_sbo = 512;
  p.fold = 1;
  p.n_orig = (int)n;
}

// Narrow matrices (n = 32 or 64) are viewed as (rows/f) x 128, f = 128/n: one full-width 128 x 128 tile with
// every TMA box useful (16 KB per stage in flight instead of 8 KB padded with zero boxes); the Gram matrix is
// the sum of the f diagonal n x n blocks.
inline int gram_tc_fold(int64_t rows, int64_t n) {
  if (n >= 128 || n < 32 || 128 % n != 0) return 1;
  const int f = (int)(128 / n);
  return (rows % f == 0) ? f : 1;
}

inline size_t gram_tc_workspace_bytes(int64_t rows, int64_t n) {
  GramTcParams p;
  const int f = gram_tc_fold(rows, n);
  gram_tc_plan(rows / f, n * f, p);
  return align_up((size_t)p.ksplit * p.num_tiles * 128 * p.tn * sizeof(float));
}

// G (n x n fp64) and optionally Gf (fp32 copy) = A^T A, A: rows x n fp32 row-major (device).
inline int gram_tc_f32(const float* A, int64_t rows, int64_t n, double* G, float* Gf, void* ws, size_t ws_bytes,
                       cudaStream_t st) {
  if (!tc_path_available()) return fail(TNB_ERR_UNSUPPORTED, "gram_tc: tcgen05/TMA path needs an sm_100 device");
  if (!gram_tc_shape_ok(rows, n)) return fail(TNB_ERR_UNSUPPORTED, "gram_tc: unsupported shape rows=%lld n=%lld", (long long)rows, (long long)n);
  if ((reinterpret_cast<uintptr_t>(A) & 15u) != 0) return fail(TNB_ERR_INVALID, "gram_tc: input must be 16-byte aligned");
  GramTcParams p;
  const int fold = gram_tc_fold(rows, n);
  const int64_t n_in = n;
  rows /= fold;
  n *= fold;
  gram_tc_plan(rows, n, p);
  p.fold = fold;
  p.n_orig = (int)n_in;
  const size_t need = (size_t)p.ksplit * p.num_tiles * 128 * p.tn * sizeof(float);
  if (ws_bytes < need) return fail(TNB_ERR_WORKSPACE, "gram_tc: workspace %zu < %zu", ws_bytes, need);
  p.partial = static_cast<float*>(ws);

  const CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;  // matches UMMA SWIZZLE_128B_BASE32B
  CUtensorMap tmap;
  cuuint64_t gdim[2] = {(cuuint64_t)n, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)n * sizeof(float)};
  cuuint32_t box[2] = {32, (cuuint32_t)TC_KC};
  cuuint32_t estr[2] = {1, 1};
  CUresult cr = get_encode_tiled()(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(A), gdim, gstride, box,
                                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return fail(TNB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)cr);

  static PerDeviceFlag attr_done;
  TNB_CUDA(ensure_dyn_smem(attr_done, gram_tc_kernel, TC_SMEM_BYTES));
  dim3 grid((unsigned)p.num_tiles, (unsigned)p.ksplit);
  gram_tc_kernel<<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(tmap, tmap, p);
  TNB_LAUNCH_CHECK();
  const int64_t total = n_in * n_in * (p.fold > 1 ? 32 : 1);  // folded form: one warp per element
  gram_tc_finalize_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, 4096), 256, 0, st>>>(p, G, Gf);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

// ---------------------------------------------------------------------------------------------
// General C (m x n) = alpha * A^T B + beta * D + gamma * E on the same kernel: A is K x m, B is K x n,
// both row-major fp32 (TF32 operands, fp32 accumulation).  Used for the filter products G*Y of the
// subspace iteration (G symmetric, so A = G).  Finalize fuses the three-term epilogue.
// ---------------------------------------------------------------------------------------------
__global__ void atb_tc_finalize_kernel(const GramTcParams p, float* __restrict__ C, int ldc, float alpha,
                                       const float* __restrict__ D, int ldd, float beta, const float* __restrict__ E,
                                       int lde, float gamma) {
  const int64_t total = (int64_t)p.m * p.n;
  const size_t split_stride = (size_t)p.num_tiles * 128 * p.tn;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / p.n), j = (int)(idx % p.n);
    const int bm = i / 128, bn = j / p.tn;
    const int tile = bm * p.num_bn + bn;
    const size_t off = ((size_t)tile * 128 + (i - bm * 128)) * (size_t)p.tn + (j - bn * p.tn);
    float s = 0.f;
    for (int z = 0; z < p.ksplit; ++z) s += p.partial[(size_t)z * split_stride + off];
    float v = alpha * s;
    if (D) v += beta * D[(size_t)i * ldd + j];
    if (E) v += gamma * E[(size_t)i * lde + j];
    C[(size_t)i * ldc + j] = v;
  }
}

inline bool atb_tc_shape_ok(int64_t K, int64_t m, int64_t n) {
  return m >= 32 && n >= 32 && m % 4 == 0 && n % 4 == 0 && m <= 65536 && n <= 65536 && K >= 1 && K < ((int64_t)1 << 31) - 64;
}
inline size_t atb_tc_workspace_bytes(int64_t K, int64_t m, int64_t n) {
  GramTcParams p;
  gram_tc_plan(K, n, p, m);
  return align_up((size_t)p.ksplit * p.num_tiles * 128 * p.tn * sizeof(float));
}

inline int encode_rowmajor_f32(CUtensorMap* tmap, const float* ptr, int64_t rows, int64_t cols, int box_rows = TC_KC) {
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)cols * sizeof(float)};
  cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult cr = get_encode_tiled()(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstride, box,
                                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return fail(TNB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)cr);
  return TNB_OK;
}

inline int atb_tc_f32(const float* A, int64_t K, int64_t m, const float* B, int64_t n, float* C, int ldc, float alpha,
                      const float* D, int ldd, float beta, const float* E, int lde, float gamma, void* ws,
                      size_t ws_bytes, cudaStream_t st) {
  if (!tc_path_available()) return fail(TNB_ERR_UNSUPPORTED, "atb_tc: tcgen05/TMA path needs an sm_100 device");
  if (!atb_tc_shape_ok(K, m, n)) return fail(TNB_ERR_UNSUPPORTED, "atb_tc: unsupported shape K=%lld m=%lld n=%lld", (long long)K, (long long)m, (long long)n);
  if (((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B)) & 15u) != 0)
    return fail(TNB_ERR_INVALID, "atb_tc: operands must be 16-byte aligned");
  GramTcParams p;
  gram_tc_plan(K, n, p, m);
  const size_t need = (size_t)p.ksplit * p.num_tiles * 128 * p.tn * sizeof(float);
  if (ws_bytes < need) return fail(TNB_ERR_WORKSPACE, "atb_tc: workspace %zu < %zu", ws_bytes, need);
  p.partial = static_cast<float*>(ws);
  CUtensorMap ta, tb;
  TNB_TRY(encode_rowmajor_f32(&ta, A, K, m));
  TNB_TRY(encode_rowmajor_f32(&tb, B, K, n));
  static PerDeviceFlag attr_done;
  TNB_CUDA(ensure_dyn_smem(attr_done, gram_tc_kernel, TC_SMEM_BYTES));
  dim3 grid((unsigned)p.num_tiles, (unsigned)p.ksplit);
  gram_tc_kernel<<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(ta, tb, p);
  TNB_LAUNCH_CHECK();
  const int64_t total = m * n;
  atb_tc_finalize_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, 4096), 256, 0, st>>>(p, C, ldc, alpha, D, ldd,
                                                                                                 beta, E, lde, gamma);
  TNB_LAUNCH_CHECK();
  return TNB_OK;
}

}  // namespace tnb

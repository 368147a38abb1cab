// The two dense projections of M-A that are genuinely GEMMs -- the detector's 6144 -> 512 over all B*T frames (cad:167, 3.2 GFLOP) and
// the direct classifier's 6144 -> 512 over the B clips (cad:526) -- on the tensor cores with fp32-level accuracy ("3xTF32"):
//
//      C[M][N] += sum_k A[m][k] * W[n][k]          A (M,K), W (N,K) fp32 row-major (K contiguous), C fp32 (M,N), pre-zeroed
//
// tcgen05 kind::tf32 multiplies 11-bit-significand operands.  A plain tf32 product is 1e-3 accurate -- enough to flip the detector's hard
// window tests (cad:217-218) against the fp32 reference -- so every fp32 operand is split in shared memory into hi = tf32(x) and the
// residual lo = x - hi, and three MMAs accumulate  hi*hi + lo*hi + hi*lo  in the fp32 TMEM accumulator (the dropped lo*lo term is 2^-22
// relative): the result matches an fp32 FMA GEMM to ~1e-6 while running on the tensor pipe instead of 137 us of FFMA.
//
// Pipeline per CTA (one 128 x 128 output tile and one slice of K; split-K over gridDim.z fills the machine):
//   warp 0      TMA producer: 128 x 32-float boxes of A and W (128-byte rows, SWIZZLE_128B) into a 3-stage ring;
//   warps 4-7   splitter: rewrite the landed tiles as hi in place and lo into the stage's twin buffers (same swizzled addresses, so no
//               layout arithmetic), then release the stage to the MMA warp;
//   warp 1      MMA issuer: 3 x 4 MMAs of M128 x N128 x K8 per stage;
//   warps 4-7   epilogue: TMEM -> registers -> shared memory -> global, coalesced red.add (one 128-byte row segment per warp instruction).
// Rows beyond M are zero-filled by TMA, so M = 32 (the classifier) uses the same kernel.  Bias / activation / dropout mask follow in
// cvad_bias_act_mask_f32, as for every split-K GEMM of linear_f32.cu.
#include <cuda.h>

#include "common.cuh"
#include "cvad_b200.h"
#include "tc_common.cuh"

namespace {

using namespace cvad_tc;

constexpr int TG_BM = 128, TG_BN = 128, TG_BK = 32;          // tile; BK floats = one 128-byte swizzle row
constexpr int TG_STAGES = 3;
constexpr int TG_TILE_BYTES = TG_BM * TG_BK * 4;             // 16 KiB per operand tile
constexpr int TG_STAGE_BYTES = 4 * TG_TILE_BYTES;            // A, W, A_lo, W_lo
constexpr size_t TG_SMEM = (size_t)TG_STAGES * TG_STAGE_BYTES + 1024;

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__global__ void __launch_bounds__(256, 1) gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                                                             float* __restrict__ C, int M, int N, int k_chunks_per_split, int k_chunks) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_full[TG_STAGES], bar_ready[TG_STAGES], bar_empty[TG_STAGES], bar_done;
  __shared__ uint32_t tmem_base_sh;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int m0 = blockIdx.x * TG_BM, n0 = blockIdx.y * TG_BN;
  const int c_begin = blockIdx.z * k_chunks_per_split;
  int c_end = c_begin + k_chunks_per_split;
  if (c_end > k_chunks) c_end = k_chunks;
  const int n_iter = c_end > c_begin ? c_end - c_begin : 0;

  if (tid == 0) {
    for (int i = 0; i < TG_STAGES; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_ready[i], 128); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_done, 1);
    fence_barrier_init();
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w);
  }
  if (warp == 2) tmem_alloc<128>(&tmem_base_sh);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    for (int it = 0; it < n_iter; ++it) {
      const int st = it % TG_STAGES;
      mbar_wait(&bar_empty[st], ((it / TG_STAGES) & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&bar_full[st], 2 * TG_TILE_BYTES);
        const uint32_t dst = smem_base + st * TG_STAGE_BYTES;
        const int k0 = (c_begin + it) * TG_BK;
        tma_load_2d(dst, &map_a, k0, m0, &bar_full[st]);
        tma_load_2d(dst + TG_TILE_BYTES, &map_w, k0, n0, &bar_full[st]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    uint32_t idesc = 0;
    idesc |= 1u << 4;                        // D = f32
    idesc |= 2u << 7;                        // A = tf32
    idesc |= 2u << 10;                       // B = tf32
    idesc |= (uint32_t)(TG_BN >> 3) << 17;
    idesc |= (uint32_t)(TG_BM >> 4) << 24;
    const uint64_t desc_hi = make_smem_desc(0, 16, 1024, UMMA_SW128);      // K-major, 128-byte rows, 8-row groups 1 KiB apart
    for (int it = 0; it < n_iter; ++it) {
      const int st = it % TG_STAGES;
      mbar_wait(&bar_ready[st], (it / TG_STAGES) & 1);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_hi = smem_base + st * TG_STAGE_BYTES, w_hi = a_hi + TG_TILE_BYTES, a_lo = a_hi + 2 * TG_TILE_BYTES,
                       w_lo = a_hi + 3 * TG_TILE_BYTES;
        const uint64_t dah = desc_hi | (uint64_t)((a_hi >> 4) & 0x3FFF), dwh = desc_hi | (uint64_t)((w_hi >> 4) & 0x3FFF);
        const uint64_t dal = desc_hi | (uint64_t)((a_lo >> 4) & 0x3FFF), dwl = desc_hi | (uint64_t)((w_lo >> 4) & 0x3FFF);
#pragma unroll
        for (int k = 0; k < TG_BK / 8; ++k) {                               // +32 bytes per K8 step
          tc_mma_tf32(tmem_base, dal + 2 * k, dwh + 2 * k, idesc, (it | k) != 0);      // small terms first
          tc_mma_tf32(tmem_base, dah + 2 * k, dwl + 2 * k, idesc, 1u);
          tc_mma_tf32(tmem_base, dah + 2 * k, dwh + 2 * k, idesc, 1u);
        }
        tc_commit(&bar_empty[st]);
      }
      __syncwarp();
    }
    if (elect_one()) tc_commit(&bar_done);
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------ splitter: x -> (tf32(x), x - tf32(x)) on both operand tiles
    const int t = tid - 128;                                     // 0..127
    for (int it = 0; it < n_iter; ++it) {
      const int st = it % TG_STAGES;
      mbar_wait(&bar_full[st], (it / TG_STAGES) & 1);
      float4* hi = reinterpret_cast<float4*>(smem_gen + st * TG_STAGE_BYTES);                 // A then W: 2 x 16 KiB = 2048 float4
      float4* lo = reinterpret_cast<float4*>(smem_gen + st * TG_STAGE_BYTES + 2 * TG_TILE_BYTES);
#pragma unroll 4
      for (int i = t; i < 2 * TG_TILE_BYTES / 16; i += 128) {
        const float4 v = hi[i];
        float4 h, l;
        h.x = to_tf32(v.x); h.y = to_tf32(v.y); h.z = to_tf32(v.z); h.w = to_tf32(v.w);
        l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
        hi[i] = h;
        lo[i] = l;
      }
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");          // generic-proxy writes -> visible to the tensor core's async proxy
      mbar_arrive(&bar_ready[st]);
    }
    if (n_iter > 0) {
      // ---------------------------------------------------------- epilogue: TMEM -> smem (row per thread) -> coalesced red.add
      mbar_wait(&bar_done, 0);
      tc_fence_after();
      const int ew = warp - 4;                                     // TMEM lanes 32*ew ..
      const int row = ew * 32 + lane;
      constexpr int LD = TG_BN + 1;                                // padded row pitch (floats): conflict-free row writes
      float* tile = reinterpret_cast<float*>(smem_gen);            // the pipeline buffers are free now: 128 x 129 floats = 66 KB
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16);
#pragma unroll
      for (int c0 = 0; c0 < TG_BN; c0 += 16) {
        uint32_t v[16];
        tmem_ld16(taddr + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 16; ++i) tile[row * LD + c0 + i] = __uint_as_float(v[i]);
      }
      __syncwarp();                                                // each warp reads back only the 32 rows it wrote
      for (int r = 0; r < 32; ++r) {
        const int m = m0 + ew * 32 + r;
        if (m >= M) break;
        float* crow = C + (long long)m * N + n0;
#pragma unroll
        for (int c = lane; c < TG_BN; c += 32)
          if (n0 + c < N) atomicAdd(crow + c, tile[(ew * 32 + r) * LD + c]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<128>(tmem_base);
}

}  // namespace

// y (M,N) fp32 must be ZERO on entry (split-K partial sums are added atomically); x (M,K), w (N,K) fp32 row-major, 16-byte aligned, K % 32 == 0.
CVAD_API int cvad_linear_fwd_tf32x3(const float* x, const float* w, float* y, int M, int N, int K, void* stream) {
  if (M <= 0 || N <= 0) return 0;
  if (K <= 0 || K % TG_BK || (((uintptr_t)x | (uintptr_t)w) & 15)) return (int)cudaErrorInvalidValue;
  CUtensorMap ma, mw;
  // 128 rows x 32 floats per box (one 128-byte swizzle row); rows past M / N read as zero
  int e = make_tmap_2d(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, x, M, K, TG_BM, TG_BK, 128);
  if (e) return e;
  e = make_tmap_2d(&mw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w, N, K, TG_BM, TG_BK, 128);
  if (e) return e;
  const int tiles = ((M + TG_BM - 1) / TG_BM) * ((N + TG_BN - 1) / TG_BN);
  const int k_chunks = K / TG_BK;
  int splits = cvad_num_sms() / tiles;
  if (splits < 1) splits = 1;
  if (splits > k_chunks) splits = k_chunks;
  const int per = (k_chunks + splits - 1) / splits;
  splits = (k_chunks + per - 1) / per;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(gemm_tf32x3_kernel, TG_SMEM, configured);
  if (ce != cudaSuccess) return (int)ce;
  gemm_tf32x3_kernel<<<dim3((M + TG_BM - 1) / TG_BM, (N + TG_BN - 1) / TG_BN, splits), 256, TG_SMEM, (cudaStream_t)stream>>>(ma, mw, y, M, N, per,
                                                                                                                               k_chunks);
  CVAD_LAUNCH_CHECK();
  return 0;
}

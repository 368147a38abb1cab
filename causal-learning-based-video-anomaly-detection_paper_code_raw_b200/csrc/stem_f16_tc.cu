// Stem of the M-A backbone, second formulation: conv 7x7 stride 2 pad 3, 1 -> 32 channels (cad:115, 145) as a tcgen05 kind::f16 implicit
// GEMM over a 2x4 space-to-depth of the frames, fused with the BatchNorm batch statistics (pass 1) or with BN + ReLU + MaxPool2d(3,2,1)
// (pass 2, cad:116-118, 146-148).  Frames whose width is a multiple of 4 take this path; stem_tc.cu (kind::tf32 over a 2x2
// space-to-depth) stays the general one.
//
// Why.  The tf32 form issues, per 128 output pixels, 8 MMAs of M128 x N32 x K8 whose operands (5 KB each) stream from shared memory:
// 66 cycles apiece against 16 of math, and in pass 2 that stream plus the max-pool's parked band saturate the shared-memory pipe
// (profiles/r02c_stem_pool_ncu_full.md).  Here X8[n][i][J][a*4+b] = x[n][2(i-2)+a][4(J-1)+b] (zero outside the frame) is an NHWC tensor
// of fp16 with 8 channels = one 16-byte "pixel" that covers a 2 x 4 patch of the frame, i.e. TWO horizontally adjacent outputs of the
// stride-2 convolution.  An accumulator row is such a pixel and carries N = 64 columns = (output parity p, channel), and over the flat
// pixel index q of X8 (geometry (Ho+3) x (Wo/2+2) per frame)
//        out[q][p*32 + c] = sum_{u<4, v<3} X8[q + u*Wq + v][0:8] * W8[u][v][p][c]      (kh = 2u+a-1, kw = 4v+b-2p-1)
// is 6 MMAs of M128 x N64 x K16 per 128 pixels = 256 outputs (the two 16-byte K chunks of an MMA are the pixel rows u and u+1: LBO = one
// row of X8): 2.3x fewer tensor-core cycles and 2.2x fewer operand bytes than the tf32 form.  Inputs are exact in fp16 whenever they are
// exact in tf32 (both keep 11 significant bits; the loader's 0..255 grayscale values through Normalize(0.5, 0.5) are odd integers below
// 512); weights are rounded to nearest fp16 where the tf32 MMA truncates.
//
// Kernels: persistent and warp-specialised like stem_tc.cu (warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM owner, warps 4-11
// epilogue in two groups on alternate sub-tiles).  The pixel stream is copied by TMA as is; tcgen05.mma performs the im2col through its
// no-swizzle K-major descriptors.
#include <cuda_fp16.h>

#include "common.cuh"
#include "cvad_b200.h"
#include "tc_common.cuh"

namespace {

using namespace cvad_tc;

constexpr int S8_C = 32;              // output channels
constexpr int S8_N = 64;              // accumulator columns: (parity, channel)
constexpr int S8_K = 7;               // kernel size
constexpr int S8_SLOTS = 8;           // TMEM accumulator ring (8 x 64 columns)
constexpr int S8_SUB = 4;             // 128-pixel sub-tiles per tile (pass 1)
constexpr int S8_MMAS = 6;            // (u0 in {0,2}) x (v in {0,1,2})
constexpr int S8_W_BYTES = S8_MMAS * 2048;   // [mma][2 K chunks][64 rows][16 B]
constexpr int S8_P = 4;               // pooled rows per band (pass 2)
constexpr int S8_ROWS = 2 * S8_P + 1; // convolution rows per band

struct Geo8 {
  int N, H, W, Ho, Wo, Wh, Hq, Wq;    // Wh = outputs pairs per row, Wq = Wh + 2
  long long np;                        // N*Hq*Wq pixels of X8 (= GEMM rows incl. junk)
  long long n_tiles;
  int seg_rows;                        // 128-byte rows (8 pixels) per stream segment of pass 1
};

struct Pool8 {
  int PH, PW, bands_per_frame, sub, seg_rows, tile_pitch;
  long long n_items;
};

// x (N,1,H,W) fp32 or uint8 -> X8 (N,Hq,Wq,8) fp16: one 16-byte pixel per thread; W % 4 == 0, so a pixel's four columns are one aligned
// 16-byte (fp32) / 4-byte (uint8) load per frame row.  uint8: x = (float(v) - mean) / std as torchvision's Normalize computes it.
template <bool U8>
__global__ void stem8_s2d_kernel(const void* __restrict__ xin, Geo8 g, float mean, float stdv, uint4* __restrict__ x8) {
  // np < 2^31 (geo8): 32-bit index arithmetic.  Four pixels per thread and iteration, their eight loads issued before the first is
  // consumed: with one pixel per iteration the kernel ran at 2.2 TB/s, latency-bound on two 4-byte loads per thread.
  constexpr int U = 4;
  const unsigned np = (unsigned)g.np, step = gridDim.x * blockDim.x;
  for (unsigned t0 = blockIdx.x * blockDim.x + threadIdx.x; t0 < np; t0 += U * step) {
    uint4 raw[U][2];               // fp32: the four columns of one frame row; uint8: .x holds them
    bool ok[U][2];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const unsigned t = t0 + k * step;
      const unsigned r = t / (unsigned)g.Wq;
      const int J = (int)(t - r * (unsigned)g.Wq);
      const unsigned nn = r / (unsigned)g.Hq;
      const int i = (int)(r - nn * (unsigned)g.Hq);
      const int h0 = 2 * (i - 2), w0 = 4 * (J - 1);
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const int h = h0 + a;
        ok[k][a] = t < np && (unsigned)h < (unsigned)g.H && w0 >= 0 && w0 < g.W;
        raw[k][a] = make_uint4(0, 0, 0, 0);
        if (ok[k][a]) {
          const long long off = ((long long)nn * g.H + h) * g.W + w0;
          if (U8) raw[k][a].x = __ldg(reinterpret_cast<const unsigned*>(reinterpret_cast<const uint8_t*>(xin) + off));
          else raw[k][a] = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(xin) + off));
        }
      }
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const unsigned t = t0 + k * step;
      if (t >= np) break;
      float v[8];
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        if (!ok[k][a]) {
#pragma unroll
          for (int b = 0; b < 4; ++b) v[a * 4 + b] = 0.f;
        } else if (U8) {
          const unsigned q = raw[k][a].x;
#pragma unroll
          for (int b = 0; b < 4; ++b) v[a * 4 + b] = ((float)((q >> (8 * b)) & 255u) - mean) / stdv;
        } else {
          v[a * 4 + 0] = __uint_as_float(raw[k][a].x); v[a * 4 + 1] = __uint_as_float(raw[k][a].y);
          v[a * 4 + 2] = __uint_as_float(raw[k][a].z); v[a * 4 + 3] = __uint_as_float(raw[k][a].w);
        }
      }
      uint4 o;
      __half2* hp = reinterpret_cast<__half2*>(&o);
#pragma unroll
      for (int q = 0; q < 4; ++q) hp[q] = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
      x8[t] = o;
    }
  }
}

__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// conv1 weights (32,1,7,7) fp32 -> shared memory [mma = (u0/2)*3 + v][chunk c][n = p*32 + cout][e = a*4 + b] fp16
// chan_scale (shared memory, may be NULL): a per-output-channel factor folded into the weights before they are rounded
__device__ __forceinline__ void stage_weights8(const float* __restrict__ w, uint8_t* smem_w, const float* chan_scale) {
  __half* dst = reinterpret_cast<__half*>(smem_w);
  for (int i = threadIdx.x; i < S8_MMAS * 2 * S8_N * 8; i += blockDim.x) {
    const int e = i & 7, n = (i >> 3) & 63, c = (i >> 9) & 1, m = i >> 10;
    const int u = 2 * (m / 3) + c, v = m % 3, a = e >> 2, b = e & 3, p = n >> 5, co = n & 31;
    const int kh = 2 * u + a - 1, kw = 4 * v + b - 2 * p - 1;
    float val = ((unsigned)kh < (unsigned)S8_K && (unsigned)kw < (unsigned)S8_K) ? w[co * S8_K * S8_K + kh * S8_K + kw] : 0.f;
    if (chan_scale) val *= chan_scale[co];
    dst[i] = __float2half_rn(val);
  }
}

__device__ __forceinline__ uint32_t idesc_f16_m128_n64() {
  uint32_t d = 0;
  d |= 1u << 4;                         // D = f32; A = B = f16 (format 0), both K-major
  d |= (uint32_t)(S8_N >> 3) << 17;
  d |= (uint32_t)(128 >> 4) << 24;
  return d;
}

// the six MMAs of one 128-pixel sub-tile whose first pixel sits at shared-memory address a0 (16-byte pixels)
__device__ __forceinline__ void issue_subtile8(uint32_t tmem_acc, uint32_t a0, uint32_t s_w, int Wq, uint64_t da_hi, uint64_t db_hi, uint32_t idesc) {
#pragma unroll
  for (int m = 0; m < S8_MMAS; ++m) {
    const uint32_t a_addr = a0 + (uint32_t)(2 * (m / 3) * Wq + (m % 3)) * 16;
    const uint64_t da = da_hi | (uint64_t)((a_addr >> 4) & 0x3FFF);
    const uint64_t db = db_hi | (uint64_t)(((s_w + m * 2048) >> 4) & 0x3FFF);
    tc_mma_f16(tmem_acc, da, db, idesc, m != 0);
  }
}

// ------------------------------------------------------------------------------------------------ pass 1: batch statistics
__global__ void __launch_bounds__(384, 1) stem8_stats_kernel(const __grid_constant__ CUtensorMap map_x8, const float* __restrict__ w, Geo8 g,
                                                             double* __restrict__ ws) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_seg_full[2], bar_seg_empty[2], bar_acc_full[S8_SLOTS], bar_acc_empty[S8_SLOTS];
  __shared__ uint32_t tmem_base_sh;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)g.seg_rows * 128;
  const uint32_t s_w = smem_base, s_seg = smem_base + S8_W_BYTES;
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  constexpr int MT = 128 * S8_SUB;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_seg_full[i], 1); mbar_init(&bar_seg_empty[i], 1); }
    for (int i = 0; i < S8_SLOTS; ++i) { mbar_init(&bar_acc_full[i], 1); mbar_init(&bar_acc_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(&map_x8);
  }
  stage_weights8(w, smem_gen, nullptr);
  if (warp == 2) tmem_alloc<512>(&tmem_base_sh);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    uint32_t cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      mbar_wait(&bar_seg_empty[st], ((cnt >> 1) & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&bar_seg_full[st], seg_bytes);
        tma_load_2d(s_seg + st * seg_bytes, &map_x8, 0, (int)(t * (MT / 8)), &bar_seg_full[st]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    const uint32_t idesc = idesc_f16_m128_n64();
    const uint64_t da_hi = make_smem_desc(0, (uint32_t)g.Wq * 16, 128, UMMA_NOSW);    // K chunk 1 = the pixel one X8 row below
    const uint64_t db_hi = make_smem_desc(0, 1024, 128, UMMA_NOSW);
    uint32_t cnt = 0, acc_cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      mbar_wait(&bar_seg_full[st], (cnt >> 1) & 1);
      tc_fence_after();
      const uint32_t seg = s_seg + st * seg_bytes;
      for (int s = 0; s < S8_SUB; ++s) {
        const uint32_t use = acc_cnt + s;
        const int slot = use % S8_SLOTS;
        mbar_wait(&bar_acc_empty[slot], ((use / S8_SLOTS) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          issue_subtile8(tmem_base + slot * S8_N, seg + (uint32_t)(s * 128) * 16, s_w, g.Wq, da_hi, db_hi, idesc);
          tc_commit(&bar_acc_full[slot]);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(&bar_seg_empty[st]);
      __syncwarp();
      acc_cnt += S8_SUB;
    }
  } else if (warp >= 4) {
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    float s[S8_C], q[S8_C];                    // per-channel sum / sum of squares over this thread's valid outputs
#pragma unroll
    for (int c = 0; c < S8_C; ++c) { s[c] = 0.f; q[c] = 0.f; }
    const int frame = g.Hq * g.Wq;
    uint32_t acc_cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
      for (int sb = eg; sb < S8_SUB; sb += 2) {
        const uint32_t use = acc_cnt + sb;
        const int slot = use % S8_SLOTS;
        mbar_wait(&bar_acc_full[slot], (use / S8_SLOTS) & 1);
        tc_fence_after();
        uint32_t a[4][16];
        const uint32_t taddr = tmem_base + slot * S8_N + ((uint32_t)(ew * 32) << 16);
#pragma unroll
        for (int k = 0; k < 4; ++k) tmem_ld16(taddr + 16 * k, a[k]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&bar_acc_empty[slot]);
        const uint32_t qq = (uint32_t)(t * MT) + sb * 128 + ew * 32 + lane;
        const uint32_t n = qq / (uint32_t)frame;
        const uint32_t rem = qq - n * (uint32_t)frame;
        const int i = (int)(rem / (uint32_t)g.Wq), J = (int)(rem - (uint32_t)i * (uint32_t)g.Wq);
        if ((long long)qq < g.np && i < g.Ho && J < g.Wh) {
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const float y0 = __uint_as_float(a[0][c]), y1 = __uint_as_float(a[1][c]);
            s[c] += y0; q[c] = fmaf(y0, y0, q[c]);
            s[16 + c] += y1; q[16 + c] = fmaf(y1, y1, q[16 + c]);
          }
          if (2 * J + 1 < g.Wo) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              const float y0 = __uint_as_float(a[2][c]), y1 = __uint_as_float(a[3][c]);
              s[c] += y0; q[c] = fmaf(y0, y0, q[c]);
              s[16 + c] += y1; q[16 + c] = fmaf(y1, y1, q[16 + c]);
            }
          }
        }
      }
      acc_cnt += S8_SUB;
    }
    // CTA reduction over the 256 row-threads (the stream segments are free: every MMA retired before its acc_full fired)
    float* red = reinterpret_cast<float*>(smem_gen + S8_W_BYTES);          // [256][65]
    const int r = tid - 128;
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
#pragma unroll
    for (int c = 0; c < S8_C; ++c) { red[r * 65 + c] = s[c]; red[r * 65 + 32 + c] = q[c]; }
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
    if (r < 64) {
      double acc = 0.0;
      for (int k = 0; k < 256; ++k) acc += (double)red[k * 65 + r];
      atomicAdd(ws + r, acc);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------------ pass 2: BN + ReLU + MaxPool2d(3,2,1)
// A work item is a BAND of one frame: S8_P pooled rows = the 2*S8_P + 1 convolution rows 2*S8_P*b - 1 .. 2*S8_P*b + 2*S8_P - 1 (one row of
// overlap with the next band).  Its pixels are contiguous in the flat X8 index: one TMA box per band, `sub` sub-tiles of 128 pixels,
// six MMAs each.  The epilogue applies BN + ReLU and parks the band as bf16 [row][column][32] in shared memory; when the band is complete
// the eight epilogue warps pool it (post-ReLU values: an absent neighbour is a 0) and write the padded-flat rows of layer1's input.
// A thread holds BOTH outputs of its pixel, so the horizontal part of the pooling window starts in registers: per band row it parks
// M[J] = max(y[2J], y[2J+1]) and X[J] = y[2J+1] (two planes of Wo/2 pixels; Wo is even on this path), and a pooled value is the maximum
// over three rows of max(M[pw], X[pw-1]) -- six shared-memory loads instead of nine, on the pipe the MMAs stream their operands through.
// A pixel's four 16-byte vectors are XOR-swizzled by (J >> 1) & 3: parking stores (lanes = consecutive pixels) and pooling reads are both
// bank-conflict free.
constexpr int S8_EG = 3;              // epilogue groups of pass 2 (4 warps each): 128 + 3 * 128 = 512 threads
__global__ void __launch_bounds__(128 + 128 * S8_EG, 1) stem8_pool_kernel(const __grid_constant__ CUtensorMap map_x8, const float* __restrict__ w,
                                                            const float* __restrict__ bias, Geo8 g, Pool8 pg, const float* __restrict__ mean,
                                                            const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, __nv_bfloat16* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_seg_full[2], bar_seg_empty[2], bar_acc_full[S8_SLOTS], bar_acc_empty[S8_SLOTS];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float s_sc[S8_C], s_sh[S8_C];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)pg.seg_rows * 128;
  const uint32_t s_w = smem_base, s_seg = smem_base + S8_W_BYTES;
  __nv_bfloat16* band = reinterpret_cast<__nv_bfloat16*>(smem_gen + S8_W_BYTES + 2 * seg_bytes);       // [S8_ROWS][tile_pitch]
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int sub = pg.sub;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_seg_full[i], 1); mbar_init(&bar_seg_empty[i], 1); }
    for (int i = 0; i < S8_SLOTS; ++i) { mbar_init(&bar_acc_full[i], 1); mbar_init(&bar_acc_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(&map_x8);
  }
  // The BatchNorm scale gamma * invstd goes INTO the weights (times a power of two that brings the largest scale to ~1, so that small
  // weights do not fall into fp16's subnormals): the epilogue is then relu(acc * 2^-k + shift) with ONE scalar instead of 32 per-channel
  // scales -- the 32 registers that let the kernel run three epilogue groups (512 threads: 128 registers per thread).
  __shared__ float s_kinv;
  if (warp == 0) {
    const float sc = invstd[lane] * gamma[lane];
    float mx = fabsf(sc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float k = mx > 0.f ? exp2f(-rintf(log2f(mx))) : 1.f;
    s_sc[lane] = sc * k;
    s_sh[lane] = (bias[lane] - mean[lane]) * sc + beta[lane];
    if (lane == 0) s_kinv = 1.f / k;
  }
  __syncthreads();
  stage_weights8(w, smem_gen, s_sc);
  if (warp == 2) tmem_alloc<512>(&tmem_base_sh);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  // first flat X8 pixel of work item t (negative for the first band of the first frame: TMA zero-fills)
  auto item_start = [&](long long t) -> long long {
    const long long n = t / pg.bands_per_frame;
    const int b = (int)(t - n * pg.bands_per_frame);
    return (n * g.Hq + (2 * S8_P * b - 1)) * (long long)g.Wq;
  };

  if (warp == 0) {
    uint32_t cnt = 0;
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      mbar_wait(&bar_seg_empty[st], ((cnt >> 1) & 1) ^ 1);
      if (elect_one()) {
        const long long p0 = item_start(t);
        const long long row = p0 >= 0 ? p0 / 8 : -((-p0 + 7) / 8);          // floor(p0 / 8)
        mbar_expect_tx(&bar_seg_full[st], seg_bytes);
        tma_load_2d(s_seg + st * seg_bytes, &map_x8, 0, (int)row, &bar_seg_full[st]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    const uint32_t idesc = idesc_f16_m128_n64();
    const uint64_t da_hi = make_smem_desc(0, (uint32_t)g.Wq * 16, 128, UMMA_NOSW);
    const uint64_t db_hi = make_smem_desc(0, 1024, 128, UMMA_NOSW);
    uint32_t cnt = 0, acc_cnt = 0;
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      const long long p0 = item_start(t);
      const long long row = p0 >= 0 ? p0 / 8 : -((-p0 + 7) / 8);
      const int off = (int)(p0 - row * 8);                          // 0..7 pixels into the box
      mbar_wait(&bar_seg_full[st], (cnt >> 1) & 1);
      tc_fence_after();
      const uint32_t seg = s_seg + st * seg_bytes;
      for (int s = 0; s < sub; ++s) {
        const uint32_t use = acc_cnt + s;
        const int slot = use % S8_SLOTS;
        mbar_wait(&bar_acc_empty[slot], ((use / S8_SLOTS) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          issue_subtile8(tmem_base + slot * S8_N, seg + (uint32_t)(off + s * 128) * 16, s_w, g.Wq, da_hi, db_hi, idesc);
          tc_commit(&bar_acc_full[slot]);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(&bar_seg_empty[st]);
      __syncwarp();
      acc_cnt += sub;
    }
  } else if (warp >= 4) {
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    const int et = tid - 128;                                       // 0 .. 128*S8_EG - 1 among the epilogue threads
    constexpr int ET = 128 * S8_EG;
    uint32_t acc_cnt = 0;
    const int groups = S8_C / 8;                                    // 16-byte vectors per pixel
    float rq[S8_C];                                                 // BatchNorm shift in registers (the scale sits in the weights)
#pragma unroll
    for (int c = 0; c < S8_C; ++c) rq[c] = s_sh[c];
    const float kinv = s_kinv;
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x) {
      const long long n = t / pg.bands_per_frame;
      const int b = (int)(t - n * pg.bands_per_frame);
      const int i0 = 2 * S8_P * b - 1;                              // first convolution row of the band
      for (int sb = eg; sb < sub; sb += S8_EG) {
        const uint32_t use = acc_cnt + sb;
        const int slot = use % S8_SLOTS;
        mbar_wait(&bar_acc_full[slot], (use / S8_SLOTS) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + slot * S8_N + ((uint32_t)(ew * 32) << 16);
        const int ql = sb * 128 + ew * 32 + lane;                   // pixel inside the band
        const int r = ql / g.Wq, J = ql - r * g.Wq;
        const bool row_in = r < S8_ROWS && J < g.Wh;
        const bool live = row_in && i0 + r >= 0 && i0 + r < g.Ho;
        // all four 16-column loads of the row (both outputs) in flight before the single wait: one TMEM round trip per sub-tile, not two
        uint32_t acc[4][16];
#pragma unroll
        for (int k = 0; k < 4; ++k) tmem_ld16(taddr + 16 * k, acc[k]);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&bar_acc_empty[slot]);
        uint32_t pk0[16], pk1[16];
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          uint32_t* pk = p ? pk1 : pk0;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float y0 = fmaxf(fmaf(__uint_as_float(acc[2 * p][2 * c]), kinv, rq[2 * c]), 0.f);
            const float y1 = fmaxf(fmaf(__uint_as_float(acc[2 * p][2 * c + 1]), kinv, rq[2 * c + 1]), 0.f);
            const float z0 = fmaxf(fmaf(__uint_as_float(acc[2 * p + 1][2 * c]), kinv, rq[16 + 2 * c]), 0.f);
            const float z1 = fmaxf(fmaf(__uint_as_float(acc[2 * p + 1][2 * c + 1]), kinv, rq[16 + 2 * c + 1]), 0.f);
            __nv_bfloat162 h0 = __floats2bfloat162_rn(y0, y1), h1 = __floats2bfloat162_rn(z0, z1);
            pk[c] = *reinterpret_cast<uint32_t*>(&h0);
            pk[8 + c] = *reinterpret_cast<uint32_t*>(&h1);
          }
        }
        if (row_in) {
          if (!live) {                                               // rows outside the frame: post-ReLU zeros never win a max
#pragma unroll
            for (int c = 0; c < 16; ++c) { pk0[c] = 0u; pk1[c] = 0u; }
          }
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const __nv_bfloat162 m = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&pk0[c]), *reinterpret_cast<__nv_bfloat162*>(&pk1[c]));
            pk0[c] = *reinterpret_cast<const uint32_t*>(&m);
          }
          const int sw = (J >> 1) & 3;
          uint4* om = reinterpret_cast<uint4*>(band + (size_t)r * pg.tile_pitch + (size_t)J * S8_C);
          uint4* ox = reinterpret_cast<uint4*>(band + (size_t)r * pg.tile_pitch + (size_t)(g.Wh + J) * S8_C);
          om[0 ^ sw] = make_uint4(pk0[0], pk0[1], pk0[2], pk0[3]);
          om[1 ^ sw] = make_uint4(pk0[4], pk0[5], pk0[6], pk0[7]);
          om[2 ^ sw] = make_uint4(pk0[8], pk0[9], pk0[10], pk0[11]);
          om[3 ^ sw] = make_uint4(pk0[12], pk0[13], pk0[14], pk0[15]);
          ox[0 ^ sw] = make_uint4(pk1[0], pk1[1], pk1[2], pk1[3]);
          ox[1 ^ sw] = make_uint4(pk1[4], pk1[5], pk1[6], pk1[7]);
          ox[2 ^ sw] = make_uint4(pk1[8], pk1[9], pk1[10], pk1[11]);
          ox[3 ^ sw] = make_uint4(pk1[12], pk1[13], pk1[14], pk1[15]);
        }
      }
      acc_cnt += sub;
      asm volatile("bar.sync 1, %0;\n" ::"n"(ET) : "memory");        // the band is complete
      // ---- pool: pooled rows S8_P*b .. S8_P*b + S8_P - 1 (band rows 2k, 2k+1, 2k+2 for the k-th of them), padded-flat output
      const int rowlen = (pg.PW + 2) * groups;                       // vectors per padded output row
      for (int v = et; v < S8_P * rowlen; v += ET) {
        const int k = v / rowlen, vv = v - k * rowlen;
        const int ph = S8_P * b + k;
        if (ph >= pg.PH) continue;
        const int pwp = vv / groups, cg = vv - pwp * groups;
        uint4 o = make_uint4(0, 0, 0, 0);
        if (pwp >= 1 && pwp <= pg.PW) {
          const int pw = pwp - 1;
          // window columns 2pw-1, 2pw, 2pw+1 = X[pw-1], M[pw]; all six loads before the first max.  pw = 0 has no left neighbour: X[0]
          // stands in (column 1, which M[0] covers anyway)
          uint4 tv[6];
          const int jx = pw > 0 ? pw - 1 : 0;
          const int offm = pw * S8_C + ((cg ^ ((pw >> 1) & 3)) * 8), offx = (g.Wh + jx) * S8_C + ((cg ^ ((jx >> 1) & 3)) * 8);
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            tv[2 * a] = *reinterpret_cast<const uint4*>(band + (size_t)(2 * k + a) * pg.tile_pitch + offm);
            tv[2 * a + 1] = *reinterpret_cast<const uint4*>(band + (size_t)(2 * k + a) * pg.tile_pitch + offx);
          }
          __nv_bfloat162 best[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) best[i] = reinterpret_cast<const __nv_bfloat162*>(&tv[0])[i];
#pragma unroll
          for (int t6 = 1; t6 < 6; ++t6)
#pragma unroll
            for (int i = 0; i < 4; ++i) best[i] = __hmax2(best[i], reinterpret_cast<const __nv_bfloat162*>(&tv[t6])[i]);
          o = *reinterpret_cast<uint4*>(best);
        }
        reinterpret_cast<uint4*>(out)[((n * (pg.PH + 2) + ph + 1) * (long long)rowlen) + vv] = o;
      }
      // the frame's top / bottom border rows belong to its first / last band
      if (b == 0)
        for (int v = et; v < rowlen; v += ET) reinterpret_cast<uint4*>(out)[(n * (pg.PH + 2)) * (long long)rowlen + v] = make_uint4(0, 0, 0, 0);
      if (b == pg.bands_per_frame - 1)
        for (int v = et; v < rowlen; v += ET)
          reinterpret_cast<uint4*>(out)[(n * (pg.PH + 2) + pg.PH + 1) * (long long)rowlen + v] = make_uint4(0, 0, 0, 0);
      asm volatile("bar.sync 1, %0;\n" ::"n"(ET) : "memory");        // the band buffer may be overwritten
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

int geo8(Geo8& g, int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0 || (W & 3)) return 1;
  g.N = N; g.H = H; g.W = W;
  g.Ho = (H - 1) / 2 + 1;
  g.Wo = (W - 1) / 2 + 1;
  g.Wh = (g.Wo + 1) / 2;
  g.Hq = g.Ho + 3;
  g.Wq = g.Wh + 2;
  g.np = (long long)N * g.Hq * g.Wq;
  const int MT = 128 * S8_SUB;
  g.n_tiles = (g.np + MT - 1) / MT;
  const int seg_px = MT + 3 * g.Wq + 2;
  g.seg_rows = (seg_px + 7) / 8;
  if (g.seg_rows > 256 || g.np + MT > 0x7fffffffLL) return 1;
  return 0;
}

int make_map8(CUtensorMap* mx, const void* x8, const Geo8& g, int box_rows) {
  // X8 as a matrix of 128-byte rows (8 pixels); the last partial row is covered by the buffer's slack
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return (int)cudaErrorNotSupported;
  memset(mx, 0, sizeof(*mx));
  cuuint64_t dims[2] = {32, (cuuint64_t)((g.np + 7) / 8)};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(mx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(x8), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

// pass-2 geometry; false when a band does not fit one TMA box / the accumulator ring / shared memory (very wide frames)
bool pool8_geo(const Geo8& g, Pool8& pg, size_t& smem) {
  pg.PH = (g.Ho - 1) / 2 + 1;
  pg.PW = (g.Wo - 1) / 2 + 1;
  pg.bands_per_frame = (pg.PH + S8_P - 1) / S8_P;
  pg.n_items = (long long)g.N * pg.bands_per_frame;
  pg.sub = (S8_ROWS * g.Wq + 127) / 128;
  const int seg_px = 128 * pg.sub + 3 * g.Wq + 2 + 8;              // + the pixel remainder of the box's 128-byte alignment
  pg.seg_rows = (seg_px + 7) / 8;
  pg.tile_pitch = ((g.Wo + 3) & ~3) * S8_C;
  const size_t band_bytes = (size_t)S8_ROWS * pg.tile_pitch * sizeof(__nv_bfloat16);
  smem = S8_W_BYTES + 2 * (size_t)pg.seg_rows * 128 + band_bytes + 1024;
  return pg.seg_rows <= 256 && pg.sub <= S8_SLOTS && smem <= 220 * 1024;
}

}  // namespace

// bytes of the X8 buffer for (N,1,H,W) frames (incl. the slack the last TMA row needs), or -1 when the shape is outside this path's range
// (W not a multiple of 4, very wide frames): callers then use the tf32 stem
CVAD_API long long cvad_stem8_bytes(int N, int H, int W) {
  Geo8 g;
  Pool8 pg;
  size_t smem;
  if (geo8(g, N, H, W) || !pool8_geo(g, pg, smem)) return -1;
  return ((g.np + 7) / 8) * 128 + 128;
}

CVAD_API int cvad_stem8_space_to_depth_f32(const float* x, int N, int H, int W, void* x8, void* stream) {
  Geo8 g;
  if (geo8(g, N, H, W) || ((uintptr_t)x & 15)) return (int)cudaErrorInvalidValue;
  long long blocks = (g.np + 255) / 256;
  if (blocks > 16LL * cvad_num_sms()) blocks = 16LL * cvad_num_sms();
  stem8_s2d_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, g, 0.f, 1.f, reinterpret_cast<uint4*>(x8));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_stem8_space_to_depth_u8(const void* x, int N, int H, int W, float mean, float stdv, void* x8, void* stream) {
  Geo8 g;
  if (geo8(g, N, H, W) || stdv == 0.f || ((uintptr_t)x & 3)) return (int)cudaErrorInvalidValue;
  long long blocks = (g.np + 255) / 256;
  if (blocks > 16LL * cvad_num_sms()) blocks = 16LL * cvad_num_sms();
  stem8_s2d_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, g, mean, stdv, reinterpret_cast<uint4*>(x8));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_stem8_f16_stats(const void* x8, const float* w, const float* bias, int N, int H, int W, double* ws, float eps, float momentum,
                                  float* mean, float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked,
                                  void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  Geo8 g;
  if (geo8(g, N, H, W)) return (int)cudaErrorInvalidValue;
  CUtensorMap mx;
  int e = make_map8(&mx, x8, g, g.seg_rows);
  if (e) return e;
  size_t smem = S8_W_BYTES + 2 * (size_t)g.seg_rows * 128 + 1024;
  const size_t red = S8_W_BYTES + 256 * 65 * 4 + 1024;
  if (smem < red) smem = red;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem8_stats_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > g.n_tiles) grid = g.n_tiles;
  stem8_stats_kernel<<<(unsigned)grid, 384, smem, st>>>(mx, w, g, ws);
  CVAD_LAUNCH_CHECK();
  // ws holds the sums of the RAW accumulator; y = acc + bias: the bias moves the mean, not the variance
  return bn_finalize_launch(ws, S8_C, (double)N * g.Ho * g.Wo, bias, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked,
                            st);
}

CVAD_API int cvad_stem8_f16_bn_relu_maxpool(const void* x8, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                            const float* invstd, const float* gamma, const float* beta, void* out, void* stream) {
  Geo8 g;
  if (geo8(g, N, H, W)) return (int)cudaErrorInvalidValue;
  Pool8 pg;
  size_t smem;
  if (!pool8_geo(g, pg, smem)) return (int)cudaErrorNotSupported;
  CUtensorMap mx;
  int e = make_map8(&mx, x8, g, pg.seg_rows);
  if (e) return e;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem8_pool_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > pg.n_items) grid = pg.n_items;
  stem8_pool_kernel<<<(unsigned)grid, 128 + 128 * S8_EG, smem, (cudaStream_t)stream>>>(mx, w, bias, g, pg, mean, invstd, gamma, beta, (__nv_bfloat16*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

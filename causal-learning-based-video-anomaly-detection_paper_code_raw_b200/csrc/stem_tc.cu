// Stem of the M-A backbone on the tensor cores: conv 7x7 stride 2 pad 3, 1 -> 32 channels (cad:115, 145) as a
// tcgen05 kind::tf32 implicit GEMM, fused with the BatchNorm batch statistics (pass 1) or with BN + ReLU (pass 2);
// MaxPool2d(3,2,1) (cad:118,148) follows as a 16-byte-vector bandwidth kernel that writes the padded-flat bf16 layout.
//
// With one input channel an im2col row has no contiguous 16-byte piece, so neither TMA nor a UMMA descriptor can address it.
// A 2x2 space-to-depth turns the problem into one they can: X4[n][i][j][a*2+b] = x[n][2(i-2)+a][2(j-2)+b] (zero outside the
// frame) is an NHWC tensor with 4 fp32 channels = one 16-byte "pixel", and the 7x7 stride-2 convolution becomes a 4x4
// stride-1 convolution over it (kh = 2u+a-1, kw = 2v+b-1; the 15 combinations outside the 7x7 window get zero weights).
// Over the flat pixel index q of X4 (geometry (Ho+3) x (Wo+3) per frame) the output is
//        out[q][:] = sum_{u,v} X4[q + u*(Wo+3) + v][0:4] * W4[u][v]            (positions with i >= Ho or j >= Wo are junk)
// and the A operand of one MMA (K = 8 tf32 = two horizontally adjacent pixels) is a VIEW OF THE RAW PIXEL STREAM: rows are
// consecutive pixels (16-byte pitch = the no-swizzle core-matrix row pitch), the second K chunk is the same stream one pixel
// later (LBO = 16 B, overlapping), 8-row groups follow at SBO = 128 B.  So TMA copies the stream into shared memory as is
// (one box of up to 32 KiB per tile) and tcgen05.mma performs the im2col through its descriptor -- no thread touches an
// input element (profiles/r01_umma_descriptor_probe.md, config 15).
//
// Kernel: persistent, warp-specialised like flatconv_tc.cu -- warp 0 TMA producer (double-buffered stream segments), warp 1
// MMA issuer (8 MMAs of M=128, N=32, K=8 per 128 positions, 16-slot TMEM accumulator ring), warp 2 TMEM owner, warps 4-11
// epilogue (two groups on alternate sub-tiles): pass 1 accumulates per-channel sum / sum of squares of the valid rows in registers across the whole CTA (no
// convolution output is ever written), pass 2 applies BN + ReLU and stores bf16 NHWC rows.
// The frozen stem needs no gradient (cad:596-598).  fp32 inputs are rounded to tf32 (10-bit mantissa) by the MMA.
#include "common.cuh"
#include "cvad_b200.h"
#include "tc_common.cuh"

namespace {

using namespace cvad_tc;

constexpr int ST_C = 32;             // output channels
constexpr int ST_K = 7;              // kernel size
constexpr int ST_SUB = 8;            // 128-position sub-tiles per tile
constexpr int ST_SLOTS = 16;         // TMEM accumulator ring (16 x 32 columns)
constexpr int ST_W_BYTES = 8 * 1024; // 8 MMAs x [2 chunks][32 rows][16 B]

struct StemGeo {
  int N, H, W, Ho, Wo, Hq, Wq;
  long long np4;          // N*Hq*Wq pixels of X4 (= GEMM rows incl. junk)
  long long n_tiles;
  int seg_rows;           // 128-byte rows (8 pixels) per stream segment
};

__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// x (N,1,H,W) fp32 -> X4 (N,Hq,Wq,4) fp32, one 16-byte pixel per thread
__global__ void stem_s2d_kernel(const float* __restrict__ x, StemGeo g, float4* __restrict__ x4) {
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < g.np4; t += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(t % g.Wq);
    const long long r = t / g.Wq;
    const int i = (int)(r % g.Hq), n = (int)(r / g.Hq);
    const int h0 = 2 * (i - 2), w0 = 2 * (j - 2);
    const float* xn = x + (long long)n * g.H * g.W;
    float v[4];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        const int h = h0 + a, w = w0 + b;
        v[a * 2 + b] = ((unsigned)h < (unsigned)g.H && (unsigned)w < (unsigned)g.W) ? __ldg(xn + (long long)h * g.W + w) : 0.f;
      }
    x4[t] = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// The same from uint8 frames (what cv2.imread hands the reference's dataset, cad:89-96): the Normalize(mean, std) of cad:1177-1179 is applied on the
// fly, x = (float(v) - mean) / std -- exactly torchvision's sub_().div_() on the FloatTensor, so the result is bit-identical to the fp32
// path while the frames cross PCIe and are read from HBM at 1 byte per pixel.  Conv padding stays 0 (it pads the NORMALISED tensor).
__global__ void stem_s2d_u8_kernel(const uint8_t* __restrict__ x, StemGeo g, float mean, float stdv, float4* __restrict__ x4) {
  // one thread = four horizontally adjacent X4 pixels = 8 source bytes from each of two frame rows (two aligned 4-byte loads per row when
  // the frame width is a multiple of 4) -> 64 contiguous output bytes
  const int wq4 = (g.Wq + 3) >> 2;
  const long long items = (long long)g.N * g.Hq * wq4;
  const bool aligned = (g.W & 3) == 0;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < items; t += (long long)gridDim.x * blockDim.x) {
    const int jq = (int)(t % wq4);
    const long long r = t / wq4;
    const int i = (int)(r % g.Hq), n = (int)(r / g.Hq);
    const int j0 = jq * 4;
    const int h0 = 2 * (i - 2), w0 = 2 * (j0 - 2);          // w0 = 4 (mod 8)
    const uint8_t* xn = x + (long long)n * g.H * g.W;
    float v[2][8];
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int h = h0 + a;
      const bool hok = (unsigned)h < (unsigned)g.H;
      const uint8_t* row = xn + (long long)h * g.W;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int w = w0 + 4 * half;
        if (hok && aligned && w >= 0 && w + 3 < g.W) {
          const unsigned q = __ldg(reinterpret_cast<const unsigned*>(row + w));
#pragma unroll
          for (int e = 0; e < 4; ++e) v[a][4 * half + e] = ((float)((q >> (8 * e)) & 255u) - mean) / stdv;
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) v[a][4 * half + e] = (hok && (unsigned)(w + e) < (unsigned)g.W) ? ((float)__ldg(row + w + e) - mean) / stdv : 0.f;
        }
      }
    }
    const long long o = (r * g.Wq) + j0;
#pragma unroll
    for (int p = 0; p < 4; ++p)
      if (j0 + p < g.Wq) x4[o + p] = make_float4(v[0][2 * p], v[0][2 * p + 1], v[1][2 * p], v[1][2 * p + 1]);
  }
}

// y = (float(v) - mean) / std over a flat uint8 buffer, 16 bytes in / 64 bytes out per thread iteration (fp32 mode of the same input path)
__global__ void u8_normalize_kernel(const uint8_t* __restrict__ x, long long n, float mean, float stdv, float* __restrict__ y) {
  const long long n16 = n / 16;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n16; t += (long long)gridDim.x * blockDim.x) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(x) + t);
    const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
      reinterpret_cast<float4*>(y)[t * 4 + k] = make_float4(((float)(w[k] & 255u) - mean) / stdv, ((float)((w[k] >> 8) & 255u) - mean) / stdv,
                                                             ((float)((w[k] >> 16) & 255u) - mean) / stdv, ((float)(w[k] >> 24) - mean) / stdv);
  }
  for (long long t = n16 * 16 + blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x)
    y[t] = ((float)__ldg(x + t) - mean) / stdv;
}

// MODE 0: statistics of the raw accumulator (ws[c] += sum acc, ws[32+c] += sum acc^2 over valid rows; the bias is folded in by
// the finalize kernel).  MODE 1: out = relu((acc + bias - mean) * invstd * gamma + beta) bf16 NHWC (N,Ho,Wo,32).
template <int MODE>
__global__ void __launch_bounds__(384, 1) stem_tf32_kernel(const __grid_constant__ CUtensorMap map_x4, const float* __restrict__ w,
                                                           const float* __restrict__ bias, StemGeo g, const float* __restrict__ mean,
                                                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, double* __restrict__ ws,
                                                           __nv_bfloat16* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_seg_full[2], bar_seg_empty[2], bar_acc_full[ST_SLOTS], bar_acc_empty[ST_SLOTS];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float s_sc[ST_C], s_sh[ST_C];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)g.seg_rows * 128;
  const uint32_t s_w = smem_base;                           // 8 KiB of packed weights
  const uint32_t s_seg = smem_base + ST_W_BYTES;            // 2 stream segments
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  constexpr int MT = 128 * ST_SUB;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_seg_full[i], 1); mbar_init(&bar_seg_empty[i], 1); }
    for (int i = 0; i < ST_SLOTS; ++i) { mbar_init(&bar_acc_full[i], 1); mbar_init(&bar_acc_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(&map_x4);
  }
  if (tid < ST_C) {
    const float sc = MODE == 1 ? invstd[tid] * gamma[tid] : 1.f;
    s_sc[tid] = sc;
    s_sh[tid] = MODE == 1 ? (bias[tid] - mean[tid]) * sc + beta[tid] : 0.f;
  }
  // weights -> [mma = u*2+vp][K chunk c][n][4 floats]; chunk c of MMA (u,vp) is tap column v = 2vp+c, element e = a*2+b
  for (int i = tid; i < 8 * 2 * ST_C * 4; i += blockDim.x) {
    const int e = i & 3, n = (i >> 2) & 31, c = (i >> 7) & 1, m = i >> 8;
    const int u = m >> 1, v = 2 * (m & 1) + c, a = e >> 1, b = e & 1;
    const int kh = 2 * u + a - 1, kw = 2 * v + b - 1;
    const float val = ((unsigned)kh < (unsigned)ST_K && (unsigned)kw < (unsigned)ST_K) ? w[n * ST_K * ST_K + kh * ST_K + kw] : 0.f;
    reinterpret_cast<float*>(smem_gen)[i] = val;
  }
  if (warp == 2) tmem_alloc<512>(&tmem_base_sh);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer: one box per tile
    uint32_t cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      mbar_wait(&bar_seg_empty[st], ((cnt >> 1) & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&bar_seg_full[st], seg_bytes);
        tma_load_2d(s_seg + st * seg_bytes, &map_x4, 0, (int)(t * (MT / 8)), &bar_seg_full[st]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    uint32_t idesc = 0;
    idesc |= 1u << 4;                 // D = f32
    idesc |= 2u << 7;                 // A = tf32
    idesc |= 2u << 10;                // B = tf32
    idesc |= (uint32_t)(ST_C >> 3) << 17;
    idesc |= (uint32_t)(128 >> 4) << 24;
    const uint64_t da_hi = make_smem_desc(0, 16, 128, UMMA_NOSW);     // pixel stream: K chunks overlap by one pixel
    const uint64_t db_hi = make_smem_desc(0, 512, 128, UMMA_NOSW);
    uint32_t cnt = 0, acc_cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      mbar_wait(&bar_seg_full[st], (cnt >> 1) & 1);
      tc_fence_after();
      const uint32_t seg = s_seg + st * seg_bytes;
      for (int s = 0; s < ST_SUB; ++s) {
        const uint32_t use = acc_cnt + s;
        const int slot = use % ST_SLOTS;
        mbar_wait(&bar_acc_empty[slot], ((use / ST_SLOTS) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const uint32_t a_addr = seg + (uint32_t)(s * 128 + (m >> 1) * g.Wq + 2 * (m & 1)) * 16;
            const uint64_t da = da_hi | (uint64_t)((a_addr >> 4) & 0x3FFF);
            const uint64_t db = db_hi | (uint64_t)(((s_w + m * 1024) >> 4) & 0x3FFF);
            tc_mma_tf32(tmem_base + slot * ST_C, da, db, idesc, m != 0);
          }
          tc_commit(&bar_acc_full[slot]);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(&bar_seg_empty[st]);
      __syncwarp();
      acc_cnt += ST_SUB;
    }
  } else if (warp >= 4) {
    // ---------------------------------------------------------------- epilogue: thread <-> TMEM lane (row) 32*(warp-4)+lane
    // two groups of four warps (warps 4-7 and 8-11) take alternate sub-tiles; warp w reads TMEM lanes 32*(w%4)..
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    // MODE 0: s / q are the per-channel sums.  MODE 1: s / q hold the BatchNorm scale / shift -- in REGISTERS: the MMAs stream their
    // operands from shared memory at the pipe's limit, and 64 broadcast loads per thread and sub-tile took a third of it away
    float s[ST_C], q[ST_C];
#pragma unroll
    for (int c = 0; c < ST_C; ++c) { s[c] = MODE == 0 ? 0.f : s_sc[c]; q[c] = MODE == 0 ? 0.f : s_sh[c]; }
    const int frame = g.Hq * g.Wq;
    uint32_t acc_cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
      for (int sb = eg; sb < ST_SUB; sb += 2) {
        const uint32_t use = acc_cnt + sb;
        const int slot = use % ST_SLOTS;
        mbar_wait(&bar_acc_full[slot], (use / ST_SLOTS) & 1);
        tc_fence_after();
        uint32_t a0[16], a1[16];
        const uint32_t taddr = tmem_base + slot * ST_C + ((uint32_t)(ew * 32) << 16);
        tmem_ld16(taddr, a0);
        tmem_ld16(taddr + 16, a1);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&bar_acc_empty[slot]);
        const uint32_t qq = (uint32_t)(t * MT) + sb * 128 + ew * 32 + lane;      // np4 < 2^31 (checked by the launcher)
        const uint32_t n = qq / (uint32_t)frame;
        const uint32_t rem = qq - n * (uint32_t)frame;
        const int i = (int)(rem / (uint32_t)g.Wq), j = (int)(rem - (uint32_t)i * (uint32_t)g.Wq);
        if ((long long)qq < g.np4 && i < g.Ho && j < g.Wo) {
          if (MODE == 0) {
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              const float y0 = __uint_as_float(a0[c]), y1 = __uint_as_float(a1[c]);
              s[c] += y0; q[c] = fmaf(y0, y0, q[c]);
              s[16 + c] += y1; q[16 + c] = fmaf(y1, y1, q[16 + c]);
            }
          } else {
            uint32_t pk[16];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float y0 = fmaxf(fmaf(__uint_as_float(a0[2 * c]), s[2 * c], q[2 * c]), 0.f);
              const float y1 = fmaxf(fmaf(__uint_as_float(a0[2 * c + 1]), s[2 * c + 1], q[2 * c + 1]), 0.f);
              const float z0 = fmaxf(fmaf(__uint_as_float(a1[2 * c]), s[16 + 2 * c], q[16 + 2 * c]), 0.f);
              const float z1 = fmaxf(fmaf(__uint_as_float(a1[2 * c + 1]), s[16 + 2 * c + 1], q[16 + 2 * c + 1]), 0.f);
              __nv_bfloat162 h0 = __floats2bfloat162_rn(y0, y1), h1 = __floats2bfloat162_rn(z0, z1);
              pk[c] = *reinterpret_cast<uint32_t*>(&h0);
              pk[8 + c] = *reinterpret_cast<uint32_t*>(&h1);
            }
            uint4* o = reinterpret_cast<uint4*>(out + (((long long)n * g.Ho + i) * g.Wo + j) * ST_C);
            o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            o[2] = make_uint4(pk[8], pk[9], pk[10], pk[11]);
            o[3] = make_uint4(pk[12], pk[13], pk[14], pk[15]);
          }
        }
      }
      acc_cnt += ST_SUB;
    }
    if (MODE == 0) {
      // CTA reduction over the 128 row-threads; the stream segments are free (every MMA retired before its acc_full fired)
      float* red = reinterpret_cast<float*>(smem_gen + ST_W_BYTES);          // [256][65]
      const int r = tid - 128;
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
#pragma unroll
      for (int c = 0; c < ST_C; ++c) { red[r * 65 + c] = s[c]; red[r * 65 + 32 + c] = q[c]; }
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
      if (r < 64) {
        double acc = 0.0;
        for (int k = 0; k < 256; ++k) acc += (double)red[k * 65 + r];
        atomicAdd(ws + r, acc);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------------------------------------------------------------------------
// Pass 2 fused with MaxPool2d(3,2,1) (cad:118,148): the 708 MB bf16 NHWC tensor between the stem and the pool is never written.
//
// A work item is a BAND of one frame: SP_P pooled rows = the 2*SP_P + 1 convolution rows 2*SP_P*b - 1 .. 2*SP_P*b + 2*SP_P - 1 (one row
// of overlap with the next band: 17 % more MMAs than pass 2 alone).  The band's positions are contiguous in the flat X4 index, so the
// stream machinery is unchanged -- one TMA box per band (it starts at the enclosing 128-byte row; the pixel remainder goes into the
// MMA descriptors' start address), SP_SUB sub-tiles of 128 positions, the same 8 MMAs each.  The epilogue applies BN + ReLU and parks
// the band as bf16 [row][column][32] in shared memory instead of HBM; when the band is complete, the eight epilogue warps pool it
// (values are post-ReLU, so an absent neighbour is a 0) and write the padded-flat rows of the next layer's input, borders included.
constexpr int SP_P = 3;                       // pooled rows per band
constexpr int SP_ROWS = 2 * SP_P + 1;         // convolution rows per band

struct PoolGeo {
  int PH, PW;                 // pooled frame
  int bands_per_frame;
  long long n_items;          // N * bands_per_frame
  int sub;                    // 128-position sub-tiles per band
  int seg_rows;               // 128-byte rows per stream segment
  int tile_pitch;             // bf16 elements per parked row (Wo * 32)
};

__global__ void __launch_bounds__(384, 1) stem_pool_kernel(const __grid_constant__ CUtensorMap map_x4, const float* __restrict__ w,
                                                           const float* __restrict__ bias, StemGeo g, PoolGeo pg, const float* __restrict__ mean,
                                                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, __nv_bfloat16* __restrict__ out) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_seg_full[2], bar_seg_empty[2], bar_acc_full[ST_SLOTS], bar_acc_empty[ST_SLOTS];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float s_sc[ST_C], s_sh[ST_C];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)pg.seg_rows * 128;
  const uint32_t s_w = smem_base;                           // 8 KiB of packed weights
  const uint32_t s_seg = smem_base + ST_W_BYTES;            // 2 stream segments
  __nv_bfloat16* band = reinterpret_cast<__nv_bfloat16*>(smem_gen + ST_W_BYTES + 2 * seg_bytes);       // [SP_ROWS][Wo][32]
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int sub = pg.sub;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_seg_full[i], 1); mbar_init(&bar_seg_empty[i], 1); }
    for (int i = 0; i < ST_SLOTS; ++i) { mbar_init(&bar_acc_full[i], 1); mbar_init(&bar_acc_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(&map_x4);
  }
  if (tid < ST_C) {
    const float sc = invstd[tid] * gamma[tid];
    s_sc[tid] = sc;
    s_sh[tid] = (bias[tid] - mean[tid]) * sc + beta[tid];
  }
  for (int i = tid; i < 8 * 2 * ST_C * 4; i += blockDim.x) {       // weights, as in stem_tf32_kernel
    const int e = i & 3, n = (i >> 2) & 31, c = (i >> 7) & 1, m = i >> 8;
    const int u = m >> 1, v = 2 * (m & 1) + c, a = e >> 1, b = e & 1;
    const int kh = 2 * u + a - 1, kw = 2 * v + b - 1;
    const float val = ((unsigned)kh < (unsigned)ST_K && (unsigned)kw < (unsigned)ST_K) ? w[n * ST_K * ST_K + kh * ST_K + kw] : 0.f;
    reinterpret_cast<float*>(smem_gen)[i] = val;
  }
  if (warp == 2) tmem_alloc<512>(&tmem_base_sh);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  // first flat X4 pixel of work item t (may be negative for the first band of the first frame: TMA zero-fills)
  auto item_start = [&](long long t) -> long long {
    const long long n = t / pg.bands_per_frame;
    const int b = (int)(t - n * pg.bands_per_frame);
    return (n * g.Hq + (2 * SP_P * b - 1)) * (long long)g.Wq;
  };

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer: one box per band
    uint32_t cnt = 0;
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x, ++cnt) {
      const int st = cnt & 1;
      mbar_wait(&bar_seg_empty[st], ((cnt >> 1) & 1) ^ 1);
      if (elect_one()) {
        const long long p0 = item_start(t);
        const long long row = p0 >= 0 ? p0 / 8 : -((-p0 + 7) / 8);          // floor(p0 / 8)
        mbar_expect_tx(&bar_seg_full[st], seg_bytes);
        tma_load_2d(s_seg + st * seg_bytes, &map_x4, 0, (int)row, &bar_seg_full[st]);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    uint32_t idesc = 0;
    idesc |= 1u << 4;                 // D = f32
    idesc |= 2u << 7;                 // A = tf32
    idesc |= 2u << 10;                // B = tf32
    idesc |= (uint32_t)(ST_C >> 3) << 17;
    idesc |= (uint32_t)(128 >> 4) << 24;
    const uint64_t da_hi = make_smem_desc(0, 16, 128, UMMA_NOSW);
    const uint64_t db_hi = make_smem_desc(0, 512, 128, UMMA_NOSW);
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
        const int slot = use % ST_SLOTS;
        mbar_wait(&bar_acc_empty[slot], ((use / ST_SLOTS) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const uint32_t a_addr = seg + (uint32_t)(off + s * 128 + (m >> 1) * g.Wq + 2 * (m & 1)) * 16;
            const uint64_t da = da_hi | (uint64_t)((a_addr >> 4) & 0x3FFF);
            const uint64_t db = db_hi | (uint64_t)(((s_w + m * 1024) >> 4) & 0x3FFF);
            tc_mma_tf32(tmem_base + slot * ST_C, da, db, idesc, m != 0);
          }
          tc_commit(&bar_acc_full[slot]);
        }
        __syncwarp();
      }
      if (elect_one()) tc_commit(&bar_seg_empty[st]);
      __syncwarp();
      acc_cnt += sub;
    }
  } else if (warp >= 4) {
    // ---------------------------------------------------------------- epilogue: park the band (BN + ReLU, bf16) in shared memory, then pool it
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    const int et = tid - 128;                                       // 0..255 among the epilogue threads
    uint32_t acc_cnt = 0;
    const int groups = ST_C / 8;                                    // 16-byte vectors per pixel
    // BatchNorm scale / shift in registers (see stem_tf32_kernel): the epilogue's shared-memory traffic competes with the MMAs' operand
    // stream, so it is kept to the parked band itself.  Band layout: column j lives in the 64-byte slot j ^ ((j >> 1) & 1) of its row (the
    // second pair of every four columns is swapped) and its four 16-byte vectors are XOR-swizzled by (j >> 1) & 3.  The parking stores
    // (lane = column) and the pooling reads are then both bank-conflict free: the pooling reads walk columns two apart, which without
    // the slot swap all fall into the same 16 banks (a 64-byte pixel covers half of them) -- ncu showed 2.76 M wavefronts where 1.40 M
    // suffice on every one of the nine pooling loads (profiles/r02c_stem_pool_ncu_full.md)
    float rs[ST_C], rq[ST_C];
#pragma unroll
    for (int c = 0; c < ST_C; ++c) { rs[c] = s_sc[c]; rq[c] = s_sh[c]; }
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x) {
      const long long n = t / pg.bands_per_frame;
      const int b = (int)(t - n * pg.bands_per_frame);
      const int i0 = 2 * SP_P * b - 1;                              // first convolution row of the band
      for (int sb = eg; sb < sub; sb += 2) {
        const uint32_t use = acc_cnt + sb;
        const int slot = use % ST_SLOTS;
        mbar_wait(&bar_acc_full[slot], (use / ST_SLOTS) & 1);
        tc_fence_after();
        uint32_t a0[16], a1[16];
        const uint32_t taddr = tmem_base + slot * ST_C + ((uint32_t)(ew * 32) << 16);
        tmem_ld16(taddr, a0);
        tmem_ld16(taddr + 16, a1);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(&bar_acc_empty[slot]);
        const int ql = sb * 128 + ew * 32 + lane;                   // position inside the band
        const int r = ql / g.Wq, j = ql - r * g.Wq;
        if (r < SP_ROWS && j < g.Wo) {
          const int i = i0 + r;
          uint32_t pk[16];
          if (i >= 0 && i < g.Ho) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float y0 = fmaxf(fmaf(__uint_as_float(a0[2 * c]), rs[2 * c], rq[2 * c]), 0.f);
              const float y1 = fmaxf(fmaf(__uint_as_float(a0[2 * c + 1]), rs[2 * c + 1], rq[2 * c + 1]), 0.f);
              const float z0 = fmaxf(fmaf(__uint_as_float(a1[2 * c]), rs[16 + 2 * c], rq[16 + 2 * c]), 0.f);
              const float z1 = fmaxf(fmaf(__uint_as_float(a1[2 * c + 1]), rs[16 + 2 * c + 1], rq[16 + 2 * c + 1]), 0.f);
              __nv_bfloat162 h0 = __floats2bfloat162_rn(y0, y1), h1 = __floats2bfloat162_rn(z0, z1);
              pk[c] = *reinterpret_cast<uint32_t*>(&h0);
              pk[8 + c] = *reinterpret_cast<uint32_t*>(&h1);
            }
          } else {
#pragma unroll
            for (int c = 0; c < 16; ++c) pk[c] = 0u;               // rows outside the frame: post-ReLU zeros never win a max
          }
          uint4* o = reinterpret_cast<uint4*>(band + (size_t)r * pg.tile_pitch + (size_t)(j ^ ((j >> 1) & 1)) * ST_C);
          const int sw = (j >> 1) & 3;
          o[0 ^ sw] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          o[1 ^ sw] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          o[2 ^ sw] = make_uint4(pk[8], pk[9], pk[10], pk[11]);
          o[3 ^ sw] = make_uint4(pk[12], pk[13], pk[14], pk[15]);
        }
      }
      acc_cnt += sub;
      asm volatile("bar.sync 1, 256;\n" ::: "memory");              // the band is complete
      // ---- pool: pooled rows SP_P*b .. SP_P*b + SP_P - 1 (band rows 2k, 2k+1, 2k+2 for the k-th of them), padded-flat output
      const int rowlen = (pg.PW + 2) * groups;                       // vectors per padded output row
      for (int v = et; v < SP_P * rowlen; v += 256) {
        const int k = v / rowlen, vv = v - k * rowlen;
        const int ph = SP_P * b + k;
        if (ph >= pg.PH) continue;
        const int pwp = vv / groups, cg = vv - pwp * groups;
        uint4 o = make_uint4(0, 0, 0, 0);
        if (pwp >= 1 && pwp <= pg.PW) {
          const int pw = pwp - 1;
          // all nine loads are issued before the first max (a branch per tap made the compiler chain them: load, use, load ...).  A window
          // column outside the frame is clamped onto its in-frame neighbour, which the window holds anyway: the max is unchanged
          uint4 tv[9];
#pragma unroll
          for (int bb = 0; bb < 3; ++bb) {
            int ww = 2 * pw - 1 + bb;
            ww = ww < 0 ? 0 : (ww >= g.Wo ? g.Wo - 1 : ww);
            const int off = (ww ^ ((ww >> 1) & 1)) * ST_C + ((cg ^ ((ww >> 1) & 3)) * 8);
#pragma unroll
            for (int a = 0; a < 3; ++a)
              tv[a * 3 + bb] = *reinterpret_cast<const uint4*>(band + (size_t)(2 * k + a) * pg.tile_pitch + off);
          }
          __nv_bfloat162 best[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) best[i] = reinterpret_cast<const __nv_bfloat162*>(&tv[0])[i];
#pragma unroll
          for (int t9 = 1; t9 < 9; ++t9)
#pragma unroll
            for (int i = 0; i < 4; ++i) best[i] = __hmax2(best[i], reinterpret_cast<const __nv_bfloat162*>(&tv[t9])[i]);
          o = *reinterpret_cast<uint4*>(best);
        }
        reinterpret_cast<uint4*>(out)[((n * (pg.PH + 2) + ph + 1) * (long long)rowlen) + vv] = o;
      }
      // the frame's top / bottom border rows belong to its first / last band
      if (b == 0)
        for (int v = et; v < rowlen; v += 256) reinterpret_cast<uint4*>(out)[(n * (pg.PH + 2)) * (long long)rowlen + v] = make_uint4(0, 0, 0, 0);
      if (b == pg.bands_per_frame - 1)
        for (int v = et; v < rowlen; v += 256)
          reinterpret_cast<uint4*>(out)[(n * (pg.PH + 2) + pg.PH + 1) * (long long)rowlen + v] = make_uint4(0, 0, 0, 0);
      asm volatile("bar.sync 1, 256;\n" ::: "memory");              // the band buffer may be overwritten
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// MaxPool2d(3,2,1) over relu'd bf16 NHWC (N,H,W,C) -> padded-flat (N,PH+2,PW+2,C) with zero border; 8 channels per thread
__global__ void maxpool3x3s2_pad_kernel(const __nv_bfloat16* __restrict__ y, int N, int H, int W, int C, int PH, int PW,
                                        __nv_bfloat16* __restrict__ out) {
  const int groups = C >> 3;
  const int rowlen = (PW + 2) * groups;
  const int rows = N * (PH + 2);
  for (int rr = blockIdx.x; rr < rows; rr += gridDim.x) {
    const int php = rr % (PH + 2), n = rr / (PH + 2);
    uint4* dst = reinterpret_cast<uint4*>(out) + (long long)rr * rowlen;
    const bool row_ok = php >= 1 && php <= PH;
    for (int v = threadIdx.x; v < rowlen; v += blockDim.x) {
      const int pwp = v / groups, cg = v - pwp * groups;
      uint4 o = make_uint4(0, 0, 0, 0);
      if (row_ok && pwp >= 1 && pwp <= PW) {
        const int ph = php - 1, pw = pwp - 1;
        __nv_bfloat162 best[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) best[i] = __floats2bfloat162_rn(0.f, 0.f);     // inputs are post-ReLU (>= 0)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const int h = 2 * ph - 1 + a;
          if ((unsigned)h >= (unsigned)H) continue;
#pragma unroll
          for (int b = 0; b < 3; ++b) {
            const int ww = 2 * pw - 1 + b;
            if ((unsigned)ww >= (unsigned)W) continue;
            const uint4 t = __ldg(reinterpret_cast<const uint4*>(y) + (((long long)n * H + h) * W + ww) * groups + cg);
            const __nv_bfloat162* tp = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
            for (int i = 0; i < 4; ++i) best[i] = __hmax2(best[i], tp[i]);
          }
        }
        o = *reinterpret_cast<uint4*>(best);
      }
      dst[v] = o;
    }
  }
}

int stem_geo(StemGeo& g, int N, int H, int W) {
  g.N = N; g.H = H; g.W = W;
  g.Ho = (H - 1) / 2 + 1;
  g.Wo = (W - 1) / 2 + 1;
  g.Hq = g.Ho + 3;
  g.Wq = g.Wo + 3;
  g.np4 = (long long)N * g.Hq * g.Wq;
  const int MT = 128 * ST_SUB;
  g.n_tiles = (g.np4 + MT - 1) / MT;
  const int seg_px = MT + 3 * g.Wq + 3;
  g.seg_rows = (seg_px + 7) / 8;
  if (g.seg_rows > 256 || g.np4 + 128 * ST_SUB > 0x7fffffffLL) return 1;      // one TMA box per tile (frames up to ~1000 px wide)
  return 0;
}

int stem_launch(int mode, const float* x4, const float* w, const float* bias, const StemGeo& g, const float* mean, const float* invstd,
                const float* gamma, const float* beta, double* ws, void* out, cudaStream_t st) {
  // X4 as a matrix of 128-byte rows (8 pixels); the last partial row is covered by the buffer's 128-byte slack
  CUtensorMap mx;
  {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return (int)cudaErrorNotSupported;
    memset(&mx, 0, sizeof(mx));
    cuuint64_t dims[2] = {32, (cuuint64_t)((g.np4 + 7) / 8)};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {32, (cuuint32_t)g.seg_rows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&mx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x4), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return (int)cudaErrorInvalidValue;
  }
  const size_t smem = ST_W_BYTES + 2 * (size_t)g.seg_rows * 128 + 1024 + (mode == 0 ? 0 : 0);
  const size_t need = smem < (size_t)(ST_W_BYTES + 256 * 65 * 4 + 1024) ? (size_t)(ST_W_BYTES + 256 * 65 * 4 + 1024) : smem;
  static size_t configured0[CVAD_MAX_DEVICES] = {}, configured1[CVAD_MAX_DEVICES] = {};
  cudaError_t ce = cvad_ensure_dyn_smem(stem_tf32_kernel<0>, need, configured0);
  if (ce == cudaSuccess) ce = cvad_ensure_dyn_smem(stem_tf32_kernel<1>, need, configured1);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > g.n_tiles) grid = g.n_tiles;
  if (mode == 0)
    stem_tf32_kernel<0><<<(unsigned)grid, 384, need, st>>>(mx, w, bias, g, mean, invstd, gamma, beta, ws, (__nv_bfloat16*)out);
  else
    stem_tf32_kernel<1><<<(unsigned)grid, 384, need, st>>>(mx, w, bias, g, mean, invstd, gamma, beta, ws, (__nv_bfloat16*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

// pass 2 + max-pool in one kernel; returns cudaErrorNotSupported when a band does not fit (very wide frames): callers fall back
int stem_pool_launch(const float* x4, const float* w, const float* bias, const StemGeo& g, const float* mean, const float* invstd,
                     const float* gamma, const float* beta, void* out, cudaStream_t st) {
  PoolGeo pg;
  pg.PH = (g.Ho - 1) / 2 + 1;
  pg.PW = (g.Wo - 1) / 2 + 1;
  pg.bands_per_frame = (pg.PH + SP_P - 1) / SP_P;
  pg.n_items = (long long)g.N * pg.bands_per_frame;
  pg.sub = (SP_ROWS * g.Wq + 127) / 128;
  const int seg_px = 128 * pg.sub + 3 * g.Wq + 3 + 8;              // + the pixel remainder of the box's 128-byte alignment
  pg.seg_rows = (seg_px + 7) / 8;
  pg.tile_pitch = ((g.Wo + 3) & ~3) * ST_C;                       // whole groups of four columns: the slot swap stays inside the row
  const size_t band_bytes = (size_t)SP_ROWS * pg.tile_pitch * sizeof(__nv_bfloat16);
  const size_t smem = ST_W_BYTES + 2 * (size_t)pg.seg_rows * 128 + band_bytes + 1024;
  if (pg.seg_rows > 256 || pg.sub > ST_SLOTS || smem > 220 * 1024) return (int)cudaErrorNotSupported;
  CUtensorMap mx;
  {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return (int)cudaErrorNotSupported;
    memset(&mx, 0, sizeof(mx));
    cuuint64_t dims[2] = {32, (cuuint64_t)((g.np4 + 7) / 8)};
    cuuint64_t strides[1] = {128};
    cuuint32_t box[2] = {32, (cuuint32_t)pg.seg_rows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&mx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(x4), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return (int)cudaErrorInvalidValue;
  }
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem_pool_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > pg.n_items) grid = pg.n_items;
  stem_pool_kernel<<<(unsigned)grid, 384, smem, st>>>(mx, w, bias, g, pg, mean, invstd, gamma, beta, (__nv_bfloat16*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

}  // namespace

CVAD_API long long cvad_stem_x4_floats(int N, int H, int W) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return -1;
  return ((g.np4 + 7) / 8) * 32 + 32;
}

CVAD_API int cvad_stem_space_to_depth_f32(const float* x, int N, int H, int W, float* x4, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  long long blocks = (g.np4 + 255) / 256;
  if (blocks > 16LL * cvad_num_sms()) blocks = 16LL * cvad_num_sms();
  stem_s2d_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, g, reinterpret_cast<float4*>(x4));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_stem_space_to_depth_u8(const void* x, int N, int H, int W, float mean, float stdv, float* x4, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W) || stdv == 0.f) return (int)cudaErrorInvalidValue;
  long long blocks = ((long long)g.N * g.Hq * ((g.Wq + 3) / 4) + 255) / 256;
  if (blocks > 16LL * cvad_num_sms()) blocks = 16LL * cvad_num_sms();
  stem_s2d_u8_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)x, g, mean, stdv, reinterpret_cast<float4*>(x4));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_u8_normalize_f32(const void* x, long long n, float mean, float stdv, float* y, void* stream) {
  if (n <= 0) return 0;
  if (stdv == 0.f || ((uintptr_t)x & 15) || ((uintptr_t)y & 15)) return (int)cudaErrorInvalidValue;
  long long blocks = (n / 16 + 255) / 256 + 1;
  if (blocks > 16LL * cvad_num_sms()) blocks = 16LL * cvad_num_sms();
  u8_normalize_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)x, n, mean, stdv, y);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_stem_tf32_stats(const float* x4, const float* w, const float* bias, int N, int H, int W, double* ws, float eps, float momentum,
                                  float* mean, float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked,
                                  void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  int e = stem_launch(0, x4, w, bias, g, nullptr, nullptr, nullptr, nullptr, ws, nullptr, st);
  if (e) return e;
  // ws holds the sums of the RAW accumulator; y = acc + bias: the bias moves the mean, not the variance
  return bn_finalize_launch(ws, ST_C, (double)N * g.Ho * g.Wo, bias, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked,
                            st);
}

CVAD_API int cvad_stem_tf32_bn_relu(const float* x4, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                    const float* invstd, const float* gamma, const float* beta, void* y, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  return stem_launch(1, x4, w, bias, g, mean, invstd, gamma, beta, nullptr, y, (cudaStream_t)stream);
}

CVAD_API int cvad_stem_tf32_bn_relu_maxpool(const float* x4, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                            const float* invstd, const float* gamma, const float* beta, void* out, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  return stem_pool_launch(x4, w, bias, g, mean, invstd, gamma, beta, out, (cudaStream_t)stream);
}

CVAD_API int cvad_pad_maxpool3x3s2_bf16(const void* y, int N, int H, int W, int C, void* out, void* stream) {
  if (C % 8) return (int)cudaErrorInvalidValue;
  const int PH = (H - 1) / 2 + 1, PW = (W - 1) / 2 + 1;
  const int rows = N * (PH + 2);
  const int blocks = rows < 16 * cvad_num_sms() ? rows : 16 * cvad_num_sms();
  maxpool3x3s2_pad_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)y, N, H, W, C, PH, PW, (__nv_bfloat16*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

// Stem of the M-A backbone on the tensor cores: conv 7x7 stride 2 pad 3, 1 -> 32 channels (cad:115, 145) as a tcgen05 implicit GEMM,
// fused with the BatchNorm batch statistics (pass 1) or with BN + ReLU (pass 2), and in pass 2 optionally with MaxPool2d(3,2,1)
// (cad:116-118, 146-148).  Two formulations share one pipeline: kind::tf32 over a 2x2 space-to-depth (the general path) and kind::f16
// over a 2x4 space-to-depth (frames whose width is a multiple of 4).
//
// tf32 over 2x2.  With one input channel an im2col row has no contiguous 16-byte piece, so neither TMA nor a UMMA descriptor can address
// it.  A 2x2 space-to-depth turns the problem into one they can: X4[n][i][j][a*2+b] = x[n][2(i-2)+a][2(j-2)+b] (zero outside the
// frame) is an NHWC tensor with 4 fp32 channels = one 16-byte "pixel", and the 7x7 stride-2 convolution becomes a 4x4
// stride-1 convolution over it (kh = 2u+a-1, kw = 2v+b-1; the 15 combinations outside the 7x7 window get zero weights).
// Over the flat pixel index q of X4 (geometry (Ho+3) x (Wo+3) per frame) the output is
//        out[q][:] = sum_{u,v} X4[q + u*(Wo+3) + v][0:4] * W4[u][v]            (positions with i >= Ho or j >= Wo are junk)
// and the A operand of one MMA (K = 8 tf32 = two horizontally adjacent pixels) is a VIEW OF THE RAW PIXEL STREAM: rows are
// consecutive pixels (16-byte pitch = the no-swizzle core-matrix row pitch), the second K chunk is the same stream one pixel
// later (LBO = 16 B, overlapping), 8-row groups follow at SBO = 128 B.  So TMA copies the stream into shared memory as is
// (one box of up to 32 KiB per tile) and tcgen05.mma performs the im2col through its descriptor -- no thread touches an
// input element (profiles/r01_umma_descriptor_probe.md, config 15).  fp32 inputs are rounded to tf32 (10-bit mantissa) by the MMA.
//
// fp16 over 2x4.  Why: the tf32 form issues, per 128 output pixels, 8 MMAs of M128 x N32 x K8 whose operands (5 KB each) stream from
// shared memory: 66 cycles apiece against 16 of math, and in pass 2 that stream plus the max-pool's parked band saturate the shared-memory
// pipe (profiles/r02c_stem_pool_ncu_full.md).  Here X8[n][i][J][a*4+b] = x[n][2(i-2)+a][4(J-1)+b] (zero outside the frame) is an NHWC
// tensor of fp16 with 8 channels = one 16-byte "pixel" that covers a 2 x 4 patch of the frame, i.e. TWO horizontally adjacent outputs of
// the stride-2 convolution.  An accumulator row is such a pixel and carries N = 64 columns = (output parity p, channel), and over the flat
// pixel index q of X8 (geometry (Ho+3) x (Wo/2+2) per frame)
//        out[q][p*32 + c] = sum_{u<4, v<3} X8[q + u*Wq + v][0:8] * W8[u][v][p][c]      (kh = 2u+a-1, kw = 4v+b-2p-1)
// is 6 MMAs of M128 x N64 x K16 per 128 pixels = 256 outputs (the two 16-byte K chunks of an MMA are the pixel rows u and u+1: LBO = one
// row of X8): 2.3x fewer tensor-core cycles and 2.2x fewer operand bytes than the tf32 form.  Inputs are exact in fp16 whenever they are
// exact in tf32 (both keep 11 significant bits; the loader's 0..255 grayscale values through Normalize(0.5, 0.5) are odd integers below
// 512); weights are rounded to nearest fp16 where the tf32 MMA truncates.
//
// Kernels: persistent, warp-specialised like flatconv_tc.cu -- warp 0 TMA producer (double-buffered stream segments), warp 1 MMA issuer
// (one formulation's MMAs per 128 positions into a TMEM accumulator ring), warp 2 TMEM owner, warps 4-11 (4-15 in the fp16 pool kernel)
// epilogue in groups of four warps on alternate sub-tiles.  Pass 1 accumulates per-channel sum / sum of squares of the valid rows in
// registers across the whole CTA (no convolution output is ever written); pass 2 applies BN + ReLU and either stores bf16 NHWC rows or
// parks a band of rows in shared memory and max-pools it.  The frozen stem needs no gradient (cad:596-598).
#include <cuda_fp16.h>

#include "common.cuh"
#include "cvad_b200.h"
#include "tc_common.cuh"

namespace {

using namespace cvad_tc;

constexpr int STEM_C = 32;            // output channels
constexpr int STEM_K = 7;             // kernel size

struct StemGeo {
  int N, H, W, Ho, Wo, Hq, Wq;
  int Wh;                 // fp16 formulation: output pairs per row (Wq = Wh + 2)
  long long np;           // N*Hq*Wq pixels of the space-to-depth stream (= GEMM rows incl. junk)
  long long n_tiles;      // pass-1 tiles
  int seg_rows;           // 128-byte rows (8 pixels) per stream segment of pass 1
};

// pass 1: s / q += one output's 32 channels (columns 0-15 in a0, 16-31 in a1) and their squares
__device__ __forceinline__ void add_sums(float (&s)[STEM_C], float (&q)[STEM_C], const uint32_t (&a0)[16], const uint32_t (&a1)[16]) {
#pragma unroll
  for (int c = 0; c < 16; ++c) {
    const float y0 = __uint_as_float(a0[c]), y1 = __uint_as_float(a1[c]);
    s[c] += y0; q[c] = fmaf(y0, y0, q[c]);
    s[16 + c] += y1; q[16 + c] = fmaf(y1, y1, q[16 + c]);
  }
}

// ------------------------------------------------------------------------------------------------------------------------------------
// The two formulations: what differs between them.  Everything else -- the segment ring, the accumulator ring, the band decomposition,
// the statistics reduction -- is the shared pipeline below.

// kind::tf32 over the 2x2 space-to-depth X4: an accumulator row is one output, 8 MMAs of M128 x N32 x K8 per 128 positions
struct StemTf32 {
  static constexpr int N = 32;                   // accumulator columns
  static constexpr int SLOTS = 16;               // TMEM accumulator ring (16 x 32 columns)
  static constexpr int TILE_SUB = 8;             // 128-position sub-tiles per pass-1 tile
  static constexpr int W_BYTES = 8 * 1024;       // 8 MMAs x [2 chunks][32 rows][16 B]
  static constexpr uint32_t B_LBO = 512;
  static constexpr uint32_t IDESC = (1u << 4)    // D = f32
                                    | (2u << 7)  // A = tf32
                                    | (2u << 10) // B = tf32
                                    | (uint32_t)(N >> 3) << 17 | (uint32_t)(128 >> 4) << 24;
  __device__ static uint32_t a_lbo(int) { return 16; }     // pixel stream: K chunks overlap by one pixel

  // weights -> [mma = u*2+vp][K chunk c][n][4 floats]; chunk c of MMA (u,vp) is tap column v = 2vp+c, element e = a*2+b
  __device__ __forceinline__ static void stage_weights(const float* __restrict__ w, uint8_t* smem_w, const float* chan_scale) {
    for (int i = threadIdx.x; i < 8 * 2 * N * 4; i += blockDim.x) {
      const int e = i & 3, n = (i >> 2) & 31, c = (i >> 7) & 1, m = i >> 8;
      const int u = m >> 1, v = 2 * (m & 1) + c, a = e >> 1, b = e & 1;
      const int kh = 2 * u + a - 1, kw = 2 * v + b - 1;
      float val = ((unsigned)kh < (unsigned)STEM_K && (unsigned)kw < (unsigned)STEM_K) ? w[n * STEM_K * STEM_K + kh * STEM_K + kw] : 0.f;
      if (chan_scale) val *= chan_scale[n];
      reinterpret_cast<float*>(smem_w)[i] = val;
    }
  }
  // the eight MMAs of one 128-position sub-tile whose first pixel sits at shared-memory address a0 (16-byte pixels)
  __device__ __forceinline__ static void issue_subtile(uint32_t tmem_acc, uint32_t a0, uint32_t s_w, int Wq, uint64_t da_hi, uint64_t db_hi) {
#pragma unroll
    for (int m = 0; m < 8; ++m) {
      const uint32_t a_addr = a0 + (uint32_t)((m >> 1) * Wq + 2 * (m & 1)) * 16;
      const uint64_t da = da_hi | (uint64_t)((a_addr >> 4) & 0x3FFF);
      const uint64_t db = db_hi | (uint64_t)(((s_w + m * 1024) >> 4) & 0x3FFF);
      tc_mma_tf32(tmem_acc, da, db, IDESC, m != 0);
    }
  }
  // pass 1: accumulator row j of an in-frame stream row holds one output, valid if j < Wo
  __device__ __forceinline__ static void add_row(const uint32_t (&a)[N / 16][16], int j, const StemGeo& g, float (&s)[STEM_C], float (&q)[STEM_C]) {
    if (j < g.Wo) add_sums(s, q, a[0], a[1]);
  }
};

// kind::f16 over the 2x4 space-to-depth X8: an accumulator row is two horizontally adjacent outputs, 6 MMAs of M128 x N64 x K16
struct StemF16 {
  static constexpr int N = 64;                   // accumulator columns: (parity, channel)
  static constexpr int SLOTS = 8;                // TMEM accumulator ring (8 x 64 columns)
  static constexpr int TILE_SUB = 4;             // 128-pixel sub-tiles per pass-1 tile
  static constexpr int MMAS = 6;                 // (u0 in {0,2}) x (v in {0,1,2})
  static constexpr int W_BYTES = MMAS * 2048;    // [mma][2 K chunks][64 rows][16 B]
  static constexpr uint32_t B_LBO = 1024;
  static constexpr uint32_t IDESC = (1u << 4)    // D = f32; A = B = f16 (format 0), both K-major
                                    | (uint32_t)(N >> 3) << 17 | (uint32_t)(128 >> 4) << 24;
  __device__ static uint32_t a_lbo(int Wq) { return (uint32_t)Wq * 16; }   // K chunk 1 = the pixel one X8 row below

  // conv1 weights (32,1,7,7) fp32 -> shared memory [mma = (u0/2)*3 + v][chunk c][n = p*32 + cout][e = a*4 + b] fp16
  __device__ __forceinline__ static void stage_weights(const float* __restrict__ w, uint8_t* smem_w, const float* chan_scale) {
    __half* dst = reinterpret_cast<__half*>(smem_w);
    for (int i = threadIdx.x; i < MMAS * 2 * N * 8; i += blockDim.x) {
      const int e = i & 7, n = (i >> 3) & 63, c = (i >> 9) & 1, m = i >> 10;
      const int u = 2 * (m / 3) + c, v = m % 3, a = e >> 2, b = e & 3, p = n >> 5, co = n & 31;
      const int kh = 2 * u + a - 1, kw = 4 * v + b - 2 * p - 1;
      float val = ((unsigned)kh < (unsigned)STEM_K && (unsigned)kw < (unsigned)STEM_K) ? w[co * STEM_K * STEM_K + kh * STEM_K + kw] : 0.f;
      if (chan_scale) val *= chan_scale[co];
      dst[i] = __float2half_rn(val);
    }
  }
  // the six MMAs of one 128-pixel sub-tile whose first pixel sits at shared-memory address a0 (16-byte pixels)
  __device__ __forceinline__ static void issue_subtile(uint32_t tmem_acc, uint32_t a0, uint32_t s_w, int Wq, uint64_t da_hi, uint64_t db_hi) {
#pragma unroll
    for (int m = 0; m < MMAS; ++m) {
      const uint32_t a_addr = a0 + (uint32_t)(2 * (m / 3) * Wq + (m % 3)) * 16;
      const uint64_t da = da_hi | (uint64_t)((a_addr >> 4) & 0x3FFF);
      const uint64_t db = db_hi | (uint64_t)(((s_w + m * 2048) >> 4) & 0x3FFF);
      tc_mma_f16(tmem_acc, da, db, IDESC, m != 0);
    }
  }
  // pass 1: accumulator row J holds the outputs 2J (valid if J < Wh) and 2J+1 (valid if also 2J+1 < Wo)
  __device__ __forceinline__ static void add_row(const uint32_t (&a)[N / 16][16], int J, const StemGeo& g, float (&s)[STEM_C], float (&q)[STEM_C]) {
    if (J < g.Wh) {
      add_sums(s, q, a[0], a[1]);
      if (2 * J + 1 < g.Wo) add_sums(s, q, a[2], a[3]);
    }
  }
};

// ------------------------------------------------------------------------------------------------------------------------------------
// The shared pipeline

template <class F>
struct StemBars {
  uint64_t seg_full[2], seg_empty[2], acc_full[F::SLOTS], acc_empty[F::SLOTS];
  uint32_t tmem_base;
};

// barrier init, weight staging (each output channel's weights times chan_scale[c] when given), TMEM allocation; returns the TMEM base
template <class F>
__device__ __forceinline__ uint32_t stem_setup(StemBars<F>& bars, const CUtensorMap* map, const float* __restrict__ w, uint8_t* smem_w,
                                               const float* chan_scale, int warp) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&bars.seg_full[i], 1); mbar_init(&bars.seg_empty[i], 1); }
    for (int i = 0; i < F::SLOTS; ++i) { mbar_init(&bars.acc_full[i], 1); mbar_init(&bars.acc_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(map);
  }
  F::stage_weights(w, smem_w, chan_scale);
  if (warp == 2) tmem_alloc<512>(&bars.tmem_base);
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return bars.tmem_base;
}

__device__ __forceinline__ void stem_teardown(int warp, uint32_t tmem_base) {
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// warp 0: one TMA box of seg_bytes per work item into the two-segment ring; box_row(t) = the item's first 128-byte stream row
template <class F, class BoxRow>
__device__ __forceinline__ void stem_produce(StemBars<F>& bars, const CUtensorMap* map, uint32_t s_seg, uint32_t seg_bytes, long long n_items,
                                             BoxRow box_row) {
  uint32_t cnt = 0;
  for (long long t = blockIdx.x; t < n_items; t += gridDim.x, ++cnt) {
    const int st = cnt & 1;
    mbar_wait(&bars.seg_empty[st], ((cnt >> 1) & 1) ^ 1);
    if (elect_one()) {
      mbar_expect_tx(&bars.seg_full[st], seg_bytes);
      tma_load_2d(s_seg + st * seg_bytes, map, 0, box_row(t), &bars.seg_full[st]);
    }
    __syncwarp();
  }
}

// warp 1: SUB sub-tiles per work item (SUB = 0: `sub`, known at run time only), each into the next slot of the accumulator ring;
// box_off(t) = the item's first pixel inside its box
template <class F, int SUB, class BoxOff>
__device__ __forceinline__ void stem_issue(StemBars<F>& bars, uint32_t tmem_base, uint32_t s_seg, uint32_t seg_bytes, uint32_t s_w, int Wq,
                                           long long n_items, int sub, BoxOff box_off) {
  const uint64_t da_hi = make_smem_desc(0, F::a_lbo(Wq), 128, UMMA_NOSW);
  const uint64_t db_hi = make_smem_desc(0, F::B_LBO, 128, UMMA_NOSW);
  const int nsub = SUB > 0 ? SUB : sub;
  uint32_t cnt = 0, acc_cnt = 0;
  for (long long t = blockIdx.x; t < n_items; t += gridDim.x, ++cnt) {
    const int st = cnt & 1;
    const int off = box_off(t);
    mbar_wait(&bars.seg_full[st], (cnt >> 1) & 1);
    tc_fence_after();
    const uint32_t seg = s_seg + st * seg_bytes;
    for (int s = 0; s < nsub; ++s) {
      const uint32_t use = acc_cnt + s;
      const int slot = use % F::SLOTS;
      mbar_wait(&bars.acc_empty[slot], ((use / F::SLOTS) & 1) ^ 1);
      tc_fence_after();
      if (elect_one()) {
        F::issue_subtile(tmem_base + slot * F::N, seg + (uint32_t)(off + s * 128) * 16, s_w, Wq, da_hi, db_hi);
        tc_commit(&bars.acc_full[slot]);
      }
      __syncwarp();
    }
    if (elect_one()) tc_commit(&bars.seg_empty[st]);
    __syncwarp();
    acc_cnt += nsub;
  }
}

// epilogue: wait for accumulator number `use`, load TMEM lanes 32*ew.. (all F::N columns, one wait) and hand the slot back to the issuer
template <class F>
__device__ __forceinline__ void stem_take_acc(StemBars<F>& bars, uint32_t tmem_base, uint32_t use, int ew, uint32_t (&acc)[F::N / 16][16]) {
  const int slot = use % F::SLOTS;
  mbar_wait(&bars.acc_full[slot], (use / F::SLOTS) & 1);
  tc_fence_after();
  const uint32_t taddr = tmem_base + slot * F::N + ((uint32_t)(ew * 32) << 16);
#pragma unroll
  for (int k = 0; k < F::N / 16; ++k) tmem_ld16(taddr + 16 * k, acc[k]);
  tmem_ld_wait();
  tc_fence_before();
  mbar_arrive(&bars.acc_empty[slot]);
}

// first flat stream pixel of band t of P pooled rows (= 2P + 1 convolution rows from row 2Pb - 1; negative for the first band of the first
// frame: TMA zero-fills), and the 128-byte stream row and pixel offset of its TMA box
__device__ __forceinline__ long long band_start(long long t, int P, int bands_per_frame, const StemGeo& g) {
  const long long n = t / bands_per_frame;
  const int b = (int)(t - n * bands_per_frame);
  return (n * g.Hq + (2 * P * b - 1)) * (long long)g.Wq;
}
__device__ __forceinline__ long long box_row_of(long long p0) { return p0 >= 0 ? p0 / 8 : -((-p0 + 7) / 8); }   // floor(p0 / 8)
__device__ __forceinline__ int box_off_of(long long p0) { return (int)(p0 - box_row_of(p0) * 8); }              // 0..7

struct BandGeo {
  int PH, PW;                 // pooled frame
  int bands_per_frame;
  long long n_items;          // N * bands_per_frame
  int sub;                    // 128-position sub-tiles per band
  int seg_rows;               // 128-byte rows per stream segment
  int tile_pitch;             // bf16 elements per parked row
};

// the frame's top / bottom padded border rows belong to its first / last band; ET epilogue threads, this one is et
__device__ __forceinline__ void band_border_rows(__nv_bfloat16* __restrict__ out, const BandGeo& pg, long long n, int b, int rowlen, int et, int ET) {
  if (b == 0)
    for (int v = et; v < rowlen; v += ET) reinterpret_cast<uint4*>(out)[(n * (pg.PH + 2)) * (long long)rowlen + v] = make_uint4(0, 0, 0, 0);
  if (b == pg.bands_per_frame - 1)
    for (int v = et; v < rowlen; v += ET)
      reinterpret_cast<uint4*>(out)[(n * (pg.PH + 2) + pg.PH + 1) * (long long)rowlen + v] = make_uint4(0, 0, 0, 0);
}

// ------------------------------------------------------------------------------------------------------------------------------------
// Space-to-depth of the frames

// x (N,1,H,W) fp32 -> X4 (N,Hq,Wq,4) fp32, one 16-byte pixel per thread
__global__ void stem_s2d_kernel(const float* __restrict__ x, StemGeo g, float4* __restrict__ x4) {
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < g.np; t += (long long)gridDim.x * blockDim.x) {
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

// x (N,1,H,W) fp32 or uint8 -> X8 (N,Hq,Wq,8) fp16: one 16-byte pixel per thread; W % 4 == 0, so a pixel's four columns are one aligned
// 16-byte (fp32) / 4-byte (uint8) load per frame row.  uint8: x = (float(v) - mean) / std as torchvision's Normalize computes it.
template <bool U8>
__global__ void stem8_s2d_kernel(const void* __restrict__ xin, StemGeo g, float mean, float stdv, uint4* __restrict__ x8) {
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

// ------------------------------------------------------------------------------------------------------------------------------------
// Pass 1: batch statistics of the raw accumulator (ws[c] += sum acc, ws[32+c] += sum acc^2 over the valid outputs; the bias is folded
// in by the finalize kernel).  An accumulator row holds one output (tf32: valid if j < Wo) or a pair (fp16: valid if J < Wh, the second
// output only if 2J+1 < Wo).
template <class F>
__global__ void __launch_bounds__(384, 1) stem_stats_kernel(const __grid_constant__ CUtensorMap map_xs, const float* __restrict__ w, StemGeo g,
                                                            double* __restrict__ ws) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ StemBars<F> bars;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)g.seg_rows * 128;
  const uint32_t s_w = smem_base, s_seg = smem_base + F::W_BYTES;        // packed weights, then 2 stream segments
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  constexpr int MT = 128 * F::TILE_SUB;
  const uint32_t tmem_base = stem_setup(bars, &map_xs, w, smem_gen, nullptr, warp);

  if (warp == 0) {
    stem_produce(bars, &map_xs, s_seg, seg_bytes, g.n_tiles, [](long long t) { return (int)(t * (MT / 8)); });
  } else if (warp == 1) {
    stem_issue<F, F::TILE_SUB>(bars, tmem_base, s_seg, seg_bytes, s_w, g.Wq, g.n_tiles, 0, [](long long) { return 0; });
  } else if (warp >= 4) {
    // thread <-> TMEM lane (row) 32*(warp-4)+lane; two groups of four warps (warps 4-7 and 8-11) take alternate sub-tiles
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    float s[STEM_C], q[STEM_C];                // per-channel sum / sum of squares over this thread's valid outputs
#pragma unroll
    for (int c = 0; c < STEM_C; ++c) { s[c] = 0.f; q[c] = 0.f; }
    const int frame = g.Hq * g.Wq;
    uint32_t acc_cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
      for (int sb = eg; sb < F::TILE_SUB; sb += 2) {
        uint32_t a[F::N / 16][16];
        stem_take_acc(bars, tmem_base, acc_cnt + sb, ew, a);
        const uint32_t qq = (uint32_t)(t * MT) + sb * 128 + ew * 32 + lane;      // np < 2^31 (checked by the launcher)
        const uint32_t n = qq / (uint32_t)frame;
        const uint32_t rem = qq - n * (uint32_t)frame;
        const int i = (int)(rem / (uint32_t)g.Wq), j = (int)(rem - (uint32_t)i * (uint32_t)g.Wq);
        if ((long long)qq < g.np && i < g.Ho) F::add_row(a, j, g, s, q);
      }
      acc_cnt += F::TILE_SUB;
    }
    // CTA reduction over the 256 row-threads; the stream segments are free (every MMA retired before its acc_full fired)
    float* red = reinterpret_cast<float*>(smem_gen + F::W_BYTES);          // [256][65]
    const int r = tid - 128;
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
#pragma unroll
    for (int c = 0; c < STEM_C; ++c) { red[r * 65 + c] = s[c]; red[r * 65 + 32 + c] = q[c]; }
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
    if (r < 64) {
      double acc = 0.0;
      for (int k = 0; k < 256; ++k) acc += (double)red[k * 65 + r];
      atomicAdd(ws + r, acc);
    }
  }
  stem_teardown(warp, tmem_base);
}

// out = relu(acc * s + q) per channel, bf16: pk[0..7] = channels 0-15 (from a0), pk[8..15] = channels 16-31 (from a1)
__device__ __forceinline__ void bn_relu_pack(const uint32_t (&a0)[16], const uint32_t (&a1)[16], const float (&s)[STEM_C], const float (&q)[STEM_C],
                                             uint32_t (&pk)[16]) {
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
}

// ------------------------------------------------------------------------------------------------------------------------------------
// tf32 pass 2: out = relu((acc + bias - mean) * invstd * gamma + beta) bf16 NHWC (N,Ho,Wo,32)
__global__ void __launch_bounds__(384, 1) stem_tf32_kernel(const __grid_constant__ CUtensorMap map_x4, const float* __restrict__ w,
                                                           const float* __restrict__ bias, StemGeo g, const float* __restrict__ mean,
                                                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, __nv_bfloat16* __restrict__ out) {
  using F = StemTf32;
  extern __shared__ uint8_t smem_raw[];
  __shared__ StemBars<F> bars;
  __shared__ float s_sc[STEM_C], s_sh[STEM_C];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)g.seg_rows * 128;
  const uint32_t s_w = smem_base, s_seg = smem_base + F::W_BYTES;
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  constexpr int MT = 128 * F::TILE_SUB;
  if (tid < STEM_C) {
    const float sc = invstd[tid] * gamma[tid];
    s_sc[tid] = sc;
    s_sh[tid] = (bias[tid] - mean[tid]) * sc + beta[tid];
  }
  const uint32_t tmem_base = stem_setup(bars, &map_x4, w, smem_gen, nullptr, warp);

  if (warp == 0) {
    stem_produce(bars, &map_x4, s_seg, seg_bytes, g.n_tiles, [](long long t) { return (int)(t * (MT / 8)); });
  } else if (warp == 1) {
    stem_issue<F, F::TILE_SUB>(bars, tmem_base, s_seg, seg_bytes, s_w, g.Wq, g.n_tiles, 0, [](long long) { return 0; });
  } else if (warp >= 4) {
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    // the BatchNorm scale / shift in REGISTERS: the MMAs stream their operands from shared memory at the pipe's limit, and 64 broadcast
    // loads per thread and sub-tile took a third of it away
    float s[STEM_C], q[STEM_C];
#pragma unroll
    for (int c = 0; c < STEM_C; ++c) { s[c] = s_sc[c]; q[c] = s_sh[c]; }
    const int frame = g.Hq * g.Wq;
    uint32_t acc_cnt = 0;
    for (long long t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
      for (int sb = eg; sb < F::TILE_SUB; sb += 2) {
        uint32_t a[2][16];
        stem_take_acc(bars, tmem_base, acc_cnt + sb, ew, a);
        const uint32_t qq = (uint32_t)(t * MT) + sb * 128 + ew * 32 + lane;      // np < 2^31 (checked by the launcher)
        const uint32_t n = qq / (uint32_t)frame;
        const uint32_t rem = qq - n * (uint32_t)frame;
        const int i = (int)(rem / (uint32_t)g.Wq), j = (int)(rem - (uint32_t)i * (uint32_t)g.Wq);
        if ((long long)qq < g.np && i < g.Ho && j < g.Wo) {
          uint32_t pk[16];
          bn_relu_pack(a[0], a[1], s, q, pk);
          uint4* o = reinterpret_cast<uint4*>(out + (((long long)n * g.Ho + i) * g.Wo + j) * STEM_C);
          o[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          o[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          o[2] = make_uint4(pk[8], pk[9], pk[10], pk[11]);
          o[3] = make_uint4(pk[12], pk[13], pk[14], pk[15]);
        }
      }
      acc_cnt += F::TILE_SUB;
    }
  }
  stem_teardown(warp, tmem_base);
}

// ------------------------------------------------------------------------------------------------------------------------------------
// Pass 2 fused with MaxPool2d(3,2,1) (cad:118,148): the 708 MB bf16 NHWC tensor between the stem and the pool is never written.
//
// A work item is a BAND of one frame: P pooled rows = the 2P + 1 convolution rows 2Pb - 1 .. 2Pb + 2P - 1 (one row of overlap with the
// next band: 17 % more MMAs than pass 2 alone at P = 3).  The band's positions are contiguous in the flat stream index, so the stream
// machinery is unchanged -- one TMA box per band (it starts at the enclosing 128-byte row; the pixel remainder goes into the MMA
// descriptors' start address), `sub` sub-tiles of 128 positions.  The epilogue applies BN + ReLU and parks the band as bf16 in shared
// memory instead of HBM; when the band is complete, the epilogue warps pool it (values are post-ReLU, so an absent neighbour is a 0) and
// write the padded-flat rows of the next layer's input, borders included.  The two formulations park differently (below).
constexpr int SP_P = 3;                       // tf32: pooled rows per band
constexpr int SP_ROWS = 2 * SP_P + 1;         // convolution rows per band
constexpr int S8_P = 4;                       // fp16: pooled rows per band
constexpr int S8_ROWS = 2 * S8_P + 1;

__global__ void __launch_bounds__(384, 1) stem_pool_kernel(const __grid_constant__ CUtensorMap map_x4, const float* __restrict__ w,
                                                           const float* __restrict__ bias, StemGeo g, BandGeo pg, const float* __restrict__ mean,
                                                           const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                           const float* __restrict__ beta, __nv_bfloat16* __restrict__ out) {
  using F = StemTf32;
  extern __shared__ uint8_t smem_raw[];
  __shared__ StemBars<F> bars;
  __shared__ float s_sc[STEM_C], s_sh[STEM_C];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)pg.seg_rows * 128;
  const uint32_t s_w = smem_base, s_seg = smem_base + F::W_BYTES;
  __nv_bfloat16* band = reinterpret_cast<__nv_bfloat16*>(smem_gen + F::W_BYTES + 2 * seg_bytes);       // [SP_ROWS][Wo][32]
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int sub = pg.sub;
  if (tid < STEM_C) {
    const float sc = invstd[tid] * gamma[tid];
    s_sc[tid] = sc;
    s_sh[tid] = (bias[tid] - mean[tid]) * sc + beta[tid];
  }
  const uint32_t tmem_base = stem_setup(bars, &map_x4, w, smem_gen, nullptr, warp);

  if (warp == 0) {
    stem_produce(bars, &map_x4, s_seg, seg_bytes, pg.n_items, [=](long long t) { return (int)box_row_of(band_start(t, SP_P, pg.bands_per_frame, g)); });
  } else if (warp == 1) {
    stem_issue<F, 0>(bars, tmem_base, s_seg, seg_bytes, s_w, g.Wq, pg.n_items, sub,
                     [=](long long t) { return box_off_of(band_start(t, SP_P, pg.bands_per_frame, g)); });
  } else if (warp >= 4) {
    // ---------------------------------------------------------------- epilogue: park the band (BN + ReLU, bf16) in shared memory, then pool it
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    const int et = tid - 128;                                       // 0..255 among the epilogue threads
    uint32_t acc_cnt = 0;
    const int groups = STEM_C / 8;                                  // 16-byte vectors per pixel
    // BatchNorm scale / shift in registers (see stem_tf32_kernel): the epilogue's shared-memory traffic competes with the MMAs' operand
    // stream, so it is kept to the parked band itself.  Band layout: column j lives in the 64-byte slot j ^ ((j >> 1) & 1) of its row (the
    // second pair of every four columns is swapped) and its four 16-byte vectors are XOR-swizzled by (j >> 1) & 3.  The parking stores
    // (lane = column) and the pooling reads are then both bank-conflict free: the pooling reads walk columns two apart, which without
    // the slot swap all fall into the same 16 banks (a 64-byte pixel covers half of them) -- ncu showed 2.76 M wavefronts where 1.40 M
    // suffice on every one of the nine pooling loads (profiles/r02c_stem_pool_ncu_full.md)
    float rs[STEM_C], rq[STEM_C];
#pragma unroll
    for (int c = 0; c < STEM_C; ++c) { rs[c] = s_sc[c]; rq[c] = s_sh[c]; }
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x) {
      const long long n = t / pg.bands_per_frame;
      const int b = (int)(t - n * pg.bands_per_frame);
      const int i0 = 2 * SP_P * b - 1;                              // first convolution row of the band
      for (int sb = eg; sb < sub; sb += 2) {
        uint32_t a[2][16];
        stem_take_acc(bars, tmem_base, acc_cnt + sb, ew, a);
        const int ql = sb * 128 + ew * 32 + lane;                   // position inside the band
        const int r = ql / g.Wq, j = ql - r * g.Wq;
        if (r < SP_ROWS && j < g.Wo) {
          const int i = i0 + r;
          uint32_t pk[16];
          if (i >= 0 && i < g.Ho) {
            bn_relu_pack(a[0], a[1], rs, rq, pk);
          } else {
#pragma unroll
            for (int c = 0; c < 16; ++c) pk[c] = 0u;               // rows outside the frame: post-ReLU zeros never win a max
          }
          uint4* o = reinterpret_cast<uint4*>(band + (size_t)r * pg.tile_pitch + (size_t)(j ^ ((j >> 1) & 1)) * STEM_C);
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
            const int off = (ww ^ ((ww >> 1) & 1)) * STEM_C + ((cg ^ ((ww >> 1) & 3)) * 8);
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
      band_border_rows(out, pg, n, b, rowlen, et, 256);
      asm volatile("bar.sync 1, 256;\n" ::: "memory");              // the band buffer may be overwritten
    }
  }
  stem_teardown(warp, tmem_base);
}

// fp16 pass 2 with the pool.  A thread holds BOTH outputs of its pixel, so the horizontal part of the pooling window starts in registers:
// per band row it parks M[J] = max(y[2J], y[2J+1]) and X[J] = y[2J+1] (two planes of Wo/2 pixels; Wo is even on this path), and a pooled
// value is the maximum over three rows of max(M[pw], X[pw-1]) -- six shared-memory loads instead of nine, on the pipe the MMAs stream their
// operands through.  A pixel's four 16-byte vectors are XOR-swizzled by (J >> 1) & 3: parking stores (lanes = consecutive pixels) and
// pooling reads are both bank-conflict free.
constexpr int S8_EG = 3;              // epilogue groups of pass 2 (4 warps each): 128 + 3 * 128 = 512 threads
__global__ void __launch_bounds__(128 + 128 * S8_EG, 1) stem8_pool_kernel(const __grid_constant__ CUtensorMap map_x8, const float* __restrict__ w,
                                                            const float* __restrict__ bias, StemGeo g, BandGeo pg, const float* __restrict__ mean,
                                                            const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, __nv_bfloat16* __restrict__ out) {
  using F = StemF16;
  extern __shared__ uint8_t smem_raw[];
  __shared__ StemBars<F> bars;
  __shared__ float s_sc[STEM_C], s_sh[STEM_C];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t seg_bytes = (uint32_t)pg.seg_rows * 128;
  const uint32_t s_w = smem_base, s_seg = smem_base + F::W_BYTES;
  __nv_bfloat16* band = reinterpret_cast<__nv_bfloat16*>(smem_gen + F::W_BYTES + 2 * seg_bytes);       // [S8_ROWS][tile_pitch]
  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int sub = pg.sub;

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
  const uint32_t tmem_base = stem_setup(bars, &map_x8, w, smem_gen, s_sc, warp);

  if (warp == 0) {
    stem_produce(bars, &map_x8, s_seg, seg_bytes, pg.n_items, [=](long long t) { return (int)box_row_of(band_start(t, S8_P, pg.bands_per_frame, g)); });
  } else if (warp == 1) {
    stem_issue<F, 0>(bars, tmem_base, s_seg, seg_bytes, s_w, g.Wq, pg.n_items, sub,
                     [=](long long t) { return box_off_of(band_start(t, S8_P, pg.bands_per_frame, g)); });
  } else if (warp >= 4) {
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    const int et = tid - 128;                                       // 0 .. 128*S8_EG - 1 among the epilogue threads
    constexpr int ET = 128 * S8_EG;
    uint32_t acc_cnt = 0;
    const int groups = STEM_C / 8;                                  // 16-byte vectors per pixel
    float rq[STEM_C];                                               // BatchNorm shift in registers (the scale sits in the weights)
#pragma unroll
    for (int c = 0; c < STEM_C; ++c) rq[c] = s_sh[c];
    const float kinv = s_kinv;
    for (long long t = blockIdx.x; t < pg.n_items; t += gridDim.x) {
      const long long n = t / pg.bands_per_frame;
      const int b = (int)(t - n * pg.bands_per_frame);
      const int i0 = 2 * S8_P * b - 1;                              // first convolution row of the band
      for (int sb = eg; sb < sub; sb += S8_EG) {
        const int ql = sb * 128 + ew * 32 + lane;                   // pixel inside the band
        const int r = ql / g.Wq, J = ql - r * g.Wq;
        const bool row_in = r < S8_ROWS && J < g.Wh;
        const bool live = row_in && i0 + r >= 0 && i0 + r < g.Ho;
        // all four 16-column loads of the row (both outputs) in flight before the single wait: one TMEM round trip per sub-tile, not two
        uint32_t acc[4][16];
        stem_take_acc(bars, tmem_base, acc_cnt + sb, ew, acc);
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
          uint4* om = reinterpret_cast<uint4*>(band + (size_t)r * pg.tile_pitch + (size_t)J * STEM_C);
          uint4* ox = reinterpret_cast<uint4*>(band + (size_t)r * pg.tile_pitch + (size_t)(g.Wh + J) * STEM_C);
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
          const int offm = pw * STEM_C + ((cg ^ ((pw >> 1) & 3)) * 8), offx = (g.Wh + jx) * STEM_C + ((cg ^ ((jx >> 1) & 3)) * 8);
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
      band_border_rows(out, pg, n, b, rowlen, et, ET);
      asm volatile("bar.sync 1, %0;\n" ::"n"(ET) : "memory");        // the band buffer may be overwritten
    }
  }
  stem_teardown(warp, tmem_base);
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

// ------------------------------------------------------------------------------------------------------------------------------------
// Host

// tf32 geometry: X4 is (Ho+3) x (Wo+3) pixels per frame
int stem_geo(StemGeo& g, int N, int H, int W) {
  g.N = N; g.H = H; g.W = W;
  g.Ho = (H - 1) / 2 + 1;
  g.Wo = (W - 1) / 2 + 1;
  g.Wh = 0;
  g.Hq = g.Ho + 3;
  g.Wq = g.Wo + 3;
  g.np = (long long)N * g.Hq * g.Wq;
  const int MT = 128 * StemTf32::TILE_SUB;
  g.n_tiles = (g.np + MT - 1) / MT;
  const int seg_px = MT + 3 * g.Wq + 3;
  g.seg_rows = (seg_px + 7) / 8;
  if (g.seg_rows > 256 || g.np + MT > 0x7fffffffLL) return 1;      // one TMA box per tile (frames up to ~1000 px wide)
  return 0;
}

// fp16 geometry: X8 is (Ho+3) x (Wh+2) pixels per frame
int geo8(StemGeo& g, int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0 || (W & 3)) return 1;
  g.N = N; g.H = H; g.W = W;
  g.Ho = (H - 1) / 2 + 1;
  g.Wo = (W - 1) / 2 + 1;
  g.Wh = (g.Wo + 1) / 2;
  g.Hq = g.Ho + 3;
  g.Wq = g.Wh + 2;
  g.np = (long long)N * g.Hq * g.Wq;
  const int MT = 128 * StemF16::TILE_SUB;
  g.n_tiles = (g.np + MT - 1) / MT;
  const int seg_px = MT + 3 * g.Wq + 2;
  g.seg_rows = (seg_px + 7) / 8;
  if (g.seg_rows > 256 || g.np + MT > 0x7fffffffLL) return 1;
  return 0;
}

// the pixel stream as a matrix of 128-byte rows (8 pixels), box_rows of them per TMA box; the last partial row is covered by the
// buffer's 128-byte slack
int stream_map(CUtensorMap* m, const void* xs, const StemGeo& g, int box_rows) {
  return make_tmap_2d(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, xs, (g.np + 7) / 8, 32, box_rows, 32, 0);
}

// dynamic shared memory of the pass-1 kernels (and of the unfused tf32 pass 2): weights, two stream segments, and at least the [256][65]
// floats of the statistics reduction
size_t pass1_smem(const StemGeo& g, int w_bytes) {
  const size_t smem = w_bytes + 2 * (size_t)g.seg_rows * 128 + 1024;
  const size_t red = w_bytes + 256 * 65 * 4 + 1024;
  return smem < red ? red : smem;
}

// pass-2 band geometry: P pooled rows per band, `slots` accumulators in the TMEM ring, w_bytes of packed weights, and `overhang` pixels
// the MMAs read past a sub-tile's 128.  False when a band does not fit one TMA box / the accumulator ring / shared memory (very wide
// frames); the callers then decline.
bool band_geo(const StemGeo& g, int P, int slots, int w_bytes, int overhang, BandGeo& pg, size_t& smem) {
  const int rows = 2 * P + 1;                                      // convolution rows per band
  pg.PH = (g.Ho - 1) / 2 + 1;
  pg.PW = (g.Wo - 1) / 2 + 1;
  pg.bands_per_frame = (pg.PH + P - 1) / P;
  pg.n_items = (long long)g.N * pg.bands_per_frame;
  pg.sub = (rows * g.Wq + 127) / 128;
  const int seg_px = 128 * pg.sub + overhang + 8;                  // + the pixel remainder of the box's 128-byte alignment
  pg.seg_rows = (seg_px + 7) / 8;
  pg.tile_pitch = ((g.Wo + 3) & ~3) * STEM_C;                      // whole groups of four columns: the tf32 slot swap stays inside the row
  const size_t band_bytes = (size_t)rows * pg.tile_pitch * sizeof(__nv_bfloat16);
  smem = w_bytes + 2 * (size_t)pg.seg_rows * 128 + band_bytes + 1024;
  return pg.seg_rows <= 256 && pg.sub <= slots && smem <= 220 * 1024;
}
bool band_geo_tf32(const StemGeo& g, BandGeo& pg, size_t& smem) { return band_geo(g, SP_P, StemTf32::SLOTS, StemTf32::W_BYTES, 3 * g.Wq + 3, pg, smem); }
bool band_geo_f16(const StemGeo& g, BandGeo& pg, size_t& smem) { return band_geo(g, S8_P, StemF16::SLOTS, StemF16::W_BYTES, 3 * g.Wq + 2, pg, smem); }

// pass 1 of formulation F over the stream xs, then the BatchNorm finalize
template <class F>
int stats_launch(const void* xs, const float* w, const float* bias, const StemGeo& g, double* ws, float eps, float momentum, float* mean,
                 float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked, cudaStream_t st) {
  CUtensorMap mx;
  const int e = stream_map(&mx, xs, g, g.seg_rows);
  if (e) return e;
  const size_t smem = pass1_smem(g, F::W_BYTES);
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem_stats_kernel<F>, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > g.n_tiles) grid = g.n_tiles;
  stem_stats_kernel<F><<<(unsigned)grid, 384, smem, st>>>(mx, w, g, ws);
  CVAD_LAUNCH_CHECK();
  // ws holds the sums of the RAW accumulator; y = acc + bias: the bias moves the mean, not the variance
  return bn_finalize_launch(ws, STEM_C, (double)g.N * g.Ho * g.Wo, bias, eps, momentum, mean, invstd, running_mean, running_var,
                            num_batches_tracked, st);
}

}  // namespace

CVAD_API long long cvad_stem_x4_floats(int N, int H, int W) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return -1;
  return ((g.np + 7) / 8) * 32 + 32;
}

CVAD_API int cvad_stem_space_to_depth_f32(const float* x, int N, int H, int W, float* x4, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  long long blocks = (g.np + 255) / 256;
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
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  return stats_launch<StemTf32>(x4, w, bias, g, ws, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked,
                                (cudaStream_t)stream);
}

CVAD_API int cvad_stem_tf32_bn_relu(const float* x4, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                    const float* invstd, const float* gamma, const float* beta, void* y, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  CUtensorMap mx;
  const int e = stream_map(&mx, x4, g, g.seg_rows);
  if (e) return e;
  const size_t smem = pass1_smem(g, StemTf32::W_BYTES);
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem_tf32_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > g.n_tiles) grid = g.n_tiles;
  stem_tf32_kernel<<<(unsigned)grid, 384, smem, (cudaStream_t)stream>>>(mx, w, bias, g, mean, invstd, gamma, beta, (__nv_bfloat16*)y);
  CVAD_LAUNCH_CHECK();
  return 0;
}

// pass 2 + max-pool in one kernel; returns cudaErrorNotSupported when a band does not fit (very wide frames): callers fall back
CVAD_API int cvad_stem_tf32_bn_relu_maxpool(const float* x4, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                            const float* invstd, const float* gamma, const float* beta, void* out, void* stream) {
  StemGeo g;
  if (stem_geo(g, N, H, W)) return (int)cudaErrorInvalidValue;
  BandGeo pg;
  size_t smem;
  if (!band_geo_tf32(g, pg, smem)) return (int)cudaErrorNotSupported;
  CUtensorMap mx;
  const int e = stream_map(&mx, x4, g, pg.seg_rows);
  if (e) return e;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem_pool_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > pg.n_items) grid = pg.n_items;
  stem_pool_kernel<<<(unsigned)grid, 384, smem, (cudaStream_t)stream>>>(mx, w, bias, g, pg, mean, invstd, gamma, beta, (__nv_bfloat16*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
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

// bytes of the X8 buffer for (N,1,H,W) frames (incl. the slack the last TMA row needs), or -1 when the shape is outside the fp16 stem's
// range (W not a multiple of 4, very wide frames): callers then use the tf32 stem
CVAD_API long long cvad_stem8_bytes(int N, int H, int W) {
  StemGeo g;
  BandGeo pg;
  size_t smem;
  if (geo8(g, N, H, W) || !band_geo_f16(g, pg, smem)) return -1;
  return ((g.np + 7) / 8) * 128 + 128;
}

CVAD_API int cvad_stem8_space_to_depth_f32(const float* x, int N, int H, int W, void* x8, void* stream) {
  StemGeo g;
  if (geo8(g, N, H, W) || ((uintptr_t)x & 15)) return (int)cudaErrorInvalidValue;
  long long blocks = (g.np + 255) / 256;
  if (blocks > 16LL * cvad_num_sms()) blocks = 16LL * cvad_num_sms();
  stem8_s2d_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, g, 0.f, 1.f, reinterpret_cast<uint4*>(x8));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_stem8_space_to_depth_u8(const void* x, int N, int H, int W, float mean, float stdv, void* x8, void* stream) {
  StemGeo g;
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
  StemGeo g;
  if (geo8(g, N, H, W)) return (int)cudaErrorInvalidValue;
  return stats_launch<StemF16>(x8, w, bias, g, ws, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked,
                               (cudaStream_t)stream);
}

CVAD_API int cvad_stem8_f16_bn_relu_maxpool(const void* x8, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                            const float* invstd, const float* gamma, const float* beta, void* out, void* stream) {
  StemGeo g;
  if (geo8(g, N, H, W)) return (int)cudaErrorInvalidValue;
  BandGeo pg;
  size_t smem;
  if (!band_geo_f16(g, pg, smem)) return (int)cudaErrorNotSupported;
  CUtensorMap mx;
  const int e = stream_map(&mx, x8, g, pg.seg_rows);
  if (e) return e;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(stem8_pool_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  long long grid = cvad_num_sms();
  if (grid > pg.n_items) grid = pg.n_items;
  stem8_pool_kernel<<<(unsigned)grid, 128 + 128 * S8_EG, smem, (cudaStream_t)stream>>>(mx, w, bias, g, pg, mean, invstd, gamma, beta,
                                                                                       (__nv_bfloat16*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

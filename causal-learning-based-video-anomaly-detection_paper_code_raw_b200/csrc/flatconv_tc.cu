// "Flat" tensor-core 3x3 convolution for the M-A backbone (cad:128-139, 150-153): forward, data-gradient and
// weight-gradient as TMA-fed tcgen05.mma GEMMs over a zero-bordered NHWC layout.
//
// Layout in HBM.  An activation with logical shape (N,H,W,C) is stored as (N, H+2, W+2, C) bf16 with a zero border
// ("padded-flat").  With q the flat pixel index of that buffer, a stride-1 3x3 convolution is a sum of nine row-shifted
// GEMMs over the SAME index space for input and output:
//        out[q][:] = sum_{kh,kw} in[q + (kh-1)*(W+2) + (kw-1)][:] * W[kh][kw]
// (border positions produce junk that nobody reads).  A stride-2 convolution reads its input from four "phase planes"
// P_ab[n][i][j] = in_padded(2(i-1)+a, 2(j-1)+b) stored in the OUTPUT's padded geometry, which makes it the same kind of
// sum: tap (kh,kw) reads plane (kh&1, kw&1) shifted by (kh>>1)*(Wo+2) + (kw>>1).  The data-gradients are the transposed
// sums (negative shifts; one launch per phase plane for stride 2).
//
// Forward / data-gradient kernel.  Persistent, warp-specialised, one CTA per SM:
//   warp 0  TMA producer, activations: per K-unit (a 32/64-channel slab of one source plane) one segment of 128*SUB + halo
//           rows, hardware-swizzled (SWIZZLE_64B / SWIZZLE_128B), double buffered;
//   warp 2  TMA producer, weights: boxes of 256 packed rows (2-8 taps each) through a ring, or loaded once and kept
//           resident when all taps fit; also owns the TMEM allocation;
//   warp 1  tcgen05.mma issuer: every tap is a ROW-SHIFTED VIEW of the resident segment (descriptor start address +
//           delta*row_bytes; the swizzle is a function of the absolute smem address, profiles/r01_umma_descriptor_probe.md),
//           M=128 x N x K=16 MMAs into a ring of TMEM accumulators;
//   warps 4-11 epilogue (two groups on alternate sub-tiles): tcgen05.ld -> +bias -> bf16 -> global, overlapped with the
//           next tile's MMAs.
// All role loops are warp-uniform and one elected lane issues, so descriptors live in uniform registers.  TMA boxes are as
// large as the hardware allows (256 rows): a box costs ~700 cycles of TMA service however small it is
// (profiles/r01_tma_box_probe.md).  An activation element is fetched from L2/HBM ~1.1-1.4x (halo) instead of 9x.
#include <cuda.h>

#include "common.cuh"
#include "cvad_b200.h"
#include "tc_common.cuh"

namespace {

using namespace cvad_tc;

constexpr int FC_MAX_UNITS = 16;
constexpr int FC_WST_MAX = 8;        // maximum weight ring depth
constexpr int FC_MAX_SLOTS = 16;     // TMEM accumulator ring
constexpr int FC_SRC_MAX = 3;        // activation-segment ring depth (2 or 3 stages, FcParams::nsrc)
constexpr int FC_BOX = 256;          // rows per big TMA box
constexpr size_t FC_SMEM_BUDGET = 222 * 1024;   // dynamic; the static part (barriers, bias, statistics) stays below 5 KB of the 227 KB

// optional profiling hook (tools/conv_probe.py): when set, the MMA-issuing warp of every CTA records the cycles it spent
// waiting on each barrier class: dbg[cta*8 + {0 total, 1 src_full, 2 w_full, 3 acc_empty, 4 work items, 5 entry ns, 6 loop start ns, 7 loop end ns}]
__device__ long long* g_fc_debug = nullptr;
constexpr int FC_DBG_CTAS = 148;     // buffer: FC_DBG_CTAS x 8 per-CTA records + {min entry ns (preset to max), max exit ns}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

struct FcUnit {
  int row_off;          // first segment row relative to the tile's first output row (may be negative)
  int col;              // first channel of the slab
  int ntaps;
  int w_row0;           // first packed weight row of the unit's first tap (n-block 0); tap i follows at + i*N
  int tap_delta[9];     // row shift of tap i inside the segment (>= 0)
  unsigned char tap_acc[9];           // accumulator set of tap i (0 unless one item fills several output planes)
  unsigned short first_mask, last_mask;   // bit i: tap i is the first / last tap of its accumulator set inside this unit
};

struct FcParams {
  long long rows;        // output rows (flat pixels)
  long long out_row_base;
  int n_units, seg_rows, sub, n_blocks, ld_out, wst, w_resident;
  int big_boxes, tail_rows;      // segment = big_boxes x 256 rows + one exact tail box (0 = none)
  // "groups": independent sub-problems per row tile walked by ONE launch (work item = tile x group x n-block).  Group g uses units
  // [group_unit0[g], + group_nunits[g]) and fills acc_sets accumulator sets (the same number in every group); set a of group g writes its
  // rows at out_row_base + group_plane[g][a] * plane_out_stride.  A stride-2 data-gradient is ONE group of four sets (the four phase
  // planes of dx computed from ONE fetch of the dy segment) or two groups of two; everything else is one group with one set.
  int n_groups, acc_sets, nsrc;
  int group_unit0[4], group_nunits[4], group_plane[4][4];
  long long plane_out_stride;
  // fused BatchNorm statistics (forward only, n_blocks == 1): per-channel sum / sum of squares of the bf16-rounded outputs over the
  // interior pixels (1..st_h, 1..st_w of every (st_h+2) x (st_w+2) image), added to st_out[0..N) / st_out[N..2N) (fp64, zeroed by the caller)
  int st_h, st_w;
  unsigned st_mul_img, st_shr_img, st_mul_row, st_shr_row;
  double* st_out;
  // fused BatchNorm-BACKWARD reductions (data-gradient only, n_blocks == 1): the rows this launch writes are the gradient dact w.r.t. the
  // output of relu(bn(raw)) of the layer below; with g = dact * (raw*ga + gb > 0) (ga = gamma*invstd, gb = beta - mean*ga) the epilogue adds
  // sum g and sum g*xhat over the interior pixels to st_out[0..N) / st_out[N..2N) -- the two per-channel sums of the BatchNorm backward,
  // which otherwise cost a full read pass over raw and dact.  planes: the rows are the four phase planes of a stride-2 input
  // (geometry (st_h+2) x (st_w+2) per plane) and map to pixel (2(i-1)+a, 2(j-1)+b) of the bw_H x bw_W interior of raw.
  // ReLU-output forward (EPI_RELU): the output interior is st_h x st_w; planes = 1 writes it as the four phase planes of the next
  // stride-2 convolution, plane_out_stride rows apart, instead of padded-flat.
  const __nv_bfloat16* bw_raw;
  const float *bw_gamma, *bw_beta, *bw_mean, *bw_invstd;
  int bw_H, bw_W, planes;
  // masked column sums (EPI_MASK, data-gradient only, n_blocks == 1): sum_mask holds N bits per output row in the rows' own layout (bit c in
  // 32-bit word c/32; the ReLU gate the BatchNorm apply of the layer below wrote, 0 on borders and empty plane positions); the epilogue adds
  // sum over rows of bf16(out) * bit to st_out[0..N) -- the BatchNorm backward's sum g, with no pixel decode and no per-column constants
  const uint32_t* sum_mask;
  FcUnit units[FC_MAX_UNITS];
};

// Column sums of a 32-row x 16-column register tile held one row per lane, for the values and their squares at once (two independent
// shuffle chains): a butterfly that halves the number of columns a lane carries at every exchange (8 + 4 + 2 + 1 shuffles) and a final
// pair exchange; afterwards every lane holds the 32-row sums of column 8*bit4 + 4*bit3 + 2*bit2 + bit1 of its lane index.
__device__ __forceinline__ void warp_colsum16_sq(const float (&x)[16], int lane, float& sum, float& sumsq) {
  float y[8], z[4], w[2], yy[8], zz[4], ww[2];
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float keep = b4 ? x[i + 8] : x[i], send = b4 ? x[i] : x[i + 8];
    y[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    yy[i] = fmaf(keep, keep, __shfl_xor_sync(0xffffffffu, send * send, 16));
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    z[i] = (b3 ? y[i + 4] : y[i]) + __shfl_xor_sync(0xffffffffu, b3 ? y[i] : y[i + 4], 8);
    zz[i] = (b3 ? yy[i + 4] : yy[i]) + __shfl_xor_sync(0xffffffffu, b3 ? yy[i] : yy[i + 4], 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    w[i] = (b2 ? z[i + 2] : z[i]) + __shfl_xor_sync(0xffffffffu, b2 ? z[i] : z[i + 2], 4);
    ww[i] = (b2 ? zz[i + 2] : zz[i]) + __shfl_xor_sync(0xffffffffu, b2 ? zz[i] : zz[i + 2], 4);
  }
  const float v = (b1 ? w[1] : w[0]) + __shfl_xor_sync(0xffffffffu, b1 ? w[0] : w[1], 2);
  const float vv = (b1 ? ww[1] : ww[0]) + __shfl_xor_sync(0xffffffffu, b1 ? ww[0] : ww[1], 2);
  sum = v + __shfl_xor_sync(0xffffffffu, v, 1);
  sumsq = vv + __shfl_xor_sync(0xffffffffu, vv, 1);
}

// the same butterfly for one 32 x 16 tile
__device__ __forceinline__ float warp_colsum16(const float (&x)[16], int lane) {
  float y[8], z[4], w[2];
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
  for (int i = 0; i < 8; ++i) y[i] = (b4 ? x[i + 8] : x[i]) + __shfl_xor_sync(0xffffffffu, b4 ? x[i] : x[i + 8], 16);
#pragma unroll
  for (int i = 0; i < 4; ++i) z[i] = (b3 ? y[i + 4] : y[i]) + __shfl_xor_sync(0xffffffffu, b3 ? y[i] : y[i + 4], 8);
#pragma unroll
  for (int i = 0; i < 2; ++i) w[i] = (b2 ? z[i + 2] : z[i]) + __shfl_xor_sync(0xffffffffu, b2 ? z[i] : z[i + 2], 4);
  const float v = (b1 ? w[1] : w[0]) + __shfl_xor_sync(0xffffffffu, b1 ? w[0] : w[1], 2);
  return v + __shfl_xor_sync(0xffffffffu, v, 1);
}

// the same butterfly for two independent 32 x 16 tiles (column sums of a and of b)
__device__ __forceinline__ void warp_colsum16_pair(const float (&a)[16], const float (&b)[16], int lane, float& sum_a, float& sum_b) {
  float y[8], z[4], w[2], yy[8], zz[4], ww[2];
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    y[i] = (b4 ? a[i + 8] : a[i]) + __shfl_xor_sync(0xffffffffu, b4 ? a[i] : a[i + 8], 16);
    yy[i] = (b4 ? b[i + 8] : b[i]) + __shfl_xor_sync(0xffffffffu, b4 ? b[i] : b[i + 8], 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    z[i] = (b3 ? y[i + 4] : y[i]) + __shfl_xor_sync(0xffffffffu, b3 ? y[i] : y[i + 4], 8);
    zz[i] = (b3 ? yy[i + 4] : yy[i]) + __shfl_xor_sync(0xffffffffu, b3 ? yy[i] : yy[i + 4], 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    w[i] = (b2 ? z[i + 2] : z[i]) + __shfl_xor_sync(0xffffffffu, b2 ? z[i] : z[i + 2], 4);
    ww[i] = (b2 ? zz[i + 2] : zz[i]) + __shfl_xor_sync(0xffffffffu, b2 ? zz[i] : zz[i + 2], 4);
  }
  const float v = (b1 ? w[1] : w[0]) + __shfl_xor_sync(0xffffffffu, b1 ? w[0] : w[1], 2);
  const float vv = (b1 ? ww[1] : ww[0]) + __shfl_xor_sync(0xffffffffu, b1 ? ww[0] : ww[1], 2);
  sum_a = v + __shfl_xor_sync(0xffffffffu, v, 1);
  sum_b = vv + __shfl_xor_sync(0xffffffffu, vv, 1);
}

// Epilogue kinds, each a separate instantiation: the epilogue of the plain kernels is timing-critical (8 warps against the MMA stream) and
// must not carry optional code.
//   EPI_PLAIN  out = conv + bias (junk on the border rows), optionally with the BatchNorm batch statistics (FcParams::st_out)
//   EPI_BW     data-gradient that also takes the BatchNorm-backward reductions (FcParams::bw_raw)
//   EPI_RELU   out = relu(conv + bias) on interior pixels and exact zeros on the border: the forward of an eval-mode BatchNorm + ReLU
//              already folded into the weights and bias; padded-flat or phase planes (FcParams::planes)
//   EPI_MASK   data-gradient that also sums its bf16 output under a per-row bitmask (FcParams::sum_mask): the successor of EPI_BW, which
//              loaded raw (as many bytes as it wrote) and formed xhat per element and slowed the MMAs; this one loads N bits per row
enum { EPI_PLAIN = 0, EPI_BW = 1, EPI_RELU = 2, EPI_MASK = 3 };
template <int ROWB, int N, int EPI>
__global__ void __launch_bounds__(384, 1) flatconv_kernel(const __grid_constant__ CUtensorMap map_src, const __grid_constant__ CUtensorMap map_tail,
                                                          const __grid_constant__ CUtensorMap map_w, const FcParams p,
                                                          const float* __restrict__ bias, __nv_bfloat16* __restrict__ out) {
  constexpr bool BW = EPI == EPI_BW, RELU = EPI == EPI_RELU, MS = EPI == EPI_MASK;
  constexpr int NSLOT = (512 / N) > FC_MAX_SLOTS ? FC_MAX_SLOTS : (512 / N);
  constexpr uint32_t TMEM_COLS = NSLOT * N;
  constexpr int TPO = FC_BOX / N;                  // taps per weight box
  constexpr int WBOX_BYTES = FC_BOX * ROWB;
  constexpr int K16 = ROWB / 32;
  constexpr uint32_t SBO = ROWB * 8;
  constexpr int LAYOUT = ROWB == 128 ? UMMA_SW128 : UMMA_SW64;

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_src_full[FC_SRC_MAX], bar_src_empty[FC_SRC_MAX], bar_w_full[FC_WST_MAX], bar_w_empty[FC_WST_MAX], bar_acc_full[FC_MAX_SLOTS],
      bar_acc_empty[FC_MAX_SLOTS];
  __shared__ uint32_t tmem_base_sh;
  __shared__ float s_bias[N];
  __shared__ float s_stat[2 * N];          // fused BatchNorm statistics of this CTA's rows (fp32 partial sums, flushed once at the end)
  __shared__ float s_ga[N], s_gb[N];       // fused BatchNorm-backward reductions: the forward's per-channel scale / shift
  for (int i = threadIdx.x; i < 2 * N; i += blockDim.x) s_stat[i] = 0.f;
  if (BW)
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
      const float ga = p.bw_gamma[i] * p.bw_invstd[i];
      s_ga[i] = ga;
      s_gb[i] = p.bw_beta[i] - p.bw_mean[i] * ga;
    }
  const long long t_entry = g_fc_debug ? (long long)globaltimer_ns() : 0;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t seg_bytes = (uint32_t)p.seg_rows * ROWB;
  const uint32_t s_src = smem_base;
  const int nsrc = p.nsrc;
  const uint32_t s_w = smem_base + nsrc * seg_bytes;

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int sub = p.sub, n_units = p.n_units, n_blocks = p.n_blocks, wst = p.wst, resident = p.w_resident;
  const int MT = 128 * sub;
  const long long n_tiles = (p.rows + MT - 1) / MT;
  const int n_groups = p.n_groups, acc_sets = p.acc_sets;
  const long long total = n_tiles * n_blocks * n_groups;
  const int item_slots = acc_sets * sub;            // accumulators one work item fills
  // work item -> (tile, group, n-block).  The groups of one tile are consecutive items, i.e. they run on neighbouring CTAs at the same
  // time and share their source segment through L2; the group index is rotated by the round (wi / gridDim.x, gridDim.x is a multiple of
  // n_groups) so that every CTA sees all groups, whose tap counts differ.
#define FC_DECODE(wi, g, q0, nb)                                                        \
  int g = 0, nb;                                                                          \
  long long q0;                                                                           \
  {                                                                                       \
    long long rest = (wi);                                                                \
    if (n_groups > 1) {                                                                   \
      g = (int)(((wi) + (wi) / gridDim.x) % n_groups);                                    \
      rest = (wi) / n_groups;                                                             \
    }                                                                                     \
    q0 = (rest / n_blocks) * MT;                                                          \
    nb = (int)(rest % n_blocks);                                                          \
  }

  if (tid == 0) {
    for (int i = 0; i < FC_SRC_MAX; ++i) { mbar_init(&bar_src_full[i], 1); mbar_init(&bar_src_empty[i], 1); }
    for (int i = 0; i < FC_WST_MAX; ++i) { mbar_init(&bar_w_full[i], 1); mbar_init(&bar_w_empty[i], 1); }
    for (int i = 0; i < FC_MAX_SLOTS; ++i) { mbar_init(&bar_acc_full[i], 1); mbar_init(&bar_acc_empty[i], 128); }
    fence_barrier_init();
    prefetch_tmap(&map_src);
    prefetch_tmap(&map_tail);
    prefetch_tmap(&map_w);
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(&tmem_base_sh);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer: activation segments
    uint32_t src_cnt = 0;
    for (long long wi = blockIdx.x; wi < total; wi += gridDim.x) {
      FC_DECODE(wi, g, q0, nb)
      (void)nb;
      const int u0 = p.group_unit0[g], nu = p.group_nunits[g];
      for (int u = u0; u < u0 + nu; ++u) {
        const int st = (int)(src_cnt % nsrc);
        mbar_wait(&bar_src_empty[st], ((src_cnt / nsrc) & 1) ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bar_src_full[st], seg_bytes);
          const int r0 = (int)(q0 + p.units[u].row_off), col = p.units[u].col;
          const uint32_t dst = s_src + st * seg_bytes;
          for (int b = 0; b < p.big_boxes; ++b) tma_load_2d(dst + b * (FC_BOX * ROWB), &map_src, col, r0 + b * FC_BOX, &bar_src_full[st]);
          if (p.tail_rows) tma_load_2d(dst + p.big_boxes * (FC_BOX * ROWB), &map_tail, col, r0 + p.big_boxes * FC_BOX, &bar_src_full[st]);
        }
        __syncwarp();
        ++src_cnt;
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ TMA producer: weight boxes (TPO taps each)
    uint32_t w_cnt = 0;
    bool first_item = true;
    for (long long wi = blockIdx.x; wi < total; wi += gridDim.x) {
      FC_DECODE(wi, g, q0, nb)
      (void)q0;
      if (resident && !first_item) break;
      const int u0 = p.group_unit0[g], nu = p.group_nunits[g];
      for (int u = u0; u < u0 + nu; ++u) {
        const int ntaps = p.units[u].ntaps, col = p.units[u].col;
        const int row0 = p.units[u].w_row0 + nb * 9 * N;
        for (int c = 0; c * TPO < ntaps; ++c) {
          const int st = resident ? c : (int)(w_cnt % wst);
          if (!resident) mbar_wait(&bar_w_empty[st], ((w_cnt / wst) & 1) ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&bar_w_full[st], WBOX_BYTES);
            tma_load_2d(s_w + st * WBOX_BYTES, &map_w, col, row0 + c * FC_BOX, &bar_w_full[st]);
          }
          __syncwarp();
          ++w_cnt;
        }
      }
      first_item = false;
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (whole warp walks the loops, one lane issues)
    const uint32_t idesc = make_idesc_bf16(128, N, 0, 0);
    const uint64_t desc_hi = make_smem_desc(0, 16, SBO, LAYOUT);
    uint32_t src_cnt = 0, w_cnt = 0, acc_cnt = 0;
    long long* dbg = g_fc_debug;
    long long t_src = 0, t_w = 0, t_acc = 0, n_items = 0;
    const long long t_begin = dbg ? clock64() : 0;
    const long long t_loop_ns = dbg ? (long long)globaltimer_ns() : 0;
    for (long long wi = blockIdx.x; wi < total; wi += gridDim.x) {
      ++n_items;
      FC_DECODE(wi, g, q0, nb)
      (void)q0;
      (void)nb;
      const int u0 = p.group_unit0[g], nu = p.group_nunits[g];
      for (int u = u0; u < u0 + nu; ++u) {
        const int ntaps = p.units[u].ntaps;
        const uint32_t first_mask = u == u0 ? p.units[u].first_mask : 0u, last_mask = u == u0 + nu - 1 ? p.units[u].last_mask : 0u;
        const int st = (int)(src_cnt % nsrc);
        long long tq = dbg ? clock64() : 0;
        mbar_wait(&bar_src_full[st], (src_cnt / nsrc) & 1);
        if (dbg) t_src += clock64() - tq;
        tc_fence_after();
        const uint32_t a_seg = s_src + st * seg_bytes;
        for (int c = 0; c * TPO < ntaps; ++c) {
          const int ws = resident ? c : (int)(w_cnt % wst);
          tq = dbg ? clock64() : 0;
          mbar_wait(&bar_w_full[ws], resident ? 0u : ((w_cnt / wst) & 1));
          if (dbg) t_w += clock64() - tq;
          tc_fence_after();
          const int tin = ntaps - c * TPO < TPO ? ntaps - c * TPO : TPO;
          for (int j = 0; j < tin; ++j) {
            const int t = c * TPO + j;
            const bool first = (first_mask >> t) & 1u;          // overwrite: the first tap of its accumulator set in the item's first unit
            const bool last = (last_mask >> t) & 1u;
            const uint32_t acc0 = acc_cnt + p.units[u].tap_acc[t] * sub;
            // descriptors advance by plain adds: (bytes >> 4) never carries out of the 14-bit address field (smem < 256 KiB)
            const uint64_t db0 = desc_hi | (uint64_t)(((s_w + ws * WBOX_BYTES + j * (N * ROWB)) >> 4) & 0x3FFF);
            const uint64_t da0 = desc_hi | (uint64_t)(((a_seg + (uint32_t)p.units[u].tap_delta[t] * ROWB) >> 4) & 0x3FFF);
            if (first) {
              // first tap of a tile: each accumulator slot must have been drained by the epilogue (overwrite, no accumulate)
              for (int s = 0; s < sub; ++s) {
                const uint32_t use = acc0 + s;
                const int slot = use % NSLOT;
                tq = dbg ? clock64() : 0;
                mbar_wait(&bar_acc_empty[slot], ((use / NSLOT) & 1) ^ 1);
                if (dbg) t_acc += clock64() - tq;
                tc_fence_after();
                if (elect_one()) {
#pragma unroll
                  for (int k = 0; k < K16; ++k) tc_mma_f16(tmem_base + slot * N, da0 + (uint64_t)(s * (128 * ROWB / 16) + 2 * k), db0 + 2 * k, idesc, k != 0);
                  if (last) tc_commit(&bar_acc_full[slot]);
                }
                __syncwarp();
              }
            } else {
              if (elect_one()) {
                uint32_t slot = acc0 % NSLOT;
                uint64_t da = da0;
                for (int s = 0; s < sub; ++s) {
#pragma unroll
                  for (int k = 0; k < K16; ++k) tc_mma_f16(tmem_base + slot * N, da + 2 * k, db0 + 2 * k, idesc, 1u);
                  if (last) tc_commit(&bar_acc_full[slot]);
                  da += 128 * ROWB / 16;
                  slot = slot + 1 == NSLOT ? 0 : slot + 1;
                }
              }
              __syncwarp();
            }
          }
          if (!resident) {
            if (elect_one()) tc_commit(&bar_w_empty[ws]);
            __syncwarp();
          }
          ++w_cnt;
        }
        if (elect_one()) tc_commit(&bar_src_empty[st]);
        __syncwarp();
        ++src_cnt;
      }
      acc_cnt += item_slots;
    }
    if (dbg && lane == 0) {
      long long* d = dbg + (long long)blockIdx.x * 8;
      d[0] = clock64() - t_begin; d[1] = t_src; d[2] = t_w; d[3] = t_acc; d[4] = n_items;
      d[5] = t_entry; d[6] = t_loop_ns; d[7] = (long long)globaltimer_ns();      // kernel entry / MMA loop start / MMA loop end (ns)
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ epilogue (TMEM lanes 32*(warp-4) ..)
    // two groups of four warps (4-7, 8-11) take alternate sub-tiles; warp w reads TMEM lanes 32*(w%4)..
    const int ew = (warp - 4) & 3, eg = (warp - 4) >> 2;
    uint32_t acc_cnt = 0;
    int cur_nb = -1;
    float st_s[N / 16], st_q[N / 16];          // fused statistics: this lane's column of every 16-column chunk, over all its tiles
#pragma unroll
    for (int i = 0; i < N / 16; ++i) { st_s[i] = 0.f; st_q[i] = 0.f; }

    // The bias add reads its operand from shared memory as a broadcast: N wavefronts per warp and sub-tile on the pipe that also
    // feeds the MMAs their operands (+18 % at N = 32).  Data-gradients have no bias (has_bias = false skips the reads); at N = 32 the
    // bias lives in registers.
    const bool has_bias = bias != nullptr;
    constexpr bool BIAS_REGS = N == 32;
    float rb[BIAS_REGS ? N : 1];
    for (long long wi = blockIdx.x; wi < total; wi += gridDim.x) {
      FC_DECODE(wi, g, q0, nb)
      if (nb != cur_nb) {                       // stage this n-block's bias once (epilogue warps only: named barrier 1)
        asm volatile("bar.sync 1, 256;\n" ::: "memory");
        for (int i = tid - 128; i < N; i += 256) s_bias[i] = bias ? __ldg(bias + nb * N + i) : 0.f;
        asm volatile("bar.sync 1, 256;\n" ::: "memory");
        cur_nb = nb;
        if (BIAS_REGS) {
#pragma unroll
          for (int i = 0; i < (BIAS_REGS ? N : 1); ++i) rb[i] = s_bias[i];
        }
      }
      for (int idx = eg; idx < item_slots; idx += 2) {        // accumulator sets in the order the MMA warp completes them
        const int a = idx / sub, s = idx - a * sub;
        const int pl = p.group_plane[g][a];
        const uint32_t use = acc_cnt + idx;
        const int slot = use % NSLOT;
        // row bookkeeping first: none of it depends on the accumulator, and the raw loads of the fused BatchNorm-backward reductions
        // are issued BEFORE the wait so that their latency hides behind the MMAs still running for this slot
        const long long q = q0 + s * 128 + ew * 32 + lane;
        const uint32_t taddr = tmem_base + slot * N + ((uint32_t)(ew * 32) << 16);
        __nv_bfloat16* orow = out + (p.out_row_base + pl * p.plane_out_stride + q) * (long long)p.ld_out + nb * N;
        bool keep = false;                    // interior pixel (the only ones BatchNorm statistics run over)
        constexpr bool bw = BW;
        const __nv_bfloat16* rrow = nullptr;  // bw: this row's pixel in raw
        if ((RELU || (p.st_out && !MS)) && q < p.rows) {
          const int qi = (int)q;
          const int n = fast_div(qi, p.st_mul_img, p.st_shr_img);
          const int r = qi - n * ((p.st_h + 2) * (p.st_w + 2));
          const int i = fast_div(r, p.st_mul_row, p.st_shr_row), j = r - i * (p.st_w + 2);
          if (!BW || !p.planes) {
            keep = i >= 1 && i <= p.st_h && j >= 1 && j <= p.st_w;
            if (bw) rrow = p.bw_raw + q * (long long)N;
            if (RELU && p.planes) {           // padded pixel (i, j) -> plane (i&1, j&1) at (i>>1 + 1, j>>1 + 1): the inverse of tc.to_phase
              const int hq = (p.st_h - 1) / 2 + 3, wq = (p.st_w - 1) / 2 + 3;
              const long long prow = ((i & 1) * 2 + (j & 1)) * p.plane_out_stride + ((long long)n * hq + (i >> 1) + 1) * wq + (j >> 1) + 1;
              orow = out + prow * (long long)p.ld_out + nb * N;
            }
          } else {
            const int hp = 2 * (i - 1) + (pl >> 1), wp = 2 * (j - 1) + (pl & 1);
            keep = hp >= 1 && hp <= p.bw_H && wp >= 1 && wp <= p.bw_W;
            rrow = p.bw_raw + (((long long)n * (p.bw_H + 2) + hp) * (p.bw_W + 2) + wp) * (long long)N;
          }
        }
        constexpr int NCH = N / 16;
        constexpr int PF = !BW ? 1 : (NCH < 4 ? NCH : 4);  // 16-column chunks of raw in flight per thread (a ring of 2*PF 16-byte registers)
        uint4 rq[PF][2];
        const bool bwk = bw && keep;
        if (BW) {
#pragma unroll
          for (int c = 0; c < PF; ++c) {
            rq[c][0] = make_uint4(0, 0, 0, 0);
            rq[c][1] = make_uint4(0, 0, 0, 0);
            if (bwk) {
              rq[c][0] = __ldg(reinterpret_cast<const uint4*>(rrow + c * 16));
              rq[c][1] = __ldg(reinterpret_cast<const uint4*>(rrow + c * 16 + 8));
            }
          }
        }
        constexpr int NW = MS ? N / 32 : 1;    // mask words of a row
        uint32_t mw[NW];
        if (MS) {
          const uint32_t* mrow = p.sum_mask + (p.out_row_base + pl * p.plane_out_stride + q) * NW;
#pragma unroll
          for (int k = 0; k < NW; ++k) mw[k] = 0u;
          if (q < p.rows) {
            if (NW % 4 == 0) {
#pragma unroll
              for (int k = 0; k < NW; k += 4) {
                const uint4 t = __ldg(reinterpret_cast<const uint4*>(mrow + k));
                mw[k] = t.x; mw[k + 1 < NW ? k + 1 : 0] = t.y; mw[k + 2 < NW ? k + 2 : 0] = t.z; mw[k + 3 < NW ? k + 3 : 0] = t.w;
              }
            } else if (NW == 2) {
              const uint2 t = __ldg(reinterpret_cast<const uint2*>(mrow));
              mw[0] = t.x; mw[NW - 1] = t.y;
            } else {
              mw[0] = __ldg(mrow);
            }
          }
        }
        mbar_wait(&bar_acc_full[slot], (use / NSLOT) & 1);
        tc_fence_after();
#pragma unroll
        for (int c0 = 0; c0 < N; c0 += 16) {
          uint32_t v[16];
          tmem_ld16(taddr + c0, v);
          tmem_ld_wait();
          uint32_t pk[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float a = __uint_as_float(v[2 * i]), b = __uint_as_float(v[2 * i + 1]);
            if (BIAS_REGS) {
              a += rb[BIAS_REGS ? c0 + 2 * i : 0];
              b += rb[BIAS_REGS ? c0 + 2 * i + 1 : 0];
            } else if (has_bias) {
              a += s_bias[c0 + 2 * i];
              b += s_bias[c0 + 2 * i + 1];
            }
            if (RELU) {
              a = keep ? fmaxf(a, 0.f) : 0.f;
              b = keep ? fmaxf(b, 0.f) : 0.f;
            }
            __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
            pk[i] = *reinterpret_cast<uint32_t*>(&h);
          }
          if (q < p.rows) {
            *reinterpret_cast<uint4*>(orow + c0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            *reinterpret_cast<uint4*>(orow + c0 + 8) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
          }
          if (MS) {                           // sum of the bf16 values just stored, under the row's mask bits
            const uint32_t bits = mw[(c0 / 32) % NW] >> (c0 & 16);
            float x[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              x[2 * i] = (bits >> (2 * i)) & 1u ? __uint_as_float(pk[i] << 16) : 0.f;
              x[2 * i + 1] = (bits >> (2 * i + 1)) & 1u ? __uint_as_float(pk[i] & 0xffff0000u) : 0.f;
            }
            st_s[c0 / 16] += warp_colsum16(x, lane);
          } else if (EPI == EPI_PLAIN && p.st_out) {     // warp-uniform: statistics of exactly the values the BatchNorm kernels will read back
            float x[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              x[2 * i] = keep ? __uint_as_float(pk[i] << 16) : 0.f;
              x[2 * i + 1] = keep ? __uint_as_float(pk[i] & 0xffff0000u) : 0.f;
            }
            float cs, cq;
            warp_colsum16_sq(x, lane, cs, cq);
            st_s[c0 / 16] += cs;
            st_q[c0 / 16] += cq;
          } else if (BW && p.st_out) {        // BatchNorm-backward sums over g = dact * relu'(bn(raw)) and g * raw, from the bf16 values just stored
            uint4 rv[2] = {rq[(c0 / 16) % PF][0], rq[(c0 / 16) % PF][1]};
            if (c0 / 16 + PF < NCH) {         // refill the ring slot just consumed
              rq[(c0 / 16) % PF][0] = make_uint4(0, 0, 0, 0);
              rq[(c0 / 16) % PF][1] = make_uint4(0, 0, 0, 0);
              if (bwk) {
                rq[(c0 / 16) % PF][0] = __ldg(reinterpret_cast<const uint4*>(rrow + c0 + PF * 16));
                rq[(c0 / 16) % PF][1] = __ldg(reinterpret_cast<const uint4*>(rrow + c0 + PF * 16 + 8));
              }
            }
            const uint32_t* rw = reinterpret_cast<const uint32_t*>(rv);
            float ga[16], gx[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float x0 = __uint_as_float(rw[i] << 16), x1 = __uint_as_float(rw[i] & 0xffff0000u);
              const float d0 = __uint_as_float(pk[i] << 16), d1 = __uint_as_float(pk[i] & 0xffff0000u);
              const float g0 = (keep && fmaf(x0, s_ga[c0 + 2 * i], s_gb[c0 + 2 * i]) > 0.f) ? d0 : 0.f;
              const float g1 = (keep && fmaf(x1, s_ga[c0 + 2 * i + 1], s_gb[c0 + 2 * i + 1]) > 0.f) ? d1 : 0.f;
              ga[2 * i] = g0;
              ga[2 * i + 1] = g1;
              gx[2 * i] = g0 * x0;
              gx[2 * i + 1] = g1 * x1;
            }
            float cs, cq;
            warp_colsum16_pair(ga, gx, lane, cs, cq);
            st_s[c0 / 16] += cs;
            st_q[c0 / 16] += cq;
          }
        }
        tc_fence_before();
        mbar_arrive(&bar_acc_empty[slot]);
      }
      acc_cnt += item_slots;
    }
    if (!RELU && p.st_out && !(lane & 1)) {   // one shared-memory add per warp and column, once per kernel
      const int col = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
#pragma unroll
      for (int i = 0; i < N / 16; ++i) {
        atomicAdd(&s_stat[i * 16 + col], st_s[i]);
        if (!MS) atomicAdd(&s_stat[N + i * 16 + col], st_q[i]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<TMEM_COLS>(tmem_base);
  if (EPI == EPI_PLAIN && p.st_out)
    for (int i = tid; i < 2 * N; i += blockDim.x) atomicAdd(p.st_out + i, (double)s_stat[i]);
  if (MS)
    for (int i = tid; i < N; i += blockDim.x) atomicAdd(p.st_out + i, (double)s_stat[i]);
  if (BW && p.st_out)                     // sum g*xhat = invstd * (sum g*x - mean * sum g), combined in fp64 (as pad_reduce_kernel does)
    for (int i = tid; i < N; i += blockDim.x) {
      const double a0 = (double)s_stat[i], a1 = (double)s_stat[N + i];
      atomicAdd(p.st_out + i, a0);
      atomicAdd(p.st_out + N + i, (a1 - (double)p.bw_mean[i] * a0) * (double)p.bw_invstd[i]);
    }
  if (g_fc_debug && tid == 0) {      // grid-wide first entry / last exit (ns) behind the per-CTA records
    atomicMin((unsigned long long*)g_fc_debug + FC_DBG_CTAS * 8, (unsigned long long)t_entry);
    atomicMax((unsigned long long*)g_fc_debug + FC_DBG_CTAS * 8 + 1, globaltimer_ns());
  }
#undef FC_DECODE
}

// ---------------------------------------------------------------------------------------------- host side
inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
// Stride-2 data-gradient: 2 = one launch, one work item per row tile fills all four phase planes of dx from ONE fetch of the dy segment
// (two items of two planes when four accumulator sets would leave the TMEM ring without a second buffer); 1 = one launch, one item per
// (tile, plane): dy is fetched four times; 0 = one launch per plane.  cvad_flat_dgrad_mode() switches (A/B measurements).
int g_dgrad_mode = 2;
// development knobs (cvad_flat_tune): [0] cap on the 128-row sub-tiles per work item for N = 128 (4 fills the whole accumulator ring,
// 2 leaves a second buffer for the epilogue); [1] activation-segment ring depth for items with several units (3 = a third stage when
// shared memory allows, 2 = always double buffering)
int g_fc_tune[4] = {2, 3, 0, 0};      // [2] != 0: single dy fetch for every stride-2 data-gradient; [3] != 0: stride-2 weight gradients with pixel-shift atoms
// Output-channel block = the MMA's N.  One M128 x N x K16 MMA streams 4 KB of A plus N*32 B of B from shared memory at ~80-90 B/cycle
// (profiles/r01g_flatconv_L0_ncu_full.md), so it is operand-bound below N = 256: take the widest N the layer allows.
inline int n_block_of(int nout) { return nout % 256 == 0 ? 256 : (nout % 128 == 0 ? 128 : (nout % 64 == 0 ? 64 : 32)); }

// fills the bookkeeping every launch needs from the units' tap lists: a single group / accumulator set unless the caller set them up,
// and the per-unit first / last masks
void finish_units(FcParams& p) {
  if (p.n_groups < 1) {
    p.n_groups = 1;
    p.group_unit0[0] = 0;
    p.group_nunits[0] = p.n_units;
  }
  if (p.acc_sets < 1) p.acc_sets = 1;
  for (int u = 0; u < p.n_units; ++u) {
    FcUnit& un = p.units[u];
    un.first_mask = un.last_mask = 0;
    for (int a = 0; a < p.acc_sets; ++a) {
      int f = -1, l = -1;
      for (int t = 0; t < un.ntaps; ++t)
        if (un.tap_acc[t] == a) {
          if (f < 0) f = t;
          l = t;
        }
      if (f >= 0) {
        un.first_mask |= (unsigned short)(1u << f);
        un.last_mask |= (unsigned short)(1u << l);
      }
    }
  }
}

template <int ROWB, int N, int EPI>
int launch_flatconv(const void* src, long long src_rows, int K, const void* wpk, long long w_rows, FcParams& p, const float* bias,
                    __nv_bfloat16* out, cudaStream_t st) {
  constexpr int TPO = FC_BOX / N;
  constexpr int NSLOT = (512 / N) > FC_MAX_SLOTS ? FC_MAX_SLOTS : (512 / N);
  finish_units(p);
  int max_delta = 0, max_chunks = 0, max_group_units = 0;
  for (int u = 0; u < p.n_units; ++u) {
    for (int t = 0; t < p.units[u].ntaps; ++t) max_delta = p.units[u].tap_delta[t] > max_delta ? p.units[u].tap_delta[t] : max_delta;
    const int ch = (p.units[u].ntaps + TPO - 1) / TPO;
    max_chunks = ch > max_chunks ? ch : max_chunks;
  }
  for (int g = 0; g < p.n_groups; ++g) max_group_units = p.group_nunits[g] > max_group_units ? p.group_nunits[g] : max_group_units;
  // rows per work item: as many 128-row sub-tiles as TMEM and shared memory allow while the machine stays filled.  TMEM: 512 columns =
  // NSLOT accumulators; an item fills acc_sets x sub of them, and the epilogue overlaps the next item's MMAs only when that is at most
  // half the ring.  N = 256 has two slots and keeps sub = 2 without a second buffer: one 128-row sub-tile per 32 KB weight box would
  // make the weight stream the limiter (measured: 84 -> 92 us at 8x12 256->256)
  static const int cand[] = {8, 6, 4, 3, 2, 1};
  int sub_max = NSLOT / p.acc_sets;
  if (NSLOT >= 4 * p.acc_sets && !(N == 128 && p.acc_sets == 1 && g_fc_tune[0] >= 4)) sub_max = NSLOT / (2 * p.acc_sets);
  if (sub_max < 1) return (int)cudaErrorInvalidValue;
  p.sub = 0;
  for (int sub : cand) {
    if (sub > sub_max) continue;
    const long long items = ((p.rows + 128LL * sub - 1) / (128LL * sub)) * p.n_blocks * p.n_groups;
    if (sub > 1 && items < (3LL * cvad_num_sms()) / 2) continue;
    const int seg = round_up(128 * sub + max_delta, 64);
    if (2 * (size_t)seg * ROWB + 1024 + 2 * (size_t)FC_BOX * ROWB > FC_SMEM_BUDGET) continue;
    p.sub = sub;
    p.seg_rows = seg;
    break;
  }
  if (!p.sub) return (int)cudaErrorInvalidValue;
  const size_t seg_bytes = (size_t)p.seg_rows * ROWB, box_bytes = (size_t)FC_BOX * ROWB;
  // a third segment stage for items made of several short units (the phase planes of a stride-2 forward: 4 / 2 / 2 / 1 taps per fetch),
  // as long as the weight ring keeps at least three boxes
  p.nsrc = 2;
  if (g_fc_tune[1] >= 3 && max_group_units > 1 && 3 * seg_bytes + 1024 + 3 * box_bytes <= FC_SMEM_BUDGET) p.nsrc = 3;
  const size_t fixed = p.nsrc * seg_bytes + 1024;
  long long wst = (long long)((FC_SMEM_BUDGET - fixed) / box_bytes);
  p.wst = (int)(wst > FC_WST_MAX ? FC_WST_MAX : wst);
  p.w_resident = (p.n_units == 1 && p.n_blocks == 1 && p.n_groups == 1 && max_chunks <= p.wst) ? 1 : 0;
  p.big_boxes = p.seg_rows / FC_BOX;
  p.tail_rows = p.seg_rows % FC_BOX;
  const size_t smem = fixed + (size_t)p.wst * FC_BOX * ROWB;
  CUtensorMap ms, mt, mw;
  int e = make_tmap_2d(&ms, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, src, src_rows, K, FC_BOX, ROWB / 2, ROWB);
  if (e) return e;
  e = make_tmap_2d(&mt, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, src, src_rows, K, p.tail_rows ? p.tail_rows : 64, ROWB / 2, ROWB);
  if (e) return e;
  e = make_tmap_2d(&mw, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, wpk, w_rows, K, FC_BOX, ROWB / 2, ROWB);
  if (e) return e;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(flatconv_kernel<ROWB, N, EPI>, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  const long long MT = 128LL * p.sub;
  const long long total = ((p.rows + MT - 1) / MT) * p.n_blocks * p.n_groups;
  int grid = (int)(total < cvad_num_sms() ? total : cvad_num_sms());
  if (grid < total) grid -= grid % p.n_groups;           // the kernel's group rotation needs whole tiles per round
  flatconv_kernel<ROWB, N, EPI><<<grid, 384, smem, st>>>(ms, mt, mw, p, bias, out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

// `K` reduction channels (the gathered tensor's channel count), `Nout` output channels.  relu: the EPI_RELU epilogue (forward only).
int run_flat(const void* src, long long src_rows, int K, const void* wpk, int Nout, const float* bias, void* out, FcParams& p, cudaStream_t st,
             bool relu = false) {
  if (K % 32 || Nout % 32) return (int)cudaErrorInvalidValue;
  if (K >= 64 && K % 64) return (int)cudaErrorInvalidValue;
  const int rowb = K >= 64 ? 128 : 64;
  const int n = n_block_of(Nout);
  p.n_blocks = Nout / n;
  p.ld_out = Nout;
  const long long w_rows = 9LL * Nout;
  __nv_bfloat16* o = (__nv_bfloat16*)out;
#define CVAD_FC(R, NN) (relu ? launch_flatconv<R, NN, EPI_RELU>(src, src_rows, K, wpk, w_rows, p, bias, o, st)          \
                        : p.bw_raw   ? launch_flatconv<R, NN, EPI_BW>(src, src_rows, K, wpk, w_rows, p, bias, o, st)   \
                        : p.sum_mask ? launch_flatconv<R, NN, EPI_MASK>(src, src_rows, K, wpk, w_rows, p, bias, o, st) \
                                     : launch_flatconv<R, NN, EPI_PLAIN>(src, src_rows, K, wpk, w_rows, p, bias, o, st))
  if (rowb == 64) {
    if (n == 32) return CVAD_FC(64, 32);
    if (n == 64) return CVAD_FC(64, 64);
    if (n == 256) return CVAD_FC(64, 256);
    return CVAD_FC(64, 128);
  }
  if (n == 32) return CVAD_FC(128, 32);
  if (n == 64) return CVAD_FC(128, 64);
  if (n == 256) return CVAD_FC(128, 256);
  return CVAD_FC(128, 128);
#undef CVAD_FC
}

// packed tap order: stride 1 natural; stride 2 grouped by phase plane (kh&1, kw&1) so every unit's taps are contiguous rows
__host__ __device__ inline int packed_tap(int stride, int i) {
  const int s2[9] = {0, 2, 6, 8, 1, 7, 3, 5, 4};
  return stride == 2 ? s2[i] : i;
}
// index of the first packed tap of source plane pl and the number of taps in it: stride 1 has one plane holding all nine taps,
// stride 2 the four phase planes
inline void plane_taps(int stride, int pl, int& first, int& count) {
  static const int f[4] = {0, 4, 6, 8}, c[4] = {4, 2, 2, 1};
  first = stride == 2 ? f[pl] : 0;
  count = stride == 2 ? c[pl] : 9;
}

// Geometry of a 3x3 convolution with input (N, H, W): the output interior h x w, its padded-flat rows (N, h+2, w+2) and their pitch
// wrow, and the number of source planes in that geometry (stride 1: the padded input itself; stride 2: its four phase planes).
struct FlatGeom {
  int stride, h, w, wrow, planes;
  long long rows;
};
inline FlatGeom flat_geom(int N, int H, int W, int stride) {
  const int h = stride == 1 ? H : (H - 1) / 2 + 1, w = stride == 1 ? W : (W - 1) / 2 + 1;
  return {stride, h, w, w + 2, stride == 1 ? 1 : 4, (long long)N * (h + 2) * (w + 2)};
}

// The epilogue's (image, row, column) decode of its output row over the geometry g (ReLU output, fused statistics): the row index is
// decoded in 32 bits.
int set_pixel_decode(FcParams& p, const FlatGeom& g) {
  if (g.rows > 0x7fffffffLL) return (int)cudaErrorInvalidValue;
  p.st_h = g.h;
  p.st_w = g.w;
  fast_div_init((unsigned)((g.h + 2) * (g.w + 2)), p.st_mul_img, p.st_shr_img);
  fast_div_init((unsigned)(g.w + 2), p.st_mul_row, p.st_shr_row);
  return 0;
}

// Appends the units of one work item that reads source planes pl0 .. pl0+n-1: one unit per K slab, walking the packed taps of those
// planes in order, the taps of plane pl0+a accumulating into set a.  Tap (kh, kw) lies shift = (kh/stride)*wrow + kw/stride rows into
// its plane.  The forward reads it at +shift from the segment start (row_off: one row and column before the output for stride 1, the
// plane's offset in the stacked phase planes for stride 2); the data-gradient, the transposed sum, at shift(2,2) - shift.
// group >= 0: the units form that group of p, whose set a writes output plane pl0+a.
void add_units(FcParams& p, const FlatGeom& g, bool dgrad, int slab, int nslab, int nblk, int pl0, int n, int group) {
  auto shift = [&](int t) { return t / 3 / g.stride * g.wrow + t % 3 / g.stride; };
  if (group >= 0) {
    p.n_groups = group + 1;
    p.acc_sets = n;
    p.group_unit0[group] = p.n_units;
    p.group_nunits[group] = nslab;
    for (int a = 0; a < n; ++a) p.group_plane[group][a] = pl0 + a;
  }
  for (int s = 0; s < nslab; ++s) {
    FcUnit& u = p.units[p.n_units++];
    u.row_off = dgrad || g.stride == 1 ? -(g.wrow + 1) : (int)(pl0 * g.rows);
    u.col = s * slab;
    for (int a = 0; a < n; ++a) {
      int first, count;
      plane_taps(g.stride, pl0 + a, first, count);
      if (a == 0) u.w_row0 = first * nblk;
      for (int i = 0; i < count; ++i, ++u.ntaps) {
        const int t = packed_tap(g.stride, first + i);
        u.tap_delta[u.ntaps] = dgrad ? shift(8) - shift(t) : shift(t);
        u.tap_acc[u.ntaps] = (unsigned char)a;
      }
    }
  }
}

// OIHW fp32 (Co, Ci, 3, 3) -> fwd [n-block][packed tap][N][Ci] bf16 (N = block of Co) and dgrad [n-block][packed tap][Nd][Co] (Nd = block of Ci)
__global__ void pack_w3x3_flat_kernel(const float* __restrict__ w, int Co, int Ci, int stride, int nf, int nd, __nv_bfloat16* __restrict__ wf,
                                      __nv_bfloat16* __restrict__ wd) {
  const int total = Co * Ci * 9;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ti = i % 9, ci = (i / 9) % Ci, co = i / (9 * Ci);
    const int tap = packed_tap(stride, ti);
    const __nv_bfloat16 v = __float2bfloat16(w[((long long)co * Ci + ci) * 9 + tap]);
    if (wf) wf[((long long)((co / nf) * 9 + ti) * nf + (co % nf)) * Ci + ci] = v;
    if (wd) wd[((long long)((ci / nd) * 9 + ti) * nd + (ci % nd)) * Co + co] = v;
  }
}

}  // namespace

// development hook: device buffer of 8 int64 per CTA (NULL switches the instrumentation off)
CVAD_API int cvad_flat_debug_buffer(long long* buf) {
  return (int)cudaMemcpyToSymbol(g_fc_debug, &buf, sizeof(buf));
}

CVAD_API int cvad_flat_dgrad_mode(int mode) {
  g_dgrad_mode = mode < 0 ? 0 : (mode > 2 ? 2 : mode);
  return 0;
}

CVAD_API int cvad_flat_tune(int key, int value) {
  if (key < 0 || key >= 4) return (int)cudaErrorInvalidValue;
  g_fc_tune[key] = value;
  return 0;
}

CVAD_API int cvad_flat_pack_w3x3_bf16(const float* w, int Cout, int Cin, int stride, void* w_fwd, void* w_dgrad, void* stream) {
  if (Cout % 32 || Cin % 32 || (stride != 1 && stride != 2)) return (int)cudaErrorInvalidValue;
  int total = Cout * Cin * 9;
  pack_w3x3_flat_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, Cout, Cin, stride, n_block_of(Cout), n_block_of(Cin),
                                                                               (__nv_bfloat16*)w_fwd, (__nv_bfloat16*)w_dgrad);
  CVAD_LAUNCH_CHECK();
  return 0;
}

namespace {
int flat_fwd(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin, int Cout, int stride, double* stats,
             int relu_phase, void* stream);
}

CVAD_API int cvad_flat_conv3x3_fwd_bf16(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                                        int stride, void* stream) {
  return flat_fwd(x, w_fwd, bias, y, N, H, W, Cin, Cout, stride, nullptr, -1, stream);
}

CVAD_API int cvad_flat_conv3x3_fwd_stats_bf16(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin,
                                              int Cout, int stride, double* stats, void* stream) {
  if (!stats || Cout != n_block_of(Cout)) return (int)cudaErrorInvalidValue;      // one output-channel block per CTA row tile
  return flat_fwd(x, w_fwd, bias, y, N, H, W, Cin, Cout, stride, stats, -1, stream);
}

CVAD_API int cvad_flat_conv3x3_fwd_relu_bf16(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin,
                                             int Cout, int stride, int phase_out, void* stream) {
  if (phase_out != 0 && phase_out != 1) return (int)cudaErrorInvalidValue;
  return flat_fwd(x, w_fwd, bias, y, N, H, W, Cin, Cout, stride, nullptr, phase_out, stream);
}

namespace {
// relu_phase: -1 = plain epilogue; 0 / 1 = EPI_RELU writing padded-flat / phase planes
int flat_fwd(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin, int Cout, int stride, double* stats,
             int relu_phase, void* stream) {
  if (stride != 1 && stride != 2) return (int)cudaErrorInvalidValue;
  const int slab = Cin >= 64 ? 64 : 32;
  const int nslab = Cin / slab;
  const FlatGeom g = flat_geom(N, H, W, stride);
  if (g.planes * nslab > FC_MAX_UNITS || (stride == 2 && 3 * g.rows > 0x7fffffffLL - (1 << 20))) return (int)cudaErrorInvalidValue;
  FcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = g.rows;
  for (int pl = 0; pl < g.planes; ++pl) add_units(p, g, false, slab, nslab, n_block_of(Cout), pl, 1, -1);
  if (stats || relu_phase >= 0) {
    if (int e = set_pixel_decode(p, g)) return e;
    p.st_out = stats;
  }
  if (relu_phase == 1) {                // the next stride-2 convolution's planes: (N, (st_h-1)/2+3, (st_w-1)/2+3) rows each
    p.planes = 1;
    p.plane_out_stride = (long long)N * ((p.st_h - 1) / 2 + 3) * ((p.st_w - 1) / 2 + 3);
  }
  return run_flat(x, g.planes * g.rows, Cin, w_fwd, Cout, bias, y, p, (cudaStream_t)stream, relu_phase >= 0);
}
}  // namespace

namespace {
struct BwStats {           // BatchNorm-backward reductions fused into the data-gradient epilogue (see FcParams::bw_raw)
  const void* raw;
  const float *gamma, *beta, *mean, *invstd;
  double* ws;
};

// raw is H x W; the rows of the launch live in the geometry g: the padded input itself (stride 1) or one phase plane (stride 2)
int set_bw(FcParams& p, const BwStats* bw, int H, int W, const FlatGeom& g) {
  if (!bw) return 0;
  p.bw_raw = (const __nv_bfloat16*)bw->raw;
  p.bw_gamma = bw->gamma; p.bw_beta = bw->beta; p.bw_mean = bw->mean; p.bw_invstd = bw->invstd;
  p.st_out = bw->ws;
  p.bw_H = H; p.bw_W = W; p.planes = g.stride == 2;
  return set_pixel_decode(p, g);
}

// sum_mask / sum_ws: the EPI_MASK column sums of dx (FcParams::sum_mask) into sum_ws[0..Cin)
int flat_dgrad(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout, int stride, const BwStats* bw,
               const void* sum_mask, double* sum_ws, void* stream) {
  // (N,H,W,Cin) is the convolution INPUT geometry.  stride 1: dy, dx padded-flat (N,H+2,W+2,.).  stride 2: dy padded-flat
  // (N,Ho+2,Wo+2,Cout), dx = four phase planes in that same geometry.
  if (stride != 1 && stride != 2) return (int)cudaErrorInvalidValue;
  const int slab = Cout >= 64 ? 64 : 32;
  const int nslab = Cout / slab;
  const int nblk = n_block_of(Cin);
  if (nslab > FC_MAX_UNITS) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  const FlatGeom g = flat_geom(N, H, W, stride);
  FcParams p;
  memset(&p, 0, sizeof(p));
  p.rows = g.rows;
  // (measured, profiles/r02c_conv_variants.md: the single fetch pays where the nine taps' weights stay resident in shared memory -- one
  // K slab, N = 32: 102 -> 92 us at 60x90 32->64 -- and loses where four accumulator sets shrink the work item to 128 rows and the weights
  // have to be streamed again for each of them: 70 -> 88 us at 30x45 64->128)
  const bool single_fetch = g_dgrad_mode == 2 && (g_fc_tune[2] ? true : (nslab == 1 && nblk == 32));
  if (stride == 1) {
    add_units(p, g, true, slab, nslab, nblk, 0, 1, -1);
  } else if (single_fetch && 2 * nslab <= FC_MAX_UNITS) {
    // One launch, and ONE fetch of each dy segment for all four phase planes of dx: a work item walks all nine taps (packed plane by
    // plane) and keeps one accumulator set per plane.  Four sets need 4 x N columns of TMEM per 128 rows: with N = 128 that is the whole
    // ring, so the planes are split into two groups of two sets whose packed taps are contiguous: {0,1} (4 + 2 taps), {2,3} (2 + 1).
    const int ngr = nblk >= 128 ? 2 : 1;
    p.plane_out_stride = g.rows;
    for (int gi = 0; gi < ngr; ++gi) add_units(p, g, true, slab, nslab, nblk, gi * (4 / ngr), 4 / ngr, gi);
  } else if (g_dgrad_mode >= 1 && 4 * nslab <= FC_MAX_UNITS) {
    // all four phase planes in one launch: plane pl is a set of work items with its own units (its 4 / 2 / 2 / 1 taps) and its own
    // output offset; one drain instead of four, but every plane fetches the dy segment again
    p.plane_out_stride = g.rows;
    for (int pl = 0; pl < 4; ++pl) add_units(p, g, true, slab, nslab, nblk, pl, 1, pl);
  } else {
    if (bw) return (int)cudaErrorNotSupported;      // the fused reductions need the one-launch form (plane index per work item)
    for (int pl = 0; pl < 4; ++pl) {
      memset(&p, 0, sizeof(p));
      p.rows = g.rows;
      p.out_row_base = pl * g.rows;
      p.sum_mask = (const uint32_t*)sum_mask;
      p.st_out = sum_ws;
      add_units(p, g, true, slab, nslab, nblk, pl, 1, -1);
      if (int e = run_flat(dy, g.rows, Cout, w_dgrad, Cin, nullptr, dx, p, st)) return e;
    }
    return 0;
  }
  if (int e = set_bw(p, bw, H, W, g)) return e;
  if (sum_mask) {
    p.sum_mask = (const uint32_t*)sum_mask;
    p.st_out = sum_ws;
  }
  return run_flat(dy, g.rows, Cout, w_dgrad, Cin, nullptr, dx, p, st);
}
}  // namespace

CVAD_API int cvad_flat_conv3x3_dgrad_bf16(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                                          void* stream) {
  return flat_dgrad(dy, w_dgrad, dx, N, H, W, Cin, Cout, stride, nullptr, nullptr, nullptr, stream);
}

CVAD_API int cvad_flat_conv3x3_dgrad_bnstats_bf16(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout,
                                                  int stride, const void* raw_in, const float* gamma, const float* beta, const float* mean,
                                                  const float* invstd, double* ws, void* stream) {
  if (!raw_in || !ws || Cin != n_block_of(Cin)) return (int)cudaErrorInvalidValue;
  BwStats bw = {raw_in, gamma, beta, mean, invstd, ws};
  return flat_dgrad(dy, w_dgrad, dx, N, H, W, Cin, Cout, stride, &bw, nullptr, nullptr, stream);
}

CVAD_API int cvad_flat_conv3x3_dgrad_masksum_bf16(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                                                  const void* mask, double* ws, void* stream) {
  if (!mask || !ws || Cin != n_block_of(Cin)) return (int)cudaErrorInvalidValue;
  return flat_dgrad(dy, w_dgrad, dx, N, H, W, Cin, Cout, stride, nullptr, mask, ws, stream);
}

// ================================================================================================ weight gradient
// dW[tap][ci][co] += sum_q  src[q + off_tap][ci] * dy[q][co]   over the flat pixel index q (dy has a ZERO border, so the
// junk positions contribute nothing).  Both operands are MN-major views of TMA-swizzled [pixel][channel] tiles (K = pixels):
//   A (M = 128): the activation segment, row-shifted per tap.  With 32 (64) input channels the four (two) 32- (64-) channel
//                atoms of the M dimension are consecutive PIXEL SHIFTS of the same tile (LBO = one pixel row), so one MMA
//                covers up to four (two) taps of a kernel row; with >= 128 channels the atoms are two channel slabs.
//   B (N = NB):  the dy tile.
// One accumulator [128 x NB] per tap group lives in TMEM for the CTA's whole pixel range; the epilogue adds it atomically
// into the OIHW fp32 gradient (a slice of the flat gradient arena).  A launch covers all tap groups (blockIdx.z = "variant":
// kernel row for wide layers, phase plane for stride 2) with ONE wave of CTAs, so the number of pixel chunks -- and with it
// the number of atomics, chunks x |dW| -- stays minimal.
namespace {

constexpr int WG_MAX_STAGES = 4;
bool g_wgrad_kh_stack = true;          // cvad_flat_wgrad_mode(0) selects the one-kernel-row-per-MMA form (A/B measurements)
// stride 2 with 32 / 64 input channels: the M atoms of an MMA are the PHASE PLANES at one pixel shift (9 taps in 4-5 MMAs per 16
// pixels) instead of pixel shifts inside one plane (6 MMAs); cvad_flat_tune(3, 0) restores the latter

struct WgGroup {
  int seg, delta;
  int atom_segs;         // 0: the M atoms are consecutive pixel shifts of one segment; k > 0: atom j is segment seg + j*k (phase planes)
  int tap[4];            // tap index of each M atom, -1 = unused lanes
};
struct WgVariant {
  int n_seg, n_groups;
  int seg_row_off[4];
  WgGroup groups[9];
};
struct WgParams {
  long long rows;        // flat pixels
  long long pix_per_cta; // multiple of qs
  int seg_rows, qs, n_stages, n_variants;
  int Cin, Cout, ci_blocks, co_blocks;
  int a_big, a_tail, b_box, max_seg;
  // KH-stacked mode (stride 1, 32/64 channels): the dy tile carries a halo of b_halo = W+2 rows on either side and the MMA's N is three
  // 32/64-channel atoms b_halo rows apart (kernel rows kh = 2, 1, 0), so one MMA covers a whole 3 x {kw} block of taps
  int b_rows, b_big, b_tail, b_halo;
  // optional staging buffer [tap][Cout][Cin] fp32 (zero on entry): the epilogue's atomics then run along Cin, i.e. along the lanes of a
  // warp (128 contiguous bytes per instruction instead of 32 addresses 36 bytes apart in the OIHW gradient); wgrad_fold_kernel adds it
  // into dw and re-zeroes it
  float* scratch;
  WgVariant v[4];
};

template <int ROWB_A, int ROWB_B, int NB, int A_SLABS, int KH>
__global__ void __launch_bounds__(256, 1) flatwgrad_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_at,
                                                           const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_bt,
                                                           const WgParams p, float* __restrict__ dw) {
  constexpr int B_SLABS = (NB * 2 + ROWB_B - 1) / ROWB_B;
  constexpr int NMMA = NB * KH;                            // the MMA's N: KH row-shifted copies of the NB-channel dy tile
  static_assert(KH == 1 || (KH == 3 && B_SLABS == 1 && NMMA <= 256), "KH stacking needs a single-slab dy tile");
  constexpr int LAY_A = ROWB_A == 128 ? UMMA_SW128 : UMMA_SW64;
  constexpr int LAY_B = ROWB_B == 128 ? UMMA_SW128 : UMMA_SW64;
  constexpr int AW = A_SLABS == 2 ? 128 : ROWB_A / 2;      // channels per M atom group that share a tap
  constexpr int CI_BLK = A_SLABS == 2 ? 128 : ROWB_A / 2;  // input channels handled by one CTA

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t bar_full[WG_MAX_STAGES], bar_empty[WG_MAX_STAGES], bar_done;
  __shared__ uint32_t tmem_base_sh;
  const WgVariant& var = p.v[blockIdx.z];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t seg1 = (uint32_t)p.seg_rows * ROWB_A;            // one slab of one segment
  const uint32_t a_bytes = (uint32_t)var.n_seg * A_SLABS * seg1;
  const uint32_t a_bytes_max = (uint32_t)p.max_seg * A_SLABS * seg1;
  const uint32_t b1 = (uint32_t)(KH == 3 ? p.b_rows : p.qs) * ROWB_B;
  const uint32_t stage_bytes = a_bytes_max + B_SLABS * b1;
  const uint32_t tx_bytes = a_bytes + B_SLABS * b1;

  const int tid = threadIdx.x, warp = uniform_warp_idx(), lane = tid & 31;
  const int qs = p.qs, n_stages = p.n_stages;
  const int cib = blockIdx.y / p.co_blocks, cob = blockIdx.y % p.co_blocks;
  const long long p_begin = (long long)blockIdx.x * p.pix_per_cta;
  long long p_end = p_begin + p.pix_per_cta;
  if (p_end > p.rows) p_end = p.rows;
  const int n_iter = p_begin < p_end ? (int)((p_end - p_begin + qs - 1) / qs) : 0;

  if (tid == 0) {
    for (int i = 0; i < WG_MAX_STAGES; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_done, 1);
    fence_barrier_init();
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_at);
    prefetch_tmap(&map_b);
  }
  if (warp == 2) tmem_alloc<512>(&tmem_base_sh);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_sh;

  if (warp == 0) {
    for (int it = 0; it < n_iter; ++it) {
      const int st = it % n_stages;
      mbar_wait(&bar_empty[st], ((it / n_stages) & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&bar_full[st], tx_bytes);
        const long long q = p_begin + (long long)it * qs;
        const uint32_t base = smem_base + st * stage_bytes;
        for (int sg = 0; sg < var.n_seg; ++sg)
          for (int sl = 0; sl < A_SLABS; ++sl) {
            const uint32_t dst = base + (sg * A_SLABS + sl) * seg1;
            const int r0 = (int)(q + var.seg_row_off[sg]), col = cib * CI_BLK + sl * 64;
            for (int b = 0; b < p.a_big; ++b) tma_load_2d(dst + b * (FC_BOX * ROWB_A), &map_a, col, r0 + b * FC_BOX, &bar_full[st]);
            if (p.a_tail) tma_load_2d(dst + p.a_big * (FC_BOX * ROWB_A), &map_at, col, r0 + p.a_big * FC_BOX, &bar_full[st]);
          }
        if (KH == 3) {                    // dy rows [q - halo, q - halo + b_rows): big boxes + one exact tail box
          const uint32_t dst = base + a_bytes_max;
          const int r0 = (int)q - p.b_halo;
          for (int b = 0; b < p.b_big; ++b) tma_load_2d(dst + b * (FC_BOX * ROWB_B), &map_b, cob * NB, r0 + b * FC_BOX, &bar_full[st]);
          if (p.b_tail) tma_load_2d(dst + p.b_big * (FC_BOX * ROWB_B), &map_bt, cob * NB, r0 + p.b_big * FC_BOX, &bar_full[st]);
        } else {
          for (int sl = 0; sl < B_SLABS; ++sl) {
            const uint32_t dst = base + a_bytes_max + sl * b1;
            for (int r = 0; r < qs; r += p.b_box) tma_load_2d(dst + r * ROWB_B, &map_b, cob * NB + sl * 64, (int)q + r, &bar_full[st]);
          }
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_bf16(128, NMMA, 1, 1);
    const uint32_t lbo_a = A_SLABS == 2 ? seg1 : ROWB_A;
    const uint64_t da_hi_shift = make_smem_desc(0, lbo_a, 8 * ROWB_A, LAY_A);
    // KH == 3: the N atoms are the same channels b_halo pixel rows apart (atom i = dy[q + (i-1)*halo] <-> kernel row kh = 2 - i)
    const uint64_t db_hi = make_smem_desc(0, KH == 3 ? (uint32_t)p.b_halo * ROWB_B : b1, 8 * ROWB_B, LAY_B);
    const int n_groups = var.n_groups;
    const int ksteps = qs / 16;
    for (int it = 0; it < n_iter; ++it) {
      const int st = it % n_stages;
      mbar_wait(&bar_full[st], (it / n_stages) & 1);
      tc_fence_after();
      const uint32_t base = smem_base + st * stage_bytes;
      if (elect_one()) {
        for (int g = 0; g < n_groups; ++g) {
          const uint32_t a0 = base + var.groups[g].seg * A_SLABS * seg1 + (uint32_t)var.groups[g].delta * ROWB_A;
          const uint32_t tacc = tmem_base + g * NMMA;
          const uint64_t da_hi = var.groups[g].atom_segs
                                     ? make_smem_desc(0, (uint32_t)var.groups[g].atom_segs * A_SLABS * seg1, 8 * ROWB_A, LAY_A)
                                     : da_hi_shift;
          for (int k = 0; k < ksteps; ++k) {
            const uint64_t da = da_hi | (uint64_t)(((a0 + k * 16 * ROWB_A) >> 4) & 0x3FFF);
            const uint64_t db = db_hi | (uint64_t)(((base + a_bytes_max + k * 16 * ROWB_B) >> 4) & 0x3FFF);
            tc_mma_f16(tacc, da, db, idesc, (it | k) != 0);
          }
        }
        tc_commit(&bar_empty[st]);
      }
      __syncwarp();
    }
    if (elect_one()) tc_commit(&bar_done);
    __syncwarp();
  }
  __syncwarp();
  if (n_iter > 0) {
    mbar_wait(&bar_done, 0);
    tc_fence_after();
    const int lq = warp & 3, half = warp >> 2;
    const int m = lq * 32 + lane;
    const int j = m / AW;
    const int ci = cib * CI_BLK + (m % AW);
    const uint32_t tlane = tmem_base + ((uint32_t)(lq * 32) << 16);
    for (int g = 0; g < var.n_groups; ++g) {
      const int tap0 = var.groups[g].tap[j];           // KH == 3: the kw of this M atom (the kernel row comes from the N atom)
#pragma unroll
      for (int c0 = 0; c0 < NMMA; c0 += 16) {
        if ((((c0 >> 4) + g) & 1) != half) continue;
        uint32_t v[16];
        tmem_ld16(tlane + g * NMMA + c0, v);
        tmem_ld_wait();
        if (tap0 >= 0 && ci < p.Cin) {
          const int tap = KH == 3 ? (2 - c0 / NB) * 3 + tap0 : tap0;
          if (p.scratch) {
            float* dst = p.scratch + ((long long)tap * p.Cout + cob * NB + (c0 % NB)) * p.Cin + ci;
#pragma unroll
            for (int i = 0; i < 16; ++i) atomicAdd(dst + (long long)i * p.Cin, __uint_as_float(v[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int co = cob * NB + (c0 % NB) + i;
              atomicAdd(dw + ((long long)co * p.Cin + ci) * 9 + tap, __uint_as_float(v[i]));
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// dw (OIHW) += scratch ([tap][Cout][Cin]); scratch = 0.  w (OIHW fp32, optional; Cin <= 256): also t[ci] += sum_{co,tap} bf16(w) * scratch,
// i.e. sum W*dW of this call's weight gradient with the weights the data-gradient multiplies by.  For every input channel that equals
// sum act*dconv over the convolution's input buffer (dconv = d/d act, zero padding and phase planes included): the BatchNorm backward of the
// layer below takes its T from here.  One element per thread in dw's order; the products gather in shared memory (a block's 256 elements
// touch ~30 input channels) and each touched channel costs one fp64 atomic per block.
__global__ void __launch_bounds__(256) wgrad_fold_kernel(float* __restrict__ scratch, float* __restrict__ dw, int Cin, int Cout,
                                                         const float* __restrict__ w, double* __restrict__ t) {
  __shared__ float s_t[256];
  if (w) {
    for (int c = threadIdx.x; c < Cin; c += blockDim.x) s_t[c] = 0.f;
    __syncthreads();
  }
  const int total = Cout * Cin * 9;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int tap = i % 9, ci = (i / 9) % Cin, co = i / (9 * Cin);
    float* s = scratch + ((long long)tap * Cout + co) * Cin + ci;
    const float v = *s;
    dw[i] += v;
    *s = 0.f;
    if (w) atomicAdd(&s_t[ci], __bfloat162float(__float2bfloat16(w[i])) * v);
  }
  if (!w) return;
  __syncthreads();
  for (int c = threadIdx.x; c < Cin; c += blockDim.x)
    if (s_t[c] != 0.f) atomicAdd(t + c, (double)s_t[c]);
}

template <int ROWB_A, int ROWB_B, int NB, int A_SLABS, int KH>
int launch_wgrad(const void* src, long long src_rows, const void* dy, WgParams& p, float* dw, cudaStream_t st) {
  constexpr int B_SLABS = (NB * 2 + ROWB_B - 1) / ROWB_B;
  constexpr int NMMA = NB * KH;
  constexpr int CI_BLK = A_SLABS == 2 ? 128 : ROWB_A / 2;
  p.ci_blocks = (p.Cin + CI_BLK - 1) / CI_BLK;
  p.co_blocks = p.Cout / NB;
  int max_delta = 0;
  p.max_seg = 0;
  for (int v = 0; v < p.n_variants; ++v) {
    if (p.v[v].n_groups * NMMA > 512) return (int)cudaErrorInvalidValue;
    p.max_seg = p.v[v].n_seg > p.max_seg ? p.v[v].n_seg : p.max_seg;
    for (int g = 0; g < p.v[v].n_groups; ++g) max_delta = p.v[v].groups[g].delta > max_delta ? p.v[v].groups[g].delta : max_delta;
  }
  const int shifts = A_SLABS == 2 ? 0 : (128 / CI_BLK - 1);   // extra rows touched by the pixel-shift atoms
  // stage size: largest qs in {512, 256, 128, 64} that leaves room for >= 2 stages
  int qs = 512;
  size_t stage = 0;
  for (;; qs >>= 1) {
    p.seg_rows = round_up(qs + max_delta + shifts, 32);
    p.b_rows = KH == 3 ? round_up(qs + 2 * p.b_halo, 32) : qs;
    stage = (size_t)p.max_seg * A_SLABS * p.seg_rows * ROWB_A + (size_t)B_SLABS * p.b_rows * ROWB_B;
    if (2 * stage + 1024 <= FC_SMEM_BUDGET || qs == 64) break;
  }
  if (2 * stage + 1024 > FC_SMEM_BUDGET) return (int)cudaErrorInvalidValue;
  p.qs = qs;
  p.n_stages = (int)((FC_SMEM_BUDGET - 1024) / stage);
  if (p.n_stages > WG_MAX_STAGES) p.n_stages = WG_MAX_STAGES;
  p.a_big = p.seg_rows / FC_BOX;
  p.a_tail = p.seg_rows % FC_BOX;
  p.b_box = qs < FC_BOX ? qs : FC_BOX;
  p.b_big = p.b_rows / FC_BOX;
  p.b_tail = p.b_rows % FC_BOX;
  const size_t smem = p.n_stages * stage + 1024;
  const int yz = p.ci_blocks * p.co_blocks * p.n_variants;
  long long chunks = cvad_num_sms() / yz;                         // one wave of CTAs
  const long long max_chunks = (p.rows + qs - 1) / qs;
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  p.pix_per_cta = ((p.rows + chunks - 1) / chunks + qs - 1) / qs * qs;
  chunks = (p.rows + p.pix_per_cta - 1) / p.pix_per_cta;
  CUtensorMap ma, mat, mb;
  int e = make_tmap_2d(&ma, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, src, src_rows, p.Cin, FC_BOX, ROWB_A / 2, ROWB_A);
  if (e) return e;
  e = make_tmap_2d(&mat, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, src, src_rows, p.Cin, p.a_tail ? p.a_tail : 32, ROWB_A / 2, ROWB_A);
  if (e) return e;
  CUtensorMap mbt;
  e = make_tmap_2d(&mb, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dy, p.rows, p.Cout, KH == 3 ? FC_BOX : p.b_box, ROWB_B / 2, ROWB_B);
  if (e) return e;
  e = make_tmap_2d(&mbt, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dy, p.rows, p.Cout, p.b_tail ? p.b_tail : 32, ROWB_B / 2, ROWB_B);
  if (e) return e;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(flatwgrad_kernel<ROWB_A, ROWB_B, NB, A_SLABS, KH>, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  flatwgrad_kernel<ROWB_A, ROWB_B, NB, A_SLABS, KH><<<dim3((unsigned)chunks, p.ci_blocks * p.co_blocks, p.n_variants), 256, smem, st>>>(ma, mat, mb, mbt, p, dw);
  CVAD_LAUNCH_CHECK();
  return 0;
}

int dispatch_wgrad(const void* src, long long src_rows, const void* dy, WgParams& p, float* dw, cudaStream_t st) {
  if (p.b_halo) {                       // KH-stacked: stride 1, 32->32 or 64->64
    if (p.Cin == 32 && p.Cout == 32) return launch_wgrad<64, 64, 32, 1, 3>(src, src_rows, dy, p, dw, st);
    if (p.Cin == 64 && p.Cout == 64) return launch_wgrad<128, 128, 64, 1, 3>(src, src_rows, dy, p, dw, st);
    return (int)cudaErrorInvalidValue;
  }
  if (p.Cin == 32 && p.Cout == 32) return launch_wgrad<64, 64, 32, 1, 1>(src, src_rows, dy, p, dw, st);
  if (p.Cin == 32 && p.Cout % 64 == 0) return launch_wgrad<64, 128, 64, 1, 1>(src, src_rows, dy, p, dw, st);
  if (p.Cin == 64 && p.Cout % 64 == 0) return launch_wgrad<128, 128, 64, 1, 1>(src, src_rows, dy, p, dw, st);
  if (p.Cin % 128 == 0 && p.Cout % 128 == 0) return launch_wgrad<128, 128, 128, 2, 1>(src, src_rows, dy, p, dw, st);
  return (int)cudaErrorInvalidValue;
}

}  // namespace

CVAD_API int cvad_flat_wgrad_mode(int kh_stack) {
  g_wgrad_kh_stack = kh_stack != 0;
  return 0;
}

namespace {
int flat_wgrad(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin, int Cout, int stride, void* stream);
}

CVAD_API int cvad_flat_conv3x3_wgrad_bf16(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin, int Cout, int stride,
                                          void* stream) {
  return flat_wgrad(x, dy, dw, nullptr, N, H, W, Cin, Cout, stride, stream);
}

namespace {
int wgrad_staged(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin, int Cout, int stride, const float* w,
                 double* t, void* stream) {
  if (!scratch) return (int)cudaErrorInvalidValue;
  int e = flat_wgrad(x, dy, dw, scratch, N, H, W, Cin, Cout, stride, stream);
  if (e) return e;
  const int total = Cout * Cin * 9;
  wgrad_fold_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(scratch, dw, Cin, Cout, w, t);
  CVAD_LAUNCH_CHECK();
  return 0;
}
}  // namespace

CVAD_API int cvad_flat_conv3x3_wgrad_staged_bf16(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin,
                                                 int Cout, int stride, void* stream) {
  return wgrad_staged(x, dy, dw, scratch, N, H, W, Cin, Cout, stride, nullptr, nullptr, stream);
}

CVAD_API int cvad_flat_conv3x3_wgrad_staged_wdot_bf16(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin,
                                                      int Cout, int stride, const float* w, double* ws, void* stream) {
  if (!w || !ws || Cin > 256) return (int)cudaErrorInvalidValue;
  return wgrad_staged(x, dy, dw, scratch, N, H, W, Cin, Cout, stride, w, ws + Cin, stream);
}

namespace {
int flat_wgrad(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin, int Cout, int stride, void* stream) {
  if (stride != 1 && stride != 2) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  const int apm = Cin == 32 ? 4 : (Cin == 64 ? 2 : 1);     // taps one MMA can cover through pixel-shift atoms
  const FlatGeom geo = flat_geom(N, H, W, stride);
  WgParams p;
  memset(&p, 0, sizeof(p));
  p.Cin = Cin; p.Cout = Cout;
  p.scratch = scratch;
  p.rows = geo.rows;
  if (stride == 1 && g_wgrad_kh_stack && ((Cin == 32 && Cout == 32) || (Cin == 64 && Cout == 64))) {
    // dW[kh][kw] = sum_q' x[q' + kw - 1] * dy[q' - (kh - 1)*Wp]: the kw taps are pixel-shift atoms of M (as below), the kh taps are
    // atoms of N one padded image row apart, so one M128 x N(3*Cout) MMA per 16 pixels covers a 3 x apm block of taps.  The operand
    // stream per 16 pixels drops from 3 x 5 KB to 7 KB (32 channels) and from 6 x 6 KB to 2 x 10 KB (64 channels).
    p.b_halo = geo.wrow;
    p.n_variants = 1;
    WgVariant& v = p.v[0];
    v.n_seg = 1;
    v.seg_row_off[0] = -1;
    for (int kw = 0; kw < 3; kw += apm) {
      WgGroup& g = v.groups[v.n_groups++];
      g.seg = 0;
      g.delta = kw;
      for (int j = 0; j < 4; ++j) g.tap[j] = (j < apm && kw + j < 3) ? kw + j : -1;
    }
    return dispatch_wgrad(x, p.rows, dy, p, dw, st);
  }
  if (stride == 1) {
    const int Wp = geo.wrow;
    // wide layers: one variant per kernel row keeps 3 accumulators of 128 columns in TMEM; narrow layers: all nine taps at once
    p.n_variants = apm == 1 ? 3 : 1;
    for (int l = 0; l < p.n_variants; ++l) {
      WgVariant& v = p.v[l];
      v.n_seg = 1;
      const int kh0 = apm == 1 ? l : 0, kh1 = apm == 1 ? l + 1 : 3;
      v.seg_row_off[0] = (kh0 - 1) * Wp - 1;
      for (int kh = kh0; kh < kh1; ++kh)
        for (int kw = 0; kw < 3; kw += apm) {
          WgGroup& g = v.groups[v.n_groups++];
          g.seg = 0;
          g.delta = (kh - kh0) * Wp + kw;
          for (int j = 0; j < 4; ++j) g.tap[j] = (j < apm && kw + j < 3) ? kh * 3 + kw + j : -1;
        }
    }
    return dispatch_wgrad(x, p.rows, dy, p, dw, st);
  }
  const int Wq = geo.wrow;
  if (3 * p.rows > 0x7fffffffLL - (1 << 20)) return (int)cudaErrorInvalidValue;
  if (apm > 1 && g_fc_tune[3] == 0) {
    // Narrow layers: all four planes are resident per stage anyway.  A tap (kh,kw) lives in plane (kh&1, kw&1) at pixel shift
    // (kh>>1, kw>>1); grouping by SHIFT makes the planes the atoms of M: shift (0,0) holds the four taps {0,1}x{0,1}, (0,1) and (1,0) two
    // each, (1,1) one -- 4 MMAs per 16 pixels at 32 channels (four atoms, LBO = one plane segment) and 5 at 64 channels (two atoms)
    // instead of 6, 9 of 16 (20) atom slots used instead of 9 of 24 (12 of 24).
    p.n_variants = 1;
    WgVariant& v = p.v[0];
    v.n_seg = 4;
    for (int pl = 0; pl < 4; ++pl) v.seg_row_off[pl] = (int)(pl * p.rows);
    auto add = [&](int seg0, int stride, int dh, int dw, int natoms) {
      WgGroup& g = v.groups[v.n_groups++];
      g.seg = seg0;
      g.delta = dh * Wq + dw;
      g.atom_segs = stride;
      for (int j = 0; j < 4; ++j) {
        g.tap[j] = -1;
        if (j >= natoms) continue;
        const int pl = seg0 + j * stride;
        if (pl > 3) continue;
        const int kh = 2 * dh + (pl >> 1), kw = 2 * dw + (pl & 1);
        if (kh < 3 && kw < 3) g.tap[j] = kh * 3 + kw;
      }
    };
    if (apm == 4) {
      for (int dh = 0; dh < 2; ++dh)
        for (int dw = 0; dw < 2; ++dw) add(0, 1, dh, dw, 4);
    } else {
      add(0, 1, 0, 0, 2); add(2, 1, 0, 0, 2);       // shift (0,0): planes {0,1}, {2,3}
      add(0, 2, 0, 1, 2);                           // shift (0,1): planes 0, 2 (kw = 2)
      add(0, 1, 1, 0, 2);                           // shift (1,0): planes 0, 1 (kh = 2)
      add(0, 1, 1, 1, 1);                           // shift (1,1): plane 0
    }
    return dispatch_wgrad(x, 4 * p.rows, dy, p, dw, st);
  }
  // per phase plane (a,b): taps with (kh&1, kw&1) = (a,b), shift (kh>>1)*Wq + (kw>>1); wide layers: one variant per plane
  p.n_variants = apm == 1 ? 4 : 1;
  for (int pl = 0; pl < 4; ++pl) {
    WgVariant& v = p.v[apm == 1 ? pl : 0];
    const int a = pl >> 1, b = pl & 1;
    const int sg = v.n_seg++;
    v.seg_row_off[sg] = (int)(pl * p.rows);
    for (int kh = a; kh < 3; kh += 2)
      for (int kw = b; kw < 3; kw += 2 * (apm > 1 ? 2 : 1)) {
        WgGroup& g = v.groups[v.n_groups++];
        g.seg = sg;
        g.delta = (kh >> 1) * Wq + (kw >> 1);
        for (int j = 0; j < 4; ++j) g.tap[j] = -1;
        g.tap[0] = kh * 3 + kw;
        if (apm > 1 && kw + 2 < 3) g.tap[1] = kh * 3 + kw + 2;      // the next same-parity tap is one plane pixel further
      }
  }
  return dispatch_wgrad(x, 4 * p.rows, dy, p, dw, st);
}
}  // namespace

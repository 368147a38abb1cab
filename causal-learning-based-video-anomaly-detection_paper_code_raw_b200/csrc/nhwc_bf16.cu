// Bandwidth kernels of the bf16 (tensor-core) M-A backbone path on the padded-flat / phase-plane layouts of flatconv_tc.cu:
//   bn_stats:  per-channel batch mean / biased variance (fp64 accumulation) + running-stat update (cad:131,136)
//   bn_apply:  y = relu((x-mean)*invstd*gamma+beta), bf16 -> bf16, zero border / phase planes for the next convolution
//   bn_bwd:    ReLU + BatchNorm backward (two passes: per-channel reductions, then dx), dgamma/dbeta accumulated in fp32; or one pass when the
//              reductions arrive from the convolution above (the "T" form, see pad_bn_relu_bwd_apply_kernel)
//   avgpool:   AdaptiveAvgPool2d((4,6)) (cad:126,155) bf16 -> fp32 features in the reference's (c,h,w) flatten order
// All loads/stores are 16-byte vectors over the channel axis (8 bf16), coalesced across threads.
#include "common.cuh"
#include "cvad_b200.h"

namespace {

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 v;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return v;
}

// ------------------------------------------------------------------------------------------------ adaptive average pool
// adaptive-pool bin bounds; 32-bit arithmetic (frame dimensions are far below 2^15: the 64-bit divisions these used to be cost the
// per-frame backward kernel more than its memory traffic)
__device__ __forceinline__ int bstart(int o, int in, int out) { return (int)(((unsigned)o * (unsigned)in) / (unsigned)out); }
__device__ __forceinline__ int bend(int o, int in, int out) { return (int)((((unsigned)(o + 1)) * (unsigned)in + (unsigned)out - 1u) / (unsigned)out); }

inline int blocks_for(long long n, int per = 256) {
  long long b = (n + per - 1) / per;
  long long cap = 16LL * cvad_num_sms();
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}


// ================================================================================================ padded-flat layout
// Activations of the flat tensor-core path (flatconv_tc.cu): (N, H+2, W+2, C) bf16 with a zero border, or -- for the
// input of a stride-2 convolution -- four phase planes P_ab[n][i][j] = padded(2(i-1)+a, 2(j-1)+b) in the geometry
// (N, Ho+2, Wo+2) of that convolution's output.  Convolution outputs (raw) and data-gradients (dact) carry junk in their
// border; every kernel below reads interiors only and writes complete buffers (zero borders where a consumer needs them).
struct PadGeo {
  int N, H, W, C;       // interior geometry of the raw / plain tensor
  int Hq, Wq;           // phase-plane geometry (Ho+2, Wo+2) when a phase layout is involved
  int lg;               // log2(C/8)
  unsigned mulW, shrW, mulH, shrH;     // x / W and x / H as umulhi(x, mul) >> shr for 0 <= x < 2^31 (mul = 0: divisor 1)
  // the same for H + 2, Hq and N: the row-walking kernels decode their row index with them (an emulated 32-bit division is ~25
  // instructions, and ncu counted 85-118 instructions per 16-byte vector in the apply kernels before these replaced four of them per row)
  unsigned mulHp, shrHp, mulHq, shrHq, mulN, shrN;
};


__device__ __forceinline__ long long plain_row(const PadGeo& g, int n, int hp, int wp) { return ((long long)n * (g.H + 2) + hp) * (g.W + 2) + wp; }
__device__ __forceinline__ long long phase_row(const PadGeo& g, int n, int hp, int wp) {
  const int pl = ((hp & 1) << 1) | (wp & 1);
  return (((long long)pl * g.N + n) * g.Hq + (hp >> 1) + 1) * g.Wq + (wp >> 1) + 1;
}

// relu(bn(raw)) -> act.  PHASE=0: plain padded act, zero border.  PHASE=1: four phase planes (zeros where no pixel maps).
// mask (optional): the ReLU gate as one bit per element in act's row layout -- byte k holds the 8 channels of act's 16-byte vector k (bit c of
// a pixel in 32-bit word c/32), 0 wherever act is zero by construction.  The data-gradient of the next convolution sums its output under
// it (the BatchNorm backward's sum g, cvad_flat_conv3x3_dgrad_masksum_bf16), 1/16 of the bytes of re-reading raw.
// Block = 256 threads, two 16-byte vectors per thread and pass (v = tid, tid + 256): every padded row of the backbone
// (368..448 vectors) is one pass with all loads issued before the first use.  PHASE=1 handles the two column-phase planes
// (a,0) and (a,1) of one plane row in the same block, so the raw row both of them sample is fetched from HBM once.
// FIN: the batch statistics are still the raw fp64 sums in fin.ws (left there by the convolution's epilogue): every thread finalises its own
// eight channels (common.cuh's BatchNorm helpers, as the separate finalize kernel, so the result is bit-identical), block 0 also publishes
// mean / invstd for the backward and updates the running statistics, and the last block past this prologue re-zeroes the sums -- one
// launch instead of two on the critical path of every layer.
struct BnFin {
  int reverse;            // walk the rows back to front (L2 reuse, see the kernel)
  double* ws;
  double count;
  float eps, momentum;
  float *mean_out, *invstd_out, *running_mean, *running_var;
  long long* nbt;
};
__device__ unsigned int g_bn_fold_ticket = 0u;

// after every thread of the block has consumed its ws values: the last block of the grid to get here zeroes ws[0, 2C)
__device__ __forceinline__ void bn_fold_release(double* ws, int C) {
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&g_bn_fold_ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last) {
    for (int j = threadIdx.x; j < 2 * C; j += blockDim.x) ws[j] = 0.0;
    if (threadIdx.x == 0) g_bn_fold_ticket = 0u;
  }
}

// Output positions are 32-bit vector indices (make_geo bounds the buffers): with 64-bit ones the mask store took the phase-plane form from
// 80 to 102 registers, i.e. from 3 to 2 resident CTAs per SM.
template <int PHASE, int R, bool FIN>
__global__ void __launch_bounds__(256) pad_bn_apply_relu_kernel(const __nv_bfloat16* __restrict__ raw, __nv_bfloat16* __restrict__ act,
                                                                uint8_t* __restrict__ mask, PadGeo g, const float* __restrict__ mean,
                                                                const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, BnFin fin) {
  const int groups = 1 << g.lg;
  const int cg = threadIdx.x & (groups - 1);
  float sc[8], sh[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cg * 8 + i;
    float mu, is;
    if (FIN) {
      const BnBatchStat s = bn_batch_stat(fin.ws, g.C, c, fin.count, nullptr);
      mu = (float)s.mean;
      is = bn_invstd(s, fin.eps);
    } else {
      mu = mean[c];
      is = invstd[c];
    }
    sc[i] = is * gamma[c];
    sh[i] = beta[c] - mu * sc[i];
  }
  if (FIN) {
    if (blockIdx.x == 0)
      for (int c = threadIdx.x; c < g.C; c += blockDim.x)
        bn_finalize_channel(fin.ws, g.C, c, fin.count, nullptr, fin.eps, fin.momentum, fin.mean_out, fin.invstd_out, fin.running_mean,
                            fin.running_var, fin.nbt);
    bn_fold_release(fin.ws, g.C);
  }
  const int Hp = g.H + 2, Wp = g.W + 2;
  const int items = PHASE ? 2 * g.N * g.Hq : g.N * Hp;          // PHASE: (a, n, i) with both b planes per item
  const int rowlen = (PHASE ? g.Wq : Wp) << g.lg;
  const int span = PHASE ? 2 * rowlen : rowlen;
  // R items (rows) per iteration: all their loads (2 per thread and row) are issued before the first is consumed, which keeps
  // 2R x 16 bytes per thread in flight -- with one row per iteration the kernel ran at 0.6 of the copy bandwidth, latency-bound
  for (int r0 = blockIdx.x * R; r0 < items; r0 += gridDim.x * R) {
    for (int v0 = threadIdx.x; v0 < span; v0 += 512) {
      uint4 x[R][2];
      bool in[R][2], ok[R][2];
      unsigned dst[R][2];
#pragma unroll
      for (int rr = 0; rr < R; ++rr) {
        // fin.reverse: rows are walked from the END of the tensor -- the convolution in front of this kernel wrote raw front to back, so
        // its last rows are what the 126 MB L2 still holds, and the convolution behind it starts reading act at the front, which this
        // kernel then wrote last
        const int r = fin.reverse ? items - 1 - (r0 + rr) : r0 + rr;
        int n = 0, hp = -1, a = 0;
        unsigned row0 = 0, row1 = 0;                              // first vector of the output row(s)
        if (r >= 0 && r < items) {
          if (PHASE) {
            const int t = fast_div(r, g.mulHq, g.shrHq);
            const int i = r - t * g.Hq;
            a = fast_div(t, g.mulN, g.shrN);
            n = t - a * g.N;
            hp = 2 * (i - 1) + a;
            row0 = (((unsigned)(2 * a) * g.N + n) * g.Hq + i) * rowlen;
            row1 = (((unsigned)(2 * a + 1) * g.N + n) * g.Hq + i) * rowlen;
          } else {
            n = fast_div(r, g.mulHp, g.shrHp);
            hp = r - n * Hp;
            row0 = (unsigned)r * rowlen;
          }
        }
        const bool row_ok = hp >= 1 && hp <= g.H;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int v = v0 + u * 256;
          in[rr][u] = v < span && r >= 0 && r < items;
          const int b = PHASE && v >= rowlen ? 1 : 0;
          const int vv = v - b * rowlen;
          const int j = vv >> g.lg;
          const int wp = PHASE ? 2 * (j - 1) + b : j;
          ok[rr][u] = in[rr][u] && row_ok && wp >= 1 && wp <= g.W;
          dst[rr][u] = (b ? row1 : row0) + vv;
          if (ok[rr][u]) x[rr][u] = __ldg(reinterpret_cast<const uint4*>(raw) + ((plain_row(g, n, hp, wp) << g.lg) + cg));
        }
      }
#pragma unroll
      for (int rr = 0; rr < R; ++rr)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (!in[rr][u]) continue;
          uint4 o = make_uint4(0, 0, 0, 0);
          unsigned bits = 0u;
          if (ok[rr][u]) {
            float f[8];
            unpack8(x[rr][u], f);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float y = fmaf(f[i], sc[i], sh[i]);
              bits |= (y > 0.f ? 1u : 0u) << i;
              f[i] = fmaxf(y, 0.f);
            }
            o = pack8(f);
          }
          reinterpret_cast<uint4*>(act)[dst[rr][u]] = o;
          if (mask) mask[dst[rr][u]] = (uint8_t)bits;
        }
    }
  }
}

constexpr int PAD_REP = 16, PAD_REP_MAXC = 512;
__device__ double g_pad_rep[PAD_REP * 2 * PAD_REP_MAXC];      // zero-initialised; every launch leaves it zero again
__device__ unsigned int g_pad_ticket = 0u;

// per-channel reductions over the INTERIOR of raw.  !BWD: sum x, sum x^2.  BWD: g = dact*(pre>0): sum g, sum g*xhat.
// dact is plain (PHASE=0) or phase planes (PHASE=1).
template <bool BWD, int PHASE>
__global__ void __launch_bounds__(256, 3) pad_reduce_kernel(const __nv_bfloat16* __restrict__ raw, const __nv_bfloat16* __restrict__ dact, PadGeo g,
                                                            const float* __restrict__ mean, const float* __restrict__ invstd,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            double* __restrict__ ws) {
  extern __shared__ float red[];             // [blockDim][16]
  const int groups = 1 << g.lg;
  const int cg = threadIdx.x & (groups - 1), slot = threadIdx.x >> g.lg, slots = blockDim.x >> g.lg;
  const int C = g.C;
  // BWD: the ReLU gate is (x*a + b > 0) with a = gamma*invstd, b = beta - mean*a; the sums are taken over g and g*x and turned into
  // sum g*xhat = invstd * (sum g*x - mean * sum g) in the fp64 combine below (half the per-thread state of carrying xhat).
  float s[8], q[8], ga[8], gb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    s[i] = 0.f; q[i] = 0.f;
    if (BWD) {
      ga[i] = gamma[cg * 8 + i] * invstd[cg * 8 + i];
      gb[i] = beta[cg * 8 + i] - mean[cg * 8 + i] * ga[i];
    }
  }
  // Interior pixels as one flat index space p = (n*H + h)*W + w, strided over the block's pixel slots; four independent
  // 16-byte loads are in flight per thread before any is consumed.
  const int P = g.N * g.H * g.W;               // < 2^31 (checked by the launcher)
  const int chunk = (P + gridDim.x - 1) / gridDim.x;
  const int p_end = min(P, (int)(blockIdx.x + 1) * chunk);
  constexpr int U = 4;               // 16-byte loads in flight per thread and tensor (the backward reads two tensors: 8 loads)
  for (int p0 = blockIdx.x * chunk + slot; p0 < p_end; p0 += U * slots) {
    uint4 xv[U], dv[U];
    bool ok[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int pp = p0 + u * slots;
      ok[u] = pp < p_end;
      if (ok[u]) {
        const int t = fast_div(pp, g.mulW, g.shrW);
        const int w = pp - t * g.W;
        const int n = fast_div(t, g.mulH, g.shrH);
        const int h = t - n * g.H;
        const long long row = plain_row(g, n, h + 1, w + 1);
        xv[u] = __ldg(reinterpret_cast<const uint4*>(raw) + ((row << g.lg) + cg));
        if (BWD) {
          const long long drow = PHASE ? phase_row(g, n, h + 1, w + 1) : row;
          dv[u] = __ldg(reinterpret_cast<const uint4*>(dact) + ((drow << g.lg) + cg));
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!ok[u]) continue;
      float f[8];
      unpack8(xv[u], f);
      if (!BWD) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { s[i] += f[i]; q[i] = fmaf(f[i], f[i], q[i]); }
      } else {
        float d[8];
        unpack8(dv[u], d);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float gg = fmaf(f[i], ga[i], gb[i]) > 0.f ? d[i] : 0.f;
          s[i] += gg;
          q[i] = fmaf(gg, f[i], q[i]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) { red[threadIdx.x * 16 + i] = s[i]; red[threadIdx.x * 16 + 8 + i] = q[i]; }
  __syncthreads();
  // Cross-CTA combine.  Hundreds of CTAs adding into the same 2*C addresses serialise in the L2 atomic unit: each CTA adds into one
  // of PAD_REP replicas instead, and the last CTA to finish (ticket counter) folds the replicas into ws and re-zeroes them.  Calls
  // are stream-ordered (as for ws itself), so one scratch suffices.
  const bool replicated = C <= PAD_REP_MAXC;
  double* dst = replicated ? g_pad_rep + (size_t)(blockIdx.x & (PAD_REP - 1)) * (2 * PAD_REP_MAXC) : ws;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g2 = c >> 3, i = c & 7;
    double a0 = 0.0, a1 = 0.0;
    for (int r = 0; r < slots; ++r) {
      a0 += (double)red[(r * groups + g2) * 16 + i];
      a1 += (double)red[(r * groups + g2) * 16 + 8 + i];
    }
    if (BWD) a1 = (a1 - (double)mean[c] * a0) * (double)invstd[c];
    atomicAdd(dst + c, a0);
    atomicAdd(dst + C + c, a1);
  }
  if (!replicated) return;
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&g_pad_ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  for (int j = threadIdx.x; j < 2 * C; j += blockDim.x) {
    double acc = 0.0;
#pragma unroll
    for (int r = 0; r < PAD_REP; ++r) {
      double* p = g_pad_rep + (size_t)r * (2 * PAD_REP_MAXC) + j;
      acc += __ldcg(p);
      __stcg(p, 0.0);
    }
    ws[j] += acc;
  }
  if (threadIdx.x == 0) g_pad_ticket = 0u;
}

// ReLU + BatchNorm backward: draw (plain padded, ZERO border) from raw and dact (plain or phase planes)
// FOLD: block 0 also adds the two sums into dgamma / dbeta and the last block past the prologue re-zeroes ws (the parameter-update kernel's
// work): no third launch.
// OCC: resident CTAs per SM the register allocation is held to (98 registers = 2 CTAs when left alone; 3 CTAs cost ~20 spilled registers)
// TS: no reduce pass in front.  ws[0, C) holds S1 = sum g (the masked-sum epilogue of the data-gradient above) and ws[C, 2C) holds
// T = sum act*dact (from the weight gradient above: sum W*dW, cvad_flat_conv3x3_wgrad_staged_wdot_bf16).  Since act = relu(gamma*xhat + beta),
// gamma * sum g*xhat = T - beta*S1, which is all the apply needs (no division by gamma).  dgamma / dbeta keep their definition: each thread
// keeps its channel group, sums g and g*x in registers, and the block adds sum g and sum g*xhat into g_bn_tsum (the layout of a BatchNorm
// workspace); the last block past the prologue re-zeroes ws, and the parameter-update launch behind the kernel consumes and re-zeroes
// g_bn_tsum.
__device__ double g_bn_tsum[2 * 256];      // zero-initialised; every TS backward leaves it zero again (stream-ordered, as ws)

template <int PHASE, int R, bool FOLD, int OCC, bool TS = false>
__global__ void __launch_bounds__(256, OCC) pad_bn_relu_bwd_apply_kernel(const __nv_bfloat16* __restrict__ raw, const __nv_bfloat16* __restrict__ dact,
                                                                    __nv_bfloat16* __restrict__ draw, PadGeo g, const float* __restrict__ mean,
                                                                    const float* __restrict__ invstd, const float* __restrict__ gamma,
                                                                    const float* __restrict__ beta, double* __restrict__ ws, double count,
                                                                    int training, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int groups = 1 << g.lg;
  const int cg = threadIdx.x & (groups - 1);
  // With a = gamma*invstd, b = beta - mean*a (the forward's scale/shift), g = dact*(x*a + b > 0), mg = mean(g), mgx = mean(g*xhat):
  //   draw = a*(g - mg - xhat*mgx) = a*g - k0 - k1*x,   k1 = a*mgx*invstd,  k0 = a*mg - k1*mean     (eval mode: k0 = k1 = 0)
  float ca[8], cb[8], k0[8], k1[8], sg[8], sgx[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cg * 8 + i;
    const float is = invstd[c], mu = mean[c];
    ca[i] = gamma[c] * is;
    cb[i] = beta[c] - mu * ca[i];
    const float mg = training ? (float)(ws[c] / count) : 0.f;
    if (TS) {
      const float gmgx = training ? (float)((ws[g.C + c] - (double)beta[c] * ws[c]) / count) : 0.f;     // gamma * mean(g*xhat)
      k1[i] = gmgx * is * is;
    } else {
      const float mgx = training ? (float)(ws[g.C + c] / count) : 0.f;
      k1[i] = ca[i] * mgx * is;
    }
    k0[i] = ca[i] * mg - k1[i] * mu;
    sg[i] = 0.f;
    sgx[i] = 0.f;
  }
  if (TS) bn_fold_release(ws, g.C);
  if (FOLD) {
    if (blockIdx.x == 0)
      for (int c = threadIdx.x; c < g.C; c += blockDim.x) bn_params_channel(ws, g.C, c, dgamma, dbeta);
    bn_fold_release(ws, g.C);
  }
  const int Hp = g.H + 2, Wp = g.W + 2;
  const int rows = g.N * Hp, rowlen = Wp << g.lg;
  // R rows per iteration, every load (2 tensors x 2 vectors x R rows per thread) issued before the first use
  for (int r0 = blockIdx.x * R; r0 < rows; r0 += gridDim.x * R) {
    for (int v0 = threadIdx.x; v0 < rowlen; v0 += 512) {
      uint4 x[R][2], dd[R][2];
      bool in[R][2], ok[R][2];
#pragma unroll
      for (int rr = 0; rr < R; ++rr) {
        const int r = r0 + rr;
        const int n = fast_div(r, g.mulHp, g.shrHp), hp = r - n * Hp;
        const bool row_ok = r < rows && hp >= 1 && hp <= g.H;
        const long long vbase = (long long)r * rowlen;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int v = v0 + u * 256;
          const int wp = v >> g.lg;
          in[rr][u] = v < rowlen && r < rows;
          ok[rr][u] = in[rr][u] && row_ok && wp >= 1 && wp <= g.W;
          if (ok[rr][u]) {
            x[rr][u] = __ldg(reinterpret_cast<const uint4*>(raw) + vbase + v);
            const long long dv = PHASE ? ((phase_row(g, n, hp, wp) << g.lg) + cg) : vbase + v;
            dd[rr][u] = __ldg(reinterpret_cast<const uint4*>(dact) + dv);
          }
        }
      }
#pragma unroll
      for (int rr = 0; rr < R; ++rr)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (!in[rr][u]) continue;
          uint4 o = make_uint4(0, 0, 0, 0);
          if (ok[rr][u]) {
            float f[8], d[8];
            unpack8(x[rr][u], f);
            unpack8(dd[rr][u], d);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float gg = fmaf(f[i], ca[i], cb[i]) > 0.f ? d[i] : 0.f;
              if (TS) {
                sg[i] += gg;
                sgx[i] = fmaf(gg, f[i], sgx[i]);
              }
              f[i] = fmaf(-k1[i], f[i], fmaf(ca[i], gg, -k0[i]));
            }
            o = pack8(f);
          }
          reinterpret_cast<uint4*>(draw)[(long long)(r0 + rr) * rowlen + v0 + u * 256] = o;
        }
    }
  }
  if (TS) {      // block sums per channel (as pad_reduce_kernel: fp32 per thread, fp64 across the block's slots), then one atomic per channel
    __shared__ float red[TS ? 256 * 16 : 1];
#pragma unroll
    for (int i = 0; i < 8; ++i) { red[threadIdx.x * 16 + i] = sg[i]; red[threadIdx.x * 16 + 8 + i] = sgx[i]; }
    __syncthreads();
    const int slots = blockDim.x >> g.lg;
    for (int c = threadIdx.x; c < g.C; c += blockDim.x) {
      const int g2 = c >> 3, i = c & 7;
      double a0 = 0.0, a1 = 0.0;
      for (int r = 0; r < slots; ++r) {
        a0 += (double)red[(r * groups + g2) * 16 + i];
        a1 += (double)red[(r * groups + g2) * 16 + 8 + i];
      }
      atomicAdd(g_bn_tsum + c, a0);
      atomicAdd(g_bn_tsum + g.C + c, (a1 - (double)mean[c] * a0) * (double)invstd[c]);
    }
  }
}

// AdaptiveAvgPool2d on a padded-flat input; out (N, C, OH, OW) fp32.  One thread = one output bin x 8 channels: 16-byte loads
// over the bin, eight strided fp32 stores (the reference's (c,h,w) flatten order, cad:155).
__global__ void avgpool_pad_fwd_kernel(const __nv_bfloat16* __restrict__ x, int N, int H, int W, int C, int OH, int OW, float* __restrict__ out) {
  const int groups = C >> 3;
  const long long total = (long long)N * OH * OW * groups;
  const int Wp = W + 2, Hp = H + 2;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(t % groups);
    long long r = t / groups;
    const int ow = (int)(r % OW); r /= OW;
    const int oh = (int)(r % OH);
    const int n = (int)(r / OH);
    const int h0 = bstart(oh, H, OH), h1 = bend(oh, H, OH), w0 = bstart(ow, W, OW), w1 = bend(ow, W, OW);
    float s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = 0.f;
    for (int h = h0; h < h1; ++h)
      for (int w = w0; w < w1; ++w) {
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(x) + (((long long)n * Hp + h + 1) * Wp + w + 1) * groups + cg), f);
#pragma unroll
        for (int i = 0; i < 8; ++i) s[i] += f[i];
      }
    const float inv = 1.f / (float)((h1 - h0) * (w1 - w0));
#pragma unroll
    for (int i = 0; i < 8; ++i) out[(((long long)n * C + cg * 8 + i) * OH + oh) * OW + ow] = s[i] * inv;
  }
}
// The same, one block per frame: the (C, OH, OW) outputs of a frame are contiguous in the result, so they are collected in shared memory
// ([bin][channel], pitch C + 4) and written as one coalesced run -- the kernel above writes eight 4-byte values 4*OH*OW bytes apart per
// thread (one 32-byte sector per value: 31 -> 12 us at 512 x 8x12x256).
__global__ void avgpool_pad_fwd_frame_kernel(const __nv_bfloat16* __restrict__ x, int N, int H, int W, int C, int OH, int OW,
                                             float* __restrict__ out) {
  extern __shared__ __align__(16) float sp[];             // [OH*OW][C + 4]
  const int bins = OH * OW, groups = C >> 3, Wp = W + 2, Hp = H + 2, pitch = C + 4;
  for (int n = blockIdx.x; n < N; n += gridDim.x) {
    for (int t = threadIdx.x; t < bins * groups; t += blockDim.x) {
      const int cg = t % groups, b = t / groups;
      const int oh = b / OW, ow = b - oh * OW;
      const int h0 = bstart(oh, H, OH), h1 = bend(oh, H, OH), w0 = bstart(ow, W, OW), w1 = bend(ow, W, OW);
      float s[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] = 0.f;
      for (int h = h0; h < h1; ++h)
        for (int w = w0; w < w1; ++w) {
          float f[8];
          unpack8(__ldg(reinterpret_cast<const uint4*>(x) + (((long long)n * Hp + h + 1) * Wp + w + 1) * groups + cg), f);
#pragma unroll
          for (int i = 0; i < 8; ++i) s[i] += f[i];
        }
      const float inv = 1.f / (float)((h1 - h0) * (w1 - w0));
      float4* d = reinterpret_cast<float4*>(sp + b * pitch + cg * 8);
      d[0] = make_float4(s[0] * inv, s[1] * inv, s[2] * inv, s[3] * inv);
      d[1] = make_float4(s[4] * inv, s[5] * inv, s[6] * inv, s[7] * inv);
    }
    __syncthreads();
    float* dst = out + (long long)n * C * bins;
    for (int i = threadIdx.x; i < C * bins; i += blockDim.x) {
      const int c = i / bins, b = i - c * bins;
      dst[i] = sp[b * pitch + c];
    }
    __syncthreads();
  }
}

// dout (N,C,OH,OW) fp32 -> dx padded-flat bf16 (interior only; the border is never read).  One thread = one pixel x 8 channels;
// a pixel lies in at most a 3x3 neighbourhood of (possibly overlapping) adaptive bins.
__global__ void avgpool_pad_bwd_kernel(const float* __restrict__ dout, int N, int H, int W, int C, int OH, int OW,
                                       __nv_bfloat16* __restrict__ dx) {
  const int groups = C >> 3;
  const long long total = (long long)N * H * W * groups;
  const int Wp = W + 2, Hp = H + 2;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(t % groups);
    long long r = t / groups;
    const int w = (int)(r % W); r /= W;
    const int h = (int)(r % H);
    const int n = (int)(r / H);
    float s[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) s[i] = 0.f;
    const int ohc = (h * OH) / H, owc = (w * OW) / W;
    for (int oh = max(0, ohc - 1); oh <= min(OH - 1, ((h + 1) * OH) / H + 1); ++oh) {
      const int h0 = bstart(oh, H, OH), h1 = bend(oh, H, OH);
      if (h < h0 || h >= h1) continue;
      for (int ow = max(0, owc - 1); ow <= min(OW - 1, ((w + 1) * OW) / W + 1); ++ow) {
        const int w0 = bstart(ow, W, OW), w1 = bend(ow, W, OW);
        if (w < w0 || w >= w1) continue;
        const float inv = 1.f / (float)((h1 - h0) * (w1 - w0));
#pragma unroll
        for (int i = 0; i < 8; ++i) s[i] += __ldg(dout + (((long long)n * C + cg * 8 + i) * OH + oh) * OW + ow) * inv;
      }
    }
    reinterpret_cast<uint4*>(dx)[(((long long)n * Hp + h + 1) * Wp + w + 1) * groups + cg] = pack8(s);
  }
}

// Same result, one CTA per frame: the frame's (C, OH, OW) gradient is staged in shared memory transposed to [bin][channel], so the
// strided fp32 reads of the kernel above (32 sectors per warp load) become one coalesced pass, and all index math is 32-bit.
__global__ void avgpool_pad_bwd_frame_kernel(const float* __restrict__ dout, int N, int H, int W, int C, int OH, int OW,
                                             __nv_bfloat16* __restrict__ dx) {
  extern __shared__ __align__(16) float sd[];              // [OH*OW][C + 4]
  const int bins = OH * OW, groups = C >> 3, Wp = W + 2, Hp = H + 2, pitch = C + 4;
  const bool uniform = H % OH == 0 && W % OW == 0;          // disjoint bins of equal size: every pixel lies in exactly one
  const int kh = H / OH, kw = W / OW;
  for (int n = blockIdx.x; n < N; n += gridDim.x) {
    const float* src = dout + (long long)n * C * bins;       // the frame's (C, OH, OW) gradients are one contiguous run: coalesced reads
    for (int i = threadIdx.x; i < C * bins; i += blockDim.x) {
      const int c = i / bins, b = i - c * bins;
      sd[b * pitch + c] = __ldg(src + i);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < H * W * groups; t += blockDim.x) {
      const int cg = t % groups, pix = t / groups;
      const int w = pix % W, h = pix / W;
      float s[8];
      if (uniform) {
        const float inv = 1.f / (float)(kh * kw);
        const float* q = sd + ((h / kh) * OW + w / kw) * pitch + cg * 8;
        const float4 lo = *reinterpret_cast<const float4*>(q), hi = *reinterpret_cast<const float4*>(q + 4);
        s[0] = lo.x * inv; s[1] = lo.y * inv; s[2] = lo.z * inv; s[3] = lo.w * inv;
        s[4] = hi.x * inv; s[5] = hi.y * inv; s[6] = hi.z * inv; s[7] = hi.w * inv;
        reinterpret_cast<uint4*>(dx)[(((long long)n * Hp + h + 1) * Wp + w + 1) * groups + cg] = pack8(s);
        continue;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) s[i] = 0.f;
      const int ohc = (h * OH) / H, owc = (w * OW) / W;
      for (int oh = max(0, ohc - 1); oh <= min(OH - 1, ((h + 1) * OH) / H + 1); ++oh) {
        const int h0 = bstart(oh, H, OH), h1 = bend(oh, H, OH);
        if (h < h0 || h >= h1) continue;
        for (int ow = max(0, owc - 1); ow <= min(OW - 1, ((w + 1) * OW) / W + 1); ++ow) {
          const int w0 = bstart(ow, W, OW), w1 = bend(ow, W, OW);
          if (w < w0 || w >= w1) continue;
          const float inv = 1.f / (float)((h1 - h0) * (w1 - w0));
          const float4 lo = *reinterpret_cast<const float4*>(sd + (oh * OW + ow) * pitch + cg * 8);
          const float4 hi = *reinterpret_cast<const float4*>(sd + (oh * OW + ow) * pitch + cg * 8 + 4);
          s[0] = fmaf(lo.x, inv, s[0]); s[1] = fmaf(lo.y, inv, s[1]); s[2] = fmaf(lo.z, inv, s[2]); s[3] = fmaf(lo.w, inv, s[3]);
          s[4] = fmaf(hi.x, inv, s[4]); s[5] = fmaf(hi.y, inv, s[5]); s[6] = fmaf(hi.z, inv, s[6]); s[7] = fmaf(hi.w, inv, s[7]);
        }
      }
      reinterpret_cast<uint4*>(dx)[(((long long)n * Hp + h + 1) * Wp + w + 1) * groups + cg] = pack8(s);
    }
    __syncthreads();
  }
}

// development knobs for the apply kernels: rows per CTA iteration (2 or 4; anything else runs 2) and CTAs per SM
inline int bn_rows_per_iter() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CVAD_BN_ROWS");
    v = e ? atoi(e) : 2;
    if (v != 2 && v != 4) v = 2;
  }
  return v;
}
inline int bn_ctas_per_sm() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CVAD_BN_CTAS");
    v = e ? atoi(e) : 8;
    if (v < 1 || v > 32) v = 8;
  }
  return v;
}

inline int make_geo(PadGeo& g, int N, int H, int W, int C, int phase) {
  if (C % 8 || C > 256 || (C / 8) & (C / 8 - 1) || (long long)N * (H + 2) * (W + 2) * 4 > 0x7fffffffLL) return 1;
  g.N = N; g.H = H; g.W = W; g.C = C;
  g.Hq = phase ? (H - 1) / 2 + 3 : 0;
  g.Wq = phase ? (W - 1) / 2 + 3 : 0;
  // the apply kernel addresses its output in 16-byte vectors with 32-bit indices
  if ((long long)N * (H + 2) * (W + 2) * (C / 8) > 0xffffffffLL || 4LL * N * g.Hq * g.Wq * (C / 8) > 0xffffffffLL) return 1;
  g.lg = 0;
  while ((8 << g.lg) < C) ++g.lg;
  fast_div_init((unsigned)W, g.mulW, g.shrW);
  fast_div_init((unsigned)H, g.mulH, g.shrH);
  fast_div_init((unsigned)(H + 2), g.mulHp, g.shrHp);
  fast_div_init((unsigned)(g.Hq > 0 ? g.Hq : 1), g.mulHq, g.shrHq);
  fast_div_init((unsigned)N, g.mulN, g.shrN);
  return 0;
}

template <bool BWD>
void launch_reduce(const __nv_bfloat16* r, const __nv_bfloat16* d, const PadGeo& g, int N, int H, int phase_in, const float* mean,
                   const float* invstd, const float* gamma, const float* beta, double* ws, cudaStream_t st) {
  const size_t sm = 256 * 16 * sizeof(float);
  // (a row-structured variant of this reduction -- fixed channel group per thread, no per-element index division -- measured 5-10 % SLOWER
  // at every backbone shape: the kernel is not instruction-bound)
  const int per_sm = BWD ? 3 : 4;                         // one wave (the kernel's launch bounds)
  const int blocks = N * H < per_sm * cvad_num_sms() ? N * H : per_sm * cvad_num_sms();
  if (BWD && phase_in) pad_reduce_kernel<BWD, 1><<<blocks, 256, sm, st>>>(r, d, g, mean, invstd, gamma, beta, ws);
  else pad_reduce_kernel<BWD, 0><<<blocks, 256, sm, st>>>(r, d, g, mean, invstd, gamma, beta, ws);
}

// Grid of a row-walking apply kernel: as many CTAs as are RESIDENT at once (occupancy x SMs), each walking its share of the rows.  A
// CTA's prologue is ~50 dependent loads of per-channel constants; with 8 x SMs CTAs -- four waves at 2 resident CTAs per SM -- the small
// layers paid it once per 2-3 row iterations (ncu: 36 us for 54 MB at 8x12x256), and the waves ended unevenly on the large ones.  Measured
// on the M-A step (A/B twice on one box): 8 x SMs CTAs everywhere 3.960 ms; resident-only for tensors with < 4 / < 8 row iterations per CTA
// 3.903 / 3.888 ms; resident-only everywhere 3.873 ms.  CVAD_BN_SMALL_GRID=k applies the rule below k iterations only (0 = never).
template <typename K>
int apply_grid(K kernel, int want) {
  const int cap = bn_ctas_per_sm() * cvad_num_sms();
  int blocks = want < cap ? want : cap;
  static int small_rule = -1;
  if (small_rule < 0) {
    const char* e = getenv("CVAD_BN_SMALL_GRID");
    small_rule = e ? atoi(e) : (1 << 20);
  }
  if (small_rule && want < small_rule * cap) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) == cudaSuccess && per_sm > 0) {
      const int resident = per_sm * cvad_num_sms();
      if (resident < blocks) blocks = resident;
    }
  }
  return blocks;
}

inline int bn_apply_reverse() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CVAD_BN_REVERSE");
    v = e ? atoi(e) : 1;
  }
  return v;
}

int launch_apply(const __nv_bfloat16* r, __nv_bfloat16* a, uint8_t* mask, const PadGeo& g, int N, int H, int phase_out, const float* mean,
                 const float* invstd, const float* gamma, const float* beta, bool finalize, const BnFin& fin_in, cudaStream_t st) {
  BnFin fin = fin_in;
  fin.reverse = bn_apply_reverse();
  const int rows = phase_out ? 2 * N * g.Hq : N * (H + 2);
  const int R = bn_rows_per_iter();
  const int want = (rows + R - 1) / R;
#define CVAD_APPLY(PH, RR, FI) \
  pad_bn_apply_relu_kernel<PH, RR, FI><<<apply_grid(pad_bn_apply_relu_kernel<PH, RR, FI>, want), 256, 0, st>>>(r, a, mask, g, mean, invstd, gamma, \
                                                                                                                beta, fin)
#define CVAD_APPLY2(PH, FI) { if (R == 2) CVAD_APPLY(PH, 2, FI); else CVAD_APPLY(PH, 4, FI); }
  if (phase_out) { if (finalize) CVAD_APPLY2(1, true) else CVAD_APPLY2(1, false) }
  else { if (finalize) CVAD_APPLY2(0, true) else CVAD_APPLY2(0, false) }
#undef CVAD_APPLY2
#undef CVAD_APPLY
  CVAD_LAUNCH_CHECK();
  return 0;
}

// CVAD_BN_FOLD=1: the finalize / parameter-gradient kernels are folded into the apply kernels; 0 (default): separate launches.  Measured
// on the M-A step (A/B on one box, twice): folded 3.936 / 3.972 ms, separate 3.912 / 3.960 ms -- every block redoing the fp64 finalize
// costs more than the two tiny launches it saves inside a replayed graph.
inline int bn_fold() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CVAD_BN_FOLD");
    v = e ? atoi(e) : 0;
  }
  return v;
}

// apply pass of the backward; with dgamma / dbeta it also performs the parameter-gradient update and re-zeroes ws (FOLD).  ts: the
// (S1, T) form (no FOLD), which also takes the parameter-gradient sums
int launch_bwd_apply(const __nv_bfloat16* r, const __nv_bfloat16* d, __nv_bfloat16* draw, const PadGeo& g, int N, int H, int W, int phase_in,
                     const float* mean, const float* invstd, const float* gamma, const float* beta, double* ws, int training, bool fold,
                     float* dgamma, float* dbeta, cudaStream_t st, bool ts = false) {
  const int rows = N * (H + 2);
  const int R = bn_rows_per_iter();
  const int want = (rows + R - 1) / R;
  const double count = (double)N * H * W;
  static int occ3 = -1;
  if (occ3 < 0) {
    const char* e = getenv("CVAD_BN_OCC");
    occ3 = e ? (atoi(e) >= 3) : 0;          // measured: 3 CTAs per SM (80 registers, ~20 spilled) is 75 us per step slower than 2 (98 registers)
  }
#define CVAD_BAPPLY(PH, RR, FO, OC, TS)                                                                                                     \
  pad_bn_relu_bwd_apply_kernel<PH, RR, FO, OC, TS><<<apply_grid(pad_bn_relu_bwd_apply_kernel<PH, RR, FO, OC, TS>, want), 256, 0, st>>>(       \
      r, d, draw, g, mean, invstd, gamma, beta, ws, count, training, dgamma, dbeta)
#define CVAD_BAPPLY2(PH, FO, TS) \
  { if (R == 2) { if (occ3) CVAD_BAPPLY(PH, 2, FO, 3, TS); else CVAD_BAPPLY(PH, 2, FO, 2, TS); } else CVAD_BAPPLY(PH, 4, FO, 1, TS); }
  if (ts) { if (phase_in) CVAD_BAPPLY2(1, false, true) else CVAD_BAPPLY2(0, false, true) }
  else if (phase_in) { if (fold) CVAD_BAPPLY2(1, true, false) else CVAD_BAPPLY2(1, false, false) }
  else { if (fold) CVAD_BAPPLY2(0, true, false) else CVAD_BAPPLY2(0, false, false) }
#undef CVAD_BAPPLY2
#undef CVAD_BAPPLY
  CVAD_LAUNCH_CHECK();
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------- padded-flat entry points
CVAD_API int cvad_pad_bn_stats_bf16(const void* raw, int N, int H, int W, int C, double* ws, float eps, float momentum, float* mean,
                                    float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked, void* stream) {
  PadGeo g;
  if (make_geo(g, N, H, W, C, 0)) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  launch_reduce<false>((const __nv_bfloat16*)raw, nullptr, g, N, H, 0, nullptr, nullptr, nullptr, nullptr, ws, st);
  CVAD_LAUNCH_CHECK();
  return bn_finalize_launch(ws, C, (double)N * H * W, nullptr, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked, st);
}

CVAD_API int cvad_bn_finalize_f64(double* ws, int C, double count, float eps, float momentum, float* mean, float* invstd, float* running_mean,
                                  float* running_var, long long* num_batches_tracked, void* stream) {
  if (C <= 0 || count <= 0) return (int)cudaErrorInvalidValue;
  return bn_finalize_launch(ws, C, count, nullptr, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked,
                            (cudaStream_t)stream);
}

CVAD_API int cvad_pad_bn_apply_relu_bf16(const void* raw, void* act, int N, int H, int W, int C, int phase_out, const float* mean,
                                         const float* invstd, const float* gamma, const float* beta, void* stream) {
  PadGeo g;
  if (make_geo(g, N, H, W, C, phase_out)) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  BnFin fin;
  memset(&fin, 0, sizeof(fin));
  return launch_apply((const __nv_bfloat16*)raw, (__nv_bfloat16*)act, nullptr, g, N, H, phase_out, mean, invstd, gamma, beta, false, fin, st);
}

namespace {
int finalize_apply(const void* raw, void* act, void* mask, int N, int H, int W, int C, int phase_out, double* ws, float eps, float momentum,
                   const float* gamma, const float* beta, float* mean, float* invstd, float* running_mean, float* running_var,
                   long long* num_batches_tracked, void* stream) {
  PadGeo g;
  if (make_geo(g, N, H, W, C, phase_out) || !ws || !mean || !invstd) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  const double count = (double)N * H * W;
  if (!bn_fold()) {
    const int e = bn_finalize_launch(ws, C, count, nullptr, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked, st);
    if (e) return e;
    BnFin none;
    memset(&none, 0, sizeof(none));
    return launch_apply((const __nv_bfloat16*)raw, (__nv_bfloat16*)act, (uint8_t*)mask, g, N, H, phase_out, mean, invstd, gamma, beta, false,
                        none, st);
  }
  BnFin fin = {0, ws, count, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked};
  return launch_apply((const __nv_bfloat16*)raw, (__nv_bfloat16*)act, (uint8_t*)mask, g, N, H, phase_out, nullptr, nullptr, gamma, beta, true,
                      fin, st);
}
}  // namespace

CVAD_API int cvad_pad_bn_finalize_apply_relu_bf16(const void* raw, void* act, int N, int H, int W, int C, int phase_out, double* ws, float eps,
                                                  float momentum, const float* gamma, const float* beta, float* mean, float* invstd,
                                                  float* running_mean, float* running_var, long long* num_batches_tracked, void* stream) {
  return finalize_apply(raw, act, nullptr, N, H, W, C, phase_out, ws, eps, momentum, gamma, beta, mean, invstd, running_mean, running_var,
                        num_batches_tracked, stream);
}

CVAD_API int cvad_pad_bn_finalize_apply_relu_mask_bf16(const void* raw, void* act, void* mask, int N, int H, int W, int C, int phase_out,
                                                       double* ws, float eps, float momentum, const float* gamma, const float* beta, float* mean,
                                                       float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked,
                                                       void* stream) {
  if (!mask) return (int)cudaErrorInvalidValue;
  return finalize_apply(raw, act, mask, N, H, W, C, phase_out, ws, eps, momentum, gamma, beta, mean, invstd, running_mean, running_var,
                        num_batches_tracked, stream);
}

CVAD_API int cvad_pad_bn_apply_relu_mask_bf16(const void* raw, void* act, void* mask, int N, int H, int W, int C, int phase_out, const float* mean,
                                              const float* invstd, const float* gamma, const float* beta, void* stream) {
  PadGeo g;
  if (!mask || make_geo(g, N, H, W, C, phase_out)) return (int)cudaErrorInvalidValue;
  BnFin fin;
  memset(&fin, 0, sizeof(fin));
  return launch_apply((const __nv_bfloat16*)raw, (__nv_bfloat16*)act, (uint8_t*)mask, g, N, H, phase_out, mean, invstd, gamma, beta, false, fin,
                      (cudaStream_t)stream);
}

CVAD_API int cvad_pad_bn_relu_bwd_bf16(const void* raw, const void* dact, void* draw, int N, int H, int W, int C, int phase_in,
                                       const float* mean, const float* invstd, const float* gamma, const float* beta, int training, double* ws,
                                       float* dgamma, float* dbeta, void* stream) {
  PadGeo g;
  if (make_geo(g, N, H, W, C, phase_in)) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  const __nv_bfloat16 *r = (const __nv_bfloat16*)raw, *d = (const __nv_bfloat16*)dact;
  launch_reduce<true>(r, d, g, N, H, phase_in, mean, invstd, gamma, beta, ws, st);
  CVAD_LAUNCH_CHECK();
  if (draw) {
    const bool fold = bn_fold() != 0;
    int e = launch_bwd_apply(r, d, (__nv_bfloat16*)draw, g, N, H, W, phase_in, mean, invstd, gamma, beta, ws, training, fold, dgamma, dbeta, st);
    if (e || fold) return e;
  }
  return bn_params_launch(ws, C, dgamma, dbeta, st);
}

// The same with the two per-channel sums already in ws (taken by the data-gradient epilogue of the layer above,
// cvad_flat_conv3x3_dgrad_bnstats_bf16): only the apply pass and the dgamma / dbeta update run -- one pass over raw and dact instead of two.
CVAD_API int cvad_pad_bn_relu_bwd_apply_bf16(const void* raw, const void* dact, void* draw, int N, int H, int W, int C, int phase_in,
                                             const float* mean, const float* invstd, const float* gamma, const float* beta, int training,
                                             double* ws, float* dgamma, float* dbeta, void* stream) {
  PadGeo g;
  if (make_geo(g, N, H, W, C, phase_in) || !draw) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  const __nv_bfloat16 *r = (const __nv_bfloat16*)raw, *d = (const __nv_bfloat16*)dact;
  const bool fold = bn_fold() != 0;
  int e = launch_bwd_apply(r, d, (__nv_bfloat16*)draw, g, N, H, W, phase_in, mean, invstd, gamma, beta, ws, training, fold, dgamma, dbeta, st);
  if (e || fold) return e;
  return bn_params_launch(ws, C, dgamma, dbeta, st);
}

// the parameter-gradient update of the TS backward, from g_bn_tsum (re-zeroed)
static __global__ void bn_tsum_params_kernel(int C, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    bn_params_channel(g_bn_tsum, C, c, dgamma, dbeta);
    g_bn_tsum[c] = 0.0;
    g_bn_tsum[C + c] = 0.0;
  }
}

// Training-mode backward without the reduce pass: ws[0, C) = sum g and ws[C, 2C) = sum act*dact are already there (see the TS form of
// pad_bn_relu_bwd_apply_kernel); one pass over raw and dact, then the parameter-gradient update.  ws is zero again afterwards.
CVAD_API int cvad_pad_bn_relu_bwd_tsum_bf16(const void* raw, const void* dact, void* draw, int N, int H, int W, int C, int phase_in,
                                            const float* mean, const float* invstd, const float* gamma, const float* beta, double* ws,
                                            float* dgamma, float* dbeta, void* stream) {
  PadGeo g;
  if (make_geo(g, N, H, W, C, phase_in) || !draw || !ws) return (int)cudaErrorInvalidValue;
  cudaStream_t st = (cudaStream_t)stream;
  int e = launch_bwd_apply((const __nv_bfloat16*)raw, (const __nv_bfloat16*)dact, (__nv_bfloat16*)draw, g, N, H, W, phase_in, mean, invstd, gamma,
                           beta, ws, 1, false, nullptr, nullptr, st, true);
  if (e) return e;
  bn_tsum_params_kernel<<<(C + 127) / 128, 128, 0, st>>>(C, dgamma, dbeta);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_pad_avgpool_bf16_fwd(const void* x, int N, int H, int W, int C, int OH, int OW, float* out, void* stream) {
  long long total = (long long)N * OH * OW * (C / 8);
  if (total <= 0 || C % 8) return total <= 0 ? 0 : (int)cudaErrorInvalidValue;
  const size_t frame_smem = (size_t)OH * OW * (C + 4) * sizeof(float);
  if (frame_smem <= 48 * 1024)
    avgpool_pad_fwd_frame_kernel<<<N < 8 * cvad_num_sms() ? N : 8 * cvad_num_sms(), 256, frame_smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)x, N, H, W, C, OH, OW, out);
  else
    avgpool_pad_fwd_kernel<<<blocks_for(total), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, N, H, W, C, OH, OW, out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_pad_avgpool_bf16_bwd(const float* dout, int N, int H, int W, int C, int OH, int OW, void* dx, void* stream) {
  long long total = (long long)N * H * W * (C / 8);
  if (total <= 0 || C % 8) return total <= 0 ? 0 : (int)cudaErrorInvalidValue;
  const size_t frame_smem = (size_t)OH * OW * (C + 4) * sizeof(float);
  if (frame_smem <= 48 * 1024)
    avgpool_pad_bwd_frame_kernel<<<N < 8 * cvad_num_sms() ? N : 8 * cvad_num_sms(), 256, frame_smem, (cudaStream_t)stream>>>(
        dout, N, H, W, C, OH, OW, (__nv_bfloat16*)dx);
  else
    avgpool_pad_bwd_kernel<<<blocks_for(total), 256, 0, (cudaStream_t)stream>>>(dout, N, H, W, C, OH, OW, (__nv_bfloat16*)dx);
  CVAD_LAUNCH_CHECK();
  return 0;
}

// M-D (causal_anomaly_detection1.py) specific kernels: the LSTM(64->64) recurrence over T (cad1:182-188, 238-239), the
// cosine-distance-to-memory anomaly score (cad1:262-301), the reconstruction MSE with its gradient and the per-clip
// error used by calculate_anomaly_scores (cad1:323-344, 545-552), and the scores of every window slot of S streams read
// from their frame rings (infer.MultiStreamAutoEncoderScorer).  Convolutions, BatchNorm and the linear layers of the
// autoencoder reuse the generic fp32 kernels (conv_f32.cu: a ConvTranspose2d forward IS the data-gradient kernel).
#include "common.cuh"
#include "cvad_b200.h"

namespace {

constexpr int LH = 64;            // hidden size (cad1:183-184: latent_dim = 64)
constexpr int LG = 4 * LH;        // gate rows i, f, g, o (torch order)

__device__ __forceinline__ float sigm(float v) { return 1.f / (1.f + expf(-v)); }

// gi (N,T,256) = x W_ih^T + b_ih precomputed.  One block of 256 threads per sequence; thread g owns gate row g of W_hh.
// saved (N,T,6,64) = i, f, g, o, c_prev, h_prev for the backward.
__global__ void __launch_bounds__(LG) lstm_fwd_kernel(const float* __restrict__ gi, const float* __restrict__ w_hh, const float* __restrict__ b_hh,
                                                      int T, float* __restrict__ hT, float* __restrict__ saved) {
  const int n = blockIdx.x, g = threadIdx.x;
  __shared__ float h[LH], c[LH], gate[LG];
  float w[LH];
#pragma unroll
  for (int i = 0; i < LH; ++i) w[i] = w_hh[g * LH + i];
  const float bias = b_hh[g];
  if (g < LH) { h[g] = 0.f; c[g] = 0.f; }
  __syncthreads();
  for (int t = 0; t < T; ++t) {
    float acc = bias + gi[((long long)n * T + t) * LG + g];
#pragma unroll
    for (int i = 0; i < LH; ++i) acc = fmaf(w[i], h[i], acc);
    gate[g] = (g >= 2 * LH && g < 3 * LH) ? tanhf(acc) : sigm(acc);
    __syncthreads();
    if (g < LH) {
      const float ig = gate[g], fg = gate[LH + g], gg = gate[2 * LH + g], og = gate[3 * LH + g];
      const float cp = c[g], hp = h[g];
      const float cn = fg * cp + ig * gg;
      if (saved) {
        float* s = saved + ((long long)n * T + t) * 6 * LH;
        s[g] = ig; s[LH + g] = fg; s[2 * LH + g] = gg; s[3 * LH + g] = og; s[4 * LH + g] = cp; s[5 * LH + g] = hp;
      }
      c[g] = cn;
      h[g] = og * tanhf(cn);
    }
    __syncthreads();
  }
  if (g < LH) hT[(long long)n * LH + g] = h[g];
}

// BPTT from dhT (N,64): dgi (N,T,256) = gradient of the pre-activations (== gradient of gi and of b_hh rows);
// dw_hh (256,64) and db_hh (256) are ADDED atomically (one block per sequence).
__global__ void __launch_bounds__(LG) lstm_bwd_kernel(const float* __restrict__ dhT, const float* __restrict__ saved,
                                                      const float* __restrict__ w_hh, int T, float* __restrict__ dgi,
                                                      float* __restrict__ dw_hh, float* __restrict__ db_hh) {
  const int n = blockIdx.x, g = threadIdx.x;
  extern __shared__ float sm[];
  float* wT = sm;                        // [LH][LG+1]: wT[i][g] = w_hh[g][i]
  float* dh = wT + LH * (LG + 1);        // [LH]
  float* dc = dh + LH;                   // [LH]
  float* dgate = dc + LH;                // [LG]
  float* hp = dgate + LG;                // [LH]
  for (int i = 0; i < LH; ++i) wT[i * (LG + 1) + g] = w_hh[g * LH + i];
  if (g < LH) { dh[g] = dhT[(long long)n * LH + g]; dc[g] = 0.f; }
  float dw[LH];
#pragma unroll
  for (int i = 0; i < LH; ++i) dw[i] = 0.f;
  float dbias = 0.f;
  __syncthreads();
  for (int t = T - 1; t >= 0; --t) {
    const float* s = saved + ((long long)n * T + t) * 6 * LH;
    if (g < LH) {
      const float ig = s[g], fg = s[LH + g], gg = s[2 * LH + g], og = s[3 * LH + g], cp = s[4 * LH + g];
      const float cn = fg * cp + ig * gg;
      const float tc = tanhf(cn);
      const float d = dh[g];
      const float dcn = dc[g] + d * og * (1.f - tc * tc);
      dgate[g] = dcn * gg * ig * (1.f - ig);                 // i
      dgate[LH + g] = dcn * cp * fg * (1.f - fg);            // f
      dgate[2 * LH + g] = dcn * ig * (1.f - gg * gg);        // g
      dgate[3 * LH + g] = d * tc * og * (1.f - og);          // o
      dc[g] = dcn * fg;
      hp[g] = s[5 * LH + g];
    }
    __syncthreads();
    const float dg = dgate[g];
    dgi[((long long)n * T + t) * LG + g] = dg;
    dbias += dg;
#pragma unroll
    for (int i = 0; i < LH; ++i) dw[i] = fmaf(dg, hp[i], dw[i]);
    if (g < LH) {
      float acc = 0.f;
      for (int k = 0; k < LG; ++k) acc = fmaf(wT[g * (LG + 1) + k], dgate[k], acc);
      dh[g] = acc;
    }
    __syncthreads();
  }
  if (dw_hh)
    for (int i = 0; i < LH; ++i) atomicAdd(dw_hh + g * LH + i, dw[i]);
  if (db_hh) atomicAdd(db_hh + g, dbias);
}

// cad1:279-294 for one query row q (D floats) by the whole block: clamp(min_m (1 - clamp(cos(q, mem_m), -1, 1)), 0, 2) / 2 over the
// first n_filled rows of mem, returned to thread 0.  sq: D floats of shared memory, red: 32.  Each row's dot product is one thread's
// sequential loop and the minimum is exact, so the value is the same at any block size (the norm of q too while D <= blockDim.x).
__device__ float memory_score_block(const float* __restrict__ q, const float* __restrict__ mem, int n_filled, int D, float eps,
                                    float* __restrict__ sq, float* __restrict__ red) {
  float part = 0.f;
  for (int i = threadIdx.x; i < D; i += blockDim.x) { const float v = q[i]; part = fmaf(v, v, part); }
  const float nrm = fmaxf(sqrtf(block_sum(part, red)), eps);
  for (int i = threadIdx.x; i < D; i += blockDim.x) sq[i] = q[i] / nrm;
  __syncthreads();
  float best = 3.f;
  for (int m = threadIdx.x; m < n_filled; m += blockDim.x) {
    const float* r = mem + (long long)m * D;
    float dot = 0.f, nn = 0.f;
    for (int i = 0; i < D; ++i) { const float v = r[i]; nn = fmaf(v, v, nn); }
    const float mn = fmaxf(sqrtf(nn), eps);
    for (int i = 0; i < D; ++i) dot = fmaf(sq[i], r[i] / mn, dot);
    const float sim = fminf(fmaxf(dot, -1.f), 1.f);
    best = fminf(best, 1.f - sim);
  }
  __syncthreads();
  // block min: warp shuffles, then one value per warp through shared memory
  for (int o = 16; o > 0; o >>= 1) best = fminf(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
  __syncthreads();
  float v = red[0];
  if (threadIdx.x == 0)
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) v = fminf(v, red[w]);
  return fminf(fmaxf(v, 0.f), 2.f) * 0.5f;
}

// score[b] = memory_score_block(seq_b) over the first n_filled memory rows (cad1:279-294)
__global__ void __launch_bounds__(128) memory_score_kernel(const float* __restrict__ seq, const float* __restrict__ mem, int n_filled, int D,
                                                           float eps, float* __restrict__ score) {
  extern __shared__ float sq[];          // normalised query [D]
  __shared__ float red[32];
  const int b = blockIdx.x;
  const float s = memory_score_block(seq + (long long)b * D, mem, n_filled, D, eps, sq, red);
  if (threadIdx.x == 0) score[b] = s;
}

// calculate_anomaly_scores (cad1:526-564) for every window slot of S streams, one CTA per slot (k, j) (stream_push, common.cuh):
// recon_err = mean over the window's T frames x E values of (recon - x_t)^2, x_t read from stream k's frame ring (fp32 per thread and
// vector, fp64 across the block, as recon_mse_kernel); mem_score = memory_score_block(z) over the first clamp(*memory_ptr, 0, memory_rows)
// rows, 0 below 10 rows; score = 0.7 recon_err + 0.3 mem_score, rounded as the two products and the sum are in torch.  Unused slots
// (j >= n_win_k) get zeros.
__global__ void __launch_bounds__(256) streams_md_scores_kernel(const float4* __restrict__ rings, long long cap, long long E4, int T, int stride,
                                                                long long m, const long long* __restrict__ cursors,
                                                                const long long* __restrict__ push, const float4* __restrict__ recon,
                                                                const float* __restrict__ z, const float* __restrict__ memory, int memory_rows,
                                                                const long long* __restrict__ memory_ptr, int D, float* __restrict__ score,
                                                                float* __restrict__ recon_err, float* __restrict__ mem_score) {
  extern __shared__ float sq[];          // normalised query [D]
  __shared__ float red[32];
  __shared__ double shd[32];
  cvad_pdl_enter();
  const long long slot = blockIdx.x;
  const int k = (int)(slot / m);
  const long long j = slot - k * m;
  const StreamPush p = stream_push(cursors, push, k, T, stride);
  if (j >= p.n_win) {
    if (threadIdx.x == 0) score[slot] = recon_err[slot] = mem_score[slot] = 0.f;
    return;
  }
  const float4* rb = recon + slot * E4;
  const float4* ring = rings + (long long)k * cap * E4;
  const long long first = (p.next + j) * stride;
  double acc = 0.0;
  for (long long e = threadIdx.x; e < E4; e += blockDim.x) {
    const float4 r = __ldg(rb + e);
    float part = 0.f;
#pragma unroll 4
    for (int t = 0; t < T; ++t) {
      const float4 x = __ldg(ring + ((first + t) % cap) * E4 + e);
      const float d0 = r.x - x.x, d1 = r.y - x.y, d2 = r.z - x.z, d3 = r.w - x.w;
      part = fmaf(d0, d0, part);
      part = fmaf(d1, d1, part);
      part = fmaf(d2, d2, part);
      part = fmaf(d3, d3, part);
    }
    acc += (double)part;
  }
  acc = block_sum_d(acc, shd);
  const long long filled = min(max(*memory_ptr, 0LL), (long long)memory_rows);       // the same value in every thread
  const float ms = filled >= 10 ? memory_score_block(z + slot * D, memory, (int)filled, D, 1e-8f, sq, red) : 0.f;
  if (threadIdx.x == 0) {
    const float re = (float)(acc / ((double)T * (double)(4 * E4)));
    recon_err[slot] = re;
    mem_score[slot] = ms;
    score[slot] = __fadd_rn(__fmul_rn(0.7f, re), __fmul_rn(0.3f, ms));
  }
}

// recon (B, ., E) with t-stride rts (0 = one reconstruction broadcast over T), frames (B,T,E).
// clip_err[b] += sum_{t,e} (recon - x)^2 / (T*E)   (pre-zeroed);  drecon (may be NULL): d(mean over B,T,E)/d recon
// VEC = 4: 16-byte accesses (E % 4 == 0, 16-byte aligned tensors), four time steps in flight per thread; VEC = 1: any E / alignment.
template <int VEC>
__global__ void __launch_bounds__(256) recon_mse_kernel(const float* __restrict__ recon, long long rts, const float* __restrict__ x, int B, int T,
                                                        long long E, double* __restrict__ clip_acc, float* __restrict__ drecon) {
  __shared__ double shd[32];
  const int b = blockIdx.y;
  const float scale = 2.f / ((float)B * (float)T * (float)E);
  const long long EV = E / VEC;
  const float* rb = recon + (long long)b * (rts ? T : 1) * E;
  const float* xb = x + (long long)b * T * E;
  float* db = drecon ? drecon + (long long)b * (rts ? T : 1) * E : nullptr;
  double acc = 0.0;
  for (long long ev = blockIdx.x * (long long)blockDim.x + threadIdx.x; ev < EV; ev += (long long)gridDim.x * blockDim.x) {
    const long long e = ev * VEC;
    float gsum[VEC], part = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) gsum[i] = 0.f;
    constexpr int U = 4;
    for (int t0 = 0; t0 < T; t0 += U) {
      float r[U][VEC], v[U][VEC];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (t0 + u >= T) continue;
        const float* rp = rb + (long long)(t0 + u) * rts + e;
        const float* xp = xb + (long long)(t0 + u) * E + e;
        if (VEC == 4) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(rp)), c = __ldg(reinterpret_cast<const float4*>(xp));
          r[u][0] = a.x; r[u][1 % VEC] = a.y; r[u][2 % VEC] = a.z; r[u][3 % VEC] = a.w;
          v[u][0] = c.x; v[u][1 % VEC] = c.y; v[u][2 % VEC] = c.z; v[u][3 % VEC] = c.w;
        } else {
          r[u][0] = __ldg(rp);
          v[u][0] = __ldg(xp);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (t0 + u >= T) continue;
        float d[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          d[i] = r[u][i] - v[u][i];
          part = fmaf(d[i], d[i], part);
          gsum[i] += d[i];
        }
        if (rts && db) {
          float* dp = db + (long long)(t0 + u) * E + e;
          if (VEC == 4) *reinterpret_cast<float4*>(dp) = make_float4(d[0] * scale, d[1 % VEC] * scale, d[2 % VEC] * scale, d[3 % VEC] * scale);
          else *dp = d[0] * scale;
        }
      }
    }
    if (!rts && db) {
      if (VEC == 4) *reinterpret_cast<float4*>(db + e) = make_float4(gsum[0] * scale, gsum[1 % VEC] * scale, gsum[2 % VEC] * scale, gsum[3 % VEC] * scale);
      else db[e] = gsum[0] * scale;
    }
    acc += (double)part;
  }
  acc = block_sum_d(acc, shd);
  if (threadIdx.x == 0) atomicAdd(clip_acc + b, acc);
}

// one block: clip_err[b] = acc[b] / per_clip, loss = mean_b clip_err, acc re-zeroed
__global__ void __launch_bounds__(256) recon_finish_kernel(double* __restrict__ clip_acc, int B, double per_clip, float* __restrict__ clip_err,
                                                           float* __restrict__ loss, float* __restrict__ nonfinite_flag) {
  __shared__ double shd[32];
  double tot = 0.0;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const double v = clip_acc[b] / per_clip;
    if (clip_err) clip_err[b] = (float)v;
    tot += v;
    clip_acc[b] = 0.0;
  }
  tot = block_sum_d(tot, shd);
  if (threadIdx.x == 0) {
    const float l = (float)(tot / B);
    if (loss) *loss = l;
    if (nonfinite_flag && !isfinite(l)) *nonfinite_flag = 1.f;
  }
}

}  // namespace

CVAD_API int cvad_lstm_fwd_f32(const float* gi, const float* w_hh, const float* b_hh, int N, int T, float* hT, float* saved, void* stream) {
  if (N <= 0) return 0;
  lstm_fwd_kernel<<<N, LG, 0, (cudaStream_t)stream>>>(gi, w_hh, b_hh, T, hT, saved);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_lstm_bwd_f32(const float* dhT, const float* saved, const float* w_hh, int N, int T, float* dgi, float* dw_hh, float* db_hh,
                               void* stream) {
  if (N <= 0) return 0;
  const size_t smem = (size_t)(LH * (LG + 1) + LH + LH + LG + LH) * sizeof(float);
  static size_t configured[CVAD_MAX_DEVICES] = {};
  const cudaError_t ce = cvad_ensure_dyn_smem(lstm_bwd_kernel, smem, configured);
  if (ce != cudaSuccess) return (int)ce;
  lstm_bwd_kernel<<<N, LG, smem, (cudaStream_t)stream>>>(dhT, saved, w_hh, T, dgi, dw_hh, db_hh);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_memory_score_f32(const float* seq, const float* memory, int B, int n_filled, int D, float* score, void* stream) {
  if (B <= 0) return 0;
  memory_score_kernel<<<B, 128, D * sizeof(float), (cudaStream_t)stream>>>(seq, memory, n_filled, D, 1e-8f, score);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_streams_md_scores_f32(const float* frame_rings, int S, long long capacity, long long E, int T, int stride, long long m,
                                        const long long* cursors, const long long* push, const float* recon, const float* z, const float* memory,
                                        int memory_rows, const long long* memory_ptr, int D, float* score, float* recon_err, float* mem_score,
                                        void* stream) {
  if (!frame_rings || !cursors || !push || !recon || !z || !memory || !memory_ptr || !score || !recon_err || !mem_score || E <= 0 || E % 4 ||
      S <= 0 || T <= 0 || stride <= 0 || capacity <= 0 || D <= 0 || memory_rows <= 0 || m < 0 || (((uintptr_t)frame_rings | (uintptr_t)recon) & 15))
    return (int)cudaErrorInvalidValue;
  if (m == 0) return 0;
  cvad_launch_pdl(streams_md_scores_kernel, dim3((unsigned)(S * m)), dim3(256), (size_t)D * sizeof(float), (cudaStream_t)stream,
                  reinterpret_cast<const float4*>(frame_rings), capacity, E / 4, T, stride, m, cursors, push, reinterpret_cast<const float4*>(recon),
                  z, memory, memory_rows, memory_ptr, D, score, recon_err, mem_score);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_recon_mse_f32(const float* recon, long long recon_t_stride, const float* frames, int B, int T, long long E, double* ws,
                                float* clip_err, float* loss, float* drecon, float* nonfinite_flag, void* stream) {
  if (B <= 0 || T <= 0 || E <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = E % 4 == 0 && recon_t_stride % 4 == 0 && (((uintptr_t)recon | (uintptr_t)frames | (uintptr_t)drecon) & 15) == 0;
  const long long ev = vec ? E / 4 : E;
  int bx = (int)((ev + 255) / 256);
  const int cap = (16 * cvad_num_sms() + B - 1) / B;        // enough CTAs to fill the machine, no more than the work
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  if (vec) recon_mse_kernel<4><<<dim3(bx, B), 256, 0, st>>>(recon, recon_t_stride, frames, B, T, E, ws, drecon);
  else recon_mse_kernel<1><<<dim3(bx, B), 256, 0, st>>>(recon, recon_t_stride, frames, B, T, E, ws, drecon);
  CVAD_LAUNCH_CHECK();
  recon_finish_kernel<<<1, 256, 0, st>>>(ws, B, (double)T * (double)E, clip_err, loss, nonfinite_flag);
  CVAD_LAUNCH_CHECK();
  return 0;
}

// The pieces of M-A0 (video_anomaly_detection.py, "vad") that differ from M-A (ma_tail.cu): small dense/masked kernels over
// (B, 5 track slots) batches, one thread per row / element, fp32.
//   det_topk_decode  vad:127-165  boxes ordered by descending confidence (torch.topk over the 3 anchors), conf > 0.5 filter,
//                                 one all-zero dummy box when no anchor survives (vad:158-160: a constant, no gradient)
//   score_rows       vad:389-397  [cur | pred | |cur - pred|] per TRACK row (M-A averages over tracks first, cad:470-472)
//   masked_mean      vad:398-399  score.mean() over the clip's tracks
//   ma0_loss         vad:516-531  MSE(scores, labels) + 0.001 * (sum of finite KL terms / number of finite KL terms), with gradients
//   window_features  streaming sliding-window inference: gathers (n_windows, T, F) clips out of a ring of per-frame features
//   streams          S rings driven by device-side cursors {frames pushed, next window} and a per-push descriptor {count, reset}, so
//                    that one captured CUDA graph serves every push of a given size for all streams at once: ring_write,
//                    window_features, then cursor_advance (stream-ordered after both); the window rule is stream_push (common.cuh)
#include "common.cuh"
#include "cvad_b200.h"

namespace {

constexpr int MAXDET = 5;     // track slots of the dense layout shared with ma_tail.cu
constexpr int NA = 3;         // anchors (vad:118)
constexpr int NF = 6;         // causal factors (vad:406)

__device__ __forceinline__ float sigmoidf_(float v) { return 1.f / (1.f + expf(-v)); }

__global__ void det_topk_decode_kernel(const float* __restrict__ bbox, const float* __restrict__ conf_logit, long long R, float* __restrict__ box,
                                       int* __restrict__ cnt, int* __restrict__ src, float* __restrict__ flag) {
  cvad_pdl_enter();
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < R; r += (long long)gridDim.x * blockDim.x) {
    float c[NA];
    int order[NA];
#pragma unroll
    for (int k = 0; k < NA; ++k) {
      c[k] = sigmoidf_(conf_logit[r * NA + k]);      // vad:139
      order[k] = k;
    }
    // descending by confidence, the lower anchor index first among equals (3 elements: a fixed compare-exchange network)
#define CVAD_CSWAP(i, j)                                                       \
  if (c[order[j]] > c[order[i]]) { const int t_ = order[i]; order[i] = order[j]; order[j] = t_; }
    CVAD_CSWAP(0, 1)
    CVAD_CSWAP(1, 2)
    CVAD_CSWAP(0, 1)
#undef CVAD_CSWAP
    int n = 0;
#pragma unroll
    for (int k = 0; k < NA; ++k) {
      const int a = order[k];
      if (c[a] > 0.5f) {                              // vad:153
#pragma unroll
        for (int e = 0; e < 4; ++e) box[(r * MAXDET + n) * 4 + e] = bbox[(r * NA + a) * 4 + e];
        src[r * MAXDET + n] = a;
        ++n;
      }
    }
    const int real = n;
    if (n == 0) {                                     // vad:158-160
      src[r * MAXDET] = -1;
      n = 1;
    } else if (flag) {
      *flag = 1.f;                                    // bbox_head receives a gradient this step
    }
    for (int k = real; k < MAXDET; ++k) {
#pragma unroll
      for (int e = 0; e < 4; ++e) box[(r * MAXDET + k) * 4 + e] = 0.f;
      if (k >= n) src[r * MAXDET + k] = -1;
    }
    cnt[r] = n;
  }
}

__global__ void det_topk_decode_bwd_kernel(const float* __restrict__ dbox, const int* __restrict__ src, const int* __restrict__ cnt, long long R,
                                           float* __restrict__ dbbox) {
  cvad_pdl_enter();
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < R; r += (long long)gridDim.x * blockDim.x) {
    float g[NA][4];
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
      for (int e = 0; e < 4; ++e) g[a][e] = 0.f;
    const int n = cnt[r];
    for (int k = 0; k < n; ++k) {
      const int a = src[r * MAXDET + k];
#pragma unroll
      for (int aa = 0; aa < NA; ++aa)
        if (aa == a)
#pragma unroll
          for (int e = 0; e < 4; ++e) g[aa][e] = dbox[(r * MAXDET + k) * 4 + e];
    }
#pragma unroll
    for (int a = 0; a < NA; ++a)
#pragma unroll
      for (int e = 0; e < 4; ++e) dbbox[(r * NA + a) * 4 + e] = g[a][e];
  }
}

__global__ void score_rows_kernel(const float* __restrict__ z, const float* __restrict__ pred, long long rows, float* __restrict__ out) {
  cvad_pdl_enter();
  const long long total = rows * NF;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(t % NF);
    const long long r = t / NF;
    const float c = z[t], p = pred[t];
    out[r * 18 + f] = c;
    out[r * 18 + 6 + f] = p;
    out[r * 18 + 12 + f] = fabsf(c - p);
  }
}

__global__ void score_rows_bwd_kernel(const float* __restrict__ z, const float* __restrict__ pred, const float* __restrict__ dout, long long rows,
                                      float* __restrict__ dz, float* __restrict__ dpred) {
  cvad_pdl_enter();
  const long long total = rows * NF;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(t % NF);
    const long long r = t / NF;
    const float d = z[t] - pred[t];
    const float gd = dout[r * 18 + 12 + f] * (float)((d > 0.f) - (d < 0.f));      // torch.abs: sign(0) = 0
    dz[t] = dout[r * 18 + f] + gd;
    dpred[t] = dout[r * 18 + 6 + f] - gd;
  }
}

__global__ void masked_mean_kernel(const float* __restrict__ s, const int* __restrict__ ntr, int B, float* __restrict__ out) {
  cvad_pdl_enter();
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    const int n = ntr[b];
    float a = 0.f;
    for (int k = 0; k < n; ++k) a += s[b * MAXDET + k];
    out[b] = a / (float)n;
  }
}

__global__ void masked_mean_bwd_kernel(const float* __restrict__ dout, const int* __restrict__ ntr, int B, float* __restrict__ ds) {
  cvad_pdl_enter();
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < B * MAXDET; t += gridDim.x * blockDim.x) {
    const int b = t / MAXDET, k = t - b * MAXDET;
    const int n = ntr[b];
    ds[t] = k < n ? dout[b] / (float)n : 0.f;
  }
}

__global__ void ma0_loss_kernel(const float* __restrict__ scores, const float* __restrict__ kl, const long long* __restrict__ labels, int B,
                                float* __restrict__ out, float* __restrict__ dscores, float* __restrict__ dkl, float* __restrict__ flag) {
  cvad_pdl_enter();
  __shared__ float sh[32];
  float mse = 0.f, ks = 0.f, nfin = 0.f;
  const float invB = 1.f / (float)B;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float d = scores[b] - (float)labels[b];
    mse += d * d;
    const float k = kl[b];
    if (fabsf(k) <= 3.0e38f) { ks += k; nfin += 1.f; }        // vad:521 keeps the finite terms
    if (dscores) dscores[b] = 2.f * d * invB;
  }
  mse = block_sum(mse, sh);
  ks = block_sum(ks, sh);
  nfin = block_sum(nfin, sh);
  __shared__ float s_inv;
  if (threadIdx.x == 0) {
    mse *= invB;
    const float klm = nfin > 0.f ? ks / nfin : 0.f;             // vad:522: sum(valid) / len(valid), else 0
    const float total = mse + 0.001f * klm;
    out[0] = total; out[1] = mse; out[2] = klm;
    s_inv = nfin > 0.f ? 0.001f / nfin : 0.f;
    if (flag && !(fabsf(total) <= 3.0e38f)) *flag = 1.f;
  }
  __syncthreads();
  if (dkl)
    for (int b = threadIdx.x; b < B; b += blockDim.x) dkl[b] = fabsf(kl[b]) <= 3.0e38f ? s_inv : 0.f;
}

// out[w][t][:] = ring[(first + w*stride + t) % cap][:]  (F floats per frame, 16-byte vectors)
__global__ void window_features_kernel(const float4* __restrict__ ring, long long cap, long long first, int stride, int T, int F4, long long n_win,
                                       float4* __restrict__ out) {
  cvad_pdl_enter();
  const long long total = n_win * T * F4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % F4);
    const long long wt = i / F4;
    const int t = (int)(wt % T);
    const long long w = wt / T;
    const long long fr = (first + w * stride + t) % cap;
    out[i] = __ldg(ring + fr * F4 + v);
  }
}

// rings[k][(base_k + r) % cap][:] = feats[k*n + r][:] for r < count_k; rows r >= count_k are not read
__global__ void streams_ring_write_kernel(const float4* __restrict__ feats, int S, long long n, int F4, float4* __restrict__ rings, long long cap,
                                          int T, int stride, const long long* __restrict__ cursors, const long long* __restrict__ push) {
  cvad_pdl_enter();
  const long long total = S * n * F4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long row = i / F4;
    const int k = (int)(row / n);
    const long long r = row - k * n;
    if (r >= push[2 * k]) continue;
    const StreamPush p = stream_push(cursors, push, k, T, stride);
    const long long fr = (p.base + r) % cap;
    rings[(k * cap + fr) * F4 + (i - row * F4)] = __ldg(feats + i);
  }
}

// out[k*m + j][t][:] = rings[k][((next_k + j)*stride + t) % cap][:] for j < n_win_k, zeros for the unused slots j >= n_win_k
__global__ void streams_window_features_kernel(const float4* __restrict__ rings, int S, long long cap, int stride, int T, int F4, long long m,
                                               const long long* __restrict__ cursors, const long long* __restrict__ push, float4* __restrict__ out) {
  cvad_pdl_enter();
  const long long total = S * m * T * F4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % F4);
    const long long st = i / F4;
    const int t = (int)(st % T);
    const long long slot = st / T;
    const int k = (int)(slot / m);
    const long long j = slot - k * m;
    const StreamPush p = stream_push(cursors, push, k, T, stride);
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < p.n_win) x = __ldg(rings + (k * cap + ((p.next + j) * stride + t) % cap) * F4 + v);
    out[i] = x;
  }
}

// cursors[k] = {frames_k, next_k + n_win_k}
__global__ void streams_cursor_advance_kernel(long long* __restrict__ cursors, int S, int T, int stride, const long long* __restrict__ push) {
  cvad_pdl_enter();
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < S; k += gridDim.x * blockDim.x) {
    const StreamPush p = stream_push(cursors, push, k, T, stride);
    cursors[2 * k] = p.frames;
    cursors[2 * k + 1] = p.next + p.n_win;
  }
}

inline int blocks_of(long long n) {
  long long b = (n + 255) / 256;
  const long long cap = 8LL * cvad_num_sms();
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

CVAD_API int cvad_det_topk_decode_f32(const float* bbox, const float* conf_logit, long long rows, float* box, int* cnt, int* src, float* flag,
                                      void* stream) {
  if (rows <= 0) return 0;
  cvad_launch_pdl(det_topk_decode_kernel, dim3(blocks_of(rows)), dim3(256), 0, (cudaStream_t)stream, bbox, conf_logit, rows, box, cnt, src, flag);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_det_topk_decode_bwd_f32(const float* dbox, const int* src, const int* cnt, long long rows, float* dbbox, void* stream) {
  if (rows <= 0) return 0;
  cvad_launch_pdl(det_topk_decode_bwd_kernel, dim3(blocks_of(rows)), dim3(256), 0, (cudaStream_t)stream, dbox, src, cnt, rows, dbbox);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_score_rows_f32(const float* z, const float* pred, long long rows, float* out18, void* stream) {
  if (rows <= 0) return 0;
  cvad_launch_pdl(score_rows_kernel, dim3(blocks_of(rows * NF)), dim3(256), 0, (cudaStream_t)stream, z, pred, rows, out18);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_score_rows_bwd_f32(const float* z, const float* pred, const float* dout18, long long rows, float* dz, float* dpred,
                                     void* stream) {
  if (rows <= 0) return 0;
  cvad_launch_pdl(score_rows_bwd_kernel, dim3(blocks_of(rows * NF)), dim3(256), 0, (cudaStream_t)stream, z, pred, dout18, rows, dz, dpred);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_masked_mean_f32(const float* s, const int* ntr, int B, float* out, void* stream) {
  if (B <= 0) return 0;
  cvad_launch_pdl(masked_mean_kernel, dim3(blocks_of(B)), dim3(256), 0, (cudaStream_t)stream, s, ntr, B, out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_masked_mean_bwd_f32(const float* dout, const int* ntr, int B, float* ds, void* stream) {
  if (B <= 0) return 0;
  cvad_launch_pdl(masked_mean_bwd_kernel, dim3(blocks_of((long long)B * MAXDET)), dim3(256), 0, (cudaStream_t)stream, dout, ntr, B, ds);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_ma0_loss_f32(const float* scores, const float* kl, const long long* labels, int B, float* out3, float* dscores, float* dkl,
                               float* nonfinite_flag, void* stream) {
  if (B <= 0) return 0;
  cvad_launch_pdl(ma0_loss_kernel, dim3(1), dim3(256), 0, (cudaStream_t)stream, scores, kl, labels, B, out3, dscores, dkl, nonfinite_flag);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_window_features_f32(const float* ring, long long capacity, long long first_frame, int stride, int T, int F, long long n_windows,
                                      float* out, void* stream) {
  if (n_windows <= 0) return 0;
  if (F % 4 || capacity <= 0 || stride <= 0 || T <= 0 || first_frame < 0) return (int)cudaErrorInvalidValue;
  cvad_launch_pdl(window_features_kernel, dim3(blocks_of(n_windows * T * (F / 4))), dim3(256), 0, (cudaStream_t)stream, 
      reinterpret_cast<const float4*>(ring), capacity, first_frame, stride, T, F / 4, n_windows, reinterpret_cast<float4*>(out));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_streams_ring_write_f32(const float* feats, int S, long long n, int F, float* rings, long long capacity, int T, int stride,
                                         const long long* cursors, const long long* push, void* stream) {
  if (F % 4 || capacity <= 0 || S <= 0 || n < 0 || T <= 0 || stride <= 0 || !feats || !rings || !cursors || !push)
    return (int)cudaErrorInvalidValue;
  if (n == 0) return 0;
  cvad_launch_pdl(streams_ring_write_kernel, dim3(blocks_of(S * n * (F / 4))), dim3(256), 0, (cudaStream_t)stream,
                  reinterpret_cast<const float4*>(feats), S, n, F / 4, reinterpret_cast<float4*>(rings), capacity, T, stride, cursors, push);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_streams_window_features_f32(const float* rings, int S, long long capacity, int stride, int T, int F, long long m,
                                              const long long* cursors, const long long* push, float* out, void* stream) {
  if (F % 4 || capacity <= 0 || S <= 0 || m < 0 || T <= 0 || stride <= 0 || !rings || !cursors || !push || !out)
    return (int)cudaErrorInvalidValue;
  if (m == 0) return 0;
  cvad_launch_pdl(streams_window_features_kernel, dim3(blocks_of(S * m * T * (F / 4))), dim3(256), 0, (cudaStream_t)stream,
                  reinterpret_cast<const float4*>(rings), S, capacity, stride, T, F / 4, m, cursors, push, reinterpret_cast<float4*>(out));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_streams_cursor_advance(long long* cursors, int S, int T, int stride, const long long* push, void* stream) {
  if (S <= 0 || T <= 0 || stride <= 0 || !cursors || !push) return (int)cudaErrorInvalidValue;
  cvad_launch_pdl(streams_cursor_advance_kernel, dim3(blocks_of(S)), dim3(256), 0, (cudaStream_t)stream, cursors, S, T, stride, push);
  CVAD_LAUNCH_CHECK();
  return 0;
}

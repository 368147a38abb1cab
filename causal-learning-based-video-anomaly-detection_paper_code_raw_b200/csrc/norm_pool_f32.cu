// BatchNorm (2-D/3-D, training and inference), max / adaptive-average pooling -- fp32, NC(D)HW-contiguous.
//
// Bandwidth kernels (K3/K5 of SURVEY.md 2.5): cad:116-153 (BatchNorm2d + ReLU + MaxPool2d(3,2,1) + AdaptiveAvgPool2d),
// mc3:39-56 (BatchNorm3d + ReLU + MaxPool3d + global average), s2:23 (AdaptiveAvgPool3d((4,4,4))),
// cad1:132-147 (BatchNorm2d + LeakyReLU(0.1)).  Statistics are accumulated in fp64 so that inputs in the
// reference's [-1, 509] range (cad:96) do not lose the variance to cancellation.
#include "common.cuh"
#include "cvad_b200.h"

namespace {

// ---------------------------------------------------------------------------------------- BN statistics
// grid (chunks, C).  ws[0..C) += sum x, ws[C..2C) += sum x^2  (fp64 atomics)
__global__ void bn_stats_kernel(const float* __restrict__ x, int N, int C, long long S, double* __restrict__ ws) {
  __shared__ double sh[32];
  const int c = blockIdx.y;
  const long long per_n = S;
  const long long total = (long long)N * per_n;
  const long long chunk = (total + gridDim.x - 1) / gridDim.x;
  const long long beg = blockIdx.x * chunk;
  const long long end = beg + chunk < total ? beg + chunk : total;
  double s = 0.0, ss = 0.0;
  for (long long i = beg + threadIdx.x; i < end; i += blockDim.x) {
    long long n = i / per_n, sp = i - n * per_n;
    float v = __ldg(x + ((long long)n * C + c) * S + sp);
    s += v;
    ss += (double)v * v;
  }
  s = block_sum_d(s, sh);
  ss = block_sum_d(ss, sh);
  if (threadIdx.x == 0 && beg < end) {
    atomicAdd(ws + c, s);
    atomicAdd(ws + C + c, ss);
  }
}

// One thread per channel: the forward finalize of every BatchNorm of the library (fp32, bf16 backbone, stems); ws re-zeroed.
__global__ void bn_finalize_kernel(double* __restrict__ ws, int C, double count, const float* __restrict__ shift, float eps, float momentum,
                                   float* __restrict__ mean, float* __restrict__ invstd, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, long long* __restrict__ num_batches_tracked) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    bn_finalize_channel(ws, C, c, count, shift, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked);
    ws[c] = 0.0;
    ws[C + c] = 0.0;
  }
}

__global__ void bn_eval_prepare_kernel(int C, float eps, const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                       float* __restrict__ mean, float* __restrict__ invstd) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    mean[c] = running_mean[c];
    invstd[c] = 1.f / sqrtf(running_var[c] + eps);
  }
}

// y = act((x - mean) * invstd * gamma + beta).  grid.x strides over the N*C planes, grid.y splits a plane into chunks (a few long planes --
// M-C at T = 256 has 32 planes of 4 MB -- must still fill the machine); 16-byte accesses when the plane size and pointers allow.
__global__ void bn_apply_kernel(const float* __restrict__ x, float* __restrict__ y, long long planes, int C, long long S,
                                const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma,
                                const float* __restrict__ beta, int act, int vec4) {
  for (long long p = blockIdx.x; p < planes; p += gridDim.x) {
    int c = (int)(p % C);
    float sc = invstd[c] * gamma[c];
    float sh = beta[c] - mean[c] * sc;
    const float* xp = x + p * S;
    float* yp = y + p * S;
    if (vec4) {
      const long long S4 = S >> 2;
      for (long long i = blockIdx.y * (long long)blockDim.x + threadIdx.x; i < S4; i += (long long)gridDim.y * blockDim.x) {
        float4 v = __ldg(reinterpret_cast<const float4*>(xp) + i);
        v.x = cvad_act(fmaf(v.x, sc, sh), act); v.y = cvad_act(fmaf(v.y, sc, sh), act);
        v.z = cvad_act(fmaf(v.z, sc, sh), act); v.w = cvad_act(fmaf(v.w, sc, sh), act);
        reinterpret_cast<float4*>(yp)[i] = v;
      }
    } else {
      for (long long i = blockIdx.y * (long long)blockDim.x + threadIdx.x; i < S; i += (long long)gridDim.y * blockDim.x)
        yp[i] = cvad_act(fmaf(xp[i], sc, sh), act);
    }
  }
}

// backward pass 1: g = dy * act'(pre); ws[c] += sum g ; ws[C+c] += sum g * xhat
// derivative of the activation expressed through its PRE-activation value
__device__ __forceinline__ float act_grad_from_pre(float pre, int act) {
  switch (act) {
    case ACT_RELU: return pre > 0.f ? 1.f : 0.f;
    case ACT_LEAKY01: return pre > 0.f ? 1.f : 0.1f;
    case ACT_SIGMOID: { const float sg = 1.f / (1.f + expf(-pre)); return sg * (1.f - sg); }
    case ACT_TANH: { const float th = tanhf(pre); return 1.f - th * th; }
    default: return 1.f;
  }
}

__global__ void bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ x, int N, int C, long long S,
                                     const float* __restrict__ mean, const float* __restrict__ invstd, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, int act, double* __restrict__ ws) {
  __shared__ double sh[32];
  const int c = blockIdx.y;
  const long long total = (long long)N * S;
  const long long chunk = (total + gridDim.x - 1) / gridDim.x;
  const long long beg = blockIdx.x * chunk;
  const long long end = beg + chunk < total ? beg + chunk : total;
  const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c];
  double s = 0.0, sx = 0.0;
  for (long long i = beg + threadIdx.x; i < end; i += blockDim.x) {
    long long n = i / S, sp = i - n * S;
    long long off = ((long long)n * C + c) * S + sp;
    float xh = (__ldg(x + off) - mu) * is;
    float pre = fmaf(xh, ga, be);
    float g = __ldg(dy + off) * act_grad_from_pre(pre, act);
    s += g;
    sx += (double)g * xh;
  }
  s = block_sum_d(s, sh);
  sx = block_sum_d(sx, sh);
  if (threadIdx.x == 0 && beg < end) {
    atomicAdd(ws + c, s);
    atomicAdd(ws + C + c, sx);
  }
}

// backward pass 2: dx = gamma*invstd*(g - sum_g/cnt - xhat*sum_gx/cnt)   (training statistics)
//                  dx = gamma*invstd*g                                   (frozen / inference statistics)
// block (0,*) of the first plane loop also emits dgamma / dbeta (accumulating) -- done by a separate tiny kernel below.
__global__ void bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x, float* __restrict__ dx, long long planes,
                                    int C, long long S, const float* __restrict__ mean, const float* __restrict__ invstd,
                                    const float* __restrict__ gamma, const float* __restrict__ beta, int act,
                                    const double* __restrict__ ws, double count, int training) {
  for (long long p = blockIdx.x; p < planes; p += gridDim.x) {
    int c = (int)(p % C);
    const float mu = mean[c], is = invstd[c], ga = gamma[c], be = beta[c];
    const float mg = training ? (float)(ws[c] / count) : 0.f;
    const float mgx = training ? (float)(ws[C + c] / count) : 0.f;
    const float k = ga * is;
    const float* xp = x + p * S;
    const float* gp = dy + p * S;
    float* dp = dx + p * S;
    for (long long i = blockIdx.y * (long long)blockDim.x + threadIdx.x; i < S; i += (long long)gridDim.y * blockDim.x) {
      float xh = (xp[i] - mu) * is;
      float pre = fmaf(xh, ga, be);
      const float g = gp[i] * act_grad_from_pre(pre, act);
      dp[i] = k * (g - mg - xh * mgx);
    }
  }
}

// the backward's parameter-gradient update, for the fp32 and the bf16 backbone BatchNorms alike; ws re-zeroed
__global__ void bn_bwd_params_kernel(double* __restrict__ ws, int C, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    bn_params_channel(ws, C, c, dgamma, dbeta);
    ws[c] = 0.0;
    ws[C + c] = 0.0;
  }
}

// ---------------------------------------------------------------------------------------- max pooling
struct PoolGeo {
  int D, H, W, OD, OH, OW, kD, kH, kW, sD, sH, sW, pD, pH, pW;
};

__global__ void maxpool_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int* __restrict__ idx, long long planes, PoolGeo g) {
  const long long osz = (long long)g.OD * g.OH * g.OW;
  const long long total = planes * osz;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long p = t / osz;
    int r = (int)(t - p * osz);
    int ow = r % g.OW; r /= g.OW;
    int oh = r % g.OH;
    int od = r / g.OH;
    const float* xp = x + p * (long long)g.D * g.H * g.W;
    float best = -INFINITY;
    int bi = -1;
    for (int a = 0; a < g.kD; ++a) {
      int id = od * g.sD - g.pD + a;
      if ((unsigned)id >= (unsigned)g.D) continue;
      for (int b = 0; b < g.kH; ++b) {
        int ih = oh * g.sH - g.pH + b;
        if ((unsigned)ih >= (unsigned)g.H) continue;
        for (int c = 0; c < g.kW; ++c) {
          int iw = ow * g.sW - g.pW + c;
          if ((unsigned)iw >= (unsigned)g.W) continue;
          int ii = (id * g.H + ih) * g.W + iw;
          float v = __ldg(xp + ii);
          if (bi < 0) bi = ii;                  // torch seeds the index with the window's first element
          if (v > best || v != v) {             // first max wins; NaN propagates (torch semantics)
            best = v;
            bi = ii;
          }
        }
      }
    }
    y[t] = best;
    if (idx) idx[t] = bi;
  }
}

__global__ void maxpool_bwd_kernel(const float* __restrict__ dy, const int* __restrict__ idx, float* __restrict__ dx, long long planes,
                                   long long isz, long long osz) {
  const long long total = planes * osz;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long p = t / osz;
    int ii = idx[t];
    if (ii >= 0) atomicAdd(dx + p * isz + ii, dy[t]);
  }
}

// ---------------------------------------------------------------------------------------- adaptive average pooling
__device__ __forceinline__ int bin_start(int o, int in, int out) { return (int)(((long long)o * in) / out); }
__device__ __forceinline__ int bin_end(int o, int in, int out) { return (int)((((long long)(o + 1)) * in + out - 1) / out); }

__global__ void adaptive_avgpool_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long planes, int D, int H, int W,
                                            int OD, int OH, int OW) {
  const long long osz = (long long)OD * OH * OW;
  const long long total = planes * osz;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long p = t / osz;
    int r = (int)(t - p * osz);
    int ow = r % OW; r /= OW;
    int oh = r % OH;
    int od = r / OH;
    int d0 = bin_start(od, D, OD), d1 = bin_end(od, D, OD);
    int h0 = bin_start(oh, H, OH), h1 = bin_end(oh, H, OH);
    int w0 = bin_start(ow, W, OW), w1 = bin_end(ow, W, OW);
    const float* xp = x + p * (long long)D * H * W;
    float s = 0.f;
    for (int a = d0; a < d1; ++a)
      for (int b = h0; b < h1; ++b)
        for (int c = w0; c < w1; ++c) s += __ldg(xp + ((long long)a * H + b) * W + c);
    y[t] = s / (float)((d1 - d0) * (h1 - h0) * (w1 - w0));
  }
}

// the same with one CTA per output bin: large bins (M-C's global pooling over T/4 x 8 x 8 = up to 4096 elements, mc3:56) as a block reduction
__global__ void __launch_bounds__(256) adaptive_avgpool_fwd_bin_kernel(const float* __restrict__ x, float* __restrict__ y, long long planes, int D,
                                                                       int H, int W, int OD, int OH, int OW) {
  __shared__ float sh[32];
  const long long osz = (long long)OD * OH * OW;
  const long long total = planes * osz;
  for (long long t = blockIdx.x; t < total; t += gridDim.x) {
    long long p = t / osz;
    int r = (int)(t - p * osz);
    int ow = r % OW; r /= OW;
    int oh = r % OH;
    int od = r / OH;
    const int d0 = bin_start(od, D, OD), d1 = bin_end(od, D, OD);
    const int h0 = bin_start(oh, H, OH), h1 = bin_end(oh, H, OH);
    const int w0 = bin_start(ow, W, OW), w1 = bin_end(ow, W, OW);
    const int bw = w1 - w0, bh = h1 - h0, n = (d1 - d0) * bh * bw;
    const float* xp = x + p * (long long)D * H * W;
    float s = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int c = i % bw, q = i / bw, b = q % bh, a = q / bh;
      s += __ldg(xp + ((long long)(d0 + a) * H + (h0 + b)) * W + (w0 + c));
    }
    s = block_sum(s, sh);
    if (threadIdx.x == 0) y[t] = s / (float)n;
    __syncthreads();
  }
}

// gather form: each input element sums the (possibly overlapping) bins that contain it
__global__ void adaptive_avgpool_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, long long planes, int D, int H, int W,
                                            int OD, int OH, int OW) {
  const long long isz = (long long)D * H * W;
  const long long osz = (long long)OD * OH * OW;
  const long long total = planes * isz;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long p = t / isz;
    int r = (int)(t - p * isz);
    int iw = r % W; r /= W;
    int ih = r % H;
    int id = r / H;
    const float* gp = dy + p * osz;
    float s = 0.f;
    for (int a = 0; a < OD; ++a) {
      int d0 = bin_start(a, D, OD), d1 = bin_end(a, D, OD);
      if (id < d0 || id >= d1) continue;
      for (int b = 0; b < OH; ++b) {
        int h0 = bin_start(b, H, OH), h1 = bin_end(b, H, OH);
        if (ih < h0 || ih >= h1) continue;
        for (int c = 0; c < OW; ++c) {
          int w0 = bin_start(c, W, OW), w1 = bin_end(c, W, OW);
          if (iw < w0 || iw >= w1) continue;
          s += __ldg(gp + ((long long)a * OH + b) * OW + c) / (float)((d1 - d0) * (h1 - h0) * (w1 - w0));
        }
      }
    }
    dx[t] = s;
  }
}

// mean over the middle axis: x (A, T, F) -> y (A, F)  (cad:568 temporal mean of backbone features) and its gradient
__global__ void mean_mid_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, long long A, int T, long long F) {
  cvad_pdl_enter();
  long long total = A * F;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long a = t / F, f = t - a * F;
    float s = 0.f;
    for (int k = 0; k < T; ++k) s += __ldg(x + (a * T + k) * F + f);
    y[t] = s / (float)T;
  }
}
__global__ void mean_mid_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, long long A, int T, long long F, int accumulate) {
  cvad_pdl_enter();
  long long total = A * T * F;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    long long f = t % F, a = t / (F * T);
    float v = __ldg(dy + a * F + f) / (float)T;
    dx[t] = accumulate ? dx[t] + v : v;
  }
}

// out[c] += sum over (n, s) of x[n][c][s]   (conv bias gradients); grid (chunks, C)
__global__ void channel_sum_add_kernel(const float* __restrict__ x, int N, int C, long long S, float* __restrict__ out) {
  __shared__ float sh[32];
  const int c = blockIdx.y;
  const long long total = (long long)N * S;
  const long long chunk = (total + gridDim.x - 1) / gridDim.x;
  const long long beg = blockIdx.x * chunk;
  const long long end = beg + chunk < total ? beg + chunk : total;
  float s = 0.f;
  for (long long i = beg + threadIdx.x; i < end; i += blockDim.x) {
    long long n = i / S, sp = i - n * S;
    s += __ldg(x + ((long long)n * C + c) * S + sp);
  }
  s = block_sum(s, sh);
  if (threadIdx.x == 0 && beg < end) atomicAdd(out + c, s);
}

// chunks per plane (grid.y) so that planes x chunks CTAs cover the machine ~8 times, each chunk at least `min_elems` elements
inline int plane_chunks(int plane_blocks, long long S, int min_elems) {
  long long want = (8LL * cvad_num_sms() + plane_blocks - 1) / plane_blocks;
  long long most = (S + min_elems - 1) / min_elems;
  long long c = want < most ? want : most;
  return (int)(c < 1 ? 1 : (c > 65535 ? 65535 : c));
}

inline int ew_blocks(long long n) {
  long long b = (n + 255) / 256;
  long long cap = 16LL * cvad_num_sms();
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

int bn_finalize_launch(double* ws, int C, double count, const float* shift, float eps, float momentum, float* mean, float* invstd,
                       float* running_mean, float* running_var, long long* nbt, cudaStream_t st) {
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(ws, C, count, shift, eps, momentum, mean, invstd, running_mean, running_var, nbt);
  CVAD_LAUNCH_CHECK();
  return 0;
}

int bn_params_launch(double* ws, int C, float* dgamma, float* dbeta, cudaStream_t st) {
  bn_bwd_params_kernel<<<(C + 127) / 128, 128, 0, st>>>(ws, C, dgamma, dbeta);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_bn_train_stats_f32(const float* x, int N, int C, long long S, double* ws, float eps, float momentum, float* mean,
                                     float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked,
                                     void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  long long total = (long long)N * S;
  int chunks = (int)((total + 8191) / 8192);
  int maxc = (8 * cvad_num_sms() + C - 1) / C;
  if (chunks > maxc) chunks = maxc;
  if (chunks < 1) chunks = 1;
  bn_stats_kernel<<<dim3(chunks, C), 256, 0, st>>>(x, N, C, S, ws);
  CVAD_LAUNCH_CHECK();
  return bn_finalize_launch(ws, C, (double)total, nullptr, eps, momentum, mean, invstd, running_mean, running_var, num_batches_tracked, st);
}

CVAD_API int cvad_bn_eval_prepare_f32(int C, float eps, const float* running_mean, const float* running_var, float* mean, float* invstd,
                                      void* stream) {
  bn_eval_prepare_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(C, eps, running_mean, running_var, mean, invstd);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_bn_apply_f32(const float* x, float* y, int N, int C, long long S, const float* mean, const float* invstd,
                               const float* gamma, const float* beta, int act, void* stream) {
  long long planes = (long long)N * C;
  int blocks = (int)(planes < 8LL * cvad_num_sms() ? planes : 8LL * cvad_num_sms());
  int threads = S >= 1024 ? 256 : (S >= 128 ? 128 : 32);
  const int vec4 = (S % 4 == 0) && ((((uintptr_t)x | (uintptr_t)y) & 15) == 0);
  bn_apply_kernel<<<dim3(blocks, plane_chunks(blocks, S, threads * (vec4 ? 16 : 4))), threads, 0, (cudaStream_t)stream>>>(
      x, y, planes, C, S, mean, invstd, gamma, beta, act, vec4);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_bn_bwd_f32(const float* dy, const float* x, float* dx, int N, int C, long long S, const float* mean,
                             const float* invstd, const float* gamma, const float* beta, int act, int training, double* ws,
                             float* dgamma, float* dbeta, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  long long total = (long long)N * S;
  int chunks = (int)((total + 8191) / 8192);
  int maxc = (8 * cvad_num_sms() + C - 1) / C;
  if (chunks > maxc) chunks = maxc;
  if (chunks < 1) chunks = 1;
  bn_bwd_reduce_kernel<<<dim3(chunks, C), 256, 0, st>>>(dy, x, N, C, S, mean, invstd, gamma, beta, act, ws);
  CVAD_LAUNCH_CHECK();
  if (dx) {
    long long planes = (long long)N * C;
    int blocks = (int)(planes < 8LL * cvad_num_sms() ? planes : 8LL * cvad_num_sms());
    int threads = S >= 1024 ? 256 : (S >= 128 ? 128 : 32);
    bn_bwd_apply_kernel<<<dim3(blocks, plane_chunks(blocks, S, threads * 4)), threads, 0, st>>>(dy, x, dx, planes, C, S, mean, invstd, gamma, beta,
                                                                                               act, ws, (double)total, training);
    CVAD_LAUNCH_CHECK();
  }
  return bn_params_launch(ws, C, dgamma, dbeta, st);
}

// Eval-mode BatchNorm folded into the convolution in front of it (SURVEY K5): w'[co][...] = w[co][...] * s, b' = (b - running_mean) * s + beta
// with s = gamma / sqrt(running_var + eps), so that conv + BN (+ ReLU in the convolution's epilogue) is ONE launch at inference.
__global__ void bn_fold_conv_kernel(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, const float* __restrict__ rm, const float* __restrict__ rv, float eps, int Cout,
                                    int per_out, float* __restrict__ w_out, float* __restrict__ b_out) {
  const int total = Cout * per_out;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int co = i / per_out;
    const float sc = gamma[co] * (1.f / sqrtf(rv[co] + eps));
    w_out[i] = w[i] * sc;
    if (i == co * per_out) b_out[co] = ((b ? b[co] : 0.f) - rm[co]) * sc + beta[co];
  }
}

CVAD_API int cvad_bn_fold_conv_f32(const float* w, const float* b, const float* gamma, const float* beta, const float* running_mean,
                                   const float* running_var, float eps, int Cout, int per_out, float* w_out, float* b_out, void* stream) {
  if (Cout <= 0 || per_out <= 0) return (int)cudaErrorInvalidValue;
  const int total = Cout * per_out;
  bn_fold_conv_kernel<<<(total + 255) / 256 < 1024 ? (total + 255) / 256 : 1024, 256, 0, (cudaStream_t)stream>>>(w, b, gamma, beta, running_mean,
                                                                                                              running_var, eps, Cout, per_out,
                                                                                                              w_out, b_out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_channel_sum_add_f32(const float* x, int N, int C, long long S, float* out, void* stream) {
  long long total = (long long)N * S;
  if (total <= 0 || C <= 0) return 0;
  int chunks = (int)((total + 16383) / 16384);
  int maxc = (4 * cvad_num_sms() + C - 1) / C;
  if (chunks > maxc) chunks = maxc;
  if (chunks < 1) chunks = 1;
  channel_sum_add_kernel<<<dim3(chunks, C), 256, 0, (cudaStream_t)stream>>>(x, N, C, S, out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_maxpool_fwd_f32(const float* x, float* y, int* idx, long long planes, int D, int H, int W, int OD, int OH, int OW,
                                  int kD, int kH, int kW, int sD, int sH, int sW, int pD, int pH, int pW, void* stream) {
  PoolGeo g{D, H, W, OD, OH, OW, kD, kH, kW, sD, sH, sW, pD, pH, pW};
  long long total = planes * OD * OH * OW;
  if (total <= 0) return 0;
  maxpool_fwd_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(x, y, idx, planes, g);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_maxpool_bwd_f32(const float* dy, const int* idx, float* dx, long long planes, long long in_size, long long out_size,
                                  void* stream) {
  // dx must be zero-initialised by the caller
  long long total = planes * out_size;
  if (total <= 0) return 0;
  maxpool_bwd_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(dy, idx, dx, planes, in_size, out_size);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_adaptive_avgpool_fwd_f32(const float* x, float* y, long long planes, int D, int H, int W, int OD, int OH, int OW,
                                           void* stream) {
  long long total = planes * OD * OH * OW;
  if (total <= 0) return 0;
  const long long bin = ((long long)(D + OD - 1) / OD) * ((H + OH - 1) / OH) * ((W + OW - 1) / OW);
  if (bin >= 256 && total <= 16LL * cvad_num_sms() * 8)      // few, large bins: one CTA per bin
    adaptive_avgpool_fwd_bin_kernel<<<(unsigned)(total < 16LL * cvad_num_sms() ? total : 16LL * cvad_num_sms()), 256, 0, (cudaStream_t)stream>>>(
        x, y, planes, D, H, W, OD, OH, OW);
  else
    adaptive_avgpool_fwd_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(x, y, planes, D, H, W, OD, OH, OW);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_adaptive_avgpool_bwd_f32(const float* dy, float* dx, long long planes, int D, int H, int W, int OD, int OH, int OW,
                                           void* stream) {
  long long total = planes * D * H * W;
  if (total <= 0) return 0;
  adaptive_avgpool_bwd_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(dy, dx, planes, D, H, W, OD, OH, OW);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_mean_mid_fwd_f32(const float* x, float* y, long long A, int T, long long F, void* stream) {
  if (A * F <= 0) return 0;
  cvad_launch_pdl(mean_mid_fwd_kernel, dim3(ew_blocks(A * F)), dim3(256), 0, (cudaStream_t)stream, x, y, A, T, F);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_mean_mid_bwd_f32(const float* dy, float* dx, long long A, int T, long long F, int accumulate, void* stream) {
  if (A * F * T <= 0) return 0;
  cvad_launch_pdl(mean_mid_bwd_kernel, dim3(ew_blocks(A * T * F)), dim3(256), 0, (cudaStream_t)stream, dy, dx, A, T, F, accumulate);
  CVAD_LAUNCH_CHECK();
  return 0;
}

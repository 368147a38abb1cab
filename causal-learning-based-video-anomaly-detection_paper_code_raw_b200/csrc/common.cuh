// Shared device helpers for the cvad_b200 kernels (sm_100a only).
#pragma once
#include <cstdlib>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define CVAD_API extern "C" __attribute__((visibility("default")))

// Every entry point returns 0 on success or the cudaError_t of the failed launch.
#define CVAD_LAUNCH_CHECK()                         \
  do {                                              \
    cudaError_t e__ = cudaGetLastError();           \
    if (e__ != cudaSuccess) return (int)e__;        \
  } while (0)

enum CvadAct { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY01 = 2, ACT_SIGMOID = 3, ACT_TANH = 4 };

__device__ __forceinline__ float cvad_act(float v, int act) {
  switch (act) {
    case ACT_RELU: return v > 0.f ? v : 0.f;
    case ACT_LEAKY01: return v > 0.f ? v : 0.1f * v;
    case ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    case ACT_TANH: return tanhf(v);
    default: return v;
  }
}

// derivative of the activation expressed through its OUTPUT y
__device__ __forceinline__ float cvad_act_grad_from_out(float y, int act) {
  switch (act) {
    case ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case ACT_LEAKY01: return y > 0.f ? 1.f : 0.1f;
    case ACT_SIGMOID: return y * (1.f - y);
    case ACT_TANH: return 1.f - y * y;
    default: return 1.f;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// block-wide sum (blockDim.x <= 1024, multiple of 32); result valid in every thread
__device__ __forceinline__ float block_sum(float v, float* sh /* >=32 floats */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  float r = (lane < nw) ? sh[lane] : 0.f;
  r = warp_sum(r);
  return r;
}
__device__ __forceinline__ double block_sum_d(double v, double* sh /* >=32 doubles */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum_d(v);
  __syncthreads();
  if (lane == 0) sh[wid] = v;
  __syncthreads();
  const int nw = (blockDim.x + 31) >> 5;
  double r = (lane < nw) ? sh[lane] : 0.0;
  r = warp_sum_d(r);
  return r;
}

// x / d for a launch constant d and 0 <= x < 2^31 as umulhi(x, mul) >> shr (mul = 0 encodes d = 1), instead of the ~20-instruction
// emulated divide: mul = ceil(2^(31 + ceil(log2 d)) / d), shr = ceil(log2 d) - 1
static inline void fast_div_init(unsigned d, unsigned& mul, unsigned& shr) {
  if (d <= 1) { mul = 0; shr = 0; return; }
  unsigned lg = 0;
  while ((1u << lg) < d) ++lg;
  const unsigned p = 31 + lg;
  mul = (unsigned)(((1ull << p) + d - 1) / d);
  shr = p - 32;
}
__device__ __forceinline__ int fast_div(int x, unsigned mul, unsigned shr) { return mul ? (int)(__umulhi((unsigned)x, mul) >> shr) : x; }

// The window rule of S streams that share one push (bbox:392-430 as a service, one stream per camera or video), shared by the feature
// rings of ma0_tail.cu and the frame rings of frames.cu.  Stream k's cursor cursors[k] = {frames pushed, next window}; its entry of the
// push descriptor push[k] = {count, reset}:
//   base   = reset ? 0 : cursors[k][0]        frames   = base + count
//   next   = reset ? 0 : cursors[k][1]        n_win    = frames >= T ? (frames - T) / stride + 1 - next : 0
// infer.window_count is the host's copy of this rule.
struct StreamPush {
  long long base, next, frames, n_win;
};

__device__ __forceinline__ StreamPush stream_push(const long long* __restrict__ cursors, const long long* __restrict__ push, int k, int T,
                                                  int stride) {
  const bool reset = push[2 * k + 1] != 0;
  StreamPush p;
  p.base = reset ? 0 : cursors[2 * k];
  p.next = reset ? 0 : cursors[2 * k + 1];
  p.frames = p.base + push[2 * k];
  p.n_win = p.frames >= T ? (p.frames - T) / stride + 1 - p.next : 0;
  return p;
}

static inline bool cvad_pdl_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("CVAD_PDL");
    on = (e && e[0] == '0') ? 0 : 1;
  }
  return on == 1;
}

// ---- programmatic dependent launch (PDL) for the chains of small, latency-bound kernels of the dense tail.
// A kernel launched through cvad_launch_pdl may be scheduled while its stream predecessor is still running; cvad_pdl_enter() -- the
// FIRST statement of such a kernel, before any global-memory access -- (1) lets the kernel's own successor be scheduled as soon as
// every CTA of this grid has started, and (2) blocks until all prerequisite grids have completed and their writes are visible.
// The data dependence is unchanged; what disappears is the ~2 us scheduling gap between dependent launches (also inside a captured
// CUDA graph, where the launches become programmatic edges).  Predecessors that never trigger simply release at completion.
__device__ __forceinline__ void cvad_pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <typename... KArgs, typename... Args>
static inline cudaError_t cvad_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = cvad_pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

static inline int cvad_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }
// Per-DEVICE host-side caches: function attributes (cudaFuncAttributeMaxDynamicSharedMemorySize) and the SM count belong to the current
// device, and one process may drive several GPUs (tests on cuda:1, single-process inference sharding), so nothing is cached per process.
constexpr int CVAD_MAX_DEVICES = 64;
static inline int cvad_current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev >= 0 && dev < CVAD_MAX_DEVICES ? dev : 0;
}
static inline int cvad_num_sms() {
  static int sms[CVAD_MAX_DEVICES] = {};
  const int dev = cvad_current_device();
  if (!sms[dev]) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    sms[dev] = n > 0 ? n : 148;
  }
  return sms[dev];
}
// Raise a kernel's dynamic shared-memory limit on the current device when `smem` exceeds what was configured there before.
template <typename Kernel>
static inline cudaError_t cvad_ensure_dyn_smem(Kernel kernel, size_t smem, size_t (&configured)[CVAD_MAX_DEVICES]) {
  const int dev = cvad_current_device();
  if (smem <= configured[dev]) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess) configured[dev] = smem;
  return e;
}

// ---- BatchNorm statistics.  Every BatchNorm reduction leaves per-channel fp64 sums in a 2*C workspace: ws[c] = sum y, ws[C + c] = sum y^2
// in the forward pass, ws[c] = sum g, ws[C + c] = sum g*xhat in the backward pass.  The helpers below are the one place that turns those
// sums into batch statistics and parameter gradients; whoever calls them re-zeroes ws afterwards.

// Batch mean and biased variance of channel c over `count` values.  shift (nullptr = none): the sums were taken over y - shift[c] (the
// stems sum their raw accumulator, before the conv bias), which moves the mean and leaves the variance.
struct BnBatchStat { double mean, var; };
__device__ __forceinline__ BnBatchStat bn_batch_stat(const double* ws, int C, int c, double count, const float* shift) {
  const double m = ws[c] / count;
  double var = ws[C + c] / count - m * m;
  if (var < 0.0) var = 0.0;
  return {shift ? m + (double)shift[c] : m, var};
}
__device__ __forceinline__ float bn_invstd(const BnBatchStat& s, float eps) { return (float)(1.0 / sqrt(s.var + (double)eps)); }

// Forward finalize of channel c: mean / invstd for the apply and backward passes, the momentum update of the running statistics (with the
// unbiased variance, as torch) when running_mean is non-null, and num_batches_tracked += 1 by channel 0 when nbt is non-null.
__device__ __forceinline__ void bn_finalize_channel(const double* ws, int C, int c, double count, const float* shift, float eps, float momentum,
                                                    float* mean, float* invstd, float* running_mean, float* running_var, long long* nbt) {
  const BnBatchStat s = bn_batch_stat(ws, C, c, count, shift);
  mean[c] = (float)s.mean;
  invstd[c] = bn_invstd(s, eps);
  if (running_mean) {
    const double unbiased = count > 1.0 ? s.var * count / (count - 1.0) : s.var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)s.mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
  if (c == 0 && nbt) *nbt += 1;
}

// Backward parameter update of channel c: dgamma += sum g*xhat, dbeta += sum g, each only when non-null.
__device__ __forceinline__ void bn_params_channel(const double* ws, int C, int c, float* dgamma, float* dbeta) {
  if (dgamma) dgamma[c] += (float)ws[C + c];
  if (dbeta) dbeta[c] += (float)ws[c];
}

// One launch of the finalize / parameter-update kernel over channels [0, C), which then re-zeroes ws[0, 2C) (norm_pool_f32.cu; library
// internal, not exported).  Return 0 or the launch error.
int bn_finalize_launch(double* ws, int C, double count, const float* shift, float eps, float momentum, float* mean, float* invstd,
                       float* running_mean, float* running_var, long long* nbt, cudaStream_t st);
int bn_params_launch(double* ws, int C, float* dgamma, float* dbeta, cudaStream_t st);

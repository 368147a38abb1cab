// Frame preparation on the device (SURVEY.md 8(f1)): what the reference's loaders do per frame on the host with OpenCV --
//   cv2.resize(frame, (360, 240)) on grayscale uint8 frames                     causal_anomaly_detection.py:89-96  (then Normalize, fused into the stem)
//   cv2.resize(img, frame_size) + BGR->RGB + /255 + (T,H,W,3)->(3,T,H,W)        avenue loaders (s1:19, 86-92; bbox:397-411)
// so that a video is uploaded ONCE as raw uint8 frames and every clip / sliding window is cut, resized and laid out where the model
// reads it, instead of crossing PCIe as fp32 per clip.
//
// cvad_resize_bilinear_u8 reproduces cv2.resize(..., interpolation=INTER_LINEAR) for 8-bit images BIT-EXACTLY: OpenCV's fixed-point
// scheme -- 11-bit coefficients saturate_cast<short>(w * 2048) from fx = (float)((dx + 0.5) * scale - 0.5), horizontal pass in int32,
// vertical pass ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2 -- including its asymmetric border rules (columns: the
// fraction is zeroed when the tap is clamped; rows: only the tap index is clamped).
#include "common.cuh"
#include "cvad_b200.h"

namespace {

struct Tap {
  int i0, i1, w0, w1;
};

__device__ __forceinline__ Tap make_tap(int d, int src, double scale, bool zero_frac_when_clamped) {
  float f = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= (float)s;
  if (zero_frac_when_clamped) {
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= src - 1) { f = 0.f; s = src - 1; }
  }
  Tap t;
  t.i0 = min(max(s, 0), src - 1);
  t.i1 = min(max(s + 1, 0), src - 1);
  t.w0 = __float2int_rn((1.f - f) * 2048.f);
  t.w1 = __float2int_rn(f * 2048.f);
  return t;
}

// cv2.resize(INTER_LINEAR) of pixel (dx, dy) of frame `frame` of src (.., sh, sw, C) into pixel `pix` of dst (.., C): the taps, then the
// fixed-point blend.
__device__ __forceinline__ void resize_pixel_u8(const uint8_t* src, long long frame, int sh, int sw, int C, int dx, int dy, double scale_x,
                                                double scale_y, uint8_t* dst, long long pix) {
  const Tap tx = make_tap(dx, sw, scale_x, true), ty = make_tap(dy, sh, scale_y, false);
  const uint8_t* f = src + frame * sh * sw * C;
  const uint8_t* r0 = f + (long long)ty.i0 * sw * C;
  const uint8_t* r1 = f + (long long)ty.i1 * sw * C;
  uint8_t* o = dst + pix * C;
  for (int c = 0; c < C; ++c) {
    const int s0 = (int)__ldg(r0 + tx.i0 * C + c) * tx.w0 + (int)__ldg(r0 + tx.i1 * C + c) * tx.w1;
    const int s1 = (int)__ldg(r1 + tx.i0 * C + c) * tx.w0 + (int)__ldg(r1 + tx.i1 * C + c) * tx.w1;
    const int v = (((ty.w0 * (s0 >> 4)) >> 16) + ((ty.w1 * (s1 >> 4)) >> 16) + 2) >> 2;
    o[c] = (uint8_t)min(max(v, 0), 255);
  }
}

// src (N, sh, sw, C) uint8 interleaved -> dst (N, dh, dw, C) uint8
__global__ void resize_bilinear_u8_kernel(const uint8_t* __restrict__ src, int N, int sh, int sw, int C, uint8_t* __restrict__ dst, int dh, int dw,
                                          double scale_x, double scale_y) {
  const long long total = (long long)N * dh * dw;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int dx = (int)(t % dw);
    const long long r = t / dw;
    const int dy = (int)(r % dh), n = (int)(r / dh);
    resize_pixel_u8(src, n, sh, sw, C, dx, dy, scale_x, scale_y, dst, t);
  }
}

// Frame rings of S streams (the window rule is stream_push, common.cuh).  src (S*n, sh, sw, C), stream-major: row r < count_k of stream k
// is resized to (dh, dw) into rings[k][(base_k + r) % cap] (rings (S, cap, dh, dw, C)); rows r >= count_k are not read.  At the ring's
// own size the resize rule is the identity and the frame is copied.
__global__ void streams_frame_write_u8_kernel(const uint8_t* __restrict__ src, int S, long long n, int sh, int sw, int C, uint8_t* __restrict__ rings,
                                              long long cap, int dh, int dw, int T, int stride, const long long* __restrict__ cursors,
                                              const long long* __restrict__ push, double scale_x, double scale_y) {
  const long long hw = (long long)dh * dw;
  const long long total = S * n * hw;
  const bool copy = sh == dh && sw == dw;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long row = t / hw, p = t - row * hw;
    const int k = (int)(row / n);
    const long long r = row - k * n;
    if (r >= push[2 * k]) continue;
    const StreamPush sp = stream_push(cursors, push, k, T, stride);
    const long long pix = (k * cap + (sp.base + r) % cap) * hw + p;
    if (copy) {
      for (int c = 0; c < C; ++c) rings[pix * C + c] = __ldg(src + t * C + c);
    } else {
      resize_pixel_u8(src, row, sh, sw, C, (int)(p % dw), (int)(p / dw), scale_x, scale_y, rings, pix);
    }
  }
}

// out (S*m, C, T, H, W) fp32: slot (k, j) = window next_k + j of stream k, frames ((next_k + j)*stride + [0, T)) % cap of its ring, as
// value * scale with channel C-1-c read for c when reverse_channels (the element rule of clips_from_frames_kernel); zeros for j >= n_win_k
__global__ void streams_clips_f32_kernel(const uint8_t* __restrict__ rings, int S, long long cap, int H, int W, int C, int T, int stride, long long m,
                                         const long long* __restrict__ cursors, const long long* __restrict__ push, float scale, int reverse_channels,
                                         float* __restrict__ out) {
  const long long hw = (long long)H * W;
  const long long total = S * m * C * T * hw;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long p = t % hw;
    long long r = t / hw;
    const int tt = (int)(r % T); r /= T;
    const int c = (int)(r % C);
    const long long slot = r / C;
    const int k = (int)(slot / m);
    const long long j = slot - k * m;
    const StreamPush sp = stream_push(cursors, push, k, T, stride);
    float v = 0.f;
    if (j < sp.n_win) {
      const long long fr = ((sp.next + j) * stride + tt) % cap;
      const int cs = reverse_channels ? C - 1 - c : c;
      v = (float)__ldg(rings + ((k * cap + fr) * hw + p) * C + cs) * scale;
    }
    out[t] = v;
  }
}

// frames (F, H, W, C) uint8 (C = 1 or 3) + clip starts -> clips (B, C, T, H, W) fp32 = value * scale, channel order optionally reversed
// (BGR -> RGB): the Avenue loaders' cvtColor + /255 + permute, and the sliding-window gather of bbox:392-411, in one pass.
__global__ void clips_from_frames_kernel(const uint8_t* __restrict__ frames, int F, int H, int W, int C, const int* __restrict__ starts, int B, int T,
                                         int frame_stride, float scale, int reverse_channels, float* __restrict__ out) {
  const long long hw = (long long)H * W;
  const long long total = (long long)B * C * T * hw;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long p = t % hw;
    long long r = t / hw;
    const int tt = (int)(r % T); r /= T;
    const int c = (int)(r % C);
    const int b = (int)(r / C);
    int fr = starts[b] + tt * frame_stride;
    fr = min(max(fr, 0), F - 1);
    const int cs = reverse_channels ? C - 1 - c : c;
    out[t] = (float)__ldg(frames + ((long long)fr * hw + p) * C + cs) * scale;
  }
}

// the same gather for the M-A input: clips (B, T, 1, H, W) uint8 from grayscale frames (F, H, W) (cad:57 sequence windows)
__global__ void clips_from_frames_u8_kernel(const uint8_t* __restrict__ frames, int F, long long hw, const int* __restrict__ starts, int B, int T,
                                            int frame_stride, uint8_t* __restrict__ out) {
  const long long total = (long long)B * T * hw;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long p = t % hw;
    const long long r = t / hw;
    const int tt = (int)(r % T), b = (int)(r / T);
    int fr = starts[b] + tt * frame_stride;
    fr = min(max(fr, 0), F - 1);
    out[t] = __ldg(frames + (long long)fr * hw + p);
  }
}

inline unsigned frame_blocks(long long n) {
  long long b = (n + 255) / 256;
  if (b < 1) b = 1;
  if (b > 16LL * cvad_num_sms()) b = 16LL * cvad_num_sms();
  return (unsigned)b;
}

// OpenCV: inv_scale = dsize / ssize (double); scale = 1. / inv_scale
inline double cv2_scale(int dst, int src) { return 1.0 / ((double)dst / src); }

}  // namespace

CVAD_API int cvad_resize_bilinear_u8(const void* src, int N, int src_h, int src_w, int C, void* dst, int dst_h, int dst_w, void* stream) {
  if (N <= 0) return 0;
  if (src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0 || C < 1 || C > 4) return (int)cudaErrorInvalidValue;
  resize_bilinear_u8_kernel<<<frame_blocks((long long)N * dst_h * dst_w), 256, 0, (cudaStream_t)stream>>>(
      (const uint8_t*)src, N, src_h, src_w, C, (uint8_t*)dst, dst_h, dst_w, cv2_scale(dst_w, src_w), cv2_scale(dst_h, src_h));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_clips_from_frames_f32(const void* frames, int F, int H, int W, int C, const int* starts, int B, int T, int frame_stride,
                                        float scale, int reverse_channels, float* out, void* stream) {
  if (B <= 0 || T <= 0) return 0;
  if (F <= 0 || H <= 0 || W <= 0 || C < 1 || C > 4) return (int)cudaErrorInvalidValue;
  clips_from_frames_kernel<<<frame_blocks((long long)B * C * T * H * W), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)frames, F, H, W, C, starts, B, T,
                                                                                                       frame_stride, scale, reverse_channels, out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_clips_from_frames_u8(const void* frames, int F, int H, int W, const int* starts, int B, int T, int frame_stride, void* out,
                                       void* stream) {
  if (B <= 0 || T <= 0) return 0;
  if (F <= 0 || H <= 0 || W <= 0) return (int)cudaErrorInvalidValue;
  clips_from_frames_u8_kernel<<<frame_blocks((long long)B * T * H * W), 256, 0, (cudaStream_t)stream>>>((const uint8_t*)frames, F, (long long)H * W, starts,
                                                                                                      B, T, frame_stride, (uint8_t*)out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_streams_frame_write_u8(const void* src, int S, long long n, int src_h, int src_w, int C, void* rings, long long capacity, int dst_h,
                                         int dst_w, int T, int stride, const long long* cursors, const long long* push, void* stream) {
  if (!src || !rings || !cursors || !push || S <= 0 || n < 0 || capacity <= 0 || T <= 0 || stride <= 0 || src_h <= 0 || src_w <= 0 || dst_h <= 0 ||
      dst_w <= 0 || C < 1 || C > 4)
    return (int)cudaErrorInvalidValue;
  if (n == 0) return 0;
  streams_frame_write_u8_kernel<<<frame_blocks(S * n * dst_h * dst_w), 256, 0, (cudaStream_t)stream>>>(
      (const uint8_t*)src, S, n, src_h, src_w, C, (uint8_t*)rings, capacity, dst_h, dst_w, T, stride, cursors, push, cv2_scale(dst_w, src_w),
      cv2_scale(dst_h, src_h));
  CVAD_LAUNCH_CHECK();
  return 0;
}

CVAD_API int cvad_streams_clips_f32(const void* rings, int S, long long capacity, int H, int W, int C, int T, int stride, long long m,
                                    const long long* cursors, const long long* push, float scale, int reverse_channels, float* out, void* stream) {
  if (!rings || !cursors || !push || !out || S <= 0 || m < 0 || capacity <= 0 || T <= 0 || stride <= 0 || H <= 0 || W <= 0 || C < 1 || C > 4)
    return (int)cudaErrorInvalidValue;
  if (m == 0) return 0;
  streams_clips_f32_kernel<<<frame_blocks(S * m * C * T * H * W), 256, 0, (cudaStream_t)stream>>>(
      (const uint8_t*)rings, S, capacity, H, W, C, T, stride, m, cursors, push, scale, reverse_channels, out);
  CVAD_LAUNCH_CHECK();
  return 0;
}

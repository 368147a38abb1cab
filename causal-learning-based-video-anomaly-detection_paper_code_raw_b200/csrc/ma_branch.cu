// M-A's causal branch behind the GRU (cad:300-502) as ONE kernel forward and ONE kernel backward: from the last GRU states hT to
// (z, kl, adj, causal) -- the trajectory encoder's output Linear, the factor MLP, the mu / log-variance heads with reparameterisation and
// KL, the node encoder, the edge MLP over track pairs, the adjacency, structured = adj z, the dynamics MLP, the scorer inputs, the three
// scorers (scorer0 dropout) and their 0.5 / 0.3 / 0.2 combination.
//
// Why: these 20 Linear layers hold ~13.5 k parameters and do ~0.1 MFLOP per clip, on 160..800 rows.  As separate launches the branch
// was a serial chain of ~12 dependent kernels forward and ~18 backward, plus ~45 beside them (the log-variance head, two scorers, one
// weight-gradient GEMM and one bias column sum per layer), every one a few KB through L2 -- and the whole chain sits on the critical path
// between the backbone's forward and its backward.  Here one CTA owns one clip at a time (the grid strides over clips: eval and
// streaming run B in the thousands), stages all parameters in shared memory before the programmatic-dependent-launch wait, and walks
// the layers with the clip's activations in shared memory, separated by __syncthreads only.  Only the nt live track rows and the
// nt (nt - 1) live edge pairs are computed: the rest contributed exact zeros before.
//
// The backward kernel recomputes the forward from (hT, eps, keep, ntr) -- nothing is saved between the two kernels -- and accumulates the
// parameter gradients of all clips it owns in shared memory, then adds them into the gradient buffers with one red.global.add.f32 per
// element (the same accumulate semantics as the weight-gradient GEMMs, summation order across CTAs unspecified).
//
// Exact rules kept from the stage kernels of ma_tail.cu: inactive track slots of z are 0, KL is the mean over the clip's nt tracks,
// adjacency entries exist only for i != j with i, j < nt, and dhT is 0 for inactive slots.
#include "common.cuh"
#include "cvad_b200.h"

namespace {

constexpr int MAXDET = 5, NF = 6, HID = 64, NPAIR = MAXDET * (MAXDET - 1);
constexpr int NT = 256;
constexpr int NL = 20;
constexpr float KEEP_SCALE = 1.25f;     // 1 / (1 - 0.2): the scorer0 dropout (cad:438)

// layer l of the branch: params[2 l] = weight (DOUT, DIN) row-major (nn.Linear), params[2 l + 1] = bias (DOUT); order in cvad_b200.h
enum { ENC, FX0, FX1, MU, LV, NODE, EDGE0, EDGE1, DYN0, DYN1, DYN2, CS0, CS1, CS2, MS0, MS1, MS2, TS0, TS1, TS2 };
constexpr int DIN[NL] = {64, 32, 32, 32, 32, 6, 64, 32, 6, 32, 32, 18, 64, 32, 12, 32, 16, 6, 32, 16};
constexpr int DOUT[NL] = {32, 32, 32, 6, 6, 32, 32, 1, 32, 32, 6, 64, 32, 1, 32, 16, 1, 32, 16, 1};

// staged in shared memory: weight rows at an odd pitch (DIN + 1; every DIN is even) so that threads over output columns j read
// conflict-free, then the bias; each layer padded to 4 floats
constexpr int stage_size(int l) { return (DOUT[l] * (DIN[l] + 1) + DOUT[l] + 3) & ~3; }
constexpr int stage_off(int l) { return l == 0 ? 0 : stage_off(l - 1) + stage_size(l - 1); }
// parameter-gradient partial sums: the global layout (weight then bias, no padding)
constexpr int grad_off(int l) { return l == 0 ? 0 : grad_off(l - 1) + DOUT[l - 1] * DIN[l - 1] + DOUT[l - 1]; }
constexpr int SP = stage_off(NL);
constexpr int SG = grad_off(NL);

template <int L>
struct Lay {
  static constexpr int din = DIN[L], dout = DOUT[L], pitch = din + 1;
  static constexpr int w = stage_off(L), b = w + dout * pitch;      // staged parameters
  static constexpr int gw = grad_off(L), gb = gw + dout * din;      // gradient partial sums
  static constexpr int nw = dout * din, items = nw + dout;       // weight-gradient items: one per weight and bias element
};

struct Params {
  const float* p[2 * NL];
};
struct Grads {
  float* p[2 * NL];
};

// one clip's forward activations (track rows; rows >= nt are never read)
struct Clip {
  float hT[MAXDET][HID], enc[MAXDET][32], h1[MAXDET][32], h2[MAXDET][32];
  float mu[MAXDET][NF], lv[MAXDET][NF], eps[MAXDET][NF], z[MAXDET][NF];
  float node[MAXDET][32], eh[NPAIR][32], e[NPAIR], adj[NF][NF], st[MAXDET][NF];
  float d1[MAXDET][32], d2[MAXDET][32], pred[MAXDET][NF];
  float sin[3 * NF];      // [cur | prd | |cur - prd|]: the causal scorer's input; the motion scorer reads [cur | prd], the temporal one cur
  float keep[64], c1[64], m1[32], t1[32], c2[32], m2[16], t2[16], s3[4];
};

// one clip's backward: gradients w.r.t. pre-activations unless noted
struct ClipGrad {
  float c1[64], m1[32], t1[32], c2[32], m2[16], t2[16];
  float sin[36];                  // w.r.t. the scorer inputs: causal 18, motion 12, temporal 6
  float zs[NF], prd[NF];          // dz of every active track through cur, dpred of every active track through prd
  float d1[MAXDET][32], d2[MAXDET][32], st[MAXDET][NF];
  float e[NPAIR];                 // edge logits
  float s1[MAXDET][32], s2[MAXDET][32];   // edge hidden gradients summed over the pairs in which the track is first / second
  float node[MAXDET][32], zs2[MAXDET][NF];   // node encoder output; dz through structured
  float mu[MAXDET][NF], lv[MAXDET][NF], h2[MAXDET][32], h1[MAXDET][32], enc[MAXDET][32];
};

constexpr int CLIP_F = ((int)(sizeof(Clip) / sizeof(float)) + 3) & ~3;      // regions start 16-byte aligned
constexpr int GRAD_F = ((int)(sizeof(ClipGrad) / sizeof(float)) + 3) & ~3;
constexpr size_t FWD_SMEM = (size_t)(SP + CLIP_F) * sizeof(float);
constexpr size_t BWD_SMEM = (size_t)(SP + CLIP_F + GRAD_F + SG) * sizeof(float);
static_assert(BWD_SMEM <= 227 * 1024, "backward shared memory");

__device__ __forceinline__ float relu(float v) { return v > 0.f ? v : 0.f; }
__device__ __forceinline__ float sigm(float v) { return cvad_act(v, ACT_SIGMOID); }

// live pair p of nt tracks: (i, j), i != j, i-major
__device__ __forceinline__ int pair_i(int p, int nt) { return p / (nt - 1); }
__device__ __forceinline__ int pair_j(int p, int nt) {
  const int i = p / (nt - 1), jj = p - i * (nt - 1);
  return jj < i ? jj : jj + 1;
}
__device__ __forceinline__ int pair_id(int i, int j, int nt) { return i * (nt - 1) + (j < i ? j : j - 1); }

// W[j] . x + b[j]
template <int L>
__device__ __forceinline__ float dense(const float* sp, int j, const float* x) {
  using Q = Lay<L>;
  const float* w = sp + Q::w + j * Q::pitch;
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < Q::din; ++k) acc = fmaf(w[k], x[k], acc);
  return acc + sp[Q::b + j];
}
// sum_j W[j][k] g[j]
template <int L>
__device__ __forceinline__ float dense_t(const float* sp, int k, const float* g) {
  using Q = Lay<L>;
  const float* w = sp + Q::w + k;
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < Q::dout; ++j) acc = fmaf(w[j * Q::pitch], g[j], acc);
  return acc;
}
// item i < nw + dout of layer L's gradient: dW[j][k] += sum_r g[r][j] x[r][k], db[j] += sum_r g[r][j]  (g, x rows at pitch gp, xp)
template <int L>
__device__ __forceinline__ void wgrad(float* sg, int i, const float* g, int gp, const float* x, int xp, int rows) {
  using Q = Lay<L>;
  float acc = 0.f;
  if (i < Q::nw) {
    const int j = i / Q::din, k = i - j * Q::din;
    for (int r = 0; r < rows; ++r) acc = fmaf(g[r * gp + j], x[r * xp + k], acc);
    sg[Q::gw + i] += acc;
  } else {
    const int j = i - Q::nw;
    for (int r = 0; r < rows; ++r) acc += g[r * gp + j];
    sg[Q::gb + j] += acc;
  }
}
// the same for a one-row, one-output layer: dW[0][k] += g x[k], db[0] += g
template <int L>
__device__ __forceinline__ void wgrad_one(float* sg, int i, float g, const float* x) {
  if (i < Lay<L>::nw) sg[Lay<L>::gw + i] += g * x[i];
  else sg[Lay<L>::gb] += g;
}

template <int L>
__device__ __forceinline__ void stage_params(const Params& P, float* sp) {
  using Q = Lay<L>;
  const float* W = P.p[2 * L];
  const float* bias = P.p[2 * L + 1];
#pragma unroll 4
  for (int i = threadIdx.x; i < Q::nw; i += NT) {
    const int j = i / Q::din, k = i - j * Q::din;
    sp[Q::w + j * Q::pitch + k] = __ldg(W + i);
  }
  if (threadIdx.x < Q::dout) sp[Q::b + threadIdx.x] = __ldg(bias + threadIdx.x);
  if constexpr (L + 1 < NL) stage_params<L + 1>(P, sp);
}

template <int L>
__device__ __forceinline__ void flush_grads(const Grads& G, const float* sg) {
  using Q = Lay<L>;
  if (float* gw = G.p[2 * L])
    for (int i = threadIdx.x; i < Q::nw; i += NT) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(gw + i), "f"(sg[Q::gw + i]) : "memory");
  if (float* gb = G.p[2 * L + 1])
    if (threadIdx.x < Q::dout) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(gb + threadIdx.x), "f"(sg[Q::gb + threadIdx.x]) : "memory");
  if constexpr (L + 1 < NL) flush_grads<L + 1>(G, sg);
}

// The forward of clip b into c (every thread of the CTA; ends with a barrier).  OUT: also write z, kl, adj, causal.
template <bool OUT>
__device__ void clip_forward(const float* sp, Clip& c, int b, int nt, const float* __restrict__ hT, const float* __restrict__ eps,
                             const float* __restrict__ keep, float* __restrict__ z_out, float* __restrict__ kl_out,
                             float* __restrict__ adj_out, float* __restrict__ causal_out) {
  const int tid = threadIdx.x;
  const int np = nt * (nt - 1);
  for (int i = tid; i < nt * HID; i += NT) (&c.hT[0][0])[i] = hT[(long long)b * MAXDET * HID + i];
  for (int i = tid; i < nt * NF; i += NT) (&c.eps[0][0])[i] = eps[(long long)b * MAXDET * NF + i];
  if (keep && tid < 64) c.keep[tid] = keep[(long long)b * 64 + tid];
  __syncthreads();
  // trajectory encoder output Linear, factor MLP
  for (int i = tid; i < nt * 32; i += NT) c.enc[i >> 5][i & 31] = dense<ENC>(sp, i & 31, c.hT[i >> 5]);
  __syncthreads();
  for (int i = tid; i < nt * 32; i += NT) c.h1[i >> 5][i & 31] = relu(dense<FX0>(sp, i & 31, c.enc[i >> 5]));
  __syncthreads();
  for (int i = tid; i < nt * 32; i += NT) c.h2[i >> 5][i & 31] = relu(dense<FX1>(sp, i & 31, c.h1[i >> 5]));
  __syncthreads();
  // mu / log-variance heads, reparameterisation, KL (warp 0: nt * 6 <= 30 lanes)
  if (tid < 32) {
    float term = 0.f;
    if (tid < nt * NF) {
      const int r = tid / NF, f = tid - r * NF;
      const float m = dense<MU>(sp, f, c.h2[r]), l = dense<LV>(sp, f, c.h2[r]);
      c.mu[r][f] = m;
      c.lv[r][f] = l;
      c.z[r][f] = m + c.eps[r][f] * expf(0.5f * l);
      term = -0.5f * (1.f + l - m * m - expf(l));
    }
    if (OUT && tid < MAXDET * NF) z_out[(long long)b * MAXDET * NF + tid] = tid < nt * NF ? c.z[tid / NF][tid % NF] : 0.f;
    term = warp_sum(term);
    if (OUT && tid == 0) kl_out[b] = term / (float)nt;
  }
  __syncthreads();
  // node encoder; cur = mean of z over the tracks
  for (int i = tid; i < nt * 32 + NF; i += NT) {
    if (i < nt * 32) {
      c.node[i >> 5][i & 31] = dense<NODE>(sp, i & 31, c.z[i >> 5]);
    } else {
      const int f = i - nt * 32;
      float s = 0.f;
      for (int k = 0; k < nt; ++k) s += c.z[k][f];
      c.sin[f] = s / (float)nt;
    }
  }
  __syncthreads();
  // edge MLP over the live pairs: hidden = relu(W [node_i | node_j] + b)
  for (int i = tid; i < np * 32; i += NT) {
    const int p = i >> 5, m = i & 31;
    const float* w = sp + Lay<EDGE0>::w + m * Lay<EDGE0>::pitch;
    const float *xi = c.node[pair_i(p, nt)], *xj = c.node[pair_j(p, nt)];
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k) acc = fmaf(w[k], xi[k], acc);
#pragma unroll
    for (int k = 0; k < 32; ++k) acc = fmaf(w[32 + k], xj[k], acc);
    c.eh[p][m] = relu(acc + sp[Lay<EDGE0>::b + m]);
  }
  __syncthreads();
  // edge probabilities into the adjacency; every other entry is 0
  for (int i = tid; i < np + NF * NF; i += NT) {
    if (i < np) {
      const float e = sigm(dense<EDGE1>(sp, 0, c.eh[i]));
      c.e[i] = e;
      c.adj[pair_i(i, nt)][pair_j(i, nt)] = e;
    } else {
      const int q = i - np, a = q / NF, bb = q - a * NF;
      if (!(a < nt && bb < nt && a != bb)) c.adj[a][bb] = 0.f;
    }
  }
  __syncthreads();
  // structured[k][i] = sum_j adj[i][j] z[k][j]
  for (int i = tid; i < nt * NF + (OUT ? NF * NF : 0); i += NT) {
    if (i < nt * NF) {
      const int k = i / NF, a = i - k * NF;
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < NF; ++j) s = fmaf(c.adj[a][j], c.z[k][j], s);
      c.st[k][a] = s;
    } else {
      adj_out[(long long)b * NF * NF + i - nt * NF] = (&c.adj[0][0])[i - nt * NF];
    }
  }
  __syncthreads();
  // dynamics MLP
  for (int i = tid; i < nt * 32; i += NT) c.d1[i >> 5][i & 31] = relu(dense<DYN0>(sp, i & 31, c.st[i >> 5]));
  __syncthreads();
  for (int i = tid; i < nt * 32; i += NT) c.d2[i >> 5][i & 31] = relu(dense<DYN1>(sp, i & 31, c.d1[i >> 5]));
  __syncthreads();
  for (int i = tid; i < nt * NF; i += NT) c.pred[i / NF][i % NF] = dense<DYN2>(sp, i % NF, c.d2[i / NF]);
  __syncthreads();
  if (tid < NF) {
    float s = 0.f;
    for (int k = 0; k < nt; ++k) s += c.pred[k][tid];
    s /= (float)nt;
    c.sin[NF + tid] = s;
    c.sin[2 * NF + tid] = fabsf(c.sin[tid] - s);
  }
  __syncthreads();
  // the three scorers, layer by layer side by side
  for (int i = tid; i < 128; i += NT) {
    if (i < 64) {
      float v = relu(dense<CS0>(sp, i, c.sin));
      if (keep) v *= c.keep[i] * KEEP_SCALE;
      c.c1[i] = v;
    } else if (i < 96) {
      c.m1[i - 64] = relu(dense<MS0>(sp, i - 64, c.sin));
    } else {
      c.t1[i - 96] = relu(dense<TS0>(sp, i - 96, c.sin));
    }
  }
  __syncthreads();
  for (int i = tid; i < 64; i += NT) {
    if (i < 32) c.c2[i] = relu(dense<CS1>(sp, i, c.c1));
    else if (i < 48) c.m2[i - 32] = relu(dense<MS1>(sp, i - 32, c.m1));
    else c.t2[i - 48] = relu(dense<TS1>(sp, i - 48, c.t1));
  }
  __syncthreads();
  if (tid < 32) {
    float s = 0.f;
    if (tid == 0) s = sigm(dense<CS2>(sp, 0, c.c2));
    else if (tid == 1) s = sigm(dense<MS2>(sp, 0, c.m2));
    else if (tid == 2) s = sigm(dense<TS2>(sp, 0, c.t2));
    if (tid < 3) c.s3[tid] = s;
    const float cs = __shfl_sync(0xffffffffu, s, 0), ms = __shfl_sync(0xffffffffu, s, 1), ts = __shfl_sync(0xffffffffu, s, 2);
    if (OUT && tid == 0) causal_out[b] = 0.5f * cs + 0.3f * ms + 0.2f * ts;
  }
  __syncthreads();
}

// The backward of clip b after clip_forward<false> (every thread; ends with a barrier).  Adds the clip's parameter gradients to sg.
__device__ void clip_backward(const float* sp, const Clip& c, ClipGrad& g, float* sg, int b, int nt, const float* __restrict__ dz_up,
                              const float* __restrict__ dkl_up, const float* __restrict__ dadj_up, const float* __restrict__ dcausal_up,
                              const bool masked, float* __restrict__ dhT) {
  const int tid = threadIdx.x;
  const int np = nt * (nt - 1);
  const float gc = dcausal_up ? dcausal_up[b] : 0.f;
  // the scorers' last layers: dpre = (coefficient * dcausal) * s (1 - s)
  const float ds0 = (gc * 0.5f) * (c.s3[0] * (1.f - c.s3[0])), ds1 = (gc * 0.3f) * (c.s3[1] * (1.f - c.s3[1])),
              ds2 = (gc * 0.2f) * (c.s3[2] * (1.f - c.s3[2]));
  for (int i = tid; i < 64 + Lay<CS2>::items + Lay<MS2>::items + Lay<TS2>::items; i += NT) {
    int t = i;
    if (t < 32) { g.c2[t] = c.c2[t] > 0.f ? sp[Lay<CS2>::w + t] * ds0 : 0.f; continue; }
    if ((t -= 32) < 16) { g.m2[t] = c.m2[t] > 0.f ? sp[Lay<MS2>::w + t] * ds1 : 0.f; continue; }
    if ((t -= 16) < 16) { g.t2[t] = c.t2[t] > 0.f ? sp[Lay<TS2>::w + t] * ds2 : 0.f; continue; }
    if ((t -= 16) < Lay<CS2>::items) { wgrad_one<CS2>(sg, t, ds0, c.c2); continue; }
    if ((t -= Lay<CS2>::items) < Lay<MS2>::items) { wgrad_one<MS2>(sg, t, ds1, c.m2); continue; }
    wgrad_one<TS2>(sg, t - Lay<MS2>::items, ds2, c.t2);
  }
  __syncthreads();
  for (int i = tid; i < 128 + Lay<CS1>::items + Lay<MS1>::items + Lay<TS1>::items; i += NT) {
    int t = i;
    if (t < 64) {
      float v = c.c1[t] > 0.f ? dense_t<CS1>(sp, t, g.c2) : 0.f;
      if (masked) v *= c.keep[t] * KEEP_SCALE;
      g.c1[t] = v;
      continue;
    }
    if ((t -= 64) < 32) { g.m1[t] = c.m1[t] > 0.f ? dense_t<MS1>(sp, t, g.m2) : 0.f; continue; }
    if ((t -= 32) < 32) { g.t1[t] = c.t1[t] > 0.f ? dense_t<TS1>(sp, t, g.t2) : 0.f; continue; }
    if ((t -= 32) < Lay<CS1>::items) { wgrad<CS1>(sg, t, g.c2, 32, c.c1, 64, 1); continue; }
    if ((t -= Lay<CS1>::items) < Lay<MS1>::items) { wgrad<MS1>(sg, t, g.m2, 16, c.m1, 32, 1); continue; }
    wgrad<TS1>(sg, t - Lay<MS1>::items, g.t2, 16, c.t1, 32, 1);
  }
  __syncthreads();
  for (int i = tid; i < 36 + Lay<CS0>::items + Lay<MS0>::items + Lay<TS0>::items; i += NT) {
    int t = i;
    if (t < 18) { g.sin[t] = dense_t<CS0>(sp, t, g.c1); continue; }
    if ((t -= 18) < 12) { g.sin[18 + t] = dense_t<MS0>(sp, t, g.m1); continue; }
    if ((t -= 12) < 6) { g.sin[30 + t] = dense_t<TS0>(sp, t, g.t1); continue; }
    if ((t -= 6) < Lay<CS0>::items) { wgrad<CS0>(sg, t, g.c1, 64, c.sin, 18, 1); continue; }
    if ((t -= Lay<CS0>::items) < Lay<MS0>::items) { wgrad<MS0>(sg, t, g.m1, 32, c.sin, 12, 1); continue; }
    wgrad<TS0>(sg, t - Lay<MS0>::items, g.t1, 32, c.sin, 6, 1);
  }
  __syncthreads();
  // through cur / prd (|.| takes the zero subgradient at a tie) to every active track
  if (tid < NF) {
    const float d = c.sin[tid] - c.sin[NF + tid];
    const float sgn = (d > 0.f) - (d < 0.f);
    const float gd = g.sin[12 + tid] * sgn;
    const float gcur = g.sin[tid] + g.sin[18 + tid] + g.sin[30 + tid] + gd;
    const float gprd = g.sin[6 + tid] + g.sin[24 + tid] - gd;
    g.zs[tid] = gcur / (float)nt;
    g.prd[tid] = gprd / (float)nt;
  }
  __syncthreads();
  // dynamics MLP backward (dpred is the same for every active track)
  for (int i = tid; i < nt * 32 + Lay<DYN2>::items; i += NT) {
    if (i < nt * 32) {
      const int r = i >> 5, m = i & 31;
      g.d2[r][m] = c.d2[r][m] > 0.f ? dense_t<DYN2>(sp, m, g.prd) : 0.f;
    } else {
      wgrad<DYN2>(sg, i - nt * 32, g.prd, 0, &c.d2[0][0], 32, nt);
    }
  }
  __syncthreads();
  for (int i = tid; i < nt * 32 + Lay<DYN1>::items; i += NT) {
    if (i < nt * 32) {
      const int r = i >> 5, m = i & 31;
      g.d1[r][m] = c.d1[r][m] > 0.f ? dense_t<DYN1>(sp, m, g.d2[r]) : 0.f;
    } else {
      wgrad<DYN1>(sg, i - nt * 32, &g.d2[0][0], 32, &c.d1[0][0], 32, nt);
    }
  }
  __syncthreads();
  for (int i = tid; i < nt * NF + Lay<DYN0>::items; i += NT) {
    if (i < nt * NF) g.st[i / NF][i % NF] = dense_t<DYN0>(sp, i % NF, g.d1[i / NF]);
    else wgrad<DYN0>(sg, i - nt * NF, &g.d1[0][0], 32, &c.st[0][0], NF, nt);
  }
  __syncthreads();
  // structured backward: dadj (plus the upstream dadj) on the live pairs -> edge logits; dz through structured
  for (int i = tid; i < np + nt * NF; i += NT) {
    if (i < np) {
      const int a = pair_i(i, nt), j = pair_j(i, nt);
      float s = 0.f;
      for (int k = 0; k < nt; ++k) s = fmaf(g.st[k][a], c.z[k][j], s);
      if (dadj_up) s += dadj_up[(long long)b * NF * NF + a * NF + j];
      g.e[i] = s * (c.e[i] * (1.f - c.e[i]));
    } else {
      const int q = i - np, k = q / NF, j = q - k * NF;
      float s = 0.f;
#pragma unroll
      for (int a = 0; a < NF; ++a) s = fmaf(g.st[k][a], c.adj[a][j], s);
      g.zs2[k][j] = s;
    }
  }
  __syncthreads();
  // edge MLP hidden layer: its gradients summed over the pairs in which track i is first (s1) / second (s2); the last layer's gradients
  for (int i = tid; i < nt * 32 + Lay<EDGE1>::items; i += NT) {
    if (i < nt * 32) {
      const int a = i >> 5, m = i & 31;
      const float w = sp[Lay<EDGE1>::w + m];
      float s1 = 0.f, s2 = 0.f;
      for (int j = 0; j < nt; ++j) {
        if (j == a) continue;
        const int pa = pair_id(a, j, nt), pb = pair_id(j, a, nt);
        s1 += c.eh[pa][m] > 0.f ? w * g.e[pa] : 0.f;
        s2 += c.eh[pb][m] > 0.f ? w * g.e[pb] : 0.f;
      }
      g.s1[a][m] = s1;
      g.s2[a][m] = s2;
    } else {
      wgrad<EDGE1>(sg, i - nt * 32, g.e, 1, &c.eh[0][0], 32, np);
    }
  }
  __syncthreads();
  // dnode[i] = W[:, :32]^T s1[i] + W[:, 32:]^T s2[i]; the hidden layer's weight gradient over the pairs, grouped by track
  for (int i = tid; i < nt * 32 + Lay<EDGE0>::items; i += NT) {
    if (i < nt * 32) {
      const int a = i >> 5, k = i & 31;
      const float* w = sp + Lay<EDGE0>::w + k;
      float acc = 0.f;
#pragma unroll
      for (int m = 0; m < 32; ++m) acc = fmaf(w[m * Lay<EDGE0>::pitch], g.s1[a][m], acc);
#pragma unroll
      for (int m = 0; m < 32; ++m) acc = fmaf(w[m * Lay<EDGE0>::pitch + 32], g.s2[a][m], acc);
      g.node[a][k] = acc;
    } else {
      const int t = i - nt * 32;
      float acc = 0.f;
      if (t < Lay<EDGE0>::nw) {
        const int m = t >> 6, k = t & 63;
        const float(*s)[32] = k < 32 ? g.s1 : g.s2;
        for (int a = 0; a < nt; ++a) acc = fmaf(s[a][m], c.node[a][k & 31], acc);
        sg[Lay<EDGE0>::gw + t] += acc;
      } else {
        const int m = t - Lay<EDGE0>::nw;
        for (int a = 0; a < nt; ++a) acc += g.s1[a][m];
        sg[Lay<EDGE0>::gb + m] += acc;
      }
    }
  }
  __syncthreads();
  // node encoder backward, the total dz, reparameterisation and KL backward
  for (int i = tid; i < nt * NF + Lay<NODE>::items; i += NT) {
    if (i < nt * NF) {
      const int r = i / NF, f = i - r * NF;
      float d = dense_t<NODE>(sp, f, g.node[r]) + g.zs2[r][f] + g.zs[f];
      if (dz_up) d += dz_up[(long long)b * MAXDET * NF + i];
      const float gk = (dkl_up ? dkl_up[b] : 0.f) / (float)nt;
      const float m = c.mu[r][f], l = c.lv[r][f];
      g.mu[r][f] = d + gk * m;
      g.lv[r][f] = d * c.eps[r][f] * 0.5f * expf(0.5f * l) + gk * (-0.5f) * (1.f - expf(l));
    } else {
      wgrad<NODE>(sg, i - nt * NF, &g.node[0][0], 32, &c.z[0][0], NF, nt);
    }
  }
  __syncthreads();
  for (int i = tid; i < nt * 32 + Lay<MU>::items + Lay<LV>::items; i += NT) {
    int t = i;
    if (t < nt * 32) {
      const int r = t >> 5, m = t & 31;
      g.h2[r][m] = c.h2[r][m] > 0.f ? dense_t<MU>(sp, m, g.mu[r]) + dense_t<LV>(sp, m, g.lv[r]) : 0.f;
      continue;
    }
    if ((t -= nt * 32) < Lay<MU>::items) { wgrad<MU>(sg, t, &g.mu[0][0], NF, &c.h2[0][0], 32, nt); continue; }
    wgrad<LV>(sg, t - Lay<MU>::items, &g.lv[0][0], NF, &c.h2[0][0], 32, nt);
  }
  __syncthreads();
  for (int i = tid; i < nt * 32 + Lay<FX1>::items; i += NT) {
    if (i < nt * 32) {
      const int r = i >> 5, m = i & 31;
      g.h1[r][m] = c.h1[r][m] > 0.f ? dense_t<FX1>(sp, m, g.h2[r]) : 0.f;
    } else {
      wgrad<FX1>(sg, i - nt * 32, &g.h2[0][0], 32, &c.h1[0][0], 32, nt);
    }
  }
  __syncthreads();
  for (int i = tid; i < nt * 32 + Lay<FX0>::items; i += NT) {
    if (i < nt * 32) g.enc[i >> 5][i & 31] = dense_t<FX0>(sp, i & 31, g.h1[i >> 5]);
    else wgrad<FX0>(sg, i - nt * 32, &g.h1[0][0], 32, &c.enc[0][0], 32, nt);
  }
  __syncthreads();
  for (int i = tid; i < MAXDET * HID + Lay<ENC>::items; i += NT) {
    if (i < MAXDET * HID) dhT[(long long)b * MAXDET * HID + i] = i < nt * HID ? dense_t<ENC>(sp, i & 63, g.enc[i >> 6]) : 0.f;
    else wgrad<ENC>(sg, i - MAXDET * HID, &g.enc[0][0], 32, &c.hT[0][0], HID, nt);
  }
  __syncthreads();
}

__device__ __forceinline__ int clip_tracks(const int* ntr, int b) { return min(max(__ldg(ntr + b), 0), MAXDET); }

__global__ void __launch_bounds__(NT) ma_branch_fwd_kernel(const Params P, const float* __restrict__ hT, const int* __restrict__ ntr,
                                                           const float* __restrict__ eps, const float* __restrict__ keep, int B,
                                                           float* __restrict__ z, float* __restrict__ kl, float* __restrict__ adj,
                                                           float* __restrict__ causal) {
  extern __shared__ __align__(16) float smem[];
  float* sp = smem;
  Clip& c = *reinterpret_cast<Clip*>(smem + SP);
  // parameters first: they do not depend on the kernel in front of this one
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  stage_params<0>(P, sp);
  asm volatile("griddepcontrol.wait;" ::: "memory");
  __syncthreads();
  for (int b = blockIdx.x; b < B; b += gridDim.x) clip_forward<true>(sp, c, b, clip_tracks(ntr, b), hT, eps, keep, z, kl, adj, causal);
}

__global__ void __launch_bounds__(NT) ma_branch_bwd_kernel(const Params P, const Grads G, const float* __restrict__ hT,
                                                           const int* __restrict__ ntr, const float* __restrict__ eps,
                                                           const float* __restrict__ keep, int B, const float* __restrict__ dz,
                                                           const float* __restrict__ dkl, const float* __restrict__ dadj,
                                                           const float* __restrict__ dcausal, float* __restrict__ dhT) {
  extern __shared__ __align__(16) float smem[];
  float* sp = smem;
  Clip& c = *reinterpret_cast<Clip*>(smem + SP);
  ClipGrad& g = *reinterpret_cast<ClipGrad*>(smem + SP + CLIP_F);
  float* sg = smem + SP + CLIP_F + GRAD_F;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  stage_params<0>(P, sp);
  for (int i = threadIdx.x; i < SG; i += NT) sg[i] = 0.f;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  __syncthreads();
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int nt = clip_tracks(ntr, b);
    clip_forward<false>(sp, c, b, nt, hT, eps, keep, nullptr, nullptr, nullptr, nullptr);
    clip_backward(sp, c, g, sg, b, nt, dz, dkl, dadj, dcausal, keep != nullptr, dhT);
  }
  flush_grads<0>(G, sg);
}

// one CTA per clip, at most as many as fit on the GPU at once (the grid strides over the rest); returns the grid or -error
template <typename K>
int grid_for(K kernel, size_t smem, int B, size_t (&configured)[CVAD_MAX_DEVICES], int (&per_sm)[CVAD_MAX_DEVICES]) {
  const cudaError_t ce = cvad_ensure_dyn_smem(kernel, smem, configured);
  if (ce != cudaSuccess) return -(int)ce;
  const int dev = cvad_current_device();
  if (per_sm[dev] == 0 && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[dev], kernel, NT, smem) != cudaSuccess) return -1;
  const long long cap = (long long)(per_sm[dev] > 0 ? per_sm[dev] : 1) * cvad_num_sms();
  return (int)(B < cap ? B : cap);
}

bool fill_params(Params& P, const void* const* params) {
  if (!params) return false;
  for (int i = 0; i < 2 * NL; ++i)
    if (!(P.p[i] = (const float*)params[i])) return false;
  return true;
}

}  // namespace

CVAD_API int cvad_ma_branch_fwd_f32(const float* hT, const int* ntr, const float* eps, const float* keep_scorer0, int B,
                                    const void* const* params, float* z, float* kl, float* adj, float* causal, void* stream) {
  if (B < 0 || !hT || !ntr || !eps || !z || !kl || !adj || !causal) return (int)cudaErrorInvalidValue;
  Params P;
  if (!fill_params(P, params)) return (int)cudaErrorInvalidValue;
  if (B == 0) return 0;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  static int per_sm[CVAD_MAX_DEVICES] = {};
  const int grid = grid_for(ma_branch_fwd_kernel, FWD_SMEM, B, configured, per_sm);
  if (grid <= 0) return grid < 0 ? -grid : (int)cudaErrorInvalidValue;
  return (int)cvad_launch_pdl(ma_branch_fwd_kernel, dim3(grid), dim3(NT), FWD_SMEM, (cudaStream_t)stream, P, hT, ntr, eps, keep_scorer0, B,
                              z, kl, adj, causal);
}

CVAD_API int cvad_ma_branch_bwd_f32(const float* hT, const int* ntr, const float* eps, const float* keep_scorer0, int B,
                                    const void* const* params, const float* dz, const float* dkl, const float* dadj, const float* dcausal,
                                    float* dhT, void* const* grads, void* stream) {
  if (B < 0 || !hT || !ntr || !eps || !dhT || !grads) return (int)cudaErrorInvalidValue;
  Params P;
  if (!fill_params(P, params)) return (int)cudaErrorInvalidValue;
  Grads G;
  for (int i = 0; i < 2 * NL; ++i) G.p[i] = (float*)grads[i];
  if (B == 0) return 0;
  static size_t configured[CVAD_MAX_DEVICES] = {};
  static int per_sm[CVAD_MAX_DEVICES] = {};
  const int grid = grid_for(ma_branch_bwd_kernel, BWD_SMEM, B, configured, per_sm);
  if (grid <= 0) return grid < 0 ? -grid : (int)cudaErrorInvalidValue;
  return (int)cvad_launch_pdl(ma_branch_bwd_kernel, dim3(grid), dim3(NT), BWD_SMEM, (cudaStream_t)stream, P, G, hT, ntr, eps, keep_scorer0, B,
                              dz, dkl, dadj, dcausal, dhT);
}

/*
 * cvad_b200.h -- C ABI of libcvad_b200.so: the B200 (sm_100a) kernels behind the causal video-anomaly hot path.
 *
 * The reference (pvvkishore/Causal-Learning-Based-Video-Anomaly-Detection_Paper_Code_Raw) is pure Python/PyTorch and has
 * no FFI of its own; its seam is the nn.Module / trainer interface (SURVEY.md 8b).  Each entry point below therefore
 * names the reference arithmetic (file:line) it replaces; the Python mirror of that interface
 * (causal-learning-based-video-anomaly-detection_paper_code_raw_b200/) binds these symbols with ctypes.
 *
 * Conventions: plain pointers to DEVICE memory and sizes, no torch types; every function is asynchronous on `stream`
 * (a cudaStream_t passed as void*), allocates nothing, keeps no global state besides a cached SM count, and returns
 * 0 or the cudaError_t of the failed launch.  All tensors are fp32 unless a name says bf16.
 */
#ifndef CVAD_B200_H
#define CVAD_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* activation codes shared by conv / linear / batch-norm epilogues */
#define CVAD_ACT_NONE 0
#define CVAD_ACT_RELU 1
#define CVAD_ACT_LEAKY01 2 /* LeakyReLU(0.1), cad1:133 */
#define CVAD_ACT_SIGMOID 3
#define CVAD_ACT_TANH 4

/* Convolution geometry.  xs / ys are ELEMENT strides of the input / output tensors in (n, c, d, h, w) order, so
 * NCDHW-contiguous torch tensors and channels-last views are both addressable; 2-D convolutions use D = kD = 1. */
typedef struct cvad_conv_desc {
  int N, Cin, Din, Hin, Win;
  int Cout, Dout, Hout, Wout;
  int kD, kH, kW, sD, sH, sW, pD, pH, pW;
  long long xs[5];
  long long ys[5];
} cvad_conv_desc;

/* Device-resident optimizer bookkeeping (one per flat parameter arena). */
typedef struct cvad_opt_state {
  double gradsq;         /* running sum of squared gradients (zeroed by cvad_adam_flat_f32)              */
  double nonfinite;      /* > 0 when a NaN/Inf gradient was seen this step                                */
  double last_gradnorm;  /* total gradient norm of the last step (what clip_grad_norm_ returns)            */
  long long step[8];     /* Adam step count per activity slot; slot 0 = tensors that always receive grads */
  long long skipped;     /* steps skipped because of a non-finite loss / gradient                         */
  double lr_device;      /* > 0: overrides the lr argument (lets a captured CUDA graph follow an LR scheduler) */
} cvad_opt_state;

/* ---- convolution, fp32 implicit GEMM (conv_f32.cu) -------------------------------------------------------------
 * nn.Conv3d / nn.Conv2d forward with fused bias + activation: s2:19-21,28-30; mc3:38,44,50; cad:115,130,135; cad1:131-146.
 * w is torch's OIDHW layout (Cout, Cin, kD, kH, kW), contiguous. */
int cvad_conv_fwd_f32(const cvad_conv_desc* d, const float* x, const float* w, const float* bias, float* y, int act, void* stream);
/* input gradient (autograd of the above; also nn.ConvTranspose2d forward, cad1:162-177).  accumulate != 0 adds into dx. */
int cvad_conv_dgrad_f32(const cvad_conv_desc* d, const float* dy, const float* w, float* dx, int accumulate, void* stream);
/* weight gradient, ADDED atomically onto dw (OIDHW) -- dw is a slice of the flat gradient arena. */
int cvad_conv_wgrad_f32(const cvad_conv_desc* d, const float* x, const float* dy, float* dw, void* stream);

/* ---- fully connected layers (linear_f32.cu) ---------------------------------------------------------------------
 * C[i][j] (+)= sum_k A(i,k) B(k,j);  A(i,k)=A[i*lda+k] if a_kmajor else A[k*lda+i];  B(k,j)=B[j*ldb+k] if b_kmajor else B[k*ldb+j].
 * Epilogue: +bias[j], activation, *mask[i][j]*mask_scale (dropout keep-mask).  splits>1: split-K with atomic adds onto a
 * pre-zeroed C and no epilogue.  gate (may be NULL): device scalar; the call does nothing unless *gate > 0 (a branch whose
 * gradient is None in the reference, SURVEY fact 6, costs no GEMM time).  nn.Linear stacks: s2:24,43-48,77-89; mc3:60-69; cad:167-179,240-246,318-326,361-367,407-413,435-461,525-538. */
int cvad_sgemm_f32(int M, int N, int K, const float* A, long long lda, int a_kmajor, const float* B, long long ldb, int b_kmajor, float* C,
                   long long ldc, const float* bias, int act, const float* mask, float mask_scale, int accumulate, int splits,
                   const float* gate, void* stream);
int cvad_bias_act_mask_f32(float* y, long long rows, int cols, const float* bias, int act, const float* mask, float mask_scale,
                           void* stream);
/* dz = dy * mask*mask_scale * act'(y)  (y is the stored, post-mask output; NULL for ACT_NONE) */
int cvad_act_mask_bwd_f32(const float* dy, const float* y, const float* mask, float mask_scale, int act, float* dz, long long n,
                          void* stream);
/* out[j] (+)= sum_i x[i*ld + j]   (bias gradients) */
int cvad_colsum_f32(const float* x, long long rows, int cols, long long ld, float* out, int accumulate, void* stream);

/* ---- batch norm / pooling (norm_pool_f32.cu); tensors are N,C,(D,)H,W contiguous with S = D*H*W -------------------
 * nn.BatchNorm2d/3d in train mode: cad:116,131,136; mc3:39,45,51; cad1:132-147.  ws = 2*C zero-initialised doubles
 * (re-zeroed by the call).  Writes batch mean / invstd and updates running stats (momentum, unbiased variance). */
int cvad_bn_train_stats_f32(const float* x, int N, int C, long long S, double* ws, float eps, float momentum, float* mean, float* invstd,
                            float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
int cvad_bn_eval_prepare_f32(int C, float eps, const float* running_mean, const float* running_var, float* mean, float* invstd,
                             void* stream);
/* y = act((x-mean)*invstd*gamma+beta) */
int cvad_bn_apply_f32(const float* x, float* y, int N, int C, long long S, const float* mean, const float* invstd, const float* gamma,
                      const float* beta, int act, void* stream);
/* backward of bn_apply (+activation): dx (may be NULL), dgamma/dbeta ADDED (may be NULL).  training=0 -> frozen statistics. */
int cvad_bn_bwd_f32(const float* dy, const float* x, float* dx, int N, int C, long long S, const float* mean, const float* invstd,
                    const float* gamma, const float* beta, int act, int training, double* ws, float* dgamma, float* dbeta, void* stream);
/* out[c] += sum_{n,s} x[n][c][s]  -- bias gradient of a convolution (autograd of s2:19-21 etc.) */
int cvad_channel_sum_add_f32(const float* x, int N, int C, long long S, float* out, void* stream);
/* nn.MaxPool2d/3d: cad:118 (3,2,1); mc3:41,47,53.  idx (int32, may be NULL) = arg-max offset inside each (n,c) plane. */
int cvad_maxpool_fwd_f32(const float* x, float* y, int* idx, long long planes, int D, int H, int W, int OD, int OH, int OW, int kD, int kH,
                         int kW, int sD, int sH, int sW, int pD, int pH, int pW, void* stream);
int cvad_maxpool_bwd_f32(const float* dy, const int* idx, float* dx, long long planes, long long in_size, long long out_size,
                         void* stream); /* dx pre-zeroed */
/* nn.AdaptiveAvgPool2d/3d: s2:23 (4,4,4); cad:126 (4,6); mc3:56 (1,1,1) */
int cvad_adaptive_avgpool_fwd_f32(const float* x, float* y, long long planes, int D, int H, int W, int OD, int OH, int OW, void* stream);
int cvad_adaptive_avgpool_bwd_f32(const float* dy, float* dx, long long planes, int D, int H, int W, int OD, int OH, int OW, void* stream);
/* mean over the middle axis of (A,T,F): cad:568 features.mean(dim=1) */
int cvad_mean_mid_fwd_f32(const float* x, float* y, long long A, int T, long long F, void* stream);
int cvad_mean_mid_bwd_f32(const float* dy, float* dx, long long A, int T, long long F, int accumulate, void* stream);

/* ---- losses (loss_optim.cu) ---------------------------------------------------------------------------------------
 * ImprovedMiniCausalVAD.compute_improved_loss, s2:135-205.  pseudo (B) in {0,1} = (rand > 0.95) drawn by the caller.
 * out8 = {total, anomaly, acyclicity, sparsity, consistency, structure, edge_count, sparsity_ratio}; dscores (B), dadj (B,256).
 * ws: cvad_mb_loss_ws_floats(B) floats.  nonfinite_flag (may be NULL) is set to 1 when the loss is NaN/Inf (s2:230). */
long long cvad_mb_loss_ws_floats(int B);
int cvad_mb_loss_f32(const float* scores, const float* adj, const float* pseudo, int B, float w_anom, float w_causal, float w_sparse,
                     float w_cons, float* ws, float* out8, float* dscores, float* dadj, float* nonfinite_flag, void* stream);
/* nn.BCELoss (mean) + gradient, mc3:240,287 (+ the NaN/Inf guards of mc3:282-292 as a device flag) */
int cvad_bce_loss_f32(const float* scores, const float* targets, int B, float* out1, float* dscores, float* nonfinite_flag, void* stream);
/* cad:649-662: out5 = {total, CE(on softmax probs), MSE(final), MSE(causal), KL}; gradients may be NULL (all or none) */
int cvad_ma_loss_f32(const float* probs, const float* final_scores, const float* causal_scores, const float* kl, const long long* labels,
                     int B, float* out5, float* dprobs, float* dfinal, float* dcausal, float* dkl, float* nonfinite_flag, void* stream);

/* ---- optimizer over a flat arena (loss_optim.cu) ---------------------------------------------------------------------
 * Arena layout: block 0 (1024 floats) is a header -- header[0] = non-finite-loss flag, header[1..7] = per-slot "this group
 * received a gradient" flags; every tensor starts on a 1024-float boundary.  block_slot[b] = -1 (header/padding), 0 (always
 * stepped) or 1..7 (stepped only when header[slot] > 0; torch skips tensors whose grad is None: cad:615-617 + SURVEY fact 6).
 * clip_grad_norm_ + AdamW: s2:236-238, cad:665-667; Adam with L2 decay and clip-if-norm>threshold: mc3:298-311. */
int cvad_sumsq_f32(const float* g, long long n, float scale, cvad_opt_state* state, void* stream);
int cvad_adam_flat_f32(float* p, const float* g, float* m, float* v, long long n, const int* block_slot, cvad_opt_state* state,
                       float grad_scale, float lr, float beta1, float beta2, float eps, float weight_decay, int decoupled, int clip_mode,
                       float max_norm, float clip_threshold, int nan_mode, void* stream);
int cvad_fill_f32(float* x, long long n, float value, void* stream);
/* out[i] = a*x[i*xs] + b*y[i*ys]   (score fusion 0.6*causal + 0.4*direct[:,1], cad:574) */
int cvad_lincomb2_f32(float* out, const float* x, long long xs, float a, const float* y, long long ys, float b, long long n, void* stream);

/* ---- M-A0 (video_anomaly_detection.py, "vad"): the pieces that differ from M-A (ma0_tail.cu) ----------------------------
 * Same dense layout as the M-A causal branch below (5 track slots per clip + counts); vad's detector keeps at most its 3 anchors. */
/* vad:127-165: the frame's anchors ordered by descending sigmoid(conf_logit) (torch.topk over all 3; equal scores keep anchor order),
 * those with confidence > 0.5 copied to box (rows,5,4) as raw bbox_head outputs (no squashing, vad:135-141); no survivor -> one all-zero
 * dummy box (vad:158-160, a constant).  cnt (rows) int32 >= 1; src (rows,5) int32 = anchor of each kept slot or -1; unused slots are
 * zero.  active_flag (may be NULL) is set to 1 when any real box was kept (bbox_head then receives a gradient; conf_head never does). */
int cvad_det_topk_decode_f32(const float* bbox, const float* conf_logit, long long rows, float* box, int* cnt, int* src, float* active_flag,
                             void* stream);
int cvad_det_topk_decode_bwd_f32(const float* dbox, const int* src, const int* cnt, long long rows, float* dbbox, void* stream);
/* vad:389-397: out18[row] = [cur | pred | |cur - pred|] per track row (rows = B*5, 6 factors); bwd uses sign(0) = 0 like torch.abs */
int cvad_score_rows_f32(const float* z, const float* pred, long long rows, float* out18, void* stream);
int cvad_score_rows_bwd_f32(const float* z, const float* pred, const float* dout18, long long rows, float* dz, float* dpred, void* stream);
/* vad:398-399: out[b] = mean of s[b, 0..ntr[b]) over the clip's tracks (s is (B,5)) */
int cvad_masked_mean_f32(const float* s, const int* ntr, int B, float* out, void* stream);
int cvad_masked_mean_bwd_f32(const float* dout, const int* ntr, int B, float* ds, void* stream);
/* vad:516-531: out3 = {total, MSE(scores, labels), KL} with KL = sum of the finite kl[b] / their number (0 when none is finite) and
 * total = MSE + 0.001*KL; gradients may be NULL (both or none) */
int cvad_ma0_loss_f32(const float* scores, const float* kl, const long long* labels, int B, float* out3, float* dscores, float* dkl,
                      float* nonfinite_flag, void* stream);
/* streaming sliding-window inference (bbox:392-430 turned into a service; SURVEY.md 8(f3)): per-frame backbone features live in a ring of
 * `capacity` frames x F floats; out (n_windows, T, F) gathers window w = frames first_frame + w*stride + [0,T) (indices modulo capacity) */
int cvad_window_features_f32(const float* ring, long long capacity, long long first_frame, int stride, int T, int F, long long n_windows,
                             float* out, void* stream);
/* S frame streams sharing one push (bbox:392-430 scores a test set video by video; a deployment serves many cameras), so that one captured
 * CUDA graph serves every push of a given size for all of them.  rings (S, capacity, F) fp32; cursors (S, 2) int64 on the device, row k =
 * {frames pushed, next window} of stream k; push (S, 2) int64 on the device, row k = {count_k in [0, n], reset_k}.  Window rule, per stream:
 *   base_k = reset_k ? 0 : cursors[k][0]     next_k = reset_k ? 0 : cursors[k][1]     frames_k = base_k + count_k
 *   n_win_k = frames_k >= T ? (frames_k - T) / stride + 1 - next_k : 0
 * ring_write: feats (S*n, F), stream-major; row r < count_k of stream k goes to rings[k][(base_k + r) % capacity], rows r >= count_k
 * are not read.  window_features: out (S*m, T, F); slot (k, j) holds window next_k + j of stream k (frames (next_k + j)*stride + [0,T)
 * modulo capacity) when j < n_win_k, zeros otherwise.  cursor_advance: cursors[k] = {frames_k, next_k + n_win_k}; issue it after the
 * other two, on the same stream. */
int cvad_streams_ring_write_f32(const float* feats, int S, long long n, int F, float* rings, long long capacity, int T, int stride,
                                const long long* cursors, const long long* push, void* stream);
int cvad_streams_window_features_f32(const float* rings, int S, long long capacity, int stride, int T, int F, long long m,
                                     const long long* cursors, const long long* push, float* out, void* stream);
int cvad_streams_cursor_advance(long long* cursors, int S, int T, int stride, const long long* push, void* stream);
/* The same streams with rings of FRAMES instead of features (frames.cu), for the 3-D clip models (M-B, M-C, M-E), whose temporal zero
 * padding makes every window's activations depend on where it starts: each window is gathered from the ring and scored whole.  Same
 * cursors, push descriptor and window rule as above; issue cvad_streams_cursor_advance after both, on the same stream.
 * frame_write_u8: src (S*n, src_h, src_w, C) interleaved uint8, stream-major (BGR for C = 3, as cv2 and video decoders deliver it); row
 *   r < count_k of stream k is resized to (dst_h, dst_w) with cvad_resize_bilinear_u8's rule (cv2.resize INTER_LINEAR, bit-exact; a copy
 *   at the same size) into rings[k][(base_k + r) % capacity], rings (S, capacity, dst_h, dst_w, C) uint8; rows r >= count_k are not read.
 * clips_f32: out (S*m, C, T, H, W) fp32 from rings (S, capacity, H, W, C); slot (k, j) holds window next_k + j of stream k (frames
 *   (next_k + j)*stride + [0,T) modulo capacity) when j < n_win_k, zeros otherwise; each value is value * scale, and channel c reads
 *   channel C-1-c when reverse_channels (BGR -> RGB): the values of cvad_clips_from_frames_f32 on the same frames.
 * Both return cudaErrorInvalidValue for a NULL pointer, a non-positive S / capacity / T / stride / size, C outside [1, 4] or a negative
 * n / m, and 0 without a launch for n = 0 / m = 0. */
int cvad_streams_frame_write_u8(const void* src, int S, long long n, int src_h, int src_w, int C, void* rings, long long capacity, int dst_h,
                                int dst_w, int T, int stride, const long long* cursors, const long long* push, void* stream);
int cvad_streams_clips_f32(const void* rings, int S, long long capacity, int H, int W, int C, int T, int stride, long long m,
                           const long long* cursors, const long long* push, float scale, int reverse_channels, float* out, void* stream);

/* ---- M-A causal branch, dense masked batched form (ma_tail.cu) -------------------------------------------------------
 * Every clip carries 5 padded track slots (the detector emits <= 5 boxes per frame, cad:178,198) and a per-clip track
 * count; rows = B*T frames.  Replaces the ragged Python-list loops of cad:206-228, 251-272, 290-307, 337-350, 375-396,
 * 418-424, 466-500 (thousands of batch-1 launches and host syncs per forward). */
/* cad:198-228: box = sigmoid(raw)*scale+offset, validity window, in-order compaction, fallback box when none valid.
 * box (rows,5,4), cnt (rows) int32 >= 1, src (rows,5) int32 = original detection index of each kept slot or -1.
 * active_flag (may be NULL) is set to 1 when any real detection was kept (the detector then receives gradients). */
int cvad_det_decode_f32(const float* raw, long long rows, float* box, int* cnt, int* src, float* active_flag, void* stream);
int cvad_det_decode_bwd_f32(const float* raw, const float* dbox, const int* src, long long rows, float* draw, void* stream);
/* cad:251-269: traj (B,5,T,4+reid_dim) = [box | reid] per kept slot, zero rows for padding; ntr[b] = max_t cnt[b,t];
 * multi_flag (may be NULL) is set to 1 when some clip has >= 2 tracks (only then does the edge MLP get gradients). */
int cvad_traj_assemble_f32(const float* box, const float* reid, const int* cnt, int B, int T, int reid_dim, float* traj, int* ntr,
                           float* multi_flag, void* stream);
int cvad_traj_assemble_bwd_f32(const float* dtraj, const int* cnt, int B, int T, int reid_dim, float* dbox, float* dreid, void* stream);
/* cad:284,298-299: nn.GRU(68->64) recurrence over T for the B*5 track slots (gi = x W_ih^T + b_ih precomputed, (B*5,T,192));
 * hT (B*5,64) last hidden state (zeros for slots >= ntr[b]); saved (B*5,T,5,64) = r,z,n,gh_n,h_prev for the backward. */
int cvad_gru_fwd_f32(const float* gi, const float* w_hh, const float* b_hh, const int* ntr, int B, int T, float* hT, float* saved,
                     void* stream);
int cvad_gru_bwd_f32(const float* dhT, const float* saved, const float* w_hh, const int* ntr, int B, int T, float* dgi, float* dw_hh,
                     float* db_hh, void* stream); /* dw_hh / db_hh are ADDED */
/* cad:328-347: z = mu + eps*exp(logvar/2) (B,5,6), kl (B) = mean over the clip's tracks of -0.5*sum(1+lv-mu^2-e^lv) */
int cvad_reparam_kl_f32(const float* mu, const float* logvar, const float* eps, const int* ntr, int B, float* z, float* kl, void* stream);
int cvad_reparam_kl_bwd_f32(const float* mu, const float* logvar, const float* eps, const int* ntr, int B, const float* dz,
                            const float* dkl, float* dmu, float* dlogvar, void* stream);
/* cad:385: pair (B,5,5,2*node_dim) = [node_i | node_j] */
int cvad_pair_concat_f32(const float* node, int B, int node_dim, float* pair, void* stream);
int cvad_pair_concat_bwd_f32(const float* dpair, int B, int node_dim, float* dnode, void* stream);
/* cad:380-390: adj (B,6,6) from edge probabilities e (B,5,5): i != j and i,j < ntr[b]; backward=1 maps dadj -> de */
int cvad_adj_assemble_f32(const float* src, const int* ntr, int B, float* dst, int backward, void* stream);
/* cad:420: structured[b,k,:] = adj[b] @ z[b,k,:] */
int cvad_structured_f32(const float* adj, const float* z, int B, float* out, void* stream);
int cvad_structured_bwd_f32(const float* adj, const float* z, const float* dout, int B, float* dadj, float* dz, void* stream);
/* cad:469-494: masked track means cur/prd, cin (B,18) = [cur|prd||cur-prd|], min (B,12) = [cur|prd], tin (B,6) = cur */
int cvad_scorer_inputs_f32(const float* z, const float* pred, const int* ntr, int B, float* cin, float* min_, float* tin, void* stream);
int cvad_scorer_inputs_bwd_f32(const float* cin, const int* ntr, int B, const float* dcin, const float* dmin, const float* dtin, float* dz,
                               float* dpred, void* stream);
/* cad:497: 0.5*causal + 0.3*motion + 0.2*temporal */
int cvad_lincomb3_f32(float* out, const float* x, float a, const float* y, float b, const float* z, float c, long long n, void* stream);
/* ---- M-A causal branch behind the GRU in one launch forward and one backward (ma_branch.cu), cad:300-502 -------------------
 * hT (B*5,64) last GRU states (rows of slots >= ntr[b] are ignored), ntr (B) int32 in [1,5], eps (B,5,6), keep_scorer0 (B,64) the dropout
 * keep-mask of the causal scorer's first layer (scaled by 1/0.8) or NULL (eval) ->
 *   z (B,5,6) (0 for slots >= ntr[b]), kl (B) = mean over the clip's tracks, adj (B,6,6) (entries only for i != j, i,j < ntr[b]),
 *   causal (B) = 0.5 causal_scorer + 0.3 motion_scorer + 0.2 temporal_scorer.
 * params: 40 pointers, weight (out,in) row-major then bias of each nn.Linear, in this order:
 *   traj_encoder.encoder (64->32); causal_extractor.encoder.0 (32->32), .2 (32->32); causal_extractor.mu_head (32->6), .logvar_head
 *   (32->6); structure_learner.node_encoder (6->32), .edge_predictor.0 (64->32), .2 (32->1); dynamics_predictor.dynamics_net.0 (6->32),
 *   .2 (32->32), .4 (32->6); anomaly_scorer.causal_scorer.0 (18->64), .3 (64->32), .5 (32->1); .motion_scorer.0 (12->32), .2 (32->16),
 *   .4 (16->1); .temporal_scorer.0 (6->32), .2 (32->16), .4 (16->1).
 * backward: recomputes the forward from (hT, ntr, eps, keep_scorer0); any of the upstream gradients dz (B,5,6), dkl (B), dadj (B,6,6),
 * dcausal (B) may be NULL (= zero); writes dhT (B*5,64) (0 for inactive slots) and ADDS the parameter gradients into grads (40 pointers in
 * the order of params; a NULL entry = that parameter needs no gradient).  The pointer arrays are host arrays, read during the call. */
int cvad_ma_branch_fwd_f32(const float* hT, const int* ntr, const float* eps, const float* keep_scorer0, int B, const void* const* params,
                           float* z, float* kl, float* adj, float* causal, void* stream);
int cvad_ma_branch_bwd_f32(const float* hT, const int* ntr, const float* eps, const float* keep_scorer0, int B, const void* const* params,
                           const float* dz, const float* dkl, const float* dadj, const float* dcausal, float* dhT, void* const* grads,
                           void* stream);
/* cad:537: nn.Softmax(dim=-1) over rows of C (small) entries */
int cvad_softmax_rows_f32(const float* x, long long rows, int C, float* y, void* stream);
int cvad_softmax_rows_bwd_f32(const float* y, const float* dy, long long rows, int C, float* dx, void* stream);

/* ---- bf16 tensor-core path of the M-A backbone (flatconv_tc.cu, nhwc_bf16.cu) ---------------------------------------------
 * The eight 3x3 convolutions, BatchNorms and pools of cad:128-139, 145-155 as tcgen05 (UMMA) GEMMs with fp32 accumulation in
 * TMEM, on a zero-bordered layout that lets TMA feed the tensor cores directly:
 * an activation (N,H,W,C) is stored "padded-flat" as (N,H+2,W+2,C) bf16; the input of a stride-2 convolution is stored as
 * four phase planes P_ab[n][i][j] = padded(2(i-1)+a, 2(j-1)+b), each in the geometry (N,Ho+2,Wo+2,C) of that convolution's
 * output, plane index a*2+b outermost.  Convolution outputs / data-gradients carry junk in their border rows. */
/* OIHW fp32 -> w_fwd [n-block][packed tap][N][Cin] bf16 (N = 128/64/32-channel block of Cout), w_dgrad likewise with the roles of
 * Cin and Cout swapped; either may be NULL.  Taps are packed in natural order for stride 1 and grouped by phase plane for stride 2,
 * so the taps one TMA box fetches are contiguous rows.  Both buffers hold 9*Cout*Cin elements. */
int cvad_flat_pack_w3x3_bf16(const float* w, int Cout, int Cin, int stride, void* w_fwd, void* w_dgrad, void* stream);
/* development hook (tools/conv_probe.py): 8 int64 per CTA receive the MMA warp's wait-cycle breakdown; NULL = off (default) */
int cvad_flat_debug_buffer(long long* buf);
/* (N,H,W,Cin) = input geometry.  stride 1: x, y padded-flat.  stride 2: x = phase planes, y padded-flat (N,Ho+2,Wo+2,Cout). */
int cvad_flat_conv3x3_fwd_bf16(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                               int stride, void* stream);
/* The same convolution with the BatchNorm batch statistics of its output (cad:131,136 in train mode) taken in the epilogue: per-channel
 * sum and sum of squares of the bf16-rounded outputs over the interior pixels are ADDED to stats[0..Cout) / stats[Cout..2*Cout) (fp64,
 * zeroed by the caller; cvad_bn_finalize_f64 turns them into mean / invstd / running statistics and re-zeroes them).
 * Cout must be 32, 64, 128 or 256. */
int cvad_flat_conv3x3_fwd_stats_bf16(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                                     int stride, double* stats, void* stream);
/* y = relu(conv3x3(x) + bias) in bf16, for an eval-mode BatchNorm already folded into w_fwd / bias (cvad_bn_fold_conv_f32 then
 * cvad_flat_pack_w3x3_bf16).  phase_out = 0: y padded-flat (N,Ho+2,Wo+2,Cout), border written as exact zeros.
 * phase_out = 1: y = the four phase planes (4,N,Ho2+2,Wo2+2,Cout) the next stride-2 convolution reads; every plane position that
 * corresponds to a padded pixel is written (0 on the border), positions with no source pixel must be zero on entry and are not touched. */
int cvad_flat_conv3x3_fwd_relu_bf16(const void* x, const void* w_fwd, const float* bias, void* y, int N, int H, int W, int Cin, int Cout,
                                    int stride, int phase_out, void* stream);
/* mean = ws[c]/count, var = ws[C+c]/count - mean^2 (biased) -> invstd; running stats with momentum and the unbiased variance
 * (nn.BatchNorm2d train mode); running_mean / running_var / num_batches_tracked may be NULL.  Re-zeroes ws. */
int cvad_bn_finalize_f64(double* ws, int C, double count, float eps, float momentum, float* mean, float* invstd, float* running_mean,
                         float* running_var, long long* num_batches_tracked, void* stream);
/* stride 1: dy, dx padded-flat.  stride 2: dy padded-flat (N,Ho+2,Wo+2,Cout), dx = phase planes. */
int cvad_flat_conv3x3_dgrad_bf16(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                                 void* stream);
/* dw (OIHW fp32) += sum over pixels; x as for the forward (padded-flat or phase planes), dy padded-flat with a ZERO border */
int cvad_flat_conv3x3_wgrad_bf16(const void* x, const void* dy, float* dw, int N, int H, int W, int Cin, int Cout, int stride, void* stream);
/* The same weight gradient with its atomics staged through scratch (9*Cout*Cin floats, [tap][Cout][Cin], ZERO on entry and again on
 * return): coalesced reductions along Cin, then one pass adds the staging buffer into dw (OIHW). */
int cvad_flat_conv3x3_wgrad_staged_bf16(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin, int Cout,
                                        int stride, void* stream);
/* Data-gradient with the BatchNorm-BACKWARD reductions of the layer below fused into its epilogue (cad:131-136 backward): the rows it writes
 * are dact = dL/d relu(bn(raw_in)); with g = dact * (bn(raw_in) > 0) it adds sum g and sum g*xhat over the interior pixels of raw_in
 * (N,H+2,W+2,Cin padded-flat) to ws[0..Cin) / ws[Cin..2Cin) (fp64, zero on entry) -- what the reduce pass of cvad_pad_bn_relu_bwd_bf16
 * computes by re-reading raw and dact.  cvad_pad_bn_relu_bwd_apply_bf16 then finishes the BatchNorm backward from those sums. */
int cvad_flat_conv3x3_dgrad_bnstats_bf16(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                                         const void* raw_in, const float* gamma, const float* beta, const float* mean, const float* invstd,
                                         double* ws, void* stream);
int cvad_pad_bn_relu_bwd_apply_bf16(const void* raw, const void* dact, void* draw, int N, int H, int W, int C, int phase_in, const float* mean,
                                    const float* invstd, const float* gamma, const float* beta, int training, double* ws, float* dgamma,
                                    float* dbeta, void* stream);
/* The BatchNorm backward's reductions without a pass of their own (cad:131-136 backward, train mode).  With act = relu(bn(raw)) of the layer
 * below, dact = dL/d act and g = dact * (act > 0):
 *   S1 = sum g: the data-gradient that writes dact sums its output under the ReLU mask the forward apply wrote (masksum below);
 *   T = sum act*dact = sum_{co,tap} W*dW for every input channel of the convolution above, taken from its staged weight gradient (wdot);
 * and gamma * sum g*xhat = T - beta*S1, so cvad_pad_bn_relu_bwd_tsum_bf16 finishes the backward in one pass over raw and dact.
 * ws: the lower layer's BatchNorm workspace, 2*C fp64 (zero on entry; S1 in [0,C), T in [C,2C); zero again after the tsum call).
 *
 * Data-gradient (as cvad_flat_conv3x3_dgrad_bf16, dx bit-identical) that also adds sum_rows bf16(dx)*bit to ws[0..Cin); mask: Cin bits per
 * row of dx in dx's own layout (cvad_pad_bn_apply_relu_mask_bf16).  Cin = 32, 64, 128 or 256. */
int cvad_flat_conv3x3_dgrad_masksum_bf16(const void* dy, const void* w_dgrad, void* dx, int N, int H, int W, int Cin, int Cout, int stride,
                                         const void* mask, double* ws, void* stream);
/* Staged weight gradient (as cvad_flat_conv3x3_wgrad_staged_bf16) that also adds T[ci] = sum_{co,tap} bf16(w)*dW of this call (w: the fp32
 * OIHW weight the data-gradient's bf16 pack was made from) to ws[Cin..2Cin).  Cin = 32, 64, 128 or 256. */
int cvad_flat_conv3x3_wgrad_staged_wdot_bf16(const void* x, const void* dy, float* dw, float* scratch, int N, int H, int W, int Cin, int Cout,
                                             int stride, const float* w, double* ws, void* stream);
/* ReLU+BN backward (training mode) from S1 / T in ws: draw padded-flat with ZERO border; dgamma += sum g*xhat, dbeta += sum g (taken in the
 * same pass; either may be NULL); ws re-zeroed */
int cvad_pad_bn_relu_bwd_tsum_bf16(const void* raw, const void* dact, void* draw, int N, int H, int W, int C, int phase_in, const float* mean,
                                   const float* invstd, const float* gamma, const float* beta, double* ws, float* dgamma, float* dbeta,
                                   void* stream);
/* development switch for the stride-2 data-gradient: 2 (default) = one launch, one work item per row tile fills all four phase planes of dx
 * from ONE fetch of the dy segment; 1 = one launch, one work item per (tile, plane); 0 = four launches */
int cvad_flat_dgrad_mode(int mode);
/* development knobs of the flat convolution's launch heuristics (A/B measurements): key 0 = sub-tiles per work item for N = 128 (2 default,
 * 4 = fill the whole accumulator ring), key 1 = activation-segment ring depth for multi-unit items (3 default, 2 = double buffering only) */
int cvad_flat_tune(int key, int value);
/* development switch: 1 (default) = stride-1 32->32 / 64->64 weight gradients stack the three kernel rows in the MMA's N dimension,
 * 0 = one kernel row per MMA */
int cvad_flat_wgrad_mode(int kh_stack);
/* batch statistics over the interior of a padded-flat raw tensor (N,H,W,C interior geometry) */
int cvad_pad_bn_stats_bf16(const void* raw, int N, int H, int W, int C, double* ws, float eps, float momentum, float* mean, float* invstd,
                           float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
/* The finalize step (cvad_bn_finalize_f64) folded into the apply pass: ws still holds the raw fp64 sums of the batch (left by
 * cvad_flat_conv3x3_fwd_stats_bf16); the kernel derives mean / invstd from them (same arithmetic, bit-identical activations), publishes
 * them for the backward, updates the running statistics (cad:116,131-136 train-mode nn.BatchNorm2d) and re-zeroes ws -- one launch on the
 * critical path of every layer instead of two. */
int cvad_pad_bn_finalize_apply_relu_bf16(const void* raw, void* act, int N, int H, int W, int C, int phase_out, double* ws, float eps,
                                         float momentum, const float* gamma, const float* beta, float* mean, float* invstd,
                                         float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
/* act = relu(bn(raw)) written padded-flat with zero border (phase_out = 0) or as the four phase planes (phase_out = 1) */
int cvad_pad_bn_apply_relu_bf16(const void* raw, void* act, int N, int H, int W, int C, int phase_out, const float* mean, const float* invstd,
                                const float* gamma, const float* beta, void* stream);
/* The two apply entries above that also write the ReLU gate: mask = numel(act)/8 bytes in act's row layout, C bits per pixel (bit c in 32-bit
 * word c/32), set where act > 0 -- the same test as the backward's -- and 0 wherever act is zero by construction (border, empty plane
 * positions) */
int cvad_pad_bn_finalize_apply_relu_mask_bf16(const void* raw, void* act, void* mask, int N, int H, int W, int C, int phase_out, double* ws,
                                              float eps, float momentum, const float* gamma, const float* beta, float* mean, float* invstd,
                                              float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
int cvad_pad_bn_apply_relu_mask_bf16(const void* raw, void* act, void* mask, int N, int H, int W, int C, int phase_out, const float* mean,
                                     const float* invstd, const float* gamma, const float* beta, void* stream);
/* ReLU+BN backward; dact padded-flat (phase_in = 0) or phase planes (phase_in = 1); draw padded-flat with ZERO border (may be NULL) */
int cvad_pad_bn_relu_bwd_bf16(const void* raw, const void* dact, void* draw, int N, int H, int W, int C, int phase_in, const float* mean,
                              const float* invstd, const float* gamma, const float* beta, int training, double* ws, float* dgamma,
                              float* dbeta, void* stream);
int cvad_pad_avgpool_bf16_fwd(const void* x, int N, int H, int W, int C, int OH, int OW, float* out, void* stream);
int cvad_pad_avgpool_bf16_bwd(const float* dout, int N, int H, int W, int C, int OH, int OW, void* dx, void* stream);

/* ---- tensor-core stem (stem_tc.cu, both formulations): conv 7x7 s2 p3, 1 -> 32 (cad:115,145) as a tcgen05 kind::tf32 implicit GEMM
 * x (N,1,H,W) fp32, w (32,1,7,7) fp32 OIHW, bias (32).  First a 2x2 space-to-depth of x into X4 (N,Ho+3,Wo+3,4) fp32 -- 16-byte
 * pixels that TMA streams and the MMA descriptor turns into im2col rows; x4 must hold cvad_stem_x4_floats(N,H,W) floats.
 * Pass 1: bn1 batch statistics of conv(x)+bias without writing the convolution output (ws = 64 zeroed doubles, re-zeroed by
 * the call; running statistics updated).  Pass 2: relu(bn1(conv)) as bf16 NHWC (N,Ho,Wo,32).  Then MaxPool2d(3,2,1) (cad:118)
 * of a post-ReLU bf16 NHWC tensor into the padded-flat layout. */
long long cvad_stem_x4_floats(int N, int H, int W);
int cvad_stem_space_to_depth_f32(const float* x, int N, int H, int W, float* x4, void* stream);
/* The frame loader's output taken as it is (cad:89-96: cv2.imread grayscale uint8 -> FloatTensor -> Normalize(0.5, 0.5), cad:1177-1179):
 * x (N,1,H,W) uint8; the space-to-depth applies (float(v) - mean) / std on the fly, bit-identical to normalising on the host, so frames
 * cross PCIe and HBM at one byte per pixel (SURVEY.md 8(f1), K1).  cvad_u8_normalize_f32 is the plain elementwise form (fp32 mode; x and
 * y 16-byte aligned). */
int cvad_stem_space_to_depth_u8(const void* x, int N, int H, int W, float mean, float stdv, float* x4, void* stream);
int cvad_u8_normalize_f32(const void* x, long long n, float mean, float stdv, float* y, void* stream);
int cvad_stem_tf32_stats(const float* x4, const float* w, const float* bias, int N, int H, int W, double* ws, float eps, float momentum,
                         float* mean, float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
int cvad_stem_tf32_bn_relu(const float* x4, const float* w, const float* bias, int N, int H, int W, const float* mean, const float* invstd,
                           const float* gamma, const float* beta, void* y, void* stream);
/* Pass 2 and the max-pool as ONE kernel: relu(bn1(conv)) is pooled out of shared memory, the (N,Ho,Wo,32) tensor between them is never
 * written; out = padded-flat (N,PH+2,PW+2,32) bf16 with its zero border.  Returns cudaErrorNotSupported (801) when a band of a very wide
 * frame does not fit in shared memory: use the two calls above / below instead. */
int cvad_stem_tf32_bn_relu_maxpool(const float* x4, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                   const float* invstd, const float* gamma, const float* beta, void* out, void* stream);

/* The stem's second formulation (also stem_tc.cu): tcgen05 kind::f16 over a 2x4 space-to-depth X8 of the frames (fp16, one 16-byte pixel =
 * a 2 x 4 patch = two adjacent outputs of the stride-2 convolution; accumulator rows carry N = 64 columns = (output parity, channel)):
 * 6 MMAs of M128 x N64 x K16 per 256 outputs instead of 16 of M128 x N32 x K8.  For frames whose width is a multiple of 4;
 * cvad_stem8_bytes returns the size of the X8 buffer or -1 when the shape is outside this path (callers then use the tf32 entries above).
 * Same contracts as cvad_stem_space_to_depth_*, cvad_stem_tf32_stats and cvad_stem_tf32_bn_relu_maxpool (cad:115-118, 145-148). */
long long cvad_stem8_bytes(int N, int H, int W);
int cvad_stem8_space_to_depth_f32(const float* x, int N, int H, int W, void* x8, void* stream);
int cvad_stem8_space_to_depth_u8(const void* x, int N, int H, int W, float mean, float stdv, void* x8, void* stream);
int cvad_stem8_f16_stats(const void* x8, const float* w, const float* bias, int N, int H, int W, double* ws, float eps, float momentum,
                         float* mean, float* invstd, float* running_mean, float* running_var, long long* num_batches_tracked, void* stream);
int cvad_stem8_f16_bn_relu_maxpool(const void* x8, const float* w, const float* bias, int N, int H, int W, const float* mean,
                                   const float* invstd, const float* gamma, const float* beta, void* out, void* stream);
int cvad_pad_maxpool3x3s2_bf16(const void* y, int N, int H, int W, int C, void* out, void* stream);

/* ---- M-D: conv autoencoder + LSTM + memory bank (md_kernels.cu), causal_anomaly_detection1.py --------------------------------
 * nn.LSTM(64->64, 1 layer) recurrence (cad1:182-188, 238-239); gi (N,T,256) = x W_ih^T + b_ih precomputed, gate order i,f,g,o;
 * hT (N,64) = last hidden state; saved (N,T,6,64) = i,f,g,o,c_prev,h_prev (may be NULL in inference). */
int cvad_lstm_fwd_f32(const float* gi, const float* w_hh, const float* b_hh, int N, int T, float* hT, float* saved, void* stream);
/* dgi (N,T,256): gradient of the gate pre-activations; dw_hh (256,64) / db_hh (256) are ADDED (may be NULL) */
int cvad_lstm_bwd_f32(const float* dhT, const float* saved, const float* w_hh, int N, int T, float* dgi, float* dw_hh, float* db_hh,
                      void* stream);
/* cad1:279-294: score[b] = clamp(min_m(1 - clamp(cos(seq_b, memory_m), -1, 1)), 0, 2) / 2 over the first n_filled rows */
int cvad_memory_score_f32(const float* seq, const float* memory, int B, int n_filled, int D, float* score, void* stream);
/* cad1:323-344, 545-547: MSE between frames (B,T,E) and a reconstruction (B,T,E) (recon_t_stride = E) or one reconstruction per
 * clip broadcast over T (recon_t_stride = 0, cad1:254-257).  ws = B zeroed doubles (re-zeroed).  clip_err (B) per-clip mean
 * error, loss = mean over everything, drecon = d loss / d recon in recon's own shape; any of the three may be NULL. */
int cvad_recon_mse_f32(const float* recon, long long recon_t_stride, const float* frames, int B, int T, long long E, double* ws,
                       float* clip_err, float* loss, float* drecon, float* nonfinite_flag, void* stream);
/* calculate_anomaly_scores (cad1:526-564) for every window slot of S streams whose frames live in rings (infer.MultiStreamAutoEncoderScorer):
 * frame_rings (S, capacity, E) fp32; cursors, push and the window rule as for cvad_streams_ring_write_f32; slot (k, j) of the (S*m)
 * outputs is window next_k + j of stream k (frames (next_k + j)*stride + [0,T) modulo capacity) when j < n_win_k.  recon (S*m, E) = one
 * decoded frame per slot, z (S*m, D) = its sequence feature.  recon_err = mean over the window's T*E values of (recon - x_t)^2; mem_score =
 * the cvad_memory_score_f32 value over the first clamp(*memory_ptr, 0, memory_rows) rows of memory (memory_rows, D), exactly 0 when fewer
 * than 10 are filled (memory_ptr is read on the device, so a captured graph follows update_memory / load_state_dict); score = 0.7 *
 * recon_err + 0.3 * mem_score.  Unused slots (j >= n_win_k) get zeros in all three.  Issue before cvad_streams_cursor_advance.
 * Returns cudaErrorInvalidValue for a NULL pointer, E <= 0 or E % 4 != 0, frame_rings / recon not 16-byte aligned, a non-positive S / T /
 * stride / capacity / D / memory_rows or a negative m, and 0 without a launch for m = 0. */
int cvad_streams_md_scores_f32(const float* frame_rings, int S, long long capacity, long long E, int T, int stride, long long m,
                               const long long* cursors, const long long* push, const float* recon, const float* z, const float* memory,
                               int memory_rows, const long long* memory_ptr, int D, float* score, float* recon_err, float* mem_score,
                               void* stream);

/* ---- evaluation tail on the device (SURVEY.md 8(f2)): the numpy / sklearn host code that follows the hot path in the reference.
 * workspace: cvad_eval_workspace_bytes(n) bytes of device memory (caller-owned, any contents).
 * cvad_sort_scores_f32        ascending sort (NaNs last, like np.sort) of n float32 scores; sorted (n) and/or order (n, int32) may be NULL.
 * cvad_percentile_sorted_f32  np.percentile(scores, q) of s1:60 / cad1:609 / cad1:709 (method 'linear', float32 arithmetic exactly as numpy
 *                             performs it for a float32 array: bit-identical threshold), from the sorted scores.
 * cvad_threshold_labels_f32   labels = (scores > *threshold) as 0/1 floats (s1:61).
 * cvad_roc_auc_f32            sklearn.metrics.roc_auc_score of mc3:388 / cad:1233-1248 as the rank statistic with average ranks for ties
 *                             (fp64); 0.0 when one class is absent.  targets: 0/1 floats.
 * cvad_mb_eval_metrics_f32    the 8 entries of s2:286-295 from scores (n) and graphs (n,row_len): mean, std, min, max, range of the scores,
 *                             mean count of entries > edge_threshold, that count / row_len, number of distinct rows (np.unique(axis=0)).
 * cvad_moving_average_f32     np.convolve(x, ones(w)/w, 'valid') of cad:1085-1087 / vad:833-835 in fp64; out holds n-w+1 doubles. */
long long cvad_eval_workspace_bytes(long long n);
int cvad_sort_scores_f32(const float* scores, long long n, void* workspace, float* sorted, int* order, void* stream);
int cvad_percentile_sorted_f32(const float* sorted, long long n, float q, float* out, void* stream);
int cvad_threshold_labels_f32(const float* scores, long long n, const float* threshold, float* labels, void* stream);
int cvad_roc_auc_f32(const float* scores, const float* targets, long long n, void* workspace, double* auc, void* stream);
int cvad_mb_eval_metrics_f32(const float* scores, const float* graphs, long long n, int row_len, float edge_threshold, void* workspace,
                             double* out8, void* stream);
int cvad_moving_average_f32(const float* x, long long n, int w, double* out, void* stream);

/* ---- fused MLP chains (mlp_chain.cu): n_layers <= 8 nn.Linear layers (widths <= 256, sum over layers of (din|1)*dout <= 50000: all weight
 * matrices of the chain are staged in shared memory) with bias, activation and dropout keep-mask in one
 * launch (forward) / one launch (data-gradient chain).  cad:167-179, 240-246, 318-326, 361-367, 407-413, 435-461, 525-538; s2:43-48, 77-89.
 * dims[n_layers+1] = {din_0, dout_0 (= din_1), ...}; acts[l] = CvadAct of layer l; weights[l] (dout,din) row-major; biases[l] / masks[l]
 * (rows,dout) may be NULL (the arrays themselves too); saves[l] (rows,dout) receives layer l's output (post activation, post mask) for
 * the backward, NULL entries / array = not stored (inference).  The arrays are host arrays, read during the call.
 * forward:  out (rows, dout_last) = chain(x (rows, din_0)).
 * backward: dy (rows, dout_last) -> dzs[l] (rows,dout_l) = gradient w.r.t. layer l's pre-activation (what the weight-gradient GEMM
 *           dW_l += dz_l^T h_{l-1} and the bias column sum consume), and dx (rows, din_0) unless NULL. */
int cvad_mlp_chain_fwd_f32(const float* x, long long rows, int n_layers, const int* dims, const int* acts, const void* const* weights,
                           const void* const* biases, const void* const* masks, const float* mask_scales, void* const* saves, float* out,
                           void* stream);
int cvad_mlp_chain_bwd_f32(const float* dy, long long rows, int n_layers, const int* dims, const int* acts, const void* const* weights,
                           const void* const* masks, const float* mask_scales, const void* const* saves, void* const* dzs, float* dx,
                           void* stream);

/* ---- 6144 -> 512 projections on the tensor cores (gemm_tf32x3_tc.cu): y (M,N) += x (M,K) @ w (N,K)^T with TMA-fed tcgen05 kind::tf32 MMAs and
 * the 3xTF32 operand split (hi*hi + lo*hi + hi*lo in the fp32 TMEM accumulator): fp32-level accuracy (~1e-6) on the tensor pipe.  Replaces
 * cvad_sgemm_f32 for the forward of cad:167 (detector, M = B*T) and cad:526 (direct classifier, M = B).  y must be zero on entry (split-K
 * partial sums are reduced atomically); K % 32 == 0; x, w 16-byte aligned; rows beyond M / N are handled by TMA zero fill. */
int cvad_linear_fwd_tf32x3(const float* x, const float* w, float* y, int M, int N, int K, void* stream);

/* Eval-mode BatchNorm folded into the preceding convolution (mc3:38-53 at inference, SURVEY K5): w_out = w * s per output channel,
 * b_out = (b - running_mean) * s + beta, s = gamma / sqrt(running_var + eps); w (Cout, per_out) contiguous, b may be NULL. */
int cvad_bn_fold_conv_f32(const float* w, const float* b, const float* gamma, const float* beta, const float* running_mean,
                          const float* running_var, float eps, int Cout, int per_out, float* w_out, float* b_out, void* stream);

/* ---- frame preparation on the device (frames.cu; SURVEY.md 8(f1)): a video's raw uint8 frames are uploaded once, clips are cut, resized and
 * laid out on the GPU instead of crossing PCIe as fp32 per clip.
 * cvad_resize_bilinear_u8     cv2.resize(img, (dst_w, dst_h)) with INTER_LINEAR on 8-bit images (cad:92, the Avenue loaders, bbox:399), BIT-EXACT:
 *                             OpenCV's 11-bit fixed-point coefficients, its two-pass rounding and its border rules.  src (N,src_h,src_w,C)
 *                             interleaved uint8 (C = 1..4) -> dst (N,dst_h,dst_w,C).
 * cvad_clips_from_frames_f32  clips (B,C,T,H,W) fp32 = frames[starts[b] + t*frame_stride] * scale, channels optionally reversed (BGR -> RGB):
 *                             cvtColor + /255 + permute of the Avenue loaders and the stride-4 window gather of bbox:392-411 in one pass.
 * cvad_clips_from_frames_u8   clips (B,T,1,H,W) uint8 from grayscale frames (F,H,W): M-A's sequence windows (cad:57), normalised by the stem. */
int cvad_resize_bilinear_u8(const void* src, int N, int src_h, int src_w, int C, void* dst, int dst_h, int dst_w, void* stream);
int cvad_clips_from_frames_f32(const void* frames, int F, int H, int W, int C, const int* starts, int B, int T, int frame_stride, float scale,
                               int reverse_channels, float* out, void* stream);
int cvad_clips_from_frames_u8(const void* frames, int F, int H, int W, const int* starts, int B, int T, int frame_stride, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CVAD_B200_H */

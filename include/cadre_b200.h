/*
 * cadre_b200.h — C ABI of libcadre_sm100.so, the sm_100a device side of the CADRE learner hot path.
 *
 * The reference (BIT-MCS/Cadre) is pure Python/PyTorch and has no FFI of its own (SURVEY.md §8b); each entry
 * point below names the reference call site it replaces. Conventions:
 *   - every function returns 0 on success, non-zero on error; cadre_last_error() returns a thread-local
 *     message; no C++ exception crosses the boundary;
 *   - pointer arguments are raw DEVICE pointers borrowed from the caller (e.g. torch.Tensor.data_ptr()) unless
 *     the name ends in _host; the library never frees them; the caller keeps them alive until the stream
 *     has drained;
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with an error.
 */
#ifndef CADRE_B200_H_
#define CADRE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* cadre_last_error(void);
/* library / build identification: "cadre_b200 sm_100a <date>" */
const char* cadre_version(void);
/* 16-bit storage / tensor-core operand type of the encoder path: 1 = IEEE fp16 (default build), 0 = bf16.
 * Every "enc16" buffer below (activations, conv / linear weights) uses this type. */
int cadre_enc_dtype(void);
/* stream-ordered device-to-device copy (test / debug helper) */
int cadre_memcpy_d2d(void* dst, const void* src, int64_t nbytes, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Dense tile operator (tcgen05 + TMEM + TMA). Replaces the cuBLAS/cuDNN calls PyTorch dispatches for
 * nn.Linear / nn.LSTMCell / F.conv2d on the path (ppo_agent/models.py:139-152,165-212;
 * carla_perception/Networks/danet_blocks/resnet.py:39-55,168-183; intertask_att.py:39-80).
 * out[M,N] = epilogue(alpha * A * B^T); kind 0: enc16 operands, kind 1: fp32 operands consumed as TF32.
 * a_mn / b_mn = 0: operand stored [M|N][K] (K contiguous); 1: stored [K][M|N] (M|N contiguous).
 * All leading dimensions / batch strides are in elements. */
typedef struct cadre_gemm_args {
  int32_t kind, a_mn, b_mn, batch;
  int32_t M, N, K, block_n;
  const void* A;
  const void* B;
  int64_t lda, a_bs, ldb, b_bs;
  void* out;
  int64_t ldc, out_bs;
  int32_t out_f32, act; /* act: 0 none, 1 ReLU, 2 LeakyReLU(0.01) */
  const float* bias;
  int64_t bias_bs;
  const void* res; /* residual, dtype of out */
  int64_t ldr, res_bs;
  const void* mask; /* out = 0 where mask <= 0, dtype of out */
  int64_t ldm, mask_bs;
  int32_t res_after_act, rows_is_k;
  const int32_t* batch_rows; /* optional per-batch valid rows (or valid K if rows_is_k) */
  float alpha;
  int32_t epi; /* 0 linear, 1 LSTM cell */
  const float* xpart;
  const float* c_prev;
  float* c_out;
  float* h_out;
  float* gates_out;
  int64_t ldx, x_bs, ldh, h_bs;
} cadre_gemm_args;
int cadre_gemm(const cadre_gemm_args* args, void* stream);

/* NHWC enc16 implicit-GEMM convolution with folded BatchNorm bias, optional residual and ReLU
 * (resnet.py:39-55 BasicBlock, danet.py:21-36 conv5a/5c/51/52, danet.py:41 conv8). in_pad = 1: the input tensor is
 * stored with a 1-pixel zero border, [B][Hin+2][Win+2][Cin] (Hin / Win stay the logical sizes). */
int cadre_conv2d_nhwc(const void* in, int B, int Hin, int Win, int Cin, const void* w, int Cout, int KH,
                      int KW, int stride, int pad, const float* bias, const void* res, int res_after_act,
                      int act, void* out, int in_pad, void* stream);

/* Halo-reuse 3x3 / stride 1 / pad 1 convolution, 64 -> 64 channels (ResNet layer1), on zero-bordered
 * activations: in / res / out are [B][H+2][W+2][64] enc16 with zero borders (kept zero by the kernel). */
/* Debug: per-CTA cycle counters ([grid][16] int64, device memory) filled by the layer1 / stem kernels while
 * the pointer is set; pass NULL to switch off. Not part of the reference interface. */
int cadre_debug_clk(long long* dev_counters);

int cadre_conv3x3_flat64(const void* in, int B, int H, int W, const void* w, const float* bias, const void* res,
                         int act, void* out, void* stream);
/* The same for 128 -> 128 channels (ResNet layer2, W <= 33): in / res / out are [B][H+2][W+2][128] enc16 with zero
 * borders, w is [128][3][3][128]; res (optional) is added before the activation (resnet.py:52-53). */
int cadre_conv3x3_flat128(const void* in, int B, int H, int W, const void* w, const float* bias, const void* res,
                          int act, void* out, void* stream);
/* cadre_conv2d_nhwc writing into a zero-bordered output tensor [B][Hout+2][Wout+2][Cout] (the border is left
 * untouched: the caller zeroes it once). Feeds the halo-reuse kernels above. */
int cadre_conv2d_nhwc_bordered_out(const void* in, int B, int Hin, int Win, int Cin, const void* w, int Cout, int KH,
                                   int KW, int stride, int pad, const float* bias, int act, void* out, int in_pad,
                                   void* stream);
/* Stride-1 convolution with a fused ResNet shortcut (resnet.py:47-53, layer2.0 / 3.0 / 4.0 conv2 + downsample):
 * out = act(conv(in, w[:, :KH*KW*Cin]) + conv1x1/s2(in2, w[:, KH*KW*Cin:]) + bias), the shortcut read on the
 * stride-2 sub-lattice of in2 [B][Hin2 (+2)][Win2 (+2)][Cin2] as Cin2/64 extra k-blocks of one implicit GEMM.
 * w is [Cout][KH*KW*Cin + Cin2] (the 1x1 weights appended along K), bias the sum of both biases;
 * (Hin2 - 1) / 2 + 1 must equal the output height (likewise for the width). in_pad / in2_pad: the input is stored
 * with a 1-pixel zero border; out_pad: out is [B][Hout+2][Wout+2][Cout] and its border is left untouched. */
int cadre_conv2d_nhwc_shortcut(const void* in, int B, int Hin, int Win, int Cin, const void* w, int Cout, int KH, int KW,
                               int pad, const float* bias, int act, void* out, int in_pad, int out_pad, const void* in2,
                               int Cin2, int Hin2, int Win2, int in2_pad, void* stream);
/* Fused stem (resnet.py:169-172): conv7x7/s2/p3 + folded BN bias -> ReLU -> MaxPool2d(3, 2, 1). in is the
 * row-pair interleaved padded image [B][75][262][2][4] (padded row 2*y2 + r, image at rows / columns 3..146 / 3..258),
 * w / bias as cadre_encoder_weights.stem_w / stem_b; out is the zero-bordered [B][38][66][64]: only its interior is
 * written, the caller zeroes the border once. */
int cadre_stem_pool(const void* in, int B, const void* w, const float* bias, void* out, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Perception encoder forward = DANet.get_latent_feature(x, "concate")
 * (carla_perception/Networks/danet.py:216-238) + CadreAgent.pre_process / get_latent_feature
 * (ppo_agent/agent.py:43-75, 97-112). Weights are prepared once by the host (BatchNorm folded into the
 * preceding conv, NHWC / K-major bf16 layouts, linear chains folded) — see cadre_b200/encoder.py. */
typedef struct cadre_encoder_weights {
  const void* stem_w;   /* enc16 [64][256]: [cout][row pair 4][kw 8][row 2][c 4], zero where kh==7 or kw==7 */
  const float* stem_b;  /* [64] conv bias and BN folded */
  const void* conv_w[19]; /* backbone convs in execution order (per block: conv1, conv2, [downsample]);
                             enc16 [Cout][KH][KW][Cin], BN folded */
  const float* conv_b[19];
  const void* head5_w;  /* conv5a | conv5c stacked on Cout: enc16 [256][3][3][512] */
  const float* head5_b; /* [256] */
  const float* pam_wqk; /* fp32 [32][128]: query_conv rows 0..15, key_conv rows 16..31 */
  const float* pam_bqk; /* [32] */
  const void* pam_wv;   /* enc16 [128][128] value_conv (runs on the tensor cores) */
  const float* pam_bv;  /* [128] */
  const void* conv51_w; /* enc16 [128][3][3][128] */
  const float* conv51_b;
  const void* conv52_w;
  const float* conv52_b;
  const void* fc1_w;    /* enc16 [3072][5120]: Linear(20480,512) x6 o {visual,bc}_conv o conv8, K = (h*8+w)*128+c */
  const float* fc1_b;   /* [3072] */
  const void* fc2_w;    /* enc16 [6][256][512], order vis q,k,v, bc q,k,v */
  const float* fc2_b;   /* [6][256] */
  float pam_gamma, cam_gamma;
} cadre_encoder_weights;

int cadre_encoder_create(void** handle, const cadre_encoder_weights* w, int max_batch);
int cadre_encoder_destroy(void* handle);
/* rgb u8 [B][144][256][3], route_fig u8 [B][256][144], measurements f64 [B][3] or NULL;
 * out fp32 [B][ld_out]: 512 latent floats (+ 18 measurement floats when measurements != NULL). */
int cadre_encoder_forward_u8(void* handle, const uint8_t* rgb, const uint8_t* route_fig,
                             const double* measurements, int B, float* out, int ld_out, void* stream);
/* x fp32 NCHW [B][4][144][256] already pre-processed (BASELINE config 2, encoder sweep). */
int cadre_encoder_forward_f32(void* handle, const float* x_nchw, int B, float* out, int ld_out, void* stream);
/* internal activation buffers for parity tests: 0 layer4 out, 1 feat_sum, 2 conv5a|5c, 3 PAM, 4 CAM, 5 fc1 (six folded
 * Linear(20480,512) + LeakyReLU), 6 the ingested image [75][262][2][4] per frame (the input of cadre_stem_pool) */
int cadre_encoder_buffer(void* handle, int which, void** ptr, int64_t* elems_per_frame);
/* Re-runs the trunk on the frames ingested by the previous forward call with a CUDA event between launches:
 * ms_out[i] = device time of launch i (<= 64), names_out = ';'-joined launch names. Measurement helper for
 * bench.py's roofline object; synchronises the stream. */
int cadre_encoder_profile(void* handle, int B, float* out, int ld_out, float* ms_out, char* names_out,
                          int names_cap, int* n_out, void* stream);
/* kernels launched by the last forward call */
int cadre_encoder_launches(void* handle);

/* ------------------------------------------------------------------------------------------------------
 * Rollout: RolloutStorage.compute_returns GAE branch (ppo_agent/storage.py:68-76) + advantage
 * normalisation with unbiased std (ppo_agent/train.py:82-88), one sequence per (env, head).
 * rewards / values / masks / returns: fp32 [E][T+1]; next_value fp32 [E]; adv fp32 [E][T].
 * values[e][T] is overwritten with next_value[e] exactly as the reference does. */
int cadre_gae(const float* rewards, float* values, const float* masks, const float* next_value, float* returns,
              float* adv, int E, int T, float gamma, float tau, int normalize, void* stream);
/* Rollout statistics of E sequences after cadre_gae, over steps t < T of returns / values fp32 [E][T+1] (the raw
 * advantage R - V is recomputed from them: returns = gae + values). out fp32 [E][6] = explained variance
 * 1 - Var(R - V) / Var(R) (NaN when Var(R) = 0), mean and std of R - V, mean and std of R, mean of V; fp64 sums,
 * population variances. One warp per sequence; E > 0, T > 0. */
int cadre_rollout_stats(const float* returns, const float* values, int E, int T, float* out, void* stream);

/* Sliding-window assembly of rollout observations (env_wrapper.py:900-914 stacks the last `seq_length` frames per
 * tick; train.py:69-72 inserts that window into the steer AND the throttle storage). unique_feats: fp32
 * [workers][num_steps + seq_length - 1][feature_dims] = encoder features of every DISTINCT frame of each worker's
 * rollout, oldest first. Writes obs[(w*2 + head)*obs_head_stride + t*obs_step_stride + j*feature_dims + :] =
 * unique_feats[w][t + j][:] for head 0..1, t < num_steps, j < seq_length (strides in floats; RolloutStorage.obs of
 * the batched pool: head stride (T+1)*seq*F, step stride seq*F). */
int cadre_window_scatter(const float* unique_feats, float* obs, int workers, int num_steps, int seq_length,
                         int feature_dims, int64_t obs_head_stride, int64_t obs_step_stride, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * PPO update = CadreAgent.update_policy (ppo_agent/agent.py:166-237) for `workers` logical workers at once
 * (forward + hand-written backward; gradients are the SUM over workers, like Shared_grad_buffers.add_gradient,
 * ppo_agent/models.py:231-239), then the chief's per-module clip + Adam (ppo_agent/chief.py:13-21).
 * Parameters / gradients / Adam moments are flat fp32 buffers of cadre_ppo_param_count() elements in the
 * layout of cadre_b200/csrc/ppo_layout.h (converted from / to reference state dicts by
 * cadre_b200/ppo_params.py). Between cadre_ppo_update and cadre_ppo_adam_step the host all-reduces (sum) the
 * gradient buffer across ranks (NCCL), which replaces the shared-memory aggregation of the reference. */
typedef struct cadre_ppo_config {
  int32_t workers;    /* logical workers (envs) whose minibatches are processed per update on this GPU */
  int32_t mini_batch; /* rows per worker per head = num_steps / mini_batch_num (storage.py:94) */
  float clip, value_coeff, clip_coeff, ent_coeff; /* agent_config.py:43-46 */
} cadre_ppo_config;

/* device pointers into one RolloutStorage (ppo_agent/storage.py:8-26) + its advantage vector */
typedef struct cadre_storage_ref {
  const float* obs;              /* [T+1][8][530] */
  const int64_t* action;         /* [T+1][1] */
  const float* value_preds;      /* [T+1][1] */
  const float* returns;          /* [T+1][1] */
  const float* action_log_probs; /* [T+1][1] */
  const float* adv;              /* [T][1] normalised advantages */
  const float* hn;               /* [T+1][530] */
  const float* cn;               /* [T+1][530] */
  const int32_t* command;        /* [T+1][1] */
} cadre_storage_ref;

int64_t cadre_ppo_param_count(void);
int cadre_ppo_create(void** handle, const cadre_ppo_config* cfg);
int cadre_ppo_destroy(void* handle);
/* storages_host: [workers][2] (steer, throttle); indices_host: int32 [workers][2][mini_batch] minibatch row
 * indices (host-generated, bit-exact torch.randperm chunks); losses: device fp32 [workers][2][3] =
 * per-worker, per-head UN-scaled (value, action, entropy) losses. grads is overwritten.
 * Staged form for a sequence of update steps on the same storages (train.py:93-110: ppo_epoch x minibatches):
 * cadre_ppo_stage uploads the storage references and the indices of n_steps <= 64 steps ([n_steps][workers][2][mb])
 * once; each following cadre_ppo_update(handle, NULL, NULL, ...) consumes the next slice (a device-side counter) and
 * advances the device-side Adam step (starting at first_adam_step), which cadre_ppo_adam_step* use when called with
 * step = 0. Such an update + adam sequence issues no host-to-device copy and can be captured in a CUDA graph. */
int cadre_ppo_stage(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host, int n_steps,
                    int first_adam_step, void* stream);
int cadre_ppo_update(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                     float* params, float* grads, float* losses, void* stream);
/* Forward only (CadreAgent.act / get_value, Model.evaluate_actions; agent.py:114-164, models.py:184-212):
 * row_out fp32 [2 heads][workers*mini_batch][36] = value, log-prob(stored action), entropy, 33 normalised
 * logits (first 3 valid for the throttle head); row order = (worker, minibatch position). */
int cadre_ppo_evaluate(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                       const float* params, float* row_out, void* stream);
int cadre_ppo_adam_step(void* handle, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                        float max_grad_norm, float lr, float beta1, float beta2, float eps, int step,
                        void* stream);
/* gradient norms of the 16 modules seen by the last adam_step: [0..7] LSTM of expert e, [8..15] actor-critic
 * of expert e (expert = head*4 + command); synchronises */
int cadre_ppo_module_norms(void* handle, float* norms16_host);
/* Data-parallel pipeline (replaces Shared_grad_buffers.add_gradient + the chief's single optimizer.step(),
 * models.py:231-239, chief.py:13-21, by per-group all-reduce + clip + Adam overlapped with the backward pass).
 * cadre_ppo_set_grad_groups(groups in {1, 2, 4, 8}): subsequent cadre_ppo_update calls produce the LSTM weight
 * gradients per group of 8 / groups experts. cadre_ppo_grad_range: the contiguous [offset, offset + count) range of the
 * flat buffers that holds group `group`'s LSTM tensors (group = -1: the actor-critic tensors of all experts) and the
 * module ids [mod_begin, mod_end) it covers (module e < 8 = LSTM of expert e, 8 + e = actor-critic of expert e: each
 * is one reference nn.Module, the unit of clip_grad_norm_). cadre_ppo_wait_grads: `stream` waits until the LAST
 * cadre_ppo_update has finished that range of `grads`. cadre_ppo_adam_step_modules: clip + Adam restricted to the
 * modules [mod_begin, mod_end). */
int cadre_ppo_set_grad_groups(void* handle, int groups);
int cadre_ppo_grad_range(void* handle, int group, int64_t* offset, int64_t* count, int* mod_begin, int* mod_end);
int cadre_ppo_wait_grads(void* handle, int group, void* stream);
int cadre_ppo_adam_step_modules(void* handle, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                                float max_grad_norm, float lr, float beta1, float beta2, float eps, int step,
                                int mod_begin, int mod_end, void* stream);
/* Synchronises and returns non-zero (cadre_last_error() explains) if a persistent LSTM recurrence kernel of an
 * earlier cadre_ppo_update / cadre_ppo_evaluate on this handle gave up waiting for a cross-CTA hand-off (its polling is
 * bounded so that a lost signal can never hang the GPU). */
int cadre_ppo_check(void* handle);
int cadre_ppo_launches(void* handle);
/* Update diagnostics (off by default). While diag_out is set, each cadre_ppo_update also writes diag_out fp32
 * [workers][2][4], means over the minibatch of worker w's head h with d = lp - old_lp: [0] approximate KL
 * expm1(d) - d, [1] old_lp - lp, [2] fraction of rows with |ratio - 1| > clip, [3] fraction of rows with
 * |v - old_v| > clip; bit-reproducible, no float atomics. While norms_out is set, each cadre_ppo_adam_step* also writes
 * the pre-clip gradient norm of every module it steps into norms_out[module] (fp32 [16], module order of
 * cadre_ppo_module_norms). Both are device pointers read at launch time: the host points them at the next row of a
 * device-side history before each staged step, which needs no synchronisation. NULL turns either off; losses,
 * gradients and parameters do not depend on the setting. */
int cadre_ppo_set_diagnostics(void* handle, float* diag_out, float* norms_out);
/* Target-KL early stopping of a phase of staged update steps (off by default; SB3's target_kl rule). While it is on,
 * each staged cadre_ppo_update also writes kl_sum_dev fp32 [2]: per head, the sum over this engine's workers of the
 * approximate KL (diag term [0] above). The caller sums kl_sum_dev over ranks (a 16-byte vector in place) and then
 * calls cadre_ppo_kl_gate on the stream of the Adam steps, before the step's first cadre_ppo_adam_step* with step = 0.
 * The gate computes KL = sum over heads of kl_sum[h] * (1 / total_workers); if KL > 1.5 * target_kl the step is not
 * applied (no norms are skipped for it, but no Adam update, no moment update, and the device Adam step goes back by
 * one), and every later step of the phase is skipped: its update routes no rows (gradients and losses are zeros) and its
 * norms and Adam step do nothing. One-step updates (indices_host set) and Adam steps with step >= 1 ignore the gate.
 * cadre_ppo_set_target_kl: target_kl = 0 turns it off; otherwise target_kl must be finite and > 0, total_workers (all
 * ranks) >= this engine's workers and kl_sum_dev set (4 floats advised: a 16-byte vector for the exchange).
 * cadre_ppo_kl_begin starts a phase (clears the stop); call it before the phase's first cadre_ppo_stage, not between
 * its chunks. cadre_ppo_stage with first_adam_step = 0 continues the device Adam step (after a stop, the steps actually
 * applied). cadre_ppo_early_stop reads the state in the order of `stream` (the stream of the gates), waits for that
 * stream only, and returns state_host int32 [5] = steps gated, steps run (applied + the one that stopped), steps applied, index of the step that stopped (-1: none), device Adam step; and kl_host fp32
 * [kl_count] (kl_count <= 4096), the KL of each step that ran (entries past "steps run" are stale). */
int cadre_ppo_set_target_kl(void* handle, float target_kl, int total_workers, float* kl_sum_dev);
int cadre_ppo_kl_begin(void* handle, void* stream);
int cadre_ppo_kl_gate(void* handle, void* stream);
int cadre_ppo_early_stop(void* handle, int32_t* state_host, float* kl_host, int kl_count, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Device-side rollout collection: replaces the host-side Categorical draw (ppo_agent/distributions.py:96-99,
 * agent.py:114-141), the per-worker RolloutStorage.insert calls (storage.py:45-58) and the per-worker get_value
 * bootstrap (train.py:66-79) with a fixed number of launches and copies per tick, whatever the worker count.
 *
 * Counter-based categorical sampler (cadre_b200/csrc/sampler.cuh). A draw is a pure function of
 * (seed, env id, tick, word, log-probs); the library holds no RNG state:
 *   x = Philox4x32-10(counter = (tick & 0xffffffff, tick >> 32, env_id, 0), key = (seed & 0xffffffff, seed >> 32)),
 *       output word `word` (the act step uses word 0 for the steer head, 1 for the throttle head); counter word 3 is
 *       0 here and the snapshot index k in cadre_ensemble_control;
 *   u = (x >> 8) * 2^-24, exact in fp32;
 *   p_j = expf(lp_j) for j < A (columns >= A are never read), c_j = inclusive prefix sum in index order;
 *   a = min{ j : c_j > u * c_{A-1} }, or max{ j : p_j > 0 } if rounding leaves none; so p_j == 0 is never drawn.
 * cadre_categorical_sample: rows of fp32 log-probabilities logp[rows][ld], env_ids int32 [rows] (device);
 * action_out int64 [rows], logp_out fp32 [rows] = lp_a bit for bit, u_out fp32 [rows] = u (may be NULL).
 * 1 <= A <= 33 (33 = steer, 3 = throttle), rows > 0, 0 <= word <= 3. */
int cadre_categorical_sample(const float* logp, int ld, int rows, int A, uint64_t seed, uint64_t tick,
                             const int32_t* env_ids, int word, int64_t* action_out, float* logp_out, float* u_out,
                             void* stream);

/* The batched tensors of a RolloutPool (cadre_b200/learner.py): `storages` = 2 * workers RolloutStorage objects,
 * storage n = 2 * worker + head, each tensor [storages][num_steps + 1][...] contiguous (storage.py:8-26). */
typedef struct cadre_rollout_pool {
  float* obs;              /* [n][T+1][seq_length][feature_dims] */
  int64_t* action;         /* [n][T+1] */
  float* action_log_probs; /* [n][T+1] */
  float* value_preds;      /* [n][T+1] */
  float* rewards;          /* [n][T+1] */
  float* masks;            /* [n][T+1] */
  int32_t* command;        /* [n][T+1] */
  float* hn;               /* [n][T+1][hidden_size] */
  float* cn;               /* [n][T+1][hidden_size] */
  int32_t storages, num_steps, seq_length, feature_dims, hidden_size;
} cadre_rollout_pool;

/* One act step of E environments into the pool at cursor `slot` (0 <= slot <= num_steps), on an engine with
 * workers = 1, mini_batch = E: storages_host / indices_host as for cadre_ppo_evaluate (the actor's [E][8][530]
 * windows and commands; indices must be 0..E-1 for both heads). Runs the forward plan and head_eval_kernel unchanged
 * (row_out as cadre_ppo_evaluate, fp32 [2][E][36]), then ONE kernel that, for environment e and head h (storage
 * n = 2e + h), draws a_h with the sampler above (env id env_ids[e], word h, A = 33 / 3) and writes
 * action[n][slot], action_log_probs[n][slot] = lp_a, value_preds[n][slot], command[n][slot], obs[n][slot] = the
 * window of e, and, only when slot < num_steps, hn[n][slot+1] / cn[n][slot+1] = hidden_hn / hidden_cn (fp32
 * [hidden_size], the agent's hidden_state), as RolloutStorage.insert does (storage.py:45-58); actions_out int64
 * [E][2] receives the draws for one device-to-host copy. The pool needs storages = 2E, seq_length = 8,
 * feature_dims = hidden_size = 530. */
int cadre_ppo_act(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                  const float* params, float* row_out, const cadre_rollout_pool* pool, int slot, uint64_t seed,
                  uint64_t tick, const int32_t* env_ids, const float* hidden_hn, const float* hidden_cn,
                  int64_t* actions_out, void* stream);
/* Rewards and masks of slot `slot` of every storage (train.py:60-72: env.step, then insert): two cudaMemcpy2DAsync
 * from host rows rewards_host / masks_host fp32 [storages] (pinned for an asynchronous copy) into the strided columns
 * [n][slot]. The caller keeps the host rows unchanged until the stream has consumed them. */
int cadre_rollout_env_results(const cadre_rollout_pool* pool, int slot, const float* rewards_host,
                              const float* masks_host, void* stream);
/* Bootstrap values of all workers in one forward (train.py:76-79, agent.py:143-164) on an engine with
 * mini_batch = 1: storages_host / indices_host as for cadre_ppo_evaluate (index num_steps of every storage, hn / cn
 * holding the agent's hidden_state at that index); row_out fp32 [2][workers][36] scratch; next_value fp32
 * [workers][2] = value of worker w's head h, exactly 0 where bit w of done_mask is set. No host synchronisation. */
int cadre_ppo_bootstrap(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                        const float* params, float* row_out, uint64_t done_mask, float* next_value, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Ensemble evaluation (eval.py:53-63): K policy snapshots act on the same E environments and their controls are
 * averaged (CadreAgent.avg_action, agent.py:83-95).
 *
 * cadre_ensemble_control: row_out fp32 [K][2][E][36] in cadre_ppo_evaluate's row format (snapshot k's rows at
 * row_out + k * 2 * E * 36). For snapshot k, environment e and head h (A = 33 / 3):
 *   greedy = 0: a = the sampler above with counter (tick lo, tick hi, env_ids[e], k), output word h; snapshot 0 thus
 *               draws what cadre_ppo_act draws for the same (seed, env id, tick);
 *   greedy = 1: a = the first index of the largest log-prob among j < A (torch.argmax's rule).
 * actions_out int64 [K][E][2] = the actions; controls_out fp64 [E][3] = (steer, throttle, brake) averaged over the K
 * snapshots: steer_table fp64 [33] (STEER_CONTROL), throttle_table fp64 [3][2] ((throttle, brake) = THROTTLE_CONTROL),
 * the three sums taken in float64 in snapshot order and divided by K, then, if K > 1 and the mean brake is below 0.5,
 * brake = 0: bit for bit numpy's mean(0) of avg_action. 1 <= K <= 64, E >= 1, greedy in {0, 1}; one launch. */
int cadre_ensemble_control(const float* row_out, int K, int E, uint64_t seed, uint64_t tick, const int32_t* env_ids,
                           int greedy, const double* steer_table, const double* throttle_table, double* controls_out,
                           int64_t* actions_out, void* stream);
/* One ensemble tick on an engine with workers = 1, mini_batch = E (storages_host / indices_host as for cadre_ppo_act:
 * the [E][8][530] windows and commands, indices 0..E-1 for both heads): for each snapshot k, the forward plan and
 * head_eval_kernel with parameters params_host[k] (K device pointers) into row_out[k] (bit-identical to
 * cadre_ppo_evaluate with those parameters), then cadre_ensemble_control's kernel once. The index table is uploaded
 * once for all K forwards. cadre_ppo_launches = K * (forward launches + 1) + 1 (the forward's own count is the one
 * cadre_ppo_evaluate reports, minus its head_eval_kernel). */
int cadre_ppo_ensemble_act(void* handle, const cadre_storage_ref* storages_host, const int32_t* indices_host,
                           const float* const* params_host, int K, float* row_out, uint64_t seed, uint64_t tick,
                           const int32_t* env_ids, int greedy, const double* steer_table, const double* throttle_table,
                           double* controls_out, int64_t* actions_out, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Gradient exchange across the ranks of one NVSwitch domain, in place: grads <- sum over ranks, every rank receives
 * the same bits. Replaces Shared_grad_buffers.add_gradient + the chief installing the summed gradient
 * (ppo_agent/models.py:231-239, ppo_agent/chief.py:13-16). The buffer must be symmetric memory: buffer_ptrs_host[r] =
 * rank r's copy as mapped into THIS process (r == rank: the local buffer), `multicast` = the multicast mapping of all
 * copies (NULL when the fabric has none), flag_ptrs_host[r] = rank r's zero-initialised flag area of
 * cadre_allreduce_flag_bytes() bytes, also symmetric memory (cadre_b200/collective.py obtains all of them from
 * torch.distributed._symmetric_memory). cadre_allreduce_sum reduces [offset, offset + count) (floats, multiples of 4);
 * all ranks must issue the same sequence of calls. use_multicast = 1: in-switch reduction (multimem.ld_reduce /
 * multimem.st); 0: peer loads summed in rank order + peer stores. cadre_allreduce_check synchronises and fails if a
 * barrier ever timed out (polling is bounded; a lost peer cannot hang the GPU). */
int cadre_allreduce_flag_bytes(void);
int cadre_allreduce_create(void** handle, int rank, int world, float* const* buffer_ptrs_host, float* multicast,
                           uint32_t* const* flag_ptrs_host, int64_t count);
/* thread blocks of 256 threads per launch (default 32, at most 256): every rank must use the same value for the same call */
int cadre_allreduce_set_blocks(void* handle, int blocks);
int cadre_allreduce_destroy(void* handle);
int cadre_allreduce_sum(void* handle, int64_t offset, int64_t count, int use_multicast, void* stream);
int cadre_allreduce_check(void* handle);

#ifdef __cplusplus
}
#endif
#endif /* CADRE_B200_H_ */

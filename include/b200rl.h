/*
 * b200rl.h -- C-ABI of libb200rl.so: the B200-native (sm_100a) PPO hot path.
 *
 * The reference (vwxyzjn/cleanrl) is pure Python/PyTorch and has NO native
 * interface; this header is the boundary SURVEY.md section 8(b) defines for it.
 * Every entry point replaces a block of torch calls inside the reference's
 * training loop (file:line cited per function, relative to the reference root).
 *
 * Conventions
 *   - plain C: raw DEVICE pointers + explicit sizes, scalars by value.  No
 *     torch / C++ types.  The caller (PyTorch in the shipped host code) owns
 *     every buffer including workspaces; nothing here allocates or frees
 *     device memory, and nothing synchronises the device.
 *   - every function only ENQUEUES work on `stream` (a cudaStream_t passed as
 *     void*; NULL = legacy default stream) and is CUDA-graph capturable.
 *   - return value: 0 on success, negative b200rl_status on failure.  The
 *     failing call's message is kept per host thread: b200rl_last_error().
 *   - "f32" = IEEE binary32.  All matrices are dense row-major unless a leading
 *     dimension / layout is spelled out.
 *   - python-double hyper-parameters (gamma, lr, betas, eps ...) are passed as
 *     double and rounded exactly where the reference rounds them.
 */
#ifndef B200RL_H
#define B200RL_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    B200RL_OK = 0,
    B200RL_ERR_INVALID_ARGUMENT = -1,
    B200RL_ERR_CUDA = -2,
    B200RL_ERR_UNSUPPORTED = -3,
    B200RL_ERR_WORKSPACE = -4
} b200rl_status;

/* library version: major*10000 + minor*100 + patch */
int b200rl_version(void);
/* message of the last failing call on this host thread ("" if none) */
const char* b200rl_last_error(void);
/* compute capability the kernels were compiled for (100 = sm_100a) */
int b200rl_compiled_arch(void);

/* Optional per-kernel timing: when enabled, every kernel launch below is bracketed by CUDA events
 * on its stream.  b200rl_profile_summary synchronises the device and writes a JSON array
 * [{"name","launches","ms","flops","bytes"}] (algorithmic flops/bytes per kernel family) into buf.
 * Do not enable during CUDA-graph capture. */
/* number of kernels this library has launched in this process (host-side counter) */
long long b200rl_launch_count(void);
void b200rl_profile_enable(int on);
void b200rl_profile_reset(void);
int b200rl_profile_summary(char* buf, size_t capacity);

/* ---------------------------------------------------------------- GAE -----
 * Reverse-scan generalised advantage estimation over a (T x N) rollout.
 * Replaces the python loop cleanrl/ppo.py:218-231 (identical in
 * ppo_atari_envpool.py:250-263, ppo_atari_multigpu.py:288-301,
 * ppo_continuous_action.py:233-246).
 *   rewards, values, dones : f32 [T, N] (N contiguous)
 *   next_value, next_done  : f32 [N]
 *   advantages, returns    : f32 [T, N] out  (returns = advantages + values)
 *   gamma, gae_lambda      : python doubles; gamma -> f32 once,
 *                            gamma*gae_lambda -> f32 once (ppo.py:230)
 *   mode 0: one thread per env, every op individually rounded (no FMA):
 *           bit-identical to the reference loop.
 *   mode 1: time-chunked affine scan (3 short dependent phases instead of T
 *           steps); re-associated, |err| ~1e-7 relative.
 */
int b200rl_gae_f32(const float* rewards, const float* values, const float* dones,
                   const float* next_value, const float* next_done,
                   float* advantages, float* returns,
                   int64_t T, int64_t N, double gamma, double gae_lambda,
                   int mode, void* stream);

/* ------------------------------------------------ categorical policy head --
 * Rollout-side policy epilogue.  Replaces Categorical(logits) + sample() +
 * log_prob() + entropy() in Agent.get_action_and_value
 * (cleanrl/ppo_atari_envpool.py:143-149, cleanrl/ppo.py:121-126) and the four
 * rollout-buffer stores ppo.py:200-202.
 *   logits  : f32 [n, A], row stride ld_logits elements
 *   noise   : f32 [n, A] Exp(1) draws from the CALLER's generator (torch's
 *             multinomial consumes exactly `empty_like(probs).exponential_(1)`),
 *             action = argmax(softmax(normalised logits) / noise), first max wins.
 *   value_in: optional f32 [n] (stride ld_value) copied to value_out (may be NULL)
 *   outputs : action i64 [n], logprob f32 [n], entropy f32 [n] (entropy may be NULL)
 */
int b200rl_categorical_sample_f32(const float* logits, int64_t ld_logits, const float* noise,
                                  const float* value_in, int64_t ld_value,
                                  int64_t n, int A,
                                  int64_t* action, float* logprob, float* entropy, float* value_out,
                                  void* stream);

/* log_prob and entropy of GIVEN actions (the action != None branch of
 * Agent.get_action_and_value, cleanrl/ppo.py:121-126).  action i64 [n] (clamped to [0,A)). */
int b200rl_categorical_eval_f32(const float* logits, int64_t ld_logits, const int64_t* action,
                                int64_t n, int A, float* logprob, float* entropy, void* stream);

/* -------------------------------------------------------------- PPO loss ---
 * Fused minibatch loss: gather by mb_inds, advantage normalisation (unbiased
 * std), ratio, both KL estimates, clipfrac, clipped surrogate, clipped value
 * loss, entropy bonus, AND the gradients wrt the policy logits / value that
 * autograd would produce.  Replaces cleanrl/ppo.py:250-285 (+ the part of
 * loss.backward() :288 above the network).
 *   new_logits : f32 [M, A] (row stride ld_logits); new_value: f32 [M] (stride ld_value)
 *   mb_inds    : i64 [M] rows of the flat batch (NULL = 0..M-1)
 *   b_*        : flat batch tensors of length B >= max(mb_inds)+1
 *                b_actions i64, b_logprobs/b_advantages/b_returns/b_values f32
 *   dlogits    : f32 [M, A] (row stride ld_dlogits) out; dvalue: f32 [M] (stride ld_dvalue) out
 *   stats      : f32 [16] out: 0 pg_loss, 1 v_loss, 2 entropy, 3 old_approx_kl,
 *                4 approx_kl, 5 clipfrac, 6 loss, 7 adv_mean, 8 adv_std
 *   workspace  : >= b200rl_ppo_loss_workspace_bytes(M) bytes, 16-B aligned.
 * Deterministic: fixed-order two-level reductions, no float atomics.
 */
size_t b200rl_ppo_loss_workspace_bytes(int64_t M);
int b200rl_ppo_loss_f32(const float* new_logits, int64_t ld_logits,
                        const float* new_value, int64_t ld_value,
                        const int64_t* mb_inds,
                        const int64_t* b_actions, const float* b_logprobs,
                        const float* b_advantages, const float* b_returns, const float* b_values,
                        int64_t M, int A,
                        double clip_coef, double ent_coef, double vf_coef,
                        int norm_adv, int clip_vloss,
                        float* dlogits, int64_t ld_dlogits, float* dvalue, int64_t ld_dvalue,
                        float* stats, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------ diagonal Gaussian policy --
 * Continuous-action twin of the three entry points above (cleanrl/ppo_continuous_action.py:134-141:
 * Normal(action_mean, exp(actor_logstd)), log_prob(a).sum(1), entropy().sum(1)).
 *   mean f32 [n, D] (row stride ld_mean), logstd f32 [D] (the state-independent actor_logstd parameter),
 *   noise f32 [n, D] N(0,1) from the caller's generator (torch.normal(mean, std) == randn*std + mean),
 *   action f32 [n, D].  The loss additionally returns dlogstd [D] (deterministic batch reduction).
 */
int b200rl_gaussian_sample_f32(const float* mean, int64_t ld_mean, const float* logstd, const float* noise,
                               const float* value_in, int64_t ld_value, int64_t n, int D,
                               float* action, float* logprob, float* entropy, float* value_out, void* stream);
int b200rl_gaussian_eval_f32(const float* mean, int64_t ld_mean, const float* logstd, const float* action,
                             int64_t n, int D, float* logprob, float* entropy, void* stream);
size_t b200rl_ppo_loss_gaussian_workspace_bytes(int64_t M);
int b200rl_ppo_loss_gaussian_f32(const float* new_mean, int64_t ld_mean, const float* logstd,
                                 const float* new_value, int64_t ld_value, const int64_t* mb_inds,
                                 const float* b_actions, const float* b_logprobs,
                                 const float* b_advantages, const float* b_returns, const float* b_values,
                                 int64_t M, int D, double clip_coef, double ent_coef, double vf_coef,
                                 int norm_adv, int clip_vloss,
                                 float* dmean, int64_t ld_dmean, float* dlogstd, float* dvalue, int64_t ld_dvalue,
                                 float* stats, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------- grad clip + Adam step ---
 * One fused optimiser step over a FLAT f32 parameter vector: optional DP
 * averaging (grads hold the all-reduced SUM; divided by world_size first, as
 * ppo_atari_multigpu.py:369-373 does), global-L2 clip_grad_norm_
 * (torch/nn/utils/clip_grad.py: coef = max_norm/(norm+1e-6) clamped to 1) and
 * Adam (torch/optim/adam.py _single_tensor_adam op order).  Replaces
 * cleanrl/ppo.py:289-290.
 *   params, exp_avg, exp_avg_sq : f32 [P] in/out;  grads: f32 [P] in
 *   step       : 1-based count of this step (bias corrections in double)
 *   max_norm   : < 0 disables clipping (dqn_atari.py has none)
 *   norm_out   : optional f32 [1] device scalar receiving the pre-clip norm
 *   workspace  : >= b200rl_clip_adam_workspace_bytes(P) bytes
 */
size_t b200rl_clip_adam_workspace_bytes(int64_t P);
int b200rl_clip_adam_f32(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                         int64_t P, int64_t step, double lr, double beta1, double beta2, double eps,
                         double max_norm, int world_size, float* norm_out,
                         void* workspace, size_t workspace_bytes, void* stream);
/* The same update with the two scalars that depend on (step, lr) -- sqrt(1 - beta2^step) and -lr / (1 - beta1^step), computed
 * on the host in double by b200rl_adam_step_scalars exactly as the by-value entry point computes them -- read from DEVICE
 * memory (step_scalars f32[2]): a captured CUDA graph of the update can be replayed for every later step / learning rate. */
int b200rl_adam_step_scalars(int64_t step, double lr, double beta1, double beta2, float* out2);
int b200rl_clip_adam_dyn_f32(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                             int64_t P, const float* step_scalars, double beta1, double beta2, double eps,
                             double max_norm, int world_size, float* norm_out,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------ fp32 network layers ------
 * Exact-arithmetic (fp32 FMA, CUDA cores) layers in the reference's own NCHW /
 * [out,in] layouts.  They carry configs 1 and 4 (64-wide MLPs,
 * cleanrl/ppo.py:100-116, ppo_continuous_action.py:112-129) and are the
 * validation mode of the NatureCNN (ppo_atari_envpool.py:123-139); the bf16
 * tensor-core path below is the fast path.
 *
 * act: 0 none, 1 ReLU, 2 tanh.  `rows` (i64, may be NULL) gathers the batch
 * dimension of x: sample i of the call reads x[rows[i]] (the minibatch gather
 * ppo.py:250 `b_obs[mb_inds]` without materialising it).
 */
enum { B200RL_ACT_NONE = 0, B200RL_ACT_RELU = 1, B200RL_ACT_TANH = 2 };
enum { B200RL_DT_F32 = 0, B200RL_DT_U8 = 1 };

/* y[n,Cout,OH,OW] = act(conv(x[n,Cin,H,W] / in_div, w[Cout,Cin,KH,KW]) + b)  (in_div = 255 for uint8 obs, 1 otherwise) */
int b200rl_conv2d_fwd_f32(const void* x, int x_dtype, const int64_t* rows, double in_div,
                          const float* w, const float* b, float* y,
                          int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride,
                          int act, void* stream);
/* Same with zero padding `pad` on every side (IMPALA-CNN 3x3 convolutions, cleanrl/ppo_procgen.py:92-93,110). */
int b200rl_conv2d_fwd_pad_f32(const void* x, int x_dtype, const int64_t* rows, double in_div,
                              const float* w, const float* b, float* y,
                              int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride, int pad,
                              int act, void* stream);
int b200rl_conv2d_bwd_data_pad_f32(const float* dy, const float* w, const float* x_post, int prev_act, float* dx,
                                   int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride, int pad, void* stream);
size_t b200rl_conv2d_bwd_weight_pad_workspace_bytes(int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride, int pad);
int b200rl_conv2d_bwd_weight_pad_f32(const void* x, int x_dtype, const int64_t* rows, double in_div,
                                     const float* dy, float* dw, float* db,
                                     int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride, int pad,
                                     void* workspace, size_t workspace_bytes, void* stream);
/* IMPALA-CNN glue (cleanrl/ppo_procgen.py:89-150), fp32 NCHW:
 *   maxpool3s2: max_pool2d(kernel 3, stride 2, padding 1) on [nc, H, W] planes -> [nc, (H+1)/2, (W+1)/2]; argmax u8 (0..8)
 *   relu / relu_bwd (dx = dy * (x > 0) + extra, extra may be NULL) / add: pre-activation residual blocks
 *   nhwc_to_nchw_u8: frames [n, H, W, C] (optionally gathered through rows) -> [n, C, H, W] */
int b200rl_maxpool3s2_fwd_f32(const float* x, int64_t nc, int H, int W, float* y, uint8_t* argmax, void* stream);
int b200rl_maxpool3s2_bwd_f32(const float* dy, const uint8_t* argmax, int64_t nc, int H, int W, float* dx, void* stream);
int b200rl_relu_f32(const float* x, int64_t n, float* y, void* stream);
int b200rl_relu_bwd_f32(const float* dy, const float* x, const float* extra, int64_t n, float* dx, void* stream);
int b200rl_add_f32(const float* a, const float* b, int64_t n, float* y, void* stream);
int b200rl_nhwc_to_nchw_u8(const uint8_t* x, const int64_t* rows, int64_t n, int H, int W, int C, uint8_t* y, void* stream);
/* dx = conv_transpose(dy, w) * act'(x_post) ; x_post = the layer input as the
 * previous layer's post-activation output (prev_act selects the derivative). */
int b200rl_conv2d_bwd_data_f32(const float* dy, const float* w, const float* x_post, int prev_act,
                               float* dx,
                               int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride,
                               void* stream);
/* dw[Cout,Cin,KH,KW] = sum_m dy * im2col(x / in_div) ; db[Cout] = sum dy.  Deterministic split
 * reduction through `workspace` (b200rl_conv2d_bwd_weight_workspace_bytes). */
size_t b200rl_conv2d_bwd_weight_workspace_bytes(int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride);
int b200rl_conv2d_bwd_weight_f32(const void* x, int x_dtype, const int64_t* rows, double in_div,
                                 const float* dy, float* dw, float* db,
                                 int64_t n, int Cin, int H, int W, int Cout, int KH, int KW, int stride,
                                 void* workspace, size_t workspace_bytes, void* stream);
/* y[n,out] = act(x[n,in] @ w[out,in]^T + b) ; x rows optionally gathered */
int b200rl_linear_fwd_f32(const float* x, const int64_t* rows, const float* w, const float* b, float* y,
                          int64_t n, int in_features, int out_features, int act, void* stream);
int b200rl_linear_bwd_data_f32(const float* dy, const float* w, const float* x_post, int prev_act, float* dx,
                               int64_t n, int in_features, int out_features, void* stream);
size_t b200rl_linear_bwd_weight_workspace_bytes(int64_t n, int in_features, int out_features);
int b200rl_linear_bwd_weight_f32(const float* x, const int64_t* rows, const float* dy, float* dw, float* db,
                                 int64_t n, int in_features, int out_features,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------- NatureCNN, bf16 tensor cores ---
 * The throughput path of Agent.network/actor/critic (cleanrl/ppo_atari_envpool.py:123-149):
 * every conv / linear contraction (forward, data-gradient, weight-gradient) is an implicit GEMM
 * on tcgen05.mma with bf16 operands and fp32 accumulation in TMEM, fed by TMA; a minibatch gather
 * (rows) is the image coordinate of conv1's TMA boxes, nothing is materialised; the two heads
 * (A+1 outputs, 1 <= A <= 23) run in fp32 on CUDA cores.
 *
 * params / grads: ONE flat f32 vector in libb200rl order
 *     conv1.w[32,4,8,8] conv1.b[32] conv2.w[64,32,4,4] conv2.b[64] conv3.w[64,64,3,3] conv3.b[64]
 *     fc.w[512,3136] fc.b[512] actor.w[A,512] critic.w[1,512] actor.b[A] critic.b[1]
 *   (each tensor in torch's own element order; b200rl_naturecnn_param_count(A) elements).
 * packed : bf16 GEMM operand copies of the weights (b200rl_naturecnn_bf16_packed_bytes), refreshed
 *          by b200rl_naturecnn_bf16_pack after every optimiser step.
 * acts   : activation + activation-gradient workspace for batch n (b200rl_naturecnn_bf16_acts_bytes);
 *          forward fills it, backward consumes it.  The caller must ZERO it once before its first use
 *          with a given n (zero-padded gradient grids rely on never-written positions staying 0).
 * obs    : obs_format B200RL_OBS_U8_NCHW  : uint8 [*, 4, 84, 84] frames as the env delivers them, or
 *          obs_format B200RL_OBS_S2D_BF16 : bf16 [*, 21, 21, 64] space-to-depth frames produced ONCE per
 *          env step by b200rl_frames_to_s2d_bf16 (channel = c*16 + sy*4 + sx of pixel (4Y+sy, 4X+sx)):
 *          conv1 (8x8 stride 4) is then a 2x2 stride-1 convolution over 128-byte pixels and the 16
 *          minibatch passes of an iteration never touch / convert the uint8 frames again.
 *          rows (i64 [n], may be NULL) selects the samples (ppo.py:250 gather) in either format; the
 *          indices are the caller's contract (not range-checked); ascending order keeps the gather
 *          DRAM-page friendly (the engine sorts every minibatch).
 * head_out / dhead : f32 [n, A+1] = [logits | value] and its gradient.
 */
enum { B200RL_OBS_U8_NCHW = 0, B200RL_OBS_S2D_BF16 = 1, B200RL_OBS_S2D_U8 = 2 };
int b200rl_frames_to_s2d_bf16(const uint8_t* obs, const int64_t* rows, int64_t n, void* out_s2d, void* stream);
/* B200RL_OBS_S2D_U8: the rollout keeps each frame as uint8 space-to-depth(4) pixels (28 224 B, the algorithmic minimum;
 * reference: fp32, 112 896 B, ppo_atari_envpool.py:203) in TWO orientations written once per env step:
 *   out_rm u8 [n, 441 grid rows, 64 channels]  -> `obs` of forward: conv1 on the integer tensor cores (kind::i8)
 *   out_cm u8 [n, 64 channels, 448 grid rows]  -> `obs_aux` of backward: conv1 weight gradient (pixels converted
 *                                                  uint8 -> fp16 in registers, fed to the MMA from tensor memory)
 * channel = c*16 + sy*4 + sx of source pixel (4Y+sy, 4X+sx), grid row = Y*21 + X; rows 441..447 of out_cm are zero. */
int b200rl_frames_to_s2d_u8(const uint8_t* obs, const int64_t* rows, int64_t n, uint8_t* out_rm, uint8_t* out_cm, void* stream);
/* Frame-stack delta upload (csrc/frame_stack.cu).  The Atari observation the reference uploads whole every step
 * (cleanrl/ppo_atari_envpool.py:185-196 stack_num=4, :226,239 `torch.Tensor(next_obs).to(device)`) is a stack of the 4 newest
 * frames: planes 0..2 of an env's observation are planes 1..3 of its previous one unless the env was reset.  Only the newest
 * plane (7 056 B instead of 28 224 B per env) has to cross PCIe; the device rebuilds rollout slot t from slot t-1:
 *   new_planes  u8 [n, 7056]   newest plane of every env
 *   full_slot   i32 [n] or NULL: -1 = shifted stack, k >= 0 = take all 4 planes from full_frames[k] (u8 [*, 4, 84, 84])
 *   prev_rm/prev_cm            the previous slot in the two B200RL_OBS_S2D_U8 orientations (must not alias the outputs) */
int b200rl_frames_delta_s2d_u8(const uint8_t* new_planes, const int32_t* full_slot, const uint8_t* full_frames,
                               const uint8_t* prev_rm, const uint8_t* prev_cm, int64_t n,
                               uint8_t* out_rm, uint8_t* out_cm, void* stream);
/* rows x row_bytes from pitched (pinned) host memory into a dense device buffer (cudaMemcpy2DAsync): the newest planes are
 * uploaded straight from the env's own observation batch, no host-side packing. */
int b200rl_h2d_rows_async(void* dst, const void* src, int64_t src_pitch, int64_t row_bytes, int64_t rows, void* stream);
/* Host-side tracker, one per vector env (HOST pointers; no stream).  It owns a private mirror of every env's last
 * observation and a pool of `threads` worker threads (0 = run inline).
 *   begin(): env i's observation starts at obs + i*env_stride (planes contiguous).  Envs with done[i] != 0 (f32, may be NULL)
 *            -- and every env on the first pass / after invalidate() -- are staged as full frames: full_out[k] (pinned,
 *            [n, planes*plane_bytes]) and slot_out[i] = k; all other envs get slot_out[i] = -1.  new_out (pinned
 *            [n, plane_bytes], may be NULL when the caller uploads the newest planes from `obs` itself) receives the newest
 *            planes.  Returns the number of full frames (>= 0; negative = error) and starts the ASYNCHRONOUS verification:
 *            the workers memcmp the first planes-1 planes of every slot -1 env against the mirror and refresh the mirror.
 *            `obs` must stay unchanged until wait() returns.
 *   wait():  joins the verification; returns how many slot -1 envs did NOT hold the shifted stack (their indices, ascending,
 *            in mismatch_out i32 [n]): the caller must re-stage those as full frames and redo the step.  Every begin() must
 *            be followed by one wait(). */
void* b200rl_stackdelta_create(int64_t n_envs, int planes, int64_t plane_bytes, int threads);
void b200rl_stackdelta_destroy(void* tracker);
void b200rl_stackdelta_invalidate(void* tracker);
int64_t b200rl_stackdelta_begin(void* tracker, const uint8_t* obs, int64_t env_stride, const float* done,
                                uint8_t* new_out, uint8_t* full_out, int32_t* slot_out);
int64_t b200rl_stackdelta_wait(void* tracker, int32_t* mismatch_out);
/* One env group's whole rollout step in ONE host call (the grouped loop of PPOEngine.collect is bounded by per-step host
 * overhead once only a plane per env crosses PCIe).  `plan` is filled once per (step, group):
 *   launch(): begin() on `tracker` (NULL = nothing to upload: the slot is rebuilt from device data only), H2D of the staged
 *             full frames / slot table / newest planes on `copy_stream` (straight from `obs` when it is pinned memory, else
 *             through new_h), then per chunk c: main_stream waits h2d_event[c] and launches graph_exec[c] (a cudaGraphExec_t
 *             holding that chunk's storage rebuild + policy + sampler), records `consumed_event`, copies the actions D2H
 *             (actions_bytes > 0) and records d2h_event.  Returns the number of whole observations staged (or < 0).
 *   join():   cudaEventSynchronize(d2h_event) (may be NULL) + wait() on `tracker` (may be NULL / nothing pending -> 0). */
typedef struct B200rlPartLaunch {
    void* tracker;
    void* copy_stream;
    void* main_stream;
    void* consumed_event;
    int32_t n, nchunks;
    int32_t chunk_lo[4], chunk_hi[4];      /* env ranges of the chunks, relative to the group */
    void* h2d_event[4];
    void* graph_exec[4];
    uint8_t* new_d; int32_t* slot_d; uint8_t* full_d;     /* device staging of the group */
    uint8_t* new_h; uint8_t* full_h; int32_t* slot_h;     /* pinned host staging of the group */
    const void* actions_d; void* actions_h; int64_t actions_bytes; void* d2h_event;
} B200rlPartLaunch;
/* numpy.random.shuffle(x) of an int64 vector on the legacy MT19937 generator (the reference's minibatch shuffle,
 * cleanrl/ppo.py:245, driven by numpy's GLOBAL RandomState), restated natively and bit-exact: key624 / pos are the state
 * words of numpy.random.get_state(); both are advanced exactly as numpy would advance them. */
int b200rl_mt19937_shuffle_i64(uint32_t* key624, int32_t* pos, int64_t* data, int64_t n);
int64_t b200rl_stackdelta_launch(const B200rlPartLaunch* plan, const uint8_t* obs, int64_t env_stride, const float* done);
int64_t b200rl_stackdelta_join(void* tracker, void* d2h_event, int32_t* mismatch_out);
int64_t b200rl_naturecnn_param_count(int A);
size_t b200rl_naturecnn_bf16_packed_bytes(int A);
size_t b200rl_naturecnn_bf16_acts_bytes(int64_t n, int obs_format);
size_t b200rl_naturecnn_bf16_workspace_bytes(int64_t n, int A);
int b200rl_naturecnn_bf16_pack(const float* params, int A, void* packed, void* stream);
int b200rl_naturecnn_bf16_forward(const void* obs, int obs_format, const int64_t* rows, int64_t n, int A,
                                  const float* params, const void* packed, void* acts,
                                  float* head_out, void* stream);
/* One rollout policy step of the bf16 NatureCNN on the uint8 rollout layout: conv tower (conv1..conv3 per image in
 * shared memory) -> fc -> heads + Categorical sample, writing action / logprob / value of n rows.  frames != NULL: uint8
 * [n,4,84,84] frames, both slot orientations (slot_rm [n,441,64], slot_cm [n,64,448]) are written from them; frames ==
 * NULL: slot_rm already holds the space-to-depth frames (slot_cm unused).  acts: the workspace of
 * b200rl_naturecnn_bf16_acts_bytes(n, B200RL_OBS_S2D_U8); noise: Exp(1) draws [n, A].  Same results, bit for bit, as
 * b200rl_frames_to_s2d_u8 + b200rl_naturecnn_bf16_forward + b200rl_categorical_sample_f32. */
int b200rl_naturecnn_bf16_rollout_step(const uint8_t* frames, uint8_t* slot_rm, uint8_t* slot_cm, int64_t n, int A,
                                       const float* params, const void* packed, void* acts, const float* noise,
                                       int64_t* action, float* logprob, float* value, void* stream);
int b200rl_naturecnn_bf16_backward(const void* obs, const void* obs_aux, int obs_format, const int64_t* rows, int64_t n, int A,
                                   const float* params, const void* packed, void* acts,
                                   const float* dhead, float* grads,
                                   void* workspace, size_t workspace_bytes, void* tail_ready_event, void* stream);
/* Data-parallel overlap (cleanrl/ppo_atari_multigpu.py:360-374 exchanges the gradient after the whole backward):
 * the backward finishes the head and fc gradients FIRST; they are the contiguous tail
 * grads[b200rl_naturecnn_grad_tail_offset(A) .. param_count) = 95 % of the vector.  When `tail_ready_event`
 * (a cudaEvent_t, may be NULL) is given, it is recorded on `stream` at that point, so the caller can all-reduce the
 * tail on another stream while the convolution gradients are still being computed. */
int64_t b200rl_naturecnn_grad_tail_offset(int A);

/* ------------------------------------------------------------ LSTM cell ---
 * Recurrent PPO agent (cleanrl/ppo_atari_lstm.py:117-160: nn.LSTM(512, 128), gate order i, f, g, o; the state is reset
 * by (1 - done) BEFORE the cell, :137-142).  The gate GEMMs are b200rl_linear_fwd_f32 calls (x W_ih^T + b_ih for all
 * steps at once, h' W_hh^T + b_hh per step); these are the elementwise parts, fp32, [n, H] row-major.
 *   mask_state : (h', c') = (1 - done[n]) * (h, c)
 *   cell_fwd   : gates_x, gates_h [n, 4H] -> h_out, c_out [n, H]; save [n, 5H] = (i, f, g, o, tanh c), may be NULL
 *   cell_bwd   : one BPTT step.  dh = dh_heads + (1 - done_next) * dh_rec_raw (dh_rec_raw = dgates_{t+1} W_hh, NULL at the
 *                last step), dc = dc_rec (NULL at the last step) + dh o (1 - tanh(c)^2); writes the pre-activation gate
 *                gradients dgates [n, 4H] and dc_rec_out = (1 - done) dc f for step t-1. */
int b200rl_lstm_mask_state_f32(const float* h, const float* c, const float* done, int64_t n, int H,
                               float* h_masked, float* c_masked, void* stream);
int b200rl_lstm_cell_fwd_f32(const float* gates_x, const float* gates_h, const float* c_masked, int64_t n, int H,
                             float* h_out, float* c_out, float* save, void* stream);
int b200rl_lstm_cell_bwd_f32(const float* dh_heads, const float* dh_rec_raw, const float* done_next, const float* dc_rec,
                             const float* save, const float* c_masked, const float* done, int64_t n, int H,
                             float* dgates, float* dc_rec_out, void* stream);

/* --------------------------------------------------------- DQN TD update ---
 * td_target = r + gamma * max_a' Q_target(s')[a'] * (1 - done); old = Q(s)[a]; loss = mean((td - old)^2)
 * (F.mse_loss, cleanrl/dqn_atari.py:220-224; huber = 1: smooth-L1) and dL/dQ [B, A] in one pass.
 *   q, q_target_next : f32 [B, A] (row strides ld_q, ld_qt); actions i64 [B]; rewards, dones f32 [B]
 *   dq f32 [B, A] out; stats f32 [2] out: td_loss, mean chosen Q (the two logged scalars, dqn_atari.py:227-228)
 * b200rl_argmax_f32: greedy action of the epsilon-greedy policy (dqn_atari.py:192-193), first maximum.
 */
size_t b200rl_dqn_td_loss_workspace_bytes(int64_t B);
int b200rl_dqn_td_loss_f32(const float* q, int64_t ld_q, const float* q_target_next, int64_t ld_qt,
                           const int64_t* actions, const float* rewards, const float* dones,
                           int64_t B, int A, double gamma, int huber,
                           float* dq, int64_t ld_dq, float* stats,
                           void* workspace, size_t workspace_bytes, void* stream);
int b200rl_argmax_f32(const float* q, int64_t ld_q, int64_t n, int A, int64_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200RL_H */

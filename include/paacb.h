/* paacb.h -- C ABI of the B200-native PAAC rollout-and-update hot path.
 *
 * The reference (arjunchandra/paac) has no native code: its hot path is Python calling
 * TensorFlow-1 ops through session.run, NumPy and PIL.  This header is the boundary a
 * maintainer binds (ctypes stub in INTEGRATION.md) to replace those calls.  Each entry
 * point cites the reference interface it stands in for (file:line in the upstream repo).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - every pointer named d_* is DEVICE memory (or pinned+mapped host memory for d_frames);
 *     the caller owns every buffer; the library allocates no device memory on the path (a context owns
 *     only its operand images of the weights, made by paacb_set_math, and a 256-byte grid-barrier block).
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), does no
 *     host synchronisation and no allocation, so a sequence of calls can be captured in a
 *     CUDA graph by the caller.
 *   - return 0 on success, a negative PAACB_E* code otherwise; paacb_last_error() gives the
 *     message (thread-local).  No exceptions cross the boundary.
 *   - layouts are the reference's: states NHWC uint8 [b,84,84,4] (oldest frame = channel 0),
 *     conv weights HWIO, fc weights [in,out]; all parameters live in ONE flat fp32 buffer in
 *     TF variable-creation order (paacb_tensor_info gives name/offset/shape).
 *   - one context per GPU per process; a context is immutable after paacb_set_* calls and may
 *     be used from one host thread at a time.  Calls on DIFFERENT streams may overlap on the device only while the
 *     parameters do not change (the acting and training forwards of one rollout): the cached operand images of the
 *     weights are written by paacb_clip_rmsprop / the first forward after paacb_params_changed and read by every forward.
 *   - the CURRENT CUDA device of the calling thread must be the context's device (PAACB_EINVAL otherwise): launches,
 *     kernel attributes and tensor maps all belong to it.
 */
#ifndef PAACB_H
#define PAACB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PAACB_VERSION 102
#define PAACB_MAX_ACTIONS 18          /* ALE full action set */
#define PAACB_MAX_TENSORS 12
#define PAACB_FRAME_H 210
#define PAACB_FRAME_W 160
#define PAACB_OBS 84
#define PAACB_STACK 4

enum { PAACB_OK = 0, PAACB_EINVAL = -1, PAACB_ECUDA = -2, PAACB_EUNSUPPORTED = -3 };
enum { PAACB_ARCH_NIPS = 0, PAACB_ARCH_NATURE = 1 };
/* arithmetic of the conv/fc contractions */
enum { PAACB_MATH_FP32 = 0,      /* SIMT fp32 FFMA: the parity anchor */
       PAACB_MATH_TF32X3 = 1,    /* tcgen05 kind::tf32, split operands (hi*hi + hi*lo + lo*hi) */
       PAACB_MATH_TF32 = 2,      /* tcgen05 kind::tf32, operands rounded to nearest tf32 */
       PAACB_MATH_BF16X3 = 3 };  /* tcgen05 kind::f16 on bf16-split operands (hi*hi + hi*lo + lo*hi), activations kept as
                                    two bf16 planes, TMA-fed patch-resident implicit GEMMs; both architectures */
enum { PAACB_CLIP_IGNORE = 0, PAACB_CLIP_GLOBAL = 1 };   /* actor_learner.py:51-58 ('local' is broken upstream) */

typedef struct paacb_ctx paacb_ctx;
typedef void* paacb_stream;           /* cudaStream_t */

int paacb_version(void);
const char* paacb_last_error(void);

/* ---- context: replaces graph construction, networks.py:102-169 + policy_v_network.py:6-57 ------ */
int paacb_create(paacb_ctx** out, int arch, int num_actions, int device);
int paacb_destroy(paacb_ctx* ctx);
int paacb_set_math(paacb_ctx* ctx, int math_mode);
int paacb_get_math(const paacb_ctx* ctx);
/* Multi-GPU: leave n_sms SMs free of the persistent conv weight-gradient CTAs (PAACB_BWD_HEAD), the kernels that run
 * while the caller's collective reduces the gradient tail, so that the collective's CTAs can be scheduled beside them. */
int paacb_set_sm_reserve(paacb_ctx* ctx, int n_sms);
/* The tensor-core modes keep operand images of the parameters (bf16 hi/lo transposes, int8 digits of conv1) in the
 * context and reuse them across forwards of the same d_params pointer: PAAC runs t_max + 2 forwards per parameter
 * update.  paacb_clip_rmsprop refreshes the images itself; a caller that writes the parameter buffer by any other
 * means (initialisation, checkpoint restore, broadcast) MUST call paacb_params_changed() afterwards. */
int paacb_params_changed(paacb_ctx* ctx);
/* nearest-resize index tables, out[y][x] = in[row[y]][col[x]]; defaults are Pillow's for
 * 210x160 -> 84x84 (what scipy.misc.imresize(..., 'nearest') used, atari_emulator.py:73). */
int paacb_set_resize_tables(paacb_ctx* ctx, const int32_t* row84, const int32_t* col84);

/* ---- parameter layout (TF variable order, SURVEY App. B) ---------------------------------------- */
int64_t paacb_param_count(const paacb_ctx* ctx);
int paacb_num_tensors(const paacb_ctx* ctx);
int paacb_tensor_info(const paacb_ctx* ctx, int index, char* name, int name_cap,
                      int64_t* offset, int* ndim, int64_t shape[4], int64_t* fan_in);
/* floats of scratch the forward / backward need for a batch of b samples */
int64_t paacb_forward_workspace_floats(const paacb_ctx* ctx, int64_t batch);
int64_t paacb_backward_workspace_floats(const paacb_ctx* ctx, int64_t batch);
/* floats of scratch paacb_clip_rmsprop needs */
int64_t paacb_optimizer_workspace_floats(const paacb_ctx* ctx);

/* ---- K1: observation pipeline.  Replaces FramePool/np.amax + imresize + ObservationPool
 * (atari_emulator.py:69-75, environment.py:42-75) and the reset rule of emulator_runner.py:26-27.
 *   d_frames      uint8 [n_envs, pairs_per_env, 2, 210, 160]  raw luminance frame pairs
 *                 (device memory or pinned+mapped host memory written by the ALE runners)
 *   pairs_per_env 1 or 4.  Slot 0 is this step's pair.  When d_reset[n] != 0 (needs 4 slots) the
 *                 four slots hold the four action-repeat pairs of get_initial_state(), oldest first.
 *   d_reset       uint8 [n_envs] or NULL
 *   d_prev        uint8 [n_envs,84,84,4] state before the step; d_next the state after (may alias d_prev). */
int paacb_preprocess_u8(const paacb_ctx* ctx, const uint8_t* d_frames, int pairs_per_env,
                        const uint8_t* d_reset, const uint8_t* d_prev, uint8_t* d_next,
                        int64_t n_envs, paacb_stream stream);

/* K1 plus the per-step rollout bookkeeping of paac.py:119-123 in the same launch:
 *   d_rewards_out[n] = d_rewards_in[n], d_over_out[n] = d_over_in[n]   (row t of the [T, N] rollout buffers; reward
 *   clipping happens in K7).  The *_in arrays are the runners' shared reward / episode_over arrays (device memory, or
 *   pinned+mapped host memory: runners.py:12-16 + paacb_host_register).  over_is_reset != 0: d_over_in[n] != 0 is also
 *   environment n's reset flag (emulator_runner.py:26-27; needs pairs_per_env == 4), OR-ed with d_reset when given. */
int paacb_observe_u8(const paacb_ctx* ctx, const uint8_t* d_frames, int pairs_per_env, const uint8_t* d_reset,
                     const uint8_t* d_prev, uint8_t* d_next, int64_t n_envs, const float* d_rewards_in,
                     const float* d_over_in, float* d_rewards_out, float* d_over_out, int over_is_reset,
                     paacb_stream stream);

/* ---- K2-K6: forward (+ sampling).  Replaces session.run([output_layer_v, output_layer_pi])
 * and __sample_policy_action (paac.py:18-45).
 *   d_params   float [P]               d_states uint8 [b,84,84,4]
 *   d_fwd_ws   float [paacb_forward_workspace_floats(b)]  activations, kept for paacb_backward
 *   d_pi       float [b,A]             d_v float [b]
 *   d_uniforms float [b] in [0,1) or NULL (no sampling); d_actions int32 [b] or NULL;
 *   d_onehot   float [b,A] or NULL (np.eye(A)[idx], paac.py:27) */
int paacb_policy_forward(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                         float* d_fwd_ws, float* d_pi, float* d_v,
                         const float* d_uniforms, int32_t* d_actions, float* d_onehot, paacb_stream stream);

/* The same forward writing samples [ws_first, ws_first + batch) of a workspace laid out for ws_capacity samples
 * (paacb_forward_workspace_floats(ws_capacity)).  PAAC's training batch is the concatenation of the t_max acting
 * batches (paac.py:92,112,151: states[t] is stored, then flattened to [T*N,...]) under UNCHANGED parameters, so the
 * learner can compute the training forward's activations step by step while the emulators run -- paacb_backward then
 * takes the assembled workspace with batch = ws_capacity.  Results are bit-identical to one forward over the whole
 * batch (every sample is computed by the same instruction sequence whatever its position in a launch). */
int paacb_policy_forward_at(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                            float* d_fwd_ws, int64_t ws_capacity, int64_t ws_first, float* d_pi, float* d_v,
                            const float* d_uniforms, int32_t* d_actions, float* d_onehot, paacb_stream stream);

/* The same forward with the sampling uniforms drawn INSIDE the heads kernel (K6, replaces np.random.multinomial of
 * paac.py:42-44 without a separate generator launch): Philox4x32-10, key = d_rng[0] (seed), counter =
 * (first_sample + i, d_rng[1] + draw_index) for sample i of this call, u = (first output word >> 8) * 2^-24.
 *   d_rng  uint64 [2] in device memory: {seed, draw base}.  paacb_rng_advance adds n to the base in stream order (once per
 *          update, n = t_max), so a captured CUDA graph of the rollout replays with fresh uniforms.
 *   first_sample  global index of this call's sample 0 (environment slices draw what the whole batch would). */
int paacb_policy_forward_sample(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                                float* d_fwd_ws, int64_t ws_capacity, int64_t ws_first, float* d_pi, float* d_v,
                                const uint64_t* d_rng, uint64_t draw_index, int64_t first_sample, int32_t* d_actions,
                                float* d_onehot, paacb_stream stream);
int paacb_rng_advance(const paacb_ctx* ctx, uint64_t* d_rng, uint64_t n, paacb_stream stream);

/* ---- K7+K8: n-step returns (paac.py:119,140-149; reward clip actor_learner.py:95-101) fused with the
 * A2C loss and its gradient w.r.t. logits and value (policy_v_network.py:29-57 + TF autodiff).
 *   d_rewards, d_episode_over, d_values  float [T,N] (raw reward, 0/1 flag, acting V(s_t))
 *   d_bootstrap_v float [N] = V(s_T);  d_actions int32 [T*N];  d_pi float [T*N,A], d_v float [T*N] from
 *   the training forward.  Outputs: d_y, d_adv float [T*N] (critic target, advantage; float64
 *   recurrence rounded to fp32 like the reference), d_dlogits float [T*N,A], d_dv float [T*N],
 *   d_loss float [1] (overwritten with the scalar loss). */
int paacb_returns_loss_grad(const paacb_ctx* ctx, const float* d_rewards, const float* d_episode_over,
                            const float* d_values, const float* d_bootstrap_v, const int32_t* d_actions,
                            const float* d_pi, const float* d_v, int t_max, int64_t n_envs,
                            double gamma, float entropy_beta,
                            float* d_y, float* d_adv, float* d_dlogits, float* d_dv, float* d_loss,
                            paacb_stream stream);

/* ---- K9: backward.  Replaces optimizer.compute_gradients(loss) (actor_learner.py:44).
 *   d_fwd_ws as left by paacb_policy_forward on the same (params, states, batch).
 *   d_grads float [P]: OVERWRITTEN with dLoss/dparams (flat, same layout as d_params). */
int paacb_backward(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                   const float* d_fwd_ws, const float* d_dlogits, const float* d_dv,
                   float* d_bwd_ws, float* d_grads, paacb_stream stream);

/* The same backward in two parts, for overlapping the gradient all-reduce with the rest of the backward (multi-GPU):
 *   PAACB_BWD_TAIL  zeroes d_grads, then computes every data gradient and the gradients of the hidden fc layer and of
 *                   both heads: d_grads[paacb_grad_tail_offset(ctx) .. P) is final (95 % of the parameters of either
 *                   architecture) and can be all-reduced while
 *   PAACB_BWD_HEAD  computes what is left of d_grads[0 .. tail offset) (the conv layers' weight gradients).
 * PAACB_BWD_ALL = both, what paacb_backward does. */
enum { PAACB_BWD_ALL = 0, PAACB_BWD_TAIL = 1, PAACB_BWD_HEAD = 2 };
int paacb_backward_part(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                        const float* d_fwd_ws, const float* d_dlogits, const float* d_dv,
                        float* d_bwd_ws, float* d_grads, int part, paacb_stream stream);
int64_t paacb_grad_tail_offset(const paacb_ctx* ctx);

/* ---- K10+K11: tf.clip_by_global_norm + ApplyRMSProp x10 (actor_learner.py:33-34,54-59,70).
 *   g = d_grads * grad_scale (1/world after an allreduce-sum); norm = ||g||_2;
 *   scale = clip * min(1/norm, 1/clip) (PAACB_CLIP_GLOBAL) or 1;  g *= scale;
 *   ms += (g*g - ms)*(1-rho); mom = momentum*mom + lr*g/sqrt(ms+eps); params -= mom.
 *   d_norm_out float [1] receives the (unclipped) global norm.  d_opt_ws: scratch. */
int paacb_clip_rmsprop(const paacb_ctx* ctx, float* d_params, float* d_ms, float* d_mom, const float* d_grads,
                       float grad_scale, float lr, float rho, float eps, float momentum,
                       float clip_norm, int clip_type, float* d_norm_out, float* d_opt_ws,
                       paacb_stream stream);

/* The same update with the learning rate read from DEVICE memory when the kernel runs (d_lr float [1]): a captured CUDA
 * graph of the update is replayed while the host anneals the rate (actor_learner.py:119-123) by writing that word. */
int paacb_clip_rmsprop_dlr(const paacb_ctx* ctx, float* d_params, float* d_ms, float* d_mom, const float* d_grads,
                           float grad_scale, const float* d_lr, float rho, float eps, float momentum,
                           float clip_norm, int clip_type, float* d_norm_out, float* d_opt_ws, paacb_stream stream);

/* ---- opt-in summaries (actor_learner.py:85-87, logger_utils.py:23-33): one pass over g = d_grads * grad_scale.
 *   d_out4 double [4] = {sum g, sum g^2, max g, min g}; mean / stddev / max / min of the RAW gradient follow on the host,
 *   those of the CLIPPED gradient are the raw ones times clip * min(1/norm, 1/clip) (the clip is one non-negative scalar),
 *   norm = sqrt(sum g^2).  d_opt_ws: the optimizer workspace (scratch).  Not on the hot path: call it when a record is due. */
int paacb_grad_stats(const paacb_ctx* ctx, const float* d_grads, float grad_scale, float* d_opt_ws, double* d_out4,
                     paacb_stream stream);

/* number of kernel launches issued through this context since creation (bench.py's gpu_launches) */
int64_t paacb_launch_count(const paacb_ctx* ctx);

/* ---- per-kernel timing with CUDA events on the launching stream (measurement aid, off by default).
 * While enabled every kernel launch is bracketed by two event records; paacb_profile_read(slot)
 * synchronises on the last recorded event and returns the accumulated device time and launch count
 * of one kernel family ("conv2_wgrad", "clip_rmsprop", ...; "unused" for absent layers). */
int paacb_profile_enable(paacb_ctx* ctx, int on);
int paacb_profile_reset(paacb_ctx* ctx);
int paacb_profile_slots(void);
int paacb_profile_read(const paacb_ctx* ctx, int slot, char* name, int name_cap, double* total_ms, int64_t* launches);

/* ---- shared-buffer plumbing for the Runners protocol (runners.py:12-16 allocates RawArray buffers
 * that forked workers write).  Page-locks an existing host range and maps it into the device address
 * space so paacb_preprocess_u8 can read the frames the workers wrote without a staging copy.
 * *d_ptr receives the device-side address.  Call from the process that owns the CUDA context. */
int paacb_host_register(void* host_ptr, size_t bytes, void** d_ptr);
int paacb_host_unregister(void* host_ptr);

#ifdef __cplusplus
}
#endif
#endif /* PAACB_H */

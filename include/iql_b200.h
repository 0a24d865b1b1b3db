/*
 * iql_b200.h -- C-ABI of the B200-native IQL(+JSRL) update engine.
 *
 * Plain C, no torch types: pointers are CUDA device pointers unless a
 * parameter says "host"; `stream` is a cudaStream_t passed as void*.
 * Every entry point returns IQL_OK (0) or an IQL_ERR_* code; the message for
 * the last failure is available through iql_last_error().
 *
 * The reference (LaurenYTaylor/jsrl-CORL) is pure Python and has no FFI layer;
 * its "boundary" is the class API of algorithms/finetune/iql.py.  Each entry
 * point below names the reference interface (file:line, relative to
 * /root/reference/algorithms/finetune/) it replaces.  The Python facade in
 * jsrl_corl_b200/ binds exactly these symbols with ctypes (INTEGRATION.md shows
 * the stub a reference maintainer would add).
 *
 * Ownership: the caller (torch) allocates every device buffer -- parameter /
 * Adam / target arenas, replay rows, workspace -- and the engine borrows the
 * pointers for the lifetime of the handle.  The library never cudaMalloc's.
 * Calls on one handle are not re-entrant.
 */
#ifndef IQL_B200_H
#define IQL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IQL_OK 0
#define IQL_ERR_INVALID 1 /* bad argument            -> ValueError            */
#define IQL_ERR_CUDA 2    /* CUDA runtime failure    -> RuntimeError          */
#define IQL_ERR_STATE 3   /* call order / not bound  -> RuntimeError          */
#define IQL_ERR_SHAPE 4   /* iql.py:530 "Actions shape missmatch" -> RuntimeError */

#define IQL_MATH_FP32_SIMT 0    /* CUDA-core FP32 validation path            */
#define IQL_MATH_TF32_TCGEN05 1 /* tcgen05.mma kind::tf32, FP32 accumulate   */

#define IQL_SAMPLE_PHILOX 0    /* indices drawn in-kernel (Philox4x32-10)     */
#define IQL_SAMPLE_INDICES 1   /* caller-supplied int64 indices [S][K][B]     */
#define IQL_SAMPLE_PRELOADED 2 /* batch already staged by iql_load_batch (K=1) */
#define IQL_SAMPLE_MT19937 3   /* numpy's RandomState.randint stream per member, drawn on the device (iql_bind_index_streams) */

/* One member's numpy index stream: uint32 words [key[624] | pos | pad], the ('MT19937', key, pos, ...) tuple of
 * RandomState.get_state() copied word for word (pos in [0, 624]; the pad word is not read). */
#define IQL_MT_STATE_WORDS 626

#define IQL_NET_Q1 0
#define IQL_NET_Q2 1
#define IQL_NET_V 2
#define IQL_NET_ACTOR 3

#define IQL_KIND_WEIGHT 0
#define IQL_KIND_BIAS 1
#define IQL_KIND_LOG_STD 2

typedef struct iql_engine iql_engine;

/* Shapes shared by all members of an ensemble (TwinQ / ValueFunction / policy
 * constructor arguments, iql.py:347-442; batch_size from TrainConfig iql.py:48). */
typedef struct iql_config {
  int32_t n_members;     /* S: independent seeds / hyper-parameter configs   */
  int32_t state_dim;
  int32_t action_dim;
  int32_t hidden_dim;    /* multiple of 4                                     */
  int32_t n_hidden;      /* >= 1                                              */
  int32_t batch_size;
  int32_t deterministic; /* 0 GaussianPolicy (iql.py:347), 1 DeterministicPolicy (iql.py:382) */
  int32_t math_mode;     /* IQL_MATH_*                                        */
  int32_t max_steps_per_call; /* K upper bound (loss ring size)               */
  int32_t reserved[7];
} iql_config;

/* Per-member hyper-parameters (ImplicitQLearning ctor iql.py:445-480, Adam
 * defaults jsrl_utils.py:263-265, CosineAnnealingLR iql.py:471).  Doubles, as
 * Python holds them; the engine derives the fp32 scalars the way torch does. */
typedef struct iql_hparams {
  double beta;
  double iql_tau;
  double discount;
  double tau; /* Polyak */
  double vf_lr, qf_lr, actor_lr; /* actor_lr = schedule base lr */
  double actor_dropout;
  double adam_beta1, adam_beta2, adam_eps;
  double lr_eta_min;
  int64_t cosine_t_max; /* 0: no schedule (max_steps=None, iql.py:472-473)  */
  uint64_t seed;        /* Philox key: index sampling and dropout masks     */
} iql_hparams;

/* Step counters of one member (checkpoint fields, iql.py:565-579). */
typedef struct iql_counters {
  int64_t v_step, q_step, actor_step; /* Adam state["step"]                  */
  int64_t sched_epoch;                /* CosineAnnealingLR.last_epoch        */
  int64_t total_it;                   /* ImplicitQLearning.total_it          */
  int64_t sample_step;                /* Philox sampling counter             */
} iql_counters;

/* Packed replay row: [ s(S) a(A) pad | s'(S) r d pad ], 16-byte aligned
 * segments, so one transition is ONE contiguous, float4-loadable row
 * (replaces the five SoA tensors of ReplayBuffer.__init__, iql.py:123-147). */
typedef struct iql_row_layout {
  int32_t state_dim, action_dim;
  int32_t row_floats; /* multiple of 4 */
  int32_t off_state, off_action, off_next_state, off_reward, off_done;
} iql_row_layout;

typedef struct iql_layout {
  int64_t param_floats;  /* per-member block size of params/exp_avg/exp_avg_sq arenas */
  int64_t q_floats;      /* leading part owned by the Q optimizer == per-member target block */
  int64_t v_begin, v_end;         /* V optimizer range inside the block        */
  int64_t actor_begin, actor_end; /* actor optimizer range                     */
  int64_t workspace_bytes;        /* for all members                           */
  int32_t n_tensors;              /* tensors per member block                  */
  int32_t reserved;
  iql_row_layout row;
} iql_layout;

typedef struct iql_tensor_info {
  int32_t net;   /* IQL_NET_*  */
  int32_t layer; /* Linear index 0..n_hidden */
  int32_t kind;  /* IQL_KIND_* */
  int32_t rows, cols; /* weight [rows, cols]; bias/log_std [rows], cols = 1 */
  int32_t ld;         /* row stride in floats (>= cols, multiple of 4 so that every row is 16-byte aligned for TMA) */
  int64_t offset; /* float offset inside the member block */
} iql_tensor_info;

const char* iql_version(void);
/* Message of the last failure on this handle (NULL handle: last failed create). */
const char* iql_last_error(const iql_engine* e);

/* ---- lifetime ---------------------------------------------------------- */
/* replaces: ImplicitQLearning.__init__ iql.py:445-480 (for S members at once) */
int iql_create(const iql_config* cfg, iql_engine** out);
void iql_destroy(iql_engine* e);
int iql_get_layout(const iql_engine* e, iql_layout* out);
int iql_tensor_at(const iql_engine* e, int32_t index, iql_tensor_info* out);

/* params / exp_avg / exp_avg_sq / grads: [S][param_floats]; target: [S][q_floats];
 * workspace: workspace_bytes.  All 128-byte aligned device memory. */
int iql_bind_state(iql_engine* e, float* params, float* exp_avg, float* exp_avg_sq,
                   float* target, float* grads, void* workspace, size_t workspace_bytes);
int iql_set_hparams(iql_engine* e, int32_t member, const iql_hparams* hp);
int iql_set_counters(iql_engine* e, int32_t member, const iql_counters* c);

/* Engine options (no counterpart in the reference: they select between equivalent B200 code paths and exist for
 * tests and measurements).  IQL_OPT_STEP_PATH must be set before iql_bind_state. */
#define IQL_OPT_STEP_PATH 1  /* 0 auto (default): 4 where it is supported and the ensemble has >= 8 members or >= 3 hidden layers, else 1;
                              1 one kernel per phase + adam_polyak; 2 chained backward + fused optimizer; 3 is not assigned;
                              4 chained backward (gradients only) + adam_polyak.  2 and 4: bind fails where unsupported --
                              the chain needs tf32, hidden 256, batch 256, 2..4 hidden layers, action_dim <= 24 and
                              state_dim + action_dim <= 256; auto takes 1 outside that */
#define IQL_OPT_KEEP_GRADS 2 /* != 0: the chained backward also stores the hidden / input weight gradients to `grads` */
int iql_set_option(iql_engine* e, int32_t key, int64_t value);
/* Which code path serves this handle (after iql_bind_state).  IQL_INFO_TENSOR_CORE_PATH == 0 under
 * IQL_MATH_TF32_TCGEN05 means the shape is outside the tcgen05 kernels (batch % 128, hidden % 256) and the FP32
 * CUDA-core kernels run instead: callers that require tensor cores must check it -- the Python facade raises when
 * math_mode="tf32" was asked for with strict=True. */
#define IQL_INFO_TENSOR_CORE_PATH 1
#define IQL_INFO_FUSED_FORWARD 2
#define IQL_INFO_CHAINED_BACKWARD 3       /* IQL_OPT_STEP_PATH 2: chained backward with the optimizer in its epilogue */
#define IQL_INFO_CHAINED_BACKWARD_GRADS 4 /* chained backward storing the gradients, adam_polyak after it (4, or auto) */
int iql_get_info(const iql_engine* e, int32_t key, int64_t* out);
int iql_get_counters(iql_engine* e, int32_t member, iql_counters* out, void* stream);
/* Per-member batch sizes (a batch-size axis of a hyper-parameter sweep, ray_hyperparam.py).  host_sizes[S] in HOST
 * memory, 1 <= B_m <= batch_size (default: every B_m = batch_size).  Member m trains on rows [0, B_m) of the engine's
 * batch: the gather writes zero rows past B_m and reads no index there, the losses and their gradients are means over
 * B_m rows, and the kernels still run on all batch_size rows (the shapes, tiles and kernel paths of the handle stay
 * those of batch_size).  In IQL_SAMPLE_PHILOX mode row b < B_m draws the index it draws at any batch size; idx_out
 * holds -1 past B_m.  Index entries past B_m (iql_train_steps, iql_train_host_step) are never read or checked.  Read by
 * the kernels at run time: a change takes effect at the next call without recapturing its graph.  iql_load_batch
 * refuses a member whose B_m != batch_size (IQL_ERR_STATE).  IQL_ERR_INVALID: a null pointer or a size out of range
 * (nothing is changed then). */
int iql_set_batch_sizes(iql_engine* e, const int32_t* host_sizes);
/* host_out[S]: the current B_m of every member. */
int iql_get_batch_sizes(iql_engine* e, int32_t* host_out);
/* Members that train (the early stopping of a hyper-parameter search, ray_hyperparam.py's ASHA scheduler).
 * host_ids[n]: member indices in HOST memory, any order, any non-empty subset; default: every member.  Retiring and
 * resuming are the same call.  The problem tables, tensor maps and chained-backward tasks are rebuilt over the listed
 * members only, so the others launch no CTA in any step, and every path choice that depends on the member count (auto
 * chained backward, CTA pairs, narrow dgrad tiles, the fused forward's wide epilogue, the tensor-core policy head) is
 * re-made from n; the workspace split chosen at iql_create (row-split output-layer backward, K-split input-layer
 * weight gradient) stays.  Inactive members are frozen: parameters, moments, target, gradients, counters and B_m keep
 * every bit, and a resumed member continues as if no time had passed.  They still serve iql_act*, inserts,
 * iql_sync_target and the tensor views.  Their iql_train_steps loss rows are NaN and their idx_out rows -1; their
 * iql_train_host_step / iql_host_step_wait losses are NaN; their index entries are never read or checked.  A host step
 * still in flight is collected first (its losses are dropped).  Host cost: the tensor maps are encoded again, and the
 * captured graphs are dropped.  IQL_ERR_INVALID: null ids, n < 1, an id out of range or listed twice (nothing changes);
 * IQL_ERR_STATE: before iql_bind_state. */
int iql_set_active_members(iql_engine* e, int32_t n, const int32_t* host_ids);
/* host_mask[S]: 1 for the members that train, 0 for the others. */
int iql_get_active_members(iql_engine* e, int8_t* host_mask);
/* replaces: copy.deepcopy(self.qf) iql.py:464,584,598 (q_target <- qf) */
int iql_sync_target(iql_engine* e, int32_t member, void* stream);

/* ---- replay data plane (no handle needed) -------------------------------- */
int iql_replay_row_layout(int32_t state_dim, int32_t action_dim, iql_row_layout* out);
/* replaces: ReplayBuffer.load_d4rl_dataset iql.py:153-169 (bulk pack of n rows
 * starting at row `first_row`; inputs are dense [n,S],[n,A],[n],[n,S],[n]) */
int iql_replay_pack(float* rows, const iql_row_layout* lay, int64_t first_row, int64_t n,
                    const float* states, const float* actions, const float* rewards,
                    const float* next_states, const float* dones, void* stream);
/* replaces: the dataset preprocessing in front of load_d4rl_dataset -- compute_mean_std / normalize_states
 * (iql.py:77-84; jsrl_w_iql.py:349-360) and the arithmetic of modify_reward (iql.py:286-297) -- fused with the pack:
 * normalize != 0 computes mean[S] and std[S] = sqrt(var) + eps of `states` with numpy's row-order fp32 summation
 * (bit-exact against states.mean(0) / states.std(0)), writes them to mean_out / std_out (device) and stores
 * (x - mean) / std for states and next_states; rewards are stored as (r / reward_div) * reward_mul - reward_sub
 * (pass 1, 1, 0 for none).  All inputs are dense device arrays as for iql_replay_pack. */
int iql_replay_ingest(float* rows, const iql_row_layout* lay, int64_t first_row, int64_t n, const float* states,
                      const float* actions, const float* rewards, const float* next_states, const float* dones,
                      int32_t normalize, float eps, float* mean_out, float* std_out, float reward_div, float reward_mul,
                      float reward_sub, void* stream);
/* replaces: ReplayBuffer.add_transition iql.py:180-196 (one fused row insert;
 * `staged_row` is a device row in packed layout) */
int iql_replay_insert(float* rows, const iql_row_layout* lay, int64_t pointer,
                      const float* staged_row, void* stream);
/* add_transition for a HOST caller (one env step of the online loop, jsrl_w_iql.py:470-478): state / action /
 * next_state are host arrays; the packed row travels in the kernel parameters (row_floats <= 960, else
 * IQL_ERR_SHAPE: stage the row and use iql_replay_insert).  One launch, no staging buffer. */
int iql_replay_insert_host(float* rows, const iql_row_layout* lay, int64_t pointer, const float* host_state,
                           const float* host_action, float reward, const float* host_next_state, float done,
                           void* stream);
/* replaces: ReplayBuffer.sample iql.py:171-178.  indices == NULL: draw them
 * in-kernel from Philox4x32-10 keyed by (seed, step); else gather the given
 * int64 indices (reference-compatible mode: numpy's MT19937 stream on host).
 * Outputs are dense [B,S],[B,A],[B,1],[B,S],[B,1]; idx_out (optional) gets the
 * indices used. */
int iql_replay_sample(const float* rows, const iql_row_layout* lay, int64_t size, int64_t batch,
                      const int64_t* indices, uint64_t seed, uint64_t step,
                      float* states, float* actions, float* rewards, float* next_states,
                      float* dones, int64_t* idx_out, void* stream);

/* ReplayBuffer.sample iql.py:171-178 for a HOST caller: `host_indices` [batch] int64 in host memory (the
 * np.random.randint draw of iql.py:172), each in [0, size).  The indices travel in the kernel parameters (256 per
 * launch): no staging buffer, no host->device copy, and the caller may reuse `host_indices` as soon as the call
 * returns.  Outputs as for iql_replay_sample. */
int iql_replay_sample_host(const float* rows, const iql_row_layout* lay, int64_t size, int64_t batch,
                           const int64_t* host_indices, float* states, float* actions, float* rewards,
                           float* next_states, float* dones, void* stream);

/* The sampler of IQL_SAMPLE_MT19937 without a handle (the np.random.randint draw of iql.py:172 for n independent
 * streams): stream i draws host_count[i] values of RandomState.randint(0, host_high[i]) from states + i *
 * IQL_MT_STATE_WORDS into out + i * stride (stride >= every count) and advances its state.  host_high / host_count are
 * host arrays, 1 <= high <= 2^32 (else IQL_ERR_INVALID, nothing drawn). */
int iql_mt19937_randint(uint32_t* states, int32_t n, const int64_t* host_high, const int64_t* host_count, int64_t* out,
                        int64_t stride, void* stream);

/* ---- the update ----------------------------------------------------------- */
/* Attach member's replay rows (several members may share one buffer). */
int iql_bind_replay(iql_engine* e, int32_t member, const float* rows, int64_t capacity, int64_t size);
int iql_set_replay_size(iql_engine* e, int32_t member, int64_t size);
/* Stage an externally sampled batch for member (drop-in `train(batch)` path):
 * dense [B,S],[B,A],[B] or [B,1],[B,S],[B] or [B,1].  IQL_ERR_STATE for a member whose B_m != B. */
int iql_load_batch(iql_engine* e, int32_t member, const float* states, const float* actions,
                   const float* rewards, const float* next_states, const float* dones,
                   void* stream);
/* replaces: K x [ReplayBuffer.sample iql.py:171 + ImplicitQLearning.train iql.py:542-563]
 * for all S members.  out_losses: [S][K][3] = value_loss, q_loss, actor_loss
 * (the log_dict of iql.py:563).  indices: [S][K][B] int64 (IQL_SAMPLE_INDICES).
 * dropout_masks: optional [S][K][n_hidden][B][H] uint8 keep-masks (test hook,
 * SURVEY.md section 7 hard-part 5); NULL = Philox masks in-kernel.
 * idx_out: optional [S][K][B] int64, the indices actually used. */
int iql_train_steps(iql_engine* e, int32_t k_steps, int32_t sample_mode, const int64_t* indices,
                    const uint8_t* dropout_masks, float* out_losses, int64_t* idx_out,
                    void* stream);
/* The numpy index streams of IQL_SAMPLE_MT19937 (replaces: the host draw np.random.randint(0, high, size=B) of
 * ReplayBuffer.sample, iql.py:172, made with each member's own RandomState as ensemble_train_loop does).  Both buffers
 * are caller-allocated device memory, borrowed for the handle's lifetime: states [S][IQL_MT_STATE_WORDS] uint32 (8-byte
 * aligned), indices [S][max_steps_per_call][batch_size] int64 (16-byte aligned; a K-step call uses its first S * K * B
 * entries as [S][K][B]).  Member m's draws in a call are exactly RandomState.randint(0, high_m, size=K * B_m) (int64):
 * step k gets draws [k B_m, (k + 1) B_m) in rows b < B_m; pad rows draw nothing.  high_m is the member's replay size
 * (iql_set_replay_size) at the call, read by the sampler at run time, so a size change needs no new graph.  A stream
 * continues across calls, graph replays and host steps; write a state to restart it.  Members that do not train draw
 * nothing and their state words keep every bit.  Refusals, with nothing drawn: IQL_ERR_STATE when no streams are bound;
 * IQL_ERR_INVALID for an active member whose size is 0 or above 2^32 (numpy's 64-bit path).  NULL, NULL unbinds. */
int iql_bind_index_streams(iql_engine* e, uint32_t* states, int64_t* indices);
/* replaces: ONE iteration of the reference's training loop as a host caller sees it --
 * `batch = replay_buffer.sample(B); log_dict = trainer.train(batch)` (offline/iql.py:631-635, finetune/iql.py:542-563),
 * whose log_dict holds the three losses as host floats every step.
 * host_indices: [S][B] int64 in HOST memory (e.g. numpy's np.random.randint stream, iql.py:172), or NULL to consume the
 * batch staged by iql_load_batch.  host_losses: [S][3] floats in HOST memory.  One CUDA-graph launch: the graph is
 * captured once on `stream` (a non-default stream) and launched on `caller_stream` (the stream the caller's own work
 * is on; may be the default stream), so the step is ordered against the caller's inserts / staged batch / later reads
 * by plain stream order.  The loss kernel writes its scalars into pinned host memory and the call returns as soon as
 * they have landed, while the step's backward / optimizer launches are still in flight. */
int iql_train_host_step(iql_engine* e, const int64_t* host_indices, float* host_losses, void* stream,
                        void* caller_stream);
/* iql_train_host_step with the indices drawn on the device from the streams of iql_bind_index_streams (one step,
 * B_m draws per active member at its replay size).  Same graph launch, pinned loss mailbox and host_losses == NULL /
 * iql_host_step_wait contract; the members' bounds travel in the pinned block where the host indices would go, so the
 * step uploads nothing from pageable memory. */
int iql_train_host_step_mt19937(iql_engine* e, float* host_losses, void* stream, void* caller_stream);
/* host_losses == NULL above returns right after the launch; this collects the losses of that step (spins on the
 * flag words, bounded; `stream` as above).  Lets the caller do its per-step host bookkeeping while the GPU works. */
int iql_host_step_wait(iql_engine* e, float* host_losses, void* stream);
/* replaces: actor(obs).mean / DeterministicPolicy.forward as used by
 * GaussianPolicy.act / DeterministicPolicy.act iql.py:371-379,403-413 in eval
 * mode: out[n,A] = clamp(max_action * tanh(MLP(states[n,S]))).  member = -1 evaluates every member's
 * policy on its own block of rows (vectorised envs): states [S][n][state_dim] -> out [S][n][action_dim]. */
int iql_act(iql_engine* e, int32_t member, const float* states, int64_t n, float max_action,
            float* out_actions, void* stream);
/* The same for ONE observation of a HOST caller -- `actor.act(state, device)` as the rollout loops call it once per
 * env step (eval_actor iql.py:218-238, jsrl_w_iql.py:445-515): host_state[state_dim] and host_action[action_dim] are
 * host arrays.  The observation travels in the kernel parameters and the action returns through pinned host memory
 * (no copies, no stream synchronisation); launched on `caller_stream`, i.e. ordered behind the host steps and
 * everything else the caller has enqueued there (`stream` is unused and kept for symmetry). */
int iql_act_host(iql_engine* e, int32_t member, const float* host_state, float max_action, float* host_action,
                 void* stream, void* caller_stream);
/* Training-mode GaussianPolicy.act (iql.py:371-379, `dist.sample()`; the learner's env steps of the online loop,
 * jsrl_w_iql.py:445-515): the parameters of the action distribution for one host observation -- host_mean[action_dim] =
 * tanh(MLP(state)) (unscaled) and host_std[action_dim] = exp(clamp(log_std, -20, 2)); the caller draws
 * mean + std * N(0, 1) on the host and clamps max_action * sample.  Same launch / mailbox as iql_act_host. */
int iql_act_host_gaussian(iql_engine* e, int32_t member, const float* host_state, float* host_mean, float* host_std,
                          void* stream, void* caller_stream);

/* ---- the online phase of an ensemble (one env step of S members at once) ---------------------------------------- */
/* Per-member action source of iql_act_host_members */
#define IQL_ACT_SKIP 0         /* the member gets nothing; its rows of host_out / host_std are left untouched          */
#define IQL_ACT_LEARNER 1      /* eval-mode action of the member's learner: clamp(max_action * tanh(MLP(s)))          */
#define IQL_ACT_LEARNER_DIST 2 /* Gaussian learner: mean = tanh(MLP(s)) (unscaled) and std = exp(clamp(log_std, -20, 2)) */
#define IQL_ACT_GUIDE 3        /* eval-mode action of the member's guide (the arena bound by iql_bind_guide)          */
#define IQL_ACT_LEARNER_DROPOUT 4      /* training-mode deterministic act: clamp(max_action * tanh(MLP_drop(s)))        */
#define IQL_ACT_LEARNER_DIST_DROPOUT 5 /* training-mode Gaussian act: mean = tanh(MLP_drop(s)) (unscaled) and std, as 2 */
/* MLP_drop is the policy MLP with nn.Dropout(p = the member's iql_hparams.actor_dropout) after every hidden ReLU, the
 * learner in training mode (GaussianPolicy.act's dist.sample(), DeterministicPolicy.act's self(state)).  Hidden unit j of
 * hidden layer l (0 <= l < n_hidden) is kept iff
 *     word (j & 3) of Philox4x32-10(counter = (j >> 2, act_step lo, act_step hi, 0x80000000 + l),
 *                                   key = (seed lo, seed hi))  >=  floor(p * 2^32)
 * (words x, y, z, w = 0..3), where seed is the member's iql_hparams.seed; a kept unit becomes relu(a) * (float)(1 / (1 - p)),
 * a dropped unit exactly 0 -- the rule of the update's dropout masks, whose counter word 3 is 1 + l, so the act masks never
 * repeat a training mask of the same key.  act_step is the member's act counter (iql_get_act_steps): every launched
 * member with code 4 or 5 draws at its counter's current value, and the counter then advances by one, whatever p is
 * (p = 0 gives codes 1 / 2 bit for bit).  No other code, no other call (iql_set_active_members included) touches it. */
/* Bind a second [S][param_floats] parameter arena with this handle's layout as the members' guides (JSRL's guide
 * policy: in practice the frozen offline ensemble's parameter arena, zero-copy).  The engine only reads it.  NULL
 * unbinds.  16-byte aligned device memory. */
int iql_bind_guide(iql_engine* e, const float* guide_params);
/* replaces: GaussianPolicy.act / DeterministicPolicy.act (iql.py:371-379, 403-413) behind jsrl_utils.learner_or_guide_action
 * (jsrl_utils.py:547-622), for every member of the ensemble in ONE launch: host_states [S][state_dim], host_source [S]
 * IQL_ACT_* codes.  host_out [S][action_dim] receives the action (or the mean of IQL_ACT_LEARNER_DIST), host_std
 * [S][action_dim] the std of IQL_ACT_LEARNER_DIST / IQL_ACT_LEARNER_DIST_DROPOUT members (may be NULL when no member asks for it).  Skipped members
 * cost no CTA.  Every active member's result is bit-identical to iql_act_host / iql_act_host_gaussian on the same
 * weights.  Observations travel through an engine-owned pinned, device-mapped block (no state_dim limit), results
 * come back through pinned memory with one flag word per member: no copies, no stream synchronisation.  Launched on
 * `caller_stream`, ordered behind the host steps like iql_act_host.  Refused (IQL_ERR_INVALID): a guide code with no
 * guide bound, a distribution code on a deterministic policy, unknown codes (nothing is launched, no counter moves). */
int iql_act_host_members(iql_engine* e, const float* host_states, const int8_t* host_source, float max_action,
                         float* host_out, float* host_std, void* stream, void* caller_stream);
/* host_out[S]: the act counters of all members (start at 0; see IQL_ACT_LEARNER_DROPOUT). */
int iql_get_act_steps(iql_engine* e, uint64_t* host_out);
/* host_in[S]: set the act counters of all members (setting a counter back to k repeats the masks drawn at k). */
int iql_set_act_steps(iql_engine* e, const uint64_t* host_in);
/* replaces: ReplayBuffer.add_transition (iql.py:180-196) for every member in ONE launch: member m's transition
 * (host_states [S][state_dim], host_actions [S][action_dim], host_rewards [S], host_next_states [S][state_dim],
 * host_dones [S], all host memory) is packed in the iql_row_layout layout, padding zeroed, and written at row
 * host_pointers[m] of the rows bound to member m by iql_bind_replay; host_pointers[m] == -1: no insert for m.
 * The packed rows travel through an engine-owned pinned, device-mapped block (any row width): two slots used in
 * turn, each reused only once the kernel has marked it consumed, so the call returns without waiting for the launch
 * and the caller may reuse its arrays at once.  Launched on `caller_stream`.  Refused (IQL_ERR_INVALID): a pointer
 * outside [0, capacity), an inserting member with no binding, two inserting members bound to the same rows. */
int iql_replay_insert_members_host(iql_engine* e, const float* host_states, const float* host_actions,
                                   const float* host_rewards, const float* host_next_states, const float* host_dones,
                                   const int64_t* host_pointers, void* stream, void* caller_stream);
/* Self-test hook for the tcgen05 TF32 GEMM building block (no reference
 * counterpart): C[M,N] = op(A) op(B), mode 0 NT (A[M,K], B[N,K]), 1 NN (A[M,K],
 * B[K,N]), 2 TN (A[K,M], B[K,N]); M multiple of 256, N <= 256 or a multiple of
 * 256, any K (TMA zero-fills tails), lda/ldb multiples of 4;
 * scratch: >= 1024 B of 128-byte aligned device memory. */
int iql_selftest_umma_gemm(int32_t mode, int32_t M, int32_t N, int32_t K, const float* A, int32_t lda,
                           const float* B, int32_t ldb, float* C, int32_t ldc, void* scratch,
                           size_t scratch_bytes, void* stream);
/* Measurement hook (bench.py roofline): run `reps` update steps with CUDA events recorded on `stream`
 * around every kernel launch of the step.  For launch slot i < *n_slots: avg_ms[i], the algorithmic
 * FLOPs and bytes of that launch (2MNK; every operand read once, every output written once) and a
 * 32-byte label at labels + 32*i.  Advances the learners by `reps` steps. */
int iql_profile_step(iql_engine* e, int32_t reps, int32_t max_slots, int32_t* n_slots, float* avg_ms,
                     double* flops, double* bytes, char* labels, void* stream);
/* number of kernel launches issued by the last iql_train_steps call */
int64_t iql_last_launch_count(const iql_engine* e);
/* Measurement hook (tools/fused_trace.py): with IQL_FUSED_TRACE set in the environment, CTA 0 of the fused
 * forward kernel records clock64 stamps of its TMA / MMA / epilogue roles for its first 8 tiles; this copies the
 * stamps of the last launch, [3 roles][8 tiles][4 layers][4 stamps] int64, to the host.  Returns the number of
 * words written, < 0 when tracing is off or `max_words` is too small. */
int iql_debug_fused_trace(long long* out, int32_t max_words);
/* IQL_STEP_TRACE=1 (with IQL_B200_DEBUG=1): per-launch start / end globaltimer stamps of the step's kernels
 * (tools/step_trace.py); reset != 0 arms the slots, otherwise copies [13][2] stamps (ns) to `out`. */
int iql_debug_step_trace(iql_engine* e, int32_t reset, unsigned long long* out, int32_t max_words, void* stream);
/* IQL_CHAIN_TRACE=1: globaltimer stamps of CTA pair 0 of the last bwd_chain launch (tools/chain_trace.py) */
int iql_debug_chain_trace(long long* out, int32_t max_words);

#ifdef __cplusplus
}
#endif
#endif /* IQL_B200_H */

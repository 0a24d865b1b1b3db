// Internal declarations shared by the engine translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/iql_b200.h"

namespace iql {

int make_row_layout(int S, int A, iql_row_layout* out);

// ---- grouped GEMM problem descriptor (one entry per member x network) -----
enum Epilogue : int {
  EPI_NONE = 0,    // C = acc                       (weight gradients)
  EPI_LINEAR = 1,  // C = acc + bias[j]             (output layer)
  EPI_RELU = 2,    // C = drop(relu(acc + bias[j])) (hidden layer, optional dropout)
  EPI_DRELU = 3,   // C = acc * [mask > 0] * scale  (activation gradient)
};

struct GemmProb {
  const float* A;
  const float* B;
  float* C;
  const float* bias;   // EPI_LINEAR / EPI_RELU
  float* dbias;        // TN mode: column sums of A (bias gradient), may be null
  const float* mask;   // EPI_DRELU: forward activation
  int M, N, K;
  int lda, ldb, ldc, ldmask;
  int epi;
  int member;
  int drop_layer;      // >= 0: hidden-layer index whose dropout applies (actor only)
  int no_store;        // 1: C is consumed only by a fused follow-up (forward-only passes), skip the store
  int row0;            // row-split output-layer backward: first batch row of this split (A, C, mask already point at it)
  // ReLU sign bits of a hidden activation, [rows][N / 32] words, bit j of word (r, c) = H[r][32 c + j] > 0:
  // written by the fused forward for the layers a tcgen05 dgrad phase masks with, read by that dgrad phase
  uint32_t* bits;
};

// Per-member scalars derived on the host the way torch derives them
// (Python float64 -> fp32 scalar operands).
struct MemberScalars {
  float beta, iql_tau, discount;
  float tau, one_minus_tau;
  float adam_w1;           // (float)(1 - beta1)
  float adam_beta2;        // (float)beta2
  float adam_one_minus_b2; // (float)(1 - beta2)
  float adam_eps;
  float drop_scale;        // (float)(1/(1-p))
  uint32_t drop_threshold; // floor(p * 2^32); 0 = no dropout
  // B_m (iql_set_batch_sizes), 1 <= B_m <= B: the member trains on rows [0, B_m) of the engine batch.  Every kernel runs
  // on all B rows; the gather writes zero rows past B_m, and the loss (loss_kernel, loss_row_grads) skips them and
  // divides by B_m, so their output-layer gradients -- and hence every gradient they feed -- are exact zeros.
  int32_t batch;
  double adam_beta1_d, adam_beta2_d;
  double vf_lr, qf_lr, actor_lr, lr_eta_min;
  int64_t cosine_t_max;
  uint64_t seed;
};

struct ReplayBinding {
  const float* rows;
  int64_t capacity;
  int64_t size;
};

// Per (member, optimizer) Adam scalars of the current step: computed once (fp64) by the loss kernel, read by every
// thread of the optimizer kernel.  Order: q, v, actor.
struct AdamScalars {
  float neg_step_size;  // -(lr / (1 - beta1^t))
  float bc2_sqrt;       // sqrt(1 - beta2^t)
};

// Context passed by value to every kernel of a step.
struct StepCtx {
  int k;                         // step offset inside this call (0..K-1)
  int K;                         // steps in this call
  int B;
  int S_dim, A_dim, H, L;
  int deterministic;
  // members this step trains (iql_set_active_members), ascending; the per-member kernels (gather, loss, optimizer,
  // operand refresh, counter advance) run one CTA row per entry and take their member from active[blockIdx]
  int n_active;
  const int32_t* active;         // [n_active] device; null when every member trains (member i = CTA row i)
  int64_t P;                     // member block floats
  int64_t PQ;                    // q range [0, PQ)
  int64_t v_begin, v_end, a_begin, a_end;
  int64_t log_std_off;           // inside member block (Gaussian only)
  iql_row_layout row;
  const MemberScalars* scalars;  // [S]
  iql_counters* counters;        // [S] device
  const ReplayBinding* replay;   // [S] device
  const int64_t* indices;        // [S][K][B] or null
  const uint8_t* dropout_masks;  // [S][K][L][B][H] or null
  int64_t* idx_out;              // [S][K][B] or null
  float* loss_ring;              // [S][Kmax][3]
  // host-step path (iql_train_host_step): pinned, device-mapped host memory [S][4] -- the loss kernel stores the three
  // losses of member m at [m][0..2], fences at system scope and then sets the word [m][3] to 1; null otherwise
  float* host_mail;
  // > 0 on the call's LAST optimizer launch (adam_polyak_kernel): it also advances the members' counters by this many
  // steps, which saves the separate advance_kernel launch -- every reader of the counters (gather, forward dropout,
  // loss kernel) precedes that launch, and nothing after it in the call reads them.  enqueue_step sets it to -1 once
  // consumed so that the caller knows not to launch advance_kernel.
  int advance_k;
  // IQL_STEP_TRACE (debug): globaltimer stamps of every launch of a step, [slot][2] = earliest CTA start / latest CTA end
  unsigned long long* stamps;
  AdamScalars* adam_sc;          // [S][3] device
  int k_max;
  int tf32;                      // 1: tcgen05 path; producers round GEMM operands to nearest TF32
  float* w_shadow;               // [S][P]  TF32-rounded copy of params (tcgen05 B operands), tf32 mode only
  float* t_shadow;               // [S][PQ] TF32-rounded copy of the target network
  // 3xTF32 input layer: x = hi + lo with both parts TF32-exact, so X W0^T = Xhi Whi + Xlo Whi + Xhi Wlo
  // runs on the tensor cores at FP32 accuracy.  lo parts of the first-layer weights / of the gathered rows:
  float* w_shadow_lo;            // [S][P]  (only the first-layer weight ranges are maintained)
  float* t_shadow_lo;            // [S][PQ]
  // ranges inside a member block whose TF32 lo parts are maintained next to the hi shadow: the first-layer weights of
  // q1, q2, v, actor (3xTF32 input layer) and [4] the policy-head weights when the head runs as a two-pass tcgen05 GEMM
  int64_t first_w_begin[5], first_w_end[5];
  // Hidden-layer weights (W_l, 1 <= l < L, and their target copies) need no TF32 shadow: during an engine call they are
  // kept in the parameter / target arenas themselves with half a TF32 ulp added to the magnitude (bit pattern + 0x1000),
  // so that the tensor cores' truncation of the fp32 operand IS round-to-nearest of the true weight.  The call's first
  // kernel adds the bias in place, the optimizer removes it from what it reads and re-adds it to what it writes, and the
  // optimizer launch of the call's LAST step writes the true values (unbias_out): outside a call the arenas always hold
  // plain fp32.  Saves the 1.5 MB per member-step of shadow writes.
  int bias_hidden;               // 1: scheme active (tcgen05 path)
  int unbias_out;                // 1: this optimizer launch is the last of the call
  int n_hid;
  int64_t hid_begin[4 * 3], hid_end[4 * 3];  // hidden weight ranges inside a member block (4 nets x (L - 1) layers)
  int64_t xrow_off_;             // per-member workspace offset of the gathered rows
  int64_t xhi_off, xlo_off;      // per-member workspace offsets of the hi / lo copies of the gathered rows (0 = off)
};

struct TensorDesc {
  iql_tensor_info info;
};

// Offsets (floats) into one member's workspace block.
struct WorkspaceLayout {
  int64_t xrow;      // [B][ROW]
  int64_t act;       // [7][L][B][H]  hidden activations H_1..H_L of the 7 forward passes
  int64_t yq;        // [6][B]        scalar heads: V(s'), V(s), tq1, tq2, q1, q2
  int64_t zpi;       // [B][Ald]      actor pre-tanh output
  int64_t gy;        // [3][B]        dL/dy of V, q1, q2
  int64_t gpi;       // [B][Ald]      dL/dz of actor
  int64_t gh;        // [4][2][B][H]  ping-pong activation gradients of the 4 trainable nets
  int64_t xhi, xlo;  // [B][ROW] each: TF32 hi / lo split of the gathered rows (tcgen05 mode)
  int64_t bits;      // [4][L-1][B][H/32] uint32: ReLU sign bits of H_1..H_{L-1} of the 4 training passes (tcgen05 mode)
  int64_t lb_scratch, lb_stride;  // [4][splits][lb_stride]: row-split partials of the output-layer backward (0: unused)
  int64_t fw_scratch, fw_stride;  // [4][splits][fw_stride]: K-split partials of the input-layer weight gradient (0: unused)
  int64_t member_floats;
  int Ald;
};

// launch slots of the step timeline (tools/step_trace.py)
enum StampSlot : int { ST_REFRESH = 0, ST_GATHER, ST_FWD, ST_POLHEAD, ST_LOSS, ST_LASTBWD, ST_LBREDUCE, ST_WGRAD, ST_DGRAD, ST_FWGRAD, ST_ADAM,
                       ST_ADVANCE, ST_CHAIN, ST_COUNT };

// forward pass ids
enum Pass : int { PASS_V_NEXT = 0, PASS_V = 1, PASS_TQ1 = 2, PASS_TQ2 = 3, PASS_Q1 = 4, PASS_Q2 = 5, PASS_PI = 6, N_PASS = 7 };

// launchers implemented in kernels_simt.cu
void launch_simt_gemm(int mode /*0 NT,1 NN,2 TN*/, const GemmProb* probs, int nprob, int maxM, int maxN,
                      const StepCtx& ctx, cudaStream_t st);
void launch_gather(const StepCtx& ctx, float* ws, int64_t ws_member_floats, int64_t xrow_off, cudaStream_t st);
void launch_loss(const StepCtx& ctx, float* ws, int64_t ws_member_floats, const WorkspaceLayout& wl,
                 const float* params, float* grads, cudaStream_t st);
void launch_adam(const StepCtx& ctx, float* params, float* exp_avg, float* exp_avg_sq, float* target,
                 const float* grads, cudaStream_t st);
void launch_advance(const StepCtx& ctx, int K, cudaStream_t st);
void launch_refresh_shadow(const StepCtx& ctx, float* params, float* target, cudaStream_t st);
void launch_gather_refresh(const StepCtx& ctx, float* ws, int64_t ws_member_floats, int64_t xrow_off, float* params, float* target,
                           cudaStream_t st);
void launch_load_batch(const StepCtx& ctx, int member, float* xrow, const float* s, const float* a, const float* r,
                       const float* s2, const float* d, cudaStream_t st);
// skinny-layer kernels (kernels_skinny.cu)
void launch_first_fwd(const GemmProb* probs, int nprob, int B, int H, int kmax, const StepCtx& ctx, cudaStream_t st);
void launch_out_fwd(const GemmProb* probs, int nprob, int B, int H, int amax, cudaStream_t st);
// ws / wl / params != null and last_bwd_recomputes_loss_grads(H, amax): the kernel derives the loss gradients of its
// rows itself (the problem tables hold 4 training nets per member: V, q1, q2, actor) and does not read gy / gpi, so
// loss_kernel need not precede it.
bool last_bwd_recomputes_loss_grads(int H, int amax, int nprob, int B);
// row-split output-layer backward: dW_L, db_L (and db_{L-1}) of problem i = sum over s of the partials the split
// problems [s * nprob + i] wrote, added in split order
// (rows = M of the wgrad problem, N valid columns per row, both tables with the leading dimension of dW; also used
// for the K-split input-layer weight gradient)
void launch_lb_reduce(const GemmProb* pw_split, const GemmProb* prev_split, const GemmProb* pw, const GemmProb* prev, int nprob,
                      int splits, cudaStream_t st);
int launch_last_bwd(const GemmProb* probs_dgrad, const GemmProb* probs_wgrad, const GemmProb* probs_prev_wgrad,
                     int nprob, int B, int H, int amax, const StepCtx& ctx, cudaStream_t st, const float* ws = nullptr,
                     int64_t ws_member_floats = 0, const WorkspaceLayout* wl = nullptr, const float* params = nullptr);
void launch_first_wgrad(const GemmProb* probs, int nprob, int B, int H, int kmax, cudaStream_t st);
void launch_act(const StepCtx& ctx, const float* actor_block, int n_members, const int64_t* w_off,
                const int64_t* b_off, const float* states, int64_t n, float max_action, float* out, cudaStream_t st);

// one observation passed by value (state_dim <= act_host_state_max()), action + flag word into pinned host memory
int act_host_state_max();
void launch_act_host(const StepCtx& ctx, const float* actor_block, const int64_t* w_off, const int64_t* b_off,
                     const float* host_state, float max_action, const float* log_std /* null: deterministic policy */, float* mail,
                     cudaStream_t st);
// iql_act_host_members: one CTA per active member, the observations and the member list in a device-mapped pinned block
// (`ids` [n] member indices, `codes` [n] IQL_ACT_* of those members, `steps` [n] their act counters, read by codes 4 / 5;
// `drop_codes`: some code is 4 or 5); results [S][2A] + flag words [S] in pinned memory
void launch_act_members(const StepCtx& ctx, const float* params, const float* guide, const int64_t* w_off, const int64_t* b_off,
                        const float* states, const int32_t* ids, const int32_t* codes, const uint64_t* steps, bool drop_codes,
                        int n, float max_action, float* mail, uint32_t* flags, cudaStream_t st);
// iql_replay_insert_members_host: one CTA per inserting member copies its packed row (device-mapped pinned block) to the
// ring bound in `replay` and raises its consumed word
void launch_insert_members(const ReplayBinding* replay, int RF, const float* rows, const int32_t* ids, const int64_t* pointers,
                           int n, uint32_t* consumed, cudaStream_t st);

}  // namespace iql

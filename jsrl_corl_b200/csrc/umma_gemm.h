// tcgen05 (UMMA) TF32 grouped GEMM used by IQL_MATH_TF32_TCGEN05.
#pragma once
#include "engine.h"

namespace iql {
// true when the phase (mode 0 NT / 1 NN / 2 TN) can run on the tcgen05 kernel
// for this batch size and hidden width (256x256x32 tiles must divide the problem).
bool umma_phase_supported(int mode, int batch, int hidden);
// Encode the two TMA tensor maps (A, B) of every problem into h_maps_out
// (2 * nprob CUtensorMap, 128 B each).  Returns 0 on success.
// tile_n = umma_tile_n(max N of the phase): the UMMA N / B-tile height used by the launch.
int umma_tile_n(int maxN);
// CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles, each CTA staging half of the B tile): umma_cta2_ok says
// whether the shape allows them, umma_cta2 whether the phase should use them; the tensor maps and the launch
// must be given the same answer (the engine stores it per phase when the state is bound).
bool umma_cta2_ok(int maxM, int maxN);
bool umma_cta2(int mode, int nprob, int maxM, int maxN, int maxK);
int umma_encode_maps(int mode, const GemmProb* h_probs, int nprob, int tile_n, void* h_maps_out, bool cta2);
// probs_out != null (forward, last hidden layer, EPI_RELU): the output-layer problem table; the scalar heads
// of its first `fuse_count` problems are evaluated in FP32 inside the epilogue.
bool umma_can_fuse_out(int act_dim);
// true when the dgrad epilogue also produces the bias gradient of the layer below (else run launch_colsum)
bool umma_dgrad_writes_dbias(int batch);
// cmaps != null (EPI_NONE / EPI_DRELU): umma_encode_store_map maps of the outputs, 1 per problem: row-layout
// epilogue with TMA stores; EPI_DRELU then masks with GemmProb::bits instead of the FP32 activation.
// split3 = 1: 3xTF32 input layer; `maps` then holds 4 maps per problem (umma_encode_maps_split): Xhi, Whi, Xlo, Wlo.
// split3 = 2: two passes A Whi + A Wlo for an A operand that is TF32-exact already (maps: A, Whi, A, Wlo): FP32-accurate
// output heads on the tensor cores.
void launch_umma_gemm(int mode, const GemmProb* probs, const void* maps, const GemmProb* probs_out, int epi, int nprob,
                      int maxM, int maxN, const StepCtx& ctx, cudaStream_t st, int split3 = 0, int fuse_count = 0,
                      bool cta2 = false, int maxK = 0, const void* cmaps = nullptr, int tile_n = 0 /* 0: umma_tile_n(maxN) */);
int umma_encode_maps_split(const GemmProb* h_hi, const GemmProb* h_lo, int nprob, int tile_n, void* h_maps_out, bool cta2);
// Fused forward (fused_fwd.cu): all hidden layers + scalar heads of every (member, pass) in one launch, hidden
// activations chained through tensor memory.  Hidden width 256, 1..FUSED_MAX_LAYERS hidden layers.
constexpr int FUSED_MAX_LAYERS = 4;
struct FusedFwdArgs {
  const GemmProb* probs[FUSED_MAX_LAYERS];  // device problem tables of forward phases 0..L-1 (same problem order in each)
  const void* maps[FUSED_MAX_LAYERS];       // [0]: umma_encode_maps_split maps (4 per problem); l >= 1: umma_encode_maps maps (2 per problem)
  const void* store_maps[FUSED_MAX_LAYERS]; // umma_encode_store_map maps of the layer outputs, 1 per problem
  const GemmProb* probs_out;                // output-layer problem table; heads of the first fuse_count problems are fused
  int L, nprob, batch, fuse_count, k0_max;
  int pair;  // run on CTA pairs (the weight maps were encoded with half-height boxes)
  int fuse_policy;  // also fuse the policy head (problems >= fuse_count of probs_out; act_dim <= 8)
};
// 2-D map of a row-major [rows][cols] fp32 output (ld floats), box 32 x 32, 128-byte swizzle (TMA store)
int umma_encode_store_map(void* h_map_out, const float* ptr, int rows, int cols, int ld);
bool fused_fwd_supported(int batch, int hidden, int n_hidden, int k0);
bool fused_fwd_pair(int batch);
bool fused_fwd_policy_head(int act_dim);  // the actor's output layer fits the fused epilogue  // whether the fused forward runs on CTA pairs for this batch size
void launch_fused_fwd(const FusedFwdArgs& a, const StepCtx& ctx, cudaStream_t st);
// Chained backward + optimizer (bwd_chain.cu): one CTA pair per (member, trainable net) runs the hidden-layer dgrad /
// wgrad phases back to back and applies Adam + Polyak in the wgrad epilogues.  Hidden width 256, batch 256,
// 2..FUSED_MAX_LAYERS hidden layers, fused forward on (it writes the ReLU sign bits the dgrad phases mask with).
// grads_only: the wgrad epilogues store the weight gradients to the grads arena instead and the optimizer runs as
// adam_polyak_kernel after the launch.
struct BwdChainArgs {
  const GemmProb* probs;  // the engine's device problem table (base)
  const void* maps;       // chain tensor maps, CTA-pair boxes: per phase 2 per task (A, B)
  const void* cmaps;      // store maps of the backward outputs, indexed by absolute problem index
  int n_phases, n_tasks, keep_grads, grads_only;
  int db_tile_order;  // grads_only: bias-gradient summation order of the single-CTA dgrad (the per-phase dgrad is not on CTA pairs)
  int kind[2 * FUSED_MAX_LAYERS];         // 0 dgrad, 1 wgrad (+ optimizer unless grads_only)
  int prob_first[2 * FUSED_MAX_LAYERS];   // first problem of the phase (task i uses prob_first + i)
  int map_first[2 * FUSED_MAX_LAYERS];    // first map of the phase inside `maps` (in maps)
  int tile_n[2 * FUSED_MAX_LAYERS], k[2 * FUSED_MAX_LAYERS], wait_dgrads[2 * FUSED_MAX_LAYERS];
  int n_seg[4];
  long long seg_lo[4][FUSED_MAX_LAYERS + 2], seg_hi[4][FUSED_MAX_LAYERS + 2];
  float *params, *exp_avg, *exp_avg_sq, *target, *grads;
};
// k0 = state_dim + action_dim: the input-layer wgrad phase runs one N tile per task, at most 256 wide
bool bwd_chain_supported(int batch, int hidden, int n_hidden, int k0, bool fused_fwd);
int bwd_chain_wgrad0_tile_n(int k0);
void launch_bwd_chain(const BwdChainArgs& a, const StepCtx& ctx, cudaStream_t st);
// bias gradients of a wgrad phase: dbias[m] = sum_k A[k][m]
void launch_colsum(const GemmProb* probs, int nprob, int maxM, cudaStream_t st);
}  // namespace iql

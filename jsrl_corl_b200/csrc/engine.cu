// C-ABI + host orchestration of the IQL update engine (see include/iql_b200.h).
//
// The handle owns only host metadata; every device byte it touches was
// allocated by the caller (torch) and bound through iql_bind_state /
// iql_bind_replay.  The first part of the caller's workspace holds the small
// device tables (per-member scalars, counters, replay bindings, grouped-GEMM
// problem descriptors, loss ring); the rest is the per-member activation area.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <tuple>
#include <string>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "engine.h"
#include "umma_gemm.h"

using namespace iql;

static thread_local std::string g_create_error;
// "auto" runs the chained backward (gradients only, IQL_OPT_STEP_PATH = 4) from this many members on with two hidden
// layers, and from one member on with three or more (each extra layer is two more per-phase launches): measured
// crossover against the per-phase backward on the B200 (profiles/r03_summary.md)
static constexpr int CHAIN_GRADS_MIN_MEMBERS = 8;

// Optional per-launch instrumentation of one update step (iql_profile_step).
struct StepTimer {
  std::vector<cudaEvent_t> ev;       // ev[i] recorded BEFORE launch i; one extra at the end
  std::vector<std::string> label;
  std::vector<double> flops, bytes;  // algorithmic work of the launch
  cudaStream_t st = nullptr;
  void mark(const char* name, double fl, double by) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    ev.push_back(e);
    label.push_back(name);
    flops.push_back(fl);
    bytes.push_back(by);
  }
  void finish() {
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    ev.push_back(e);
  }
};

struct Phase {
  int mode;      // 0 NT, 1 NN, 2 TN
  int first;     // index into problem table
  int count;
  int maxM, maxN;
  int maxK = 0;  // largest K over the problems of the phase
  bool cta2 = false;  // tcgen05 kernel runs this phase on CTA pairs (decided when the tensor maps are encoded)
  bool rowepi = false;  // tcgen05 kernel uses the row-layout epilogue: TMA stores, ReLU sign bits as the dgrad mask
  int K;         // common K of the phase (0 if mixed)
  bool umma_ok;  // eligible for the tcgen05 kernel
  int epi;       // common epilogue of the phase
  int kind;      // PH_*: dedicated skinny-layer kernel, or generic grouped GEMM
  int tile_n = 0;  // N tile of the tcgen05 kernel (0: umma_tile_n(maxN)); 128 for CTA-pair dgrad launches with few problems
};
enum { PH_GENERIC = 0, PH_FIRST_FWD = 1, PH_OUT_FWD = 2, PH_LAST_WGRAD = 3, PH_LAST_DGRAD = 4, PH_FIRST_WGRAD = 5 };

// The skinny-layer kernels keep one operand in shared memory; a layer whose operand does not fit takes the generic GEMM.
static bool skinny_enabled() {
  static const bool on = dbg_getenv("IQL_B200_NO_SKINNY") == nullptr;
  return on;
}

// input-layer forward (first_fwd_kernel): K = state_dim + action_dim up to 72
static bool first_fwd_skinny_ok(int k0) { return skinny_enabled() && k0 <= 72; }

// input-layer weight gradient (first_wgrad_kernel): the batch's rows of X at the padded K
static bool first_wgrad_skinny_ok(int batch, int k0) {
  const int kpad = k0 <= 24 ? 24 : (k0 <= 40 ? 40 : 72);
  return first_fwd_skinny_ok(k0) && ((size_t)batch * kpad + 512 * (kpad + 1)) * 4 <= 200 * 1024;
}

// output-layer forward (out_fwd_kernel): the padded head weights [apad][H]
static bool out_fwd_skinny_ok(int hidden, int action_dim) {
  const int apad = action_dim <= 1 ? 1 : (action_dim <= 8 ? 8 : (action_dim <= 24 ? 24 : 64));
  return skinny_enabled() && action_dim <= 64 && (size_t)apad * hidden * 4 <= 200 * 1024;
}

// The output-layer backward runs on the skinny kernels (last_bwd_v4 / last_bwd_kernel<24>, the output-layer operand in
// shared memory) up to 24 actions; wider heads take two generic GEMMs.  The chained backward starts from the skinny
// kernels' outputs, so bind time and every step must agree on this rule.
static bool last_bwd_skinny_ok(int batch, int action_dim) {
  const int apad = action_dim <= 1 ? 1 : (action_dim <= 8 ? 8 : 24);
  return skinny_enabled() && action_dim <= 24 && ((size_t)batch * apad + 256 * apad) * 4 <= 200 * 1024;
}

// The shape runs on the tcgen05 kernels.  TF32 math alone is not enough: outside the batch / hidden widths the tensor-core
// kernels take, a TF32 engine runs the FP32 CUDA-core kernels.
static bool tensor_core_path(const iql_config& c) {
  return c.math_mode == IQL_MATH_TF32_TCGEN05 && umma_phase_supported(0, c.batch_size, c.hidden_dim);
}

using GraphKey = std::tuple<int, int, uintptr_t>;  // (sample mode or host-step variant, K, index pointer)

struct iql_engine {
  iql_config cfg;
  iql_layout layout;
  WorkspaceLayout wl;
  std::vector<iql_tensor_info> tensors;
  int64_t w_off[4][16], b_off[4][16];
  int w_ld[4][16];
  int64_t log_std_off = 0;
  // output-layer backward split by batch rows (few problems, large batch): lb_splits > 1, split problem tables at
  // h_probs[lb_first ...] ordered [dgrad | wgrad | prev wgrad][split][member][net]
  int lb_splits = 1;
  int64_t lb_first = 0;
  // input-layer weight gradient (tcgen05 path) split along the batch (K) dimension: fw_splits > 1, split problems in
  // fw_phase ([split][member][net]); partial dW_0 / db_0 in the scratch region, reduced by lb_reduce_kernel
  int fw_splits = 1;
  Phase fw_phase;
  // bound device memory
  float *params = nullptr, *exp_avg = nullptr, *exp_avg_sq = nullptr, *target = nullptr, *grads = nullptr;
  char* ws = nullptr;
  size_t ws_bytes = 0;
  // device tables inside the workspace
  MemberScalars* d_scalars = nullptr;
  iql_counters* d_counters = nullptr;
  ReplayBinding* d_replay = nullptr;
  GemmProb* d_probs = nullptr;
  char* d_maps = nullptr;        // [2 * nprob] CUtensorMap (128 B each), tcgen05 phases only
  std::vector<char> h_maps;
  int64_t* d_act_off = nullptr;  // [2][L+1]
  float* d_loss_ring = nullptr;
  AdamScalars* d_adam_sc = nullptr;  // [S][3], written by the loss kernel, read by the optimizer kernel
  int32_t* d_active = nullptr;   // [S] device copy of `active` (the first active.size() entries)
  float* d_wshadow = nullptr;    // [S][P]  TF32-rounded params  (tcgen05 mode)
  float* d_tshadow = nullptr;    // [S][PQ] TF32-rounded target
  float* d_wshadow_lo = nullptr; // lo parts (first-layer ranges) for the 3xTF32 input layer
  float* d_tshadow_lo = nullptr;
  char* d_maps_first = nullptr;  // [4 * S * N_PASS] CUtensorMap: Xhi, Whi, Xlo, Wlo of the input-layer forward
  std::vector<char> h_maps_first;
  char* d_maps_c = nullptr;      // [nprob] CUtensorMap of the outputs of the backward tcgen05 phases (TMA stores)
  std::vector<char> h_maps_c;
  char* d_maps_store = nullptr;  // [L][S * N_PASS] CUtensorMap: activation outputs of the fused forward (TMA stores)
  std::vector<char> h_maps_store;
  // chained backward + optimizer (bwd_chain.cu): phase list, CTA-pair tensor maps, small-parameter ranges
  bool chain = false;
  bool chain_grads = false;      // the chain stores the weight gradients; adam_polyak_kernel runs after it
  int step_path = 0;             // iql_set_option(IQL_OPT_STEP_PATH): 0 auto, 1 per-phase kernels, 2 chained backward +
                                 // optimizer, 4 chained backward (gradients) + adam_polyak_kernel (2 and 4 required)
  int keep_grads = 0;            // iql_set_option(IQL_OPT_KEEP_GRADS): the chained backward also stores the weight gradients
  BwdChainArgs chain_args;
  char* d_maps_chain = nullptr;
  std::vector<char> h_maps_chain;
  // policy heads wider than the fused forward's epilogue handles (8 < act_dim <= 32): z = H_L Wp^T + b as a two-pass
  // tcgen05 GEMM (H_L is stored TF32-exact, Wp = hi + lo) instead of the FP32 SIMT kernel
  bool pol_umma = false;
  char* d_maps_pol = nullptr;
  std::vector<char> h_maps_pol;
  bool bias_hidden = false;      // hidden-layer weights carry the TF32 rounding bias in place during a call (engine.h), no shadow
  bool split_first = false;      // input layer runs as 3xTF32 tcgen05 GEMM
  bool fused_fwd = false;        // whole forward (hidden layers + scalar heads) runs as one fused tcgen05 launch
  bool fused_pair = false;       // ... on CTA pairs (cta_group::2), one pair per 256 batch rows
  float* d_ws_f = nullptr;       // activation area
  int64_t tables_bytes = 0;
  // host shadows
  std::vector<MemberScalars> h_scalars;
  std::vector<iql_hparams> h_hparams;
  std::vector<iql_counters> h_counters;
  std::vector<ReplayBinding> h_replay;
  std::vector<GemmProb> h_probs;
  std::vector<Phase> fwd_phases, bwd_phases;
  bool bound = false, tables_dirty = true, scalars_dirty = true, counters_dirty = true, replay_dirty = true;
  std::vector<char> preloaded;
  // members that train (iql_set_active_members), ascending.  The problem tables, tensor maps and chain tasks hold these
  // members only, and every bind-time choice that depends on the member count is made from active.size().
  std::vector<int32_t> active;
  std::vector<char> is_active;   // [S]
  int64_t last_launches = 0;
  std::string err;
  // CUDA graphs of iql_train_steps and iql_train_host_step with their launch counts (launch_graph)
  std::map<GraphKey, std::pair<cudaGraphExec_t, int64_t>> graphs;
  // the hidden-layer weight-gradient launches are leaves of the backward: they run on a side stream next to the
  // dgrad chain so that the partially filled last wave of one persistent kernel is covered by the other
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_side = nullptr, ev_fork_g = nullptr, ev_gather = nullptr;
  bool use_graphs = true;
  // host-step path (iql_train_host_step): pinned, device-mapped host block = [S][B] int64 indices | [S][4] floats
  // (losses + flag word, written by the loss kernel); an event ordering a caller's stream behind the last host step
  unsigned long long* d_stamps = nullptr;  // IQL_STEP_TRACE: [ST_COUNT][2] globaltimer stamps (debug)
  float* h_act = nullptr;        // iql_act_host: pinned, device-mapped [action_dim floats | flag word]
  char* h_mail = nullptr;
  bool mail_pending = false;     // a host step has been launched and its losses not collected yet
  cudaStream_t host_step_stream = nullptr;  // the caller's stream the last host step was launched on
  bool host_step_stream_set = false;
  cudaEvent_t ev_in = nullptr;
  // online phase of an ensemble (iql_act_host_members / iql_replay_insert_members_host)
  const float* guide = nullptr;  // [S][P] guide parameter arena (iql_bind_guide), read only
  char* h_actm = nullptr;        // pinned, device-mapped: states [S][state_dim] | ids [S] | codes [S] | steps [S] | results [S][2A] | flags [S]
  std::vector<uint64_t> act_steps;  // [S] act counters of the dropout codes (IQL_ACT_LEARNER_DROPOUT)
  char* h_ins = nullptr;         // pinned, device-mapped: 2 slots of rows [S][RF] | ids [S] | pointers [S] | consumed [S]
  int ins_slot = 0;              // slot the next insert call fills
  int ins_n[2] = {0, 0};         // rows launched from each slot (their consumed words are awaited before the slot is refilled)
  cudaStream_t ins_stream[2] = {nullptr, nullptr};
};

static int fail(iql_engine* e, int code, const std::string& msg) {
  if (e) e->err = msg;
  else g_create_error = msg;
  return code;
}

#define CUDA_TRY(e, call)                                                                  \
  do {                                                                                     \
    cudaError_t _err = (call);                                                             \
    if (_err != cudaSuccess)                                                               \
      return fail(e, IQL_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_err)); \
  } while (0)

extern "C" const char* iql_version(void) { return "iql_b200 0.1 (sm_100a)"; }

extern "C" const char* iql_last_error(const iql_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

static int net_in_dim(const iql_config& c, int net) {
  return (net == IQL_NET_Q1 || net == IQL_NET_Q2) ? c.state_dim + c.action_dim : c.state_dim;
}
static int net_out_dim(const iql_config& c, int net) { return net == IQL_NET_ACTOR ? c.action_dim : 1; }

// Problems in the tables of `members` training members: forward and backward phases, then the row-split copies of the
// output-layer backward and the K-split copies of the input-layer weight gradient (build_problems)
static int64_t problem_count(const iql_engine* e, int members) {
  const int L = e->cfg.n_hidden;
  return (int64_t)members * ((L + 1) * N_PASS + 4 * (L + 1) + 4 * L) +
         (e->lb_splits > 1 ? (int64_t)12 * members * e->lb_splits : 0) + (e->fw_splits > 1 ? (int64_t)4 * members * e->fw_splits : 0);
}

// The device tables at the head of the workspace, in this order, each 256-byte aligned; sized for every member.  Returns
// their size in bytes.  With the workspace `base` it also points the d_* tables into it; with base == nullptr it only
// sizes them (iql_create), so the size and the pointers always come from the same list.
static int64_t place_tables(iql_engine* e, char* base) {
  const int S = e->cfg.n_members, L = e->cfg.n_hidden;
  const int64_t nprob = problem_count(e, S);
  int64_t tb = 0;
  auto tab = [&](auto*& ptr, int64_t bytes) {
    if (base) ptr = reinterpret_cast<std::remove_reference_t<decltype(ptr)>>(base + tb);
    tb = round_up(tb + bytes, 256);
  };
  tab(e->d_scalars, sizeof(MemberScalars) * S);
  tab(e->d_counters, sizeof(iql_counters) * S);
  tab(e->d_replay, sizeof(ReplayBinding) * S);
  tab(e->d_probs, sizeof(GemmProb) * nprob);
  tab(e->d_maps, 128 * 2 * nprob);
  tab(e->d_act_off, sizeof(int64_t) * 2 * (L + 1));
  tab(e->d_loss_ring, sizeof(float) * 3 * (int64_t)S * e->cfg.max_steps_per_call);
  tab(e->d_adam_sc, sizeof(AdamScalars) * 3 * S);
  tab(e->d_active, sizeof(int32_t) * S);
  if (e->cfg.math_mode == IQL_MATH_TF32_TCGEN05) {
    tab(e->d_wshadow, sizeof(float) * (int64_t)S * e->layout.param_floats);
    tab(e->d_tshadow, sizeof(float) * (int64_t)S * e->layout.q_floats);
    tab(e->d_wshadow_lo, sizeof(float) * (int64_t)S * e->layout.param_floats);
    tab(e->d_tshadow_lo, sizeof(float) * (int64_t)S * e->layout.q_floats);
    tab(e->d_maps_first, (int64_t)128 * 4 * S * N_PASS);
    tab(e->d_maps_store, (int64_t)128 * L * S * N_PASS);
    tab(e->d_maps_c, (int64_t)128 * nprob);
    tab(e->d_maps_chain, (int64_t)128 * 2 * 4 * S * (2 * L));  // chain maps: <= 2L - 1 phases x 4 S tasks x (A, B)
    tab(e->d_maps_pol, (int64_t)128 * 4 * S);                   // policy-head maps: H_L, Wp hi, H_L, Wp lo
  }
  return tb;
}

static void build_layout(iql_engine* e) {
  const iql_config& c = e->cfg;
  const int L = c.n_hidden, H = c.hidden_dim;
  int64_t off = 0;
  auto add = [&](int net, int layer, int kind, int rows, int cols) {
    iql_tensor_info t;
    memset(&t, 0, sizeof(t));
    t.net = net; t.layer = layer; t.kind = kind; t.rows = rows; t.cols = cols; t.offset = off;
    // weight rows are padded to a multiple of 4 floats: 16-byte aligned rows are what TMA needs to
    // stream the first-layer weights (K = 11..69) into the tcgen05 pipeline; padding stays zero
    t.ld = (kind == IQL_KIND_WEIGHT) ? (int)round_up(cols, 4) : 1;
    e->tensors.push_back(t);
    off = round_up(off + (int64_t)rows * t.ld, 32);  // every tensor starts 128-byte aligned
    return t.offset;
  };
  // order == reference optimizer parameter order: qf.parameters() = q1 then q2 (iql.py:422-423),
  // vf, actor (log_std registered after net but listed first by nn.Module? no: see below)
  for (int net = 0; net < 4; ++net) {
    if (net == IQL_NET_V) { e->layout.q_floats = off; e->layout.v_begin = off; }
    if (net == IQL_NET_ACTOR) {
      e->layout.v_end = off;
      e->layout.actor_begin = off;
      if (!c.deterministic) e->log_std_off = add(net, 0, IQL_KIND_LOG_STD, c.action_dim, 1);
    }
    for (int l = 0; l <= L; ++l) {
      const int in = (l == 0) ? net_in_dim(c, net) : H;
      const int out = (l == L) ? net_out_dim(c, net) : H;
      e->w_off[net][l] = add(net, l, IQL_KIND_WEIGHT, out, in);
      e->w_ld[net][l] = (int)round_up(in, 4);
      e->b_off[net][l] = add(net, l, IQL_KIND_BIAS, out, 1);
    }
  }
  e->layout.actor_end = off;
  e->layout.param_floats = off;
  e->layout.n_tensors = (int)e->tensors.size();
  make_row_layout(c.state_dim, c.action_dim, &e->layout.row);

  // workspace (per member, floats; every region 128-byte aligned)
  WorkspaceLayout& wl = e->wl;
  const int64_t B = c.batch_size;
  wl.Ald = (int)round_up(c.action_dim, 4);
  int64_t w = 0;
  auto region = [&](int64_t n) { int64_t o = w; w = round_up(w + n, 32); return o; };
  wl.xrow = region(B * e->layout.row.row_floats);
  wl.act = region((int64_t)N_PASS * L * B * H);
  wl.yq = region(6 * B);
  wl.zpi = region(B * wl.Ald);
  wl.gy = region(3 * B);
  wl.gpi = region(B * wl.Ald);
  wl.gh = region((int64_t)4 * 2 * B * H);
  // row split of the output-layer backward: enough CTAs to fill the GPU when there are few problems and many rows
  e->lb_splits = 1;
  wl.lb_scratch = 0;
  wl.lb_stride = 0;
  // (stress shape: 4 problems x 4096 rows; single learners: 4 problems x 256 rows, 8 splits of 32 rows)
  if ((B >= 2048 || c.n_members <= 4) && c.action_dim <= 24 && (H % 4) == 0 && dbg_getenv("IQL_B200_NO_LASTBWD_SPLIT") == nullptr) {
    const int64_t ctas = (int64_t)4 * c.n_members * ((H + 255) / 256);
    int sp = 1;
    while (ctas * sp < 148 && B / (sp * 2) >= 32 && B % (sp * 2) == 0 && sp < 32) sp *= 2;
    if (sp > 1) {
      e->lb_splits = sp;
      wl.lb_stride = round_up((int64_t)std::max(c.action_dim, 1) * H + 32 + H, 32);  // dW partial, db partial, db_{L-1} partial
      wl.lb_scratch = region((int64_t)4 * sp * wl.lb_stride);
    }
  }
  e->fw_splits = 1;
  wl.fw_scratch = 0;
  wl.fw_stride = 0;
  if (B >= 2048 && c.math_mode == IQL_MATH_TF32_TCGEN05 && dbg_getenv("IQL_B200_NO_FIRST_WGRAD_SPLIT") == nullptr) {
    const int64_t tiles = (int64_t)4 * c.n_members * ((H + 127) / 128);
    int sp = 1;
    while (tiles * sp < 148 && B / (sp * 2) >= 256 && B % (sp * 2) == 0 && sp < 16) sp *= 2;
    if (sp > 1) {
      e->fw_splits = sp;
      const int64_t ldmax = round_up(c.state_dim + c.action_dim, 4);
      wl.fw_stride = round_up((int64_t)H * ldmax + H, 32);  // dW_0 partial [H][ld], db_0 partial [H]
      wl.fw_scratch = region((int64_t)4 * sp * wl.fw_stride);
    }
  }
  wl.xhi = wl.xlo = wl.bits = 0;
  if (c.math_mode == IQL_MATH_TF32_TCGEN05) {
    wl.xhi = region(B * e->layout.row.row_floats);
    wl.xlo = region(B * e->layout.row.row_floats);
    wl.bits = region((int64_t)4 * (L > 1 ? L - 1 : 0) * B * (H / 32 + 1));
  }
  wl.member_floats = w;

  e->tables_bytes = place_tables(e, nullptr);
  e->layout.workspace_bytes = e->tables_bytes + (int64_t)c.n_members * wl.member_floats * (int64_t)sizeof(float);
}

extern "C" int iql_create(const iql_config* cfg, iql_engine** out) {
  if (!cfg || !out) return fail(nullptr, IQL_ERR_INVALID, "iql_create: null argument");
  if (cfg->n_members <= 0 || cfg->state_dim <= 0 || cfg->action_dim <= 0 || cfg->batch_size <= 0)
    return fail(nullptr, IQL_ERR_INVALID, "iql_create: n_members, state_dim, action_dim, batch_size must be positive");
  if (cfg->n_hidden < 1 || cfg->n_hidden > 15) return fail(nullptr, IQL_ERR_INVALID, "iql_create: n_hidden must be in [1, 15]");
  if (cfg->hidden_dim <= 0 || (cfg->hidden_dim & 3)) return fail(nullptr, IQL_ERR_INVALID, "iql_create: hidden_dim must be a positive multiple of 4");
  if (cfg->math_mode != IQL_MATH_FP32_SIMT && cfg->math_mode != IQL_MATH_TF32_TCGEN05)
    return fail(nullptr, IQL_ERR_INVALID, "iql_create: unknown math_mode");
  if (cfg->max_steps_per_call <= 0) return fail(nullptr, IQL_ERR_INVALID, "iql_create: max_steps_per_call must be positive");
  if (!cfg->deterministic && cfg->action_dim > 64)
    return fail(nullptr, IQL_ERR_INVALID, "iql_create: Gaussian policies support action_dim <= 64");
  iql_engine* e = new iql_engine();
  e->cfg = *cfg;
  memset(&e->layout, 0, sizeof(e->layout));
  memset(e->w_off, 0, sizeof(e->w_off));
  memset(e->b_off, 0, sizeof(e->b_off));
  memset(e->w_ld, 0, sizeof(e->w_ld));
  build_layout(e);
  const int S = cfg->n_members;
  e->h_scalars.resize(S);
  e->h_hparams.resize(S);
  e->h_counters.assign(S, iql_counters{0, 0, 0, 0, 0, 0});
  e->act_steps.assign(S, 0);
  e->h_replay.assign(S, ReplayBinding{nullptr, 0, 0});
  e->preloaded.assign(S, 0);
  e->active.resize(S);
  for (int m = 0; m < S; ++m) e->active[m] = m;
  e->is_active.assign(S, 1);
  iql_hparams def;
  memset(&def, 0, sizeof(def));
  def.beta = 3.0; def.iql_tau = 0.7; def.discount = 0.99; def.tau = 0.005;
  def.vf_lr = def.qf_lr = def.actor_lr = 3e-4;
  def.adam_beta1 = 0.9; def.adam_beta2 = 0.999; def.adam_eps = 1e-8;
  def.cosine_t_max = 1000000;
  for (int m = 0; m < S; ++m) {
    e->h_scalars[m].batch = cfg->batch_size;
    def.seed = (uint64_t)m;
    iql_set_hparams(e, m, &def);
  }
  const char* g = dbg_getenv("IQL_B200_GRAPHS");
  if (g && g[0] == '0') e->use_graphs = false;
  *out = e;
  return IQL_OK;
}

static void drop_graphs(iql_engine* e) {
  for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second.first);
  e->graphs.clear();
}

extern "C" void iql_destroy(iql_engine* e) {
  if (!e) return;
  drop_graphs(e);
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_side) cudaEventDestroy(e->ev_side);
  if (e->ev_fork_g) cudaEventDestroy(e->ev_fork_g);
  if (e->ev_gather) cudaEventDestroy(e->ev_gather);
  if (e->side) cudaStreamDestroy(e->side);
  if (e->ev_in) cudaEventDestroy(e->ev_in);
  if (e->h_mail) cudaFreeHost(e->h_mail);
  if (e->h_act) cudaFreeHost(e->h_act);
  if (e->h_actm) cudaFreeHost(e->h_actm);
  if (e->h_ins) cudaFreeHost(e->h_ins);  // synchronises with the device: no insert launch still reads the slots
  if (e->d_stamps) cudaFree(e->d_stamps);
  delete e;
}

extern "C" int iql_get_layout(const iql_engine* e, iql_layout* out) {
  if (!e || !out) return IQL_ERR_INVALID;
  *out = e->layout;
  return IQL_OK;
}

extern "C" int iql_tensor_at(const iql_engine* e, int32_t index, iql_tensor_info* out) {
  if (!e || !out || index < 0 || index >= (int)e->tensors.size()) return IQL_ERR_INVALID;
  *out = e->tensors[index];
  return IQL_OK;
}

extern "C" int iql_set_hparams(iql_engine* e, int32_t member, const iql_hparams* hp) {
  if (!e || !hp || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_set_hparams: bad member or null");
  if (hp->actor_dropout < 0.0 || hp->actor_dropout >= 1.0) return fail(e, IQL_ERR_INVALID, "iql_set_hparams: actor_dropout must be in [0, 1)");
  if (hp->cosine_t_max < 0) return fail(e, IQL_ERR_INVALID, "iql_set_hparams: cosine_t_max must be >= 0");
  e->h_hparams[member] = *hp;
  MemberScalars& s = e->h_scalars[member];
  const int32_t batch = s.batch;  // set by iql_set_batch_sizes, not a hyper-parameter of iql_hparams
  memset(&s, 0, sizeof(s));
  s.batch = batch;
  s.beta = (float)hp->beta;
  s.iql_tau = (float)hp->iql_tau;
  s.discount = (float)hp->discount;
  s.tau = (float)hp->tau;
  s.one_minus_tau = (float)(1.0 - hp->tau);
  s.adam_w1 = (float)(1.0 - hp->adam_beta1);
  s.adam_beta2 = (float)hp->adam_beta2;
  s.adam_one_minus_b2 = (float)(1.0 - hp->adam_beta2);
  s.adam_eps = (float)hp->adam_eps;
  s.drop_scale = (float)(1.0 / (1.0 - hp->actor_dropout));
  s.drop_threshold = dropout_threshold(hp->actor_dropout);
  s.adam_beta1_d = hp->adam_beta1;
  s.adam_beta2_d = hp->adam_beta2;
  s.vf_lr = hp->vf_lr; s.qf_lr = hp->qf_lr; s.actor_lr = hp->actor_lr; s.lr_eta_min = hp->lr_eta_min;
  s.cosine_t_max = hp->cosine_t_max;
  s.seed = hp->seed;
  e->scalars_dirty = true;
  return IQL_OK;
}

extern "C" int iql_set_option(iql_engine* e, int32_t key, int64_t value) {
  if (!e) return IQL_ERR_INVALID;
  if (key == IQL_OPT_STEP_PATH) {
    if (value < 0 || value > 4 || value == 3)
      return fail(e, IQL_ERR_INVALID, "iql_set_option: IQL_OPT_STEP_PATH must be 0 (auto), 1 (per-phase kernels), 2 (chained backward + "
                                      "optimizer) or 4 (chained backward, optimizer in its own kernel)");
    if (e->bound && e->step_path != (int)value) return fail(e, IQL_ERR_STATE, "iql_set_option: IQL_OPT_STEP_PATH must be set before iql_bind_state");
    e->step_path = (int)value;
    return IQL_OK;
  }
  if (key == IQL_OPT_KEEP_GRADS) {
    e->keep_grads = value != 0;
    drop_graphs(e);  // the flag is baked into captured launches
    return IQL_OK;
  }
  return fail(e, IQL_ERR_INVALID, "iql_set_option: unknown key");
}

extern "C" int iql_get_info(const iql_engine* e, int32_t key, int64_t* out) {
  if (!e || !out) return IQL_ERR_INVALID;
  switch (key) {
    case IQL_INFO_TENSOR_CORE_PATH: *out = tensor_core_path(e->cfg) ? 1 : 0; return IQL_OK;   // 0: the FP32 CUDA-core kernels run this shape
    case IQL_INFO_FUSED_FORWARD: *out = e->bound && e->fused_fwd ? 1 : 0; return IQL_OK;
    case IQL_INFO_CHAINED_BACKWARD: *out = e->bound && e->chain && !e->chain_grads ? 1 : 0; return IQL_OK;
    case IQL_INFO_CHAINED_BACKWARD_GRADS: *out = e->bound && e->chain && e->chain_grads ? 1 : 0; return IQL_OK;
    default: return IQL_ERR_INVALID;
  }
}

extern "C" int iql_set_counters(iql_engine* e, int32_t member, const iql_counters* c) {
  if (!e || !c || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_set_counters: bad member or null");
  e->h_counters[member] = *c;
  e->counters_dirty = true;
  return IQL_OK;
}

extern "C" int iql_get_counters(iql_engine* e, int32_t member, iql_counters* out, void* stream) {
  (void)stream;  // the host shadow advances in lock-step with the device copy
  if (!e || !out || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_get_counters: bad member or null");
  *out = e->h_counters[member];
  return IQL_OK;
}

extern "C" int iql_set_batch_sizes(iql_engine* e, const int32_t* host_sizes) {
  if (!e || !host_sizes) return fail(e, IQL_ERR_INVALID, "iql_set_batch_sizes: null argument");
  const int S = e->cfg.n_members;
  for (int m = 0; m < S; ++m)
    if (host_sizes[m] < 1 || host_sizes[m] > e->cfg.batch_size)
      return fail(e, IQL_ERR_INVALID, "iql_set_batch_sizes: member " + std::to_string(m) + " has batch size " +
                                          std::to_string(host_sizes[m]) + ", outside [1, " + std::to_string(e->cfg.batch_size) + "]");
  for (int m = 0; m < S; ++m) e->h_scalars[m].batch = host_sizes[m];
  e->scalars_dirty = true;  // uploaded with the scalars before the next launch; the graphs read the table at run time
  return IQL_OK;
}

extern "C" int iql_get_batch_sizes(iql_engine* e, int32_t* host_out) {
  if (!e || !host_out) return fail(e, IQL_ERR_INVALID, "iql_get_batch_sizes: null argument");
  for (int m = 0; m < e->cfg.n_members; ++m) host_out[m] = e->h_scalars[m].batch;
  return IQL_OK;
}

static void build_problems(iql_engine* e) {
  const iql_config& c = e->cfg;
  const int Sa = (int)e->active.size(), L = c.n_hidden, H = c.hidden_dim, B = c.batch_size;
  const int ROW = e->layout.row.row_floats;
  const WorkspaceLayout& wl = e->wl;
  const int64_t P = e->layout.param_floats, PQ = e->layout.q_floats;
  const bool use_shadow = tensor_core_path(c);
  // hidden-layer weights as tcgen05 operands: read from the arenas themselves (biased in place during a call) instead of
  // from a TF32-rounded shadow copy
  e->bias_hidden = use_shadow && L >= 2 && L <= 4 && dbg_getenv("IQL_B200_NO_BIASED_WEIGHTS") == nullptr;
  const bool hid_shadow = use_shadow && !e->bias_hidden;
  e->h_probs.clear();
  e->fwd_phases.clear();
  e->bwd_phases.clear();
  struct PassDef { int net; bool tgt; int in_off; int k0; };
  const PassDef passes[N_PASS] = {
      {IQL_NET_V, false, e->layout.row.off_next_state, c.state_dim},
      {IQL_NET_V, false, 0, c.state_dim},
      {IQL_NET_Q1, true, 0, c.state_dim + c.action_dim},
      {IQL_NET_Q2, true, 0, c.state_dim + c.action_dim},
      {IQL_NET_Q1, false, 0, c.state_dim + c.action_dim},
      {IQL_NET_Q2, false, 0, c.state_dim + c.action_dim},
      {IQL_NET_ACTOR, false, 0, c.state_dim},
  };
  auto wsm = [&](int m) { return e->d_ws_f + (int64_t)m * wl.member_floats; };
  auto actp = [&](int m, int f, int l) { return wsm(m) + wl.act + ((int64_t)(f * L + l)) * B * H; };
  auto blank = [&]() { GemmProb p; memset(&p, 0, sizeof(p)); p.drop_layer = -1; return p; };
  // sign bits of activation index a (0-based: output of forward layer a) of training pass slot t (V, q1, q2, actor)
  auto bitsp = [&](int m, int t, int a) {
    return reinterpret_cast<uint32_t*>(wsm(m) + wl.bits) + ((int64_t)(t * (L - 1) + a)) * B * (H / 32);
  };
  // ---- forward phases, layer 0..L ----
  for (int l = 0; l <= L; ++l) {
    Phase ph; ph.mode = 0; ph.first = (int)e->h_probs.size(); ph.maxM = B; ph.maxN = 0; ph.K = 0; ph.umma_ok = false;
    // pass-major order: the six scalar-head passes of all members first, the policy pass last
    for (int f = 0; f < N_PASS; ++f)
      for (const int m : e->active) {
        const PassDef& pd = passes[f];
        const float* blk = pd.tgt ? e->target + (int64_t)m * PQ : e->params + (int64_t)m * P;
        GemmProb p = blank();
        p.member = m;
        p.M = B;
        if (l == 0) { p.A = wsm(m) + wl.xrow + pd.in_off; p.lda = ROW; p.K = pd.k0; }
        else { p.A = actp(m, f, l - 1); p.lda = H; p.K = H; }
        p.B = blk + e->w_off[pd.net][l];
        if (hid_shadow && l >= 1 && l < L)  // hidden-layer weights feed tcgen05: the TF32-rounded copy (or, bias_hidden, the arena itself)
          p.B = (pd.tgt ? e->d_tshadow + (int64_t)m * PQ : e->d_wshadow + (int64_t)m * P) + e->w_off[pd.net][l];
        p.ldb = e->w_ld[pd.net][l];
        p.bias = blk + e->b_off[pd.net][l];
        if (l < L) {
          p.N = H; p.C = actp(m, f, l); p.ldc = H; p.epi = EPI_RELU;
          p.drop_layer = (f == PASS_PI) ? l : -1;
          // H_L of the forward-only passes (V(s'), target Q) is consumed only by the fused output Linear
          p.no_store = (l == L - 1 && (f == PASS_V_NEXT || f == PASS_TQ1 || f == PASS_TQ2)) ? 1 : 0;
          const int tslot = (f == PASS_V) ? 0 : (f == PASS_Q1) ? 1 : (f == PASS_Q2) ? 2 : (f == PASS_PI) ? 3 : -1;
          if (use_shadow && tslot >= 0 && l < L - 1) p.bits = bitsp(m, tslot, l);  // sign bits of H_{l+1}, for dgrad
        } else if (f == PASS_PI) {
          p.N = c.action_dim; p.C = wsm(m) + wl.zpi; p.ldc = wl.Ald; p.epi = EPI_LINEAR;
        } else {
          p.N = 1; p.C = wsm(m) + wl.yq + (int64_t)f * B; p.ldc = 1; p.epi = EPI_LINEAR;
        }
        if (p.N > ph.maxN) ph.maxN = p.N;
        e->h_probs.push_back(p);
      }
    ph.count = (int)e->h_probs.size() - ph.first;
    ph.K = (l >= 1) ? H : 0;
    ph.umma_ok = true;  // every forward layer has a tcgen05 form (K tails / N < 32 are zero-filled by TMA)
    ph.epi = (l < L) ? EPI_RELU : EPI_LINEAR;
    ph.kind = (l == 0) ? PH_FIRST_FWD : (l == L ? PH_OUT_FWD : PH_GENERIC);
    e->fwd_phases.push_back(ph);
  }
  // ---- backward phases ----
  struct TrainDef { int net; int pass; };
  const TrainDef tr[4] = {{IQL_NET_V, PASS_V}, {IQL_NET_Q1, PASS_Q1}, {IQL_NET_Q2, PASS_Q2}, {IQL_NET_ACTOR, PASS_PI}};
  auto ghp = [&](int m, int t, int which) { return wsm(m) + wl.gh + ((int64_t)(t * 2 + which)) * B * H; };
  for (int l = L; l >= 0; --l) {
    // weight gradient  dW_l = G_l^T H_l   (TN)
    Phase pw; pw.mode = 2; pw.first = (int)e->h_probs.size(); pw.maxM = 0; pw.maxN = 0; pw.K = B; pw.umma_ok = (l < L);
    pw.epi = EPI_NONE;
    pw.kind = (l == L) ? PH_LAST_WGRAD : (l == 0 ? PH_FIRST_WGRAD : PH_GENERIC);
    for (const int m : e->active)
      for (int t = 0; t < 4; ++t) {
        const int net = tr[t].net, f = tr[t].pass;
        const PassDef& pd = passes[f];
        GemmProb p = blank();
        p.member = m;
        p.K = B;
        if (l == L) {
          if (t == 3) { p.A = wsm(m) + wl.gpi; p.lda = wl.Ald; p.M = c.action_dim; }
          else { p.A = wsm(m) + wl.gy + (int64_t)t * B; p.lda = 1; p.M = 1; }
        } else { p.A = ghp(m, t, (L - 1 - l) & 1); p.lda = H; p.M = H; }
        if (l == 0) { p.B = wsm(m) + wl.xrow + pd.in_off; p.ldb = ROW; p.N = pd.k0; }
        else { p.B = actp(m, f, l - 1); p.ldb = H; p.N = H; }
        p.C = e->grads + (int64_t)m * P + e->w_off[net][l];
        p.ldc = e->w_ld[net][l];
        p.dbias = e->grads + (int64_t)m * P + e->b_off[net][l];
        p.epi = EPI_NONE;
        if (p.M > pw.maxM) pw.maxM = p.M;
        if (p.N > pw.maxN) pw.maxN = p.N;
        e->h_probs.push_back(p);
      }
    pw.count = (int)e->h_probs.size() - pw.first;
    e->bwd_phases.push_back(pw);
    if (l == 0) break;
    // activation gradient  G_{l-1} = (G_l W_l) * [H_l > 0]   (NN)
    Phase px; px.mode = 1; px.first = (int)e->h_probs.size(); px.maxM = B; px.maxN = H; px.K = (l < L) ? H : 0; px.umma_ok = (l < L);
    px.epi = EPI_DRELU;
    px.kind = (l == L) ? PH_LAST_DGRAD : PH_GENERIC;
    for (const int m : e->active)
      for (int t = 0; t < 4; ++t) {
        const int net = tr[t].net, f = tr[t].pass;
        GemmProb p = blank();
        p.member = m;
        p.M = B; p.N = H;
        if (l == L) {
          if (t == 3) { p.A = wsm(m) + wl.gpi; p.lda = wl.Ald; p.K = c.action_dim; }
          else { p.A = wsm(m) + wl.gy + (int64_t)t * B; p.lda = 1; p.K = 1; }
        } else { p.A = ghp(m, t, (L - 1 - l) & 1); p.lda = H; p.K = H; }
        p.B = ((hid_shadow && l < L) ? e->d_wshadow : e->params) + (int64_t)m * P + e->w_off[net][l];
        p.ldb = e->w_ld[net][l];
        p.C = ghp(m, t, (L - l) & 1);
        p.ldc = H;
        p.mask = actp(m, f, l - 1);
        p.ldmask = H;
        if (use_shadow && l < L) p.bits = bitsp(m, t, l - 1);  // same activation as p.mask, 1 bit per element
        p.epi = EPI_DRELU;
        p.drop_layer = (t == 3) ? (l - 1) : -1;
        // bias gradient of the layer below = column sums of the gradient this problem produces
        // (written by the tcgen05 dgrad epilogue; the FP32 kernels compute it in their wgrad instead)
        p.dbias = e->grads + (int64_t)m * P + e->b_off[net][l - 1];
        e->h_probs.push_back(p);
      }
    px.count = (int)e->h_probs.size() - px.first;
    e->bwd_phases.push_back(px);
  }
  // row-split copies of the output-layer backward problems: every split is a problem of its own over B / splits rows
  // whose weight / bias gradient partials go to the scratch region; lb_reduce_kernel adds them up in split order
  e->lb_first = (int64_t)e->h_probs.size();
  if (e->lb_splits > 1 && e->bwd_phases.size() >= 3) {
    const int sp = e->lb_splits, Bs = B / sp;
    const Phase pw0 = e->bwd_phases[0], pn0 = e->bwd_phases[1], pv0 = e->bwd_phases[2];
    for (int which = 0; which < 3; ++which)
      for (int s_ = 0; s_ < sp; ++s_)
        for (int mi = 0; mi < Sa; ++mi)
          for (int t = 0; t < 4; ++t) {
            const int m = e->active[mi], i = mi * 4 + t;  // position of (member, net) in the phase
            float* scr = wsm(m) + wl.lb_scratch + ((int64_t)t * sp + s_) * wl.lb_stride;
            GemmProb p;
            if (which == 0) {  // dgrad: rows [s Bs, (s + 1) Bs)
              p = e->h_probs[pn0.first + i];
              p.A += (int64_t)s_ * Bs * p.lda;
              p.C += (int64_t)s_ * Bs * p.ldc;
              p.mask += (int64_t)s_ * Bs * p.ldmask;
              p.M = Bs;
              p.row0 = s_ * Bs;
            } else if (which == 1) {  // wgrad: partial dW_L [A][H], partial db_L
              p = e->h_probs[pw0.first + i];
              p.C = scr;  // ldc stays that of dW_L (= H)
              p.dbias = scr + (int64_t)std::max(c.action_dim, 1) * H;
              p.K = Bs;
            } else {  // wgrad of the layer below: only its bias gradient (column sums of the G this kernel produces)
              p = e->h_probs[pv0.first + i];
              p.dbias = scr + (int64_t)std::max(c.action_dim, 1) * H + 32;
            }
            e->h_probs.push_back(p);
          }
  }
  // K-split copies of the input-layer weight-gradient problems (G_0 and X rows [s Bs, (s + 1) Bs))
  e->fw_phase = Phase();
  if (e->fw_splits > 1 && !e->bwd_phases.empty() && e->bwd_phases.back().kind == PH_FIRST_WGRAD) {
    const int sp = e->fw_splits, Bs = B / sp;
    const Phase p0 = e->bwd_phases.back();
    Phase pf = p0;
    pf.first = (int)e->h_probs.size();
    pf.K = Bs;
    for (int s_ = 0; s_ < sp; ++s_)
      for (int mi = 0; mi < Sa; ++mi)
        for (int t = 0; t < 4; ++t) {
          const int m = e->active[mi];
          GemmProb p = e->h_probs[p0.first + mi * 4 + t];
          float* scr = wsm(m) + wl.fw_scratch + ((int64_t)t * sp + s_) * wl.fw_stride;
          p.A += (int64_t)s_ * Bs * p.lda;
          p.B += (int64_t)s_ * Bs * p.ldb;
          p.K = Bs;
          p.C = scr;  // same ldc as dW_0
          p.dbias = p.dbias ? scr + (int64_t)p.M * p.ldc : nullptr;
          e->h_probs.push_back(p);
        }
    pf.count = (int)e->h_probs.size() - pf.first;
    e->fw_phase = pf;
  } else {
    e->fw_splits = 1;
  }
}

// The part of binding that depends on which members train: problem tables, tensor maps, the chained backward's task
// list and every path choice made from the member count.  Run by iql_bind_state and again by iql_set_active_members;
// the workspace split (lb_splits / fw_splits) stays as iql_create sized it.
static int bind_tables(iql_engine* e) {
  const int Sa = (int)e->active.size(), L = e->cfg.n_hidden;
  const int64_t nprob = problem_count(e, Sa);
  build_problems(e);
  const bool tc_mode = tensor_core_path(e->cfg);
  // 3xTF32 input layer, and on top of it the fused forward (all hidden layers of a tile chained through TMEM)
  e->split_first = tc_mode && dbg_getenv("IQL_B200_NO_SPLIT_FIRST") == nullptr;
  e->fused_fwd = e->split_first && umma_can_fuse_out(e->cfg.action_dim) &&
                 fused_fwd_supported(e->cfg.batch_size, e->cfg.hidden_dim, e->cfg.n_hidden, e->cfg.state_dim + e->cfg.action_dim);
  e->fused_pair = e->fused_fwd && fused_fwd_pair(e->cfg.batch_size);
  for (auto* phases : {&e->fwd_phases, &e->bwd_phases})
    for (Phase& ph : *phases) {
      ph.maxK = 0;
      for (int i = 0; i < ph.count; ++i) ph.maxK = std::max(ph.maxK, e->h_probs[ph.first + i].K);
      // phases run by the fused forward: the weight boxes are full tiles, or half tiles when it runs on CTA pairs
      const bool in_fused = e->fused_fwd && ph.mode == 0 && ph.kind != PH_OUT_FWD;
      ph.cta2 = in_fused ? e->fused_pair : (ph.umma_ok && umma_cta2(ph.mode, ph.count, ph.maxM, ph.maxN, ph.maxK));
      // few dgrad problems (single learners, small ensembles): two N = 128 (or four N = 64) units per problem on more CTA
      // pairs -- fewer MMAs and one epilogue chunk per warp instead of two on the step's critical path
      ph.tile_n = 0;
      if (!in_fused && ph.cta2 && ph.mode == 1 && ph.kind == PH_GENERIC && ph.maxN % 256 == 0 && 2 * ph.count * (ph.maxN / 256) <= 74 &&
          dbg_getenv("IQL_B200_NO_NARROW_DGRAD") == nullptr)
        ph.tile_n = (4 * ph.count * (ph.maxN / 256) <= 74 && dbg_getenv("IQL_B200_NO_DGRAD_N64") == nullptr) ? 64 : 128;  // single learners: four units
      // backward hidden-layer phases: row-layout epilogue (TMA stores; dgrad masks with the sign bits the fused
      // forward wrote -- without the fused forward the bits do not exist and dgrad keeps the FP32 mask)
      // (the same epilogue on the weight-gradient phase measured 46.4 vs 44.2 us: it stays on the transposing one)
      const bool hidden_dgrad = tc_mode && ph.umma_ok && ph.kind == PH_GENERIC && (ph.maxN % 32) == 0 && ph.mode == 1 &&
                                e->fused_fwd;
      ph.rowepi = (hidden_dgrad || (ph.mode == 2 && ph.kind == PH_GENERIC && tc_mode && dbg_getenv("IQL_B200_ROWEPI_WGRAD"))) &&
                  dbg_getenv("IQL_B200_NO_ROWEPI") == nullptr;
    }
  if (e->fw_splits > 1) {
    Phase& pf = e->fw_phase;
    pf.maxK = 0;
    for (int i = 0; i < pf.count; ++i) pf.maxK = std::max(pf.maxK, e->h_probs[pf.first + i].K);
    pf.cta2 = pf.umma_ok && umma_cta2(pf.mode, pf.count, pf.maxM, pf.maxN, pf.maxK);
    pf.rowepi = false;
  }
  if ((int64_t)e->h_probs.size() != nprob) return fail(e, IQL_ERR_STATE, "internal: problem count mismatch");
  e->h_maps.assign((size_t)128 * 2 * nprob, 0);
  if (e->cfg.math_mode == IQL_MATH_TF32_TCGEN05) {
    auto encode = [&](const Phase& ph) {
      if (!ph.umma_ok || !umma_phase_supported(ph.mode, e->cfg.batch_size, e->cfg.hidden_dim)) return 0;
      return umma_encode_maps(ph.mode, e->h_probs.data() + ph.first, ph.count, ph.tile_n ? ph.tile_n : umma_tile_n(ph.maxN),
                              e->h_maps.data() + (size_t)256 * ph.first, ph.cta2);
    };
    for (const Phase& ph : e->fwd_phases) if (encode(ph)) return fail(e, IQL_ERR_CUDA, "cuTensorMapEncodeTiled failed (forward phase)");
    // 3xTF32 input layer: hi / lo operand maps of the first forward phase
    if (e->split_first) {
      const Phase& ph = e->fwd_phases[0];
      std::vector<GemmProb> hi(e->h_probs.begin() + ph.first, e->h_probs.begin() + ph.first + ph.count), lo = hi;
      const int64_t P = e->layout.param_floats, PQ = e->layout.q_floats;
      for (int i = 0; i < ph.count; ++i) {
        const GemmProb& g = e->h_probs[ph.first + i];
        const int m = g.member;
        const float* wsm = e->d_ws_f + (int64_t)m * e->wl.member_floats;
        const int64_t a_off = g.A - (wsm + e->wl.xrow);  // column offset of this pass's input inside the row
        hi[i].A = wsm + e->wl.xhi + a_off;
        lo[i].A = wsm + e->wl.xlo + a_off;
        const float* pblk = e->params + (int64_t)m * P;
        const float* tblk = e->target + (int64_t)m * PQ;
        const bool tgt = (g.B >= tblk && g.B < tblk + PQ);
        const int64_t w_off = tgt ? (g.B - tblk) : (g.B - pblk);
        hi[i].B = (tgt ? e->d_tshadow + (int64_t)m * PQ : e->d_wshadow + (int64_t)m * P) + w_off;
        lo[i].B = (tgt ? e->d_tshadow_lo + (int64_t)m * PQ : e->d_wshadow_lo + (int64_t)m * P) + w_off;
      }
      e->h_maps_first.assign((size_t)128 * 4 * ph.count, 0);
      if (umma_encode_maps_split(hi.data(), lo.data(), ph.count, umma_tile_n(ph.maxN), e->h_maps_first.data(), ph.cta2))
        return fail(e, IQL_ERR_CUDA, "cuTensorMapEncodeTiled failed (3xTF32 input layer)");
    }
    for (const Phase& ph : e->bwd_phases) if (encode(ph)) return fail(e, IQL_ERR_CUDA, "cuTensorMapEncodeTiled failed (backward phase)");
    if (e->fw_splits > 1 && encode(e->fw_phase)) return fail(e, IQL_ERR_CUDA, "cuTensorMapEncodeTiled failed (split input-layer wgrad)");
    e->h_maps_c.assign((size_t)128 * nprob, 0);
    for (const Phase& ph : e->bwd_phases)
      if (ph.rowepi)
        for (int i = 0; i < ph.count; ++i) {
          const GemmProb& g = e->h_probs[ph.first + i];
          if (umma_encode_store_map(e->h_maps_c.data() + (size_t)128 * (ph.first + i), g.C, g.M, g.N, g.ldc))
            return fail(e, IQL_ERR_CUDA, "cuTensorMapEncodeTiled failed (backward outputs)");
        }
    e->h_maps_store.clear();
    if (e->fused_fwd) {  // outputs H_1..H_L of every forward problem, stored by TMA from the fused kernel
      const int np = e->fwd_phases[0].count;
      e->h_maps_store.assign((size_t)128 * L * np, 0);
      for (int l = 0; l < L; ++l)
        for (int i = 0; i < np; ++i) {
          const GemmProb& g = e->h_probs[e->fwd_phases[l].first + i];
          if (umma_encode_store_map(e->h_maps_store.data() + (size_t)128 * (l * np + i), g.C, g.M, g.N, g.ldc))
            return fail(e, IQL_ERR_CUDA, "cuTensorMapEncodeTiled failed (fused forward outputs)");
        }
    }
  }
  // ---- wide policy head on the tensor cores (two-pass: H_L Wp_hi + H_L Wp_lo) ----
  e->pol_umma = false;
  e->h_maps_pol.clear();
  if (tc_mode && e->fused_fwd && !fused_fwd_policy_head(e->cfg.action_dim) && e->cfg.action_dim <= 32 &&
      dbg_getenv("IQL_B200_NO_POL_UMMA") == nullptr) {
    const Phase& pout = e->fwd_phases[L];
    const int n_scalar = (N_PASS - 1) * Sa;
    std::vector<GemmProb> hi(e->h_probs.begin() + pout.first + n_scalar, e->h_probs.begin() + pout.first + pout.count), lo = hi;
    const int64_t P = e->layout.param_floats;
    for (size_t i = 0; i < hi.size(); ++i) {
      const int m = hi[i].member;
      const int64_t w_off = hi[i].B - (e->params + (int64_t)m * P);
      hi[i].B = e->d_wshadow + (int64_t)m * P + w_off;
      lo[i].B = e->d_wshadow_lo + (int64_t)m * P + w_off;
    }
    e->h_maps_pol.assign((size_t)128 * 4 * hi.size(), 0);
    if ((int)hi.size() == Sa &&
        umma_encode_maps_split(hi.data(), lo.data(), (int)hi.size(), umma_tile_n(e->cfg.action_dim), e->h_maps_pol.data(), false) == 0)
      e->pol_umma = true;
    else
      e->h_maps_pol.clear();
  }
  // ---- chained backward: phase list and CTA-pair maps ----
  e->chain = e->chain_grads = false;
  e->h_maps_chain.clear();
  // IQL_OPT_STEP_PATH = 2 (opt-in): optimizer in the wgrad epilogue.  Measured on the 64-member ensemble it streams the
  // optimizer state at 72 % of the HBM peak against 99 % for adam_polyak_kernel and ends up 10 % behind the per-phase
  // kernels (DESIGN.md section 8).  IQL_OPT_STEP_PATH = 4: the chain computes the gradients only and adam_polyak_kernel
  // follows.  "auto" takes 4 from CHAIN_GRADS_MIN_MEMBERS members on, or with 3+ hidden layers: below that the
  // per-phase kernels' narrow dgrad units spread a two-layer step of few tasks over more SMs (DESIGN.md section 8).
  const bool want_chain = e->step_path == 2 || e->step_path == 4 ||
                          (e->step_path == 0 && (Sa >= CHAIN_GRADS_MIN_MEMBERS || e->cfg.n_hidden >= 3));
  if (tc_mode && want_chain && e->fw_splits == 1 && last_bwd_skinny_ok(e->cfg.batch_size, e->cfg.action_dim) &&
      bwd_chain_supported(e->cfg.batch_size, e->cfg.hidden_dim, e->cfg.n_hidden, e->cfg.state_dim + e->cfg.action_dim,
                          e->fused_fwd)) {
    const int ntask = 4 * Sa;
    BwdChainArgs& ca = e->chain_args;
    memset(&ca, 0, sizeof(ca));
    e->h_maps_chain.assign((size_t)128 * 2 * ntask * (2 * L), 0);
    int np = 0;
    bool ok = (int)e->bwd_phases.size() == 2 * L + 1;
    auto add_phase = [&](int kind, const Phase& ph, int tile_n, int k, int wait) {
      if (!ok) return;
      if (ph.count != ntask) { ok = false; return; }
      ca.kind[np] = kind; ca.prob_first[np] = ph.first; ca.map_first[np] = 2 * ntask * np;
      ca.tile_n[np] = tile_n; ca.k[np] = k; ca.wait_dgrads[np] = wait;
      if (umma_encode_maps(kind == 0 ? 1 : 2, e->h_probs.data() + ph.first, ph.count, tile_n,
                           e->h_maps_chain.data() + (size_t)128 * ca.map_first[np], true)) ok = false;
      ++np;
    };
    for (int l = L - 1; l >= 1 && ok; --l) {
      const Phase& pw = e->bwd_phases[2 * (L - l)];      // dW_l = dZ_l^T H_l
      const Phase& px = e->bwd_phases[2 * (L - l) + 1];  // dZ_{l-1} = (dZ_l W_l) * [H_l > 0]
      if (!px.rowepi || px.mode != 1 || pw.mode != 2) { ok = false; break; }
      ca.db_tile_order = px.cta2 ? 0 : 1;  // bias gradients summed as the per-phase dgrad of this shape sums them
      add_phase(0, px, 256, e->cfg.hidden_dim, L - 1 - l);
      add_phase(1, pw, 256, e->cfg.batch_size, L - 1 - l);
    }
    if (ok) {
      const Phase& p0 = e->bwd_phases[2 * L];
      add_phase(1, p0, bwd_chain_wgrad0_tile_n(p0.maxN), e->cfg.batch_size, L - 1);
    }
    if (ok) {
      ca.n_phases = np;
      ca.n_tasks = ntask;
      // parameters no phase covers: everything of a net except the weights of layers 0..L-1; adjacent tensors merge
      const int slot_net[4] = {IQL_NET_V, IQL_NET_Q1, IQL_NET_Q2, IQL_NET_ACTOR};
      for (int t = 0; t < 4 && ok; ++t) {
        int n = 0;
        for (size_t i = 0; i < e->tensors.size(); ++i) {
          const iql_tensor_info& ti = e->tensors[i];
          if (ti.net != slot_net[t]) continue;
          if (ti.kind == IQL_KIND_WEIGHT && ti.layer < L) continue;
          const int64_t lo = ti.offset;
          const int64_t hi = (i + 1 < e->tensors.size()) ? e->tensors[i + 1].offset : e->layout.param_floats;
          if (n > 0 && ca.seg_hi[t][n - 1] == lo) ca.seg_hi[t][n - 1] = hi;
          else if (n < FUSED_MAX_LAYERS + 2) { ca.seg_lo[t][n] = lo; ca.seg_hi[t][n] = hi; ++n; }
          else ok = false;
        }
        ca.n_seg[t] = n;
      }
    }
    e->chain = ok;
    e->chain_grads = ok && e->step_path != 2;
    if (!ok) e->h_maps_chain.clear();
  }
  if ((e->step_path == 2 || e->step_path == 4) && !e->chain)
    return fail(e, IQL_ERR_INVALID, "iql_bind_state: IQL_OPT_STEP_PATH = chained backward, but this shape / math mode does not support it "
                                    "(needs tf32, hidden 256, batch 256, 2..4 hidden layers, action_dim <= 24, "
                                    "state_dim + action_dim <= 256)");
  return IQL_OK;
}

extern "C" int iql_bind_state(iql_engine* e, float* params, float* exp_avg, float* exp_avg_sq, float* target,
                              float* grads, void* workspace, size_t workspace_bytes) {
  if (!e) return IQL_ERR_INVALID;
  if (!params || !exp_avg || !exp_avg_sq || !target || !grads || !workspace)
    return fail(e, IQL_ERR_INVALID, "iql_bind_state: null device pointer");
  if ((int64_t)workspace_bytes < e->layout.workspace_bytes) return fail(e, IQL_ERR_INVALID, "iql_bind_state: workspace too small");
  const uintptr_t all = (uintptr_t)params | (uintptr_t)exp_avg | (uintptr_t)exp_avg_sq | (uintptr_t)target |
                        (uintptr_t)grads | (uintptr_t)workspace;
  if (all & 127) return fail(e, IQL_ERR_INVALID, "iql_bind_state: pointers must be 128-byte aligned");
  e->params = params; e->exp_avg = exp_avg; e->exp_avg_sq = exp_avg_sq; e->target = target; e->grads = grads;
  e->ws = (char*)workspace; e->ws_bytes = workspace_bytes;
  place_tables(e, e->ws);
  e->d_ws_f = (float*)(e->ws + e->tables_bytes);
  int rc = bind_tables(e);
  if (rc != IQL_OK) return rc;
  if (!e->side) {  // optional: without it the backward simply stays on one stream
    if (cudaStreamCreateWithFlags(&e->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_side, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_fork_g, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->ev_gather, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      e->side = nullptr;
    }
  }
  if (dbg_getenv("IQL_STEP_TRACE") && !e->d_stamps && cudaMalloc((void**)&e->d_stamps, sizeof(unsigned long long) * 2 * ST_COUNT) != cudaSuccess) {
    cudaGetLastError();
    e->d_stamps = nullptr;
  }
  e->bound = true;
  e->tables_dirty = e->scalars_dirty = e->counters_dirty = e->replay_dirty = true;
  drop_graphs(e);
  return IQL_OK;
}

static int flush_tables(iql_engine* e, cudaStream_t st) {
  const int S = e->cfg.n_members, L = e->cfg.n_hidden;
  if (e->tables_dirty) {
    CUDA_TRY(e, cudaMemcpyAsync(e->d_probs, e->h_probs.data(), sizeof(GemmProb) * e->h_probs.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(e, cudaMemcpyAsync(e->d_maps, e->h_maps.data(), e->h_maps.size(), cudaMemcpyHostToDevice, st));
    if (!e->h_maps_first.empty())
      CUDA_TRY(e, cudaMemcpyAsync(e->d_maps_first, e->h_maps_first.data(), e->h_maps_first.size(), cudaMemcpyHostToDevice, st));
    if (!e->h_maps_c.empty())
      CUDA_TRY(e, cudaMemcpyAsync(e->d_maps_c, e->h_maps_c.data(), e->h_maps_c.size(), cudaMemcpyHostToDevice, st));
    if (!e->h_maps_store.empty())
      CUDA_TRY(e, cudaMemcpyAsync(e->d_maps_store, e->h_maps_store.data(), e->h_maps_store.size(), cudaMemcpyHostToDevice, st));
    if (!e->h_maps_chain.empty())
      CUDA_TRY(e, cudaMemcpyAsync(e->d_maps_chain, e->h_maps_chain.data(), e->h_maps_chain.size(), cudaMemcpyHostToDevice, st));
    if (!e->h_maps_pol.empty())
      CUDA_TRY(e, cudaMemcpyAsync(e->d_maps_pol, e->h_maps_pol.data(), e->h_maps_pol.size(), cudaMemcpyHostToDevice, st));
    std::vector<int64_t> off(2 * (L + 1));
    for (int l = 0; l <= L; ++l) {
      off[l] = e->w_off[IQL_NET_ACTOR][l];
      off[L + 1 + l] = e->b_off[IQL_NET_ACTOR][l];
    }
    CUDA_TRY(e, cudaMemcpyAsync(e->d_act_off, off.data(), sizeof(int64_t) * off.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(e, cudaMemcpyAsync(e->d_active, e->active.data(), sizeof(int32_t) * e->active.size(), cudaMemcpyHostToDevice, st));
    // loss rows of members that do not train read NaN (all-ones bytes) until they train again
    const size_t ring_row = sizeof(float) * 3 * (size_t)e->cfg.max_steps_per_call;
    for (int m = 0; m < S; ++m)
      if (!e->is_active[m]) CUDA_TRY(e, cudaMemsetAsync((char*)e->d_loss_ring + ring_row * m, 0xFF, ring_row, st));
    CUDA_TRY(e, cudaStreamSynchronize(st));  // `off` is a stack temporary
    e->tables_dirty = false;
  }
  if (e->scalars_dirty) {
    CUDA_TRY(e, cudaMemcpyAsync(e->d_scalars, e->h_scalars.data(), sizeof(MemberScalars) * S, cudaMemcpyHostToDevice, st));
    e->scalars_dirty = false;
  }
  if (e->counters_dirty) {
    CUDA_TRY(e, cudaMemcpyAsync(e->d_counters, e->h_counters.data(), sizeof(iql_counters) * S, cudaMemcpyHostToDevice, st));
    e->counters_dirty = false;
  }
  if (e->replay_dirty) {
    CUDA_TRY(e, cudaMemcpyAsync(e->d_replay, e->h_replay.data(), sizeof(ReplayBinding) * S, cudaMemcpyHostToDevice, st));
    e->replay_dirty = false;
  }
  return IQL_OK;
}

static StepCtx make_ctx(const iql_engine* e) {
  StepCtx c;
  memset(&c, 0, sizeof(c));
  c.B = e->cfg.batch_size;
  c.S_dim = e->cfg.state_dim; c.A_dim = e->cfg.action_dim; c.H = e->cfg.hidden_dim; c.L = e->cfg.n_hidden;
  c.deterministic = e->cfg.deterministic;
  c.n_active = (int)e->active.size();
  c.active = (int)e->active.size() < e->cfg.n_members ? e->d_active : nullptr;
  c.P = e->layout.param_floats; c.PQ = e->layout.q_floats;
  c.v_begin = e->layout.v_begin; c.v_end = e->layout.v_end;
  c.a_begin = e->layout.actor_begin; c.a_end = e->layout.actor_end;
  c.log_std_off = e->log_std_off;
  c.row = e->layout.row;
  c.scalars = e->d_scalars; c.counters = e->d_counters; c.replay = e->d_replay;
  c.loss_ring = e->d_loss_ring;
  c.adam_sc = e->d_adam_sc;
  c.k_max = e->cfg.max_steps_per_call;
  c.tf32 = tensor_core_path(e->cfg);
  c.w_shadow = e->d_wshadow;
  c.t_shadow = e->d_tshadow;
  c.w_shadow_lo = e->d_wshadow_lo;
  c.t_shadow_lo = e->d_tshadow_lo;
  for (int n = 0; n < 4; ++n) {
    c.first_w_begin[n] = e->split_first ? e->w_off[n][0] : 0;
    c.first_w_end[n] = e->split_first ? e->w_off[n][0] + (int64_t)e->cfg.hidden_dim * e->w_ld[n][0] : 0;
  }
  c.bias_hidden = (c.tf32 && e->bias_hidden) ? 1 : 0;
  c.n_hid = 0;
  if (c.bias_hidden)
    for (int n = 0; n < 4; ++n)
      for (int l = 1; l < e->cfg.n_hidden; ++l) {
        c.hid_begin[c.n_hid] = e->w_off[n][l];
        c.hid_end[c.n_hid] = e->w_off[n][l] + (int64_t)e->cfg.hidden_dim * e->w_ld[n][l];
        ++c.n_hid;
      }
  const int Lh = e->cfg.n_hidden;
  c.first_w_begin[4] = e->pol_umma ? e->w_off[IQL_NET_ACTOR][Lh] : 0;
  c.first_w_end[4] = e->pol_umma ? e->w_off[IQL_NET_ACTOR][Lh] + (int64_t)e->cfg.action_dim * e->w_ld[IQL_NET_ACTOR][Lh] : 0;
  c.stamps = e->d_stamps;
  c.xrow_off_ = e->wl.xrow;
  c.xhi_off = (c.tf32 && e->split_first) ? e->wl.xhi : 0;
  c.xlo_off = (c.tf32 && e->split_first) ? e->wl.xlo : 0;
  return c;
}

extern "C" int iql_sync_target(iql_engine* e, int32_t member, void* stream) {
  if (!e || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_sync_target: bad member");
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_sync_target: state not bound");
  const int64_t PQ = e->layout.q_floats, P = e->layout.param_floats;
  CUDA_TRY(e, cudaMemcpyAsync(e->target + member * PQ, e->params + member * P, PQ * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return IQL_OK;
}

extern "C" int iql_bind_replay(iql_engine* e, int32_t member, const float* rows, int64_t capacity, int64_t size) {
  if (!e || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_bind_replay: bad member");
  if (!rows || capacity <= 0 || size < 0 || size > capacity) return fail(e, IQL_ERR_INVALID, "iql_bind_replay: bad rows/capacity/size");
  if ((uintptr_t)rows & 15) return fail(e, IQL_ERR_INVALID, "iql_bind_replay: rows must be 16-byte aligned");
  e->h_replay[member] = ReplayBinding{rows, capacity, size};
  e->replay_dirty = true;
  return IQL_OK;
}

extern "C" int iql_set_replay_size(iql_engine* e, int32_t member, int64_t size) {
  if (!e || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_set_replay_size: bad member");
  if (size < 0 || size > e->h_replay[member].capacity) return fail(e, IQL_ERR_INVALID, "iql_set_replay_size: size out of range");
  e->h_replay[member].size = size;
  e->replay_dirty = true;
  return IQL_OK;
}

extern "C" int iql_load_batch(iql_engine* e, int32_t member, const float* states, const float* actions,
                              const float* rewards, const float* next_states, const float* dones, void* stream) {
  if (!e || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_load_batch: bad member");
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_load_batch: state not bound");
  if (!states || !actions || !rewards || !next_states || !dones) return fail(e, IQL_ERR_INVALID, "iql_load_batch: null batch tensor");
  if (e->h_scalars[member].batch != e->cfg.batch_size)
    return fail(e, IQL_ERR_STATE, "iql_load_batch: the member's batch size (iql_set_batch_sizes) differs from the engine's");
  StepCtx ctx = make_ctx(e);
  float* xrow = e->d_ws_f + (int64_t)member * e->wl.member_floats + e->wl.xrow;
  launch_load_batch(ctx, member, xrow, states, actions, rewards, next_states, dones, (cudaStream_t)stream);
  CUDA_TRY(e, cudaGetLastError());
  e->preloaded[member] = 1;
  return IQL_OK;
}

// The chained backward (bwd_chain.cu) after the output-layer backward: hidden dgrad / wgrad chain and input-layer wgrad,
// plus Adam + Polyak in the wgrad epilogues unless the engine runs it gradient-only.  With `tm`, the work of the launch
// goes to the timer's last slot.
static void launch_chain(iql_engine* e, const StepCtx& ctx, cudaStream_t st, StepTimer* tm) {
  if (tm) {  // operands read once; dZ written; the weight gradients written (gradient-only) or the optimizer state streamed
    double fl = 0, by = 0;
    for (size_t i = 2; i < e->bwd_phases.size(); ++i) {
      const Phase& q = e->bwd_phases[i];
      for (int j = 0; j < q.count; ++j) {
        const GemmProb& g = e->h_probs[q.first + j];
        fl += 2.0 * g.M * g.N * g.K;
        by += 4.0 * ((double)g.M * g.K + (double)g.N * g.K + (q.mode == 1 || e->chain_grads ? (double)g.M * g.N : 0.0));
      }
    }
    if (!e->chain_grads)  // p, m, v in and out + shadows
      by += e->active.size() * 4.0 * ((6.0 + 1.0) * e->layout.param_floats + 3.0 * e->layout.q_floats);
    tm->flops.back() = fl;
    tm->bytes.back() = by;
  }
  BwdChainArgs ca = e->chain_args;
  ca.probs = e->d_probs;
  ca.maps = e->d_maps_chain;
  ca.cmaps = e->d_maps_c;
  ca.keep_grads = e->keep_grads;
  ca.grads_only = e->chain_grads ? 1 : 0;
  ca.params = e->params; ca.exp_avg = e->exp_avg; ca.exp_avg_sq = e->exp_avg_sq; ca.target = e->target; ca.grads = e->grads;
  launch_bwd_chain(ca, ctx, st);
}

// one update step for all members; returns number of launches
// gather: sample + gather this step's rows first.  gather_next: the NEXT step's gather (ctx.k + 1) runs on the side
// stream next to this step's optimizer launch -- nothing after the input-layer weight gradient reads the row
// buffers, the gather is pure latency and the optimizer pure bandwidth -- and the caller passes gather = false for
// that next step.
static int enqueue_step(iql_engine* e, StepCtx& ctx, bool gather, cudaStream_t st_main, StepTimer* tm = nullptr,
                        bool gather_next = false) {
  int launches = 0;
  cudaStream_t st = st_main;  // the stream run_phase launches on (switched to e->side for the wgrad leaves)
  // the math mode only: on a shape outside the tcgen05 kernels (tensor_core_path false) it is still true
  const bool tf32_math = e->cfg.math_mode == IQL_MATH_TF32_TCGEN05;
  const double S_d = (double)e->active.size();
  if (gather) {
    if (tm) tm->mark("gather", 0, 2.0 * S_d * e->cfg.batch_size * e->layout.row.row_floats * 4);
    launch_gather(ctx, e->d_ws_f, e->wl.member_floats, e->wl.xrow, st);
    ++launches;
  }
  const iql_config& c = e->cfg;
  const int B = c.batch_size, H = c.hidden_dim, A = c.action_dim, K0 = c.state_dim + c.action_dim;
  const bool first_ok = first_fwd_skinny_ok(K0);
  const bool first_wgrad_ok = first_wgrad_skinny_ok(B, K0);
  const bool out_ok = out_fwd_skinny_ok(H, A);
  const bool last_ok = last_bwd_skinny_ok(B, A);
  static const bool no_side = dbg_getenv("IQL_B200_NO_SIDE_STREAM") != nullptr;
  const bool loss_recomputed = last_ok && e->bwd_phases.size() >= 2 &&
                               last_bwd_recomputes_loss_grads(H, A, e->bwd_phases[0].count * e->lb_splits, B / e->lb_splits) &&
                               e->bwd_phases[0].kind == PH_LAST_WGRAD && e->bwd_phases[1].kind == PH_LAST_DGRAD &&
                               e->bwd_phases[0].count % 4 == 0;
  bool skip_next = false, skip_colsum = false;
  // the reduction of the row-split output-layer backward (single learners) only feeds the optimizer: it leaves the
  // critical path last_bwd -> dgrad -> ... through the side stream (8 us of a 57 us single-learner step)
  const bool lb_side = tf32_math && !tm && !no_side && e->side != nullptr;
  bool lb_on_side = false;
  auto run_phase = [&](const Phase& ph, const Phase* next, const Phase* next2) {
    if (skip_next) { skip_next = false; return; }
    const GemmProb* pp = e->d_probs + ph.first;
    // Mixed precision: the input layer (observations, K = 11..69) and the output heads run in FP32 on CUDA
    // cores; every hidden-layer GEMM and the first-layer weight gradient run as TF32 tcgen05 GEMMs.  TF32 on the
    // input layer doubles the value-loss error (measured 1.2e-3 -> 2.6e-3) for < 10 % of the step time.
    const bool split = ph.kind == PH_FIRST_FWD && e->split_first;  // 3xTF32: FP32-accurate on tensor cores
    const bool umma = tf32_math && ph.umma_ok && umma_phase_supported(ph.mode, B, H) &&
                      !(ph.kind == PH_FIRST_FWD && !split && first_ok);
    // forward, last hidden layer on the tensor cores: the FP32 output Linear is fused into the epilogue, the next phase skipped
    const bool fuse_out = umma && ph.mode == 0 && ph.epi == EPI_RELU && next && next->kind == PH_OUT_FWD && H == 256 &&
                          umma_can_fuse_out(A);
    if (tm) {  // algorithmic work: 2MNK flops; each operand read once, the output written once
      double fl = 0, by = 0;
      auto add = [&](const Phase& q) {
        for (int i = 0; i < q.count; ++i) {
          const GemmProb& g = e->h_probs[q.first + i];
          fl += 2.0 * g.M * g.N * g.K;
          by += 4.0 * ((double)g.M * g.K + (double)g.N * g.K + (g.no_store ? 0.0 : (double)g.M * g.N) + (g.mask ? (double)g.M * g.N : 0.0));
        }
      };
      add(ph);
      if (fuse_out || (next && ph.kind == PH_LAST_WGRAD && next->kind == PH_LAST_DGRAD)) add(*next);
      static const char* kinds[] = {"gemm", "first_fwd", "out_fwd", "last_bwd", "last_dgrad", "first_wgrad"};
      static const char* modes[] = {"fwd", "dgrad", "wgrad"};
      char nm[32];
      snprintf(nm, sizeof(nm), "%s_%s", ph.kind == PH_GENERIC ? "hidden" : kinds[ph.kind], modes[ph.mode]);
      tm->mark(nm, fl, by);
    }
    if (umma && ph.kind == PH_OUT_FWD) {
      // the heads stay in FP32: TF32 rounding of Q and V would be amplified by adv = q - v and exp(beta * adv)
      if (out_ok) launch_out_fwd(pp, ph.count, B, H, A, st);
      else launch_simt_gemm(ph.mode, pp, ph.count, ph.maxM, ph.maxN, ctx, st);
    } else if (umma && ph.kind != PH_LAST_WGRAD) {
      const int n_scalar = (N_PASS - 1) * (int)e->active.size();  // problems with a scalar head (V, Q passes)
      launch_umma_gemm(ph.mode, pp, split ? e->d_maps_first : e->d_maps + (size_t)256 * ph.first,
                       fuse_out ? e->d_probs + next->first : nullptr, ph.epi, ph.count, ph.maxM, ph.maxN, ctx, st, split,
                       n_scalar, ph.cta2, ph.maxK, ph.rowepi ? e->d_maps_c + (size_t)128 * ph.first : nullptr, ph.tile_n);
      if (fuse_out) {  // the policy head (N = act_dim) stays with the FP32 output-layer kernel
        const GemmProb* pa = e->d_probs + next->first + n_scalar;
        if (out_ok) launch_out_fwd(pa, ph.count - n_scalar, B, H, A, st);
        else launch_simt_gemm(0, pa, ph.count - n_scalar, B, A, ctx, st);
        ++launches;
        skip_next = true;
      }
      if (ph.mode == 1 && umma_dgrad_writes_dbias(B)) skip_colsum = true;  // the dgrad epilogue wrote db of the layer below
      if (ph.mode == 2) {
        if (skip_colsum) skip_colsum = false;  // db already written by the fused output-layer backward
        else { launch_colsum(pp, ph.count, ph.maxM, st); ++launches; }
      }
    } else if (ph.kind == PH_FIRST_FWD && first_ok) {
      launch_first_fwd(pp, ph.count, B, H, K0, ctx, st);
    } else if (ph.kind == PH_OUT_FWD && out_ok) {
      launch_out_fwd(pp, ph.count, B, H, A, st);
    } else if (ph.kind == PH_LAST_WGRAD && last_ok && next && next->kind == PH_LAST_DGRAD) {
      // fused wgrad + dgrad of the output layer; it also emits db_{L-1} when layer L-1 is a hidden-layer
      // tcgen05 wgrad phase (whose kernel does not produce bias gradients)
      const bool emit_db = next2 && tf32_math && next2->umma_ok && umma_phase_supported(2, B, H);
      if (e->lb_splits > 1 && e->bwd_phases.size() >= 3 && ph.first == e->bwd_phases[0].first) {
        const int sp = e->lb_splits, n = ph.count * sp;
        const GemmProb* t0 = e->d_probs + e->lb_first;
        launches += launch_last_bwd(t0, t0 + n, emit_db ? t0 + 2 * n : nullptr, n, B / sp, H, A, ctx, st,
                                    loss_recomputed ? e->d_ws_f : nullptr, e->wl.member_floats, &e->wl, e->params);
        if (lb_side) {
          cudaEventRecord(e->ev_fork, st_main);
          cudaStreamWaitEvent(e->side, e->ev_fork, 0);
          launch_lb_reduce(t0 + n, emit_db ? t0 + 2 * n : nullptr, pp, emit_db ? e->d_probs + next2->first : nullptr, ph.count, sp, e->side);
          cudaEventRecord(e->ev_side, e->side);
          lb_on_side = true;
        } else {
          launch_lb_reduce(t0 + n, emit_db ? t0 + 2 * n : nullptr, pp, emit_db ? e->d_probs + next2->first : nullptr, ph.count, sp, st);
        }
      } else
      launches += -1 + launch_last_bwd(e->d_probs + next->first, pp, emit_db ? e->d_probs + next2->first : nullptr, ph.count, B, H, A, ctx, st,
                      loss_recomputed ? e->d_ws_f : nullptr, e->wl.member_floats, &e->wl, e->params);
      skip_next = true;
      skip_colsum = emit_db;
    } else if (ph.kind == PH_FIRST_WGRAD && first_wgrad_ok) {
      launch_first_wgrad(pp, ph.count, B, H, K0, st);
    } else {
      launch_simt_gemm(ph.mode, pp, ph.count, ph.maxM, ph.maxN, ctx, st);
    }
    ++launches;
  };
  if (tf32_math && e->fused_fwd) {
    // one launch for layers 0..L-1 + scalar heads; the policy head (N = act_dim) stays with the FP32 output kernel
    const int L = c.n_hidden;
    const int n_scalar = (N_PASS - 1) * (int)e->active.size();
    const Phase& pout = e->fwd_phases[L];
    FusedFwdArgs fa;
    memset(&fa, 0, sizeof(fa));
    for (int l = 0; l < L; ++l) {
      fa.probs[l] = e->d_probs + e->fwd_phases[l].first;
      fa.maps[l] = (l == 0) ? (const void*)e->d_maps_first : (const void*)(e->d_maps + (size_t)256 * e->fwd_phases[l].first);
      fa.store_maps[l] = e->d_maps_store + (size_t)128 * l * e->fwd_phases[0].count;
    }
    fa.probs_out = e->d_probs + pout.first;
    fa.pair = e->fused_pair ? 1 : 0;
    const bool pol_fused = fused_fwd_policy_head(A);
    fa.fuse_policy = pol_fused ? 1 : 0;
    fa.L = L; fa.nprob = e->fwd_phases[0].count; fa.batch = B; fa.fuse_count = n_scalar; fa.k0_max = e->fwd_phases[0].maxK;
    if (tm) {  // operands read once, the activations of the training passes written once
      double fl = 0, by = 0;
      for (int l = 0; l <= L; ++l) {
        const Phase& q = e->fwd_phases[l];
        for (int i = 0; i < q.count; ++i) {
          const GemmProb& g = e->h_probs[q.first + i];
          const bool kept = e->h_probs[e->fwd_phases[L - 1].first + i].no_store == 0;
          fl += 2.0 * g.M * g.N * g.K * (l == 0 ? 3.0 : 1.0);
          if (l == L && i >= n_scalar && !pol_fused) { fl -= 2.0 * g.M * g.N * g.K; continue; }  // policy head: its own launch
          by += 4.0 * ((l == 0 ? (double)g.M * g.K : 0.0) + (double)g.N * g.K + ((l == L || kept) ? (double)g.M * g.N : 0.0));
        }
      }
      tm->mark("fused_fwd", fl, by);
    }
    launch_fused_fwd(fa, ctx, st);
    ++launches;
    const GemmProb* pa = e->d_probs + pout.first + n_scalar;
    if (!pol_fused) {
    if (tm) {
      double fl = 0, by = 0;
      for (int i = n_scalar; i < pout.count; ++i) {
        const GemmProb& g = e->h_probs[pout.first + i];
        fl += 2.0 * g.M * g.N * g.K;
        by += 4.0 * ((double)g.M * g.K + (double)g.N * g.K + (double)g.M * g.N);
      }
      tm->mark("policy_head", fl, by);
    }
    if (e->pol_umma)
      launch_umma_gemm(0, pa, e->d_maps_pol, nullptr, EPI_LINEAR, pout.count - n_scalar, B, A, ctx, st, 2, 0, false, H);
    else if (out_ok) launch_out_fwd(pa, pout.count - n_scalar, B, H, A, st);
    else launch_simt_gemm(0, pa, pout.count - n_scalar, B, A, ctx, st);
    ++launches;
    }
  } else {
    for (size_t i = 0; i < e->fwd_phases.size(); ++i)
      run_phase(e->fwd_phases[i], i + 1 < e->fwd_phases.size() ? &e->fwd_phases[i + 1] : nullptr, nullptr);
  }
  // The output-layer backward derives the loss gradients of its rows itself, so loss_kernel (logged losses, log_std
  // gradient, Adam scalars of the step: all needed by the optimizer launch only) leaves the critical path and
  // runs on the side stream next to the backward.
  const bool loss_on_side = loss_recomputed && !tm && !no_side && e->side != nullptr;
  if (tm) tm->mark("loss", 0, S_d * e->cfg.batch_size * 4.0 * (8 + 3 * e->wl.Ald));
  if (loss_on_side) {
    cudaEventRecord(e->ev_fork, st_main);
    cudaStreamWaitEvent(e->side, e->ev_fork, 0);
    launch_loss(ctx, e->d_ws_f, e->wl.member_floats, e->wl, e->params, e->grads, e->side);
    cudaEventRecord(e->ev_side, e->side);
  } else {
    launch_loss(ctx, e->d_ws_f, e->wl.member_floats, e->wl, e->params, e->grads, st);
  }
  ++launches;
  // per-kernel timing (tm) keeps everything on one stream
  const bool two_streams = tf32_math && !tm && !no_side && e->side != nullptr;
  int forks = 0;
  // chained backward: the output-layer backward (phases 0, 1) runs as before, everything after it -- hidden dgrad /
  // wgrad chain, input-layer wgrad (+ Adam + Polyak unless gradient-only) -- is ONE launch on CTA pairs.  Bind time set
  // e->chain only for shapes it serves (tf32, skinny output-layer backward, 2L + 1 phases), so what it reports runs.
  const bool chain = e->chain;
  for (size_t i = 0; i < e->bwd_phases.size(); ++i) {
    if (chain && i >= 2) break;
    const Phase& ph = e->bwd_phases[i];
    const Phase* n1 = i + 1 < e->bwd_phases.size() ? &e->bwd_phases[i + 1] : nullptr;
    const Phase* n2 = i + 2 < e->bwd_phases.size() ? &e->bwd_phases[i + 2] : nullptr;
    const bool leaf = two_streams && ph.mode == 2 && ph.kind == PH_GENERIC && ph.umma_ok &&
                      umma_phase_supported(2, B, H) && !skip_next;
    if (ph.kind == PH_FIRST_WGRAD && e->fw_splits > 1 && tf32_math && ph.umma_ok && umma_phase_supported(2, B, H) && !skip_next) {
      // few problems x a long batch: the tcgen05 kernel runs the K-split copies (enough tiles to fill the GPU), then the
      // partial dW_0 / db_0 are added up in split order
      run_phase(e->fw_phase, nullptr, nullptr);  // batch > 256: the phase also runs colsum_kernel (partial db_0)
      launch_lb_reduce(e->d_probs + e->fw_phase.first, nullptr, e->d_probs + ph.first, nullptr, ph.count, e->fw_splits, st);
      ++launches;
      continue;
    }
    if (leaf) {
      // G_l (written by the previous launch) -> side stream.  The previous leaf must be done first: the dgrad that
      // follows on the main stream overwrites the ping-pong buffer that leaf was reading.
      if (forks > 0) cudaStreamWaitEvent(st_main, e->ev_side, 0);
      cudaEventRecord(e->ev_fork, st_main);
      cudaStreamWaitEvent(e->side, e->ev_fork, 0);
      st = e->side;
      run_phase(ph, n1, n2);
      st = st_main;
      cudaEventRecord(e->ev_side, e->side);
      ++forks;
    } else {
      run_phase(ph, n1, n2);
    }
  }
  // chained backward (gradients only): the chain reads nothing the side stream writes (loss kernel: logged losses,
  // log_std gradient, Adam scalars; row-split reduction: dW_L, db_L), so it starts right after the output-layer backward
  if (chain && e->chain_grads) {
    if (tm) tm->mark("bwd_chain_grads", 0, 0);
    launch_chain(e, ctx, st, tm);
    ++launches;
  }
  if (forks > 0 || loss_on_side || lb_on_side) cudaStreamWaitEvent(st_main, e->ev_side, 0);  // join before the optimizer
  // Adam: read g, p, m, v + target; write p, m, v + target (+ the TF32 shadow copies in tcgen05 mode)
  if (tm) {
    // TF32 operand copies the optimizer maintains: everything except the hidden-layer weights when those carry the
    // rounding bias in place (no shadow), plus the lo parts of the first-layer (and wide policy-head) ranges
    double shadow_p = 0, shadow_t = 0;
    if (ctx.tf32) {
      double hid_p = 0, hid_q = 0, lo_p = 0, lo_q = 0;
      for (int i = 0; i < ctx.n_hid; ++i) {
        hid_p += (double)(ctx.hid_end[i] - ctx.hid_begin[i]);
        if (ctx.hid_begin[i] < ctx.PQ) hid_q += (double)(ctx.hid_end[i] - ctx.hid_begin[i]);
      }
      for (int r = 0; r < 5; ++r) {
        lo_p += (double)(ctx.first_w_end[r] - ctx.first_w_begin[r]);
        if (ctx.first_w_begin[r] < ctx.PQ) lo_q += (double)(ctx.first_w_end[r] - ctx.first_w_begin[r]);
      }
      shadow_p = (double)e->layout.param_floats - hid_p + lo_p;
      shadow_t = (double)e->layout.q_floats - hid_q + lo_q;
    }
    tm->mark("adam_polyak", 0, S_d * 4.0 * (7.0 * e->layout.param_floats + 2.0 * e->layout.q_floats + shadow_p + shadow_t));
  }
  // (chained backward + optimizer: its input-layer weight-gradient phase still reads the gathered rows, so the next
  // step's gather cannot run beside it; the caller then gathers at the top of every step)
  const bool fork_gather = gather_next && !tm && e->side != nullptr && !(chain && !e->chain_grads);
  if (fork_gather) {
    StepCtx next = ctx;
    next.k = ctx.k + 1;
    cudaEventRecord(e->ev_fork_g, st_main);
    cudaStreamWaitEvent(e->side, e->ev_fork_g, 0);
    launch_gather(next, e->d_ws_f, e->wl.member_floats, e->wl.xrow, e->side);
    cudaEventRecord(e->ev_gather, e->side);
    ++launches;
  }
  ctx.unbias_out = (ctx.k == ctx.K - 1) ? 1 : 0;  // the call's last optimizer launch leaves plain fp32 in the arenas
  if (chain && !e->chain_grads) {
    if (tm) tm->label.back() = "bwd_chain";
    launch_chain(e, ctx, st, tm);
  } else {
    launch_adam(ctx, e->params, e->exp_avg, e->exp_avg_sq, e->target, e->grads, st);
    if (ctx.advance_k > 0) ctx.advance_k = -1;  // consumed: the optimizer launch advanced the counters
  }
  ++launches;
  if (fork_gather) cudaStreamWaitEvent(st_main, e->ev_gather, 0);
  if (tm) tm->finish();
  return launches;
}

// Launch the graph cached under `key` on `run`.  On a miss, `body` (enqueues the launches on `capture`, returns how many)
// is captured into a new graph first.  *launches receives the graph's launch count.
template <class Body>
static int launch_graph(iql_engine* e, const GraphKey& key, cudaStream_t capture, cudaStream_t run, const char* who, Body&& body,
                        int64_t* launches) {
  auto it = e->graphs.find(key);
  if (it == e->graphs.end()) {
    cudaGraph_t graph = nullptr;
    CUDA_TRY(e, cudaStreamBeginCapture(capture, cudaStreamCaptureModeThreadLocal));
    const int64_t n = body();
    cudaError_t cerr = cudaStreamEndCapture(capture, &graph);
    if (cerr != cudaSuccess) return fail(e, IQL_ERR_CUDA, std::string(who) + ": graph capture: " + cudaGetErrorString(cerr));
    cudaGraphExec_t exec = nullptr;
    CUDA_TRY(e, cudaGraphInstantiate(&exec, graph, 0));
    cudaGraphDestroy(graph);
    it = e->graphs.emplace(key, std::make_pair(exec, n)).first;
  }
  CUDA_TRY(e, cudaGraphLaunch(it->second.first, run));
  *launches = it->second.second;
  return IQL_OK;
}

// The host shadow of the counters moves with the device copy: a call of k steps advances every member that trained
static void advance_counters(iql_engine* e, int k) {
  for (const int m : e->active) {
    iql_counters& c = e->h_counters[m];
    c.v_step += k; c.q_step += k; c.actor_step += k; c.total_it += k; c.sample_step += k;
    if (e->h_hparams[m].cosine_t_max > 0) c.sched_epoch += k;
  }
}

extern "C" int iql_train_steps(iql_engine* e, int32_t k_steps, int32_t sample_mode, const int64_t* indices,
                               const uint8_t* dropout_masks, float* out_losses, int64_t* idx_out, void* stream) {
  if (!e) return IQL_ERR_INVALID;
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_train_steps: state not bound");
  if (k_steps <= 0 || k_steps > e->cfg.max_steps_per_call) return fail(e, IQL_ERR_INVALID, "iql_train_steps: k_steps out of range");
  const int S = e->cfg.n_members;
  cudaStream_t st = (cudaStream_t)stream;
  if (sample_mode == IQL_SAMPLE_INDICES) {
    if (!indices) return fail(e, IQL_ERR_INVALID, "iql_train_steps: IQL_SAMPLE_INDICES needs indices");
  } else if (sample_mode == IQL_SAMPLE_PRELOADED) {
    if (k_steps != 1) return fail(e, IQL_ERR_INVALID, "iql_train_steps: IQL_SAMPLE_PRELOADED runs exactly one step");
    for (const int m : e->active)
      if (!e->preloaded[m]) return fail(e, IQL_ERR_STATE, "iql_train_steps: no batch staged (call iql_load_batch)");
  } else if (sample_mode != IQL_SAMPLE_PHILOX) {
    return fail(e, IQL_ERR_INVALID, "iql_train_steps: unknown sample_mode");
  }
  if (sample_mode != IQL_SAMPLE_PRELOADED)
    for (const int m : e->active) {
      if (!e->h_replay[m].rows) return fail(e, IQL_ERR_STATE, "iql_train_steps: replay buffer not bound");
      if (e->h_replay[m].size <= 0 && sample_mode == IQL_SAMPLE_PHILOX)
        return fail(e, IQL_ERR_INVALID, "iql_train_steps: cannot sample from an empty replay buffer");
    }
  int rc = flush_tables(e, st);
  if (rc != IQL_OK) return rc;

  StepCtx ctx = make_ctx(e);
  ctx.K = k_steps;
  if (ctx.tf32) launch_refresh_shadow(ctx, e->params, e->target, st);
  ctx.indices = (sample_mode == IQL_SAMPLE_INDICES) ? indices : nullptr;
  ctx.dropout_masks = dropout_masks;
  ctx.idx_out = idx_out;
  const bool gather = sample_mode != IQL_SAMPLE_PRELOADED;
  static const bool no_overlap_gather = dbg_getenv("IQL_B200_NO_GATHER_AHEAD") != nullptr || dbg_getenv("IQL_B200_NO_SIDE_STREAM") != nullptr;
  // (not with the chained backward + optimizer: its last phase still reads the gathered rows, see enqueue_step)
  const bool overlap_gather = !no_overlap_gather && e->side != nullptr && st != nullptr && !(e->chain && !e->chain_grads);
  auto k_step_loop = [&]() -> int64_t {
    int64_t n = 0;
    for (int k = 0; k < k_steps; ++k) {
      ctx.k = k;
      if (k == k_steps - 1) ctx.advance_k = k_steps;
      const bool ahead = gather && overlap_gather && k + 1 < k_steps;  // step k+1's gather rides along step k's optimizer
      n += enqueue_step(e, ctx, gather && (k == 0 || !overlap_gather), st, nullptr, ahead);
    }
    if (ctx.advance_k != -1) { launch_advance(ctx, k_steps, st); ++n; }
    return n;
  };
  // the legacy default stream cannot be captured; the facade runs the engine on its own stream
  // Graphs: the K-step Philox loop, and the single preloaded step of the drop-in `train(batch)` path (its ~11
  // launches would otherwise be launch-latency bound).  Keyed by sample mode and K.
  // (the index pointer is baked into the captured kernels, so the INDICES variant is keyed by it: callers that
  // reuse one staging buffer -- the Python facade does -- replay one graph; at most 16 graphs are kept)
  const bool graphable = e->use_graphs && st != nullptr && !dropout_masks && !idx_out &&
                         (k_steps > 1 || sample_mode == IQL_SAMPLE_PRELOADED);
  const GraphKey graph_key((int)sample_mode, (int)k_steps, sample_mode == IQL_SAMPLE_INDICES ? (uintptr_t)indices : (uintptr_t)0);
  if (graphable && e->graphs.size() >= 16 && e->graphs.find(graph_key) == e->graphs.end()) drop_graphs(e);
  int64_t launches = 0;
  if (graphable) {
    rc = launch_graph(e, graph_key, st, st, "iql_train_steps", k_step_loop, &launches);
    if (rc != IQL_OK) return rc;
  } else {
    launches = k_step_loop();
  }
  CUDA_TRY(e, cudaGetLastError());
  advance_counters(e, k_steps);
  for (const int m : e->active) e->preloaded[m] = 0;
  if (idx_out)  // the gather writes the rows of the members that trained; the others read -1 (all-ones bytes)
    for (int m = 0; m < S; ++m)
      if (!e->is_active[m])
        CUDA_TRY(e, cudaMemsetAsync(idx_out + (size_t)m * k_steps * e->cfg.batch_size, 0xFF,
                                    sizeof(int64_t) * (size_t)k_steps * e->cfg.batch_size, st));
  if (out_losses) {
    const size_t row = sizeof(float) * 3 * (size_t)k_steps;
    CUDA_TRY(e, cudaMemcpy2DAsync(out_losses, row, e->d_loss_ring, sizeof(float) * 3 * (size_t)e->cfg.max_steps_per_call, row, S,
                                  cudaMemcpyDeviceToDevice, st));
  }
  e->last_launches = launches;
  return IQL_OK;
}

// ---------------------------------------------------------------------------
// Host-driven single step: the reference's loop `batch = rb.sample(B); log = trainer.train(batch)`
// (algorithms/offline/iql.py:631-635, finetune/iql.py:542-563) returns the three losses to the host every step.
// One call = one CUDA graph launch (TF32 operand refresh, gather of the host-drawn indices read straight from
// pinned memory, the whole step, counter advance).  The loss kernel stores its scalars into device-mapped pinned
// memory and raises a flag word; this function spins on that word and returns as soon as the losses of the step are on
// the host -- while the step's backward and optimizer launches are still running, so the caller's host work for the
// next step (index draw, Python) overlaps them.
// ---------------------------------------------------------------------------
// Pinned, device-mapped host block of the host-driven entry points (kernels read and write it at its host address),
// allocated zeroed on first use together with ev_in, the event order_behind_host_step records.
static int pinned_block(iql_engine* e, void** block, size_t bytes, const char* who) {
  if (*block) return IQL_OK;
  if ((!e->ev_in && cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming) != cudaSuccess) ||
      cudaHostAlloc(block, bytes, cudaHostAllocMapped) != cudaSuccess) {
    cudaGetLastError();
    *block = nullptr;
    return fail(e, IQL_ERR_CUDA, std::string(who) + ": pinned block / event allocation failed");
  }
  memset(*block, 0, bytes);
  return IQL_OK;
}

// The caller's stream waits for the stream of the last host step when the two differ
static int order_behind_host_step(iql_engine* e, cudaStream_t cur) {
  if (e->host_step_stream_set && e->host_step_stream != cur) {
    CUDA_TRY(e, cudaEventRecord(e->ev_in, e->host_step_stream));
    CUDA_TRY(e, cudaStreamWaitEvent(cur, e->ev_in, 0));
  }
  return IQL_OK;
}

// Spin until the device has raised `flag` (pinned host memory); bounded, and a failed launch is noticed through the stream.
static int spin_flag(iql_engine* e, volatile uint32_t* flag, cudaStream_t st, const char* who) {
  const auto t0 = std::chrono::steady_clock::now();
  uint32_t spins = 0;
  while (*flag == 0u) {
    if ((++spins & 0x3FFFu) == 0u) {
      const cudaError_t q = cudaStreamQuery(st);
      if (q == cudaSuccess) {
        if (*flag == 0u) return fail(e, IQL_ERR_CUDA, std::string(who) + ": the launch finished without reporting its result");
        break;
      }
      if (q != cudaErrorNotReady) return fail(e, IQL_ERR_CUDA, std::string(who) + ": " + cudaGetErrorString(q));
      if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(20))
        return fail(e, IQL_ERR_CUDA, std::string(who) + ": timed out waiting for the device");
    }
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  return IQL_OK;
}

extern "C" int iql_host_step_wait(iql_engine* e, float* host_losses, void* stream);

// Collect a host step still in flight (its losses are dropped), so that its flag words and index block can be reused
static int collect_host_step(iql_engine* e) {
  if (!e->mail_pending) return IQL_OK;
  std::vector<float> sink(3 * (size_t)e->cfg.n_members);
  return iql_host_step_wait(e, sink.data(), e->host_step_stream);
}

extern "C" int iql_train_host_step(iql_engine* e, const int64_t* host_indices, float* host_losses, void* stream,
                                   void* caller_stream) {
  if (!e) return IQL_ERR_INVALID;
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_train_host_step: state not bound");
  cudaStream_t st = (cudaStream_t)stream, cur = (cudaStream_t)caller_stream;
  if (!st) return fail(e, IQL_ERR_INVALID, "iql_train_host_step: needs a non-default stream (graph capture)");
  const int S = e->cfg.n_members, B = e->cfg.batch_size;
  const bool gather = host_indices != nullptr;
  for (const int m : e->active) {
    if (gather && !e->h_replay[m].rows) return fail(e, IQL_ERR_STATE, "iql_train_host_step: replay buffer not bound");
    if (!gather && !e->preloaded[m]) return fail(e, IQL_ERR_STATE, "iql_train_host_step: no batch staged (call iql_load_batch)");
  }
  const size_t idx_bytes = sizeof(int64_t) * (size_t)S * B;
  int rc = pinned_block(e, (void**)&e->h_mail, idx_bytes + sizeof(float) * 4 * S, "iql_train_host_step");
  if (rc != IQL_OK) return rc;
  int64_t* mail_idx = (int64_t*)e->h_mail;
  float* mail = (float*)(e->h_mail + idx_bytes);
  rc = collect_host_step(e);  // one step in flight at a time: its gather may not have read the index block yet
  if (rc != IQL_OK) return rc;
  if (gather)
    for (const int m : e->active) {  // rows of members that do not train are never read
      const int64_t cap = e->h_replay[m].capacity;
      for (int b = 0; b < e->h_scalars[m].batch; ++b) {  // entries past B_m are never read
        const int64_t i = host_indices[(size_t)m * B + b];
        if (i < 0 || i >= cap) return fail(e, IQL_ERR_INVALID, "iql_train_host_step: index outside the bound replay buffer");
        mail_idx[(size_t)m * B + b] = i;
      }
    }
  for (const int m : e->active) reinterpret_cast<volatile uint32_t*>(mail)[m * 4 + 3] = 0u;
  std::atomic_thread_fence(std::memory_order_seq_cst);
  // The graph is captured on `stream` (capture needs a non-default stream) but LAUNCHED on the caller's stream: the
  // step is then ordered against everything the caller enqueues (inserted rows, a staged batch, later reads of the
  // weights) by plain stream order -- no event record / wait pairs around every step.  Other engine calls order their
  // stream against the caller's (iql_act_host, the Python guard around iql_train_steps).  A caller that hops between
  // streams gets the two ordered by an event.
  cudaStream_t run = cur;
  rc = order_behind_host_step(e, run);
  if (rc != IQL_OK) return rc;
  e->host_step_stream = run;
  e->host_step_stream_set = true;
  rc = flush_tables(e, run);
  if (rc != IQL_OK) return rc;
  auto one_step = [&]() -> int64_t {
    StepCtx ctx = make_ctx(e);
    ctx.K = 1;
    ctx.k = 0;
    ctx.indices = gather ? mail_idx : nullptr;  // unified addressing: the pinned block is device-visible at its host address
    ctx.host_mail = mail;
    int64_t n = 0;
    // the TF32 operand refresh and the gather are independent: one launch, which releases the forward at once
    const bool fork_refresh = ctx.tf32 && gather;
    if (fork_refresh) {
      launch_gather_refresh(ctx, e->d_ws_f, e->wl.member_floats, e->wl.xrow, e->params, e->target, st);
      ++n;
    } else if (ctx.tf32) {
      launch_refresh_shadow(ctx, e->params, e->target, st);
      ++n;
    }
    ctx.advance_k = 1;
    n += enqueue_step(e, ctx, gather && !fork_refresh, st, nullptr, false);
    if (ctx.advance_k != -1) { launch_advance(ctx, 1, st); ++n; }
    return n;
  };
  rc = launch_graph(e, GraphKey(gather ? 101 : 102, 1, 0), st, run, "iql_train_host_step", one_step, &e->last_launches);
  if (rc != IQL_OK) return rc;
  advance_counters(e, 1);
  for (const int m : e->active) e->preloaded[m] = 0;
  e->mail_pending = true;
  if (!host_losses) return IQL_OK;  // the caller collects the losses with iql_host_step_wait
  return iql_host_step_wait(e, host_losses, run);
}

extern "C" int iql_host_step_wait(iql_engine* e, float* host_losses, void* stream) {
  if (!e || !host_losses) return IQL_ERR_INVALID;
  if (!e->h_mail || !e->mail_pending) return fail(e, IQL_ERR_STATE, "iql_host_step_wait: no host step in flight");
  e->mail_pending = false;
  (void)stream;
  cudaStream_t st = e->host_step_stream;  // the stream the step was launched on (a failed launch is noticed through it)
  const int S = e->cfg.n_members, B = e->cfg.batch_size;
  float* mail = (float*)(e->h_mail + sizeof(int64_t) * (size_t)S * B);
  // wait for the flag words of the members the step trained (bounded: a failed launch never raises them); the active
  // set cannot have changed since the launch, iql_set_active_members collects a pending step first
  for (const int m : e->active) {
    int rc = spin_flag(e, reinterpret_cast<volatile uint32_t*>(mail) + m * 4 + 3, st, "iql_host_step_wait");
    if (rc != IQL_OK) return rc;
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  for (int m = 0; m < S; ++m)
    for (int j = 0; j < 3; ++j)
      host_losses[m * 3 + j] = e->is_active[m] ? reinterpret_cast<volatile float*>(mail)[m * 4 + j] : NAN;
  return IQL_OK;
}

// Members that train.  The problem tables, tensor maps and chain tasks are rebuilt over the active members only, so the
// others launch no CTA and their arena rows, counters and batch sizes stay as they are; the path choices that depend on
// the member count are re-made from the new count.  Host work (tensor-map encoding), paid once per change.
extern "C" int iql_set_active_members(iql_engine* e, int32_t n, const int32_t* host_ids) {
  if (!e) return IQL_ERR_INVALID;
  const int S = e->cfg.n_members;
  if (!host_ids || n <= 0) return fail(e, IQL_ERR_INVALID, "iql_set_active_members: need at least one member id");
  std::vector<char> mask(S, 0);
  for (int i = 0; i < n; ++i) {
    const int32_t m = host_ids[i];
    if (m < 0 || m >= S) return fail(e, IQL_ERR_INVALID, "iql_set_active_members: member " + std::to_string(m) + " out of range");
    if (mask[m]) return fail(e, IQL_ERR_INVALID, "iql_set_active_members: member " + std::to_string(m) + " listed twice");
    mask[m] = 1;
  }
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_set_active_members: state not bound");
  int rc = collect_host_step(e);  // the in-flight host step's flag words belong to the old set
  if (rc != IQL_OK) return rc;
  const std::vector<int32_t> old = e->active;
  e->active.clear();
  for (int m = 0; m < S; ++m)
    if (mask[m]) e->active.push_back(m);
  rc = bind_tables(e);
  if (rc != IQL_OK) {  // cannot happen for a set the old tables were built for; restore it anyway
    e->active = old;
    bind_tables(e);
    return rc;
  }
  e->is_active = mask;
  e->tables_dirty = true;
  drop_graphs(e);  // the tables' sizes are baked into the launches
  return IQL_OK;
}

extern "C" int iql_get_active_members(iql_engine* e, int8_t* host_mask) {
  if (!e || !host_mask) return fail(e, IQL_ERR_INVALID, "iql_get_active_members: null argument");
  for (int m = 0; m < e->cfg.n_members; ++m) host_mask[m] = e->is_active[m];
  return IQL_OK;
}

// IQL_STEP_TRACE=1 (debug): reset / read the step timeline.  reset != 0 arms the slots (min = ~0, max = 0) on `stream`;
// otherwise synchronises the device and copies [ST_COUNT][2] globaltimer stamps (ns) to `out`.
extern "C" int iql_debug_step_trace(iql_engine* e, int32_t reset, unsigned long long* out, int32_t max_words, void* stream) {
  if (!e || !e->d_stamps) return -1;
  if (reset) {
    std::vector<unsigned long long> init(2 * ST_COUNT);
    for (int i = 0; i < ST_COUNT; ++i) { init[2 * i] = ~0ull; init[2 * i + 1] = 0ull; }
    if (cudaMemcpyAsync(e->d_stamps, init.data(), sizeof(unsigned long long) * init.size(), cudaMemcpyHostToDevice, (cudaStream_t)stream) != cudaSuccess ||
        cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess)
      return -2;
    return 0;
  }
  if (!out || max_words < 2 * ST_COUNT) return -1;
  if (cudaDeviceSynchronize() != cudaSuccess) return -2;
  if (cudaMemcpy(out, e->d_stamps, sizeof(unsigned long long) * 2 * ST_COUNT, cudaMemcpyDeviceToHost) != cudaSuccess) return -2;
  return 2 * ST_COUNT;
}

extern "C" int64_t iql_last_launch_count(const iql_engine* e) { return e ? e->last_launches : 0; }

extern "C" int iql_act(iql_engine* e, int32_t member, const float* states, int64_t n, float max_action,
                       float* out_actions, void* stream) {
  if (!e || member < -1 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_act: bad member");
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_act: state not bound");
  if (!states || !out_actions || n < 0) return fail(e, IQL_ERR_INVALID, "iql_act: null or negative n");
  if (n == 0) return IQL_OK;
  int rc = flush_tables(e, (cudaStream_t)stream);
  if (rc != IQL_OK) return rc;
  StepCtx ctx = make_ctx(e);
  const int L = e->cfg.n_hidden;
  // member == -1: all members at once, states [S][n][state_dim] -> actions [S][n][action_dim]
  const int first = member < 0 ? 0 : member, count = member < 0 ? e->cfg.n_members : 1;
  launch_act(ctx, e->params + (int64_t)first * e->layout.param_floats, count, e->d_act_off, e->d_act_off + (L + 1), states,
             n, max_action, out_actions, (cudaStream_t)stream);
  CUDA_TRY(e, cudaGetLastError());
  return IQL_OK;
}

// One env step of policy.act for a HOST caller (iql.py:371-379, 403-413; the rollout loops eval_actor iql.py:218-238 and
// jsrl_w_iql.py:445-515 call it once per env step): the observation rides in the kernel parameters, the action comes
// back through device-mapped pinned memory with a flag word the host spins on -- one launch, no copies, no stream
// synchronisation.  Ordered after everything queued on `stream` (the last update) and on `caller_stream`.
static int act_host_impl(iql_engine* e, int32_t member, const float* host_state, float max_action, float* host_action,
                         float* host_std, void* stream, void* caller_stream);

extern "C" int iql_act_host(iql_engine* e, int32_t member, const float* host_state, float max_action, float* host_action,
                            void* stream, void* caller_stream) {
  return act_host_impl(e, member, host_state, max_action, host_action, nullptr, stream, caller_stream);
}

// Training-mode GaussianPolicy.act (iql.py:371-379: `dist.sample()`): the kernel returns the distribution's parameters --
// mean = tanh(MLP(s)) (unscaled) and std = exp(clamp(log_std, -20, 2)) -- and the caller draws the sample on the host.
extern "C" int iql_act_host_gaussian(iql_engine* e, int32_t member, const float* host_state, float* host_mean, float* host_std,
                                     void* stream, void* caller_stream) {
  if (e && e->cfg.deterministic) return fail(e, IQL_ERR_INVALID, "iql_act_host_gaussian: the policy is deterministic");
  if (!host_std) return fail(e, IQL_ERR_INVALID, "iql_act_host_gaussian: null std");
  return act_host_impl(e, member, host_state, 1.0f, host_mean, host_std, stream, caller_stream);
}

static int act_host_impl(iql_engine* e, int32_t member, const float* host_state, float max_action, float* host_action,
                         float* host_std, void* stream, void* caller_stream) {
  if (!e || member < 0 || member >= e->cfg.n_members) return fail(e, IQL_ERR_INVALID, "iql_act_host: bad member");
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_act_host: state not bound");
  if (!host_state || !host_action) return fail(e, IQL_ERR_INVALID, "iql_act_host: null state or action");
  if (e->cfg.state_dim > act_host_state_max()) return fail(e, IQL_ERR_INVALID, "iql_act_host: state_dim too large for the by-value path (use iql_act)");
  cudaStream_t st = (cudaStream_t)stream, cur = (cudaStream_t)caller_stream;
  const int A = e->cfg.action_dim, L = e->cfg.n_hidden;
  int rc = pinned_block(e, (void**)&e->h_act, sizeof(float) * (2 * A + 1), "iql_act_host");
  if (rc != IQL_OK) return rc;
  volatile uint32_t* flag = reinterpret_cast<volatile uint32_t*>(e->h_act + 2 * A);
  *flag = 0u;
  std::atomic_thread_fence(std::memory_order_seq_cst);
  // launched on the caller's stream, like the host step: ordered behind the last update by stream order (a K-step call
  // on the engine's stream is ordered against the caller's stream by the Python guard around iql_train_steps)
  (void)st;
  rc = order_behind_host_step(e, cur);
  if (rc != IQL_OK) return rc;
  rc = flush_tables(e, cur);
  if (rc != IQL_OK) return rc;
  StepCtx ctx = make_ctx(e);
  const float* block = e->params + (int64_t)member * e->layout.param_floats;
  launch_act_host(ctx, block, e->d_act_off, e->d_act_off + (L + 1), host_state, max_action,
                  (host_std && !e->cfg.deterministic) ? block + e->log_std_off : nullptr, e->h_act, cur);
  CUDA_TRY(e, cudaGetLastError());
  rc = spin_flag(e, flag, cur, "iql_act_host");
  if (rc != IQL_OK) return rc;
  for (int i = 0; i < A; ++i) host_action[i] = reinterpret_cast<volatile float*>(e->h_act)[i];
  if (host_std)
    for (int i = 0; i < A; ++i) host_std[i] = reinterpret_cast<volatile float*>(e->h_act)[A + i];
  return IQL_OK;
}

// ---------------------------------------------------------------------------
// Online phase of an ensemble: one act launch and one ring-insert launch per env step for all members
// ---------------------------------------------------------------------------
static size_t align16(size_t n) { return (n + 15) & ~(size_t)15; }

extern "C" int iql_bind_guide(iql_engine* e, const float* guide_params) {
  if (!e) return IQL_ERR_INVALID;
  if ((uintptr_t)guide_params & 15) return fail(e, IQL_ERR_INVALID, "iql_bind_guide: the guide arena must be 16-byte aligned");
  e->guide = guide_params;
  return IQL_OK;
}

extern "C" int iql_act_host_members(iql_engine* e, const float* host_states, const int8_t* host_source, float max_action,
                                    float* host_out, float* host_std, void* stream, void* caller_stream) {
  if (!e) return IQL_ERR_INVALID;
  if (!host_states || !host_source || !host_out) return fail(e, IQL_ERR_INVALID, "iql_act_host_members: null states, sources or output");
  const int S = e->cfg.n_members, Sd = e->cfg.state_dim, A = e->cfg.action_dim, L = e->cfg.n_hidden;
  int n = 0;
  for (int m = 0; m < S; ++m) {
    const int c = host_source[m];
    if (c < IQL_ACT_SKIP || c > IQL_ACT_LEARNER_DIST_DROPOUT)
      return fail(e, IQL_ERR_INVALID, "iql_act_host_members: unknown source code " + std::to_string(c));
    if (c == IQL_ACT_GUIDE && !e->guide) return fail(e, IQL_ERR_INVALID, "iql_act_host_members: a member asks for its guide, but no guide is bound (iql_bind_guide)");
    const bool dist = c == IQL_ACT_LEARNER_DIST || c == IQL_ACT_LEARNER_DIST_DROPOUT;
    if (dist && e->cfg.deterministic)
      return fail(e, IQL_ERR_INVALID, "iql_act_host_members: the distribution code needs a Gaussian policy; this one is deterministic");
    if (dist && !host_std) return fail(e, IQL_ERR_INVALID, "iql_act_host_members: null std with distribution members");
    n += c != IQL_ACT_SKIP;
  }
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_act_host_members: state not bound");
  if (n == 0) return IQL_OK;
  const size_t off_ids = align16(sizeof(float) * (size_t)S * Sd), off_codes = off_ids + align16(sizeof(int32_t) * S);
  const size_t off_steps = off_codes + align16(sizeof(int32_t) * S), off_mail = off_steps + align16(sizeof(uint64_t) * S);
  const size_t off_flags = off_mail + align16(sizeof(float) * (size_t)S * 2 * A);
  int rc = pinned_block(e, (void**)&e->h_actm, off_flags + sizeof(uint32_t) * S, "iql_act_host_members");
  if (rc != IQL_OK) return rc;
  float* states = (float*)e->h_actm;
  int32_t* ids = (int32_t*)(e->h_actm + off_ids);
  int32_t* codes = (int32_t*)(e->h_actm + off_codes);
  uint64_t* steps = (uint64_t*)(e->h_actm + off_steps);
  float* mail = (float*)(e->h_actm + off_mail);
  volatile uint32_t* flags = (volatile uint32_t*)(e->h_actm + off_flags);
  // the previous call returned only after every flag of its launch was raised: the block is free to refill
  memcpy(states, host_states, sizeof(float) * (size_t)S * Sd);
  int j = 0;
  bool drop_codes = false;
  for (int m = 0; m < S; ++m)
    if (host_source[m] != IQL_ACT_SKIP) {
      ids[j] = m;
      codes[j] = host_source[m];
      steps[j] = e->act_steps[m];
      flags[m] = 0u;
      drop_codes |= codes[j] == IQL_ACT_LEARNER_DROPOUT || codes[j] == IQL_ACT_LEARNER_DIST_DROPOUT;
      ++j;
    }
  std::atomic_thread_fence(std::memory_order_seq_cst);
  cudaStream_t cur = (cudaStream_t)caller_stream;
  (void)stream;
  rc = order_behind_host_step(e, cur);
  if (rc != IQL_OK) return rc;
  rc = flush_tables(e, cur);
  if (rc != IQL_OK) return rc;
  StepCtx ctx = make_ctx(e);
  launch_act_members(ctx, e->params, e->guide, e->d_act_off, e->d_act_off + (L + 1), states, ids, codes, steps, drop_codes, n,
                     max_action, mail, (uint32_t*)flags, cur);
  CUDA_TRY(e, cudaGetLastError());
  for (int i = 0; i < n && drop_codes; ++i)  // the masks of the dropout codes are drawn: their counters move on, whatever p is
    if (codes[i] == IQL_ACT_LEARNER_DROPOUT || codes[i] == IQL_ACT_LEARNER_DIST_DROPOUT) ++e->act_steps[ids[i]];
  for (int i = 0; i < n; ++i) {
    rc = spin_flag(e, flags + ids[i], cur, "iql_act_host_members");
    if (rc != IQL_OK) return rc;
  }
  for (int i = 0; i < n; ++i) {
    const int m = ids[i];
    const volatile float* row = mail + (size_t)m * 2 * A;
    for (int k = 0; k < A; ++k) host_out[(size_t)m * A + k] = row[k];
    if (codes[i] == IQL_ACT_LEARNER_DIST || codes[i] == IQL_ACT_LEARNER_DIST_DROPOUT)
      for (int k = 0; k < A; ++k) host_std[(size_t)m * A + k] = row[A + k];
  }
  return IQL_OK;
}

extern "C" int iql_get_act_steps(iql_engine* e, uint64_t* host_out) {
  if (!e || !host_out) return fail(e, IQL_ERR_INVALID, "iql_get_act_steps: null argument");
  std::copy(e->act_steps.begin(), e->act_steps.end(), host_out);
  return IQL_OK;
}

extern "C" int iql_set_act_steps(iql_engine* e, const uint64_t* host_in) {
  if (!e || !host_in) return fail(e, IQL_ERR_INVALID, "iql_set_act_steps: null argument");
  std::copy(host_in, host_in + e->cfg.n_members, e->act_steps.begin());
  return IQL_OK;
}

extern "C" int iql_replay_insert_members_host(iql_engine* e, const float* host_states, const float* host_actions,
                                              const float* host_rewards, const float* host_next_states, const float* host_dones,
                                              const int64_t* host_pointers, void* stream, void* caller_stream) {
  if (!e) return IQL_ERR_INVALID;
  if (!host_states || !host_actions || !host_rewards || !host_next_states || !host_dones || !host_pointers)
    return fail(e, IQL_ERR_INVALID, "iql_replay_insert_members_host: null argument");
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_replay_insert_members_host: state not bound");
  const int S = e->cfg.n_members;
  const iql_row_layout& lay = e->layout.row;
  const int Sd = lay.state_dim, A = lay.action_dim, RF = lay.row_floats;
  std::vector<std::pair<const float*, int>> rings;
  for (int m = 0; m < S; ++m) {
    const int64_t p = host_pointers[m];
    if (p == -1) continue;
    const ReplayBinding& b = e->h_replay[m];
    if (!b.rows) return fail(e, IQL_ERR_INVALID, "iql_replay_insert_members_host: member " + std::to_string(m) + " has no replay binding");
    if (p < 0 || p >= b.capacity)
      return fail(e, IQL_ERR_INVALID, "iql_replay_insert_members_host: pointer " + std::to_string(p) + " of member " + std::to_string(m) +
                                          " is outside [0, " + std::to_string(b.capacity) + ")");
    rings.emplace_back(b.rows, m);
  }
  const int n = (int)rings.size();
  if (n == 0) return IQL_OK;
  std::sort(rings.begin(), rings.end());
  for (int i = 1; i < n; ++i)
    if (rings[i].first == rings[i - 1].first)
      return fail(e, IQL_ERR_INVALID, "iql_replay_insert_members_host: members " + std::to_string(rings[i - 1].second) + " and " +
                                          std::to_string(rings[i].second) + " share one ring; members must not see each other's transitions");
  const size_t off_ids = align16(sizeof(float) * (size_t)S * RF), off_ptr = off_ids + align16(sizeof(int32_t) * S);
  const size_t off_cons = off_ptr + align16(sizeof(int64_t) * S), slot_bytes = align16(off_cons + sizeof(uint32_t) * S);
  int rc = pinned_block(e, (void**)&e->h_ins, 2 * slot_bytes, "iql_replay_insert_members_host");
  if (rc != IQL_OK) return rc;
  const int s = e->ins_slot;
  char* slot = e->h_ins + s * slot_bytes;
  float* rows = (float*)slot;
  int32_t* ids = (int32_t*)(slot + off_ids);
  int64_t* ptrs = (int64_t*)(slot + off_ptr);
  volatile uint32_t* consumed = (volatile uint32_t*)(slot + off_cons);
  // guard: the launch that last read this slot must have consumed every row of it (it was issued two calls ago, so
  // this almost never waits; it is a spin on pinned words, not a stream synchronisation)
  for (int i = 0; i < e->ins_n[s]; ++i) {
    rc = spin_flag(e, consumed + i, e->ins_stream[s], "iql_replay_insert_members_host");
    if (rc != IQL_OK) return rc;
  }
  int i = 0;
  for (int m = 0; m < S; ++m) {
    if (host_pointers[m] == -1) continue;
    float* r = rows + (size_t)i * RF;
    memset(r, 0, sizeof(float) * RF);
    memcpy(r + lay.off_state, host_states + (size_t)m * Sd, sizeof(float) * Sd);
    memcpy(r + lay.off_action, host_actions + (size_t)m * A, sizeof(float) * A);
    memcpy(r + lay.off_next_state, host_next_states + (size_t)m * Sd, sizeof(float) * Sd);
    r[lay.off_reward] = host_rewards[m];
    r[lay.off_done] = host_dones[m];
    ids[i] = m;
    ptrs[i] = host_pointers[m];
    consumed[i] = 0u;
    ++i;
  }
  std::atomic_thread_fence(std::memory_order_seq_cst);
  cudaStream_t cur = (cudaStream_t)caller_stream;
  (void)stream;
  rc = order_behind_host_step(e, cur);
  if (rc != IQL_OK) return rc;
  rc = flush_tables(e, cur);
  if (rc != IQL_OK) return rc;
  launch_insert_members(e->d_replay, RF, rows, ids, ptrs, n, (uint32_t*)consumed, cur);
  CUDA_TRY(e, cudaGetLastError());
  e->ins_n[s] = n;
  e->ins_stream[s] = cur;
  e->ins_slot = s ^ 1;
  return IQL_OK;
}

// Self-test of the tcgen05 GEMM on one dense problem (tests/test_gpu_umma.py):
// C[M,N] = op(A) op(B) with the operand layouts of `mode` (0 NT, 1 NN, 2 TN), plain store.
extern "C" int iql_selftest_umma_gemm(int32_t mode, int32_t M, int32_t N, int32_t K, const float* A, int32_t lda,
                                      const float* B, int32_t ldb, float* C, int32_t ldc, void* scratch,
                                      size_t scratch_bytes, void* stream) {
  const bool allow_pair = !(mode & 0x100);  // test hook: mode | 0x100 keeps the single-CTA kernel
  const int tile_n_arg = (mode & 0x400) ? 64 : ((mode & 0x200) ? 128 : 0);  // test hooks: mode | 0x200 / 0x400 run N = 128 / 64 tiles
  mode &= 0xFF;
  if (mode < 0 || mode > 2 || M <= 0 || N <= 0 || K <= 0 || (M % 256) || (N > 256 && (N % 256)))
    return fail(nullptr, IQL_ERR_INVALID, "iql_selftest_umma_gemm: M multiple of 256 and N <= 256 or a multiple of 256 required");
  if ((lda & 3) || (ldb & 3)) return fail(nullptr, IQL_ERR_INVALID, "iql_selftest_umma_gemm: lda, ldb must be multiples of 4 (TMA row alignment)");
  if (!A || !B || !C || !scratch || scratch_bytes < 1024 || ((uintptr_t)scratch & 127))
    return fail(nullptr, IQL_ERR_INVALID, "iql_selftest_umma_gemm: null pointer or scratch < 1024 B / unaligned");
  GemmProb p;
  memset(&p, 0, sizeof(p));
  p.A = A; p.B = B; p.C = C; p.M = M; p.N = N; p.K = K; p.lda = lda; p.ldb = ldb; p.ldc = ldc;
  p.epi = EPI_NONE; p.drop_layer = -1;
  alignas(64) char maps[256];
  const bool cta2 = allow_pair && umma_cta2_ok(M, N);
  if (umma_encode_maps(mode, &p, 1, tile_n_arg ? tile_n_arg : umma_tile_n(N), maps, cta2)) return fail(nullptr, IQL_ERR_CUDA, "iql_selftest_umma_gemm: cuTensorMapEncodeTiled failed");
  cudaStream_t st = (cudaStream_t)stream;
  char* d = (char*)scratch;
  if (cudaMemcpyAsync(d, maps, 256, cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaMemcpyAsync(d + 256, &p, sizeof(p), cudaMemcpyHostToDevice, st) != cudaSuccess ||
      cudaStreamSynchronize(st) != cudaSuccess)
    return fail(nullptr, IQL_ERR_CUDA, "iql_selftest_umma_gemm: upload failed");
  StepCtx ctx;
  memset(&ctx, 0, sizeof(ctx));
  launch_umma_gemm(mode, (const GemmProb*)(d + 256), d, nullptr, EPI_NONE, 1, M, N, ctx, st, false, 0, cta2, K, nullptr, tile_n_arg);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(nullptr, IQL_ERR_CUDA, std::string("iql_selftest_umma_gemm: ") + cudaGetErrorString(err));
  return IQL_OK;
}

extern "C" int iql_profile_step(iql_engine* e, int32_t reps, int32_t max_slots, int32_t* n_slots, float* avg_ms,
                                double* flops, double* bytes, char* labels, void* stream) {
  if (!e || !n_slots || !avg_ms || !flops || !bytes || !labels || reps <= 0 || max_slots <= 0)
    return fail(e, IQL_ERR_INVALID, "iql_profile_step: null or non-positive argument");
  if (!e->bound) return fail(e, IQL_ERR_STATE, "iql_profile_step: state not bound");
  for (const int m : e->active)
    if (!e->h_replay[m].rows || e->h_replay[m].size <= 0) return fail(e, IQL_ERR_STATE, "iql_profile_step: replay buffer not bound");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = flush_tables(e, st);
  if (rc != IQL_OK) return rc;
  StepCtx ctx = make_ctx(e);
  ctx.K = 1;
  std::vector<double> acc;
  StepTimer last;
  for (int r = 0; r < reps; ++r) {
    if (ctx.tf32) launch_refresh_shadow(ctx, e->params, e->target, st);  // every rep is a call of its own (K = 1)
    StepTimer tm;
    tm.st = st;
    ctx.k = 0;
    enqueue_step(e, ctx, true, st, &tm);
    launch_advance(ctx, 1, st);
    CUDA_TRY(e, cudaStreamSynchronize(st));
    advance_counters(e, 1);
    if (acc.empty()) acc.assign(tm.label.size(), 0.0);
    for (size_t i = 0; i + 1 < tm.ev.size() && i < acc.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, tm.ev[i], tm.ev[i + 1]);
      acc[i] += ms;
    }
    for (cudaEvent_t ev : tm.ev) cudaEventDestroy(ev);
    tm.ev.clear();
    last = tm;
  }
  const int n = (int)std::min<size_t>(acc.size(), (size_t)max_slots);
  *n_slots = n;
  for (int i = 0; i < n; ++i) {
    avg_ms[i] = (float)(acc[i] / reps);
    flops[i] = last.flops[i];
    bytes[i] = last.bytes[i];
    snprintf(labels + 32 * i, 32, "%s", last.label[i].c_str());
  }
  return IQL_OK;
}

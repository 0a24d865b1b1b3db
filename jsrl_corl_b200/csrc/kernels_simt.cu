// FP32 CUDA-core ("SIMT") kernels of the IQL update: grouped GEMM with fused
// epilogues, the replay gather into the step workspace, the loss / output-
// gradient kernel, and the fused Adam + Polyak + cosine-LR kernel.
//
// This is the validation path of the engine (IQL_MATH_FP32_SIMT): plain fp32
// FMAs in a fixed summation order, no tensor cores.  The math follows the
// reference step algorithms/finetune/iql.py:482-563 (see SURVEY.md section 9).
#include <math.h>

#include "common.cuh"
#include "engine.h"
#include "adam.cuh"

namespace iql {

// ===========================================================================
// grouped SGEMM, 64x64x16 tiles, 256 threads, 4x4 register tile per thread.
//   A_KC: A(i,k) stored with k contiguous (row-major [M][K]); else [K][M].
//   B_KC: B(k,j) stored with k contiguous (row-major [N][K]); else [K][N].
//   NT (fwd  Y = X W^T)      : A_KC=1, B_KC=1
//   NN (dgrad dX = dZ W)     : A_KC=1, B_KC=0
//   TN (wgrad dW = dZ^T X)   : A_KC=0, B_KC=0
// ===========================================================================
constexpr int BM = 64, BN = 64, BK = 16, LDS_PAD = 4;

template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(256) simt_gemm_kernel(const GemmProb* __restrict__ probs, StepCtx ctx) {
  const GemmProb p = probs[blockIdx.z];
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  if (m0 >= p.M || n0 >= p.N) return;

  __shared__ __align__(16) float As[BK][BM + LDS_PAD];
  __shared__ __align__(16) float Bs[BK][BN + LDS_PAD];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
  const bool do_bsum = (!A_KC) && p.dbias != nullptr && blockIdx.x == 0 && tx == 0;

  for (int k0 = 0; k0 < p.K; k0 += BK) {
    // ---- stage A tile ----
    if (A_KC) {
      const int k = tid & 15;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int i = (tid >> 4) + r * 16;
        float v = 0.f;
        if (m0 + i < p.M && k0 + k < p.K) v = p.A[(int64_t)(m0 + i) * p.lda + k0 + k];
        As[k][i] = v;
      }
    } else {
      const int i = tid & 63;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int k = (tid >> 6) + r * 4;
        float v = 0.f;
        if (m0 + i < p.M && k0 + k < p.K) v = p.A[(int64_t)(k0 + k) * p.lda + m0 + i];
        As[k][i] = v;
      }
    }
    // ---- stage B tile ----
    if (B_KC) {
      const int k = tid & 15;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int j = (tid >> 4) + r * 16;
        float v = 0.f;
        if (n0 + j < p.N && k0 + k < p.K) v = p.B[(int64_t)(n0 + j) * p.ldb + k0 + k];
        Bs[k][j] = v;
      }
    } else {
      const int j = tid & 63;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int k = (tid >> 6) + r * 4;
        float v = 0.f;
        if (n0 + j < p.N && k0 + k < p.K) v = p.B[(int64_t)(k0 + k) * p.ldb + n0 + j];
        Bs[k][j] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
      if (do_bsum) {
#pragma unroll
        for (int i = 0; i < 4; ++i) bsum[i] += a[i];
      }
    }
    __syncthreads();
  }

  // ---- epilogue ----
  const MemberScalars* sc = ctx.scalars + p.member;
  const bool philox_drop = (p.epi == EPI_RELU) && p.drop_layer >= 0 && sc->drop_threshold != 0u;
  uint64_t step = 0;
  if (philox_drop) step = (uint64_t)(ctx.counters[p.member].actor_step + ctx.k);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = m0 + ty * 4 + i;
    if (row >= p.M) continue;
    const int col0 = n0 + tx * 4;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = acc[i][j];
    if (p.epi == EPI_LINEAR || p.epi == EPI_RELU) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (col0 + j < p.N) v[j] += p.bias[col0 + j];
    }
    if (p.epi == EPI_RELU) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.f);
      if (philox_drop) {
        if (ctx.dropout_masks) {
          // injected keep-masks [S][K][L][B][H] (test hook)
          const uint8_t* mk = ctx.dropout_masks +
                              ((((int64_t)p.member * ctx.K + ctx.k) * ctx.L + p.drop_layer) * ctx.B + row) * (int64_t)ctx.H;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (col0 + j < p.N) v[j] = mk[col0 + j] ? v[j] * sc->drop_scale : 0.f;
        } else {
          const uint32_t quad = (uint32_t)(((int64_t)row * p.N + col0) >> 2);
          const Philox4 r = philox_dropout_quad(sc->seed, step, (uint32_t)p.drop_layer, quad);
          const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) v[j] = (w[j] >= sc->drop_threshold) ? v[j] * sc->drop_scale : 0.f;
        }
      }
    } else if (p.epi == EPI_DRELU) {
      // d relu (and the dropout scale: H = relu(Z) * keep / (1-p), so [H > 0] == [Z > 0 and kept])
      const float dscale = (p.drop_layer >= 0 && sc->drop_threshold != 0u) ? sc->drop_scale : 1.0f;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (col0 + j < p.N) v[j] = (p.mask[(int64_t)row * p.ldmask + col0 + j] > 0.f) ? v[j] * dscale : 0.f;
    }
    float* crow = p.C + (int64_t)row * p.ldc;
    if (col0 + 3 < p.N && ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0)) {
      *reinterpret_cast<float4*>(crow + col0) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (col0 + j < p.N) crow[col0 + j] = v[j];
    }
  }
  if (do_bsum) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int row = m0 + ty * 4 + i;
      if (row < p.M) p.dbias[row] = bsum[i];
    }
  }
}

void launch_simt_gemm(int mode, const GemmProb* probs, int nprob, int maxM, int maxN, const StepCtx& ctx,
                      cudaStream_t st) {
  dim3 grid((maxN + BN - 1) / BN, (maxM + BM - 1) / BM, nprob);
  if (mode == 0) simt_gemm_kernel<true, true><<<grid, 256, 0, st>>>(probs, ctx);
  else if (mode == 1) simt_gemm_kernel<true, false><<<grid, 256, 0, st>>>(probs, ctx);
  else simt_gemm_kernel<false, false><<<grid, 256, 0, st>>>(probs, ctx);
}

// member served by CTA row i of a per-member kernel (StepCtx::active; null when every member trains, which saves the
// dependent load at the head of every per-member kernel of a full ensemble's step)
__device__ __forceinline__ int member_of(const StepCtx& ctx, int i) { return ctx.active ? ctx.active[i] : i; }

// ===========================================================================
// replay gather into the step workspace: xrow[m][b][:] = rows_m[idx][:]
// ===========================================================================
__device__ __forceinline__ void gather_body(const StepCtx& ctx, float* __restrict__ ws, int64_t ws_member_floats, int64_t xrow_off,
                                            int bx) {
  const int m = member_of(ctx, blockIdx.y);
  const int RF = ctx.row.row_floats, Q = RF >> 2;
  const int t = bx * blockDim.x + threadIdx.x;
  stamp_begin(ctx.stamps, ST_GATHER);
  if (t >= ctx.B * Q) return;
  const int b = t / Q, q = t - b * Q;
  const ReplayBinding rb = ctx.replay[m];
  // rows past the member's batch B_m are zeros (a finite forward whatever the history) and read no index
  const bool pad = b >= ctx.scalars[m].batch;
  int64_t idx = -1;
  if (!pad) {
    if (ctx.indices) {
      idx = ctx.indices[((int64_t)m * ctx.K + ctx.k) * ctx.B + b];
    } else {
      const uint64_t step = (uint64_t)(ctx.counters[m].sample_step + ctx.k);
      idx = philox_index(ctx.scalars[m].seed, step, (uint32_t)b, (uint64_t)rb.size);
    }
  }
  if (q == 0 && ctx.idx_out) ctx.idx_out[((int64_t)m * ctx.K + ctx.k) * ctx.B + b] = idx;
  const float4 v = pad ? make_float4(0.f, 0.f, 0.f, 0.f) : __ldg(reinterpret_cast<const float4*>(rb.rows + idx * RF) + q);
  float* wm = ws + m * ws_member_floats;
  reinterpret_cast<float4*>(wm + xrow_off + (int64_t)b * RF)[q] = v;
  if (ctx.xhi_off) {  // TF32 hi / lo split of the row for the 3xTF32 input layer
    const float4 hi = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
    reinterpret_cast<float4*>(wm + ctx.xhi_off + (int64_t)b * RF)[q] = hi;
    reinterpret_cast<float4*>(wm + ctx.xlo_off + (int64_t)b * RF)[q] =
        make_float4(round_tf32(v.x - hi.x), round_tf32(v.y - hi.y), round_tf32(v.z - hi.z), round_tf32(v.w - hi.w));
  }
  stamp_end(ctx.stamps, ST_GATHER);
}

__global__ void __launch_bounds__(256) gather_kernel(StepCtx ctx, float* __restrict__ ws, int64_t ws_member_floats,
                                                     int64_t xrow_off) {
  gather_body(ctx, ws, ws_member_floats, xrow_off, (int)blockIdx.x);
}

void launch_gather(const StepCtx& ctx, float* ws, int64_t ws_member_floats, int64_t xrow_off, cudaStream_t st) {
  const int threads = ctx.B * (ctx.row.row_floats >> 2);
  dim3 grid((threads + 255) / 256, ctx.n_active);
  gather_kernel<<<grid, 256, 0, st>>>(ctx, ws, ws_member_floats, xrow_off);
}

__global__ void load_batch_kernel(iql_row_layout lay, int B, float* __restrict__ xrow, float* __restrict__ xhi,
                                  float* __restrict__ xlo, const float* __restrict__ s,
                                  const float* __restrict__ a, const float* __restrict__ r,
                                  const float* __restrict__ s2, const float* __restrict__ d) {
  const int RF = lay.row_floats, S = lay.state_dim, A = lay.action_dim;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * RF) return;
  const int row = i / RF, c = i - row * RF;
  float v = 0.f;
  if (c < S) v = s[(int64_t)row * S + c];
  else if (c < S + A) v = a[(int64_t)row * A + (c - S)];
  else if (c >= lay.off_next_state && c < lay.off_next_state + S) v = s2[(int64_t)row * S + (c - lay.off_next_state)];
  else if (c == lay.off_reward) v = r[row];
  else if (c == lay.off_done) v = d[row];
  xrow[i] = v;
  if (xhi) {
    const float hi = round_tf32(v);
    xhi[i] = hi;
    xlo[i] = round_tf32(v - hi);
  }
}

void launch_load_batch(const StepCtx& ctx, int member, float* xrow, const float* s, const float* a, const float* r,
                       const float* s2, const float* d, cudaStream_t st) {
  (void)member;
  const int n = ctx.B * ctx.row.row_floats;
  // xrow points at this member's gathered-row region; the hi / lo copies live at fixed offsets from it
  float* xhi = ctx.xhi_off ? xrow + (ctx.xhi_off - ctx.xrow_off_) : nullptr;
  float* xlo = ctx.xhi_off ? xrow + (ctx.xlo_off - ctx.xrow_off_) : nullptr;
  load_batch_kernel<<<(n + 255) / 256, 256, 0, st>>>(ctx.row, ctx.B, xrow, xhi, xlo, s, a, r, s2, d);
}

// ===========================================================================
// losses and output gradients (one CTA per member)
//   value_loss  iql.py:489-490,301-302     q_loss  iql.py:506-508
//   actor_loss  iql.py:524-534 (+ torch Normal.log_prob)
// ===========================================================================
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int LOSS_MAX_A = 64;  // log_std gradient slots reduced in shared memory

__global__ void __launch_bounds__(256) loss_kernel(StepCtx ctx, float* __restrict__ ws, int64_t ws_member_floats,
                                                   WorkspaceLayout wl, const float* __restrict__ params,
                                                   float* __restrict__ grads) {
  // per-warp partial sums: [0..3] = value / q1 / q2 / actor loss terms, [4 + a] = d loss / d log_std[a].
  // One shuffle tree per quantity and ONE block barrier; summation order is fixed (rows by lane, warps 0..7).
  __shared__ float red[8][4 + LOSS_MAX_A];
  stamp_begin(ctx.stamps, ST_LOSS);
  if (blockIdx.x >= ctx.n_active) {
    // Extra CTAs (idle SMs, next to the loss CTAs): the Adam scalars of this step for the optimizer kernel --
    // torch computes the bias corrections and the step size in Python floats, CosineAnnealingLR in closed form.
    // 6 threads per member: thread (o, which) takes one fp64 pow, the pair combines through a shuffle.
    const int slot = (blockIdx.x - ctx.n_active) * 42 + threadIdx.x / 6;
    const int o = (threadIdx.x % 6) >> 1, which = threadIdx.x & 1;  // o: 0 q, 1 v, 2 actor
    const bool act = threadIdx.x < 252 && slot < ctx.n_active;
    const int idx = act ? member_of(ctx, slot) : 0;
    double pw = 0.0, lr = 0.0;
    if (act) {
      const MemberScalars sc = ctx.scalars[idx];
      const iql_counters c = ctx.counters[idx];
      int64_t t;
      if (o == 0) { lr = sc.qf_lr; t = c.q_step + ctx.k + 1; }
      else if (o == 1) { lr = sc.vf_lr; t = c.v_step + ctx.k + 1; }
      else {
        t = c.actor_step + ctx.k + 1;
        if (sc.cosine_t_max > 0) {
          const double e = (double)(c.sched_epoch + ctx.k);
          lr = sc.lr_eta_min + (sc.actor_lr - sc.lr_eta_min) * (1.0 + cos(M_PI * e / (double)sc.cosine_t_max)) * 0.5;
        } else {
          lr = sc.actor_lr;
        }
      }
      pw = pow(which ? sc.adam_beta2_d : sc.adam_beta1_d, (double)t);
    }
    const double other = __shfl_xor_sync(0xffffffffu, pw, 1);  // lanes 2j / 2j+1 hold beta1^t / beta2^t
    if (act && which == 0) {
      AdamScalars as;
      as.neg_step_size = (float)(-(lr / (1.0 - pw)));
      as.bc2_sqrt = (float)sqrt(1.0 - other);
      ctx.adam_sc[idx * 3 + o] = as;
    }
    stamp_end(ctx.stamps, ST_LOSS);
    return;
  }
  const int m = member_of(ctx, blockIdx.x);
  const int B = ctx.B, A = ctx.A_dim, RF = ctx.row.row_floats, Ald = wl.Ald;
  float* w = ws + m * ws_member_floats;
  const float* xrow = w + wl.xrow;
  const float* yq = w + wl.yq;
  const float* zpi = w + wl.zpi;
  float* gy = w + wl.gy;
  float* gpi = w + wl.gpi;
  const MemberScalars sc = ctx.scalars[m];
  // the member's own batch: means over rows [0, B_m); pad rows are skipped (exp(beta * adv) of a zero row may overflow)
  // and get exact-zero output gradients
  const int Bm = sc.batch;
  const float inv_b = 1.0f / (float)Bm;
  const float w_neg = fabsf(sc.iql_tau - 1.0f), w_pos = fabsf(sc.iql_tau);
  const float* log_std = params + m * ctx.P + ctx.log_std_off;
  constexpr float HALF_LOG_2PI = 0.9189385332046727f;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool gauss = !ctx.deterministic;
  for (int j = lane; j < 4 + LOSS_MAX_A; j += 32) red[warp][j] = 0.f;
  __syncwarp();

  float v_acc = 0.f, q1_acc = 0.f, q2_acc = 0.f, a_acc = 0.f;
  for (int b0 = 0; b0 < B; b0 += blockDim.x) {  // uniform trip count: every lane takes part in the shuffles
    const int b = b0 + threadIdx.x;
    const bool valid = b < Bm;
    const bool pad = !valid && b < B;
    float adv = 0.f, e = 0.f, eb = 0.f;
    const float* xr = xrow + (int64_t)(valid ? b : 0) * RF;
    if (pad) {
      gy[0 * B + b] = 0.f;
      gy[1 * B + b] = 0.f;
      gy[2 * B + b] = 0.f;
    }
    if (valid) {
      const float next_v = yq[PASS_V_NEXT * B + b];
      const float v = yq[PASS_V * B + b];
      const float tq = fminf(yq[PASS_TQ1 * B + b], yq[PASS_TQ2 * B + b]);
      const float q1 = yq[PASS_Q1 * B + b], q2 = yq[PASS_Q2 * B + b];
      const float r = xr[ctx.row.off_reward], d = xr[ctx.row.off_done];
      // --- V (expectile) ---
      adv = tq - v;
      const float wt = adv < 0.f ? w_neg : w_pos;
      v_acc += wt * (adv * adv);
      gy[0 * B + b] = -((wt * inv_b) * (2.0f * adv));
      // --- Q (TD) ---
      const float target = r + ((1.0f - d) * sc.discount) * next_v;
      const float d1 = q1 - target, d2 = q2 - target;
      q1_acc += d1 * d1;
      q2_acc += d2 * d2;
      gy[1 * B + b] = d1 * (2.0f * inv_b) * 0.5f;
      gy[2 * B + b] = d2 * (2.0f * inv_b) * 0.5f;
      // --- policy (AWR) weight ---
      e = fminf(expf(sc.beta * adv), 100.0f);
      eb = e * inv_b;
    }
    float bc = 0.f;
    for (int a = 0; a < A; ++a) {
      float dls = 0.f;
      if (valid) {
        const float mu = tanhf(zpi[(int64_t)b * Ald + a]);
        const float act = xr[ctx.row.off_action + a];
        float gmu;
        if (!gauss) {
          const float diff = mu - act;
          bc += diff * diff;
          gmu = eb * (2.0f * diff);
        } else {
          const float ls = fminf(fmaxf(log_std[a], -20.0f), 2.0f);
          const float sd = expf(ls);
          const float var = sd * sd;
          const float diff = act - mu;
          const float logp = -(diff * diff) / (2.0f * var) - logf(sd) - HALF_LOG_2PI;
          bc -= logp;
          gmu = -eb * diff / var;
          dls = eb * (1.0f - diff * diff / var);
        }
        gpi[(int64_t)b * Ald + a] = gmu * (1.0f - mu * mu);
      } else if (pad) {
        gpi[(int64_t)b * Ald + a] = 0.f;
      }
      if (gauss && a < LOSS_MAX_A) {
        dls = warp_sum(dls);
        if (lane == 0) red[warp][4 + a] += dls;
      }
    }
    a_acc += e * bc;
  }
  v_acc = warp_sum(v_acc);
  q1_acc = warp_sum(q1_acc);
  q2_acc = warp_sum(q2_acc);
  a_acc = warp_sum(a_acc);
  if (lane == 0) {
    red[warp][0] = v_acc; red[warp][1] = q1_acc; red[warp][2] = q2_acc; red[warp][3] = a_acc;
  }
  __syncthreads();
  const int j = threadIdx.x;
  if (j < 4 + (gauss ? min(A, LOSS_MAX_A) : 0)) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][j];
    red[0][j] = s;  // slot j is only read by thread j before this write
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float* out = ctx.loss_ring + ((int64_t)m * ctx.k_max + ctx.k) * 3;
    out[0] = red[0][0] * inv_b;
    out[1] = (red[0][1] * inv_b + red[0][2] * inv_b) * 0.5f;
    out[2] = red[0][3] * inv_b;
    if (ctx.host_mail) {  // the host is spinning on the flag word: losses first, system-scope fence, then the flag
      volatile float* mail = ctx.host_mail + (int64_t)m * 4;
      mail[0] = out[0]; mail[1] = out[1]; mail[2] = out[2];
      __threadfence_system();
      *reinterpret_cast<volatile uint32_t*>(mail + 3) = 1u;
    }
  }
  if (gauss && j < min(A, LOSS_MAX_A)) {
    const float lsr = log_std[j];
    grads[m * ctx.P + ctx.log_std_off + j] = (lsr >= -20.0f && lsr <= 2.0f) ? red[0][4 + j] : 0.f;
  }
  stamp_end(ctx.stamps, ST_LOSS);
}

void launch_loss(const StepCtx& ctx, float* ws, int64_t ws_member_floats, const WorkspaceLayout& wl,
                 const float* params, float* grads, cudaStream_t st) {
  loss_kernel<<<ctx.n_active + (ctx.n_active + 41) / 42, 256, 0, st>>>(ctx, ws, ws_member_floats, wl, params, grads);
}

// ===========================================================================
// fused Adam (3 optimisers) + Polyak target update + cosine LR
//   torch.optim.Adam defaults (jsrl_utils.py:263-265), soft_update iql.py:72-74,
//   CosineAnnealingLR iql.py:471 (closed form of the same schedule).
// ===========================================================================
// grid (ceil(P / 4 / 256 / ADAM_UNROLL), S): a thread owns ADAM_UNROLL float4 groups 256 * 4 floats apart, all of
// whose loads are issued before the first dependent instruction; no block barrier, no per-block fp64 prologue (the
// step's Adam scalars come from the loss kernel).  Measured on the 64-member ensemble (704 MB per launch): 132 us
// with the per-block prologue, 109 / 113 / 116 us without it at ADAM_UNROLL = 1 / 2 / 4 -- 99 % of the measured
// HBM copy peak at 1.
constexpr int ADAM_UNROLL = 1;
__global__ void __launch_bounds__(256) adam_polyak_kernel(StepCtx ctx, float* __restrict__ params,
                                                          float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq,
                                                          float* __restrict__ target,
                                                          const float* __restrict__ grads) {
  const int m = member_of(ctx, blockIdx.y);
  const MemberScalars* sc = ctx.scalars + m;
  stamp_begin(ctx.stamps, ST_ADAM);
  pdl_wait();  // gradients, Adam scalars of the step: written by the launches before this one
  if (ctx.advance_k > 0 && blockIdx.x == 0 && threadIdx.x == 0) {  // advance_kernel's work, folded into the call's last launch
    iql_counters c = ctx.counters[m];
    c.v_step += ctx.advance_k;
    c.q_step += ctx.advance_k;
    c.actor_step += ctx.advance_k;
    c.total_it += ctx.advance_k;
    c.sample_step += ctx.advance_k;
    if (sc->cosine_t_max > 0) c.sched_epoch += ctx.advance_k;
    ctx.counters[m] = c;
  }
  const float adam_w1 = sc->adam_w1, adam_beta2 = sc->adam_beta2, adam_one_minus_b2 = sc->adam_one_minus_b2;
  const float adam_eps = sc->adam_eps, tau = sc->tau, one_minus_tau = sc->one_minus_tau;
  const int64_t base = ((int64_t)blockIdx.x * ADAM_UNROLL * 256 + threadIdx.x) * 4;
  float4 g4[ADAM_UNROLL], p4[ADAM_UNROLL], m4[ADAM_UNROLL], v4[ADAM_UNROLL], t4[ADAM_UNROLL];
  AdamScalars as[ADAM_UNROLL];
#pragma unroll
  for (int u = 0; u < ADAM_UNROLL; ++u) {
    const int64_t i = base + (int64_t)u * 256 * 4;
    if (i < ctx.P) {
      const int64_t off = m * ctx.P + i;
      g4[u] = *reinterpret_cast<const float4*>(grads + off);
      p4[u] = *reinterpret_cast<const float4*>(params + off);
      m4[u] = *reinterpret_cast<const float4*>(exp_avg + off);
      v4[u] = *reinterpret_cast<const float4*>(exp_avg_sq + off);
      t4[u] = (i < ctx.PQ) ? *reinterpret_cast<const float4*>(target + m * ctx.PQ + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      as[u] = ctx.adam_sc[m * 3 + (i < ctx.PQ ? 0 : (i < ctx.v_end ? 1 : 2))];
    }
  }
#pragma unroll
  for (int u = 0; u < ADAM_UNROLL; ++u) {
    const int64_t i = base + (int64_t)u * 256 * 4;
    if (i < ctx.P)
      adam_quad(ctx, m, i, g4[u], p4[u], m4[u], v4[u], t4[u], as[u], adam_w1, adam_beta2, adam_one_minus_b2, adam_eps, tau,
                one_minus_tau, params, exp_avg, exp_avg_sq, target);
  }
  stamp_end(ctx.stamps, ST_ADAM);
}

// TF32-rounded operand copies of params / target, rebuilt at the start of every engine call so that weights
// written from outside (checkpoint loads, parameter surgery through the torch views) are always picked up.
__device__ __forceinline__ void refresh_body(const StepCtx& ctx, float* __restrict__ params, float* __restrict__ target, int bx) {
  const int m = member_of(ctx, blockIdx.y);
  const int64_t i = ((int64_t)bx * blockDim.x + threadIdx.x) * 4;
  stamp_begin(ctx.stamps, ST_REFRESH);
  bool first_layer = false;
#pragma unroll
  for (int r = 0; r < 5; ++r) first_layer |= (i >= ctx.first_w_begin[r] && i < ctx.first_w_end[r]);
  const bool hidden = in_hidden_weights(ctx, i);  // these enter the call biased in place and have no shadow (engine.h)
  if (i < ctx.P) {
    const float4 v = *reinterpret_cast<const float4*>(params + m * ctx.P + i);
    if (hidden) {
      *reinterpret_cast<float4*>(params + m * ctx.P + i) = make_float4(tf32_bias(v.x), tf32_bias(v.y), tf32_bias(v.z), tf32_bias(v.w));
    } else {
      const float4 hi = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
      *reinterpret_cast<float4*>(ctx.w_shadow + m * ctx.P + i) = hi;
      if (first_layer)
        *reinterpret_cast<float4*>(ctx.w_shadow_lo + m * ctx.P + i) =
            make_float4(round_tf32(v.x - hi.x), round_tf32(v.y - hi.y), round_tf32(v.z - hi.z), round_tf32(v.w - hi.w));
    }
  }
  if (i < ctx.PQ) {
    const float4 v = *reinterpret_cast<const float4*>(target + m * ctx.PQ + i);
    if (hidden) {
      *reinterpret_cast<float4*>(target + m * ctx.PQ + i) = make_float4(tf32_bias(v.x), tf32_bias(v.y), tf32_bias(v.z), tf32_bias(v.w));
    } else {
      const float4 hi = make_float4(round_tf32(v.x), round_tf32(v.y), round_tf32(v.z), round_tf32(v.w));
      *reinterpret_cast<float4*>(ctx.t_shadow + m * ctx.PQ + i) = hi;
      if (first_layer)
        *reinterpret_cast<float4*>(ctx.t_shadow_lo + m * ctx.PQ + i) =
            make_float4(round_tf32(v.x - hi.x), round_tf32(v.y - hi.y), round_tf32(v.z - hi.z), round_tf32(v.w - hi.w));
    }
  }
  stamp_end(ctx.stamps, ST_REFRESH);
}

__global__ void __launch_bounds__(256) refresh_shadow_kernel(StepCtx ctx, float* __restrict__ params, float* __restrict__ target) {
  refresh_body(ctx, params, target, (int)blockIdx.x);
}

void launch_refresh_shadow(const StepCtx& ctx, float* params, float* target, cudaStream_t st) {
  dim3 grid((unsigned)((ctx.P / 4 + 255) / 256), ctx.n_active);
  refresh_shadow_kernel<<<grid, 256, 0, st>>>(ctx, params, target);
}

// Operand refresh and gather of a host step in ONE launch (they are independent; the first n_gather blocks of a member
// gather, the rest refresh): the fused forward then has a single predecessor, which releases it at once
// (griddepcontrol.launch_dependents) so that its set-up -- barrier init, TMEM allocation, tensor-map prefetch -- runs
// beside this kernel instead of after it.
__global__ void __launch_bounds__(256) gather_refresh_kernel(StepCtx ctx, float* __restrict__ ws, int64_t ws_member_floats,
                                                             int64_t xrow_off, float* __restrict__ params,
                                                             float* __restrict__ target, int n_gather) {
  pdl_trigger();
  if ((int)blockIdx.x < n_gather) gather_body(ctx, ws, ws_member_floats, xrow_off, (int)blockIdx.x);
  else refresh_body(ctx, params, target, (int)blockIdx.x - n_gather);
}

void launch_gather_refresh(const StepCtx& ctx, float* ws, int64_t ws_member_floats, int64_t xrow_off, float* params, float* target,
                           cudaStream_t st) {
  const int n_gather = (ctx.B * (ctx.row.row_floats >> 2) + 255) / 256;
  dim3 grid((unsigned)(n_gather + (ctx.P / 4 + 255) / 256), ctx.n_active);
  gather_refresh_kernel<<<grid, 256, 0, st>>>(ctx, ws, ws_member_floats, xrow_off, params, target, n_gather);
}

void launch_adam(const StepCtx& ctx, float* params, float* exp_avg, float* exp_avg_sq, float* target,
                 const float* grads, cudaStream_t st) {
  const int64_t quads = (ctx.P + 3) / 4;
  dim3 grid((unsigned)((quads + 256 * ADAM_UNROLL - 1) / (256 * ADAM_UNROLL)), ctx.n_active);
  launch_pdl(adam_polyak_kernel, grid, dim3(256), 0, st, 1, ctx, params, exp_avg, exp_avg_sq, target, grads);
}

__global__ void advance_kernel(StepCtx ctx, int K) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ctx.n_active) return;
  const int m = member_of(ctx, i);
  iql_counters c = ctx.counters[m];
  c.v_step += K;
  c.q_step += K;
  c.actor_step += K;
  c.total_it += K;
  c.sample_step += K;
  if (ctx.scalars[m].cosine_t_max > 0) c.sched_epoch += K;
  ctx.counters[m] = c;
}

void launch_advance(const StepCtx& ctx, int K, cudaStream_t st) {
  advance_kernel<<<(ctx.n_active + 127) / 128, 128, 0, st>>>(ctx, K);
}

// ===========================================================================
// actor inference (eval mode): out = clamp(max_action * tanh(MLP(s)))
// One CTA of 32 warps per state row, activations in shared memory.  A single observation per env step is pure
// latency (three dependent layers, 256 KB of weights each through one SM), so every warp keeps four output neurons
// = 8 independent 16-byte weight loads per lane in flight, and a layer costs about one L2 round trip plus the
// streaming of its weights.  `state_val` != null: the observation rides in the kernel parameters (host callers,
// iql_act_host); `mail` != null: the action goes to device-mapped pinned host memory, fenced, followed by a flag word.
// ===========================================================================
constexpr int ACT_THREADS = 1024, ACT_NEURONS = 4, ACT_STATE_MAX = 512;
struct ActState { float v[ACT_STATE_MAX]; };

// Training-mode dropout of the act (iql_act_host_members codes 4 / 5): hidden unit j of layer l is kept iff word j & 3
// of philox_act_dropout_quad(seed, step, l, j >> 2) is >= threshold, and a kept unit becomes relu(a) * scale -- the rule
// of the update's forward epilogues, on the act's own Philox stream.
struct ActDropout {
  uint64_t seed, step;
  uint32_t threshold;
  float scale;
};

// DROP = false is the eval-mode body; `drop` is read only when DROP is true.
template <bool DROP>
__device__ __forceinline__ void act_body(int S, int A, int H, int L, const float* __restrict__ block,
                                         const int64_t* __restrict__ w_off, const int64_t* __restrict__ b_off,
                                         const float* __restrict__ state, float max_action, float* __restrict__ out, float* sm,
                                         const ActDropout& drop = ActDropout{}) {
  const int width = ((H > S ? H : S) + 3) & ~3;
  float* cur = sm;
  float* nxt = sm + width;
  for (int i = threadIdx.x; i < width; i += blockDim.x) cur[i] = i < S ? state[i] : 0.f;  // zero tail: rows are padded to 4 floats
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  int in_dim = S;
  for (int l = 0; l <= L; ++l) {
    const int out_dim = (l == L) ? A : H;
    const float* W = block + w_off[l];
    const float* bias = block + b_off[l];
    const int ldw = (in_dim + 3) & ~3;  // weight rows are padded to a multiple of 4 floats (the padding is zero)
    const int nq = ldw >> 2;
    for (int j0 = warp * ACT_NEURONS; j0 < out_dim; j0 += nwarp * ACT_NEURONS) {
      float acc[ACT_NEURONS];
#pragma unroll
      for (int u = 0; u < ACT_NEURONS; ++u) acc[u] = 0.f;
      for (int q = lane; q < nq; q += 32) {
        const float4 x = *reinterpret_cast<const float4*>(cur + 4 * q);
        float4 w[ACT_NEURONS];
#pragma unroll
        for (int u = 0; u < ACT_NEURONS; ++u)
          w[u] = (j0 + u < out_dim) ? __ldg(reinterpret_cast<const float4*>(W + (int64_t)(j0 + u) * ldw) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < ACT_NEURONS; ++u)
          acc[u] = fmaf(w[u].x, x.x, fmaf(w[u].y, x.y, fmaf(w[u].z, x.z, fmaf(w[u].w, x.w, acc[u]))));
      }
#pragma unroll
      for (int u = 0; u < ACT_NEURONS; ++u) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[u] += __shfl_xor_sync(0xffffffffu, acc[u], o);
      }
      if (lane < ACT_NEURONS && j0 + lane < out_dim) {
        float a = acc[0];
#pragma unroll
        for (int u = 1; u < ACT_NEURONS; ++u) a = (lane == u) ? acc[u] : a;
        a += bias[j0 + lane];
        if (l < L) {
          float h = fmaxf(a, 0.f);
          if constexpr (DROP) {
            // j0 is a multiple of 4: the warp's four neurons are exactly one Philox quad
            const Philox4 r = philox_act_dropout_quad(drop.seed, drop.step, (uint32_t)l, (uint32_t)(j0 >> 2));
            const uint32_t w = lane == 0 ? r.x : lane == 1 ? r.y : lane == 2 ? r.z : r.w;
            h = (w >= drop.threshold) ? h * drop.scale : 0.f;
          }
          nxt[j0 + lane] = h;
        } else {
          out[j0 + lane] = fminf(fmaxf(max_action * tanhf(a), -max_action), max_action);
        }
      }
    }
    if (l < L)
      for (int i = out_dim + threadIdx.x; i < width; i += blockDim.x) nxt[i] = 0.f;
    __syncthreads();
    float* t = cur; cur = nxt; nxt = t;
    in_dim = out_dim;
  }
}

__global__ void __launch_bounds__(ACT_THREADS) act_kernel(int S, int A, int H, int L, const float* __restrict__ block0,
                                                          int64_t member_stride, const int64_t* __restrict__ w_off,
                                                          const int64_t* __restrict__ b_off,
                                                          const float* __restrict__ states, float max_action,
                                                          float* __restrict__ out) {
  extern __shared__ float sm[];  // 2 * round_up(max(H, S), 4)
  // blockIdx.y = ensemble member (vectorised-env mode: every member's policy on its own rows), blockIdx.x = row
  const int64_t row = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
  act_body<false>(S, A, H, L, block0 + blockIdx.y * member_stride, w_off, b_off, states + row * S, max_action, out + row * A, sm);
}

// one observation from the kernel parameters, the action into pinned host memory + flag word (iql_act_host)
__global__ void __launch_bounds__(ACT_THREADS) act_host_kernel(int S, int A, int H, int L, const float* __restrict__ block,
                                                               const int64_t* __restrict__ w_off,
                                                               const int64_t* __restrict__ b_off,
                                                               const __grid_constant__ ActState state, float max_action,
                                                               const float* __restrict__ log_std, float* __restrict__ mail) {
  extern __shared__ float sm[];
  const int width = ((H > S ? H : S) + 3) & ~3;
  float* res = sm + 2 * width;  // [A]
  act_body<false>(S, A, H, L, block, w_off, b_off, state.v, max_action, res, sm);
  __syncthreads();
  if (threadIdx.x < 32) {  // mailbox: [A] actions | [A] std = exp(clamp(log_std, -20, 2)) (Gaussian policies) | flag word
    for (int i = threadIdx.x; i < A; i += 32) {
      reinterpret_cast<volatile float*>(mail)[i] = res[i];
      reinterpret_cast<volatile float*>(mail)[A + i] = log_std ? expf(fminf(fmaxf(log_std[i], -20.0f), 2.0f)) : 0.f;
    }
    __threadfence_system();
    __syncwarp();
    if (threadIdx.x == 0) *reinterpret_cast<volatile uint32_t*>(mail + 2 * A) = 1u;
  }
}

void launch_act(const StepCtx& ctx, const float* actor_block, int n_members, const int64_t* w_off,
                const int64_t* b_off, const float* states, int64_t n, float max_action, float* out, cudaStream_t st) {
  const int width = ((ctx.H > ctx.S_dim ? ctx.H : ctx.S_dim) + 3) & ~3;
  dim3 grid((unsigned)n, (unsigned)n_members);
  act_kernel<<<grid, ACT_THREADS, 2 * width * sizeof(float), st>>>(ctx.S_dim, ctx.A_dim, ctx.H, ctx.L, actor_block, ctx.P, w_off,
                                                                   b_off, states, max_action, out);
}

// every active member of an ensemble in one launch (iql_act_host_members): CTA i serves member ids[i] with the learner
// arena or the guide arena; the observations are read from device-mapped pinned memory, the results go to the member's
// mailbox row [2A] (action or mean | std) followed by the member's flag word.  For codes 0-3 act_body is the
// single-observation body unchanged, so every member's result is bit-identical to act_host_kernel's; codes 4 / 5 add the
// member's dropout (key and p from its MemberScalars) drawn at act counter steps[i].  DROP_CODES = false (no member of
// the launch asks for dropout) compiles the kernel without the dropout body, so launches of codes 0-3 alone run the
// instructions they ran before codes 4 / 5 existed.
template <bool DROP_CODES>
__global__ void __launch_bounds__(ACT_THREADS) act_members_kernel(int S, int A, int H, int L, const float* __restrict__ params,
                                                                  const float* __restrict__ guide, int64_t P,
                                                                  const int64_t* __restrict__ w_off,
                                                                  const int64_t* __restrict__ b_off, int64_t log_std_off,
                                                                  const float* states, const int32_t* ids, const int32_t* codes,
                                                                  const uint64_t* steps, const MemberScalars* __restrict__ scalars,
                                                                  float max_action, float* mail, uint32_t* flags) {
  extern __shared__ float sm[];
  const int width = ((H > S ? H : S) + 3) & ~3;
  float* res = sm + 2 * width;  // [A]
  const int m = ids[blockIdx.x], code = codes[blockIdx.x];
  const float* block = (code == IQL_ACT_GUIDE ? guide : params) + (int64_t)m * P;
  const bool dist = code == IQL_ACT_LEARNER_DIST || (DROP_CODES && code == IQL_ACT_LEARNER_DIST_DROPOUT);
  const bool drop = DROP_CODES && (code == IQL_ACT_LEARNER_DROPOUT || code == IQL_ACT_LEARNER_DIST_DROPOUT);
  if (drop && scalars[m].drop_threshold != 0u) {  // p = 0: the eval-mode body, as in the update's epilogues
    const ActDropout d{scalars[m].seed, steps[blockIdx.x], scalars[m].drop_threshold, scalars[m].drop_scale};
    act_body<true>(S, A, H, L, block, w_off, b_off, states + (int64_t)m * S, dist ? 1.0f : max_action, res, sm, d);
  } else {
    act_body<false>(S, A, H, L, block, w_off, b_off, states + (int64_t)m * S, dist ? 1.0f : max_action, res, sm);
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    float* row = mail + (int64_t)m * 2 * A;
    for (int i = threadIdx.x; i < A; i += 32) {
      reinterpret_cast<volatile float*>(row)[i] = res[i];
      if (dist) reinterpret_cast<volatile float*>(row)[A + i] = expf(fminf(fmaxf(block[log_std_off + i], -20.0f), 2.0f));
    }
    __threadfence_system();
    __syncwarp();
    if (threadIdx.x == 0) reinterpret_cast<volatile uint32_t*>(flags)[m] = 1u;
  }
}

void launch_act_members(const StepCtx& ctx, const float* params, const float* guide, const int64_t* w_off, const int64_t* b_off,
                        const float* states, const int32_t* ids, const int32_t* codes, const uint64_t* steps, bool drop_codes,
                        int n, float max_action, float* mail, uint32_t* flags, cudaStream_t st) {
  const int width = ((ctx.H > ctx.S_dim ? ctx.H : ctx.S_dim) + 3) & ~3;
  (drop_codes ? act_members_kernel<true> : act_members_kernel<false>)<<<n, ACT_THREADS, (2 * width + ctx.A_dim) * sizeof(float), st>>>(
      ctx.S_dim, ctx.A_dim, ctx.H, ctx.L, params, guide, ctx.P, w_off, b_off, ctx.deterministic ? 0 : ctx.log_std_off, states,
      ids, codes, steps, ctx.scalars, max_action, mail, flags);
}

int act_host_state_max() { return ACT_STATE_MAX; }

void launch_act_host(const StepCtx& ctx, const float* actor_block, const int64_t* w_off, const int64_t* b_off,
                     const float* host_state, float max_action, const float* log_std, float* mail, cudaStream_t st) {
  const int width = ((ctx.H > ctx.S_dim ? ctx.H : ctx.S_dim) + 3) & ~3;
  ActState s;
  for (int i = 0; i < ACT_STATE_MAX; ++i) s.v[i] = i < ctx.S_dim ? host_state[i] : 0.f;
  act_host_kernel<<<1, ACT_THREADS, (2 * width + ctx.A_dim) * sizeof(float), st>>>(ctx.S_dim, ctx.A_dim, ctx.H, ctx.L, actor_block,
                                                                                   w_off, b_off, s, max_action, log_std, mail);
}

}  // namespace iql

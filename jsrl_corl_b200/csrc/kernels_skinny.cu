// CUDA-core kernels for the "skinny" ends of the MLPs: first layer (K = obs or
// obs+act, 11..69) and last layer (N = 1 or act_dim).  These GEMMs carry < 10 %
// of the FLOPs but have no tensor-core shape; they are HBM/L2-bound row
// streams, so each kernel makes ONE coalesced pass over the big [B, H] operand
// with the small operand held in registers / shared memory, and sums in a
// fixed order (deterministic, fp32).
//
//   first_fwd   H1 = drop(relu(X W0^T + b0))                      (iql.py:329-333 forward)
//   out_fwd     y  = H_L W_L^T + b_L                               (output Linear)
//   last_bwd    dW_L = G_L^T H_L, db_L = colsum(G_L),
//               G_{L-1} = (G_L W_L) * [H_L > 0] * scale            (autograd of the output Linear + ReLU/Dropout)
//   first_wgrad dW_0 = G_0^T X, db_0 = colsum(G_0)
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "engine.h"

namespace iql {

// ---------------------------------------------------------------------------
// first layer forward.  grid (nprob, ceil(B/64), ceil(H/(128*NC))), 128 threads.
// thread = NC output columns; their W0 rows live in registers; X rows are broadcast from smem
// (one LDS.128 feeds 4*NC FMAs).
// ---------------------------------------------------------------------------
template <int KMAX, int NC>
__global__ void __launch_bounds__(128) first_fwd_kernel(const GemmProb* __restrict__ probs, StepCtx ctx) {
  constexpr int RT = 64;
  __shared__ __align__(16) float xs[RT][KMAX];
  const GemmProb p = probs[blockIdx.x];
  const int r0 = blockIdx.y * RT;
  const int nb = blockIdx.z * 128 * NC + threadIdx.x;
  const int K = p.K;
  if (r0 >= p.M) return;
  for (int i = threadIdx.x; i < RT * KMAX; i += 128) {
    const int r = i / KMAX, k = i - r * KMAX;
    float v = 0.f;
    if (r0 + r < p.M && k < K) v = p.A[(int64_t)(r0 + r) * p.lda + k];
    xs[r][k] = v;
  }
  float w[NC][KMAX];
  float bias[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    const int n = nb + c * 128;
    bias[c] = (n < p.N) ? p.bias[n] : 0.f;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) w[c][k] = (n < p.N && k < K) ? p.B[(int64_t)n * p.ldb + k] : 0.f;
  }
  __syncthreads();
  const MemberScalars* sc = ctx.scalars + p.member;
  const bool drop = p.drop_layer >= 0 && sc->drop_threshold != 0u;
  uint64_t dstep = 0;
  if (drop) dstep = (uint64_t)(ctx.counters[p.member].actor_step + ctx.k);
  const int rows = min(RT, p.M - r0);
  for (int r = 0; r < rows; ++r) {
    float acc[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c] = 0.f;
#pragma unroll
    for (int k4 = 0; k4 < KMAX; k4 += 4) {
      const float4 x = *reinterpret_cast<const float4*>(&xs[r][k4]);
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        acc[c] = fmaf(x.x, w[c][k4], acc[c]);
        acc[c] = fmaf(x.y, w[c][k4 + 1], acc[c]);
        acc[c] = fmaf(x.z, w[c][k4 + 2], acc[c]);
        acc[c] = fmaf(x.w, w[c][k4 + 3], acc[c]);
      }
    }
    const int row = r0 + r;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int n = nb + c * 128;
      if (n >= p.N) continue;
      float v = fmaxf(acc[c] + bias[c], 0.f);
      if (drop) {
        if (ctx.dropout_masks) {
          const uint8_t* mk = ctx.dropout_masks +
                              ((((int64_t)p.member * ctx.K + ctx.k) * ctx.L + p.drop_layer) * ctx.B + row) * (int64_t)ctx.H;
          v = mk[n] ? v * sc->drop_scale : 0.f;
        } else {
          const int64_t e = (int64_t)row * p.N + n;
          const Philox4 ph = philox_dropout_quad(sc->seed, dstep, (uint32_t)p.drop_layer, (uint32_t)(e >> 2));
          const uint32_t ws = (e & 3) == 0 ? ph.x : (e & 3) == 1 ? ph.y : (e & 3) == 2 ? ph.z : ph.w;
          v = (ws >= sc->drop_threshold) ? v * sc->drop_scale : 0.f;
        }
      }
      p.C[(int64_t)row * p.ldc + n] = ctx.tf32 ? round_tf32(v) : v;  // A operand of the next (tcgen05) layer
    }
  }
}

void launch_first_fwd(const GemmProb* probs, int nprob, int B, int H, int kmax, const StepCtx& ctx, cudaStream_t st) {
  if (kmax <= 24) first_fwd_kernel<24, 2><<<dim3(nprob, (B + 63) / 64, (H + 255) / 256), 128, 0, st>>>(probs, ctx);
  else if (kmax <= 40) first_fwd_kernel<40, 2><<<dim3(nprob, (B + 63) / 64, (H + 255) / 256), 128, 0, st>>>(probs, ctx);
  else first_fwd_kernel<72, 1><<<dim3(nprob, (B + 63) / 64, (H + 127) / 128), 128, 0, st>>>(probs, ctx);
}

// ---------------------------------------------------------------------------
// output layer forward.  grid (nprob, ceil(B/rows)), 256 threads = 8 warps, one warp per row at a time, lanes stride
// the hidden dimension.  `rows` per CTA is chosen by the launcher so that the launch is a whole number of waves
// (the stress shape ran 896 CTAs on 740 resident slots: 1.21 waves, i.e. twice the time of one).
// ---------------------------------------------------------------------------
template <int AMAX>
__global__ void __launch_bounds__(256) out_fwd_kernel(const GemmProb* __restrict__ probs, int rows) {
  extern __shared__ float wsm[];  // [N][K]
  const GemmProb p = probs[blockIdx.x];
  const int K = p.K, N = p.N;
  if ((K & 3) == 0 && (p.ldb & 3) == 0) {
    const int k4n = K >> 2;
    for (int i = threadIdx.x; i < N * k4n; i += 256) {
      const int n = i / k4n, k4 = i - n * k4n;
      reinterpret_cast<float4*>(wsm)[i] = __ldg(reinterpret_cast<const float4*>(p.B + (int64_t)n * p.ldb) + k4);
    }
  } else {
    for (int i = threadIdx.x; i < N * K; i += 256) wsm[i] = p.B[(int64_t)(i / K) * p.ldb + (i % K)];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int rr = warp; rr < rows; rr += 8) {
    const int row = blockIdx.y * rows + rr;
    if (row >= p.M) break;
    float acc[AMAX];
#pragma unroll
    for (int m = 0; m < AMAX; ++m) acc[m] = 0.f;
    const float* h = p.A + (int64_t)row * p.lda;
    if (((K | p.lda) & 3) == 0) {  // 16-byte loads of the row and of the weights
      const float4* h4 = reinterpret_cast<const float4*>(h);
      for (int k4 = lane; k4 < (K >> 2); k4 += 32) {
        const float4 x = h4[k4];
#pragma unroll
        for (int m = 0; m < AMAX; ++m) {
          if (m < N) {
            const float4 w = *reinterpret_cast<const float4*>(&wsm[m * K + 4 * k4]);
            acc[m] = fmaf(x.x, w.x, acc[m]);
            acc[m] = fmaf(x.y, w.y, acc[m]);
            acc[m] = fmaf(x.z, w.z, acc[m]);
            acc[m] = fmaf(x.w, w.w, acc[m]);
          }
        }
      }
    } else {
      for (int k = lane; k < K; k += 32) {
        const float x = h[k];
#pragma unroll
        for (int m = 0; m < AMAX; ++m)
          if (m < N) acc[m] = fmaf(x, wsm[m * K + k], acc[m]);
      }
    }
#pragma unroll
    for (int m = 0; m < AMAX; ++m) {
      if (m < N) {
        float v = acc[m];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) p.C[(int64_t)row * p.ldc + m] = v + p.bias[m];
      }
    }
  }
}

// Wide heads (8 < N <= 24, the pen-human policy head): one thread per batch row, the [K][AMAX] weights transposed in
// shared memory and read back as broadcast 16-byte loads (6 per k for 24 FMAs).  The warp-per-row kernel above spends
// its time in 8 dependent strided loads and 120 shuffles per row (159 us for 256 members x 256 rows on a B200).
template <int AMAX>
__global__ void __launch_bounds__(128) out_fwd_rows_kernel(const GemmProb* __restrict__ probs) {
  extern __shared__ float wsm[];  // [K][AMAX], columns >= N zero
  const GemmProb p = probs[blockIdx.x];
  const int K = p.K, N = p.N;
  for (int i = threadIdx.x; i < AMAX * K; i += 128) {
    const int m = i / K, k = i - m * K;  // coalesced along k
    wsm[k * AMAX + m] = (m < N) ? __ldg(p.B + (int64_t)m * p.ldb + k) : 0.f;
  }
  __syncthreads();
  const int row = blockIdx.y * 128 + threadIdx.x;
  if (row >= p.M) return;
  float acc[AMAX];
#pragma unroll
  for (int m = 0; m < AMAX; ++m) acc[m] = 0.f;
  const float4* h4 = reinterpret_cast<const float4*>(p.A + (int64_t)row * p.lda);
#pragma unroll 4
  for (int k4 = 0; k4 < (K >> 2); ++k4) {
    const float4 x = __ldg(h4 + k4);
    const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4* wr = reinterpret_cast<const float4*>(wsm + (4 * k4 + j) * AMAX);
#pragma unroll
      for (int m4 = 0; m4 < AMAX / 4; ++m4) {
        const float4 w = wr[m4];
        acc[4 * m4 + 0] = fmaf(xs[j], w.x, acc[4 * m4 + 0]);
        acc[4 * m4 + 1] = fmaf(xs[j], w.y, acc[4 * m4 + 1]);
        acc[4 * m4 + 2] = fmaf(xs[j], w.z, acc[4 * m4 + 2]);
        acc[4 * m4 + 3] = fmaf(xs[j], w.w, acc[4 * m4 + 3]);
      }
    }
  }
  float* out = p.C + (int64_t)row * p.ldc;
#pragma unroll
  for (int m = 0; m < AMAX; ++m)
    if (m < N) out[m] = acc[m] + p.bias[m];
}

// rows per CTA: the multiple of 8 that minimises (waves of resident CTAs) x (rows + the weight staging, ~8 rows' worth)
template <int AMAX>
static void launch_out_fwd_t(const GemmProb* probs, int nprob, int B, size_t sm, cudaStream_t st) {
  static int per_sm = 0, n_sm = 0;
  static size_t sm_of = 0;
  static bool attr[64] = {};
  if (first_use_on_device(attr)) cudaFuncSetAttribute(out_fwd_kernel<AMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (!per_sm || sm_of != sm) {
    sm_of = sm;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, out_fwd_kernel<AMAX>, 256, sm) != cudaSuccess || per_sm <= 0) per_sm = 1;
    if (n_sm <= 0) n_sm = 148;
  }
  const int64_t slots = (int64_t)per_sm * n_sm;
  int best = 32;
  int64_t best_cost = -1;
  for (int rows = 8; rows <= ((B + 7) / 8) * 8; rows += 8) {
    const int64_t ctas = (int64_t)nprob * ((B + rows - 1) / rows);
    const int64_t cost = ((ctas + slots - 1) / slots) * (rows + 8);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = rows; }
  }
  out_fwd_kernel<AMAX><<<dim3(nprob, (B + best - 1) / best), 256, sm, st>>>(probs, best);
}

void launch_out_fwd(const GemmProb* probs, int nprob, int B, int H, int amax, cudaStream_t st) {
  const size_t sm = (size_t)amax * H * sizeof(float);
  if (amax <= 1) launch_out_fwd_t<1>(probs, nprob, B, sm, st);
  else if (amax <= 8) launch_out_fwd_t<8>(probs, nprob, B, sm, st);
  else if (amax <= 24) {
    static const bool no_rows = dbg_getenv("IQL_B200_NO_OUT_ROWS") != nullptr;
    static bool attr[64] = {};
    if (first_use_on_device(attr))
      cudaFuncSetAttribute(out_fwd_rows_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    const bool big = (int64_t)nprob * ((B + 127) / 128) >= 296;
    if (big && (H & 3) == 0 && !no_rows)
      out_fwd_rows_kernel<24><<<dim3(nprob, (B + 127) / 128), 128, (size_t)24 * H * sizeof(float), st>>>(probs);
    else launch_out_fwd_t<24>(probs, nprob, B, sm, st);
  } else launch_out_fwd_t<64>(probs, nprob, B, sm, st);
}

// ---------------------------------------------------------------------------
// last layer backward (fused wgrad + dgrad + ReLU/dropout mask).
// grid (nprob, ceil(H/64)), 256 threads = 64 columns x 4 row groups.
//   pn: the dgrad problem  (A = G_L [B][ldg], K = A_out, B = W_L [A_out][H], C = G_{L-1}, mask = H_L)
//   pw: the wgrad problem  (C = dW_L [A_out][H], dbias = db_L)
// ---------------------------------------------------------------------------
template <int AMAX>
__global__ void __launch_bounds__(256) last_bwd_kernel(const GemmProb* __restrict__ probs_dgrad,
                                                       const GemmProb* __restrict__ probs_wgrad,
                                                       const GemmProb* __restrict__ probs_prev_wgrad, StepCtx ctx,
                                                       int sel_n, int sel_off) {
  extern __shared__ float sm[];  // G tile [B][AMAX] then reduction scratch [4][64][AMAX]
  // sel_n > 0: this launch covers sel_n of every 4 problems (the training nets of a member, table order), from sel_off
  const int pi = sel_n > 0 ? (int)(blockIdx.x / sel_n) * 4 + sel_off + (int)(blockIdx.x % sel_n) : (int)blockIdx.x;
  const GemmProb pn = probs_dgrad[pi];
  const GemmProb pw = probs_wgrad[pi];
  // bias gradient of layer L-1 (the wgrad problem of the NEXT backward phase), when that layer is a hidden one
  float* dbias_prev = probs_prev_wgrad ? probs_prev_wgrad[pi].dbias : nullptr;
  const int B = pn.M, H = pn.N, AO = pn.K;
  float* gs = sm;
  float* red = sm + (size_t)B * AMAX;
  for (int i = threadIdx.x; i < B * AMAX; i += 256) {
    const int b = i / AMAX, m = i - b * AMAX;
    gs[i] = (m < AO) ? pn.A[(int64_t)b * pn.lda + m] : 0.f;
  }
  const int tn = threadIdx.x & 63, bg = threadIdx.x >> 6;
  const int n = blockIdx.y * 64 + tn;
  float w[AMAX], dw[AMAX];
#pragma unroll
  for (int m = 0; m < AMAX; ++m) {
    w[m] = (m < AO && n < H) ? pn.B[(int64_t)m * pn.ldb + n] : 0.f;
    dw[m] = 0.f;
  }
  const MemberScalars* sc = ctx.scalars + pn.member;
  const float dscale = (pn.drop_layer >= 0 && sc->drop_threshold != 0u) ? sc->drop_scale : 1.0f;
  __syncthreads();
  const int rows_per = (B + 3) / 4;
  const int b_lo = bg * rows_per, b_hi = min(B, b_lo + rows_per);
  float csum = 0.f;  // column sum of the produced G_{L-1} = bias gradient of layer L-1
  if (n < H) {
    constexpr int RB = 8;  // rows per batch: 8 independent loads in flight per thread
    if (AO == 1) {  // scalar heads (Q, V): uniform per CTA
      const float w0 = w[0];
      float d0 = 0.f;
      for (int b0 = b_lo; b0 < b_hi; b0 += RB) {
        float hv[RB];
#pragma unroll
        for (int j = 0; j < RB; ++j) hv[j] = (b0 + j < b_hi) ? __ldg(pn.mask + (int64_t)(b0 + j) * pn.ldmask + n) : 0.f;
#pragma unroll
        for (int j = 0; j < RB; ++j) {
          if (b0 + j < b_hi) {
            const float g = gs[(b0 + j) * AMAX];
            d0 = fmaf(g, hv[j], d0);
            const float o = (hv[j] > 0.f) ? (g * w0) * dscale : 0.f;
            csum += o;
            pn.C[(int64_t)(b0 + j) * pn.ldc + n] = ctx.tf32 ? round_tf32(o) : o;
          }
        }
      }
      dw[0] = d0;
    } else {
      for (int b0 = b_lo; b0 < b_hi; b0 += RB) {
        float hv[RB];
#pragma unroll
        for (int j = 0; j < RB; ++j) hv[j] = (b0 + j < b_hi) ? __ldg(pn.mask + (int64_t)(b0 + j) * pn.ldmask + n) : 0.f;
#pragma unroll
        for (int j = 0; j < RB; ++j) {
          if (b0 + j < b_hi) {
            float gsum = 0.f;
#pragma unroll
            for (int m = 0; m < AMAX; ++m) {
              const float g = gs[(b0 + j) * AMAX + m];
              gsum = fmaf(g, w[m], gsum);
              dw[m] = fmaf(g, hv[j], dw[m]);
            }
            const float o = (hv[j] > 0.f) ? gsum * dscale : 0.f;
            csum += o;
            pn.C[(int64_t)(b0 + j) * pn.ldc + n] = ctx.tf32 ? round_tf32(o) : o;
          }
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < AMAX; ++m) red[(bg * 64 + tn) * AMAX + m] = dw[m];
  __shared__ float cred[4][64];
  cred[bg][tn] = csum;
  __syncthreads();
  if (bg == 0 && n < H) {
#pragma unroll
    for (int m = 0; m < AMAX; ++m) {
      if (m < AO) {
        const float s = ((red[(0 * 64 + tn) * AMAX + m] + red[(1 * 64 + tn) * AMAX + m]) +
                         red[(2 * 64 + tn) * AMAX + m]) + red[(3 * 64 + tn) * AMAX + m];
        pw.C[(int64_t)m * pw.ldc + n] = s;
      }
    }
    if (dbias_prev != nullptr) dbias_prev[n] = ((cred[0][tn] + cred[1][tn]) + cred[2][tn]) + cred[3][tn];
  }
  if (blockIdx.y == 0 && pw.dbias != nullptr && threadIdx.x < AO) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += gs[b * AMAX + threadIdx.x];
    pw.dbias[threadIdx.x] = s;
  }
}

// Vectorised variant for A_out <= 8 and H % 4 == 0: a thread owns 4 consecutive columns (16-byte loads of H_L,
// 16-byte stores of G_{L-1}); 256 threads = 64 column quads (256 columns) x 4 row groups, so at H = 256 one CTA
// covers a whole problem: the loss gradients are staged once and every thread streams 64 rows.
// Loss gradients of one batch row for training-net slot t (0 V, 1 q1, 2 q2, 3 actor): the same expressions, in the
// same order, as loss_kernel (kernels_simt.cu), which keeps producing the logged losses, the log_std gradient and
// the global gy / gpi copies -- off the critical path, on the side stream -- while this kernel no longer waits
// for it.  g[a], a < AMAX; entries >= the head width are 0.
template <int AMAX>
__device__ __forceinline__ void loss_row_grads(const StepCtx& ctx, const MemberScalars& sc, const float* __restrict__ w,
                                               const WorkspaceLayout& wl, const float* __restrict__ log_std, int t, int b,
                                               float* g) {
  const int B = ctx.B, RF = ctx.row.row_floats;
#pragma unroll
  for (int a = 0; a < AMAX; ++a) g[a] = 0.f;
  if (b >= sc.batch) return;  // pad row of a member with B_m < B: zero gradient (loss_kernel)
  const float* yq = w + wl.yq;
  const float inv_b = 1.0f / (float)sc.batch;
  const float v = yq[PASS_V * B + b];
  const float tq = fminf(yq[PASS_TQ1 * B + b], yq[PASS_TQ2 * B + b]);
  const float adv = tq - v;
  if (t == 0) {  // V (expectile)
    const float w_neg = fabsf(sc.iql_tau - 1.0f), w_pos = fabsf(sc.iql_tau);
    const float wt = adv < 0.f ? w_neg : w_pos;
    g[0] = -((wt * inv_b) * (2.0f * adv));
  } else if (t <= 2) {  // Q (TD)
    const float* xr = w + wl.xrow + (int64_t)b * RF;
    const float next_v = yq[PASS_V_NEXT * B + b];
    const float q = yq[(t == 1 ? PASS_Q1 : PASS_Q2) * B + b];
    const float r = xr[ctx.row.off_reward], d = xr[ctx.row.off_done];
    const float target = r + ((1.0f - d) * sc.discount) * next_v;
    const float dq = q - target;
    g[0] = dq * (2.0f * inv_b) * 0.5f;
  } else {  // policy (AWR)
    const float* xr = w + wl.xrow + (int64_t)b * RF;
    const float* zpi = w + wl.zpi;
    const float e = fminf(expf(sc.beta * adv), 100.0f);
    const float eb = e * inv_b;
    const bool gauss = !ctx.deterministic;
#pragma unroll
    for (int a = 0; a < AMAX; ++a) {
      if (a < ctx.A_dim) {
        const float mu = tanhf(zpi[(int64_t)b * wl.Ald + a]);
        const float act = xr[ctx.row.off_action + a];
        float gmu;
        if (!gauss) {
          const float diff = mu - act;
          gmu = eb * (2.0f * diff);
        } else {
          const float ls = fminf(fmaxf(log_std[a], -20.0f), 2.0f);
          const float sd = expf(ls);
          const float var = sd * sd;
          const float diff = act - mu;
          gmu = -eb * diff / var;
        }
        g[a] = gmu * (1.0f - mu * mu);
      }
    }
  }
}

// ws != null: the G tile comes from loss_row_grads (problem index % 4 = training-net slot, the table order of the
// engine) instead of the gy / gpi arrays loss_kernel writes.
template <int AMAX>
__global__ void __launch_bounds__(256) last_bwd_v4_kernel(const GemmProb* __restrict__ probs_dgrad,
                                                          const GemmProb* __restrict__ probs_wgrad,
                                                          const GemmProb* __restrict__ probs_prev_wgrad, StepCtx ctx,
                                                          const float* __restrict__ ws, int64_t ws_member_floats,
                                                          WorkspaceLayout wl, const float* __restrict__ params, int sel_n,
                                                          int sel_off) {
  extern __shared__ float sm[];  // G tile [B][AMAX], then reduction scratch [4 row groups][256 columns][AMAX + 1]
  stamp_begin(ctx.stamps, ST_LASTBWD);
  pdl_trigger();
  const int pi = sel_n > 0 ? (int)(blockIdx.x / sel_n) * 4 + sel_off + (int)(blockIdx.x % sel_n) : (int)blockIdx.x;
  const GemmProb pn = probs_dgrad[pi];
  const GemmProb pw = probs_wgrad[pi];
  float* dbias_prev = probs_prev_wgrad ? probs_prev_wgrad[pi].dbias : nullptr;
  pdl_wait();  // the static problem tables are read above; the forward's outputs below
  const int B = pn.M, H = pn.N, AO = pn.K;
  float* gs = sm;
  float* red = sm + (size_t)B * AMAX;
  if (ws != nullptr) {
    const MemberScalars msc = ctx.scalars[pn.member];
    const float* wmem = ws + (int64_t)pn.member * ws_member_floats;
    const float* log_std = params + (int64_t)pn.member * ctx.P + ctx.log_std_off;
    const int t = pi & 3;
    for (int b = threadIdx.x; b < B; b += 256) {
      float g[AMAX];
      loss_row_grads<AMAX>(ctx, msc, wmem, wl, log_std, t, b + pn.row0, g);
#pragma unroll
      for (int a = 0; a < AMAX; ++a) gs[b * AMAX + a] = g[a];
    }
  } else {
    for (int i = threadIdx.x; i < B * AMAX; i += 256) {
      const int b = i / AMAX, m = i - b * AMAX;
      gs[i] = (m < AO) ? pn.A[(int64_t)b * pn.lda + m] : 0.f;
    }
  }
  const int tq = threadIdx.x & 63, bg = threadIdx.x >> 6;
  const int n = blockIdx.y * 256 + tq * 4;  // first of this thread's 4 columns
  const bool act = n < H;                  // H % 4 == 0: all four or none
  float4 w[AMAX], dw[AMAX];
#pragma unroll
  for (int m = 0; m < AMAX; ++m) {
    w[m] = (m < AO && act) ? *reinterpret_cast<const float4*>(pn.B + (int64_t)m * pn.ldb + n) : make_float4(0.f, 0.f, 0.f, 0.f);
    dw[m] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const MemberScalars* sc = ctx.scalars + pn.member;
  const float dscale = (pn.drop_layer >= 0 && sc->drop_threshold != 0u) ? sc->drop_scale : 1.0f;
  const bool tf32 = ctx.tf32 != 0;
  __syncthreads();
  const int rows_per = (B + 3) / 4;
  const int b_lo = bg * rows_per, b_hi = min(B, b_lo + rows_per);
  float4 csum = make_float4(0.f, 0.f, 0.f, 0.f);
  if (act) {
    constexpr int RB = 8;
    for (int b0 = b_lo; b0 < b_hi; b0 += RB) {
      float4 hv[RB];
#pragma unroll
      for (int j = 0; j < RB; ++j)
        hv[j] = (b0 + j < b_hi) ? __ldg(reinterpret_cast<const float4*>(pn.mask + (int64_t)(b0 + j) * pn.ldmask + n))
                                : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < RB; ++j) {
        if (b0 + j < b_hi) {
          float4 gsum = make_float4(0.f, 0.f, 0.f, 0.f);
          if (AO == 1) {  // scalar heads (Q, V): uniform per CTA
            const float g = gs[(b0 + j) * AMAX];
            gsum.x = g * w[0].x; gsum.y = g * w[0].y; gsum.z = g * w[0].z; gsum.w = g * w[0].w;
            dw[0].x = fmaf(g, hv[j].x, dw[0].x); dw[0].y = fmaf(g, hv[j].y, dw[0].y);
            dw[0].z = fmaf(g, hv[j].z, dw[0].z); dw[0].w = fmaf(g, hv[j].w, dw[0].w);
          } else {
#pragma unroll
            for (int m = 0; m < AMAX; ++m) {
              const float g = gs[(b0 + j) * AMAX + m];
              gsum.x = fmaf(g, w[m].x, gsum.x); gsum.y = fmaf(g, w[m].y, gsum.y);
              gsum.z = fmaf(g, w[m].z, gsum.z); gsum.w = fmaf(g, w[m].w, gsum.w);
              dw[m].x = fmaf(g, hv[j].x, dw[m].x); dw[m].y = fmaf(g, hv[j].y, dw[m].y);
              dw[m].z = fmaf(g, hv[j].z, dw[m].z); dw[m].w = fmaf(g, hv[j].w, dw[m].w);
            }
          }
          float4 o;
          o.x = (hv[j].x > 0.f) ? gsum.x * dscale : 0.f; o.y = (hv[j].y > 0.f) ? gsum.y * dscale : 0.f;
          o.z = (hv[j].z > 0.f) ? gsum.z * dscale : 0.f; o.w = (hv[j].w > 0.f) ? gsum.w * dscale : 0.f;
          csum.x += o.x; csum.y += o.y; csum.z += o.z; csum.w += o.w;
          if (tf32) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
          *reinterpret_cast<float4*>(pn.C + (int64_t)(b0 + j) * pn.ldc + n) = o;
        }
      }
    }
  }
  // reduce the 4 row groups in a fixed order: red[bg][column][m], column = 4 tq + i; slot AMAX holds csum
  constexpr int RS = AMAX + 1;
#pragma unroll
  for (int m = 0; m < AMAX; ++m) {
    red[(bg * 256 + tq * 4 + 0) * RS + m] = dw[m].x; red[(bg * 256 + tq * 4 + 1) * RS + m] = dw[m].y;
    red[(bg * 256 + tq * 4 + 2) * RS + m] = dw[m].z; red[(bg * 256 + tq * 4 + 3) * RS + m] = dw[m].w;
  }
  red[(bg * 256 + tq * 4 + 0) * RS + AMAX] = csum.x; red[(bg * 256 + tq * 4 + 1) * RS + AMAX] = csum.y;
  red[(bg * 256 + tq * 4 + 2) * RS + AMAX] = csum.z; red[(bg * 256 + tq * 4 + 3) * RS + AMAX] = csum.w;
  __syncthreads();
  for (int i = threadIdx.x; i < 256 * RS; i += 256) {  // one (column, m) sum per thread-iteration
    const int col = i / RS, m = i - col * RS;
    const int nn = blockIdx.y * 256 + col;
    if (nn >= H) continue;
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < 4; ++g) s += red[(g * 256 + col) * RS + m];
    if (m < AO) pw.C[(int64_t)m * pw.ldc + nn] = s;
    else if (m == AMAX && dbias_prev != nullptr) dbias_prev[nn] = s;
  }
  if (blockIdx.y == 0 && pw.dbias != nullptr && threadIdx.x < AO) {
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += gs[b * AMAX + threadIdx.x];
    pw.dbias[threadIdx.x] = s;
  }
  stamp_end(ctx.stamps, ST_LASTBWD);
}

// The vectorised kernel covers 256 columns x ALL batch rows per CTA: with few problems and a large batch (stress
// shape: 4 problems x 4096 rows x 1024 columns = 16 CTAs) it leaves the GPU empty; the generic kernel then has 4x
// the CTAs (64 columns each) and measured 3x faster.
static bool last_bwd_v4_fills(int nprob, int B, int H) { return !(B >= 2048 && (int64_t)nprob * ((H + 255) / 256) < 64); }

bool last_bwd_recomputes_loss_grads(int H, int amax, int nprob, int B) {
  return dbg_getenv("IQL_B200_NO_LASTBWD_V4") == nullptr && dbg_getenv("IQL_B200_NO_LOSS_OVERLAP") == nullptr && (H % 4) == 0 && amax <= 8 &&
         last_bwd_v4_fills(nprob, B, H);
}

int launch_last_bwd(const GemmProb* probs_dgrad, const GemmProb* probs_wgrad, const GemmProb* probs_prev_wgrad,
                     int nprob, int B, int H, int amax, const StepCtx& ctx, cudaStream_t st, const float* ws,
                     int64_t ws_member_floats, const WorkspaceLayout* wl, const float* params) {
  dim3 grid(nprob, (H + 63) / 64);
  auto smem = [&](int a) { return ((size_t)B * a + 4 * 64 * a) * sizeof(float); };
  auto smem4 = [&](int a) { return ((size_t)B * a + 4 * 256 * (a + 1)) * sizeof(float); };
  static bool attr[64] = {};
  static bool no_v4 = false;
  if (first_use_on_device(attr)) {
    cudaFuncSetAttribute(last_bwd_kernel<24>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(last_bwd_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(last_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(last_bwd_v4_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(last_bwd_v4_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    no_v4 = dbg_getenv("IQL_B200_NO_LASTBWD_V4") != nullptr;
  }
  const bool v4 = !no_v4 && (H % 4) == 0 && amax <= 8 && smem4(8) <= 200 * 1024 && last_bwd_v4_fills(nprob, B, H);
  const dim3 grid4(nprob, (H + 255) / 256);
  WorkspaceLayout wlv;
  memset(&wlv, 0, sizeof(wlv));
  if (wl) wlv = *wl;
  const float* wsp = (wl && nprob % 4 == 0) ? ws : nullptr;  // 4 training nets per member, in table order
  if (v4 && amax <= 1)
    launch_pdl(last_bwd_v4_kernel<1>, grid4, dim3(256), smem4(1), st, 1, probs_dgrad, probs_wgrad, probs_prev_wgrad, ctx, wsp,
               ws_member_floats, wlv, params, 0, 0);
  else if (v4)
    launch_pdl(last_bwd_v4_kernel<8>, grid4, dim3(256), smem4(8), st, 1, probs_dgrad, probs_wgrad, probs_prev_wgrad, ctx, wsp,
               ws_member_floats, wlv, params, 0, 0);
  else if (amax <= 1) last_bwd_kernel<1><<<grid, 256, smem(1), st>>>(probs_dgrad, probs_wgrad, probs_prev_wgrad, ctx, 0, 0);
  else if (amax <= 8) last_bwd_kernel<8><<<grid, 256, smem(8), st>>>(probs_dgrad, probs_wgrad, probs_prev_wgrad, ctx, 0, 0);
  else if (!no_v4 && (H % 4) == 0 && nprob % 4 == 0 && wl != nullptr && smem4(1) <= 200 * 1024) {
    // wide policy head (pen: 24 actions): the three scalar-head nets of every member (V, Q1, Q2: problems 0..2 of each
    // group of 4, table order) take the vectorised kernel, only the actor (problem 3) the generic one
    launch_pdl(last_bwd_v4_kernel<1>, dim3(nprob / 4 * 3, (H + 255) / 256), dim3(256), smem4(1), st, 1, probs_dgrad, probs_wgrad,
               probs_prev_wgrad, ctx, (const float*)nullptr, ws_member_floats, wlv, params, 3, 0);
    last_bwd_kernel<24><<<dim3(nprob / 4, (H + 63) / 64), 256, smem(24), st>>>(probs_dgrad, probs_wgrad, probs_prev_wgrad, ctx, 1, 3);
    return 2;
  } else last_bwd_kernel<24><<<grid, 256, smem(24), st>>>(probs_dgrad, probs_wgrad, probs_prev_wgrad, ctx, 0, 0);
  return 1;  // kernels launched
}

__global__ void __launch_bounds__(256) lb_reduce_kernel(const GemmProb* __restrict__ pw_split, const GemmProb* __restrict__ prev_split,
                                                        const GemmProb* __restrict__ pw, const GemmProb* __restrict__ prev, int nprob,
                                                        int splits) {
  const int i = blockIdx.x;
  const GemmProb o = pw[i];
  const int R = o.M, W = o.N, ld = o.ldc;  // dW is [R][W] with leading dimension ld in the output and in every partial
  const int n_dw = R * W, n_all = n_dw + R + (prev ? W : 0);
  for (int e = blockIdx.y * 256 + threadIdx.x; e < n_all; e += gridDim.y * 256) {
    float s = 0.f;
    if (e < n_dw) {
      const int a = e / W, n = e - a * W;
      for (int k = 0; k < splits; ++k) s += pw_split[k * nprob + i].C[(int64_t)a * ld + n];
      o.C[(int64_t)a * ld + n] = s;
    } else if (e < n_dw + R) {
      if (o.dbias != nullptr) {
        for (int k = 0; k < splits; ++k) s += pw_split[k * nprob + i].dbias[e - n_dw];
        o.dbias[e - n_dw] = s;
      }
    } else {
      float* dst = prev[i].dbias;
      if (dst != nullptr) {
        for (int k = 0; k < splits; ++k) s += prev_split[k * nprob + i].dbias[e - n_dw - R];
        dst[e - n_dw - R] = s;
      }
    }
  }
}

void launch_lb_reduce(const GemmProb* pw_split, const GemmProb* prev_split, const GemmProb* pw, const GemmProb* prev, int nprob,
                      int splits, cudaStream_t st) {
  lb_reduce_kernel<<<dim3(nprob, 8), 256, 0, st>>>(pw_split, prev_split, pw, prev, nprob, splits);
}

// ---------------------------------------------------------------------------
// first layer weight gradient.  grid (nprob, ceil(H/(SLOTS*NC))), NT threads = SLOTS column slots x 4 row groups,
// NC columns per thread (the X row fetched from shared memory is reused NC times).
//   p: TN problem (A = G_0 [B][H] (K = B rows, M = H), B = X [B][ldx] (N = K0), C = dW_0 [H][K0], dbias = db_0)
// Sized so that the whole launch is ONE wave at the reference's shapes (KMAX = 24: 1024 CTAs of 128 threads, 7 per
// SM): with 512 larger CTAs the second, 15 % full wave doubled the kernel time.
// ---------------------------------------------------------------------------
template <int KMAX, int NC, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) first_wgrad_kernel(const GemmProb* __restrict__ probs) {
  extern __shared__ float sm[];  // X [B][KMAX]; afterwards the reduction scratch [4][SLOTS*NC][KMAX + 1] in the same bytes
  const GemmProb p = probs[blockIdx.x];
  const int B = p.K, H = p.M, K0 = p.N;
  constexpr int SLOTS = NT / 4;
  constexpr int CW = SLOTS * NC;  // columns per CTA
  float* xs = sm;
  float* red = sm;  // aliases xs once the main loop is done
  // X rows are 16-byte aligned and ldb is a multiple of 4: float4 loads, columns >= K0 (the next fields of the
  // replay row) zeroed
  for (int i = threadIdx.x; i < B * (KMAX / 4); i += NT) {
    const int b = i / (KMAX / 4), k4 = (i - b * (KMAX / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (k4 < K0 && k4 + 4 <= p.ldb) v = __ldg(reinterpret_cast<const float4*>(p.B + (int64_t)b * p.ldb + k4));
    if (k4 + 0 >= K0) v.x = 0.f;
    if (k4 + 1 >= K0) v.y = 0.f;
    if (k4 + 2 >= K0) v.z = 0.f;
    if (k4 + 3 >= K0) v.w = 0.f;
    *reinterpret_cast<float4*>(&xs[b * KMAX + k4]) = v;
  }
  const int tn = threadIdx.x % SLOTS, bg = threadIdx.x / SLOTS;
  const int n0 = blockIdx.y * CW + tn;
  float acc[NC][KMAX];
  float bsum[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    bsum[c] = 0.f;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) acc[c][k] = 0.f;
  }
  __syncthreads();
  const int rows_per = (B + 3) / 4;
  const int b_lo = bg * rows_per, b_hi = min(B, b_lo + rows_per);
  // RU rows per trip with all their G loads issued before the first FMA: the loop is bound by the latency of the
  // (coalesced) G reads, so what matters is how many of them each thread keeps in flight
  constexpr int RU = MINB >= 4 ? 4 : 8;
  for (int b = b_lo; b < b_hi; b += RU) {
    float g[RU][NC];
#pragma unroll
    for (int r = 0; r < RU; ++r)
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const int n = n0 + c * SLOTS;
        g[r][c] = (b + r < b_hi && n < H) ? __ldg(&p.A[(int64_t)(b + r) * p.lda + n]) : 0.f;
      }
#pragma unroll
    for (int r = 0; r < RU; ++r) {
      const int br = min(b + r, B - 1);  // rows past b_hi carry g = 0
#pragma unroll
      for (int c = 0; c < NC; ++c) bsum[c] += g[r][c];
#pragma unroll
      for (int k4 = 0; k4 < KMAX; k4 += 4) {
        const float4 x = *reinterpret_cast<const float4*>(&xs[br * KMAX + k4]);
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          acc[c][k4] = fmaf(g[r][c], x.x, acc[c][k4]);
          acc[c][k4 + 1] = fmaf(g[r][c], x.y, acc[c][k4 + 1]);
          acc[c][k4 + 2] = fmaf(g[r][c], x.z, acc[c][k4 + 2]);
          acc[c][k4 + 3] = fmaf(g[r][c], x.w, acc[c][k4 + 3]);
        }
      }
    }
  }
  __syncthreads();  // the reduction scratch reuses the X tile
  constexpr int RS = KMAX + 1;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    float* mine = red + (size_t)(bg * CW + c * SLOTS + tn) * RS;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) mine[k] = acc[c][k];
    mine[KMAX] = bsum[c];
  }
  __syncthreads();
  // the CTA cooperatively finishes the CW x (K0 + 1) outputs of this column block (fixed order)
  for (int i = threadIdx.x; i < CW * RS; i += NT) {
    const int c = i / RS, k = i - c * RS;
    const int nn = blockIdx.y * CW + c;
    if (nn >= H) continue;
    const float s = ((red[(size_t)(0 * CW + c) * RS + k] + red[(size_t)(1 * CW + c) * RS + k]) +
                     red[(size_t)(2 * CW + c) * RS + k]) + red[(size_t)(3 * CW + c) * RS + k];
    if (k < K0) p.C[(int64_t)nn * p.ldc + k] = s;
    else if (k == KMAX && p.dbias != nullptr) p.dbias[nn] = s;
  }
}

void launch_first_wgrad(const GemmProb* probs, int nprob, int B, int H, int kmax, cudaStream_t st) {
  auto smem = [&](int k, int cw) { return std::max((size_t)B * k, (size_t)4 * cw * (k + 1)) * sizeof(float); };
  static bool attr[64] = {};
  if (first_use_on_device(attr)) {
    cudaFuncSetAttribute(first_wgrad_kernel<24, 2, 128, 7>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(first_wgrad_kernel<40, 2, 256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(first_wgrad_kernel<72, 1, 256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  }
  if (kmax <= 24) first_wgrad_kernel<24, 2, 128, 7><<<dim3(nprob, (H + 63) / 64), 128, smem(24, 64), st>>>(probs);
  else if (kmax <= 40) first_wgrad_kernel<40, 2, 256, 1><<<dim3(nprob, (H + 127) / 128), 256, smem(40, 128), st>>>(probs);
  else first_wgrad_kernel<72, 1, 256, 1><<<dim3(nprob, (H + 63) / 64), 256, smem(72, 64), st>>>(probs);
}

}  // namespace iql

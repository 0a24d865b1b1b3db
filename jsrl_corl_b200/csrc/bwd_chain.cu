// Chained backward + optimizer of the IQL step on CTA pairs (IQL_MATH_TF32_TCGEN05, hidden width 256, batch 256).
// sm_100a only.
//
// One CTA pair owns one (member, trainable network) task and runs its hidden-layer backward as a chain of tcgen05
// GEMM phases without leaving the kernel -- reference: loss.backward() + optimizer.step() + soft_update of
// algorithms/finetune/iql.py:491-494, 509-515, 536-540 --
//
//     for l = L-1 .. 1:   dZ_{l-1} = (dZ_l W_l) * [H_l > 0]           dgrad  (sign-bit mask, TMA store, db_{l-1} = column sums)
//                         W_l     <- Adam(W_l, dZ_l^T H_l)            wgrad  with the OPTIMIZER IN THE EPILOGUE
//     W_0 <- Adam(W_0, dZ_0^T X)                                       input-layer wgrad, optimizer in the epilogue
//     biases, output layer, log_std <- Adam(...)                       from the gradients the output-layer backward wrote
//
// dZ_{L-1}, dW_L, db_L, db_{L-1} come from the output-layer backward kernel that precedes this launch.  The weight
// gradients of the big matrices never exist in memory: the FP32 accumulator of a wgrad phase is read from tensor
// memory, transposed through a per-warp staging tile and consumed by adam_quad() together with the parameter, its
// two moments (and the target network for the Q nets, Polyak with the post-Adam weights) in coalesced 16-byte
// accesses.  This replaces four launches (hidden dgrad, hidden wgrad, input-layer wgrad, adam_polyak) and removes
// the gradient arena round trip and the re-read of dZ from HBM by three different kernels (the pair that wrote a
// dZ tile reads it back from L2 microseconds later).
//
// Structure = umma_gemm.cu's CTA-pair kernel with a heterogeneous phase list per work unit: warp 0 lane 0 TMA
// producer, warp 1 lane 0 MMA issuer (leader CTA), warps 2-17 epilogue; 4-stage ring of 32 KB stages; two 256-column
// accumulators, so the (long, memory-bound) optimizer epilogue of one phase overlaps the main loop of the next.
// The only intra-task dependency through memory is dgrad -> consumers of its dZ output: every epilogue warp of
// BOTH CTAs waits for its TMA stores to complete and arrives (release.cluster) on the `gready` barrier of both CTAs;
// the producers wait on it (acquire.cluster + fence.proxy.async) before the first load that depends on it.
// W_l is overwritten by the wgrad_l epilogue only after the MMAs of dgrad_l (issued earlier, completed in order) have
// consumed the shared-memory copy of the old W_l.
//
// Gradient-only mode (grads_only, IQL_OPT_STEP_PATH = 4): the wgrad epilogues store the FP32 weight gradients from the
// staging tile to the grads arena (16-byte stores, exact zeros in the row padding of the input layer, as the per-phase
// kernels write them) and the task-end small-parameter pass is skipped; adam_polyak_kernel runs after the launch.
// The epilogue streams at the HBM rate of a plain store instead of the 72 % the in-epilogue optimizer reaches
// (DESIGN.md section 8), and the chain keeps what it is good at: one launch for the hidden-layer backward, every dZ
// read back from L2 by the pair that wrote it.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "adam.cuh"
#include "common.cuh"
#include "tcgen05.cuh"
#include "umma_gemm.h"

namespace iql {

namespace {

constexpr int C_TILE_M = 128, C_TILE_K = 32, C_UMMA_K = 8, C_STAGES = 4;
constexpr int C_STAGE_A = C_TILE_M * C_TILE_K * 4;  // 16 KB: this CTA's 128 rows (or 128 M-columns) of A
constexpr int C_STAGE_B = 128 * C_TILE_K * 4;       // 16 KB: this CTA's half of the B tile (N <= 256)
constexpr int C_STAGE = C_STAGE_A + C_STAGE_B;
constexpr int C_RING = C_STAGES * C_STAGE;
constexpr int C_EPI_WARPS = 16, C_CGROUPS = 4;
constexpr int C_STG_BYTES = 5120;  // per-warp staging: 32 x 36 floats (transposing epilogue) or a swizzled 32 x 32 box
constexpr int C_AUX_BYTES = 4 * 256 * 4;  // bias-gradient sums [4 lane quarters][256]
constexpr int C_PEER_SLOTS = 3;
constexpr int C_EPI_SMEM = C_EPI_WARPS * C_STG_BYTES + C_AUX_BYTES + C_PEER_SLOTS * 4 * 256 * 4;
constexpr int C_SMEM = C_RING + C_EPI_SMEM + 1024 /*align*/ + 512 /*barriers*/;
constexpr int C_THREADS = 576;
constexpr int C_MAX_PHASES = 2 * FUSED_MAX_LAYERS;
constexpr int C_MAX_SEG = FUSED_MAX_LAYERS + 2;

enum { CH_DGRAD = 0, CH_WGRAD = 1 };

struct ChainPhase {
  int kind;         // CH_DGRAD / CH_WGRAD
  int prob_first;   // the phase's first problem in the engine's table; task i uses prob_first + i
  int map_first;    // first tensor map of the phase in the chain map table (2 per task: A, B)
  int tile_n;       // UMMA N: 256, or 64 / 128 for the input-layer weight gradient
  int nkb;          // k-blocks of 32
  int wait_dgrads;  // dgrad epilogues of this task that must have completed before the phase's first load
  int a_mn, b_mn;   // operand majors (0 K-major, 1 MN-major)
  uint32_t idesc;
};

struct ChainParams {
  int n_phases, n_dgrad, n_tasks, keep_grads, grads_only;
  int db_tile_order;  // gradient-only: bias gradients in the summation order of the single-CTA per-phase dgrad
  ChainPhase ph[C_MAX_PHASES];
  // parameters the phases do not cover (biases, output layer, log_std), per network slot (V, q1, q2, actor):
  // flat ranges [lo, hi) inside a member block, multiples of 4 floats
  int n_seg[4];
  long long seg_lo[4][C_MAX_SEG], seg_hi[4][C_MAX_SEG];
  int dbg;           // IQL_CHAIN_DBG timing probes (results are WRONG when set): 1 no optimizer math / stores, 2 no state loads
  long long* trace;  // IQL_CHAIN_TRACE: globaltimer stamps of pair 0, [3 roles][C_TRACE_TASKS][C_MAX_PHASES + 1][4]
};

constexpr int C_TRACE_TASKS = 4;
constexpr int C_TRACE_WORDS = 3 * C_TRACE_TASKS * (C_MAX_PHASES + 1) * 4;

__device__ __forceinline__ void ctrace(const ChainParams& cp, int role, int task_it, int pi, int slot) {
  if (cp.trace && blockIdx.x == 0 && task_it < C_TRACE_TASKS) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    cp.trace[((role * C_TRACE_TASKS + task_it) * (C_MAX_PHASES + 1) + pi) * 4 + slot] = t;
  }
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p) : "memory"); }

// Optimizer on NB row groups (4 rows each, one per lane octet) x 4 columns per lane of a staged 32 x 32 gradient chunk.
// All state loads of the batch are issued before the first dependent instruction; NB is chosen so that they fit the
// 96-register budget of the kernel without spilling (4 x 3 float4 for V / actor, 2 x 4 float4 for the Q nets with
// their target): spilled loads serialise on the scoreboard, which cost 6 us per batch in the first version.
template <int NB, bool Q>
__device__ __forceinline__ void adam_rows(const StepCtx& ctx, const float* __restrict__ stg, int rl0, int lr, int lc, int col,
                                          int ncols, int member, int64_t idx0, int istep, int64_t mo, int64_t to,
                                          float neg_step, float inv_bc2, float a_w1, float a_b2, float a_1mb2, float a_eps,
                                          float tau, float omt, bool first_layer, int keep_grads, int dbg,
                                          float* __restrict__ params, float* __restrict__ exp_avg,
                                          float* __restrict__ exp_avg_sq, float* __restrict__ target, float* __restrict__ grads) {
  float4 p4[NB], m4[NB], v4[NB], t4[NB];
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    const int64_t ix = idx0 + i * istep;
    t4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (dbg & 2) { p4[i] = m4[i] = v4[i] = t4[i]; continue; }
    p4[i] = __ldcs(reinterpret_cast<const float4*>(params + mo + ix));
    m4[i] = __ldcs(reinterpret_cast<const float4*>(exp_avg + mo + ix));
    v4[i] = __ldcs(reinterpret_cast<const float4*>(exp_avg_sq + mo + ix));
    if (Q) t4[i] = __ldcs(reinterpret_cast<const float4*>(target + to + ix));
  }
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    const int64_t ix = idx0 + i * istep;
    float4 g4 = *reinterpret_cast<const float4*>(&stg[(rl0 + 4 * i + lr) * 36 + lc]);
    if (col + 3 >= ncols) {  // row padding of the input-layer weights stays exactly zero
      if (col >= ncols) g4.x = 0.f;
      if (col + 1 >= ncols) g4.y = 0.f;
      if (col + 2 >= ncols) g4.z = 0.f;
      g4.w = 0.f;
    }
    if (keep_grads) *reinterpret_cast<float4*>(grads + mo + ix) = g4;
    if (dbg & 1) {
      if (p4[i].x + m4[i].y + v4[i].z + t4[i].w + g4.x == 1234.5f) params[0] = 0.f;  // keep the loads alive
      continue;
    }
    adam_quad_fast(ctx, member, ix, g4, p4[i], m4[i], v4[i], t4[i], neg_step, inv_bc2, a_w1, a_b2, a_1mb2, a_eps, tau, omt,
                   first_layer, params, exp_avg, exp_avg_sq, target);
  }
}

__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

// (18 warps = 5 on two of the four schedulers: 16384 / 5 / 32 = 102 registers per thread at most -> ptxas settles on 96)
// GRADS_ONLY: gradient-only instance (ChainParams::grads_only), compiled without the optimizer code
template <bool GRADS_ONLY>
__global__ void __launch_bounds__(C_THREADS, 1)
bwd_chain_kernel(const GemmProb* __restrict__ probs, const CUtensorMap* __restrict__ maps, const CUtensorMap* __restrict__ cmaps,
                 const ChainParams cp, const StepCtx ctx, float* __restrict__ params, float* __restrict__ exp_avg,
                 float* __restrict__ exp_avg_sq, float* __restrict__ target, float* __restrict__ grads) {
  extern __shared__ uint8_t smem_raw[];
  // step timeline: gradient-only instance only (the stamp registers push the fused-optimizer instance into spills)
  if (GRADS_ONLY) stamp_begin(ctx.stamps, ST_CHAIN);
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  uint8_t* epi_smem = smem + C_RING;
  float* csum_s = reinterpret_cast<float*>(epi_smem + C_EPI_WARPS * C_STG_BYTES);            // [4][256]
  float* peer_csum = reinterpret_cast<float*>(epi_smem + C_EPI_WARPS * C_STG_BYTES + C_AUX_BYTES);  // [3][4][256]
  // barriers: full[4] empty[4] tfull[2] tempty[2] csfull[3] gready | tmem slot
  const uint32_t bars = base + C_RING + C_EPI_SMEM;
  const uint32_t full0 = bars, empty0 = bars + 8 * C_STAGES, tfull0 = bars + 16 * C_STAGES, tempty0 = tfull0 + 16;
  const uint32_t csfull0 = tempty0 + 16, gready = csfull0 + 8 * C_PEER_SLOTS, tslot = gready + 8;
  volatile uint32_t* tslot_ptr = reinterpret_cast<volatile uint32_t*>(smem + C_RING + C_EPI_SMEM + (tslot - bars));
  const uint32_t rank = cluster_ctarank();
  const int worker = (int)(blockIdx.x >> 1), n_workers = (int)(gridDim.x >> 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < C_STAGES; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull0 + 8 * b, 1);
      mbar_init(tempty0 + 8 * b, 2 * C_EPI_WARPS);  // the epilogue warps of both CTAs release the leader's barrier
    }
    for (int b = 0; b < C_PEER_SLOTS; ++b) mbar_init(csfull0 + 8 * b, 256);
    mbar_init(gready, 2 * C_EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tslot), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *tslot_ptr;
  pdl_wait();  // dZ_{L-1} and the small gradients come from the output-layer backward launched before this kernel

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, gpar = 0;
      const uint32_t full0_lead = mapa_u32(full0, 0);
      int task_it = 0;
      for (int u = worker; u < cp.n_tasks; u += n_workers, ++task_it) {
        int gseen = 0;
        for (int pi = 0; pi < cp.n_phases; ++pi) {
          const ChainPhase& ph = cp.ph[pi];
          ctrace(cp, 0, task_it, pi, 0);
          const CUtensorMap* mapA = maps + ph.map_first + 2 * u;
          const CUtensorMap* mapB = mapA + 1;
          asm volatile("prefetch.tensormap [%0];" ::"l"(mapA) : "memory");
          asm volatile("prefetch.tensormap [%0];" ::"l"(mapB) : "memory");
          while (gseen < ph.wait_dgrads) {  // a dZ this phase loads was written by a dgrad epilogue of this task
            mbar_wait_cluster(gready, gpar);
            gpar ^= 1u;
            ++gseen;
            fence_proxy_async_all();
          }
          ctrace(cp, 0, task_it, pi, 1);
          const int b_rows = ph.tile_n >> 1;
          const uint32_t tx_bytes = 2u * (uint32_t)(C_STAGE_A + b_rows * C_TILE_K * 4);
          const int m0 = (int)rank * C_TILE_M, n0 = (int)rank * b_rows;
          for (int kb = 0; kb < ph.nkb; ++kb) {
            mbar_wait(empty0 + 8 * stage, phase ^ 1);
            const uint32_t sa = base + stage * C_STAGE, sb = sa + C_STAGE_A;
            const uint32_t fb = full0_lead + 8 * stage;
            const int k0 = kb * C_TILE_K;
            if (rank == 0) mbar_expect_tx(full0 + 8 * stage, tx_bytes);
            if (ph.a_mn) tma_load_3d_cg2(sa, mapA, fb, 0, k0, m0 >> 5);
            else tma_load_2d_cg2(sa, mapA, fb, k0, m0);
            if (ph.b_mn) tma_load_3d_cg2(sb, mapB, fb, 0, k0, n0 >> 5);
            else tma_load_2d_cg2(sb, mapB, fb, k0, n0);
            if (++stage == (uint32_t)C_STAGES) { stage = 0; phase ^= 1; }
          }
          ctrace(cp, 0, task_it, pi, 2);
        }
        while (gseen < cp.n_dgrad) {  // keep the barrier's phase parity in step with the epilogues
          mbar_wait_cluster(gready, gpar);
          gpar ^= 1u;
          ++gseen;
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (lane == 0 && rank == 0) {
      uint32_t stage = 0, phase = 0, it = 0;
      int task_it = 0;
      for (int u = worker; u < cp.n_tasks; u += n_workers, ++task_it)
        for (int pi = 0; pi < cp.n_phases; ++pi, ++it) {
          const ChainPhase& ph = cp.ph[pi];
          const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
          ctrace(cp, 1, task_it, pi, 0);
          mbar_wait(tempty0 + 8 * buf, acc_phase ^ 1);
          tc_fence_after();
          ctrace(cp, 1, task_it, pi, 1);
          const uint32_t tacc = tmem_base + buf * 256;
          // K-major SW128: SBO 1024 B, layout 2, K step 32 B; MN-major SW128/32B atoms: LBO 4096 B, SBO 512 B, layout 1,
          // K step 1024 B (umma_gemm.cu)
          const uint32_t a_lbo = ph.a_mn ? (4096u >> 4) : 1u, a_sbo = ph.a_mn ? (512u >> 4) : (1024u >> 4);
          const uint32_t a_lay = ph.a_mn ? 1u : 2u, a_ks = ph.a_mn ? (1024u >> 4) : (32u >> 4);
          const uint32_t b_lbo = ph.b_mn ? (4096u >> 4) : 1u, b_sbo = ph.b_mn ? (512u >> 4) : (1024u >> 4);
          const uint32_t b_lay = ph.b_mn ? 1u : 2u, b_ks = ph.b_mn ? (1024u >> 4) : (32u >> 4);
          for (int kb = 0; kb < ph.nkb; ++kb) {
            mbar_wait(full0 + 8 * stage, phase);
            tc_fence_after();
            if (kb == 0) ctrace(cp, 1, task_it, pi, 2);
            const uint32_t sa = base + stage * C_STAGE, sb = sa + C_STAGE_A;
            const uint64_t adesc0 = make_desc(sa, a_lbo, a_sbo, a_lay);
            const uint64_t bdesc0 = make_desc(sb, b_lbo, b_sbo, b_lay);
#pragma unroll
            for (int ks = 0; ks < C_TILE_K / C_UMMA_K; ++ks)
              umma_tf32_cg2(tacc, adesc0 + (uint64_t)(ks * a_ks), bdesc0 + (uint64_t)(ks * b_ks), ph.idesc, (kb | ks) != 0);
            umma_commit_cg2(empty0 + 8 * stage);
            if (++stage == (uint32_t)C_STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit_cg2(tfull0 + 8 * buf);
          ctrace(cp, 1, task_it, pi, 3);
        }
    }
  } else {
    // ===================== epilogue (warps 2..17) =====================
    const int q = warp & 3;          // TMEM lane quarter
    const int ch = (warp - 2) >> 2;  // column group: chunks ch, ch + 4
    uint8_t* stg_b = epi_smem + (warp - 2) * C_STG_BYTES;  // 1024-byte aligned (5120 = 5 * 1024)
    float* stg = reinterpret_cast<float*>(stg_b);
    const int lr = lane >> 3, lc = (lane & 7) * 4;
    const int et = threadIdx.x - 64;  // 0..511 among the epilogue threads
    uint32_t it = 0, dcount = 0;
    const uint32_t tempty0_lead = mapa_u32(tempty0, 0);
    const uint32_t gready_own = mapa_u32(gready, rank), gready_peer = mapa_u32(gready, rank ^ 1u);
    auto acc_release = [&](uint32_t buf) { mbar_arrive_cluster(tempty0_lead + 8 * buf); };
    const bool tracer = warp == 2 && lane == 0;
    int task_it = -1;
    for (int u = worker; u < cp.n_tasks; u += n_workers) {
      ++task_it;
      const int slot = u & 3;  // training-net slot of the task: 0 V, 1 q1, 2 q2, 3 actor (table order of the engine)
      int member = 0;
      for (int pi = 0; pi < cp.n_phases; ++pi, ++it) {
        const ChainPhase& ph = cp.ph[pi];
        const GemmProb p = probs[ph.prob_first + u];
        member = p.member;
        const uint32_t buf = it & 1, acc_phase = (it >> 1) & 1;
        const int n_chunks = ph.tile_n >> 5;
        const int row_base = (int)rank * C_TILE_M + q * 32;
        if (tracer) ctrace(cp, 2, task_it, pi, 0);
        if (ph.kind == CH_DGRAD) {
          // ---- row layout: lane = batch row; ReLU sign bits; TMA store; bias gradient of the layer below ----
          const MemberScalars* sc = ctx.scalars + p.member;
          const float dscale = (p.drop_layer >= 0 && sc->drop_threshold != 0u) ? sc->drop_scale : 1.0f;
          const int row = row_base + lane;
          const int nw = p.ldmask >> 5;
          uint32_t wbits[2];
#pragma unroll
          for (int i = 0; i < 2; ++i) wbits[i] = __ldg(p.bits + (int64_t)row * nw + ch + i * C_CGROUPS);
          mbar_wait(tfull0 + 8 * buf, acc_phase);
          tc_fence_after();
          if (tracer) ctrace(cp, 2, task_it, pi, 1);
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int c = ch + i * C_CGROUPS;
            uint32_t r[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 256 + c * 32), r);
            tmem_ld_wait();
            if (i == 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) acc_release(buf);
            }
            const uint32_t w = wbits[i];
#pragma unroll
            for (int j2 = 0; j2 < 32; ++j2)
              r[j2] = ((w >> j2) & 1u) ? __float_as_uint(round_tf32(__uint_as_float(r[j2]) * dscale)) : 0u;
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
#pragma unroll
            for (int j2 = 0; j2 < 8; ++j2)
              *reinterpret_cast<float4*>(&stg[lane * 32 + 4 * (j2 ^ (lane & 7))]) =
                  make_float4(__uint_as_float(r[4 * j2]), __uint_as_float(r[4 * j2 + 1]), __uint_as_float(r[4 * j2 + 2]),
                              __uint_as_float(r[4 * j2 + 3]));
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(cmaps + ph.prob_first + u, smem_u32(stg), c * 32, row_base);
              bulk_commit();
            }
            float cs = 0.f;  // column `lane` of the parked chunk over its 32 rows
#pragma unroll
            for (int rr = 0; rr < 32; ++rr) cs += stg[rr * 32 + 4 * ((lane >> 2) ^ (rr & 7)) + (lane & 3)];
            csum_s[q * 256 + c * 32 + lane] = cs;
          }
          // the dZ tile must be complete in memory before any consumer (this pair's producers) loads it
          if (lane == 0) {
            bulk_wait0();
            fence_proxy_async_all();
            mbar_arrive_cluster(gready_own);
            mbar_arrive_cluster(gready_peer);
          }
          // bias gradient: add the lane quarters, then the two CTAs (fixed order).  db_tile_order: the order of the
          // per-phase dgrad when it runs one CTA per problem (both 128-row M tiles in one CTA, quarter q of the second
          // tile added to quarter q of the first, then the quarters), so that the bias gradients match it bit for bit
          asm volatile("bar.sync 1, 512;" ::: "memory");
          if (GRADS_ONLY && cp.db_tile_order && et < 256) {
            const uint32_t cslot = dcount % C_PEER_SLOTS, par = (dcount / C_PEER_SLOTS) & 1u;
            float* pc = &peer_csum[cslot * 4 * 256 + et];
            if (rank != 0) {
#pragma unroll
              for (int qq = 0; qq < 4; ++qq) st_cluster_f32(mapa_u32(smem_u32(pc + qq * 256), 0), csum_s[qq * 256 + et]);
              mbar_arrive_cluster(mapa_u32(csfull0 + 8 * cslot, 0));
            } else {
              mbar_wait_cluster(csfull0 + 8 * cslot, par);
              float own = csum_s[et] + pc[0];
#pragma unroll
              for (int qq = 1; qq < 4; ++qq) own += csum_s[qq * 256 + et] + pc[qq * 256];
              if (p.dbias != nullptr && et < p.N) p.dbias[et] = own;
            }
          } else if (et < 256) {
            float own = ((csum_s[et] + csum_s[256 + et]) + csum_s[512 + et]) + csum_s[768 + et];
            const uint32_t cslot = dcount % C_PEER_SLOTS, par = (dcount / C_PEER_SLOTS) & 1u;
            if (rank != 0) {
              st_cluster_f32(mapa_u32(smem_u32(&peer_csum[cslot * 4 * 256 + et]), 0), own);
              mbar_arrive_cluster(mapa_u32(csfull0 + 8 * cslot, 0));
            } else {
              mbar_wait_cluster(csfull0 + 8 * cslot, par);
              own += peer_csum[cslot * 4 * 256 + et];
              if (p.dbias != nullptr && et < p.N) p.dbias[et] = own;
            }
          }
          asm volatile("bar.sync 1, 512;" ::: "memory");  // csum_s is reused; db is visible to the small-parameter pass
          if (tracer) ctrace(cp, 2, task_it, pi, 3);
          ++dcount;
        } else {
          // ---- weight gradient: transpose through the staging tile, optimizer (or the gradient store) on the way out ----
          const int64_t i0 = (int64_t)(p.C - grads) - (int64_t)p.member * ctx.P;  // flat offset of W_l in the member block
          const int ld = p.ldc, ncols = p.N;
          const MemberScalars* sc = ctx.scalars + p.member;
          const float a_w1 = sc->adam_w1, a_b2 = sc->adam_beta2, a_1mb2 = sc->adam_one_minus_b2, a_eps = sc->adam_eps;
          const float tau = sc->tau, omt = sc->one_minus_tau;
          const bool is_q = i0 < ctx.PQ;
          const bool first_layer = pi == cp.n_phases - 1;  // the input-layer phase also maintains the lo shadows (3xTF32)
          const AdamScalars as = ctx.adam_sc[p.member * 3 + (is_q ? 0 : (i0 < ctx.v_end ? 1 : 2))];
          const float inv_bc2 = 1.0f / as.bc2_sqrt;
          const int64_t mo = (int64_t)p.member * ctx.P, to = (int64_t)p.member * ctx.PQ;
          // Work units of a lane quarter = (32-column chunk, half of its 32 rows).  Full-width phases: this warp takes
          // both halves of chunks ch and ch + 4.  Narrow phases (input layer, N <= 128): unit w = 2 c + half goes to
          // column group w % 4, so that all 16 warps share the few chunks that exist.
          const bool wide = n_chunks >= 2 * C_CGROUPS;
          const int n_units = wide ? 2 : (2 * n_chunks - ch + C_CGROUPS - 1) / C_CGROUPS;
          // the optimizer state this warp is about to stream does not depend on the accumulator: pull it into L2 while
          // the MMAs of the phase still run (one 128-byte line per lane = row, per array and unit)
          if (!GRADS_ONLY && !(cp.dbg & 4)) {
            for (int un = 0; un < n_units; ++un) {
              const int wu = ch + un * C_CGROUPS;
              const int c = wide ? wu : (wu >> 1);
              if (c * 32 >= ld) continue;
              const int64_t ix = i0 + (int64_t)(row_base + lane) * ld + c * 32;
              prefetch_l2(params + mo + ix);
              prefetch_l2(exp_avg + mo + ix);
              prefetch_l2(exp_avg_sq + mo + ix);
              if (is_q) prefetch_l2(target + to + ix);
            }
          }
          mbar_wait(tfull0 + 8 * buf, acc_phase);
          tc_fence_after();
          if (tracer) ctrace(cp, 2, task_it, pi, 1);
          bool released = false;
#pragma unroll 1
          for (int un = 0; un < n_units; ++un) {
            const int wu = ch + un * C_CGROUPS;
            const int c = wide ? wu : (wu >> 1);
            const int h_lo = wide ? 0 : (wu & 1), h_hi = wide ? 2 : (wu & 1) + 1;
            uint32_t r[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 256 + c * 32), r);
            tmem_ld_wait();
            if (un == n_units - 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) acc_release(buf);
              released = true;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j)
              *reinterpret_cast<float4*>(&stg[lane * 36 + 4 * j]) =
                  make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                              __uint_as_float(r[4 * j + 3]));
            __syncwarp();
            const int col = c * 32 + lc;
            if (GRADS_ONLY && col < ld) {
              // lane octet lr, row group i: row 4 i + lr of the half, 32 consecutive columns = one 128-byte line
#pragma unroll 1
              for (int half = h_lo; half < h_hi; ++half) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  const int rl = half * 16 + 4 * i + lr;
                  float4 g4 = *reinterpret_cast<const float4*>(&stg[rl * 36 + lc]);
                  if (col + 3 >= ncols) {  // row padding of the input-layer weights: exact zeros
                    if (col >= ncols) g4.x = 0.f;
                    if (col + 1 >= ncols) g4.y = 0.f;
                    if (col + 2 >= ncols) g4.z = 0.f;
                    g4.w = 0.f;
                  }
                  *reinterpret_cast<float4*>(grads + mo + i0 + (int64_t)(row_base + rl) * ld + col) = g4;
                }
              }
            } else if (!GRADS_ONLY && col < ld) {
              const int istep = 4 * ld;  // row group i is 4 rows further
#pragma unroll 1
              for (int half = h_lo; half < h_hi; ++half) {
                const int64_t idx0 = i0 + (int64_t)(row_base + half * 16 + lr) * ld + col;
                if (is_q) {
#pragma unroll 1
                  for (int sb = 0; sb < 2; ++sb)
                    adam_rows<2, true>(ctx, stg, half * 16 + sb * 8, lr, lc, col, ncols, p.member, idx0 + (int64_t)sb * 2 * istep, istep,
                                       mo, to, as.neg_step_size, inv_bc2, a_w1, a_b2, a_1mb2, a_eps, tau, omt, first_layer,
                                       cp.keep_grads, cp.dbg, params, exp_avg, exp_avg_sq, target, grads);
                } else {
                  adam_rows<4, false>(ctx, stg, half * 16, lr, lc, col, ncols, p.member, idx0, istep, mo, to, as.neg_step_size,
                                      inv_bc2, a_w1, a_b2, a_1mb2, a_eps, tau, omt, first_layer, cp.keep_grads, cp.dbg, params,
                                      exp_avg, exp_avg_sq, target, grads);
                }
              }
            }
            __syncwarp();
          }
          if (!released) {  // narrow phases: this warp had no unit
            tc_fence_before();
            __syncwarp();
            if (lane == 0) acc_release(buf);
          }
          if (tracer) ctrace(cp, 2, task_it, pi, 3);
        }
      }
      if (tracer) ctrace(cp, 2, task_it, cp.n_phases, 0);
      if (GRADS_ONLY) continue;
      // ---- small parameters of the task (biases, output layer, log_std): leader CTA, gradients from the grads arena;
      // the segments are laid end to end over the 512 threads so that all their loads are in flight together ----
      asm volatile("bar.sync 1, 512;" ::: "memory");
      if (rank == 0) {
        const MemberScalars* sc = ctx.scalars + member;
        const float a_w1 = sc->adam_w1, a_b2 = sc->adam_beta2, a_1mb2 = sc->adam_one_minus_b2, a_eps = sc->adam_eps;
        const float tau = sc->tau, omt = sc->one_minus_tau;
        const int64_t mo = (int64_t)member * ctx.P, to = (int64_t)member * ctx.PQ;
        const int64_t lo0 = cp.seg_lo[slot][0];
        const bool is_q = lo0 < ctx.PQ;
        const AdamScalars as = ctx.adam_sc[member * 3 + (is_q ? 0 : (lo0 < ctx.v_end ? 1 : 2))];
        const float inv_bc2 = 1.0f / as.bc2_sqrt;
        int64_t total = 0;
        for (int s = 0; s < cp.n_seg[slot]; ++s) total += (cp.seg_hi[slot][s] - cp.seg_lo[slot][s]) >> 2;
        for (int64_t e = et; e < total; e += 512) {
          int64_t rem = e, i = 0;
          for (int s = 0; s < cp.n_seg[slot]; ++s) {
            const int64_t n4 = (cp.seg_hi[slot][s] - cp.seg_lo[slot][s]) >> 2;
            if (rem < n4) { i = cp.seg_lo[slot][s] + 4 * rem; break; }
            rem -= n4;
          }
          const float4 g4 = *reinterpret_cast<const float4*>(grads + mo + i);
          const float4 p4 = *reinterpret_cast<const float4*>(params + mo + i);
          const float4 m4 = *reinterpret_cast<const float4*>(exp_avg + mo + i);
          const float4 v4 = *reinterpret_cast<const float4*>(exp_avg_sq + mo + i);
          const float4 t4 = is_q ? *reinterpret_cast<const float4*>(target + to + i) : make_float4(0.f, 0.f, 0.f, 0.f);
          const bool lo_too = i >= ctx.first_w_begin[4] && i < ctx.first_w_end[4];  // policy head run as a two-pass tcgen05 GEMM
          adam_quad_fast(ctx, member, i, g4, p4, m4, v4, t4, as.neg_step_size, inv_bc2, a_w1, a_b2, a_1mb2, a_eps, tau, omt, lo_too,
                         params, exp_avg, exp_avg_sq, target);
        }
      }
      if (tracer) ctrace(cp, 2, task_it, cp.n_phases, 1);
    }
    bulk_wait0();
  }
  tc_fence_before();
  __syncwarp();
  cluster_sync();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  if (GRADS_ONLY) stamp_end(ctx.stamps, ST_CHAIN);
}

}  // namespace

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static long long* chain_trace_buffer() {  // allocated once (at bind time, never inside a capture) when IQL_CHAIN_TRACE is set
  static long long* buf = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    if (dbg_getenv("IQL_CHAIN_TRACE") && cudaMalloc(&buf, sizeof(long long) * C_TRACE_WORDS) == cudaSuccess)
      cudaMemset(buf, 0, sizeof(long long) * C_TRACE_WORDS);
    else
      buf = nullptr;
  }
  return buf;
}

extern "C" int iql_debug_chain_trace(long long* out, int32_t max_words) {
  long long* buf = chain_trace_buffer();
  if (!buf || !out || max_words < C_TRACE_WORDS) return -1;
  if (cudaDeviceSynchronize() != cudaSuccess) return -2;
  if (cudaMemcpy(out, buf, sizeof(long long) * C_TRACE_WORDS, cudaMemcpyDeviceToHost) != cudaSuccess) return -2;
  return C_TRACE_WORDS;
}

bool bwd_chain_supported(int batch, int hidden, int n_hidden, int k0, bool fused_fwd) {
  chain_trace_buffer();
  return fused_fwd && batch == 2 * C_TILE_M && hidden == 256 && n_hidden >= 2 && n_hidden <= FUSED_MAX_LAYERS &&
         k0 <= 256 && umma_phase_supported(1, batch, hidden);
}

int bwd_chain_wgrad0_tile_n(int k0) { return k0 <= 64 ? 64 : (k0 <= 128 ? 128 : 256); }

void launch_bwd_chain(const BwdChainArgs& a, const StepCtx& ctx, cudaStream_t st) {
  static bool attr[64] = {};
  if (first_use_on_device(attr)) {
    cudaFuncSetAttribute(bwd_chain_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C_SMEM);
    cudaFuncSetAttribute(bwd_chain_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C_SMEM);
  }
  ChainParams cp;
  memset(&cp, 0, sizeof(cp));
  cp.n_phases = a.n_phases;
  cp.n_tasks = a.n_tasks;
  cp.keep_grads = a.keep_grads;
  cp.grads_only = a.grads_only;
  cp.db_tile_order = a.db_tile_order;
  int dg = 0;
  for (int i = 0; i < a.n_phases; ++i) {
    ChainPhase& ph = cp.ph[i];
    ph.kind = a.kind[i];
    ph.prob_first = a.prob_first[i];
    ph.map_first = a.map_first[i];
    ph.tile_n = a.tile_n[i];
    ph.nkb = (a.k[i] + C_TILE_K - 1) / C_TILE_K;
    ph.wait_dgrads = a.wait_dgrads[i];
    ph.a_mn = (ph.kind == CH_WGRAD);
    ph.b_mn = 1;
    // c = F32 [4,6), a = b = TF32, a_major [15], b_major [16], N >> 3 [17,23), M >> 4 [24,29): M = 256 per pair
    ph.idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)ph.a_mn << 15) | ((uint32_t)ph.b_mn << 16) |
               ((uint32_t)(ph.tile_n >> 3) << 17) | ((uint32_t)((2 * C_TILE_M) >> 4) << 24);
    if (ph.kind == CH_DGRAD) ++dg;
  }
  cp.n_dgrad = dg;
  cp.trace = chain_trace_buffer();
  {
    static const int dbg = dbg_getenv("IQL_CHAIN_DBG") ? atoi(dbg_getenv("IQL_CHAIN_DBG")) : 0;
    cp.dbg = dbg;
  }
  for (int s = 0; s < 4; ++s) {
    cp.n_seg[s] = a.n_seg[s];
    for (int j = 0; j < a.n_seg[s]; ++j) { cp.seg_lo[s][j] = a.seg_lo[s][j]; cp.seg_hi[s][j] = a.seg_hi[s][j]; }
  }
  static int n_sm = 0;
  if (!n_sm) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    if (n_sm <= 0) n_sm = 148;
  }
  const int workers = a.n_tasks < n_sm / 2 ? a.n_tasks : n_sm / 2;
  launch_pdl(a.grads_only ? bwd_chain_kernel<true> : bwd_chain_kernel<false>, dim3(2 * workers), dim3(C_THREADS), C_SMEM, st, 2, a.probs, (const CUtensorMap*)a.maps,
             (const CUtensorMap*)a.cmaps, cp, ctx, a.params, a.exp_avg, a.exp_avg_sq, a.target, a.grads);
}

}  // namespace iql

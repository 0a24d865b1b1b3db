// Replay data plane: packed transition rows, bulk pack, ring insert, and the
// Philox-indexed gather.  Replaces ReplayBuffer.{load_d4rl_dataset,sample,
// add_transition} (reference algorithms/finetune/iql.py:122-196).
//
// HBM layout: one transition == one contiguous row of `row_floats` fp32
// (multiple of 4, so every row is 16-byte aligned):
//     [ s(S) | a(A) | pad to 4 | s'(S) | r | d | pad to 4 ]
// A sample is therefore ONE contiguous 128..480-byte read issued as float4
// loads by adjacent lanes, instead of five sub-sector reads from five arrays.
#include "common.cuh"
#include "engine.h"

namespace iql {

int make_row_layout(int S, int A, iql_row_layout* out) {
  if (S <= 0 || A <= 0 || !out) return IQL_ERR_INVALID;
  int sa = (int)round_up(S + A, 4);
  out->state_dim = S;
  out->action_dim = A;
  out->off_state = 0;
  out->off_action = S;
  out->off_next_state = sa;
  out->off_reward = sa + S;
  out->off_done = sa + S + 1;
  out->row_floats = (int)round_up(sa + S + 2, 4);
  return IQL_OK;
}

static bool layout_ok(const iql_row_layout* lay) {
  if (!lay) return false;
  iql_row_layout t;
  if (make_row_layout(lay->state_dim, lay->action_dim, &t) != IQL_OK) return false;
  return t.row_floats == lay->row_floats && t.off_action == lay->off_action &&
         t.off_next_state == lay->off_next_state && t.off_reward == lay->off_reward &&
         t.off_done == lay->off_done && lay->off_state == 0;
}

// ---- bulk pack: dense SoA -> packed rows ---------------------------------
__global__ void replay_pack_kernel(float* __restrict__ rows, iql_row_layout lay, int64_t first_row, int64_t n,
                                   const float* __restrict__ s, const float* __restrict__ a,
                                   const float* __restrict__ r, const float* __restrict__ s2,
                                   const float* __restrict__ d) {
  const int RF = lay.row_floats, S = lay.state_dim, A = lay.action_dim;
  int64_t total = n * RF;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = i / RF;
    int c = (int)(i - row * RF);
    float v = 0.f;
    if (c < S) v = s[row * S + c];
    else if (c < S + A) v = a[row * A + (c - S)];
    else if (c >= lay.off_next_state && c < lay.off_next_state + S) v = s2[row * S + (c - lay.off_next_state)];
    else if (c == lay.off_reward) v = r[row];
    else if (c == lay.off_done) v = d[row];
    rows[(first_row + row) * RF + c] = v;
  }
}

// ---- dataset ingest: column statistics with numpy's summation order, then normalise + rescale + pack ----------
// numpy reduces a C-contiguous [n][S] float32 array along axis 0 row by row -- one running fp32 sum per column, no
// pairwise blocking -- so `states.mean(0)` / `states.std(0)` (compute_mean_std, finetune/iql.py:77-80) are reproduced
// bit for bit by ONE thread per column that walks the rows in order; 8 loads are in flight per thread and the adds are
// applied in row order.  mode 0: sum of x -> mean = sum / n.  mode 1: sum of (x - mean)^2 -> std = sqrt(sum / n) + eps.
__global__ void colstat_kernel(const float* __restrict__ x, int64_t n, int S, int mode, const float* __restrict__ mean_in,
                               float eps, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= S) return;
  const float mu = mode ? mean_in[c] : 0.f;
  float acc = 0.f;
  int64_t i = 0;
  for (; i + 8 <= n; i += 8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = x[(i + j) * S + c];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (mode) { const float d = __fsub_rn(v[j], mu); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
      else acc = __fadd_rn(acc, v[j]);
    }
  }
  for (; i < n; ++i) {
    const float v = x[i * S + c];
    if (mode) { const float d = __fsub_rn(v, mu); acc = __fadd_rn(acc, __fmul_rn(d, d)); }
    else acc = __fadd_rn(acc, v);
  }
  const float q = __fdiv_rn(acc, (float)n);
  out[c] = mode ? __fadd_rn(__fsqrt_rn(q), eps) : q;
}

// pack with the reference's preprocessing applied on the way: states and next states (x - mean) / std
// (normalize_states, finetune/iql.py:83-84), rewards (r / div) * mul - sub (modify_reward, :286-297: locomotion
// div = max_ret - min_ret, mul = max_episode_steps; antmaze sub = 1), each operation rounded like numpy's float32 ops
__global__ void replay_ingest_kernel(float* __restrict__ rows, iql_row_layout lay, int64_t first_row, int64_t n,
                                     const float* __restrict__ s, const float* __restrict__ a, const float* __restrict__ r,
                                     const float* __restrict__ s2, const float* __restrict__ d,
                                     const float* __restrict__ mean, const float* __restrict__ stdv, float rdiv, float rmul,
                                     float rsub, int scale_reward) {
  const int RF = lay.row_floats, S = lay.state_dim, A = lay.action_dim;
  const int64_t total = n * RF;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / RF;
    const int c = (int)(i - row * RF);
    float v = 0.f;
    if (c < S) {
      v = s[row * S + c];
      if (mean) v = __fdiv_rn(__fsub_rn(v, mean[c]), stdv[c]);
    } else if (c < S + A) {
      v = a[row * A + (c - S)];
    } else if (c >= lay.off_next_state && c < lay.off_next_state + S) {
      const int k = c - lay.off_next_state;
      v = s2[row * S + k];
      if (mean) v = __fdiv_rn(__fsub_rn(v, mean[k]), stdv[k]);
    } else if (c == lay.off_reward) {
      v = r[row];
      if (scale_reward) v = __fmul_rn(__fdiv_rn(v, rdiv), rmul);
      if (rsub != 0.f) v = __fsub_rn(v, rsub);
    } else if (c == lay.off_done) {
      v = d[row];
    }
    rows[(first_row + row) * RF + c] = v;
  }
}

__global__ void replay_insert_kernel(float* __restrict__ rows, int RF, int64_t pointer,
                                     const float* __restrict__ staged) {
  for (int c = threadIdx.x; c < RF; c += blockDim.x) rows[pointer * RF + c] = staged[c];  // any row width
}

// add_transition for a host caller: the packed row rides in the kernel parameters (rows of up to 960 floats), so an
// insert is one launch with no staging row, no host->device copy and nothing to guard against reuse
constexpr int ROW_BYVAL_MAX = 960;
struct RowPack { float v[ROW_BYVAL_MAX]; };
__global__ void replay_insert_byval_kernel(float* __restrict__ rows, int RF, int64_t pointer, const __grid_constant__ RowPack row) {
  for (int c = threadIdx.x; c < RF; c += blockDim.x) rows[pointer * RF + c] = row.v[c];
}

// add_transition of S members at once (iql_replay_insert_members_host): CTA i copies the packed row i of the
// device-mapped pinned input slot to row pointers[i] of the ring bound to member ids[i], then marks its part of the slot
// consumed.  Every load of the slot has returned once the CTA passes the barrier (each value was stored), so the host
// may overwrite the row as soon as the word is raised -- the guard never waits for the rest of the stream.
__global__ void replay_insert_members_kernel(const ReplayBinding* __restrict__ replay, int RF, const float* rows,
                                             const int32_t* ids, const int64_t* pointers, uint32_t* consumed) {
  const int i = blockIdx.x;
  const int m = ids[i];
  const int64_t p = pointers[i];
  float* dst = const_cast<float*>(replay[m].rows) + p * RF;
  const float* src = rows + (int64_t)i * RF;
  for (int c = threadIdx.x; c < RF; c += blockDim.x) dst[c] = src[c];
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    reinterpret_cast<volatile uint32_t*>(consumed)[i] = 1u;
  }
}

void launch_insert_members(const ReplayBinding* replay, int RF, const float* rows, const int32_t* ids, const int64_t* pointers,
                           int n, uint32_t* consumed, cudaStream_t st) {
  const int threads = RF < 256 ? ((RF + 31) / 32) * 32 : 256;
  replay_insert_members_kernel<<<n, threads, 0, st>>>(replay, RF, rows, ids, pointers, consumed);
}

// ---- sample: Philox (or given) indices + vectorised row gather ------------
// One thread per float4 of a row; the RF/4 lanes of a row are adjacent, so the
// row read is a single coalesced burst.  The row is then scattered to the five
// dense outputs the reference API returns.
__global__ void replay_sample_kernel(const float* __restrict__ rows, iql_row_layout lay, int64_t size, int64_t batch,
                                     const int64_t* __restrict__ indices, uint64_t seed, uint64_t step,
                                     float* __restrict__ so, float* __restrict__ ao, float* __restrict__ ro,
                                     float* __restrict__ s2o, float* __restrict__ dout,
                                     int64_t* __restrict__ idx_out) {
  const int RF = lay.row_floats, S = lay.state_dim, A = lay.action_dim;
  const int Q = RF >> 2;
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= batch * Q) return;
  int64_t b = t / Q;
  int q = (int)(t - b * Q);
  int64_t idx = indices ? indices[b] : philox_index(seed, step, (uint32_t)b, (uint64_t)size);
  if (q == 0 && idx_out) idx_out[b] = idx;
  float4 v = __ldg(reinterpret_cast<const float4*>(rows + idx * RF) + q);
  float vals[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int c = q * 4 + j;
    float x = vals[j];
    if (c < S) so[b * S + c] = x;
    else if (c < S + A) ao[b * A + (c - S)] = x;
    else if (c >= lay.off_next_state && c < lay.off_next_state + S) s2o[b * S + (c - lay.off_next_state)] = x;
    else if (c == lay.off_reward) ro[b] = x;
    else if (c == lay.off_done) dout[b] = x;
  }
}

// Host-drawn indices passed BY VALUE in the kernel parameters (up to 256 per launch): the reference draws its
// indices with numpy on the host every step (iql.py:172); this way they reach the gather without a staging buffer,
// a host->device copy or anything the next sample() call could overwrite while this launch is still queued.
struct IdxPack { int64_t v[256]; };
__global__ void __launch_bounds__(256) replay_sample_byval_kernel(const float* __restrict__ rows, iql_row_layout lay, int b0, int nb,
                                                                  const __grid_constant__ IdxPack idx,
                                                                  float* __restrict__ so, float* __restrict__ ao,
                                                                  float* __restrict__ ro, float* __restrict__ s2o,
                                                                  float* __restrict__ dout) {
  const int RF = lay.row_floats, S = lay.state_dim, A = lay.action_dim;
  const int Q = RF >> 2;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nb * Q) return;
  const int bl = t / Q, q = t - bl * Q;
  const int64_t b = b0 + bl;
  const float4 v = __ldg(reinterpret_cast<const float4*>(rows + idx.v[bl] * RF) + q);
  const float vals[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = q * 4 + j;
    const float x = vals[j];
    if (c < S) so[b * S + c] = x;
    else if (c < S + A) ao[b * A + (c - S)] = x;
    else if (c >= lay.off_next_state && c < lay.off_next_state + S) s2o[b * S + (c - lay.off_next_state)] = x;
    else if (c == lay.off_reward) ro[b] = x;
    else if (c == lay.off_done) dout[b] = x;
  }
}

}  // namespace iql

using namespace iql;

extern "C" int iql_replay_row_layout(int32_t state_dim, int32_t action_dim, iql_row_layout* out) {
  return make_row_layout(state_dim, action_dim, out);
}

extern "C" int iql_replay_pack(float* rows, const iql_row_layout* lay, int64_t first_row, int64_t n,
                               const float* states, const float* actions, const float* rewards,
                               const float* next_states, const float* dones, void* stream) {
  if (!layout_ok(lay) || !rows || n < 0 || first_row < 0) return IQL_ERR_INVALID;
  if (n == 0) return IQL_OK;
  if (!states || !actions || !rewards || !next_states || !dones) return IQL_ERR_INVALID;
  int64_t total = n * lay->row_floats;
  int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  replay_pack_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rows, *lay, first_row, n, states, actions, rewards,
                                                               next_states, dones);
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

extern "C" int iql_replay_ingest(float* rows, const iql_row_layout* lay, int64_t first_row, int64_t n, const float* states,
                                 const float* actions, const float* rewards, const float* next_states, const float* dones,
                                 int32_t normalize, float eps, float* mean_out, float* std_out, float reward_div,
                                 float reward_mul, float reward_sub, void* stream) {
  if (!layout_ok(lay) || !rows || n < 0 || first_row < 0) return IQL_ERR_INVALID;
  if (n == 0) return IQL_OK;
  if (!states || !actions || !rewards || !next_states || !dones) return IQL_ERR_INVALID;
  if (normalize && (!mean_out || !std_out)) return IQL_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  const int S = lay->state_dim;
  if (normalize) {
    colstat_kernel<<<(S + 31) / 32, 32, 0, st>>>(states, n, S, 0, nullptr, 0.f, mean_out);
    colstat_kernel<<<(S + 31) / 32, 32, 0, st>>>(states, n, S, 1, mean_out, eps, std_out);
  }
  const int64_t total = n * lay->row_floats;
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  replay_ingest_kernel<<<blocks, 256, 0, st>>>(rows, *lay, first_row, n, states, actions, rewards, next_states, dones,
                                                normalize ? mean_out : nullptr, normalize ? std_out : nullptr, reward_div,
                                                reward_mul, reward_sub, (reward_div != 1.0f || reward_mul != 1.0f) ? 1 : 0);
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

extern "C" int iql_replay_insert(float* rows, const iql_row_layout* lay, int64_t pointer, const float* staged_row,
                                 void* stream) {
  if (!layout_ok(lay) || !rows || !staged_row || pointer < 0) return IQL_ERR_INVALID;
  int threads = (lay->row_floats + 31) / 32 * 32;
  if (threads > 256) threads = 256;  // wide rows (2 S + A > ~250 floats) loop inside the kernel
  replay_insert_kernel<<<1, threads, 0, (cudaStream_t)stream>>>(rows, lay->row_floats, pointer, staged_row);
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

extern "C" int iql_replay_sample(const float* rows, const iql_row_layout* lay, int64_t size, int64_t batch,
                                 const int64_t* indices, uint64_t seed, uint64_t step, float* states,
                                 float* actions, float* rewards, float* next_states, float* dones,
                                 int64_t* idx_out, void* stream) {
  if (!layout_ok(lay) || !rows || batch < 0) return IQL_ERR_INVALID;
  if (batch == 0) return IQL_OK;
  if (size <= 0 && !indices) return IQL_ERR_INVALID;  // np.random.randint(0, 0) raises ValueError
  if (!states || !actions || !rewards || !next_states || !dones) return IQL_ERR_INVALID;
  int64_t threads = batch * (lay->row_floats >> 2);
  int blocks = (int)((threads + 255) / 256);
  replay_sample_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rows, *lay, size, batch, indices, seed, step, states,
                                                                 actions, rewards, next_states, dones, idx_out);
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

extern "C" int iql_replay_sample_host(const float* rows, const iql_row_layout* lay, int64_t size, int64_t batch,
                                      const int64_t* host_indices, float* states, float* actions, float* rewards,
                                      float* next_states, float* dones, void* stream) {
  if (!layout_ok(lay) || !rows || batch < 0 || size <= 0) return IQL_ERR_INVALID;
  if (batch == 0) return IQL_OK;
  if (!host_indices || !states || !actions || !rewards || !next_states || !dones) return IQL_ERR_INVALID;
  const int Q = lay->row_floats >> 2;
  IdxPack pack;
  for (int64_t b0 = 0; b0 < batch; b0 += 256) {
    const int nb = (int)(batch - b0 < 256 ? batch - b0 : 256);
    for (int i = 0; i < nb; ++i) {
      const int64_t v = host_indices[b0 + i];
      if (v < 0 || v >= size) return IQL_ERR_INVALID;
      pack.v[i] = v;
    }
    for (int i = nb; i < 256; ++i) pack.v[i] = 0;
    replay_sample_byval_kernel<<<(nb * Q + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rows, *lay, (int)b0, nb, pack, states, actions,
                                                                                        rewards, next_states, dones);
  }
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

extern "C" int iql_replay_insert_host(float* rows, const iql_row_layout* lay, int64_t pointer, const float* host_state,
                                      const float* host_action, float reward, const float* host_next_state, float done,
                                      void* stream) {
  if (!layout_ok(lay) || !rows || pointer < 0 || !host_state || !host_action || !host_next_state) return IQL_ERR_INVALID;
  if (lay->row_floats > ROW_BYVAL_MAX) return IQL_ERR_SHAPE;  // wider rows: stage the row and use iql_replay_insert
  RowPack p;
  const int S = lay->state_dim, A = lay->action_dim, RF = lay->row_floats;
  for (int c = 0; c < RF; ++c) p.v[c] = 0.f;
  for (int i = 0; i < S; ++i) p.v[lay->off_state + i] = host_state[i];
  for (int i = 0; i < A; ++i) p.v[lay->off_action + i] = host_action[i];
  for (int i = 0; i < S; ++i) p.v[lay->off_next_state + i] = host_next_state[i];
  p.v[lay->off_reward] = reward;
  p.v[lay->off_done] = done;
  replay_insert_byval_kernel<<<1, RF < 256 ? ((RF + 31) / 32) * 32 : 256, 0, (cudaStream_t)stream>>>(rows, RF, pointer, p);
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

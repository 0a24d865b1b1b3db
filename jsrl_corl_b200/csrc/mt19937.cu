// numpy's legacy index stream on the device: RandomState.randint(0, high, size=n) (int64), the draw behind
// ReplayBuffer.sample (reference algorithms/finetune/iql.py:172) and behind ensemble_train_loop's per-member
// index_rng[m].randint, reproduced word for word from the generator state RandomState.get_state() returns.
//
// The stream (numpy's legacy bounded-integer rule, masked rejection, for 1 <= high <= 2^32):
//   rng = high - 1; rng == 0 -> zeros, and no word is consumed;
//   mask = smallest 2^k - 1 >= rng; per output repeat v = temper(next_word()) & mask until v <= rng.
// next_word() is MT19937 (624 words, lazy twist: the key is twisted when a word is needed at pos == 624, so a draw
// that consumes word 623 leaves pos = 624 and the key untwisted).  K calls of size B equal one call of size K * B.
//
// One CTA per stream keeps the 624 key words in shared memory.  A round tempers, masks and tests every word still
// unread in the current key block at once (one word per thread), compacts the accepted words in stream order (warp
// ballot + popc, shared per-warp prefix), writes them up to the requested count and moves pos past the last word it
// consumed.  The twist runs in its three dependent parallel phases; each reads all its inputs before any write.
#include "common.cuh"
#include "engine.h"

namespace iql {

constexpr int MT_N = 624, MT_M = 397;
constexpr int MT_THREADS = 640;  // >= 624: one thread per word of a key block
constexpr int MT_WARPS = MT_THREADS / 32;
static_assert(IQL_MT_STATE_WORDS >= MT_N + 1, "state row: key[624], pos");

__device__ __forceinline__ uint32_t mt_twist_word(uint32_t cur, uint32_t next, uint32_t far) {
  const uint32_t y = (cur & 0x80000000u) | (next & 0x7FFFFFFFu);
  return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908B0DFu : 0u);
}

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9D2C5680u;
  y ^= (y << 15) & 0xEFC60000u;
  y ^= y >> 18;
  return y;
}

// numpy's mt19937_gen: i < 227 reads key[i + 397] (old); 227 <= i < 623 reads key[i - 227] (new, from the phase before);
// i = 623 reads key[0] (phase 1) and key[396] (phase 2), so it joins phase 3.  Every phase reads, syncs, then writes.
__device__ __forceinline__ void mt_twist(uint32_t* key) {
  const int t = threadIdx.x;
#pragma unroll
  for (int phase = 0; phase < 3; ++phase) {
    const int i = phase * (MT_N - MT_M) + t;
    const int last = phase < 2 ? (phase + 1) * (MT_N - MT_M) : MT_N;
    uint32_t v = 0;
    const bool mine = i < last;
    if (mine) {
      const int far = phase == 0 ? i + MT_M : i - (MT_N - MT_M);
      v = mt_twist_word(key[i], key[i + 1 < MT_N ? i + 1 : 0], key[far]);
    }
    __syncthreads();
    if (mine) key[i] = v;
    __syncthreads();
  }
}

// One CTA draws `count` values of randint(0, rng + 1) from the stream at `state` ([IQL_MT_STATE_WORDS]: key[624], pos)
// and stores value j at out[(j / rowlen) * rowstride + j % rowlen]; the state row is advanced past the words consumed.
__device__ void mt_randint_block(uint32_t* __restrict__ state, uint32_t rng, int64_t count, int64_t* __restrict__ out,
                                 int64_t rowlen, int64_t rowstride) {
  __shared__ uint32_t key[MT_N];
  __shared__ int warp_cnt[MT_WARPS];
  __shared__ int last_word;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (count <= 0) return;
  if (rng == 0) {  // randint(0, 1): zeros, no word consumed
    for (int64_t j = t; j < count; j += blockDim.x) out[(j / rowlen) * rowstride + j % rowlen] = 0;
    return;
  }
  uint32_t mask = rng;
  mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
  for (int i = t; i < MT_N; i += blockDim.x) key[i] = state[i];
  int pos = (int)state[MT_N];
  __syncthreads();
  bool twisted = false;
  int64_t done = 0;
  while (done < count) {  // block-uniform
    if (pos >= MT_N) {
      mt_twist(key);
      twisted = true;
      pos = 0;
    }
    const int i = pos + t;
    uint32_t v = 0;
    bool acc = false;
    if (i < MT_N) {
      v = mt_temper(key[i]) & mask;
      acc = v <= rng;
    }
    const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, acc);
    if (lane == 0) warp_cnt[warp] = __popc(ballot);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < MT_WARPS; ++w) {
      const int c = warp_cnt[w];
      before += w < warp ? c : 0;
      total += c;
    }
    const int64_t rank = done + before + __popc(ballot & ((1u << lane) - 1u));
    if (acc && rank < count) {
      out[(rank / rowlen) * rowstride + rank % rowlen] = (int64_t)v;
      if (rank == count - 1) last_word = i;
    }
    __syncthreads();
    if (done + total >= count) {
      pos = last_word + 1;
      done = count;
    } else {
      done += total;
      pos = MT_N;
    }
    __syncthreads();  // warp_cnt / last_word are rewritten by the next round
  }
  if (twisted)
    for (int i = t; i < MT_N; i += blockDim.x) state[i] = key[i];
  if (t == 0) state[MT_N] = (uint32_t)pos;
}

// The engine's sampler: CTA i serves active member m = active[i] (all members when active is null).  It draws the K x B_m
// indices of the call's K steps at the member's bound `high` -- from the replay table, or from host_high[m] (a host step:
// the device-mapped pinned block) -- into indices[m][k][b], b < B_m; the gather then reads them like caller indices.
__global__ void __launch_bounds__(MT_THREADS) mt19937_members_kernel(StepCtx ctx, uint32_t* __restrict__ states,
                                                                     int64_t* __restrict__ indices, const int64_t* host_high) {
  const int m = ctx.active ? ctx.active[blockIdx.x] : (int)blockIdx.x;
  const int64_t high = host_high ? host_high[m] : ctx.replay[m].size;
  const int64_t bm = ctx.scalars[m].batch;
  mt_randint_block(states + (int64_t)m * IQL_MT_STATE_WORDS, (uint32_t)(high - 1), (int64_t)ctx.K * bm,
                   indices + (int64_t)m * ctx.K * ctx.B, bm, ctx.B);
}

void launch_mt19937_members(const StepCtx& ctx, uint32_t* states, int64_t* indices, const int64_t* host_high, cudaStream_t st) {
  mt19937_members_kernel<<<ctx.n_active, MT_THREADS, 0, st>>>(ctx, states, indices, host_high);
}

// Handle-free form (iql_mt19937_randint): stream i of a launch draws count[i] values at bound high[i] into
// out + i * stride; the bounds and counts travel in the kernel parameters, 256 streams per launch.
struct MtJobs {
  int64_t high[256];
  int64_t count[256];
};

__global__ void __launch_bounds__(MT_THREADS) mt19937_randint_kernel(uint32_t* __restrict__ states, int64_t* __restrict__ out,
                                                                     int64_t stride, const __grid_constant__ MtJobs jobs) {
  const int i = blockIdx.x;
  const int64_t n = jobs.count[i];
  mt_randint_block(states + (int64_t)i * IQL_MT_STATE_WORDS, (uint32_t)(jobs.high[i] - 1), n, out + (int64_t)i * stride,
                   n > 0 ? n : 1, 0);
}

}  // namespace iql

using namespace iql;

extern "C" int iql_mt19937_randint(uint32_t* states, int32_t n, const int64_t* host_high, const int64_t* host_count,
                                   int64_t* out, int64_t stride, void* stream) {
  if (!states || !host_high || !host_count || n < 0) return IQL_ERR_INVALID;
  if (n == 0) return IQL_OK;
  int64_t most = 0;
  for (int i = 0; i < n; ++i) {
    if (host_high[i] < 1 || host_high[i] > ((int64_t)1 << 32) || host_count[i] < 0) return IQL_ERR_INVALID;
    most = host_count[i] > most ? host_count[i] : most;
  }
  if (most > 0 && (!out || stride < most)) return IQL_ERR_INVALID;
  for (int i0 = 0; i0 < n; i0 += 256) {
    const int nb = n - i0 < 256 ? n - i0 : 256;
    MtJobs jobs;
    for (int i = 0; i < 256; ++i) {
      jobs.high[i] = i < nb ? host_high[i0 + i] : 1;
      jobs.count[i] = i < nb ? host_count[i0 + i] : 0;
    }
    mt19937_randint_kernel<<<nb, MT_THREADS, 0, (cudaStream_t)stream>>>(states + (int64_t)i0 * IQL_MT_STATE_WORDS,
                                                                        out ? out + i0 * stride : nullptr, stride, jobs);
  }
  return cudaGetLastError() == cudaSuccess ? IQL_OK : IQL_ERR_CUDA;
}

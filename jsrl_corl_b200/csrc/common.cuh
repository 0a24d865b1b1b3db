// Shared device/host helpers for the IQL engine (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

namespace iql {

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), the counter-based generator behind index
// sampling and dropout masks.  Restated on the CPU in oracle/philox.py and
// oracle/philox_ref.c; the two are compared bit for bit in tests.
// ---------------------------------------------------------------------------
#define IQL_PHILOX_M0 0xD2511F53u
#define IQL_PHILOX_M1 0xCD9E8D57u
#define IQL_PHILOX_W0 0x9E3779B9u
#define IQL_PHILOX_W1 0xBB67AE85u

#define IQL_STREAM_SAMPLE 0u        // counter word 3 for replay index sampling
#define IQL_STREAM_DROPOUT_BASE 1u  // + hidden layer index, for dropout masks
// + hidden layer index, for the dropout masks of the training-mode act (iql_act_host_members codes 4 / 5); the update
// streams above use words 0 .. 1 + n_hidden, so the act masks never repeat a training mask of the same key
#define IQL_STREAM_ACT_DROPOUT_BASE 0x80000000u

struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
  uint64_t p = (uint64_t)a * (uint64_t)b;
  hi = (uint32_t)(p >> 32);
  lo = (uint32_t)p;
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(IQL_PHILOX_M0, c0, hi0, lo0);
    philox_mulhilo(IQL_PHILOX_M1, c2, hi1, lo1);
    uint32_t n0 = hi1 ^ c1 ^ k0;
    uint32_t n1 = lo1;
    uint32_t n2 = hi0 ^ c3 ^ k1;
    uint32_t n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += IQL_PHILOX_W0;
    k1 += IQL_PHILOX_W1;
  }
  Philox4 o{c0, c1, c2, c3};
  return o;
}

// Uniform index in [0, size): the b-th draw of (seed, step).  Two indices per
// Philox block: counter = (b >> 1, step_lo, step_hi, STREAM_SAMPLE); the 64-bit
// word (hi<<32 | lo) of lanes (x,y) for even b, (z,w) for odd b, mapped with
// a 64x64->128 multiply-high (bias < size / 2^64).
__host__ __device__ __forceinline__ int64_t philox_index(uint64_t seed, uint64_t step, uint32_t b, uint64_t size) {
  Philox4 r = philox4x32_10(b >> 1, (uint32_t)step, (uint32_t)(step >> 32), IQL_STREAM_SAMPLE,
                            (uint32_t)seed, (uint32_t)(seed >> 32));
  uint64_t u = (b & 1u) ? (((uint64_t)r.w << 32) | r.z) : (((uint64_t)r.y << 32) | r.x);
#ifdef __CUDA_ARCH__
  return (int64_t)__umul64hi(u, size);
#else
  return (int64_t)(((unsigned __int128)u * (unsigned __int128)size) >> 64);
#endif
}

// Dropout keep decisions for 4 consecutive elements (quad = element_index / 4)
// of hidden layer `layer` at update `step`: keep iff word >= threshold where
// threshold = floor(p * 2^32).
__host__ __device__ __forceinline__ Philox4 philox_dropout_quad(uint64_t seed, uint64_t step, uint32_t layer,
                                                                uint32_t quad) {
  return philox4x32_10(quad, (uint32_t)step, (uint32_t)(step >> 32), IQL_STREAM_DROPOUT_BASE + layer,
                       (uint32_t)seed, (uint32_t)(seed >> 32));
}

// The same for the act kernel: neurons 4 * quad .. 4 * quad + 3 of hidden layer `layer` at act counter `act_step`
// (restated on the CPU in tests/act_mask_oracle.py).
__host__ __device__ __forceinline__ Philox4 philox_act_dropout_quad(uint64_t seed, uint64_t act_step, uint32_t layer,
                                                                    uint32_t quad) {
  return philox4x32_10(quad, (uint32_t)act_step, (uint32_t)(act_step >> 32), IQL_STREAM_ACT_DROPOUT_BASE + layer,
                       (uint32_t)seed, (uint32_t)(seed >> 32));
}

__host__ __device__ __forceinline__ uint32_t dropout_threshold(double p) {
  double t = p * 4294967296.0;
  if (t <= 0.0) return 0u;
  if (t >= 4294967295.0) return 4294967295u;
  return (uint32_t)t;
}

// Round-to-nearest TF32 (10-bit mantissa).  tcgen05 kind::tf32 TRUNCATES the low 13 mantissa bits of its fp32
// operands, a systematic shrink of ~1e-3 per GEMM; operands that were rounded to nearest beforehand pass through
// the truncation unchanged, which turns the bias into zero-mean rounding noise.
// Same result as `cvt.rna.tf32.f32` (nearest, ties away from zero) for finite values, but two integer ALU ops
// instead of a quarter-rate XU conversion: add half an ulp of the 13 dropped bits to the magnitude, clear them.
__device__ __forceinline__ float round_tf32(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// Every IQL_* environment switch of the library (path selection for A/B measurements, probes, traces: INTEGRATION.md
// section 4) is a DEBUG facility behind one master flag: without IQL_B200_DEBUG=1 in the environment none of them is
// read, so none of them is API.  Supported, documented selection goes through iql_set_option().
static inline const char* dbg_getenv(const char* name) {
  static int on = -1;
  if (on < 0) on = getenv("IQL_B200_DEBUG") ? 1 : 0;
  return on ? getenv(name) : nullptr;
}

// ---------------------------------------------------------------------------
// Programmatic dependent launch: a kernel launched with launch_pdl may become resident and run its set-up (barrier
// init, TMEM allocation, reads of the static problem tables) while the preceding kernel of the stream drains; it
// must call pdl_wait() before it reads anything that kernel wrote -- or writes anything that kernel reads.
// Without a trigger the successor is released when every CTA of this kernel has exited (it still saves the launch
// latency and its set-up: +3.5 % on the 64-member step).  pdl_trigger() at the top of a kernel releases the
// successor as soon as all of this kernel's CTAs are running, so that it fills SMs as they drain; measured per
// kernel: helps after last_bwd (+1.2 %), neutral in adam, hurts in the persistent tcgen05 kernels (their successors
// then sit on SMs the stragglers' co-runners could use: -7 % in umma_gemm, -1.4 % in fused_fwd), so only last_bwd
// calls it.  IQL_B200_NO_PDL switches the launch attribute off.
// ---------------------------------------------------------------------------
// step timeline (IQL_STEP_TRACE): thread 0 of every CTA folds its start / end into the launch's slot
__device__ __forceinline__ void stamp_begin(unsigned long long* stamps, int slot) {
  if (stamps && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    atomicMin(stamps + 2 * slot, t);
  }
}
__device__ __forceinline__ void stamp_end(unsigned long long* stamps, int slot) {
  if (stamps && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    atomicMax(stamps + 2 * slot + 1, t);
  }
}

__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE attribute: true the first time this call site
// runs on the current device (engines on several GPUs of one process each need their own call).
static inline bool first_use_on_device(bool* seen /* [64], zero-initialised */) {
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  if (seen[dev]) return false;
  seen[dev] = true;
  return true;
}

static inline bool pdl_enabled() {
  static int v = -1;
  if (v < 0) v = dbg_getenv("IQL_B200_NO_PDL") ? 0 : 1;
  return v != 0;
}

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     int cluster_x, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  int n = 0;
  if (pdl_enabled()) {
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster_x > 1) {
    at[n].id = cudaLaunchAttributeClusterDimension;
    at[n].val.clusterDim.x = (unsigned)cluster_x;
    at[n].val.clusterDim.y = 1;
    at[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = at;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace iql

// common.cuh -- shared device helpers: numerics, reductions, Philox, error plumbing.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <utility>

namespace gmvae {

typedef __nv_bfloat16 bf16;

// ----------------------------------------------------------------------------- host errors
void set_error(const std::string& msg);
#define GM_CHECK_CUDA(expr)                                                                  \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      ::gmvae::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ + \
                         ":" + std::to_string(__LINE__) + ")");                              \
      return -2;                                                                             \
    }                                                                                        \
  } while (0)
#define GM_REQUIRE(cond, msg)                   \
  do {                                          \
    if (!(cond)) {                              \
      ::gmvae::set_error(std::string(msg));     \
      return -1;                                \
    }                                           \
  } while (0)
#define GM_TRY(expr)           \
  do {                         \
    int _r = (expr);           \
    if (_r != 0) return _r;    \
  } while (0)

// ----------------------------------------------------------------------------- launches
// Programmatic dependent launch: every kernel of the step is launched with the
// programmatic-stream-serialization attribute, so its CTAs may become resident (and run their
// prologue: barrier init, TMEM allocation, descriptor prefetch) while the previous kernel drains.
// Each kernel calls griddep_wait() before it touches global memory -- that returns only when the
// previous grid has completed and its writes are visible -- and griddep_launch() right after, which
// lets the next kernel's CTAs be scheduled as soon as SM resources free up.
extern bool g_use_pdl;
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = (pdl && g_use_pdl) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// the same with thread-block clusters of `cluster` CTAs along x (CTA pairs of the chained kernel)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = (pdl && g_use_pdl) ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// ----------------------------------------------------------------------------- conversions
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

// ----------------------------------------------------------------------------- numerics (fp32)
// log(1+e^t), the same asymptote handling as tf.nn.softplus / torch.logaddexp(t,0).
__device__ __forceinline__ float softplus_f(float t) { return fmaxf(t, 0.f) + log1pf(expf(-fabsf(t))); }
__device__ __forceinline__ float sigmoid_f(float t) {
  // stable for both signs
  float e = expf(-fabsf(t));
  float s = 1.f / (1.f + e);
  return t >= 0.f ? s : e * s;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Sum over the block, result valid in thread 0. `scratch` >= 32 floats of shared memory.
__device__ __forceinline__ float block_sum(float v, float* scratch) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  float r = 0.f;
  if (w == 0) {
    int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? scratch[lane] : 0.f;
    r = warp_sum(r);
  }
  return r;
}

// ----------------------------------------------------------------------------- loss accumulators
// The three un-normalised loss sums (nll, kl, nent) live in the tail of the gradient buffer so that
// one all-reduce covers them.  Each is spread over 32 fp32 slots (slot chosen by the adding block)
// and summed in double by the finalising kernel: thousands of same-sized addends into ONE fp32
// accumulator round in a correlated way (measured: 1.6e-4 relative on the 16 384-sample KAT).
enum { ACC_NLL = 0, ACC_KL = 32, ACC_NENT = 64, ACC_PER_TERM = 32, ACC_SLOTS = 96 };
// Deterministic mode (gmvae_config::deterministic): sums whose addends arrive in no fixed order are taken in fixed point, as
// int64 multiples of 2^-FX_SHIFT.  Integer addition is associative, so the total does not depend on the order of arrival; the
// reduction step (det_reduce_kernel) converts it to fp32.  Resolution 1.5e-11 per addend.  Sum i lives in fx[2i]; fx[2i + 1]
// flags an addend that is not finite or beyond +-2^26 (whose fixed-point form would saturate), and the reduction step then
// writes NaN, as a NaN addend would have made of the default mode's float sum.  A sum of in-range addends beyond +-2^27 wraps
// unflagged; the sums taken this way (loss terms, VAE_GMP prior gradients: means over the batch) stay far below that.
enum { FX_SHIFT = 36 };
__device__ __forceinline__ void fx_add(unsigned long long* fx, int i, float v) {
  if (fabsf(v) < 67108864.f) atomicAdd(fx + 2 * i, (unsigned long long)__float2ll_rn(v * (float)(1ull << FX_SHIFT)));   // two's complement
  else atomicOr(fx + 2 * i + 1, 1ull);                                                                                 // also NaN
}
// The training step passes the accumulator base with bit 0 set in deterministic mode: it then points at the fixed-point sums
// above, one per term (index term / ACC_PER_TERM).
inline float* acc_fixed_tag(unsigned long long* fx) { return reinterpret_cast<float*>(reinterpret_cast<uintptr_t>(fx) | 1u); }
__device__ __forceinline__ void acc_add(float* acc, int term, float v) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(acc);
  if (a & 1u) { fx_add(reinterpret_cast<unsigned long long*>(a & ~(uintptr_t)1), term / ACC_PER_TERM, v); return; }
  atomicAdd(acc + term + ((blockIdx.x + (threadIdx.x >> 5)) & (ACC_PER_TERM - 1)), v);
}
__device__ __forceinline__ float acc_total(const float* acc, int term) {
  double s = 0.0;
  for (int i = 0; i < ACC_PER_TERM; ++i) s += (double)acc[term + i];
  return (float)s;
}

// ----------------------------------------------------------------------------- Philox4x32-10
// (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123 known-answer vectors are checked
// through the host build of this struct, tests/test_input_cpu.py.)  __host__ __device__ so that the same source is
// exercised on the CPU by the tests; the device code is the `__CUDA_ARCH__` branch.
struct Philox {
  __host__ __device__ static __forceinline__ uint32_t mulhi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
  }
  __host__ __device__ static __forceinline__ void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    uint32_t hi0 = mulhi(M0, c[0]), lo0 = M0 * c[0];
    uint32_t hi1 = mulhi(M1, c[2]), lo1 = M1 * c[2];
    uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
  }
  // 4 random words for (seed, stream, counter)
  __host__ __device__ static __forceinline__ void gen(uint64_t seed, uint64_t stream, uint64_t ctr, uint32_t (&out)[4]) {
    uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)stream, (uint32_t)(stream >> 32)};
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      round(c, k0, k1);
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
  }
};
// uniform in (0,1): never 0, never 1.  (r>>9)+0.5 is exact in fp32 (23 bits + half), so the
// largest value is 1 - 2^-24 and the smallest 2^-24.
__host__ __device__ __forceinline__ float u01(uint32_t r) { return ((float)(r >> 9) + 0.5f) * (1.0f / 8388608.0f); }

}  // namespace gmvae

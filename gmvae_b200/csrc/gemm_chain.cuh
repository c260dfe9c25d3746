// gemm_chain.cuh -- a CHAIN of dependent GEMMs in ONE persistent tcgen05 kernel.
//
// At the reference's layer sizes (784-512-512, batch 16 384) one layer is 256 output tiles on 148
// SMs: 1.73 waves.  Launched one kernel per GEMM (gemm_tc.cuh), every layer pays the pipeline fill,
// the wave quantisation and the exposed epilogue of its last tile.  Here the GEMMs of a whole
// section of the step (e.g. decoder forward + Bernoulli likelihood + decoder backward: 9 GEMMs) are
// jobs of one launch.  The tiles of all jobs form one sequence, dealt round-robin to the persistent
// CTAs, so the tail of job j overlaps the head of job j+1 and the TMA->MMA->epilogue pipeline never
// drains in between.
//
// Data dependencies are per 128-row block: a job that consumes the rows another job of the chain
// produces waits (TMA producer thread, ld.acquire.gpu spin) on a counter the producing tiles'
// epilogue warps increment (st -> fence -> red.add) -- forward/dgrad jobs wait for ONE row block,
// weight-gradient jobs for the row blocks their batch slice covers.  Every tile depends only on
// tiles with a smaller index in the sequence and each CTA walks its tiles in increasing order with
// all CTAs co-resident (grid <= number of SMs, 1 CTA/SM), so the waits cannot deadlock.
//
// Everything the one-GEMM kernel fixes at compile time (tile width, operand majorness, epilogue
// functor) is a run-time field of the job here; the mechanics (TMA ring, single-thread MMA issue,
// double-buffered TMEM accumulator, 16 epilogue warps with smem-staged coalesced I/O) are the same.
#pragma once
#include "gemm_tc.cuh"
#include "chain_sched.cuh"

namespace gmvae {
namespace tc {

enum EpiKind : int { EK_NONE = -1, EK_STORE_BF16 = 0, EK_STORE_F32 = 1, EK_BCE = 2, EK_RELUMASK = 3, EK_ATOMIC = 4,
                     // "row" jobs: no GEMM, the epilogue warps run a distribution head on a block of 128 rows
                     EK_ROWS_FIRST = 16, EK_ROWS_Y_FWD = 16, EK_ROWS_Z_FWD = 17, EK_ROWS_Z_BWD = 18, EK_ROWS_Y_BWD = 19 };

// Parameters of the row jobs (same math as head_*_kernel in kernels.cuh; bf16 training step only).
struct RowsYFwd { const float* logits; const float* u; int K; float inv_T, inv_bg; float* y_f32; bf16* y_act; int ld_yact; float* acc; };
struct RowsZFwd { const float* enc_out; const float* eps; const float* prior_out; int prior_mode, Z; float c, sigma_min, inv_bg;
                  bf16* z_act; int ld_z; float* acc; };
struct RowsZBwd { const float* enc_out; const float* eps; const float* prior_out; const float* dz_dec; int prior_mode, Z; float c, sigma_min, inv_bg;
                  bf16* d_enc_out; bf16* d_prior_out; int ld_out; float* db_enc; float* db_prior; };
struct RowsYBwd { const float* logits; const float* y_f32; const float* dy; int K; float inv_T, inv_bg; bf16* dlogits; int ld_out; float* db; };
template <class Epi> struct epi_kind { static constexpr int value = EK_NONE; };
template <> struct epi_kind<EpiStore<bf16, EPI_PLAIN>> { static constexpr int value = EK_STORE_BF16; };
template <> struct epi_kind<EpiStore<float, EPI_PLAIN>> { static constexpr int value = EK_STORE_F32; };
template <> struct epi_kind<EpiBCE<bf16>> { static constexpr int value = EK_BCE; };
template <> struct epi_kind<EpiReluMask<bf16, bf16>> { static constexpr int value = EK_RELUMASK; };
template <> struct epi_kind<EpiAtomicAdd> { static constexpr int value = EK_ATOMIC; };

// 1-bit ReLU masks between the forward and the backward jobs of a layer (written by the forward epilogue, one coalesced 128-byte line per
// warp and 32 columns; read by the data-gradient epilogue with one 4-byte load per row issued ahead of the accumulator) instead of a
// TMA load of the bf16 activation box in the epilogue's critical path.  Switched per step by the host (engine.cu, DBG_NO_RELU_BITS).
constexpr bool CHAIN_RELU_BITS = true;
static_assert(SCHED_BLOCK_M == BLOCK_M, "chain_sched.cuh and gemm_tc.cuh agree on the tile height");
constexpr int CHAIN_MAX_JOBS = 40;     // a whole forward + backward pass of the 3-MLP model is 33 jobs
constexpr int CHAIN_MAX_MAPS = 112;    // tensor maps of all jobs (operands, TMA-stored outputs, ReLU-mask sources)
constexpr int CHAIN_STAGES = 4;
constexpr int CHAIN_STAGE_BYTES = A_STAGE_BYTES + 256 * BLOCK_K * 2;   // room for the widest tile (48 KB)
// CTA-pair mode (cta_group::2, see gemm_tc.cuh): a stage holds this CTA's 128 rows of A and HALF of the B tile's columns
#ifndef GMVAE_PAIR_STAGES
#define GMVAE_PAIR_STAGES 6       // experiment hook (GMVAE_NVCC_FLAGS=-DGMVAE_PAIR_STAGES=3: +7 % per k-block -- the ring depth does not pace the main loop)
#endif
constexpr int CHAIN_STAGES_PAIR = GMVAE_PAIR_STAGES;
constexpr int CHAIN_STAGE_BYTES_PAIR = A_STAGE_BYTES + 128 * BLOCK_K * 2;   // 32 KB
static_assert(CHAIN_STAGES_PAIR * CHAIN_STAGE_BYTES_PAIR <= CHAIN_STAGES * CHAIN_STAGE_BYTES, "both modes use the same ring area");
constexpr int CHAIN_PATCH_BYTES = 2048;   // per epilogue warp: 32 rows x 64 B, the box of one TMA store (SWIZZLE_64B like the tensor map)
constexpr int CHAIN_CARVE_BYTES = CHAIN_STAGES * CHAIN_STAGE_BYTES + EPI_WARPS * CHAIN_PATCH_BYTES + 256 /*barriers*/ + 256 * 4 /*bias*/ + 256 * 4 /*column sums*/;
constexpr int CHAIN_SMEM_BYTES = 232448;  // everything an SM offers one CTA (227 KB); the carve-out needs all but 768 bytes of it
static_assert(CHAIN_CARVE_BYTES + 512 <= CHAIN_SMEM_BYTES, "shared-memory budget");

// Passed by value as the kernel's __grid_constant__ parameter.  Two capacities: the recording buffer (a whole
// forward + backward pass in one launch, about 26 KB of the 32 KB parameter space) and a small one (8 KB) used when
// the recorded section fits -- the parameter block is copied at every launch, ~3 us for the large one.
template <int MAXJ, int MAXM>
struct ChainParamsT {
  int njobs, nmaps;
  int* counters;
  long long* trace;    // test hook: clock64 stamps of CTA `trace_cta`, 16 per processed tile (null in production)
  int trace_cta;
  int abl;             // timing-only ablations (builds with -DGMVAE_CHAIN_ABL; results are garbage): 1 epilogues skip their work, 2 no TMA loads, 4 no MMAs
  unsigned long long* jobstat;   // test hook: 8 counters per job over ALL CTAs (globaltimer ns): [0] first tile start, [1] last tile end,
                                 // [2] producer dependency wait, [3] MMA issue->commit, [4] epilogue rows, [5] epilogue wait for the
                                 // accumulator, [6] tiles, [7] MMA wait for a free accumulator (null in production)
  alignas(64) CUtensorMap maps[MAXM];
  ChainJob jobs[MAXJ];
};
constexpr int CHAIN_SMALL_JOBS = 10, CHAIN_SMALL_MAPS = 44;
typedef ChainParamsT<CHAIN_MAX_JOBS, CHAIN_MAX_MAPS> ChainParams;
typedef ChainParamsT<CHAIN_SMALL_JOBS, CHAIN_SMALL_MAPS> ChainParamsSmall;
static_assert(sizeof(ChainParams) <= 32000, "kernel parameter space");

#ifndef GMVAE_POLL_NS
#define GMVAE_POLL_NS 40          // back-off between two polls of a row-block counter (experiment hook)
#endif
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// Release of a row block: everything this thread wrote (and what the warp's other lanes wrote before the __syncwarp that precedes the
// call) becomes visible at gpu scope before the counter moves: one release-scoped reduction.  (`legacy`, GMVAE_CHAIN_ABL=8: the form used
// until late in round 2 -- __threadfence(), i.e. fence.sc.gpu = MEMBAR.SC + L1 invalidate, then a relaxed atomic; 8.7 % of the epilogue
// warps' stall samples sat on that fence.  Same-box A/B: 0.3593 -> 0.3558 ms per cfg4 step, 2.031 -> 2.011 ms at 131 072 rows.)
__device__ __forceinline__ void release_counter(int* ctr, int legacy) {
  if (!legacy) {
    asm volatile("red.release.gpu.global.add.s32 [%0], %1;" ::"l"(ctr), "r"(1) : "memory");
  } else {
    __threadfence();
    atomicAdd(ctr, 1);
  }
}
// bounded like mbar_wait: a scheduling bug ends as a trapped launch, not as a hung GPU
__device__ __forceinline__ void wait_counter(const int* p, int target) {
  if (ld_acquire_gpu(p) >= target) return;
  const long long t0 = clock64();
  while (ld_acquire_gpu(p) < target) {
    __nanosleep(GMVAE_POLL_NS);
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}

__device__ __forceinline__ uint64_t make_smem_desc_rt(uint32_t smem_addr, int mn_major) {
  const uint64_t lbo = mn_major ? (uint64_t)(BLOCK_K * 128) : 0;
  const uint64_t sbo = 1024;
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((lbo >> 4) << 16) | ((sbo >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

struct ChainShared {
  uint8_t* smem; uint64_t* full_bar; uint64_t* empty_bar; uint64_t* tmem_full_bar; uint64_t* tmem_empty_bar;
  uint8_t* patches; float* sbias_all; float* scs_all; uint32_t tmem_base; uint64_t* op_bar;
};

// ---- bulk-tensor stores (TMA): shared -> global, tracked in bulk async-groups of the issuing thread
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, uint32_t src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Patch addressing = the tensor map's swizzle: rows of RB bytes (128: SWIZZLE_128B, 64: SWIZZLE_64B),
// 16-byte unit u of row r.
template <int RB> __device__ __forceinline__ uint32_t patch_unit(uint32_t patch, int r, int u) {
  return RB == 128 ? patch + r * 128 + ((u ^ (r & 7)) << 4) : patch + r * 64 + ((u ^ ((r >> 1) & 3)) << 4);
}

// Column sums of a bf16 patch (32 rows) added into the CTA accumulator scs[0 .. RB/2).
template <int RB>
__device__ __forceinline__ void patch_colsum_bf16(uint32_t patch, float* scs, int ncols, int lane) {
  constexpr int WORDS = RB / 4;                 // 32-bit words (column pairs) per row: 32 or 16
  constexpr int GROUPS = 32 / WORDS;            // 1 or 2 row groups walked by different lanes
  const int w = lane % WORDS, grp = lane / WORDS;
  float s0 = 0.f, s1 = 0.f;
#pragma unroll 8
  for (int i = 0; i < 32 / GROUPS; ++i) {
    const int r = grp * (32 / GROUPS) + i;
    const uint32_t t = lds32(patch_unit<RB>(patch, r, w >> 2) + 4 * (w & 3));
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t));
    s0 += f.x; s1 += f.y;
  }
  if (GROUPS == 2) { s0 += __shfl_xor_sync(0xffffffffu, s0, 16); s1 += __shfl_xor_sync(0xffffffffu, s1, 16); }
  if (grp == 0) {
    const uint32_t a = smem_addr(scs) + 8 * w;
    if (2 * w < ncols && s0 != 0.f) asm volatile("red.shared.add.f32 [%0], %1;" ::"r"(a), "f"(s0) : "memory");
    if (2 * w + 1 < ncols && s1 != 0.f) asm volatile("red.shared.add.f32 [%0], %1;" ::"r"(a + 4), "f"(s1) : "memory");
  }
}

__device__ __forceinline__ void pack16(const float* v, uint4& lo, uint4& hi) {
  lo.x = pack_bf16x2(v[0], v[1]); lo.y = pack_bf16x2(v[2], v[3]); lo.z = pack_bf16x2(v[4], v[5]); lo.w = pack_bf16x2(v[6], v[7]);
  hi.x = pack_bf16x2(v[8], v[9]); hi.y = pack_bf16x2(v[10], v[11]); hi.z = pack_bf16x2(v[12], v[13]); hi.w = pack_bf16x2(v[14], v[15]);
}

// ---- q(y|x) head on one row held in registers (K <= 16): shared by the row jobs and the fused epilogues ----
// Warp-collective (all 32 lanes call; `valid` masks rows beyond the batch) and deliberately NOT inlined: the thin
// GEMM jobs that host them sit on the critical path of the chain and must not inherit their register footprint.
// forward: lg = logits (with bias).  Writes y (fp32 + zero-padded bf16 operand row), returns sum_k p log p of the row.
// Math of the heads inside the chained kernel (bf16 training step only): fast intrinsics.  The fp32 validation mode never
// runs these (kernels.cuh heads).  __expf is good to ~2 ulp relative.  __logf(s) is good to an ABSOLUTE ~1e-7 near s = 1,
// which is enough where the result is O(1) or is added to one: the BCE loss, and the y head's lse = ml + log(sl), whose
// absolute error of ~ulp(ml) per row stays far below the bf16 bars even when q(y|x) is nearly one-hot.  It is not
// enough for softplus(t) = log(1 + e), e = exp(t), on its own as a scale: below t ~ -5 the sum 1 + e drops the low bits of
// e (relative error 5e-4 at sigma = 1e-4, 6e-2 at 1e-6, and sigma = 0 -- log 0, 1/0 -- below 6e-8), so the z heads take
// log1p_fast, which is accurate to ~1 ulp relative for small e as well.
__device__ __forceinline__ float exp2f_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// log(1 + e) for e in [0, 1]: below 2^-7 the series e (1 - e/2 + e^2/3) (truncation e^4/4 < 2^-23 e), above it __logf(1 + e)
__device__ __forceinline__ float log1p_fast(float e) {
  return e < 0.0078125f ? e * fmaf(e, fmaf(e, 0.33333334f, -0.5f), 1.f) : __logf(1.f + e);
}
__device__ __forceinline__ float fast_softplus(float t) { return fmaxf(t, 0.f) + log1p_fast(__expf(-fabsf(t))); }
__device__ __forceinline__ float fast_sigmoid(float t) {
  const float e = __expf(-fabsf(t));
  const float s = __fdividef(1.f, 1.f + e);
  return t >= 0.f ? s : e * s;
}
// row of K floats at p (8-byte aligned when K is even): vector loads / stores
__device__ __forceinline__ void ld_row16(const float* p, int K, float* v, float fill) {
  if ((K & 1) == 0) {
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
      if (k < K) { const float2 t = __ldcg(reinterpret_cast<const float2*>(p + k)); v[k] = t.x; v[k + 1] = t.y; }
      else { v[k] = fill; v[k + 1] = fill; }
    }
  } else {
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = k < K ? __ldcg(p + k) : fill;
  }
}
__device__ __forceinline__ void st_row16(float* p, int K, const float* v) {
  if ((K & 1) == 0) {
#pragma unroll
    for (int k = 0; k < 16; k += 2)
      if (k < K) *reinterpret_cast<float2*>(p + k) = make_float2(v[k], v[k + 1]);
  } else {
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) p[k] = v[k];
  }
}
// `noise`: the row's Gumbel noise if the caller has fetched it already (ahead of the accumulator), else nullptr
__device__ __noinline__ float y_head_fwd_row(const float* lg, const RowsYFwd& prm, int64_t row, bool valid, const float* noise = nullptr) {
  if (!valid) return 0.f;
  const int K = prm.K;
  float a[16];
  if (noise) {
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = noise[k];
  } else {
    ld_row16(prm.u + row * K, K, a, 0.f);                     // Gumbel noise g = -log(-log u), prepared by the step's first kernel
  }
  float ml = -INFINITY, ma = -INFINITY;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    if (k < K) {
      a[k] = (lg[k] + a[k]) * prm.inv_T;
      ml = fmaxf(ml, lg[k]);
    } else {
      a[k] = -INFINITY;
    }
    ma = fmaxf(ma, a[k]);
  }
  float sl = 0.f, sa = 0.f;
  float pl[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    pl[k] = 0.f;
    if (k < K) { a[k] = __expf(a[k] - ma); pl[k] = __expf(lg[k] - ml); sl += pl[k]; sa += a[k]; }
  }
  const float lse = ml + __logf(sl), inv_sa = __fdividef(1.f, sa), inv_sl = __fdividef(1.f, sl);
  float y[16];
  float ent = 0.f;
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    y[k] = 0.f;
    if (k < K) {
      ent = fmaf(pl[k] * inv_sl, lg[k] - lse, ent);          // p log p
      y[k] = a[k] * inv_sa;
    }
  }
  st_row16(prm.y_f32 + row * K, K, y);
  uint4* dst = reinterpret_cast<uint4*>(prm.y_act + row * prm.ld_yact);
  dst[0] = make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
  if (prm.ld_yact > 8) dst[1] = make_uint4(pack_bf16x2(y[8], y[9]), pack_bf16x2(y[10], y[11]), pack_bf16x2(y[12], y[13]), pack_bf16x2(y[14], y[15]));
  return ent;
}
// backward: g = dy of the row.  Writes dlogits (bf16, zero-padded); the column sums of the stored values over the
// warp's rows (bias gradient of encoder_y's last layer) are added to the shared-memory accumulator scs[0..K).
__device__ __noinline__ void y_head_bwd_row(const float* g, const RowsYBwd& prm, int64_t row, bool valid, float* scs) {
  const int K = prm.K;
  float lg[16], o[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) o[k] = 0.f;
  if (valid) {
    float y[16];
    ld_row16(prm.logits + row * K, K, lg, -INFINITY);
    ld_row16(prm.y_f32 + row * K, K, y, 0.f);
    float ml = -INFINITY, ydy = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) { ml = fmaxf(ml, lg[k]); ydy = fmaf(y[k], g[k], ydy); }
    float sl = 0.f;
    float pl[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      pl[k] = 0.f;
      if (k < K) { pl[k] = __expf(lg[k] - ml); sl += pl[k]; }
    }
    const float lse = ml + __logf(sl), inv_sl = __fdividef(1.f, sl);
    float plogp = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) { lg[k] -= lse; pl[k] *= inv_sl; plogp = fmaf(pl[k], lg[k], plogp); }
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) o[k] = __bfloat162float(__float2bfloat16_rn(y[k] * (g[k] - ydy) * prm.inv_T + pl[k] * (lg[k] - plogp) * prm.inv_bg));
    uint4* dst = reinterpret_cast<uint4*>(prm.dlogits + row * prm.ld_out);
    dst[0] = make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
    if (prm.ld_out > 8) dst[1] = make_uint4(pack_bf16x2(o[8], o[9]), pack_bf16x2(o[10], o[11]), pack_bf16x2(o[12], o[13]), pack_bf16x2(o[14], o[15]));
  }
  // Column sums over the warp's 32 rows: a transposing butterfly -- every step halves the values a lane carries while it doubles the
  // rows they cover (8 + 4 + 2 + 1 + 1 = 16 shuffles; sixteen separate warp sums were 80 and ten serialised shared-memory atomics,
  // a third of this head's 15 us on the step's critical path).  Lanes 2c and 2c + 1 end up with the sum of column c.
  const int lane = (int)threadIdx.x & 31;
#pragma unroll
  for (int w = 8, bit = 16; w >= 1; w >>= 1, bit >>= 1) {
    const bool up = (lane & bit) != 0;                        // upper half of the lanes keeps the upper half of the columns
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float send = up ? o[i] : o[i + w];
      const float keep = up ? o[i + w] : o[i];
      o[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
  }
  const float t = o[0] + __shfl_xor_sync(0xffffffffu, o[0], 1);
  const int col = lane >> 1;
  if ((lane & 1) == 0 && col < K && t != 0.f) atomicAdd(scs + col, t);
}

// The epilogue warps' share of one job.  `it` counts the tiles this CTA has processed since the
// start of the kernel (accumulator buffer = it & 1).
//
// Output path (J.gw > 0): a warp owns the 32 rows of its TMEM lane quadrant and walks "groups" of
// J.gw 16-column chunks.  Lane = row: the lane converts its row of a chunk and writes it into the
// warp's patch at the position the output tensor map's swizzle expects; when the group is complete
// one lane issues ONE bulk-tensor store (or reduce-add, for weight gradients) of the 32-row x 128-byte
// (64-byte) box.  Global memory sees full lines from the TMA unit instead of 32-byte pieces from the
// LSU (measured before: ~16 B/clk/SM, the limiter of the whole step), rows/columns beyond M/N are
// clipped by the tensor map, and no st.global is issued by the epilogue warps at all.  The ReLU mask
// source of the backward pass arrives the same way (TMA load of the box into the patch).
template <class Epi, int KIND, int CL>
__device__ __forceinline__ void chain_epilogue_job(const ChainJob& J, const CUtensorMap* maps, int* counters, const ChainShared& S, int& it,
                                                   uint32_t& op_phase, int warp, int lane, long long* trace, int jidx,
                                                   unsigned long long* jobstat = nullptr, int abl = 0) {
  constexpr int CW = 16;
  constexpr bool PAIR = CL >= 2;
  Epi epi = *reinterpret_cast<const Epi*>(J.epi);
  // GEMM tiles are dealt round-robin to the walkers (CTAs, CTA pairs or 4-CTA clusters); every CTA of a walker takes the same steps
  const int G = (int)gridDim.x / CL;
  const int cidx = (int)blockIdx.x / CL;
  const int rank = (int)blockIdx.x % CL;                 // place in the cluster
  int first, wstride;
  if (!chain_walk<1>(J, cidx, G, first, wstride) || first >= J.walk_total) return;
  const int M = J.M, N = J.N, BN = J.block_n;
  const int nchunk = BN / CW;
  const int e = warp - 2, quad = warp & 3, slot = e >> 2;
  const int et = (int)threadIdx.x - 64;
  float* const cs_dst = epi.colsum_dst();
  const float* const bias = epi.bias_ptr();
  float* const scs_all = S.scs_all;
  const uint32_t patch = smem_addr(S.patches + e * CHAIN_PATCH_BYTES);
  uint64_t* const op_bar = S.op_bar + e;
  const int gw = J.gw;
  int cs_n0 = -1;
  int staged_n0 = -1;                                     // n-tile whose bias sits in the staging buffer
  float fuse_acc = 0.f;                                  // fused y head: sum p log p (forward) of this thread's rows
  bool fuse_bwd = false;
  if constexpr (KIND == EK_STORE_F32) fuse_bwd = J.fuse == EK_ROWS_Y_BWD;   // its bias-gradient sums use the CTA accumulator
  if (cs_dst || fuse_bwd) { for (int i = et; i < 256; i += EPI_WARPS * 32) scs_all[i] = 0.f; }
  auto cs_flush = [&]() {
    for (int i = et; i < BN; i += EPI_WARPS * 32) {
      const float v = scs_all[i];
      if (v != 0.f && cs_n0 + i < N) atomicAdd(cs_dst + cs_n0 + i, v);
      scs_all[i] = 0.f;
    }
  };
  for (int l = first; l < J.walk_total; l += wstride, ++it) {
    int z, mb, n0;
    chain_tile<CL>(J, l, rank, z, mb, n0);
    const int m0 = mb * BLOCK_M;
    const int as = it & 1; const uint32_t ap = (it >> 1) & 1;
    const int mrow0 = m0 + quad * 32;
    const int m = mrow0 + lane;
    float* sbias = S.sbias_all;
    // bias of this tile's columns, staged when the CTA moves to another n-tile (with an even number of walkers and n-tiles a CTA
    // keeps its n-tile through a whole job: the two block-wide barriers are then paid once per job, not once per tile)
    if (n0 != staged_n0) {                                  // uniform over the epilogue warps
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");   // (every warp has finished the previous tile's reads)
      const uint32_t sb = smem_addr(sbias);
      float shift = 0.f;
      if constexpr (KIND == EK_BCE) shift = epi.gen_bias;     // logits = MLP(z) + bias_init (base.py:135)
      for (int i = et; i < BN; i += EPI_WARPS * 32) sts32f(sb + 4 * i, ((bias && n0 + i < N) ? __ldg(bias + n0 + i) : 0.f) + shift);
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      staged_n0 = n0;
    }
    if (cs_dst && cs_n0 != n0) {
      if (cs_n0 >= 0) {
        cs_flush();
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      }
      cs_n0 = n0;
    }
    const bool mvalid = m < M;
#ifdef GMVAE_CHAIN_ABL
    if (abl & 1) {
      mbar_wait(&S.tmem_full_bar[it & 1], (it >> 1) & 1);
      tc_fence_after(); tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_leader(&S.tmem_empty_bar[it & 1]); else mbar_arrive(&S.tmem_empty_bar[it & 1]);
        if (J.sig_base >= 0) { __threadfence(); atomicAdd(counters + J.sig_base + mb, 1); }
      }
      continue;
    }
#endif
    const bool tr = trace && e == 0 && lane == 0 && it < 64;
    if (tr) { trace[16 * it + 6] = clock64(); trace[16 * it + 15] = jidx; trace[16 * it + 14] = l; }
    const bool js = jobstat && e == 0 && lane == 0;
    unsigned long long js_t0 = 0, js_t1 = 0;
    // The epilogue's own operand (ReLU mask source) is fetched ahead of the accumulator, i.e. possibly
    // before the TMA producer has seen this tile's dependencies: the warp checks the operand's producer itself.
    if (J.epi_dep >= 0 && m0 < M) {                         // (a pair's phantom half has no producer to wait for)
      if (lane == 0) { wait_counter(counters + J.deps[J.epi_dep].base + mb, J.deps[J.epi_dep].target); fence_proxy_async_global(); }
      __syncwarp();
    }
    const uint32_t taddr = S.tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * 256);
    bool acc_ready = false;
    auto wait_acc = [&]() {
      if (!acc_ready) {
        if (tr) trace[16 * it + 7] = clock64();
        if (js) js_t0 = gtimer();
        mbar_wait(&S.tmem_full_bar[as], ap);
        tc_fence_after();
        if (tr) trace[16 * it + 8] = clock64();
        if (js) js_t1 = gtimer();
        acc_ready = true;
      }
    };

    if (KIND == EK_STORE_F32 || gw == 0) {
     if constexpr (KIND == EK_STORE_F32 || KIND == EK_ATOMIC) {
      // thin fp32 outputs (logits, [mu|raw], dz, dy) and weight gradients whose row stride is not a
      // multiple of 16 bytes: each lane stores / accumulates its own row fragment
      EpiCtx ctx{nullptr, max(0, min(32, M - mrow0)), sbias, scs_all};
      float noise[CW];
      bool have_noise = false;
      if constexpr (KIND == EK_STORE_F32) {
        // fused forward y head: the row's Gumbel noise (written by the step's first kernel, complete before this launch reads anything)
        // is fetched while the accumulator is still being computed
        if (J.fuse == EK_ROWS_Y_FWD && slot == 0 && mvalid) {
          const RowsYFwd& yp = *reinterpret_cast<const RowsYFwd*>(J.epi2);
          ld_row16(yp.u + (int64_t)m * yp.K, yp.K, noise, 0.f);
          have_noise = true;
        }
      }
      wait_acc();
#pragma unroll 1
      for (int ci = slot; ci < nchunk && n0 + ci * CW < N; ci += 4) {
        const int n = n0 + ci * CW;
        uint32_t r[CW];
        tmem_ld16_issue(taddr + ci * CW, r);
        tmem_ld16_wait(r);
        float v[CW];
#pragma unroll
        for (int i = 0; i < CW; ++i) v[i] = __uint_as_float(r[i]);
        ctx.sbias = sbias + ci * CW;
        if constexpr (KIND == EK_STORE_F32) {
          if (J.fuse != 0) {
            // N <= 16: the lane holds the whole row -- the y head runs right here, no extra job / launch / dependency stage
            float lg[CW];
#pragma unroll
            for (int i = 0; i < CW; ++i) lg[i] = fmaf(v[i], epi.scale, sbias[i]);
            if (J.fuse == EK_ROWS_Y_FWD) {
              if (mvalid) {
                if (epi.ld == N) st_row16(epi.out + (int64_t)m * epi.ld, N, lg);   // logits: read again by the backward head
                else {
#pragma unroll
                  for (int i = 0; i < CW; ++i)
                    if (i < N) epi.out[(int64_t)m * epi.ld + i] = lg[i];
                }
              }
              fuse_acc += y_head_fwd_row(lg, *reinterpret_cast<const RowsYFwd*>(J.epi2), (int64_t)m, mvalid, have_noise ? noise : nullptr);
            } else {
              y_head_bwd_row(lg, *reinterpret_cast<const RowsYBwd*>(J.epi2), (int64_t)m, mvalid, scs_all);
            }
            continue;
          }
        }
        typename Epi::template Pre<CW> pre;
        epi.template row<CW>(m, n, v, min(CW, N - n), mvalid, pre, ctx);
      }
     }
    } else if constexpr (KIND != EK_STORE_F32) {
      const int ngroups = (nchunk + gw - 1) / gw;
#pragma unroll 1
      for (int g = slot; g < ngroups && n0 + g * gw * CW < N; g += 4) {
        const int gcol = g * gw * CW;                        // first column of the group within the tile
        // the previous bulk store issued from this patch must have read it before it is overwritten
        if (lane == 0) bulk_wait_read0();
        uint32_t hbits = 0;
        bool use_bits = false;
        if constexpr (KIND == EK_RELUMASK) {
          use_bits = CHAIN_RELU_BITS && epi.relu_bits != nullptr;
          if (!use_bits) fence_proxy_async();   // this warp's earlier generic reads of the patch precede the TMA write
        }
        __syncwarp();
        if constexpr (KIND == EK_RELUMASK) {
          if (use_bits) {
            // 32 mask bits of this lane's row for the group's 32 columns (written by the forward job of this layer)
            if (mvalid) hbits = __ldcg(epi.relu_bits + (int64_t)((n0 + gcol) >> 5) * epi.ld_bits + m);   // L2: written by another SM in this launch
          } else if (lane == 0) {
            mbar_expect_tx(op_bar, (uint32_t)CHAIN_PATCH_BYTES);
            tma_load_2d(&maps[J.c], op_bar, S.patches + e * CHAIN_PATCH_BYTES, n0 + gcol, mrow0);
          }
        }
        uint32_t obits = 0; int obits_chunks = 0;
        uint4 xq[2];
        if constexpr (KIND == EK_BCE) {
          // image bytes of this lane's row (16 per chunk), fetched ahead of the accumulator
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int n = n0 + gcol + c * CW;
            xq[c] = make_uint4(0, 0, 0, 0);
            if (c < gw && mvalid && n < N) {
              const uint8_t* px = epi.x + (int64_t)m * epi.ldx + n;
              if (n + CW <= N && (reinterpret_cast<uintptr_t>(px) & 15) == 0) {
                xq[c] = *reinterpret_cast<const uint4*>(px);
              } else {
                uint8_t* b = reinterpret_cast<uint8_t*>(&xq[c]);
                for (int i = 0; i < CW && n + i < N; ++i) b[i] = px[i];
              }
            }
          }
        }
        wait_acc();
        if constexpr (KIND == EK_RELUMASK) {
          if (!use_bits) {
            mbar_wait(op_bar, op_phase);
            op_phase ^= 1;
          }
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int ci = g * gw + c;
          if (c < gw && ci < nchunk && n0 + ci * CW < N) {       // warp-uniform
            uint32_t r[CW];
            tmem_ld16_issue(taddr + ci * CW, r);
            float bb[CW];
            if constexpr (KIND == EK_STORE_BF16 || KIND == EK_BCE) {
              const uint32_t sb = smem_addr(sbias + ci * CW);
#pragma unroll
              for (int i = 0; i < CW; i += 4) { float4 t = lds128f(sb + 4 * i); bb[i] = t.x; bb[i + 1] = t.y; bb[i + 2] = t.z; bb[i + 3] = t.w; }
            }
            uint4 h0, h1;
            if constexpr (KIND == EK_RELUMASK) {
              if (!use_bits) { h0 = lds128(patch_unit<64>(patch, lane, 2 * c)); h1 = lds128(patch_unit<64>(patch, lane, 2 * c + 1)); }
            }
            tmem_ld16_wait(r);
            float v[CW];
#pragma unroll
            for (int i = 0; i < CW; ++i) v[i] = __uint_as_float(r[i]);
            if constexpr (KIND == EK_ATOMIC) {
              // fp32 rows of 64 bytes: one chunk per group, units 0 .. 3
#pragma unroll
              for (int u = 0; u < 4; ++u)
                sts128(patch_unit<64>(patch, lane, u),
                       make_uint4(__float_as_uint(v[4 * u]), __float_as_uint(v[4 * u + 1]), __float_as_uint(v[4 * u + 2]), __float_as_uint(v[4 * u + 3])));
            } else {
              if constexpr (KIND == EK_STORE_BF16) {
#pragma unroll
                for (int i = 0; i < CW; ++i) {
                  v[i] = fmaf(v[i], epi.scale, bb[i]);
                  if (epi.relu == 1) v[i] = fmaxf(v[i], 0.f);
                  else if (epi.relu == 2) v[i] = sigmoid_f(v[i] + epi.shift);
                }
                if (CHAIN_RELU_BITS && epi.relu_bits) {
                  // [v == 0] for v >= +0 is the top bit of bits(v) - 1; one funnel shift per element appends it
                  // (element e of the group ends at bit 31 - e; complemented when the word is stored)
#pragma unroll
                  for (int i = 0; i < CW; ++i) obits = __funnelshift_l(__float_as_uint(v[i]) - 1u, obits, 1);
                  ++obits_chunks;
                }
              } else if constexpr (KIND == EK_RELUMASK) {
               if (use_bits) {
#pragma unroll
                for (int i = 0; i < CW; ++i) v[i] = ((hbits >> (31 - (c * CW + i))) & 1u) ? v[i] : 0.f;
               } else {
                const __nv_bfloat162* ph0 = reinterpret_cast<const __nv_bfloat162*>(&h0);
                const __nv_bfloat162* ph1 = reinterpret_cast<const __nv_bfloat162*>(&h1);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const float2 a = __bfloat1622float2(ph0[k]), b = __bfloat1622float2(ph1[k]);
                  v[2 * k] = a.x > 0.f ? v[2 * k] : 0.f; v[2 * k + 1] = a.y > 0.f ? v[2 * k + 1] : 0.f;
                  v[8 + 2 * k] = b.x > 0.f ? v[8 + 2 * k] : 0.f; v[8 + 2 * k + 1] = b.y > 0.f ? v[8 + 2 * k + 1] : 0.f;
                }
               }
              } else if constexpr (KIND == EK_BCE) {
                const int nvalid = min(CW, N - (n0 + ci * CW));
                float ll = 0.f;
                if (nvalid == CW && m0 + BLOCK_M <= M) {
                  // Whole chunk inside the matrix (warp-uniform).  x in {0,1}: with t = (1 - 2x) l, i.e. l with its sign bit
                  // flipped where x = 1,   x l - softplus(l) = -softplus(t)   and   sigmoid(l) - x = (1 - 2x) sigmoid(t):
                  // one exponential, one reciprocal, one logarithm and ~14 other instructions per element (the epilogue warps
                  // are issue-bound here: 25 K elements per tile against an 8-k-block main loop).
                  const uint32_t* xw = reinterpret_cast<const uint32_t*>(&xq[c]);
#pragma unroll
                  for (int i = 0; i < CW; ++i) {
                    const uint32_t sgn = (xw[i >> 2] << (31 - 8 * (i & 3))) & 0x80000000u;     // bit 0 of byte i -> sign bit
                    const float t = __uint_as_float(__float_as_uint(v[i] + bb[i]) ^ sgn);
                    const float e = exp2f_approx(fabsf(t) * -1.4426950408889634f);
                    const float d = 1.f + e;
                    const float r = rcp_approx(d);
                    ll -= fmaxf(t, 0.f);
                    ll = fmaf(lg2_approx(d), -0.6931471805599453f, ll);
                    const float sg = r * (t >= 0.f ? 1.f : e);
                    v[i] = __uint_as_float(__float_as_uint(sg * epi.inv_bg) ^ sgn);
                  }
                } else {
                  const uint8_t* xb = reinterpret_cast<const uint8_t*>(&xq[c]);
#pragma unroll
                  for (int i = 0; i < CW; ++i) {
                    const float lg = v[i] + bb[i];
                    // byte -> float without the conversion pipe: 2^23 + b is exact in fp32
                    const float xv = __uint_as_float(0x4B000000u | (uint32_t)xb[i]) - 8388608.f;
                    // bf16 mode only: fast intrinsics (exp(-|l|) in (0,1], log(1+e) with 1+e in (1,2]: abs error ~1e-7)
                    const float ex = __expf(-fabsf(lg));
                    const float sp = fmaxf(lg, 0.f) + __logf(1.f + ex);
                    const float inv1pe = __fdividef(1.f, 1.f + ex);
                    const float sg = lg >= 0.f ? inv1pe : ex * inv1pe;
                    const bool ok = mvalid && i < nvalid;
                    ll += ok ? fmaf(xv, lg, -sp) : 0.f;
                    v[i] = ok ? (sg - xv) * epi.inv_bg : 0.f;
                  }
                }
                epi.partial += ll;
              }
              uint4 lo, hi;
              pack16(v, lo, hi);
              sts128(patch_unit<64>(patch, lane, 2 * c), lo); sts128(patch_unit<64>(patch, lane, 2 * c + 1), hi);
            }
          }
        }
        if constexpr (KIND == EK_STORE_BF16) {
          if (CHAIN_RELU_BITS && epi.relu_bits && mvalid) {
            if (obits_chunks < 2) obits = (obits << 16) | 0xFFFFu;     // the group's second chunk lies beyond N
            epi.relu_bits[(int64_t)((n0 + gcol) >> 5) * epi.ld_bits + m] = ~obits;   // a warp's 32 rows: one 128-byte line
          }
        }
        fence_proxy_async();                                  // generic-proxy writes to the patch -> visible to the bulk store
        __syncwarp();
        if (lane == 0) {
          if constexpr (KIND == EK_ATOMIC) {
            if (J.zslice) tma_store_3d(&maps[J.d], patch, n0 + gcol, mrow0, z);
            else tma_reduce_add_2d(&maps[J.d], patch, n0 + gcol, mrow0);
          } else {
            tma_store_2d(&maps[J.d], patch, n0 + gcol, mrow0);
          }
          bulk_commit();
        }
        if constexpr (KIND == EK_RELUMASK || KIND == EK_BCE) {
          if (cs_dst) {
            const int ncols = min(gw * CW, N - (n0 + gcol));
            patch_colsum_bf16<64>(patch, scs_all + gcol, ncols, lane);
          }
        }
      }
    }
    tc_fence_before();
    if (tr) trace[16 * it + 9] = clock64();
    if constexpr (KIND == EK_STORE_F32) {
      if (J.fuse != 0) fence_proxy_async_global();   // the fused head's bf16 rows are read through TMA by later jobs
    }
    __syncwarp();
    if (lane == 0) {
      if (PAIR) mbar_arrive_leader(&S.tmem_empty_bar[as]);   // the leader's MMA warp waits for the epilogue warps of both CTAs
      else mbar_arrive(&S.tmem_empty_bar[as]);
      if (J.sig_base >= 0) {
        // rows stored by the bulk copies (async proxy) must be complete and visible before the row block is released
        if constexpr (KIND != EK_STORE_F32) { bulk_wait0(); fence_proxy_async_global(); }
        release_counter(counters + J.sig_base + mb, abl & 8);
      }
    }
    if (tr) trace[16 * it + 10] = clock64();
    if (js) {
      const unsigned long long t2 = gtimer();
      atomicMax(jobstat + 8 * jidx + 1, t2);
      atomicAdd(jobstat + 8 * jidx + 4, t2 - js_t1);
      atomicAdd(jobstat + 8 * jidx + 5, js_t1 - js_t0);
      atomicAdd(jobstat + 8 * jidx + 6, 1ull);
    }
  }
  epi.finish_warp();
  if constexpr (KIND == EK_STORE_F32) {
    if (J.fuse == EK_ROWS_Y_FWD) {
      const RowsYFwd& yp = *reinterpret_cast<const RowsYFwd*>(J.epi2);
      const float sacc = warp_sum(fuse_acc);
      if (lane == 0 && sacc != 0.f) acc_add(yp.acc, ACC_NENT, sacc * yp.inv_bg);
    } else if (J.fuse == EK_ROWS_Y_BWD) {
      const RowsYBwd& yp = *reinterpret_cast<const RowsYBwd*>(J.epi2);
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      if (et < yp.K && yp.db && scs_all[et] != 0.f) atomicAdd(yp.db + et, scs_all[et]);
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    }
  }
  if (cs_dst && cs_n0 >= 0) {
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    cs_flush();
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  }
}

// ---- row jobs ---------------------------------------------------------------------------------
// Data written earlier in this launch by other SMs is read with ld.global.cg (L2), never through L1.
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

template <int KIND, class P, int CL>
__device__ __forceinline__ void chain_rows_job(const ChainJob& J, int* counters, const ChainShared& S, int warp, int lane,
                                               unsigned long long* jobstat = nullptr, int jidx = 0, int abl = 0) {
  const P prm = *reinterpret_cast<const P*>(J.epi);
  int first, wstride;
  if (!chain_walk<CL>(J, (int)blockIdx.x, (int)gridDim.x, first, wstride) || first >= J.total_tiles) return;
  const int M = J.M;
  const int et = (int)threadIdx.x - 64;                 // 0 .. 511
  constexpr int NT = EPI_WARPS * 32;
  float red_acc = 0.f;                                   // kl / nent partial of this thread over the job's tiles
  float cs[16];                                          // column-sum partials (bias gradients) of this thread (z head)
#pragma unroll
  for (int i = 0; i < 16; ++i) cs[i] = 0.f;
  if constexpr (KIND == EK_ROWS_Y_BWD) {                 // the y head accumulates its column sums in the CTA accumulator as it goes
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    for (int i = et; i < 256; i += NT) S.scs_all[i] = 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  }
  // A tile is 1/sub of a 128-row block (J.tiles_n = sub): the z heads use 32-row tiles -- one float4 item per epilogue thread -- so
  // that a head stage spreads over every CTA instead of one CTA per row block; every tile signals its block's counter.
  const int sub = J.tiles_n, rpt = BLOCK_M / sub;
  for (int l = first; l < J.total_tiles; l += wstride) {
    const int mb = l / sub, m0 = l * rpt;
    const int rows = max(0, min(rpt, M - m0));
    const bool js = jobstat && warp == 2 && lane == 0;
    unsigned long long js_t0 = 0, js_t1 = 0;
    if (js) js_t0 = gtimer();
    if (lane == 0) {
      for (int d = 0; d < J.ndeps; ++d) wait_counter(counters + J.deps[d].base + mb, J.deps[d].target);
    }
    __syncwarp();
    if (js) { js_t1 = gtimer(); atomicMin(jobstat + 8 * jidx + 0, js_t0); atomicAdd(jobstat + 8 * jidx + 2, js_t1 - js_t0); }
    if constexpr (KIND == EK_ROWS_Z_FWD) {
      const int Z = prm.Z, tpr = Z >> 2;
      for (int t = et; t < rows * tpr; t += NT) {
        const int b = m0 + t / tpr, j = (t % tpr) * 4;
        const float4 mu = ldcg4(prm.enc_out + (int64_t)b * 2 * Z + j), raw = ldcg4(prm.enc_out + (int64_t)b * 2 * Z + Z + j);
        const float4 e4 = ldcg4(prm.eps + (int64_t)b * Z + j);
        float4 mp = make_float4(0.f, 0.f, 0.f, 0.f), rp = mp;
        if (prm.prior_mode == 2) { mp = ldcg4(prm.prior_out + (int64_t)b * 2 * Z + j); rp = ldcg4(prm.prior_out + (int64_t)b * 2 * Z + Z + j); }
        const float* MU = &mu.x; const float* RAW = &raw.x; const float* E = &e4.x; const float* MP = &mp.x; const float* RP = &rp.x;
        float z[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float sg = fmaxf(fast_softplus(RAW[q] + prm.c), prm.sigma_min);
          z[q] = fmaf(sg, E[q], MU[q]);
          // log q - log p = -e^2/2 - log sg + tt^2/2 + log sp = (tt^2 - e^2)/2 + log(sp / sg)
          float d = -0.5f * E[q] * E[q];
          if (prm.prior_mode == 0) {
            d = fmaf(0.5f * z[q], z[q], d) - __logf(sg);
          } else if (prm.prior_mode == 2) {
            const float sp = fmaxf(fast_softplus(RP[q] + prm.c), prm.sigma_min);
            const float isp = __fdividef(1.f, sp);
            const float tt = (z[q] - MP[q]) * isp;
            d = fmaf(0.5f * tt, tt, d) - __logf(sg * isp);
          } else {
            d -= __logf(sg);
          }
          red_acc += d;
        }
        *reinterpret_cast<uint2*>(prm.z_act + (int64_t)b * prm.ld_z + j) = make_uint2(pack_bf16x2(z[0], z[1]), pack_bf16x2(z[2], z[3]));
      }
    } else if constexpr (KIND == EK_ROWS_Z_BWD) {
      const int Z = prm.Z, tpr = Z >> 2;                 // NT % tpr == 0 (checked by the host): a thread keeps its 4 columns
      const int j = (et % tpr) * 4;
      for (int t = et; t < rows * tpr; t += NT) {
        const int b = m0 + t / tpr;
        const float4 mu = ldcg4(prm.enc_out + (int64_t)b * 2 * Z + j), raw = ldcg4(prm.enc_out + (int64_t)b * 2 * Z + Z + j);
        const float4 e4 = ldcg4(prm.eps + (int64_t)b * Z + j), dzd = ldcg4(prm.dz_dec + (int64_t)b * Z + j);
        float4 mp = make_float4(0.f, 0.f, 0.f, 0.f), rp = mp;
        if (prm.prior_mode == 2) { mp = ldcg4(prm.prior_out + (int64_t)b * 2 * Z + j); rp = ldcg4(prm.prior_out + (int64_t)b * 2 * Z + Z + j); }
        const float* MU = &mu.x; const float* RAW = &raw.x; const float* E = &e4.x; const float* DZ = &dzd.x;
        const float* MP = &mp.x; const float* RP = &rp.x;
        float g0[4], g1[4], a0[4], a1[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          // softplus(t) and sigmoid(t) from ONE exponential: e = exp(-|t|), softplus = max(t,0) + log(1+e), sigmoid = (t>=0 ? 1 : e)/(1+e)
          const float tq = RAW[q] + prm.c;
          const float eq = __expf(-fabsf(tq)), iq = __fdividef(1.f, 1.f + eq);
          const float spq = fmaxf(tq, 0.f) + log1p_fast(eq);
          const float sgm_q = tq >= 0.f ? iq : eq * iq;
          const float sg = fmaxf(spq, prm.sigma_min);
          const float z = fmaf(sg, E[q], MU[q]);
          float dz = DZ[q];
          a0[q] = 0.f; a1[q] = 0.f;
          if (prm.prior_mode == 0) {
            dz += z * prm.inv_bg;
          } else {
            const float tp = RP[q] + prm.c;
            const float ep = __expf(-fabsf(tp)), ip = __fdividef(1.f, 1.f + ep);
            const float spp = fmaxf(tp, 0.f) + log1p_fast(ep);
            const float sgm_p = tp >= 0.f ? ip : ep * ip;
            const float sp = fmaxf(spp, prm.sigma_min);
            const float d = z - MP[q];
            const float isp = __fdividef(1.f, sp);
            const float isp2 = isp * isp;
            dz += d * isp2 * prm.inv_bg;
            const float dsp = (isp - d * d * isp2 * isp) * prm.inv_bg;
            a0[q] = __bfloat162float(__float2bfloat16_rn(-d * isp2 * prm.inv_bg));
            a1[q] = __bfloat162float(__float2bfloat16_rn(spp >= prm.sigma_min ? dsp * sgm_p : 0.f));
          }
          const float dsg = dz * E[q] - prm.inv_bg * __fdividef(1.f, sg);
          g0[q] = __bfloat162float(__float2bfloat16_rn(dz));
          g1[q] = __bfloat162float(__float2bfloat16_rn(spq >= prm.sigma_min ? dsg * sgm_q : 0.f));
          cs[q] += g0[q]; cs[4 + q] += g1[q]; cs[8 + q] += a0[q]; cs[12 + q] += a1[q];     // sums of the values as stored
        }
        *reinterpret_cast<uint2*>(prm.d_enc_out + (int64_t)b * prm.ld_out + j) = make_uint2(pack_bf16x2(g0[0], g0[1]), pack_bf16x2(g0[2], g0[3]));
        *reinterpret_cast<uint2*>(prm.d_enc_out + (int64_t)b * prm.ld_out + Z + j) = make_uint2(pack_bf16x2(g1[0], g1[1]), pack_bf16x2(g1[2], g1[3]));
        if (prm.prior_mode == 2) {
          *reinterpret_cast<uint2*>(prm.d_prior_out + (int64_t)b * prm.ld_out + j) = make_uint2(pack_bf16x2(a0[0], a0[1]), pack_bf16x2(a0[2], a0[3]));
          *reinterpret_cast<uint2*>(prm.d_prior_out + (int64_t)b * prm.ld_out + Z + j) = make_uint2(pack_bf16x2(a1[0], a1[1]), pack_bf16x2(a1[2], a1[3]));
        }
      }
    } else if constexpr (KIND == EK_ROWS_Y_FWD) {
      if (et < BLOCK_M) {                                   // warps 0-3, whole warps
        const int64_t row = m0 + et;
        const bool valid = et < rows;
        float lg[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) lg[k] = -INFINITY;
        if (valid) ld_row16(prm.logits + row * prm.K, prm.K, lg, -INFINITY);
        red_acc += y_head_fwd_row(lg, prm, row, valid);
      }
    } else if constexpr (KIND == EK_ROWS_Y_BWD) {
      if (et < BLOCK_M) {
        const int64_t row = m0 + et;
        const bool valid = et < rows;
        float g[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) g[k] = (valid && k < prm.K) ? __ldcg(prm.dy + row * prm.K + k) : 0.f;
        y_head_bwd_row(g, prm, row, valid, S.scs_all);
      }
    }
    // release the row block: the rows are read by later jobs through TMA (async proxy) and by plain loads
    fence_proxy_async_global();
    __syncwarp();
    if (lane == 0 && J.sig_base >= 0) release_counter(counters + J.sig_base + mb, abl & 8);
    if (js) {
      const unsigned long long t2 = gtimer();
      atomicMax(jobstat + 8 * jidx + 1, t2); atomicAdd(jobstat + 8 * jidx + 4, t2 - js_t1); atomicAdd(jobstat + 8 * jidx + 6, 1ull);
    }
  }
  // ---- per-job reductions of this CTA
  if constexpr (KIND == EK_ROWS_Z_FWD || KIND == EK_ROWS_Y_FWD) {
    const float s = warp_sum(red_acc);
    if (lane == 0 && s != 0.f) acc_add(prm.acc, KIND == EK_ROWS_Z_FWD ? ACC_KL : ACC_NENT, s * prm.inv_bg);
  }
  if constexpr (KIND == EK_ROWS_Z_BWD) {
    // bias gradients: register partials -> CTA accumulator in shared memory -> one atomic per column
    float* const scs = S.scs_all;                        // 256 floats
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    for (int i = et; i < 256; i += NT) scs[i] = 0.f;
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    const int Z = prm.Z, j = (et % (Z >> 2)) * 4;
#pragma unroll
    for (int p4 = 0; p4 < 4; ++p4)
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (cs[4 * p4 + q] != 0.f) atomicAdd(scs + p4 * Z + j + q, cs[4 * p4 + q]);
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    for (int col = et; col < 4 * Z; col += NT) {
      const int p4 = col / Z, jj = col % Z;
      const float t = scs[col];
      if (prm.db_enc && t != 0.f && (p4 < 2 || prm.prior_mode == 2)) atomicAdd((p4 < 2 ? prm.db_enc : prm.db_prior) + (p4 & 1) * Z + jj, t);
    }
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  }
  if constexpr (KIND == EK_ROWS_Y_BWD) {
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
    if (et < prm.K && S.scs_all[et] != 0.f && prm.db) atomicAdd(prm.db + et, S.scs_all[et]);
    asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
  }
}

// CL = CTAs per walker: 1 (single CTAs, cta_group::1), 2 (CTA pairs, cta_group::2), 4 (QUAD: clusters of two CTA pairs that take the two
// n-tiles of a row block together and load its A rows ONCE -- each CTA loads half of its 128 rows and multicasts them to the CTA of the
// same rank in the other pair.  The operand stream from L2 is what bounds the kernel (profiles/r2_ablation_loads.md): 96 instead of
// 128 KB per two 256 x 256 x 64 steps).
template <class Params, int CL>
__global__ void __launch_bounds__(NUM_THREADS2, 1) gemm_chain_kernel(const __grid_constant__ Params p) {
  constexpr bool PAIR = CL >= 2, QUAD = CL == 4;
  constexpr int STAGES = PAIR ? CHAIN_STAGES_PAIR : CHAIN_STAGES, STAGE_BYTES = PAIR ? CHAIN_STAGE_BYTES_PAIR : CHAIN_STAGE_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  if (smem - smem_raw + CHAIN_CARVE_BYTES > CHAIN_SMEM_BYTES) __trap();   // dynamic shared memory starts (at most 512 B off) a 1 KB boundary
  uint8_t* patches = smem + STAGES * STAGE_BYTES;                       // 1024-byte aligned: TMA boxes with 64-byte swizzle
  uint64_t* bars = reinterpret_cast<uint64_t*>(patches + EPI_WARPS * CHAIN_PATCH_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tmem_full_bar = bars + 2 * STAGES;
  uint64_t* tmem_empty_bar = bars + 2 * STAGES + 2;
  uint64_t* op_bar = bars + 2 * STAGES + 4;                             // [EPI_WARPS] epilogue operand boxes
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(op_bar + EPI_WARPS);
  float* sbias_all = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);
  float* scs_all = sbias_all + 256;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // GEMM tiles: G walkers (CTAs, or CTA pairs), this one is number c; `rank` = this CTA's place in its pair
  const int G = (int)gridDim.x / CL, c = (int)blockIdx.x / CL;
  const int crank = (int)blockIdx.x % CL;                   // place in the cluster; pair h = crank >> 1, place in the pair = crank & 1
  const int rank = crank & 1;
  long long* const trace = (p.trace && (int)blockIdx.x == p.trace_cta) ? p.trace : nullptr;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < p.nmaps; ++i) tma_prefetch_desc(&p.maps[i]);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], QUAD ? 2 : 1); }   // quad: a slot is free when BOTH pairs' MMAs have read it (the sibling CTA writes into it)
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full_bar[s], 1); mbar_init(&tmem_empty_bar[s], PAIR ? 2 * EPI_WARPS : EPI_WARPS); }
    for (int s = 0; s < EPI_WARPS; ++s) mbar_init(&op_bar[s], 1);
    fence_barrier_init();
  } else if (warp == 1) {
    if (PAIR) tmem_alloc_pair(tmem_slot, 512); else tmem_alloc(tmem_slot, 512);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) {
    if (cluster_ctarank() != (uint32_t)crank) __trap();     // the pair must be two CTAs of one cluster, leader = even block
    cluster_sync_all();                                       // the peer's barriers exist before anything is signalled on them
  }
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  griddep_wait();
  griddep_launch();

  if (warp == 0) {
    // ===== TMA producer =====
    // The WHOLE warp walks the schedule with uniform control flow -- loop state, job fields and addresses stay in uniform registers -- and
    // one elected lane issues the barrier / TMA instructions.  (Run by a single thread inside `if (lane == 0)` the same loop compiled to
    // ~130 dependent instructions per k-block -- indexed constant loads, R2UR moves and a vote loop around every UTMALDG -- and that
    // instruction chain, not L2 or the tensor pipe, paced the main loop: profiles/r2_ablation_loads.md.)
    int stage = 0; uint32_t phase = 0;
    int pit = 0;
    for (int j = 0; j < p.njobs; ++j) {
      const ChainJob& J = p.jobs[j];
      if (J.kind >= EK_ROWS_FIRST) continue;              // row jobs have no GEMM
      const int BN = J.block_n, kb1 = J.kb1, kb_total = J.kb1 + J.kb2, a_mn = J.a_mn, b_mn = J.b_mn, ndeps = J.ndeps;
      const int JM = J.M, JN = J.N, kps = J.kb_per_split, walk_total = J.walk_total, share = J.share;
      const CUtensorMap* const ta1 = &p.maps[J.a1];
      const CUtensorMap* const tb1 = &p.maps[J.b1];
      const CUtensorMap* const ta2 = &p.maps[J.a2];
      const CUtensorMap* const tb2 = &p.maps[J.b2];
      // pair mode: this CTA loads its 128 rows of A and HALF of the B tile (K-major: BN/2 rows; MN-major: 64-column slabs)
      const int bhalf = BN >> 1;
      const int b_slabs = PAIR ? (bhalf + 63) / 64 : BN / 64;
      const uint32_t b_bytes = PAIR ? (uint32_t)(b_mn ? b_slabs * (BLOCK_K * 128) : bhalf * BLOCK_K * 2) : (uint32_t)(BN * BLOCK_K * 2);
      const uint32_t tx_bytes = (PAIR ? 2u : 1u) * ((uint32_t)A_STAGE_BYTES + b_bytes);    // pair: both CTAs' loads land on the leader's barrier
      bool any_seg2 = false;
      for (int d = 0; d < ndeps; ++d) any_seg2 = any_seg2 || J.deps[d].seg2 != 0;
      int first, wstride;
      if (!chain_walk<1>(J, c, G, first, wstride)) continue;
      for (int l = first; l < walk_total; l += wstride, ++pit) {
        int z, mb, n0;
        chain_tile<CL>(J, l, crank, z, mb, n0);
        const int m0 = mb * BLOCK_M;
        const bool real = a_mn || m0 < JM;                 // K-major A: rows m0.. exist (a pair's second half may lie beyond M)
        const int n_eff = min(BN, (JN - n0 + 15) & ~15);
        const int nb = PAIR ? n0 + rank * (n_eff >> 1) : n0;  // first B column this CTA loads
        const int kb_begin = z * kps, kb_end = min(kb_total, kb_begin + kps);
        const bool tr = trace && pit < 64 && lane == 0;
        if (tr) trace[16 * pit + 0] = clock64();
        unsigned long long js_t0 = 0;
        if (p.jobstat) js_t0 = gtimer();
        if (ndeps > 0) {
          for (int d = 0; d < ndeps; ++d) {
            const ChainDep& D = J.deps[d];
            if (D.seg2) continue;
            if (!D.by_k) {
              if (real) wait_counter(p.counters + D.base + mb, D.target);
            } else {
              // every row block of the k-range: one counter per lane, polled in parallel (one thread walking them paid an L2 round
              // trip per block -- 9 us per weight-gradient tile at cfg4)
              const int lo = (kb_begin * BLOCK_K) / BLOCK_M, hi = min(D.nblocks - 1, (kb_end * BLOCK_K - 1) / BLOCK_M);
              for (int b0 = lo; b0 <= hi; b0 += 32) {
                if (b0 + lane <= hi) wait_counter(p.counters + D.base + b0 + lane, D.target);
                __syncwarp();
              }
            }
          }
          fence_proxy_async_global();                       // (every lane: whichever is elected below has acquired and fenced)
          __syncwarp();
        }
        if (tr) trace[16 * pit + 1] = clock64();
        if (p.jobstat && lane == 0) { atomicMin(p.jobstat + 8 * j + 0, js_t0); atomicAdd(p.jobstat + 8 * j + 2, gtimer() - js_t0); }
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          if (kb == kb1 && any_seg2) {
            // operands of the second K segment may arrive later: the first segment's MMAs run while their producer finishes
            for (int d = 0; d < ndeps; ++d)
              if (J.deps[d].seg2 && real) wait_counter(p.counters + J.deps[d].base + mb, J.deps[d].target);
            fence_proxy_async_global();
          }
          mbar_wait(&empty_bar[stage], phase ^ 1);
          const bool seg2 = kb >= kb1;
          const CUtensorMap* const ta = seg2 ? ta2 : ta1;
          const CUtensorMap* const tb = seg2 ? tb2 : tb1;
          const int k_elem = (seg2 ? kb - kb1 : kb) * BLOCK_K;
          uint8_t* const sa = smem + stage * STAGE_BYTES;
          uint8_t* const sb = sa + A_STAGE_BYTES;
          uint64_t* const fb = &full_bar[stage];
          if (elect_one()) {
#ifdef GMVAE_CHAIN_ABL
            if (p.abl & 2) {
              if (!PAIR || rank == 0) mbar_arrive(fb);
            } else
#endif
            {
              if (!PAIR || rank == 0) mbar_expect_tx(fb, tx_bytes);
              auto ld = [&](const CUtensorMap* m, void* dst, int c0, int c1) {
                if (PAIR) tma_load_2d_pair(m, fb, dst, c0, c1); else tma_load_2d(m, fb, dst, c0, c1);
              };
              if (QUAD) {
                // A in two halves of 64 rows (8 KB; the K-major maps of this mode have 64-row boxes).  Shared rows: this CTA loads half
                // h and multicasts it to the CTA of the same rank in the other pair, which loads the other half for both.
                const int hh = crank >> 1;
                if (share) {
                  const uint16_t mask = (uint16_t)((1u << rank) | (1u << (rank + 2)));
                  if (a_mn) tma_load_2d_pair_mc(ta, fb, sa + hh * 8192, m0 + hh * 64, k_elem, mask);
                  else tma_load_2d_pair_mc(ta, fb, sa + hh * 8192, k_elem, m0 + hh * 64, mask);
                } else {
#pragma unroll
                  for (int i = 0; i < 2; ++i) {
                    if (a_mn) ld(ta, sa + i * 8192, m0 + i * 64, k_elem); else ld(ta, sa + i * 8192, k_elem, m0 + i * 64);
                  }
                }
              } else if (a_mn) {
#pragma unroll
                for (int i = 0; i < BLOCK_M / 64; ++i) ld(ta, sa + i * (BLOCK_K * 128), m0 + i * 64, k_elem);
              } else {
                ld(ta, sa, k_elem, m0);
              }
              if (b_mn) {
                for (int i = 0; i < b_slabs; ++i) ld(tb, sb + i * (BLOCK_K * 128), nb + i * 64, k_elem);
              } else {
                ld(tb, sb, k_elem, nb);
              }
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (tr) trace[16 * pit + 2] = clock64();
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (the warp walks the schedule uniformly, one elected lane issues; in pair mode the leader CTA's warp, for both CTAs) =====
    int stage = 0; uint32_t phase = 0;
    int it = 0;
    for (int j = 0; (!PAIR || rank == 0) && j < p.njobs; ++j) {
      const ChainJob& J = p.jobs[j];
      if (J.kind >= EK_ROWS_FIRST) continue;
      const int kb_total = J.kb1 + J.kb2, kps = J.kb_per_split, walk_total = J.walk_total, BN = J.block_n, JN = J.N;
      const int a_mn = J.a_mn, b_mn = J.b_mn;
      const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
                              ((uint32_t)((PAIR ? 2 * BLOCK_M : BLOCK_M) >> 4) << 24);
      const uint64_t a_step = a_mn ? (UMMA_K * 128) >> 4 : (UMMA_K * 2) >> 4;
      const uint64_t b_step = b_mn ? (UMMA_K * 128) >> 4 : (UMMA_K * 2) >> 4;
      const uint64_t adesc_hi = make_smem_desc_rt(0, a_mn), bdesc_hi = make_smem_desc_rt(0, b_mn);
      int first, wstride;
      if (!chain_walk<1>(J, c, G, first, wstride)) continue;
      for (int l = first; l < walk_total; l += wstride, ++it) {
        int z, mb_unused, n0;
        chain_tile<CL>(J, l, crank, z, mb_unused, n0);
        const int kb_begin = z * kps, kb_end = min(kb_total, kb_begin + kps);
        const int as = it & 1; const uint32_t ap = (it >> 1) & 1;
        // a ragged last n-tile runs a narrower MMA (N multiple of 16): the zero-filled columns are not multiplied
        const int n_eff = min(BN, (JN - n0 + 15) & ~15);
        const uint32_t idesc = idesc0 | ((uint32_t)(n_eff >> 3) << 17);
        const bool tr = trace && it < 64 && lane == 0;
        if (tr) trace[16 * it + 3] = clock64();
        unsigned long long js_t0 = 0, js_t1 = 0;
        if (p.jobstat) js_t0 = gtimer();
        mbar_wait(&tmem_empty_bar[as], ap ^ 1);
        tc_fence_after();
        if (p.jobstat) js_t1 = gtimer();
        const uint32_t tmem_d = tmem_base + (uint32_t)(as * 256);
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          if (tr && kb == kb_begin) trace[16 * it + 4] = clock64();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint64_t adesc = adesc_hi | (uint64_t)((sa & 0x3FFFF) >> 4);
          const uint64_t bdesc = bdesc_hi | (uint64_t)(((sa + A_STAGE_BYTES) & 0x3FFFF) >> 4);
          if (elect_one()) {
#ifdef GMVAE_CHAIN_ABL
            if (!(p.abl & 4))
#endif
#pragma unroll
            for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
              if (PAIR) umma_bf16_pair(adesc + (uint64_t)k * a_step, bdesc + (uint64_t)k * b_step, tmem_d, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
              else umma_bf16(adesc + (uint64_t)k * a_step, bdesc + (uint64_t)k * b_step, tmem_d, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
            }
            if (QUAD) umma_commit_mc(&empty_bar[stage], (uint16_t)0xF);      // the slot is released in all four CTAs
            else if (PAIR) umma_commit_pair(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (elect_one()) {
          if (QUAD) umma_commit_mc(&tmem_full_bar[as], (uint16_t)(3u << (crank & 2)));
          else if (PAIR) umma_commit_pair(&tmem_full_bar[as]); else umma_commit(&tmem_full_bar[as]);
        }
        if (tr) trace[16 * it + 5] = clock64();
        if (p.jobstat && lane == 0) { atomicAdd(p.jobstat + 8 * j + 3, gtimer() - js_t1); atomicAdd(p.jobstat + 8 * j + 7, js_t1 - js_t0); }
      }
    }
  } else {
    // ===== epilogue warps =====
    ChainShared S{smem, full_bar, empty_bar, tmem_full_bar, tmem_empty_bar, patches, sbias_all, scs_all, tmem_base, op_bar};
    int it = 0;
    uint32_t op_phase = 0;
    for (int j = 0; j < p.njobs; ++j) {
      const ChainJob& J = p.jobs[j];
      switch (J.kind) {
        case EK_STORE_BF16: chain_epilogue_job<EpiStore<bf16, EPI_PLAIN>, EK_STORE_BF16, CL>(J, p.maps, p.counters, S, it, op_phase, warp, lane, trace, j, p.jobstat, p.abl); break;
        case EK_STORE_F32: chain_epilogue_job<EpiStore<float, EPI_PLAIN>, EK_STORE_F32, CL>(J, p.maps, p.counters, S, it, op_phase, warp, lane, trace, j, p.jobstat, p.abl); break;
        case EK_BCE: chain_epilogue_job<EpiBCE<bf16>, EK_BCE, CL>(J, p.maps, p.counters, S, it, op_phase, warp, lane, trace, j, p.jobstat, p.abl); break;
        case EK_RELUMASK: chain_epilogue_job<EpiReluMask<bf16, bf16>, EK_RELUMASK, CL>(J, p.maps, p.counters, S, it, op_phase, warp, lane, trace, j, p.jobstat, p.abl); break;
        case EK_ATOMIC: chain_epilogue_job<EpiAtomicAdd, EK_ATOMIC, CL>(J, p.maps, p.counters, S, it, op_phase, warp, lane, trace, j, p.jobstat, p.abl); break;
#ifndef GMVAE_NO_ROWS
        case EK_ROWS_Y_FWD: chain_rows_job<EK_ROWS_Y_FWD, RowsYFwd, CL>(J, p.counters, S, warp, lane, p.jobstat, j, p.abl); break;
        case EK_ROWS_Z_FWD: chain_rows_job<EK_ROWS_Z_FWD, RowsZFwd, CL>(J, p.counters, S, warp, lane, p.jobstat, j, p.abl); break;
        case EK_ROWS_Z_BWD: chain_rows_job<EK_ROWS_Z_BWD, RowsZBwd, CL>(J, p.counters, S, warp, lane, p.jobstat, j, p.abl); break;
        case EK_ROWS_Y_BWD: chain_rows_job<EK_ROWS_Y_BWD, RowsYBwd, CL>(J, p.counters, S, warp, lane, p.jobstat, j, p.abl); break;
#endif
        default: break;
      }
    }
  }
  if (warp >= 2 && lane == 0) bulk_wait0();     // outstanding bulk stores read this CTA's shared memory
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();                 // no CTA of a pair leaves (or frees tensor memory) while the other may still signal it
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_pair(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace tc
}  // namespace gmvae

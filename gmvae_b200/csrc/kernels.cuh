// kernels.cuh -- the non-GEMM kernels of the training step: input conversion, noise, the
// distribution "heads" (Gumbel-softmax / entropy, reparameterised Gaussian sample and KL terms,
// mixture prior), bias gradients, TF-form Adam and the bf16 operand refresh.
#pragma once
#include "common.cuh"
#include "epilogue.cuh"

namespace gmvae {


// bf16 GEMM-operand copy of one weight matrix
struct ShadowEntry {
  const float* w; bf16* w_bf16;
  long long off;             // flat offset of the matrix in the parameter buffer
  int rows, cols, ld_w;
  int tiles_x, tile_begin;   // tiles along cols; first flat tile index of this entry
};

struct DeviceState {           // owned by the handle, lives on the device
  long long step;              // global_step (runners.py:171)
  unsigned long long seed;
  unsigned int adam_blocks;    // blocks of the running Adam launch that have read the state (the last one advances it)
  unsigned int pad;
  double beta1_power, beta2_power;   // beta^step: tf.train.AdamOptimizer's non-trainable beta1_power / beta2_power accumulators
};

// ---- x: bool bytes -> GEMM operand type (vae.py:75, gmvae.py:86,104: tf.cast(x, float32)) ----
template <typename T>
__device__ __forceinline__ void convert_x_body(const uint8_t* __restrict__ x, T* __restrict__ out, int64_t n, int64_t block) {
  int64_t i = (block * blockDim.x + threadIdx.x) * 16;
  if (i + 16 <= n) {
    uint4 t = *reinterpret_cast<const uint4*>(x + i);
    const uint8_t* p = reinterpret_cast<const uint8_t*>(&t);
    __align__(16) T v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = from_f32<T>((float)p[j]);
    uint4* dst = reinterpret_cast<uint4*>(out + i);            // n*sizeof(T) stays 16-byte aligned
    const uint4* src = reinterpret_cast<const uint4*>(v);
#pragma unroll
    for (int j = 0; j < (int)(16 * sizeof(T) / 16); ++j) dst[j] = src[j];
  } else {
    for (int64_t j = i; j < n; ++j) out[j] = from_f32<T>((float)x[j]);
  }
}
template <typename T>
__global__ void convert_x_kernel(const uint8_t* __restrict__ x, T* __restrict__ out, int64_t n) {
  griddep_wait();
  griddep_launch();
  convert_x_body<T>(x, out, n, blockIdx.x);
}

// generic variant: rows of D bytes -> rows of ld elements (ld >= D; padding left untouched)
template <typename T>
__global__ void convert_x_rows_kernel(const uint8_t* __restrict__ x, T* __restrict__ out, int B, int D, int ld) {
  griddep_wait();
  griddep_launch();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)B * D) {
    int64_t r = i / D, c = i % D;
    out[r * ld + c] = from_f32<T>((float)x[i]);
  }
}

// ---- noise (only when the caller does not inject it) -----------------------------------------
// eps ~ N(0,1) (tf.random_normal inside MultivariateNormalDiag.sample), u ~ U(tiny,1)
// (RelaxedOneHotCategorical.sample).  Keyed by (seed, step, stream id, element index).
// `gumbel` != 0: the uniforms are stored as Gumbel noise g = -log(-log u) (what RelaxedOneHotCategorical.sample adds to the
// logits, SURVEY Appendix B.5) -- the two logarithms run here, in a fully parallel coalesced kernel, instead of in the
// q(y|x) head, which sits on the critical path of the step.
__device__ __forceinline__ float gumbel_of(float u) { return -logf(-logf(u)); }
__device__ __forceinline__ void fill_noise_body(float* __restrict__ eps, int64_t n_eps, float* __restrict__ u, int64_t n_u,
                                                const DeviceState* st, uint64_t rank_stream, int64_t block, int gumbel = 0, uint64_t draw = 0) {
  // keyed by (seed, global_step, draw, rank, element): `draw` is 0 inside a training step (the device step counter advances, so a
  // captured graph draws fresh noise at every replay) and a host counter for every other call (encode, run_model, summaries), which
  // do not advance the step -- the reference draws fresh noise on every sess.run
  const uint64_t seed = st->seed ^ (draw * 0xD6E8FEB86659FD93ull), step = (uint64_t)st->step;
  int64_t i = block * blockDim.x + threadIdx.x;
  int64_t q_eps = (n_eps + 3) / 4, q_u = (n_u + 3) / 4;
  uint32_t r[4];
  if (i < q_eps) {
    Philox::gen(seed ^ (step * 0x9E3779B97F4A7C15ull), rank_stream * 2, (uint64_t)i, r);
    float a0 = sqrtf(-2.f * logf(u01(r[0]))), a1 = sqrtf(-2.f * logf(u01(r[2])));
    float s0, c0, s1, c1;
    sincospif(2.f * u01(r[1]), &s0, &c0);
    sincospif(2.f * u01(r[3]), &s1, &c1);
    float v[4] = {a0 * c0, a0 * s0, a1 * c1, a1 * s1};
    for (int j = 0; j < 4; ++j)
      if (i * 4 + j < n_eps) eps[i * 4 + j] = v[j];
  } else if (i < q_eps + q_u) {
    int64_t k = i - q_eps;
    Philox::gen(seed ^ (step * 0x9E3779B97F4A7C15ull), rank_stream * 2 + 1, (uint64_t)k, r);
    for (int j = 0; j < 4; ++j)
      if (k * 4 + j < n_u) u[k * 4 + j] = gumbel ? gumbel_of(u01(r[j])) : u01(r[j]);
  }
}
__global__ void fill_noise_kernel(float* __restrict__ eps, int64_t n_eps, float* __restrict__ u, int64_t n_u,
                                  const DeviceState* st, uint64_t rank_stream, int gumbel, uint64_t draw) {
  griddep_wait();
  griddep_launch();
  fill_noise_body(eps, n_eps, u, n_u, st, rank_stream, blockIdx.x, gumbel, draw);
}
// injected uniforms (parity tests, run_model(..., gumbel_u=)) -> Gumbel noise
__global__ void gumbel_from_u_kernel(const float* __restrict__ u, float* __restrict__ g, int64_t n) {
  griddep_wait();
  griddep_launch();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) g[i] = gumbel_of(u[i]);
}
// first launch of a training step: blocks [0, x_blocks) convert the image bytes, the rest draw the noise
template <typename T>
__global__ void prologue_kernel(const uint8_t* __restrict__ x, T* __restrict__ out, int64_t n, int x_blocks, float* __restrict__ eps,
                                int64_t n_eps, float* __restrict__ u, int64_t n_u, const DeviceState* st, uint64_t rank_stream, uint64_t draw) {
  griddep_wait();
  griddep_launch();
  if ((int)blockIdx.x < x_blocks) convert_x_body<T>(x, out, n, blockIdx.x);
  else fill_noise_body(eps, n_eps, u, n_u, st, rank_stream, (int64_t)blockIdx.x - x_blocks, 1, draw);
}

// ---- q(y|x) head, forward (gmvae.py:238-240, 262-263; utils.py:165-170) ------------------------
// One warp per row.  p = softmax(l); nent += sum_k p log p / B;  y = softmax((l + g)/T),
// g = -log(-log u).  y is written twice: fp32 for the backward pass and as the zero-padded GEMM
// operand of encoder_gmm layer 0 / prior_gmm.
constexpr int HEAD_MAXK = 128;
template <typename ActT>
__global__ void head_y_fwd_kernel(const float* __restrict__ logits, const float* __restrict__ gum, int B, int K, float inv_T,
                                  float inv_bg, float* __restrict__ y_f32, ActT* __restrict__ y_act, int ld_yact,
                                  float* __restrict__ acc) {
  griddep_wait();
  griddep_launch();
  __shared__ float scratch[32];
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  float ent = 0.f;
  if (row < B) {
    float l[HEAD_MAXK / 32], a[HEAD_MAXK / 32];
    float ml = -INFINITY, ma = -INFINITY;
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      l[i] = -INFINITY; a[i] = -INFINITY;
      if (k < K) {
        l[i] = logits[(int64_t)row * K + k];
        // gum = Gumbel noise -log(-log u); objective M passes null: y := softmax(logits) = q(y|x) itself
        a[i] = gum ? (l[i] + gum[(int64_t)row * K + k]) * inv_T : l[i];
      }
      ml = fmaxf(ml, l[i]); ma = fmaxf(ma, a[i]);
    }
    ml = warp_max(ml); ma = warp_max(ma);
    float sl = 0.f, nm = 0.f, sa = 0.f;
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      if (k < K) { if (l[i] == ml) nm += 1.f; else sl += expf(l[i] - ml); sa += expf(a[i] - ma); }
    }
    sl = warp_sum(sl); nm = warp_sum(nm); sa = warp_sum(sa);
    const float lo = lse_above_max(sl, nm), inv_sa = 1.f / sa;
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      if (k < K) {
        float logp = (l[i] - ml) - lo;
        ent += expf(logp) * logp;
        float y = expf(a[i] - ma) * inv_sa;
        y_f32[(int64_t)row * K + k] = y;
        y_act[(int64_t)row * ld_yact + k] = from_f32<ActT>(y);
      } else if (k < ld_yact) {
        y_act[(int64_t)row * ld_yact + k] = from_f32<ActT>(0.f);
      }
    }
  }
  float s = block_sum(ent, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_NENT, s * inv_bg);
}

// ---- q(y|x) head, backward --------------------------------------------------------------------
// dl = softmax-Jacobian((l+g)/T)^T dy / T  +  d nent/dl,   d nent/dl_j = p_j (log p_j - sum p log p)/B
template <typename ActT>
__global__ void head_y_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ y_f32,
                                  const float* __restrict__ dy, int B, int K, float inv_T, float inv_bg,
                                  ActT* __restrict__ dlogits, int ld_out, float* __restrict__ db) {
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  float cs[HEAD_MAXK / 32];                            // per-lane column sums (bias gradient of encoder_y's last layer)
#pragma unroll
  for (int i = 0; i < HEAD_MAXK / 32; ++i) cs[i] = 0.f;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < B; row += gridDim.x * wpb) {
  float l[HEAD_MAXK / 32], y[HEAD_MAXK / 32], g[HEAD_MAXK / 32];
  float ml = -INFINITY, ydy = 0.f;
#pragma unroll
  for (int i = 0; i < HEAD_MAXK / 32; ++i) {
    int k = lane + 32 * i;
    l[i] = -INFINITY; y[i] = 0.f; g[i] = 0.f;
    if (k < K) {
      l[i] = logits[(int64_t)row * K + k];
      y[i] = y_f32[(int64_t)row * K + k];
      g[i] = dy ? dy[(int64_t)row * K + k] : 0.f;
    }
    ml = fmaxf(ml, l[i]);
    ydy += y[i] * g[i];
  }
  ml = warp_max(ml); ydy = warp_sum(ydy);
  float sl = 0.f, nm = 0.f;
#pragma unroll
  for (int i = 0; i < HEAD_MAXK / 32; ++i)
    if (lane + 32 * i < K) { if (l[i] == ml) nm += 1.f; else sl += expf(l[i] - ml); }
  sl = warp_sum(sl); nm = warp_sum(nm);
  const float lo = lse_above_max(sl, nm);
  float plogp = 0.f;
#pragma unroll
  for (int i = 0; i < HEAD_MAXK / 32; ++i)
    if (lane + 32 * i < K) { float lp = (l[i] - ml) - lo; plogp += expf(lp) * lp; }
  plogp = warp_sum(plogp);
#pragma unroll
  for (int i = 0; i < HEAD_MAXK / 32; ++i) {
    int k = lane + 32 * i;
    if (k < K) {
      float lp = (l[i] - ml) - lo;
      ActT o = from_f32<ActT>(y[i] * (g[i] - ydy) * inv_T + expf(lp) * (lp - plogp) * inv_bg);
      dlogits[(int64_t)row * ld_out + k] = o;
      cs[i] += to_f32<ActT>(o);
    } else if (k < ld_out) {
      dlogits[(int64_t)row * ld_out + k] = from_f32<ActT>(0.f);
    }
  }
  }
  if (db) {
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      if (k < K && cs[i] != 0.f) atomicAdd(db + k, cs[i]);
    }
  }
}

// ---- q(y|x) head for HEAD_MAXK < K <= HEAD_WIDE_MAXK (GMVAE, objective R) --------------------------
// The math of head_y_fwd_kernel / head_y_bwd_kernel, one warp per row with MAXK / 32 values per lane.  MAXK (256, 512 or
// 1024) is the smallest that holds K (engine.cu head_y_wide_fwd / _bwd), so a 129-wide head does not pay for 1024 registers'
// worth of row.  Objective R only: the Gumbel noise and dy are always present.  Blocks of HEAD_WIDE_THREADS threads.
constexpr int HEAD_WIDE_MAXK = 1024, HEAD_WIDE_THREADS = 256;
template <typename ActT, int MAXK>
__global__ void __launch_bounds__(HEAD_WIDE_THREADS) head_y_wide_fwd_kernel(const float* __restrict__ logits, const float* __restrict__ gum,
                                                                            int B, int K, float inv_T, float inv_bg, float* __restrict__ y_f32,
                                                                            ActT* __restrict__ y_act, int ld_yact, float* __restrict__ acc) {
  constexpr int NI = MAXK / 32;
  griddep_wait();
  griddep_launch();
  __shared__ float scratch[32];
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (HEAD_WIDE_THREADS / 32) + (threadIdx.x >> 5);
  float ent = 0.f;
  if (row < B) {
    const float* lr = logits + (int64_t)row * K; const float* gr = gum + (int64_t)row * K;
    float l[NI], a[NI];
    float ml = -INFINITY, ma = -INFINITY;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int k = lane + 32 * i;
      l[i] = -INFINITY; a[i] = -INFINITY;
      if (k < K) { l[i] = lr[k]; a[i] = (l[i] + gr[k]) * inv_T; }
      ml = fmaxf(ml, l[i]); ma = fmaxf(ma, a[i]);
    }
    ml = warp_max(ml); ma = warp_max(ma);
    float sl = 0.f, nm = 0.f, sa = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i)
      if (lane + 32 * i < K) { if (l[i] == ml) nm += 1.f; else sl += expf(l[i] - ml); sa += expf(a[i] - ma); }
    sl = warp_sum(sl); nm = warp_sum(nm); sa = warp_sum(sa);
    const float lo = lse_above_max(sl, nm), inv_sa = 1.f / sa;
    float* yr = y_f32 + (int64_t)row * K; ActT* ar = y_act + (int64_t)row * ld_yact;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int k = lane + 32 * i;
      if (k < K) {
        const float logp = (l[i] - ml) - lo;
        ent += expf(logp) * logp;
        const float y = expf(a[i] - ma) * inv_sa;
        yr[k] = y;
        ar[k] = from_f32<ActT>(y);
      } else if (k < ld_yact) {
        ar[k] = from_f32<ActT>(0.f);
      }
    }
  }
  const float s = block_sum(ent, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_NENT, s * inv_bg);
}

// Rows are strided over the grid.  With `db` (default mode) each warp sums its rows' stored dl per column in its own slice of
// shared memory, and the block adds the slices with one global atomic per column; deterministic mode passes null and takes the
// bias gradient from its fixed-order column sum (engine.cu bias_grad).
template <typename ActT, int MAXK>
__global__ void __launch_bounds__(HEAD_WIDE_THREADS) head_y_wide_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ y_f32,
                                                                            const float* __restrict__ dy, int B, int K, float inv_T, float inv_bg,
                                                                            ActT* __restrict__ dlogits, int ld_out, float* __restrict__ db) {
  constexpr int NI = MAXK / 32, WARPS = HEAD_WIDE_THREADS / 32;
  griddep_wait();
  griddep_launch();
  __shared__ float cs[WARPS][MAXK];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (db) {
#pragma unroll
    for (int i = 0; i < NI; ++i) cs[w][lane + 32 * i] = 0.f;
  }
  for (int row = blockIdx.x * WARPS + w; row < B; row += gridDim.x * WARPS) {
    const float* lr = logits + (int64_t)row * K; const float* yr = y_f32 + (int64_t)row * K; const float* gr = dy + (int64_t)row * K;
    float l[NI], y[NI], g[NI];
    float ml = -INFINITY, ydy = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int k = lane + 32 * i;
      l[i] = -INFINITY; y[i] = 0.f; g[i] = 0.f;
      if (k < K) { l[i] = lr[k]; y[i] = yr[k]; g[i] = gr[k]; }
      ml = fmaxf(ml, l[i]);
      ydy += y[i] * g[i];
    }
    ml = warp_max(ml); ydy = warp_sum(ydy);
    float sl = 0.f, nm = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i)
      if (lane + 32 * i < K) { if (l[i] == ml) nm += 1.f; else sl += expf(l[i] - ml); }
    sl = warp_sum(sl); nm = warp_sum(nm);
    const float lo = lse_above_max(sl, nm);
    float plogp = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i)
      if (lane + 32 * i < K) { const float lp = (l[i] - ml) - lo; plogp += expf(lp) * lp; }
    plogp = warp_sum(plogp);
    ActT* orow = dlogits + (int64_t)row * ld_out;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int k = lane + 32 * i;
      if (k < K) {
        const float lp = (l[i] - ml) - lo;
        const ActT o = from_f32<ActT>(y[i] * (g[i] - ydy) * inv_T + expf(lp) * (lp - plogp) * inv_bg);
        orow[k] = o;
        if (db) cs[w][k] += to_f32<ActT>(o);
      } else if (k < ld_out) {
        orow[k] = from_f32<ActT>(0.f);
      }
    }
  }
  if (db) {
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += HEAD_WIDE_THREADS) {
      float t = 0.f;
#pragma unroll
      for (int j = 0; j < WARPS; ++j) t += cs[j][k];
      if (t != 0.f) atomicAdd(db + k, t);
    }
  }
}

// ---- q(z|.) head, forward (base.py:69-70; gmvae.py:248,258; vae.py:171,181) ---------------------
// enc_out = [mu | raw] (B x 2Z).  sigma = max(softplus(raw + c), sigma_min); z = mu + sigma eps.
// KL accumulator gets log q(z) - log p(z) summed over the batch, divided by the global batch:
//   log q(z) = -0.5 eps^2 - log sigma (-Z/2 log 2pi, cancels against the prior's constant)
//   prior_mode 0 (VAE):       log p = -0.5 z^2
//   prior_mode 1 (VAE_GMP):   handled by gmp_prior_kernel; only the log q part is added here
//   prior_mode 2 (GMVAE, R):  prior_out = [mu_p | raw_p] per row, log p = -0.5 ((z-mu_p)/s_p)^2 - log s_p
template <typename ActT>
__global__ void head_z_fwd_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps,
                                  const float* __restrict__ prior_out, int prior_mode, int B, int Z, float c,
                                  float sigma_min, float inv_bg, ActT* __restrict__ z_act, int ld_z, float* __restrict__ z_f32,
                                  float* __restrict__ acc) {
  griddep_wait();
  griddep_launch();
  __shared__ float scratch[32];
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float kl = 0.f;
  if (i < (int64_t)B * Z) {
    int b = (int)(i / Z), j = (int)(i % Z);
    float mu = enc_out[(int64_t)b * 2 * Z + j], raw = enc_out[(int64_t)b * 2 * Z + Z + j];
    float sg = fmaxf(softplus_f(raw + c), sigma_min);
    float e = eps[i];
    float z = fmaf(sg, e, mu);
    z_act[(int64_t)b * ld_z + j] = from_f32<ActT>(z);
    if (z_f32) z_f32[i] = z;
    float logq = -0.5f * e * e - logf(sg);
    float logp = 0.f;
    if (prior_mode == 0) {
      logp = -0.5f * z * z;
    } else if (prior_mode == 2) {
      float mp = prior_out[(int64_t)b * 2 * Z + j], rp = prior_out[(int64_t)b * 2 * Z + Z + j];
      float sp = fmaxf(softplus_f(rp + c), sigma_min);
      float t = (z - mp) / sp;
      logp = -0.5f * t * t - logf(sp);
    }
    kl = logq - logp;
  }
  float s = block_sum(kl, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_KL, s * inv_bg);
}

// ---- q(z|.) head, backward ---------------------------------------------------------------------
// dz = dz_dec + d kl/dz;  d mu_q = dz;  d sigma_q = dz eps - 1/(B sigma_q);  d raw = d sigma * sigmoid(raw+c)
// GMVAE: d mu_p = -(z-mu_p)/(B s_p^2); d s_p = (1/s_p - (z-mu_p)^2/s_p^3)/B.
template <typename ActT>
__global__ void head_z_bwd_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps,
                                  const float* __restrict__ prior_out, const float* __restrict__ dz_dec,
                                  const float* __restrict__ dz_prior, int prior_mode, int B, int Z, float c,
                                  float sigma_min, float inv_bg, ActT* __restrict__ d_enc_out,
                                  ActT* __restrict__ d_prior_out, int ld_out) {
  griddep_wait();
  griddep_launch();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * Z) return;
  int b = (int)(i / Z), j = (int)(i % Z);
  float mu = enc_out[(int64_t)b * 2 * Z + j], raw = enc_out[(int64_t)b * 2 * Z + Z + j];
  float spq = softplus_f(raw + c);
  float sg = fmaxf(spq, sigma_min);
  float e = eps[i];
  float z = fmaf(sg, e, mu);
  float dz = dz_dec[i];
  if (prior_mode == 0) {
    dz += z * inv_bg;
  } else if (prior_mode == 1) {
    dz += dz_prior[i];
  } else {
    float mp = prior_out[(int64_t)b * 2 * Z + j], rp = prior_out[(int64_t)b * 2 * Z + Z + j];
    float spp = softplus_f(rp + c);
    float sp = fmaxf(spp, sigma_min);
    float d = z - mp;
    float isp2 = 1.f / (sp * sp);
    dz += d * isp2 * inv_bg;
    float dsp = (1.f / sp - d * d * isp2 / sp) * inv_bg;
    d_prior_out[(int64_t)b * ld_out + j] = from_f32<ActT>(-d * isp2 * inv_bg);
    d_prior_out[(int64_t)b * ld_out + Z + j] = from_f32<ActT>(spp >= sigma_min ? dsp * sigmoid_f(rp + c) : 0.f);
  }
  float dsg = dz * e - inv_bg / sg;
  d_enc_out[(int64_t)b * ld_out + j] = from_f32<ActT>(dz);
  d_enc_out[(int64_t)b * ld_out + Z + j] = from_f32<ActT>(spq >= sigma_min ? dsg * sigmoid_f(raw + c) : 0.f);
}

// Persistent variant of head_z_bwd that also reduces the bias gradients of the last encoder layer
// (and of prior_gmm) over the batch: thread <-> latent dimension j, row lanes stride over the batch,
// one shared-memory reduction and 2-4 atomics per column per block.  Requires Z <= blockDim.x.
template <typename ActT>
__global__ void head_z_bwd_cs_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps,
                                     const float* __restrict__ prior_out, const float* __restrict__ dz_dec,
                                     const float* __restrict__ dz_prior, int prior_mode, int B, int Z, float c, float sigma_min,
                                     float inv_bg, ActT* __restrict__ d_enc_out, ActT* __restrict__ d_prior_out, int ld_out,
                                     float* __restrict__ db_enc, float* __restrict__ db_prior) {
  griddep_wait();
  griddep_launch();
  extern __shared__ float red[];                       // [4][blockDim.x]
  const int lanes = blockDim.x / Z;                    // row lanes per block
  const int j = threadIdx.x % Z, rl = threadIdx.x / Z;
  float s_mu = 0.f, s_raw = 0.f, s_pmu = 0.f, s_praw = 0.f;
  if (rl < lanes) {
    for (int b = blockIdx.x * lanes + rl; b < B; b += gridDim.x * lanes) {
      const int64_t i = (int64_t)b * Z + j;
      float mu = enc_out[(int64_t)b * 2 * Z + j], raw = enc_out[(int64_t)b * 2 * Z + Z + j];
      float spq = softplus_f(raw + c);
      float sg = fmaxf(spq, sigma_min);
      float e = eps[i];
      float z = fmaf(sg, e, mu);
      float dz = dz_dec[i];
      if (prior_mode == 0) {
        dz += z * inv_bg;
      } else if (prior_mode == 1) {
        dz += dz_prior[i];
      } else {
        float mp = prior_out[(int64_t)b * 2 * Z + j], rp = prior_out[(int64_t)b * 2 * Z + Z + j];
        float spp = softplus_f(rp + c);
        float sp = fmaxf(spp, sigma_min);
        float d = z - mp;
        float isp2 = 1.f / (sp * sp);
        dz += d * isp2 * inv_bg;
        float dsp = (1.f / sp - d * d * isp2 / sp) * inv_bg;
        ActT a0 = from_f32<ActT>(-d * isp2 * inv_bg), a1 = from_f32<ActT>(spp >= sigma_min ? dsp * sigmoid_f(rp + c) : 0.f);
        d_prior_out[(int64_t)b * ld_out + j] = a0; d_prior_out[(int64_t)b * ld_out + Z + j] = a1;
        s_pmu += to_f32<ActT>(a0); s_praw += to_f32<ActT>(a1);          // sums of the values as stored
      }
      float dsg = dz * e - inv_bg / sg;
      ActT g0 = from_f32<ActT>(dz), g1 = from_f32<ActT>(spq >= sigma_min ? dsg * sigmoid_f(raw + c) : 0.f);
      d_enc_out[(int64_t)b * ld_out + j] = g0; d_enc_out[(int64_t)b * ld_out + Z + j] = g1;
      s_mu += to_f32<ActT>(g0); s_raw += to_f32<ActT>(g1);
    }
  }
  const int n = blockDim.x;
  red[threadIdx.x] = s_mu; red[n + threadIdx.x] = s_raw; red[2 * n + threadIdx.x] = s_pmu; red[3 * n + threadIdx.x] = s_praw;
  __syncthreads();
  if (threadIdx.x < Z) {
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
    for (int l = 0; l < lanes; ++l) {
      t0 += red[l * Z + j]; t1 += red[n + l * Z + j]; t2 += red[2 * n + l * Z + j]; t3 += red[3 * n + l * Z + j];
    }
    if (t0 != 0.f) atomicAdd(db_enc + j, t0);
    if (t1 != 0.f) atomicAdd(db_enc + Z + j, t1);
    if (prior_mode == 2) {
      if (t2 != 0.f) atomicAdd(db_prior + j, t2);
      if (t3 != 0.f) atomicAdd(db_prior + Z + j, t3);
    }
  }
}

// ---- vectorised / row-per-thread variants of the heads (the bf16 training step at the reference's sizes) ----
// The kernels above keep one element (or one warp per row) per thread, which at a batch of 16 384 is bound by
// the latency of a handful of dependent 4-byte loads.  These variants move 16 bytes per load:
//   z heads: thread <-> 4 consecutive latent dimensions of one row (Z % 4 == 0, Z <= 256, 16-byte aligned rows);
//   y heads: thread <-> one row, the K <= 16 mixture components in registers (no warp shuffles).
__device__ __forceinline__ uint2 pack_bf16x4(float a, float b, float c, float d) { return make_uint2(pack_bf16x2(a, b), pack_bf16x2(c, d)); }
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__global__ void head_z_fwd_v4_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps,
                                     const float* __restrict__ prior_out, int prior_mode, int B, int Z, float c,
                                     float sigma_min, float inv_bg, bf16* __restrict__ z_act, int ld_z, float* __restrict__ z_f32,
                                     float* __restrict__ acc) {
  griddep_wait();
  griddep_launch();
  __shared__ float scratch[32];
  const int tpr = Z >> 2;                                  // threads per row
  const int64_t total = (int64_t)B * tpr;
  float kl = 0.f;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(t / tpr), j = (int)(t % tpr) * 4;
    const float4 mu = *reinterpret_cast<const float4*>(enc_out + (int64_t)b * 2 * Z + j);
    const float4 raw = *reinterpret_cast<const float4*>(enc_out + (int64_t)b * 2 * Z + Z + j);
    const float4 e4 = *reinterpret_cast<const float4*>(eps + (int64_t)b * Z + j);
    float4 mp = make_float4(0.f, 0.f, 0.f, 0.f), rp = mp;
    if (prior_mode == 2) {
      mp = *reinterpret_cast<const float4*>(prior_out + (int64_t)b * 2 * Z + j);
      rp = *reinterpret_cast<const float4*>(prior_out + (int64_t)b * 2 * Z + Z + j);
    }
    const float* MU = &mu.x; const float* RAW = &raw.x; const float* E = &e4.x; const float* MP = &mp.x; const float* RP = &rp.x;
    float z[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float sg = fmaxf(softplus_f(RAW[q] + c), sigma_min);
      z[q] = fmaf(sg, E[q], MU[q]);
      const float logq = -0.5f * E[q] * E[q] - logf(sg);
      float logp = 0.f;
      if (prior_mode == 0) {
        logp = -0.5f * z[q] * z[q];
      } else if (prior_mode == 2) {
        const float sp = fmaxf(softplus_f(RP[q] + c), sigma_min);
        const float tt = (z[q] - MP[q]) / sp;
        logp = -0.5f * tt * tt - logf(sp);
      }
      kl += logq - logp;
    }
    *reinterpret_cast<uint2*>(z_act + (int64_t)b * ld_z + j) = pack_bf16x4(z[0], z[1], z[2], z[3]);
    if (z_f32) *reinterpret_cast<float4*>(z_f32 + (int64_t)b * Z + j) = make_float4(z[0], z[1], z[2], z[3]);
  }
  float s = block_sum(kl, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_KL, s * inv_bg);
}

// backward of the z head + the bias gradients of the last encoder layer and of prior_gmm (column sums of
// the values as stored).  blockDim.x = 256; dynamic shared memory = 16 * 256 floats.
__global__ void head_z_bwd_v4_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps,
                                     const float* __restrict__ prior_out, const float* __restrict__ dz_dec,
                                     const float* __restrict__ dz_prior, int prior_mode, int B, int Z, float c, float sigma_min,
                                     float inv_bg, bf16* __restrict__ d_enc_out, bf16* __restrict__ d_prior_out, int ld_out,
                                     float* __restrict__ db_enc, float* __restrict__ db_prior) {
  griddep_wait();
  griddep_launch();
  extern __shared__ float red[];                        // [4 pieces][rows per iteration][Z]
  const int tpr = Z >> 2, rpi = blockDim.x / tpr;       // threads per row, rows per block iteration
  const int jt = threadIdx.x % tpr, rl = threadIdx.x / tpr;
  const int j = jt * 4;
  float s[4][4];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = 0; q < 4; ++q) s[p][q] = 0.f;
  if (rl < rpi) {
    for (int b = blockIdx.x * rpi + rl; b < B; b += gridDim.x * rpi) {
      const float4 mu = *reinterpret_cast<const float4*>(enc_out + (int64_t)b * 2 * Z + j);
      const float4 raw = *reinterpret_cast<const float4*>(enc_out + (int64_t)b * 2 * Z + Z + j);
      const float4 e4 = *reinterpret_cast<const float4*>(eps + (int64_t)b * Z + j);
      const float4 dzd = *reinterpret_cast<const float4*>(dz_dec + (int64_t)b * Z + j);
      float4 mp = make_float4(0.f, 0.f, 0.f, 0.f), rp = mp, dzp = mp;
      if (prior_mode == 2) {
        mp = *reinterpret_cast<const float4*>(prior_out + (int64_t)b * 2 * Z + j);
        rp = *reinterpret_cast<const float4*>(prior_out + (int64_t)b * 2 * Z + Z + j);
      } else if (prior_mode == 1) {
        dzp = *reinterpret_cast<const float4*>(dz_prior + (int64_t)b * Z + j);
      }
      const float* MU = &mu.x; const float* RAW = &raw.x; const float* E = &e4.x; const float* DZ = &dzd.x;
      const float* MP = &mp.x; const float* RP = &rp.x; const float* DZP = &dzp.x;
      float g0[4], g1[4], a0[4], a1[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float spq = softplus_f(RAW[q] + c);
        const float sg = fmaxf(spq, sigma_min);
        const float z = fmaf(sg, E[q], MU[q]);
        float dz = DZ[q];
        a0[q] = 0.f; a1[q] = 0.f;
        if (prior_mode == 0) {
          dz += z * inv_bg;
        } else if (prior_mode == 1) {
          dz += DZP[q];
        } else {
          const float spp = softplus_f(RP[q] + c);
          const float sp = fmaxf(spp, sigma_min);
          const float d = z - MP[q];
          const float isp2 = 1.f / (sp * sp);
          dz += d * isp2 * inv_bg;
          const float dsp = (1.f / sp - d * d * isp2 / sp) * inv_bg;
          a0[q] = bf16_round(-d * isp2 * inv_bg);
          a1[q] = bf16_round(spp >= sigma_min ? dsp * sigmoid_f(RP[q] + c) : 0.f);
        }
        const float dsg = dz * E[q] - inv_bg / sg;
        g0[q] = bf16_round(dz);
        g1[q] = bf16_round(spq >= sigma_min ? dsg * sigmoid_f(RAW[q] + c) : 0.f);
        s[0][q] += g0[q]; s[1][q] += g1[q]; s[2][q] += a0[q]; s[3][q] += a1[q];   // sums of the values as stored
      }
      *reinterpret_cast<uint2*>(d_enc_out + (int64_t)b * ld_out + j) = pack_bf16x4(g0[0], g0[1], g0[2], g0[3]);
      *reinterpret_cast<uint2*>(d_enc_out + (int64_t)b * ld_out + Z + j) = pack_bf16x4(g1[0], g1[1], g1[2], g1[3]);
      if (prior_mode == 2) {
        *reinterpret_cast<uint2*>(d_prior_out + (int64_t)b * ld_out + j) = pack_bf16x4(a0[0], a0[1], a0[2], a0[3]);
        *reinterpret_cast<uint2*>(d_prior_out + (int64_t)b * ld_out + Z + j) = pack_bf16x4(a1[0], a1[1], a1[2], a1[3]);
      }
    }
#pragma unroll
    for (int p = 0; p < 4; ++p)
      *reinterpret_cast<float4*>(red + ((size_t)p * rpi + rl) * Z + j) = make_float4(s[p][0], s[p][1], s[p][2], s[p][3]);
  }
  __syncthreads();
  for (int col = threadIdx.x; col < 4 * Z; col += blockDim.x) {
    const int p = col / Z, jj = col % Z;
    if (p >= 2 && prior_mode != 2) continue;
    float t = 0.f;
    for (int l = 0; l < rpi; ++l) t += red[((size_t)p * rpi + l) * Z + jj];
    if (t != 0.f) atomicAdd((p < 2 ? db_enc : db_prior) + (p & 1) * Z + jj, t);
  }
}

// q(y|x) head forward, one row per thread (K <= 16)
__global__ void head_y_fwd_row_kernel(const float* __restrict__ logits, const float* __restrict__ gum, int B, int K, float inv_T,
                                      float inv_bg, float* __restrict__ y_f32, bf16* __restrict__ y_act, int ld_yact,
                                      float* __restrict__ acc) {
  griddep_wait();
  griddep_launch();
  __shared__ float scratch[32];
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  float ent = 0.f;
  if (row < B) {
    float l[16], a[16];
    float ml = -INFINITY, ma = -INFINITY;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      l[k] = -INFINITY; a[k] = -INFINITY;
      if (k < K) {
        l[k] = logits[(int64_t)row * K + k];
        a[k] = gum ? (l[k] + gum[(int64_t)row * K + k]) * inv_T : l[k];
      }
      ml = fmaxf(ml, l[k]); ma = fmaxf(ma, a[k]);
    }
    float sl = 0.f, nm = 0.f, sa = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) { a[k] = expf(a[k] - ma); if (l[k] == ml) nm += 1.f; else sl += expf(l[k] - ml); sa += a[k]; }
    const float lo = lse_above_max(sl, nm), inv_sa = 1.f / sa;
    float y[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      y[k] = 0.f;
      if (k < K) {
        const float logp = (l[k] - ml) - lo;
        ent += expf(logp) * logp;
        y[k] = a[k] * inv_sa;
        y_f32[(int64_t)row * K + k] = y[k];
      }
    }
    // zero-padded bf16 operand row (ld_yact is a multiple of 8, at most 16)
    uint4* dst = reinterpret_cast<uint4*>(y_act + (int64_t)row * ld_yact);
    dst[0] = make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
    if (ld_yact > 8) dst[1] = make_uint4(pack_bf16x2(y[8], y[9]), pack_bf16x2(y[10], y[11]), pack_bf16x2(y[12], y[13]), pack_bf16x2(y[14], y[15]));
  }
  float s = block_sum(ent, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_NENT, s * inv_bg);
}

// q(y|x) head backward, one row per thread (K <= 16), fused bias gradient of encoder_y's last layer
__global__ void head_y_bwd_row_kernel(const float* __restrict__ logits, const float* __restrict__ y_f32,
                                      const float* __restrict__ dy, int B, int K, float inv_T, float inv_bg,
                                      bf16* __restrict__ dlogits, int ld_out, float* __restrict__ db) {
  griddep_wait();
  griddep_launch();
  __shared__ float cs_s[16];
  if (threadIdx.x < 16) cs_s[threadIdx.x] = 0.f;
  __syncthreads();
  float cs[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) cs[k] = 0.f;
  for (int row = blockIdx.x * blockDim.x + threadIdx.x; row < B; row += gridDim.x * blockDim.x) {
    float l[16], y[16], g[16];
    float ml = -INFINITY, ydy = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      l[k] = -INFINITY; y[k] = 0.f; g[k] = 0.f;
      if (k < K) {
        l[k] = logits[(int64_t)row * K + k];
        y[k] = y_f32[(int64_t)row * K + k];
        g[k] = dy ? dy[(int64_t)row * K + k] : 0.f;
      }
      ml = fmaxf(ml, l[k]);
      ydy += y[k] * g[k];
    }
    float sl = 0.f, nm = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) { if (l[k] == ml) nm += 1.f; else sl += expf(l[k] - ml); }
    const float lo = lse_above_max(sl, nm);
    float plogp = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k)
      if (k < K) { l[k] = (l[k] - ml) - lo; plogp += expf(l[k]) * l[k]; }
    float o[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      o[k] = 0.f;
      if (k < K) {
        o[k] = bf16_round(y[k] * (g[k] - ydy) * inv_T + expf(l[k]) * (l[k] - plogp) * inv_bg);
        cs[k] += o[k];
      }
    }
    uint4* dst = reinterpret_cast<uint4*>(dlogits + (int64_t)row * ld_out);
    dst[0] = make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
    if (ld_out > 8) dst[1] = make_uint4(pack_bf16x2(o[8], o[9]), pack_bf16x2(o[10], o[11]), pack_bf16x2(o[12], o[13]), pack_bf16x2(o[14], o[15]));
  }
  if (db) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float t = warp_sum(cs[k]);
      if ((threadIdx.x & 31) == 0 && k < K && t != 0.f) atomicAdd(cs_s + k, t);
    }
    __syncthreads();
    if (threadIdx.x < K && cs_s[threadIdx.x] != 0.f) atomicAdd(db + threadIdx.x, cs_s[threadIdx.x]);
  }
}

// ---- inference helpers (gmvae.py:109-188, vae.py:80-123) ------------------------------------------
// z_mean = mu, z_sample = mu + sigma eps from the encoder's [mu|raw] output
__global__ void encode_out_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps, int B, int Z, float c, float sigma_min,
                                  float* __restrict__ z_mean, float* __restrict__ z_sample) {
  griddep_wait();
  griddep_launch();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)B * Z) {
    int b = (int)(i / Z), j = (int)(i % Z);
    float mu = enc_out[(int64_t)b * 2 * Z + j];
    float sg = fmaxf(softplus_f(enc_out[(int64_t)b * 2 * Z + Z + j] + c), sigma_min);
    z_mean[i] = mu;
    z_sample[i] = fmaf(sg, eps[i], mu);
  }
}
template <typename T>
__global__ void to_act_kernel(const float* __restrict__ in, int rows, int cols, T* __restrict__ out, int ld) {
  griddep_wait();
  griddep_launch();
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)rows * cols) out[(i / cols) * ld + i % cols] = from_f32<T>(in[i]);
}
// mode 2: GMVAE prior_gmm(one_hot(k)) = (Wp[k,:Z] + bp[:Z], softplus(Wp[k,Z:] + bp[Z:] + c));
// mode 1: VAE_GMP components (loc, softplus(raw_scale_diag)); mode 0: standard normal.
__global__ void prior_params_kernel(const float* __restrict__ a, const float* __restrict__ b, int mode, int K, int Z, float c,
                                    float sigma_min, float* __restrict__ mu, float* __restrict__ sigma) {
  griddep_wait();
  griddep_launch();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K * Z) return;
  int k = i / Z, j = i % Z;
  if (mode == 2) {
    mu[i] = a[k * 2 * Z + j] + b[j];
    sigma[i] = fmaxf(softplus_f(a[k * 2 * Z + Z + j] + b[Z + j] + c), sigma_min);
  } else if (mode == 1) {
    mu[i] = a[i]; sigma[i] = softplus_f(b[i]);
  } else {
    mu[i] = 0.f; sigma[i] = 1.f;
  }
}

// ---- the callable distribution layer (base.py:63-83, 130-146, 193-209; gmvae_condition / gmvae_dist_*) -------------
// [mu | raw] rows of a ConditionalNormal's MLP -> mu, sigma = max(softplus(raw + c), sigma_min)   (base.py:69-70)
__global__ void normal_params_kernel(const float* __restrict__ outs, int n, int Z, float c, float sigma_min, float* __restrict__ mu,
                                     float* __restrict__ sigma) {
  griddep_wait();
  griddep_launch();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)n * Z) {
    const int64_t b = i / Z; const int j = (int)(i % Z);
    mu[i] = outs[b * 2 * Z + j];
    sigma[i] = fmaxf(softplus_f(outs[b * 2 * Z + Z + j] + c), sigma_min);
  }
}
__global__ void add_scalar_kernel(float* __restrict__ v, int64_t n, float s) {
  griddep_wait();
  griddep_launch();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] += s;
}
// op 0: MultivariateNormalDiag.sample      out[n,d] = a + b * c            (a = loc, b = scale_diag, c = eps)
// op 1: Bernoulli.mean                     out[n,d] = sigmoid(a)           (a = logits)
__global__ void dist_map_kernel(int op, const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c, int64_t n,
                                float* __restrict__ out) {
  griddep_wait();
  griddep_launch();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = op == 0 ? fmaf(b[i], c[i], a[i]) : sigmoid_f(a[i]);
}
// One warp per row.
// op 0: MultivariateNormalDiag.log_prob(z) = -1/2 sum ((z-mu)/sigma)^2 - sum log sigma - d/2 log 2 pi      (a = loc, b = scale_diag, c = z)
// op 1: Independent(Bernoulli(logits),1).log_prob(x) = sum x l - max(l,0) - log1p(exp(-|l|))              (a = logits, c = x as float)
// op 2: RelaxedOneHotCategorical.sample = softmax((logits + g)/T), g = -log(-log u)                       (a = logits, c = u, out [n,d])
__global__ void dist_row_kernel(int op, const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c, int n, int d,
                                float inv_T, float* __restrict__ out) {
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const int64_t base = (int64_t)row * d;
  if (op == 2) {
    float m = -INFINITY;
    for (int j = lane; j < d; j += 32) m = fmaxf(m, (a[base + j] + gumbel_of(c[base + j])) * inv_T);
    m = warp_max(m);
    float s = 0.f;
    for (int j = lane; j < d; j += 32) s += expf((a[base + j] + gumbel_of(c[base + j])) * inv_T - m);
    s = warp_sum(s);
    for (int j = lane; j < d; j += 32) out[base + j] = expf((a[base + j] + gumbel_of(c[base + j])) * inv_T - m) / s;
    return;
  }
  float acc = 0.f;
  for (int j = lane; j < d; j += 32) {
    if (op == 0) {
      const float t = (c[base + j] - a[base + j]) / b[base + j];
      acc += -0.5f * t * t - logf(b[base + j]) - 0.9189385332046727f;
    } else {
      // x l - max(l, 0) is exact for x in {0, 1}; subtracting softplus(l) whole would round a well-predicted pixel's
      // -log1p(exp(-|l|)) away against |l| (a logit of 14 gives 0 or -9.5e-7 instead of -8.3e-7)
      const float l = a[base + j];
      acc += (c[base + j] * l - fmaxf(l, 0.f)) - log1pf(expf(-fabsf(l)));
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

// ---- VAE_GMP mixture prior (vae.py:231-244, 181): forward value and every gradient -------------
// log p(z) = logsumexp_k [ log_softmax(m)_k + log N(z; loc_k, softplus(raw_scale_k)) ]
// One warp per row; lanes stride over Z.  Adds -log p / B to the KL accumulator, writes
// d kl/dz (prior part) to dz_prior, and accumulates d loc, d raw_scale_diag, d mixture_logits (deterministic mode: into the
// fixed-point sums fx = [K mixture logits | K*Z loc | K*Z raw_scale_diag] instead).
__global__ void gmp_prior_kernel(const float* __restrict__ z, const float* __restrict__ loc,
                                 const float* __restrict__ raw_scale, const float* __restrict__ mix_logits, int B, int K,
                                 int Z, float inv_bg, float* __restrict__ dz_prior, float* __restrict__ d_loc,
                                 float* __restrict__ d_raw_scale, float* __restrict__ d_mix, float* __restrict__ acc,
                                 unsigned long long* __restrict__ fx) {
  griddep_wait();
  griddep_launch();
  extern __shared__ float sm[];  // per warp: K log-weights
  __shared__ float scratch[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float* lw = sm + w * K;
  const int row = blockIdx.x * nw + w;
  float neg_logp = 0.f;
  if (row < B) {
    // log_softmax of the mixture logits
    float mm = -INFINITY;
    for (int k = lane; k < K; k += 32) mm = fmaxf(mm, mix_logits[k]);
    mm = warp_max(mm);
    float ms = 0.f;
    for (int k = lane; k < K; k += 32) ms += expf(mix_logits[k] - mm);
    ms = warp_sum(ms);
    const float mlse = mm + logf(ms);
    float best = -INFINITY;
    for (int k = 0; k < K; ++k) {
      float s = 0.f;
      for (int j = lane; j < Z; j += 32) {
        float sc = softplus_f(raw_scale[k * Z + j]);
        float t = (z[(int64_t)row * Z + j] - loc[k * Z + j]) / sc;
        s += -0.5f * t * t - logf(sc);
      }
      s = warp_sum(s) + (mix_logits[k] - mlse);
      if (lane == 0) lw[k] = s;
      best = fmaxf(best, s);
    }
    __syncwarp();
    float se = 0.f;
    for (int k = lane; k < K; k += 32) se += expf(lw[k] - best);
    se = warp_sum(se);
    const float logp = best + logf(se);
    neg_logp = lane == 0 ? -logp : 0.f;
    for (int j = lane; j < Z; j += 32) dz_prior[(int64_t)row * Z + j] = 0.f;
    for (int k = 0; k < K; ++k) {
      const float r = expf(lw[k] - logp);  // responsibility
      if (lane == 0) {
        const float g = -(r - expf(mix_logits[k] - mlse)) * inv_bg;
        if (fx) fx_add(fx, k, g); else atomicAdd(d_mix + k, g);
      }
      for (int j = lane; j < Z; j += 32) {
        float raw = raw_scale[k * Z + j];
        float sc = softplus_f(raw);
        float d = z[(int64_t)row * Z + j] - loc[k * Z + j];
        float is2 = 1.f / (sc * sc);
        dz_prior[(int64_t)row * Z + j] += r * d * is2 * inv_bg;
        float dsc = -r * (d * d * is2 / sc - 1.f / sc) * inv_bg;
        if (fx) {
          fx_add(fx, K + k * Z + j, -r * d * is2 * inv_bg);
          fx_add(fx, K + K * Z + k * Z + j, dsc * sigmoid_f(raw));
        } else {
          atomicAdd(d_loc + k * Z + j, -r * d * is2 * inv_bg);
          atomicAdd(d_raw_scale + k * Z + j, dsc * sigmoid_f(raw));
        }
      }
    }
  }
  float s = block_sum(neg_logp, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_KL, s * inv_bg);
}


// ======================================================================================
// Objective "marginal" (north_star; SURVEY.md Appendix A.3): the reference's own blocks evaluated
// at y = e_k for every component k, weighted by pi = q(y|x), analytic Gaussian KL.  Rows of the
// per-component tensors are r = b*K + k.
// ======================================================================================

// prior_gmm(e_k) = rows of Wp + bp (the reference evaluates prior_gmm at one-hot y, gmvae.py:170-173)
__global__ void prior_table_kernel(const float* __restrict__ Wp, const float* __restrict__ bp, int K, int Z2, float* __restrict__ tab) {
  griddep_wait();
  griddep_launch();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K * Z2) tab[i] = Wp[i] + bp[i % Z2];
}

// h1[b,k,:] = relu(xproj[b,:] + W1[D+k,:] + b1): the x-projection of encoder_gmm layer 0 is computed
// once per sample and broadcast over the K one-hot components.
template <typename ActT>
__global__ void expand_h1_kernel(const float* __restrict__ xproj, int64_t ldx, const float* __restrict__ Wy, const float* __restrict__ b1,
                                 int rows, int K, int H, ActT* __restrict__ out, int64_t ldo) {
  griddep_wait();
  griddep_launch();
  const int64_t total = (int64_t)rows * (H / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / (H / 4)), n = (int)(i % (H / 4)) * 4;
    const int b = r / K, k = r % K;
    const float4 xp = *reinterpret_cast<const float4*>(xproj + (int64_t)b * ldx + n);
    const float4 wy = *reinterpret_cast<const float4*>(Wy + (int64_t)k * H + n);
    const float4 bb = *reinterpret_cast<const float4*>(b1 + n);
    float v[4] = {fmaxf(xp.x + wy.x + bb.x, 0.f), fmaxf(xp.y + wy.y + bb.y, 0.f), fmaxf(xp.z + wy.z + bb.z, 0.f),
                  fmaxf(xp.w + wy.w + bb.w, 0.f)};
    store_frag<4>(out + (int64_t)r * ldo + n, v, 4);
  }
}

// One warp per row r = (b,k): z = mu_q + sigma_q eps;  KL_k = sum_j [log(s_p/s_q) + (s_q^2 + (mu_q-mu_p)^2)/(2 s_p^2) - 1/2];
// kl accumulator += pi[b,k] KL_k / B;  klrow[r] = KL_k (needed for d loss / d pi).
template <typename ActT>
__global__ void head_z_m_fwd_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps, const float* __restrict__ tab,
                                    const float* __restrict__ pi, int row0, int rows, int K, int Z, float c, float sigma_min,
                                    float inv_bg, ActT* __restrict__ z_act, int ld_z, float* __restrict__ klrow, float* __restrict__ acc) {
  griddep_wait();
  griddep_launch();
  __shared__ float scratch[32];
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float part = 0.f;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows; r += gridDim.x * wpb) {
    const int k = (row0 + r) % K;
    float kl = 0.f;
    for (int j = lane; j < Z; j += 32) {
      float mu = enc_out[(int64_t)r * 2 * Z + j], raw = enc_out[(int64_t)r * 2 * Z + Z + j];
      float sq = fmaxf(softplus_f(raw + c), sigma_min);
      float mp = tab[k * 2 * Z + j], sp = fmaxf(softplus_f(tab[k * 2 * Z + Z + j] + c), sigma_min);
      float e = eps[(int64_t)(row0 + r) * Z + j];
      z_act[(int64_t)r * ld_z + j] = from_f32<ActT>(fmaf(sq, e, mu));
      float d = mu - mp;
      kl += logf(sp / sq) + (sq * sq + d * d) / (2.f * sp * sp) - 0.5f;
    }
    kl = warp_sum(kl);
    if (lane == 0) { klrow[row0 + r] = kl; part += pi[row0 + r] * kl; }
  }
  float s = block_sum(part, scratch);
  if (threadIdx.x == 0 && s != 0.f) acc_add(acc, ACC_KL, s * inv_bg);
}

// Backward of the z head for objective M.  Thread <-> latent dimension j, row lanes stride over the
// chunk (same layout as head_z_bwd_cs_kernel): d_enc_out, the bias gradient of the last encoder_gmm
// layer, and the gradient w.r.t. the prior table (accumulated per component in shared memory).
template <typename ActT>
__global__ void head_z_m_bwd_kernel(const float* __restrict__ enc_out, const float* __restrict__ eps, const float* __restrict__ tab,
                                    const float* __restrict__ pi, const float* __restrict__ dz_dec, int row0, int rows, int K, int Z,
                                    float c, float sigma_min, float inv_bg, ActT* __restrict__ d_enc_out, int ld_out,
                                    float* __restrict__ db_enc, float* __restrict__ dtab) {
  griddep_wait();
  griddep_launch();
  extern __shared__ float sm[];                        // [2][blockDim.x] column sums, then [K][2Z] table gradient
  const int n = blockDim.x;
  float* dt = sm + 2 * n;
  for (int i = threadIdx.x; i < K * 2 * Z; i += n) dt[i] = 0.f;
  __syncthreads();
  const int lanes = n / Z;
  const int j = threadIdx.x % Z, rl = threadIdx.x / Z;
  float s_mu = 0.f, s_raw = 0.f;
  if (rl < lanes) {
    for (int r = blockIdx.x * lanes + rl; r < rows; r += gridDim.x * lanes) {
      const int k = (row0 + r) % K;
      float mu = enc_out[(int64_t)r * 2 * Z + j], raw = enc_out[(int64_t)r * 2 * Z + Z + j];
      float spq = softplus_f(raw + c), sq = fmaxf(spq, sigma_min);
      float mp = tab[k * 2 * Z + j], rp = tab[k * 2 * Z + Z + j];
      float spp = softplus_f(rp + c), sp = fmaxf(spp, sigma_min);
      float e = eps[(int64_t)(row0 + r) * Z + j];
      float w = pi[row0 + r] * inv_bg;
      float dz = dz_dec[(int64_t)r * Z + j];
      float d = mu - mp, isp2 = 1.f / (sp * sp);
      float dmu = dz + w * d * isp2;
      float dsq = dz * e + w * (sq * isp2 - 1.f / sq);
      ActT g0 = from_f32<ActT>(dmu), g1 = from_f32<ActT>(spq >= sigma_min ? dsq * sigmoid_f(raw + c) : 0.f);
      d_enc_out[(int64_t)r * ld_out + j] = g0; d_enc_out[(int64_t)r * ld_out + Z + j] = g1;
      s_mu += to_f32<ActT>(g0); s_raw += to_f32<ActT>(g1);
      float dsp = w * (1.f / sp - (sq * sq + d * d) * isp2 / sp);
      atomicAdd(dt + k * 2 * Z + j, -w * d * isp2);
      atomicAdd(dt + k * 2 * Z + Z + j, spp >= sigma_min ? dsp * sigmoid_f(rp + c) : 0.f);
    }
  }
  sm[threadIdx.x] = s_mu; sm[n + threadIdx.x] = s_raw;
  __syncthreads();
  if (threadIdx.x < Z) {
    float t0 = 0.f, t1 = 0.f;
    for (int l = 0; l < lanes; ++l) { t0 += sm[l * Z + j]; t1 += sm[n + l * Z + j]; }
    if (t0 != 0.f) atomicAdd(db_enc + j, t0);
    if (t1 != 0.f) atomicAdd(db_enc + Z + j, t1);
  }
  for (int i = threadIdx.x; i < K * 2 * Z; i += n)
    if (dt[i] != 0.f) atomicAdd(dtab + i, dt[i]);
}

// tab[k,:] = Wp[k,:] + bp  =>  dWp[k,:] += dtab[k,:],  dbp += sum_k dtab[k,:]
__global__ void prior_table_bwd_kernel(const float* __restrict__ dtab, int K, int Z2, float* __restrict__ dWp, float* __restrict__ dbp) {
  griddep_wait();
  griddep_launch();
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < Z2) {
    float s = 0.f;
    for (int k = 0; k < K; ++k) { float v = dtab[k * Z2 + j]; dWp[k * Z2 + j] += v; s += v; }
    dbp[j] += s;
  }
}

// dxproj[b,:] = sum_k dh1[b,k,:]  (ActT, the dY of the x-part weight gradient); dWy[k,:] += sum_b dh1[b,k,:];
// db1 += sum_{b,k} dh1.  A block owns 64 columns and a range of samples; each of its 4 row lanes
// accumulates the per-component sums in a private shared-memory slice (no atomics in the loop).
template <typename ActT>
__global__ void reduce_k_kernel(const ActT* __restrict__ dh1, int64_t ldh, int b0, int nb, int K, int H, ActT* __restrict__ dxproj,
                                int64_t ldx, float* __restrict__ dWy, float* __restrict__ db1, int samples_per_block) {
  griddep_wait();
  griddep_launch();
  extern __shared__ float sm[];                        // [nty][K][64]
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6, nty = blockDim.x >> 6;
  const int n = blockIdx.x * 64 + tx;
  float* mine = sm + (size_t)ty * K * 64 + tx;
  for (int k = 0; k < K; ++k) mine[k * 64] = 0.f;
  const int s0 = blockIdx.y * samples_per_block, s1 = min(nb, s0 + samples_per_block);
  if (n < H) {
    for (int s = s0 + ty; s < s1; s += nty) {
      const ActT* src = dh1 + (int64_t)s * K * ldh + n;
      float tot = 0.f;
#pragma unroll 4
      for (int k = 0; k < K; ++k) {
        float v = to_f32<ActT>(src[(int64_t)k * ldh]);
        tot += v;
        mine[k * 64] += v;
      }
      dxproj[(int64_t)(b0 + s) * ldx + n] = from_f32<ActT>(tot);
    }
  }
  __syncthreads();
  if (n < H) {
    float t = 0.f;
    for (int k = ty; k < K; k += nty) {
      float v = 0.f;
      for (int l = 0; l < nty; ++l) v += sm[((size_t)l * K + k) * 64 + tx];
      if (v != 0.f) atomicAdd(dWy + (int64_t)k * H + n, v);
      t += v;
    }
    if (t != 0.f) atomicAdd(db1 + n, t);
  }
}

// d loss / d logits_y for objective M: loss_y = sum_k pi_k c_k + sum_k pi_k log pi_k with
// c_k = KL_k - rec_k;  dl_j = pi_j (c_j - sum_k pi_k c_k)/B + pi_j (log pi_j - sum pi log pi)/B.
template <typename ActT>
__global__ void head_y_m_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ pi, const double* __restrict__ rec,
                                    const float* __restrict__ klrow, int B, int K, float inv_bg, ActT* __restrict__ dlogits, int ld_out,
                                    float* __restrict__ db) {
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  float cs[HEAD_MAXK / 32];
#pragma unroll
  for (int i = 0; i < HEAD_MAXK / 32; ++i) cs[i] = 0.f;
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < B; row += gridDim.x * wpb) {
    float p[HEAD_MAXK / 32], cc[HEAD_MAXK / 32], l[HEAD_MAXK / 32];
    double cd[HEAD_MAXK / 32];
    float ml = -INFINITY;
    double pcd = 0.0;
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      p[i] = 0.f; cd[i] = 0.0; l[i] = -INFINITY;
      if (k < K) {
        l[i] = logits[(int64_t)row * K + k];
        p[i] = pi[(int64_t)row * K + k];
        cd[i] = (double)klrow[(int64_t)row * K + k] - rec[(int64_t)row * K + k];
      }
      ml = fmaxf(ml, l[i]);
      pcd += (double)p[i] * cd[i];
    }
    // c_j - sum_k pi_k c_k cancels the common ~ -rec magnitude: done in double
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) pcd += __shfl_xor_sync(0xffffffffu, pcd, o);
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) cc[i] = (float)(cd[i] - pcd);
    const float pc = 0.f;
    ml = warp_max(ml);
    float sl = 0.f, nm = 0.f;
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i)
      if (lane + 32 * i < K) { if (l[i] == ml) nm += 1.f; else sl += expf(l[i] - ml); }
    sl = warp_sum(sl); nm = warp_sum(nm);
    const float lo = lse_above_max(sl, nm);
    float plogp = 0.f;
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i)
      if (lane + 32 * i < K) { float lp = (l[i] - ml) - lo; plogp += expf(lp) * lp; }
    plogp = warp_sum(plogp);
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      if (k < K) {
        float lp = (l[i] - ml) - lo;
        ActT o = from_f32<ActT>((p[i] * (cc[i] - pc) + expf(lp) * (lp - plogp)) * inv_bg);
        dlogits[(int64_t)row * ld_out + k] = o;
        cs[i] += to_f32<ActT>(o);
      } else if (k < ld_out) {
        dlogits[(int64_t)row * ld_out + k] = from_f32<ActT>(0.f);
      }
    }
  }
  if (db) {
#pragma unroll
    for (int i = 0; i < HEAD_MAXK / 32; ++i) {
      int k = lane + 32 * i;
      if (k < K && cs[i] != 0.f) atomicAdd(db + k, cs[i]);
    }
  }
}

// ---- bias gradients: db[n] += sum_m dY[m,n] -----------------------------------------------------
// Each thread owns 8 consecutive columns (one 16-byte load per row for bf16); a block covers
// 256 columns x `rows_per_block` rows with 8 row-lanes, reduced through shared memory.
// part != null (deterministic mode): row block y stores its sums to part[y * N + n] (every column, zeros too) instead of adding
// them to db; det_reduce_kernel adds the row blocks in order.
template <typename T>
__global__ void colsum_kernel(const T* __restrict__ dY, int64_t ld, int M, int N, int rows_per_block, float* __restrict__ db,
                              float* __restrict__ part) {
  griddep_wait();
  griddep_launch();
  __shared__ float sm[8][32][9];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n0 = blockIdx.x * 256 + tx * 8;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  if (n0 < N) {
    const int nv = min(8, N - n0);
    for (int r = r0 + ty; r < r1; r += 8) {
      float v[8];
      load_frag<8>(dY + (int64_t)r * ld + n0, v, nv);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += v[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sm[ty][tx][j] = s[j];
  __syncthreads();
  // 256 threads: thread t sums column t of the block over the 8 row-lanes
  const int c = threadIdx.x, cx = c >> 3, cj = c & 7;
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) t += sm[i][cx][cj];
  const int n = blockIdx.x * 256 + c;
  if (part) { if (n < N) part[(int64_t)blockIdx.y * N + n] = t; return; }
  if (n < N && t != 0.f) atomicAdd(db + n, t);
}

// ---- deterministic mode: the reduction step ------------------------------------------------------
// One launch after the step's last GEMM, before the gradient exchange.  Segment blockIdx.y is a rows x cols block of the gradient
// buffer, element (r, c) at dst[r * ld_dst + c]:
//   part != null: part[0 * part_stride + r * ld_part + c] + part[1 * part_stride + ...] + ...  (nparts partials: the k-splits of a
//                 weight gradient, chain_sched.cuh det_slice_index, or the row blocks of a column sum -- added in index order)
//   fx != null:   the fixed-point sum r * cols + c (common.cuh fx_add), NaN if it was flagged
constexpr int DET_MAX_SEGS = 64;
struct DetSeg { float* dst; const float* part; const unsigned long long* fx; long long part_stride; int rows, cols, nparts, ld_dst, ld_part, pad; };
struct DetSegs { int nseg; DetSeg s[DET_MAX_SEGS]; };
__global__ void det_reduce_kernel(const __grid_constant__ DetSegs segs) {
  griddep_wait();
  griddep_launch();
  const DetSeg& g = segs.s[blockIdx.y];
  const long long n = (long long)g.rows * g.cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / g.cols), c = (int)(i % g.cols);
    float v = 0.f;
    if (g.fx) {
      const unsigned long long* f = g.fx + FX_WORDS * i;
      const long long coarse = (long long)f[2];
      v = (f[1] & 1ull) ? __int_as_float(0x7fffffff)
        : ((f[1] & 2ull) || coarse >= (1ll << 26) || coarse <= -(1ll << 26)) ? (float)coarse
        : (float)((double)(long long)f[0] * (1.0 / (double)(1ull << FX_SHIFT)));
    } else {
      const float* p = g.part + (long long)r * g.ld_part + c;
      for (int s = 0; s < g.nparts; ++s) v += p[(long long)s * g.part_stride];
    }
    g.dst[(long long)r * g.ld_dst + c] = v;
  }
}

// ---- loss terms ---------------------------------------------------------------------------------
__global__ void finalize_loss_kernel(const float* __restrict__ acc, float* __restrict__ out) {
  griddep_wait();
  griddep_launch();
  if (threadIdx.x == 0) {
    float nll = acc_total(acc, ACC_NLL), kl = acc_total(acc, ACC_KL), ne = acc_total(acc, ACC_NENT);
    out[0] = nll + kl + ne;  // gmvae.py:267 / vae.py:185
    out[1] = nll; out[2] = kl; out[3] = ne;
  }
}

// ---- tf.train.AdamOptimizer (runners.py:181-183; SURVEY.md Appendix B.6) ------------------------
// lr_t = lr sqrt(1-b2^t)/(1-b1^t); m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2;
// theta -= lr_t m / (sqrt(v) + eps).   t = step+1 read from the device; one flat pass.
// Also (training step only, `zero_grads`): the gradient buffer and the loss accumulators are cleared once read, so the next step
// starts from zeros without a separate memset node.  8 elements per thread, every load issued before the block waits for lr_t.
constexpr int ADAM_THREADS = 256, ADAM_VEC = 2;              // float4 groups per thread
struct AdamPeer {                                            // all null / 0 outside the peer-memory data-parallel path
  const unsigned long long* flags;                           // [world] "shard r of the reduced gradients has landed" epochs (my memory)
  unsigned long long* epoch;                                 // the exchange epoch counter of this rank
  float* own_grads;                                          // this rank's gradient buffer (cleared here)
  int world; long long timeout_cycles;
};
__global__ void __launch_bounds__(ADAM_THREADS) adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            int64_t n, float lr, float b1, float b2, float eps, DeviceState* st,
                            float* __restrict__ acc, float* __restrict__ loss_out,
                            const ShadowEntry* __restrict__ shadows, int n_shadows, int zero_grads, AdamPeer peer) {
  griddep_wait();
  griddep_launch();
  __shared__ float lr_t_s;
  __shared__ int e0_s;
  // Data parallel over peer memory (peer.cuh): this launch is the last phase of the all-reduce.  `g` is the reduced-gradient
  // buffer the shard owners push into; wait until all `world` shards of this epoch have landed (one polling thread per block).
  // `gz` is what gets cleared: this rank's own gradient buffer (every owner has pulled from it before publishing its shard).
  float* gz = g;
  float* accz = acc;
  if (peer.flags) {
    if (threadIdx.x == 0) {
      const unsigned long long epoch = *peer.epoch + 1;
      const long long t0 = clock64();
      for (int r = 0; r < peer.world; ++r) {
        unsigned long long v;
        do {
          asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(peer.flags + r) : "memory");
          if (v < epoch) { __nanosleep(64); if (clock64() - t0 > peer.timeout_cycles) __trap(); }
        } while (v < epoch);
      }
    }
    __syncthreads();
    gz = peer.own_grads; accz = peer.own_grads + n;
  }
  if (blockIdx.x == 0 && threadIdx.x == 32) {
    if (loss_out) {                                          // loss terms (gmvae.py:267 / vae.py:185), same as finalize_loss_kernel
      float nll = acc_total(acc, ACC_NLL), kl = acc_total(acc, ACC_KL), ne = acc_total(acc, ACC_NENT);
      loss_out[0] = nll + kl + ne; loss_out[1] = nll; loss_out[2] = kl; loss_out[3] = ne;
    }
    if (zero_grads)
      for (int i = 0; i < ACC_SLOTS; ++i) accz[i] = 0.f;
  }
  const int64_t i0 = (int64_t)blockIdx.x * ADAM_THREADS * 4 * ADAM_VEC;
  // operands first: the loads are in flight while thread 0 works out the step size
  float4 pp[ADAM_VEC], gg[ADAM_VEC], mm[ADAM_VEC], vv[ADAM_VEC];
  int64_t idx[ADAM_VEC];
#pragma unroll
  for (int u = 0; u < ADAM_VEC; ++u) {
    idx[u] = i0 + ((int64_t)u * ADAM_THREADS + threadIdx.x) * 4;
    if (idx[u] + 4 <= n) {
      pp[u] = *reinterpret_cast<float4*>(p + idx[u]); gg[u] = __ldcg(reinterpret_cast<const float4*>(g + idx[u]));
      mm[u] = *reinterpret_cast<float4*>(m + idx[u]); vv[u] = *reinterpret_cast<float4*>(v + idx[u]);
    }
  }
  if (threadIdx.x == 0) {
    // lr_t = lr sqrt(1 - beta2^t) / (1 - beta1^t), t = step + 1, from the running powers (as TF keeps them)
    const double b1t = st->beta1_power * (double)b1, b2t = st->beta2_power * (double)b2;
    lr_t_s = (float)((double)lr * sqrt(1.0 - b2t) / (1.0 - b1t));
    // global_step += 1 and the powers advance once every block of this launch has read them: the last block to get here does it
    __threadfence();
    if (atomicAdd(&st->adam_blocks, 1u) == gridDim.x - 1) {
      st->adam_blocks = 0; st->step += 1; st->beta1_power = b1t; st->beta2_power = b2t;
      if (peer.flags) *peer.epoch += 1;                      // every block of this launch has passed its wait: the exchange epoch is over
    }
  } else if (threadIdx.x == 64) {
    // the weight matrix the block's first element belongs to (entries are sorted by flat offset); the block's
    // elements almost always lie in the same matrix, so the threads only step forward from here
    int lo = 0, hi = n_shadows;                             // first entry with off > i0
    while (lo < hi) { int mid = (lo + hi) >> 1; if (shadows[mid].off <= i0) lo = mid + 1; else hi = mid; }
    e0_s = lo - 1;
  }
  __syncthreads();
  const float lr_t = lr_t_s;
  int e = e0_s;
#pragma unroll
  for (int u = 0; u < ADAM_VEC; ++u) {
    const int64_t i = idx[u];
    if (i >= n) continue;
    // tensors start on 16-byte boundaries, so a group of 4 never straddles two
    while (e + 1 < n_shadows && shadows[e + 1].off <= i) ++e;
    bf16* wb = nullptr; int cols = 0, ld_w = 0; int64_t rel = 0, lim = 0;
    if (e >= 0) {
      const ShadowEntry& E = shadows[e];
      rel = i - E.off; lim = (int64_t)E.rows * E.cols;
      if (rel < lim) { wb = E.w_bf16; cols = E.cols; ld_w = E.ld_w; }
    }
    if (i + 4 <= n) {
      float* P = &pp[u].x; const float* G = &gg[u].x; float* Mm = &mm[u].x; float* V = &vv[u].x;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        Mm[j] = b1 * Mm[j] + (1.f - b1) * G[j];
        V[j] = b2 * V[j] + (1.f - b2) * G[j] * G[j];
        P[j] -= lr_t * Mm[j] / (sqrtf(V[j]) + eps);
      }
      *reinterpret_cast<float4*>(p + i) = pp[u]; *reinterpret_cast<float4*>(m + i) = mm[u]; *reinterpret_cast<float4*>(v + i) = vv[u];
      if (zero_grads) *reinterpret_cast<float4*>(gz + i) = make_float4(0.f, 0.f, 0.f, 0.f);
      if (wb) {                                               // bf16 GEMM operand copy [rows, ld_w] of the updated weights
        if (cols == ld_w && rel + 4 <= lim) {
          *reinterpret_cast<uint2*>(wb + rel) = make_uint2(pack_bf16x2(P[0], P[1]), pack_bf16x2(P[2], P[3]));
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int64_t el = rel + j;
            if (el < lim) wb[(el / cols) * ld_w + (el % cols)] = __float2bfloat16_rn(P[j]);
          }
        }
      }
    } else {
      for (int64_t k = i; k < n; ++k) {
        const float gk = __ldcg(g + k);
        float mk = b1 * m[k] + (1.f - b1) * gk;
        float vk = b2 * v[k] + (1.f - b2) * gk * gk;
        m[k] = mk; v[k] = vk;
        p[k] -= lr_t * mk / (sqrtf(vk) + eps);
        if (zero_grads) gz[k] = 0.f;
        if (wb) { const int64_t el = rel + (k - i); if (el < lim) wb[(el / cols) * ld_w + (el % cols)] = __float2bfloat16_rn(p[k]); }
      }
    }
  }
}

// ---- bf16 operand copies of the weight matrices --------------------------------------------------
// For W [rows=in, cols=out] fp32: w_bf16 [in, ld_w] (dgrad B operand, K-major over `out`) and
// wt_bf16 [out, ld_wt] (forward B operand, K-major over `in`).  One entry per matrix; a 32x32
// tile per block, transposed through shared memory.  Block (0,0,0) also advances global_step.
__global__ void refresh_shadows_kernel(const ShadowEntry* __restrict__ entries, int n_entries) {
  griddep_wait();
  griddep_launch();
  int e = 0;
  while (e + 1 < n_entries && (int)blockIdx.x >= entries[e + 1].tile_begin) ++e;
  const ShadowEntry E = entries[e];
  const int t = blockIdx.x - E.tile_begin;
  const int c0 = (t % E.tiles_x) * 32, r0 = (t / E.tiles_x) * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int r = r0 + i, c = c0 + threadIdx.x;
    float v = (r < E.rows && c < E.cols) ? E.w[(int64_t)r * E.cols + c] : 0.f;
    if (r < E.rows && c < E.ld_w) E.w_bf16[(int64_t)r * E.ld_w + c] = __float2bfloat16_rn(v);
  }
}
__global__ void bump_step_kernel(DeviceState* st) {
  griddep_wait();
  griddep_launch(); st->step += 1; }

}  // namespace gmvae

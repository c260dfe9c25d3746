/*
 * gmvae_abi.h -- C ABI of libgmvae_b200.so, the B200-native (sm_100a) training step of
 * mazrk7/gmvae (VAE / VAE_GMP / GMVAE on flattened binarised images).
 *
 * The reference has no FFI of its own: its hot path sits behind a Python object API
 * (scripts/{base,vae,gmvae}.py) that builds a TF-1.13 graph, and behind
 * `sess.run([train_op, global_step])` (scripts/runners.py:231-232).  This header is the
 * boundary a maintainer binds instead of that graph; each entry point names the reference
 * lines it replaces.  The Python host in gmvae_b200/ binds it with ctypes; INTEGRATION.md
 * shows the stub.
 *
 * Conventions
 *   - plain C: pointers and sizes only, no C++ / torch types.
 *   - every buffer is a DEVICE pointer owned by the caller (PyTorch tensors in our host);
 *     the library owns only the handle, its TMA descriptors, CUDA graph and NCCL communicator.
 *   - all work is enqueued on the caller's stream (`stream` is a cudaStream_t passed as
 *     void*); no hidden synchronisation, no allocation after gmvae_bind().
 *   - int return: 0 = OK, negative = error; message via gmvae_last_error() (thread-local).
 *   - a handle is bound to one device and is not thread-safe; one process per GPU.
 *   - there is NO CPU fallback: every entry point that computes requires an sm_100 device.
 */
#ifndef GMVAE_ABI_H_
#define GMVAE_ABI_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define GMVAE_API __attribute__((visibility("default")))
#else
#define GMVAE_API
#endif

#define GMVAE_ABI_VERSION 1
#define GMVAE_MAX_HIDDEN_LAYERS 8
#define GMVAE_NAME_LEN 64

/* run_gmvae.py:14-16 `--model` */
enum { GMVAE_MODEL_VAE = 0, GMVAE_MODEL_VAE_GMP = 1, GMVAE_MODEL_GMVAE = 2 };
/* objective: REFERENCE = what gmvae.py:238-267 computes (one relaxed y, one z, MC KL);
 *            MARGINAL  = q(y|x)-weighted per-component ELBO with analytic KL (north_star). */
enum { GMVAE_OBJECTIVE_REFERENCE = 0, GMVAE_OBJECTIVE_MARGINAL = 1 };
/* precision of the GEMM path: FP32 = SIMT validation mode (rel 1e-5), BF16 = tcgen05 tiles */
enum { GMVAE_PRECISION_FP32 = 0, GMVAE_PRECISION_BF16 = 1 };

typedef struct gmvae_handle gmvae_handle;

/* What runners.create_model (runners.py:65-103) passes to create_gmvae / create_vae
 * (gmvae.py:277-287, vae.py:191-200) plus the optimiser of runners.py:181. */
typedef struct gmvae_config {
  int32_t abi_version;        /* GMVAE_ABI_VERSION */
  int32_t model;              /* GMVAE_MODEL_* */
  int32_t objective;          /* GMVAE_OBJECTIVE_* (GMVAE only) */
  int32_t precision;          /* GMVAE_PRECISION_* */
  int32_t data_size;          /* 784 */
  int32_t latent_size;        /* --latent_size */
  int32_t mixture_components; /* --mixture_components */
  int32_t num_hidden;         /* len(fcnet_hidden_sizes) */
  int32_t hidden_sizes[GMVAE_MAX_HIDDEN_LAYERS];
  int32_t max_batch;          /* largest per-device batch this handle will see */
  float sigma_min;            /* runners.py:84 (0.0) */
  float raw_sigma_bias;       /* runners.py:85 (0.5) */
  float gen_bias_init;        /* gmvae.py:284 */
  float temperature;          /* runners.py:86 (1.0) */
  float learning_rate;        /* --learning_rate; tf.train.AdamOptimizer defaults below */
  float beta1, beta2, epsilon;
  int32_t device;             /* CUDA ordinal */
  /* 1: bitwise-reproducible training steps.  Two steps with the same build, device type, configuration, parameters, Adam state,
   * global step, seed and inputs give identical gradients, loss terms, parameters and Adam moments (eager or graph, one GPU or
   * the peer-memory exchange; not the NCCL all-reduce).  Sums whose addends arrive in no fixed order are taken in a fixed order
   * or in integer fixed point; costs step time (DESIGN.md section 9).  objective=reference only; 0 (default): the fastest plan. */
  int32_t deterministic;
  int32_t reserved[6];
} gmvae_config;

/* One trainable variable of the flat parameter buffer.  Names are the reference's TF
 * variable names (`{module}_fcnet/linear_{i}/{w,b}`, `loc`, `raw_scale_diag`,
 * `mixture_logits`; base.py:53,60 / vae.py:233-238) so a TF checkpoint maps 1:1. */
typedef struct gmvae_param_desc {
  char name[GMVAE_NAME_LEN];
  int64_t offset;             /* in floats, into params / grads / adam_m / adam_v */
  int32_t rows, cols;         /* weights [rows=in, cols=out] row-major; vectors rows=1 */
} gmvae_param_desc;

/* Construction = create_gmvae / create_vae (gmvae.py:277-355, vae.py:191-271). */
GMVAE_API int gmvae_create(const gmvae_config* cfg, gmvae_handle** out);
GMVAE_API void gmvae_destroy(gmvae_handle* h);

/* Flat layout of tf.trainable_variables() (runners.py:182). param_count includes the
 * 16-byte alignment padding between tensors; grad_count = param_count + 96 (the tail holds
 * the loss accumulators, 32 fp32 slots per term, so that one all-reduce covers both). */
GMVAE_API int64_t gmvae_param_count(const gmvae_handle* h);
GMVAE_API int64_t gmvae_grad_count(const gmvae_handle* h);
GMVAE_API int gmvae_num_params(const gmvae_handle* h);
GMVAE_API int gmvae_param_table(const gmvae_handle* h, gmvae_param_desc* out, int cap);

GMVAE_API size_t gmvae_workspace_bytes(const gmvae_handle* h);
/* params/adam_m/adam_v: float[param_count]; grads: float[grad_count]; workspace: bytes above. */
GMVAE_API int gmvae_bind(gmvae_handle* h, float* params, float* grads, float* adam_m, float* adam_v,
               void* workspace, size_t workspace_bytes);
/* Call after writing `params` from outside (initialisation, checkpoint restore): refreshes
 * the bf16 operand copies the tensor-core path reads. */
GMVAE_API int gmvae_params_updated(gmvae_handle* h, void* stream);

/* loss = model.run_model(images, targets[, labels]) (gmvae.py:223-274, vae.py:153-188)
 * followed by opt.compute_gradients (runners.py:182).
 *   x_u8        [batch, data_size] bytes in {0,1} (the reference feeds bool; targets == images)
 *   global_batch divisor of the batch means (== batch on one GPU; sum over ranks under DP)
 *   eps         [batch, Z] (REFERENCE / VAE) or [batch, K, Z] (MARGINAL) N(0,1) noise, or NULL
 *               to draw it on the device (Philox, keyed by seed and the device step counter)
 *   gumbel_u    [batch, K] uniforms in [tiny,1) for the relaxed one-hot sample, or NULL
 *   loss_terms  device float[4] = {loss, nll, kl_div_z, nent}; written by
 *               gmvae_finalize_loss (after the all-reduce under DP)
 * Gradients land in `grads` (overwritten). */
GMVAE_API int gmvae_forward_backward(gmvae_handle* h, const uint8_t* x_u8, int batch, int global_batch,
                           const float* eps, const float* gumbel_u, void* stream);
GMVAE_API int gmvae_finalize_loss(gmvae_handle* h, float* loss_terms, void* stream);

/* opt.apply_gradients (runners.py:183): TF-form Adam on the flat buffer, then
 * global_step += 1 and the beta-power accumulators advance (all on the device). */
GMVAE_API int gmvae_adam_step(gmvae_handle* h, void* stream);
GMVAE_API int gmvae_get_step(gmvae_handle* h, int64_t* step, void* stream);   /* synchronises */
GMVAE_API int gmvae_set_step(gmvae_handle* h, int64_t step, void* stream);    /* checkpoint restore */
GMVAE_API int gmvae_set_seed(gmvae_handle* h, uint64_t seed);

/* Data parallelism (new; the reference is single-device, runners.py:193): one NCCL
 * all-reduce(sum) over grads[0:grad_count].  No-op when no communicator is attached. */
GMVAE_API int gmvae_nccl_unique_id(char out[128]);
GMVAE_API int gmvae_nccl_init(gmvae_handle* h, const char id[128], int world_size, int rank);
GMVAE_API int gmvae_allreduce_grads(gmvae_handle* h, void* stream);

/* The exchange step as the library's own kernels over NVLink peer memory, fused with the optimiser (csrc/peer.cuh), in place of
 * ncclAllReduce: every rank's gradient buffer lives in a symmetric region all ranks map (cudaIpc); one `exchange` kernel per step
 * pulls this rank's shard of every rank's gradients, adds them in rank order and pushes the sums to every rank, and the Adam kernel
 * is the all-reduce's last phase (it waits for the shards, reads the reduced gradients, clears this rank's buffer).
 * export() allocates this rank's region and returns its cudaIpcMemHandle_t (64 bytes); the caller gathers the handles of all ranks
 * (rank order, own included), passes them to attach() and puts a barrier before the first step.  attach() MOVES the gradient buffer
 * into the region: gmvae_peer_grads() is where the gradients are from then on (float[grad_count]); steps captured before are
 * dropped.  One node, P2P-capable GPUs, world_size <= 16.  Flag waits are bounded by GMVAE_PEER_TIMEOUT_S (default 120 s). */
GMVAE_API int gmvae_peer_export(gmvae_handle* h, int world_size, int rank, char out[64]);
GMVAE_API int gmvae_peer_attach(gmvae_handle* h, const char* handles);
GMVAE_API float* gmvae_peer_grads(gmvae_handle* h);

/* One whole iteration of the hot loop `sess.run([train_op, global_step])`
 * (runners.py:231-232): forward_backward -> allreduce -> finalize_loss -> adam_step.
 * capture() records it once into a CUDA graph for fixed pointers; launch() replays it. */
GMVAE_API int gmvae_train_step(gmvae_handle* h, const uint8_t* x_u8, int batch, int global_batch,
                     const float* eps, const float* gumbel_u, float* loss_terms, void* stream);
GMVAE_API int gmvae_step_graph_capture(gmvae_handle* h, const uint8_t* x_u8, int batch, int global_batch,
                             const float* eps, const float* gumbel_u, float* loss_terms,
                             void* stream);
GMVAE_API int gmvae_step_graph_launch(gmvae_handle* h, void* stream);

/* Forward-only helpers behind the model classes' inference methods
 * (gmvae.py:109-188, vae.py:80-123).  out buffers are device float arrays.
 *   encode : x -> (optional) logits_y [batch,K], z_mean [batch,Z], z_sample [batch,Z]
 *   decode : z [n,Z] -> Bernoulli mean sigmoid(logits) [n, data_size]
 *   prior  : GMVAE prior_gmm(one_hot(k)) table -> mu [K,Z], sigma [K,Z] */
GMVAE_API int gmvae_encode(gmvae_handle* h, const uint8_t* x_u8, int batch, const float* eps,
                 const float* gumbel_u, float* logits_y, float* z_mean, float* z_sample,
                 void* stream);
GMVAE_API int gmvae_decode(gmvae_handle* h, const float* z, int n, float* x_mean, void* stream);
GMVAE_API int gmvae_prior_table(gmvae_handle* h, float* mu, float* sigma, void* stream);

/* The callable distribution layer: Conditional{Normal,Bernoulli,Categorical}.condition(tensor_list) (base.py:63-72, 130-135,
 * 193-198) = concat(inputs) -> MLP -> distribution parameters, on caller tensors (device float arrays, row-major):
 *   GMVAE_COND_DECODER   in1 = z [n,Z]                    -> out_a = Bernoulli logits [n, data_size] (MLP(z) + bias_init)
 *   GMVAE_COND_ENCODER   in1 = x [n,D] (in2 = y [n,K] for the GMVAE's encoder_gmm) -> out_a = mu, out_b = sigma [n,Z]
 *   GMVAE_COND_ENCODER_Y in1 = x [n,D]                    -> out_a = logits of q(y|x) [n,K]
 *   GMVAE_COND_PRIOR_GMM in1 = y [n,K]                    -> out_a = mu, out_b = sigma [n,Z]
 * with sigma = max(softplus(raw + raw_sigma_bias), sigma_min) (base.py:69-70).  The model accessors decoder(z), encoder(x),
 * encoder_y(x), encoder_gmm(x,y), prior_gmm(y) (gmvae.py:49-107, vae.py:41-78) are these.
 * gmvae_dist_*: sample / log_prob / mean of the distributions those classes return (base.py:75-83, 138-146, 201-209):
 * MultivariateNormalDiag(loc, scale_diag), Independent(Bernoulli(logits), 1), RelaxedOneHotCategorical(T, logits).  Noise is
 * passed in (eps ~ N(0,1), u ~ U(0,1)); log_prob outputs are float[n]. */
enum { GMVAE_COND_DECODER = 0, GMVAE_COND_ENCODER = 1, GMVAE_COND_ENCODER_Y = 2, GMVAE_COND_PRIOR_GMM = 3 };
GMVAE_API int gmvae_condition(gmvae_handle* h, int which, const float* in1, const float* in2, int n, float* out_a, float* out_b,
                    void* stream);
GMVAE_API int gmvae_dist_normal_sample(const float* mu, const float* sigma, const float* eps, int64_t n, float* out, void* stream);
GMVAE_API int gmvae_dist_normal_log_prob(const float* mu, const float* sigma, const float* z, int n, int d, float* out, void* stream);
GMVAE_API int gmvae_dist_bernoulli_log_prob(const float* logits, const float* x, int n, int d, float* out, void* stream);
GMVAE_API int gmvae_dist_bernoulli_mean(const float* logits, int64_t n, float* out, void* stream);
GMVAE_API int gmvae_dist_relaxed_sample(const float* logits, const float* u, int n, int k, float temperature, float* out, void* stream);

/* Input pipeline on the device = runners.create_dataset._preprocess (runners.py:44-47):
 *     image = cast(image, float32) / 255. ;  image = image < random.uniform(shape(image))
 * (dynamic, inverted binarisation: a pixel is 1 with probability 1 - intensity).
 *   intensities [n_rows, data_size] bytes 0..255, device-resident (MNIST train = 47 MB)
 *   row_index   device int64[batch], each in [0, n_rows): source row of every output row, or NULL
 *               = rows 0..batch-1 of `intensities` (pass `intensities + first_row * data_size` for a
 *               contiguous batch: the reference batches first and shuffles batches, runners.py:50-57)
 *   draw        counter of this draw (e.g. the global step); uniforms are Philox4x32-10 keyed by
 *               (seed, draw, rank, element), 24-bit, open interval (0,1), never stored
 *   x_u8        [batch, data_size] bytes in {0,1}: what gmvae_forward_backward / gmvae_train_step take */
GMVAE_API int gmvae_binarize(gmvae_handle* h, const uint8_t* intensities, int64_t n_rows, const int64_t* row_index,
                   int batch, uint64_t draw, uint8_t* x_u8, void* stream);

/* Bit-packed binary images: packed [batch, ceil(data_size/8)] bytes, pixel 8j+k of a row in bit (7-k) of byte j
 * (numpy.packbits order) -> x_u8 [batch, data_size] bytes in {0,1}.  The inputs of this path are binary (runners.py:44-47), so a
 * host batch crosses PCIe as 98 bytes per image instead of 784. */
GMVAE_API int gmvae_unpack_bits(gmvae_handle* h, const uint8_t* packed, int batch, uint8_t* x_u8, void* stream);

/* Kernel-level test hook: C[M,N] = A[M,K] * B[K,N] through the same GEMM kernels the step
 * uses (impl 0 = fp32 SIMT, 1 = tcgen05 bf16).  A, B, C are device float arrays, row-major;
 * transA/transB say the stored matrix is the transpose ([K,M] / [N,K]).  Used by tests/. */
GMVAE_API int gmvae_debug_gemm(gmvae_handle* h, int impl, int transA, int transB, int M, int N, int K,
                     const float* A, const float* B, float* C, int split_k, void* stream);

/* Test hook: the step's own noise generator (Philox4x32-10) writing n_eps N(0,1) draws and n_u
 * uniforms in the OPEN interval (0,1) into caller buffers (either may be NULL / 0). */
GMVAE_API int gmvae_debug_noise(gmvae_handle* h, float* eps, int64_t n_eps, float* u, int64_t n_u, void* stream);
/* Test hook: per-tile clock64 stamps of CTA `cta` of each chained-GEMM launch (8 launches x 64 tiles x 16 int64,
 * device memory) for the following steps; null switches it off. */
GMVAE_API int gmvae_debug_chain_trace(gmvae_handle* h, long long* trace, int cta);

/* Test hooks: per-job counters of the first chained launch of a step, summed over all CTAs (8 uint64 per job, globaltimer ns:
 * first start, last end, dependency wait, MMA issue time, epilogue time, accumulator wait, tiles, accumulator-free wait; the
 * caller presets [0] of every job to ~0 and the rest to 0; 40 jobs), and the descriptions of those jobs (8 ints per job:
 * epilogue kind, M, N, k-blocks, tiles, splits, tile width, dependencies; returns the number of jobs). */
GMVAE_API int gmvae_debug_chain_jobstat(gmvae_handle* h, unsigned long long* stat);
GMVAE_API int gmvae_debug_chain_jobs(gmvae_handle* h, int* out, int cap_jobs);

/* Per-launch profile: with profiling on, a CUDA event is recorded after every launch of the
 * (eager) step; read() returns the summed device time and launch count per kernel class:
 * 0 tcgen05 GEMM fwd/dgrad, 1 tcgen05 GEMM wgrad, 2 SIMT GEMM, 3 distribution heads,
 * 4 bias gradients, 5 Adam + bf16 operand refresh, 6 misc (convert, noise, finalize), 7 the gradient exchange
 * (all-reduce; in-stream, so its interval is the exposed communication time).  n_classes >= 8. */
GMVAE_API int gmvae_profile_enable(gmvae_handle* h, int on);
GMVAE_API int gmvae_profile_read(gmvae_handle* h, double* ms_by_class, int64_t* launches_by_class, int n_classes);

/* Number of kernels this library has launched on behalf of the handle (bench "gpu_launches"). */
GMVAE_API int64_t gmvae_launch_count(const gmvae_handle* h);

GMVAE_API const char* gmvae_last_error(void);
GMVAE_API const char* gmvae_build_info(void);

#ifdef __cplusplus
}
#endif
#endif /* GMVAE_ABI_H_ */

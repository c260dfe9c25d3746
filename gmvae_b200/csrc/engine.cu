// engine.cu -- the GMVAE / VAE / VAE_GMP training step on B200 and its C ABI (include/gmvae_abi.h).
//
// One iteration of the reference's hot loop `sess.run([train_op, global_step])`
// (/root/reference/scripts/runners.py:231-232) = forward (gmvae.py:238-267 / vae.py:167-185)
// + reverse-mode gradients of every trainable variable (runners.py:182) + TF-form Adam
// (runners.py:183), expressed as a fixed sequence of kernels on the caller's stream.
#include <nccl.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include "../../include/gmvae_abi.h"
#include "common.cuh"
#include "epilogue.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "gemm_chain.cuh"
#include "kernels.cuh"
#include "input.cuh"
#include "peer.cuh"

namespace gmvae {

bool g_use_pdl = true;
static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }

// ============================================================================ TMA descriptors
namespace tc {
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

long long* g_trace = nullptr;

int g_reserved_sms = 0;   // SMs left to the NCCL kernels while a data-parallel step is running

int current_device() { int dev = 0; cudaGetDevice(&dev); return dev < 0 ? 0 : dev % 64; }
int num_sms() {
  static int n_by_dev[64] = {};
  int& n = n_by_dev[current_device()];
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return std::max(8, n - g_reserved_sms);
}

// 2-D tensor of `elem_bytes`-wide elements (2: bf16, 4: fp32, 1: bytes), row-major [outer, inner] with `outer_stride`
// elements between rows; box = {box_inner, box_outer}; swizzle span in bytes (128 / 64 / 0); out-of-bounds
// elements read as zero and are not written.
int make_tmap(CUtensorMap* out, const void* ptr, int elem_bytes, uint64_t inner, uint64_t outer, uint64_t outer_stride,
              uint32_t box_inner, uint32_t box_outer, int swizzle) {
  typedef std::tuple<const void*, int, uint64_t, uint64_t, uint64_t, uint32_t, uint32_t, int> Key;
  static thread_local std::map<Key, CUtensorMap> cache;
  Key key(ptr, elem_bytes, inner, outer, outer_stride, box_inner, box_outer, swizzle);
  auto it = cache.find(key);
  if (it != cache.end()) { *out = it->second; return 0; }
  EncodeTiledFn fn = get_encode_fn();
  GM_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  GM_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA operand base must be 16-byte aligned");
  GM_REQUIRE((outer_stride * (uint64_t)elem_bytes) % 16 == 0, "TMA operand row stride must be a multiple of 16 bytes");
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstride[1] = {outer_stride * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                                                                                      : CU_TENSOR_MAP_DATA_TYPE_UINT8;
  const CUtensorMapSwizzle sw = swizzle == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                                             : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(out, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return -3;
  }
  if (cache.size() > 4096) cache.clear();
  cache[key] = *out;
  return 0;
}
int make_tmap_bf16(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t outer, uint64_t outer_stride,
                   uint32_t box_inner, uint32_t box_outer) {
  return make_tmap(out, ptr, 2, inner, outer, outer_stride, box_inner, box_outer, 128);
}
// fp32 [slices][outer][inner] with `ld` floats between rows and outer * ld between slices (deterministic mode's weight-gradient
// partials, chain_sched.cuh det_slice_index); box = {box_inner, box_outer, 1}: a box never crosses into the next slice
int make_tmap_slices_f32(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t outer, uint64_t slices, uint64_t ld,
                         uint32_t box_inner, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  GM_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  GM_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && ld % 4 == 0, "TMA slices need 16-byte aligned rows");
  cuuint64_t gdim[3] = {inner, outer, slices};
  cuuint64_t gstride[2] = {ld * 4, outer * ld * 4};
  cuuint32_t box[3] = {box_inner, box_outer, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (slices) failed with CUresult " + std::to_string((int)r));
    return -3;
  }
  return 0;
}
}  // namespace tc

// ============================================================================ model description
static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct Linear {
  int in = 0, out = 0;
  int64_t w_off = 0, b_off = 0;
  bf16* w_bf16 = nullptr;  int ld_w = 0;    // [in, ld_w]: K-major B of the data-gradient GEMM, MN-major B of the forward GEMM
};
struct Mlp {
  std::string name;
  std::vector<Linear> layers;
};

// A (sub-)matrix of a Linear: rows [row0, row0+in) of W.
struct LinView {
  const float* w; float* dw; const float* b; float* db;
  int in, out, ldw32;               // fp32 row stride (= full `out`)
  const bf16* w_bf16; int ld_w;     // [in, ld_w], already offset to row row0
};

enum { DBG_NO_TC = 1, DBG_NO_TC_WGRAD = 2, DBG_NO_TWO_SEG = 4, DBG_SYNC_EACH = 8, DBG_BN128 = 16, DBG_NO_FUSED_COLSUM = 32,
       DBG_NO_PDL = 128, DBG_NO_CHAIN = 512, DBG_NO_ROW_JOBS = 1024, DBG_NO_SPREAD = 4096, DBG_NO_FUSE_HEADS = 16384,
       DBG_COMM_OVERLAP = 32768 /* data parallel: all-reduce the gradient buffer in three buckets on a side stream while the backward
                                   pass is still running (the chained kernel is cut at the bucket boundaries, GMVAE_COMM_SMS SMs are left
                                   to NCCL).  Measured SLOWER than one in-stream all-reduce after a single chained launch (cfg4 per GPU, N=2: 0.536 vs
                                   0.467 ms, N=8: 0.591 vs 0.497 ms): the cuts cost more than the overlap hides.  Off by default. */,
       DBG_ROW_JOBS = 8192 /* force the distribution heads to run as row jobs of the chained kernel (the whole forward + backward
                              pass is ONE launch).  Default: on for batches of >= 32 row blocks.  Measured: cfg4 (128 blocks) 0.415 ms
                              vs 0.423 ms with the heads as 4 kernels between 5 chained launches; batch 100: 0.240 vs 0.199 ms. */,
       DBG_NO_PAIR = 65536 /* run the one-launch plan on single CTAs (tcgen05 cta_group::1, 128 x 256 tiles) instead of CTA pairs */,
       DBG_NO_QUAD = 131072 /* CTA pairs without the 4-CTA clusters that share the A rows of a row block's two n-tiles by TMA multicast */,
       DBG_WG_LATE = 262144 /* one-launch plan: every weight-gradient job after the data-gradient chain instead of interleaved with it
                                (measured: 0.378 vs 0.350 ms at cfg4 -- the chain alone leaves the SMs 80 % idle) */,
       DBG_NO_PARTITION = 524288 /* backward pass: chain and weight-gradient jobs on the same CTA pairs (no walker partition) */,
       DBG_NO_RELU_BITS = 2048 /* one-launch plan: read the ReLU mask of the backward pass from the bf16 activation (TMA load in the epilogue)
                                  instead of the 1-bit masks the forward epilogues write */ };
// kernel classes of the per-launch profile (gmvae_profile_read)
enum { PC_START = -1, PC_TC_GEMM = 0, PC_TC_WGRAD = 1, PC_SIMT_GEMM = 2, PC_HEADS = 3, PC_BIAS_GRAD = 4, PC_ADAM = 5, PC_MISC = 6,
       PC_COMM = 7, PC_COUNT = 8 };

}  // namespace gmvae

using namespace gmvae;

struct gmvae_handle {
  gmvae_config cfg;
  int D, Z, K, L;                      // L = layers per MLP = num_hidden + 1
  std::vector<int> hidden;
  std::vector<gmvae_param_desc> table;
  int64_t n_params = 0;                // padded flat count
  Mlp prior_gmm, decoder, encoder_y, encoder;   // `encoder` = encoder (VAE) / encoder_gmm (GMVAE)
  int64_t loc_off = -1, raw_scale_off = -1, mix_off = -1;
  // bound buffers
  float *params = nullptr, *grads = nullptr, *adam_m = nullptr, *adam_v = nullptr;
  uint8_t* ws = nullptr; size_t ws_bytes = 0;
  // workspace carve-outs (bytes offsets resolved at bind)
  struct Buf { size_t off = 0, bytes = 0; };
  std::map<std::string, Buf> bufs;
  size_t ws_needed = 0;
  std::vector<ShadowEntry> shadow_host;
  ShadowEntry* shadow_dev = nullptr; int shadow_tiles = 0;
  DeviceState* state = nullptr;
  uint64_t seed_host = 0;                // host copy of state->seed (it changes only through gmvae_set_seed)
  bool grads_clean = false;              // the gradient buffer and the loss accumulators are all zero (the training step's Adam clears them)
  bool graph_has_memset = true;          // the captured step starts with its own clearing memset
  uint64_t draws = 0;                    // noise draws made outside training steps (mixed into the Philox key, kernels.cuh fill_noise_body)
  bool in_train_step = false;
  int64_t launches = 0;
  int debug_flags = 0;
  // per-launch CUDA-event profile (off by default; bench.py turns it on for a few eager steps)
  bool profiling = false;
  std::vector<std::pair<cudaEvent_t, int>> marks;
  // NCCL: gradients are all-reduced in buckets ordered by backward readiness, on a side stream
  ncclComm_t comm = nullptr; int world = 1, rank = 0;
  cudaStream_t comm_stream = nullptr;
  cudaEvent_t comm_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int comm_ev_next = 0;
  bool overlap_comm = false;             // set by gmvae_train_step
  // experimental: the exchange step as our own kernels over NVLink peer memory (peer.cuh); off unless gmvae_peer_attach was called
  bool peer_ready = false;
  void* peer_region = nullptr;           // this rank's symmetric region (cudaMalloc, exported through cudaIpc)
  void* peer_mapped[peer::MAX_WORLD] = {};   // other ranks' regions as mapped into this process
  long long peer_timeout_cycles = 0;         // bound of the flag waits (GMVAE_PEER_TIMEOUT_S, default 120 s)
  float* grads_bound = nullptr;              // the caller's gradient buffer (gmvae_bind); `grads` moves into the symmetric region on attach
  peer::Layout peer_layout;
  peer::Peers peer_ptrs;
  int64_t reduced_upto = 0;              // floats of `grads` already handed to NCCL this step
  int64_t bucket_end[2] = {0, 0};        // flat offsets where bucket 0 (decoder) / 1 (encoder, prior) end
  int chunk_samples = 0;                 // objective M: samples per chunk of per-component rows
  // GEMM chains (gemm_chain.cuh): while chain_on, tensor-core GEMMs are recorded as jobs of one launch
  bool chain_on = false;
  tc::ChainParams chain;
  struct ChainWriter { const char* lo; const char* hi; int job; };
  std::vector<ChainWriter> chain_writers;
  int chain_tiles = 0;
  int max_quads = 0;
  int* chain_counters = nullptr; int chain_counter_cap = 0, chain_counter_next = 0;
  long long* chain_trace = nullptr; int chain_trace_cta = 0, chain_launch_idx = 0;   // test hook (gmvae_debug_chain_trace)
  unsigned long long* chain_jobstat = nullptr;     // test hook (gmvae_debug_chain_jobstat): 8 counters per job of the step's first chained launch
  std::vector<int> chain_jobdesc;                  // 8 ints per job of that launch: kind, M, N, k-blocks, tiles, splits, block_n, ndeps
  bool chain_flush_after = false;
  bool row_jobs = false;                          // this step: distribution heads run as row jobs of the chained kernel
  bool quad_opt_in = false;                       // GMVAE_CHAIN_QUAD=1 (read at gmvae_create)
  int chain_split_opt = 0;                        // GMVAE_CHAIN_SPLIT=<pairs on the dependent chain> (0: no walker partition)
  int wide_bn = 0;                                // tile width of jobs with more than 128 output columns (0: 256); GMVAE_CHAIN_BN
  std::vector<std::function<int()>>* wg_late = nullptr;   // one-launch plan: every weight-gradient GEMM is recorded after the data-gradient chain
  // walker partition of the backward pass (ChainJob::wfirst / wcount): 0 = every walker, 1 = the dependent chain (data gradients, heads),
  // 2 = weight gradients.  part_tiles: tiles recorded per class (the round-robin phase of the next job of that class).
  int cur_part = 0, part_chain_walkers = 0, part_walkers = 0, part_tiles[3] = {0, 0, 0};
  bool part_on = false, part_last_mlp = false, part_tail = false;
  bool chain_quad = false;                        // ... in clusters of two pairs sharing A rows by multicast (gemm_chain.cuh, CL = 4)
  bool chain_pair = false;                        // this step: the chained kernel runs on CTA pairs (cta_group::2, 256-row tiles)
  // a y head to be fused into the epilogue of the next thin fp32 GEMM job (set by the step driver, consumed by chain_add)
  struct FuseReq { int kind = 0; unsigned char prm[tc::CHAIN_EPI2_BYTES]; std::vector<std::pair<const void*, size_t>> writes; bool consumed = false; };
  FuseReq fuse_next;
  bool last_gemm_chained = false;                 // set by the GEMM dispatch: the last GEMM became a job of the chain
  std::map<const void*, bool> relu_bits_valid;    // hidden activation -> its 1-bit ReLU mask was written this step
  // deterministic mode (gmvae_config::deterministic): the segments the reduction step of this step sums (det_reduce_kernel) and the
  // partial rows of the column sums handed out so far (floats of the "det.part" buffer)
  bool det = false;
  std::vector<DetSeg> det_segs;
  std::vector<std::function<int()>> det_colsums;  // column sums of this step, launched after its last chained launch
  int64_t det_part_next = 0, det_part_cap = 0;    // floats of "det.part" (column-sum partial rows)
  int64_t det_wg_next = 0, det_wg_cap = 0;        // floats of "det.wg" (weight-gradient k-split slices)
  // graph
  cudaGraphExec_t graph_exec = nullptr;

  bool bf16_mode() const { return cfg.precision == GMVAE_PRECISION_BF16; }
  size_t act_size() const { return bf16_mode() ? 2 : 4; }
  template <typename T> T* buf(const std::string& name) const {
    auto it = bufs.find(name);
    return it == bufs.end() ? nullptr : reinterpret_cast<T*>(ws + it->second.off);
  }
};

namespace gmvae {

static void add_param(gmvae_handle* h, const std::string& name, int rows, int cols, int64_t* off_out) {
  gmvae_param_desc d;
  memset(&d, 0, sizeof(d));
  snprintf(d.name, GMVAE_NAME_LEN, "%s", name.c_str());
  d.offset = h->n_params; d.rows = rows; d.cols = cols;
  h->table.push_back(d);
  if (off_out) *off_out = h->n_params;
  h->n_params += round_up(rows * cols, 4);   // keep every tensor 16-byte aligned
}

static void build_mlp(gmvae_handle* h, Mlp& m, const std::string& name, int in, const std::vector<int>& sizes) {
  m.name = name;
  int prev = in;
  for (size_t i = 0; i < sizes.size(); ++i) {
    Linear l; l.in = prev; l.out = sizes[i];
    add_param(h, name + "_fcnet/linear_" + std::to_string(i) + "/w", l.in, l.out, &l.w_off);
    add_param(h, name + "_fcnet/linear_" + std::to_string(i) + "/b", 1, l.out, &l.b_off);
    m.layers.push_back(l);
    prev = sizes[i];
  }
}

static void plan_buf(gmvae_handle* h, const std::string& name, size_t bytes) {
  gmvae_handle::Buf b; b.off = h->ws_needed; b.bytes = bytes;
  h->bufs[name] = b;
  h->ws_needed += (bytes + 255) / 256 * 256;
}

static void plan_mlp_bufs(gmvae_handle* h, const Mlp& m, size_t B, size_t asz) {
  for (size_t i = 0; i + 1 < m.layers.size(); ++i) {
    plan_buf(h, m.name + ".h" + std::to_string(i), B * round_up(m.layers[i].out, 8) * asz);
    plan_buf(h, m.name + ".dh" + std::to_string(i), B * round_up(m.layers[i].out, 8) * asz);
    plan_buf(h, m.name + ".bits" + std::to_string(i), (size_t)round_up((int)B, 32) * (size_t)((m.layers[i].out + 31) / 32) * 4);   // 1-bit ReLU masks (chained kernel)
  }
}

static void plan_shadows(gmvae_handle* h, Mlp& m) {
  for (auto& l : m.layers) {
    l.ld_w = round_up(l.out, 8);
    plan_buf(h, "shadow.w." + std::to_string(l.w_off), (size_t)l.in * l.ld_w * 2);
  }
}

// deterministic mode: row blocks of a bias-gradient column sum (a function of nothing but the shapes)
constexpr int DET_ROW_BLOCKS = 64;
static int wgrad_split(const gmvae_handle* h, int in, int out, int M, bool pair, bool quad);

static int plan(gmvae_handle* h) {
  const gmvae_config& c = h->cfg;
  h->D = c.data_size; h->Z = c.latent_size; h->K = c.model == GMVAE_MODEL_VAE ? 1 : c.mixture_components;
  h->hidden.assign(c.hidden_sizes, c.hidden_sizes + c.num_hidden);
  h->L = c.num_hidden + 1;
  const int D = h->D, Z = h->Z, K = h->K;
  auto with = [&](int last) { std::vector<int> v = h->hidden; v.push_back(last); return v; };
  // The variables are the reference's (gmvae.py:321-353, vae.py:231-268), laid out in the flat
  // buffer in the order their gradients become final during the backward pass, so that the
  // data-parallel all-reduce can start on the decoder's range while the encoders are still running.
  if (c.model == GMVAE_MODEL_GMVAE) {
    build_mlp(h, h->decoder, "decoder", Z, with(D));
    h->bucket_end[0] = h->n_params;
    build_mlp(h, h->encoder, "encoder_gmm", D + K, with(2 * Z));
    build_mlp(h, h->prior_gmm, "prior_gmm", K, std::vector<int>{2 * Z});
    h->bucket_end[1] = h->n_params;
    build_mlp(h, h->encoder_y, "encoder_y", D, with(K));
  } else {
    build_mlp(h, h->decoder, "decoder", Z, with(D));
    h->bucket_end[0] = h->n_params;
    if (c.model == GMVAE_MODEL_VAE_GMP) {
      add_param(h, "loc", K, Z, &h->loc_off);
      add_param(h, "raw_scale_diag", K, Z, &h->raw_scale_off);
      add_param(h, "mixture_logits", 1, K, &h->mix_off);
    }
    h->bucket_end[1] = h->n_params;                         // nothing else is final before the end
    build_mlp(h, h->encoder, "encoder", D, with(2 * Z));
  }
  // ---- workspace ----
  const size_t Bfull = (size_t)c.max_batch, asz = h->act_size();
  const int Kp = round_up(K, 8);
  // Objective M evaluates K components per sample: rows r = b*K + k, processed in chunks of whole
  // samples so that the per-component activations never exceed `rows_cap` rows (SURVEY.md H6).
  h->chunk_samples = (int)Bfull;
  if (c.objective == GMVAE_OBJECTIVE_MARGINAL) {
    const char* env = getenv("GMVAE_M_CHUNK_ROWS");
    long max_rows = env ? atol(env) : 131072;
    long bc = std::max(1L, max_rows / K);
    if (bc > 64) bc = bc / 64 * 64;
    h->chunk_samples = (int)std::min<long>((long)Bfull, bc);
  }
  const size_t B = c.objective == GMVAE_OBJECTIVE_MARGINAL ? (size_t)h->chunk_samples * K : Bfull;   // row capacity
  plan_buf(h, "x_act", Bfull * round_up(D, 8) * asz);
  plan_buf(h, "eps", Bfull * (c.objective == GMVAE_OBJECTIVE_MARGINAL ? K : 1) * Z * 4);
  plan_buf(h, "dec.dlogits", B * round_up(D, 8) * asz);
  plan_buf(h, "dz", B * Z * 4);
  plan_buf(h, "enc_out", B * 2 * Z * 4);
  plan_buf(h, "d_enc_out", B * round_up(2 * Z, 8) * asz);
  plan_buf(h, "z_act", B * round_up(Z, 8) * asz);
  plan_mlp_bufs(h, h->decoder, B, asz);
  plan_mlp_bufs(h, h->encoder, B, asz);
  if (c.model == GMVAE_MODEL_GMVAE) {
    plan_mlp_bufs(h, h->encoder_y, Bfull, asz);
    plan_buf(h, "u", Bfull * K * 4);
    plan_buf(h, "logits_y", Bfull * K * 4);
    plan_buf(h, "y_f32", Bfull * K * 4);
    plan_buf(h, "y_act", Bfull * Kp * asz);
    plan_buf(h, "dlogits_y", Bfull * Kp * asz);
    const size_t H0 = (size_t)(h->hidden.empty() ? 2 * Z : h->hidden[0]);
    if (c.objective == GMVAE_OBJECTIVE_MARGINAL) {
      plan_buf(h, "tab", (size_t)K * 2 * Z * 4);
      plan_buf(h, "dtab", (size_t)K * 2 * Z * 4);
      plan_buf(h, "xproj", Bfull * H0 * 4);
      plan_buf(h, "dxproj", Bfull * round_up((int)H0, 8) * asz);
      plan_buf(h, "rec", Bfull * K * 8);
      plan_buf(h, "klrow", Bfull * K * 4);
    } else {
      plan_buf(h, "prior_out", Bfull * 2 * Z * 4);
      plan_buf(h, "d_prior_out", Bfull * round_up(2 * Z, 8) * asz);
      plan_buf(h, "dy", Bfull * K * 4);
      plan_buf(h, "pre_y", Bfull * H0 * 4);
    }
  }
  if (c.model == GMVAE_MODEL_VAE_GMP) {
    plan_buf(h, "z_f32", B * Z * 4);
    plan_buf(h, "dz_prior", B * Z * 4);
  }
  if (h->bf16_mode()) {
    plan_shadows(h, h->decoder); plan_shadows(h, h->encoder);
    if (c.model == GMVAE_MODEL_GMVAE) { plan_shadows(h, h->encoder_y); plan_shadows(h, h->prior_gmm); }
  }
  plan_buf(h, "infer.acc", ACC_SLOTS * 4);
  if (c.deterministic) {
    // one column sum per bias per step, DET_ROW_BLOCKS partial rows each; fixed-point sums of the three loss terms and of the
    // VAE_GMP prior's gradients
    int64_t cols = 0;
    for (const Mlp* m : {&h->decoder, &h->encoder, &h->encoder_y, &h->prior_gmm})
      for (const Linear& l : m->layers) cols += l.out;
    h->det_part_cap = cols * DET_ROW_BLOCKS;
    plan_buf(h, "det.part", (size_t)h->det_part_cap * 4);
    plan_buf(h, "det.fx", (size_t)(3 + (c.model == GMVAE_MODEL_VAE_GMP ? K + 2 * K * Z : 0)) * 16);
    // k-split slices of every weight gradient, for max_batch (the split count grows with the batch) in either plan
    h->det_wg_cap = 0;
    for (const Mlp* m : {&h->decoder, &h->encoder, &h->encoder_y, &h->prior_gmm})
      for (size_t i = 0; i < m->layers.size(); ++i) {
        const Linear& l = m->layers[i];
        std::vector<int> views{l.in};
        if (m == &h->encoder && i == 0 && c.model == GMVAE_MODEL_GMVAE) views = {D, K};    // [x, y] W: two weight-gradient jobs
        for (int in : views) {
          const int kb = (int)((Bfull + tc::BLOCK_K - 1) / tc::BLOCK_K);
          int S = 1;
          for (bool pair : {false, true}) S = std::max(S, wgrad_split(h, in, l.out, (int)Bfull, pair, false));
          S = std::min(S, kb);
          h->det_wg_cap += round_up((int)std::min<int64_t>((int64_t)S * in * tc::det_slice_ld(l.out), 1LL << 30), 64);
        }
      }
    plan_buf(h, "det.wg", (size_t)h->det_wg_cap * 4);
  }
  h->chain_counter_cap = 64 * (int)((Bfull + 127) / 128 + 2);
  plan_buf(h, "chain.counters", (size_t)h->chain_counter_cap * 4);
  return 0;
}

static LinView view(const gmvae_handle* h, const Linear& l, int row0 = 0, int rows = -1) {
  if (rows < 0) rows = l.in - row0;
  LinView v;
  v.w = h->params + l.w_off + (int64_t)row0 * l.out;
  v.dw = h->grads + l.w_off + (int64_t)row0 * l.out;
  v.b = h->params + l.b_off; v.db = h->grads + l.b_off;
  v.in = rows; v.out = l.out; v.ldw32 = l.out;
  v.w_bf16 = l.w_bf16 ? l.w_bf16 + (int64_t)row0 * l.ld_w : nullptr; v.ld_w = l.ld_w;
  return v;
}

// An event after every launch; the time between consecutive events on the in-order stream is
// that launch's duration (plus the launch gap).  PC_START marks carry no duration.
static int profile_mark(gmvae_handle* h, cudaStream_t st, int cls) {
  cudaEvent_t e;
  GM_CHECK_CUDA(cudaEventCreate(&e));
  GM_CHECK_CUDA(cudaEventRecord(e, st));
  h->marks.emplace_back(e, cls);
  return 0;
}

// Hands grads[reduced_upto, upto) to NCCL on the side stream once everything enqueued on `st` so
// far (which produced that range) has finished.  No-op outside gmvae_train_step / without a
// communicator.  All ranks issue the same sequence of collectives.
static int chain_flush(gmvae_handle* h, cudaStream_t st);
static int comm_bucket(gmvae_handle* h, cudaStream_t st, int64_t upto) {
  if (!h->comm || h->world == 1 || !h->overlap_comm || upto <= h->reduced_upto) return 0;
  GM_TRY(chain_flush(h, st));
  cudaEvent_t ev = h->comm_ev[h->comm_ev_next++ % 8];
  GM_CHECK_CUDA(cudaEventRecord(ev, st));
  GM_CHECK_CUDA(cudaStreamWaitEvent(h->comm_stream, ev, 0));
  ncclResult_t r = ncclAllReduce(h->grads + h->reduced_upto, h->grads + h->reduced_upto, (size_t)(upto - h->reduced_upto), ncclFloat,
                                 ncclSum, h->comm, h->comm_stream);
  if (r != ncclSuccess) { set_error(std::string("ncclAllReduce: ") + ncclGetErrorString(r)); return -5; }
  h->reduced_upto = upto;
  h->launches++;
  return 0;
}

// ============================================================================ GEMM dispatch
#define GM_LAUNCHED(h, st, cls)                                              \
  do {                                                                       \
    (h)->launches++;                                                         \
    if ((h)->profiling) GM_TRY(profile_mark(h, st, cls));                    \
    if ((h)->debug_flags & DBG_SYNC_EACH) GM_CHECK_CUDA(cudaStreamSynchronize(st)); \
  } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
// extent of a dimension whose buffer is zero-padded to a multiple of 8 elements (16 bytes)
static inline int kpad(int k, int64_t ld) { return (int)std::min<int64_t>(ld, round_up(k, 8)); }

template <typename TA>
static bool tc_ok_fwd(const gmvae_handle* h, const TA* A, int64_t lda, const LinView& L) {
  return std::is_same<TA, bf16>::value && h->bf16_mode() && !(h->debug_flags & DBG_NO_TC) && L.w_bf16 && lda % 8 == 0 &&
         aligned16(A) && aligned16(L.w_bf16);
}
template <typename TD>
static bool tc_ok_dgrad(const gmvae_handle* h, const TD* dY, int64_t ldy, const LinView& L) {
  return std::is_same<TD, bf16>::value && h->bf16_mode() && !(h->debug_flags & DBG_NO_TC) && L.w_bf16 && ldy % 8 == 0 &&
         aligned16(dY) && aligned16(L.w_bf16);
}


// ============================================================================ GEMM chains
// Launches the recorded jobs as one persistent kernel (gemm_chain.cuh).  Must be called before
// anything else is enqueued on `st` that reads what the jobs write.
// CTA pairs of the chained kernel the device can co-schedule (every cluster must be resident at once: the row-block waits assume it)
static int pair_max_clusters(gmvae_handle* h, int* out) {
  static int max_clusters_by_dev[64] = {};
  int& max_clusters = max_clusters_by_dev[tc::current_device()];
  if (max_clusters == 0) {
    GM_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_chain_kernel<tc::ChainParams, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::CHAIN_SMEM_BYTES));
    cudaLaunchConfig_t qc = {};
    qc.gridDim = dim3(tc::num_sms() & ~1); qc.blockDim = dim3(tc::NUM_THREADS2); qc.dynamicSmemBytes = tc::CHAIN_SMEM_BYTES;
    cudaLaunchAttribute qa[1];
    qa[0].id = cudaLaunchAttributeClusterDimension; qa[0].val.clusterDim.x = 2; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
    qc.attrs = qa; qc.numAttrs = 1;
    int n = 0;
    GM_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&n, tc::gemm_chain_kernel<tc::ChainParams, 2>, &qc));
    GM_REQUIRE(n >= 1, "the device cannot co-schedule a CTA pair of the chained kernel");
    max_clusters = n;
  }
  *out = max_clusters;
  return 0;
}

static int chain_flush(gmvae_handle* h, cudaStream_t st) {
  h->chain_flush_after = false;
  h->last_gemm_chained = false;
  if (h->chain.njobs == 0) return 0;
  static bool attr_set_by_dev[64] = {};                      // cudaFuncSetAttribute is per device
  bool& attr_set = attr_set_by_dev[tc::current_device()];
  if (!attr_set) {
    GM_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_chain_kernel<tc::ChainParams, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::CHAIN_SMEM_BYTES));
    GM_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_chain_kernel<tc::ChainParamsSmall, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::CHAIN_SMEM_BYTES));
    attr_set = true;
  }
  h->chain.counters = h->chain_counters;
  h->chain.trace = (h->chain_trace && h->chain_launch_idx < 8) ? h->chain_trace + (size_t)h->chain_launch_idx * 64 * 16 : nullptr;
  h->chain.trace_cta = h->chain_trace_cta;
  { static const int abl = getenv("GMVAE_CHAIN_ABL") ? atoi(getenv("GMVAE_CHAIN_ABL")) : 0; h->chain.abl = abl; }
  h->chain.jobstat = (h->chain_jobstat && h->chain_launch_idx == 0) ? h->chain_jobstat : nullptr;
  if (h->chain.jobstat) {
    h->chain_jobdesc.clear();
    for (int j = 0; j < h->chain.njobs; ++j) {
      const tc::ChainJob& J = h->chain.jobs[j];
      const int d[8] = {J.kind, J.M, J.N, J.kb1 + J.kb2, J.total_tiles, J.num_splits, J.block_n, J.ndeps};
      h->chain_jobdesc.insert(h->chain_jobdesc.end(), d, d + 8);
    }
  }
  h->chain_launch_idx++;
  if (h->chain_quad) {
    // clusters of two CTA pairs; chain_tiles counts double tiles
    const int clusters = std::max(1, std::min(h->chain_tiles, h->max_quads));
    GM_CHECK_CUDA(launch_k_cluster(tc::gemm_chain_kernel<tc::ChainParams, 4>, dim3(4 * clusters), dim3(tc::NUM_THREADS2), (size_t)tc::CHAIN_SMEM_BYTES, st, true, 4,
                           h->chain));
  } else if (h->chain_pair) {
    // CTA pairs: clusters of 2 (the two SMs of a TPC); chain_tiles counts pair tiles.  Every cluster must be resident at once
    // (the row-block waits assume it), so the grid is capped by what the device can co-schedule.
    int max_clusters = 0;
    GM_TRY(pair_max_clusters(h, &max_clusters));
    const int pairs = std::max(1, std::min(std::min(h->chain_tiles, tc::num_sms() / 2), max_clusters));
    GM_CHECK_CUDA(launch_k_cluster(tc::gemm_chain_kernel<tc::ChainParams, 2>, dim3(2 * pairs), dim3(tc::NUM_THREADS2), (size_t)tc::CHAIN_SMEM_BYTES, st, true, 2,
                           h->chain));
  } else {
  const int grid = std::min(h->chain_tiles, tc::num_sms());
  if (h->chain.njobs <= tc::CHAIN_SMALL_JOBS && h->chain.nmaps <= tc::CHAIN_SMALL_MAPS) {
    static tc::ChainParamsSmall small;                      // the launch copies it
    small.njobs = h->chain.njobs; small.nmaps = h->chain.nmaps; small.counters = h->chain.counters;
    small.trace = h->chain.trace; small.trace_cta = h->chain.trace_cta; small.jobstat = h->chain.jobstat; small.abl = h->chain.abl;
    memcpy(small.maps, h->chain.maps, sizeof(CUtensorMap) * h->chain.nmaps);
    memcpy(small.jobs, h->chain.jobs, sizeof(tc::ChainJob) * h->chain.njobs);
    GM_CHECK_CUDA(launch_k(tc::gemm_chain_kernel<tc::ChainParamsSmall, 1>, dim3(grid), dim3(tc::NUM_THREADS2), (size_t)tc::CHAIN_SMEM_BYTES, st, true, small));
  } else {
    GM_CHECK_CUDA(launch_k(tc::gemm_chain_kernel<tc::ChainParams, 1>, dim3(grid), dim3(tc::NUM_THREADS2), (size_t)tc::CHAIN_SMEM_BYTES, st, true, h->chain));
  }
  }
  h->chain.njobs = 0; h->chain.nmaps = 0; h->chain_tiles = 0; h->chain_writers.clear();
  h->launches++;
  if (h->profiling) GM_TRY(profile_mark(h, st, 0 /*PC_TC_GEMM*/));
  if (h->debug_flags & DBG_SYNC_EACH) GM_CHECK_CUDA(cudaStreamSynchronize(st));
  return 0;
}

template <typename T, int MODE> static void writer_range(const EpiStore<T, MODE>& e, int M, const char*& lo, const char*& hi) {
  lo = reinterpret_cast<const char*>(e.out); hi = lo + (int64_t)M * e.ld * sizeof(T);
}
template <typename T> static void writer_range(const EpiBCE<T>& e, int M, const char*& lo, const char*& hi) {
  lo = reinterpret_cast<const char*>(e.dlogits); hi = lo + (int64_t)M * e.ld * sizeof(T);
}
template <typename T, typename HT> static void writer_range(const EpiReluMask<T, HT>& e, int M, const char*& lo, const char*& hi) {
  lo = reinterpret_cast<const char*>(e.out); hi = lo + (int64_t)M * e.ld * sizeof(T);
}
static void writer_range(const EpiAtomicAdd&, int, const char*& lo, const char*& hi) { lo = hi = nullptr; }

// What the chained kernel's epilogue writes through TMA (pointer, row stride, element size) and, for the
// backward ReLU mask, reads through TMA.
struct ChainIO { const void* out; int64_t ld; int elem; const void* opnd; int64_t ld_opnd; bool ok; };
static ChainIO chain_io(const EpiStore<bf16, EPI_PLAIN>& e) { return {e.out, e.ld, 2, nullptr, 0, true}; }
static ChainIO chain_io(const EpiStore<float, EPI_PLAIN>& e) { return {nullptr, e.ld, 4, nullptr, 0, true}; }     // per-row stores
static ChainIO chain_io(const EpiBCE<bf16>& e) {
  return {e.dlogits, e.ld, 2, nullptr, 0, e.row_weight == nullptr && e.row_sum == nullptr && e.x_row_div == 1};
}
static ChainIO chain_io(const EpiReluMask<bf16, bf16>& e) { return {e.out, e.ld, 2, e.h, e.ldh, true}; }
static ChainIO chain_io(const EpiAtomicAdd& e) {
  const bool tma = e.ld % 4 == 0 && (reinterpret_cast<uintptr_t>(e.out) & 15) == 0;
  return {tma ? e.out : nullptr, e.ld, 4, nullptr, 0, true};
}

// Appends C = A1*B1 (+ A2*B2) with epilogue `epi` to the chain being recorded.  Dependencies on
// earlier jobs of the chain are inferred from the operand pointers: an operand that lies in the
// output of a recorded job makes this job wait for that job's row blocks.
template <class Epi>
static int chain_add(gmvae_handle* h, const tc::Operand& A1, const tc::Operand& B1, const tc::Operand* A2, const tc::Operand* B2,
                     int M, int N, int block_n, bool a_mn, bool b_mn, int split_k, const Epi& epi, cudaStream_t st) {
  static_assert(tc::epi_kind<Epi>::value != tc::EK_NONE, "epilogue not supported by the chained kernel");
  static_assert(sizeof(Epi) <= tc::CHAIN_EPI_BYTES, "epilogue parameters do not fit the job record");
  const bool pair = h->chain_pair, quad = h->chain_quad;
  // ---- dependencies
  const void* reads[4] = {A1.ptr, A2 ? A2->ptr : nullptr, a_mn ? (const void*)B1.ptr : nullptr, epi.read_ptr()};
  tc::ChainDep deps[tc::CHAIN_MAX_DEPS]; int ndeps = 0, epi_dep = -1;
  bool need_flush = h->chain.njobs >= tc::CHAIN_MAX_JOBS || h->chain.nmaps + 6 > tc::CHAIN_MAX_MAPS;
  for (int i = 0; i < 4 && !need_flush; ++i) {
    const char* p = reinterpret_cast<const char*>(reads[i]);
    if (!p) continue;
    for (const auto& w : h->chain_writers) {
      if (p < w.lo || p >= w.hi) continue;
      const tc::ChainJob& P = h->chain.jobs[w.job];
      if (p != w.lo || P.sig_base < 0) { need_flush = true; break; }          // offset view / no counters: order by kernel boundary
      int dup = -1;
      for (int d = 0; d < ndeps; ++d) if (deps[d].base == P.sig_base) dup = d;
      if (dup >= 0) {
        if (i == 3) { if (deps[dup].by_k) { need_flush = true; break; } epi_dep = dup; }
        if (i != 1) deps[dup].seg2 = 0;
        continue;
      }
      if (ndeps == tc::CHAIN_MAX_DEPS) { need_flush = true; break; }
      if (i == 3) epi_dep = ndeps;
      // by_k: this operand's rows are the contraction dimension (weight gradient over the batch)
      const bool by_k = a_mn && i != 3;
      // an operand of the second K segment only (i == 1, K-major jobs): its rows are needed when that segment starts
      deps[ndeps++] = tc::ChainDep{P.sig_base, tc::EPI_WARPS * P.tiles_n * P.num_splits, by_k ? 1 : 0, (P.M + tc::BLOCK_M - 1) / tc::BLOCK_M,
                                   (i == 1 && !a_mn) ? 1 : 0};
    }
  }
  if (need_flush) { GM_TRY(chain_flush(h, st)); ndeps = 0; epi_dep = -1; }
  // ---- the job
  tc::ChainJob& J = h->chain.jobs[h->chain.njobs];
  auto mk = [&](int* idx, const tc::Operand& o, bool mn, int box_rows) -> int {
    CUtensorMap* m = &h->chain.maps[h->chain.nmaps];
    *idx = h->chain.nmaps++;
    if (mn) return tc::make_tmap_bf16(m, o.ptr, (uint64_t)o.rows, (uint64_t)o.k, (uint64_t)o.ld, 64, tc::BLOCK_K);
    return tc::make_tmap_bf16(m, o.ptr, (uint64_t)o.k, (uint64_t)o.rows, (uint64_t)o.ld, tc::BLOCK_K, (uint32_t)box_rows);
  };
  const int b_box_rows = pair ? block_n / 2 : block_n;                 // K-major B: a CTA of a pair loads half of the tile's rows
  GM_REQUIRE(!pair || block_n % 16 == 0, "pair tiles need a tile width that is a multiple of 16");
  const int a_box_rows = quad ? 64 : tc::BLOCK_M;                      // quad mode loads A in halves of 64 rows
  GM_TRY(mk(&J.a1, A1, a_mn, a_box_rows));
  GM_TRY(mk(&J.b1, B1, b_mn, b_box_rows));
  J.kb1 = (A1.k + tc::BLOCK_K - 1) / tc::BLOCK_K; J.kb2 = 0;
  if (A2 && B2) {
    GM_TRY(mk(&J.a2, *A2, a_mn, a_box_rows));
    GM_TRY(mk(&J.b2, *B2, b_mn, b_box_rows));
    J.kb2 = (A2->k + tc::BLOCK_K - 1) / tc::BLOCK_K;
  } else {
    J.a2 = J.a1; J.b2 = J.b1;
  }
  const int kb_total = J.kb1 + J.kb2;
  tc::chain_job_geometry(J, M, N, block_n, split_k, kb_total, a_mn, quad ? 4 : pair ? 2 : 1);      // chain_sched.cuh
  J.b_mn = b_mn ? 1 : 0; J.kind = tc::epi_kind<Epi>::value;
  J.tile_base = h->chain_tiles;
  {
    const int part = h->part_on ? h->cur_part : 0;
    J.wfirst = part == 2 ? h->part_chain_walkers : 0;
    J.wcount = part == 1 ? h->part_chain_walkers : part == 2 ? h->part_walkers - h->part_chain_walkers : 0;
    J.tile_base = part == 0 ? h->chain_tiles : h->part_tiles[part];
    h->part_tiles[part] += J.walk_total;
  }
  J.ndeps = ndeps; J.epi_dep = epi_dep;
  for (int d = 0; d < ndeps; ++d) J.deps[d] = deps[d];
  const char *lo, *hi;
  writer_range(epi, M, lo, hi);
  J.sig_base = -1;
  if (lo) {
    const int ncount = tc::chain_job_counters(M, quad ? 4 : pair ? 2 : 1);
    if (h->chain_counter_next + ncount <= h->chain_counter_cap) {
      J.sig_base = h->chain_counter_next; h->chain_counter_next += ncount;
    } else {
      h->chain_flush_after = true;     // out of counters: later readers are ordered by the kernel boundary
    }
    h->chain_writers.push_back({lo, hi, h->chain.njobs});
  }
  // epilogue I/O through TMA: boxes of 32 rows x 64 bytes (one patch of the kernel)
  const ChainIO io = chain_io(epi);
  J.gw = 0; J.c = J.a1; J.d = J.a1;
  J.zslice = (h->det && tc::epi_kind<Epi>::value == tc::EK_ATOMIC) ? 1 : 0;
  GM_REQUIRE(!J.zslice || io.out, "deterministic mode: weight-gradient slices need 16-byte rows");
  if (io.out) {
    J.gw = io.elem == 2 ? 2 : 1;
    J.d = h->chain.nmaps++;
    if (J.zslice)   // k-split z stores into slice z (lin_wgrad sized the buffer for these splits)
      GM_TRY(tc::make_tmap_slices_f32(&h->chain.maps[J.d], io.out, (uint64_t)N, (uint64_t)M, (uint64_t)J.num_splits, (uint64_t)io.ld, 16, 32));
    else
      GM_TRY(tc::make_tmap(&h->chain.maps[J.d], io.out, io.elem, (uint64_t)N, (uint64_t)M, (uint64_t)io.ld, io.elem == 2 ? 32 : 16, 32, 64));
    if (io.opnd) {
      J.c = h->chain.nmaps++;
      GM_TRY(tc::make_tmap(&h->chain.maps[J.c], io.opnd, 2, (uint64_t)N, (uint64_t)M, (uint64_t)io.ld_opnd, 32, 32, 64));
    }
  }
  memset(J.epi, 0, sizeof(J.epi));
  memcpy(J.epi, &epi, sizeof(Epi));
  J.fuse = 0;
  if (h->fuse_next.kind != 0 && tc::epi_kind<Epi>::value == tc::EK_STORE_F32 && N <= 16 && J.sig_base >= 0) {
    J.fuse = h->fuse_next.kind;
    memcpy(J.epi2, h->fuse_next.prm, sizeof(J.epi2));
    for (const auto& w : h->fuse_next.writes)
      if (w.first) h->chain_writers.push_back({reinterpret_cast<const char*>(w.first), reinterpret_cast<const char*>(w.first) + w.second, h->chain.njobs});
    h->fuse_next.consumed = true;
  }
  h->chain_tiles += J.walk_total;
  h->chain.njobs++;
  h->last_gemm_chained = true;
  if (h->chain_flush_after) GM_TRY(chain_flush(h, st));
  return 0;
}
// Appends a row job (a distribution head run by the epilogue warps on 128-row blocks) to the chain.
// `reads`: buffers whose rows it consumes; `writes`: {pointer, bytes} of every buffer it produces.
template <class P>
static int chain_add_rows(gmvae_handle* h, int kind, const P& prm, int M, std::initializer_list<const void*> reads,
                          std::initializer_list<std::pair<const void*, size_t>> writes, cudaStream_t st, int sub = 1) {
  static_assert(sizeof(P) <= tc::CHAIN_EPI_BYTES, "row-job parameters do not fit the job record");
  const int tiles_m = (M + tc::BLOCK_M - 1) / tc::BLOCK_M;
  tc::ChainDep deps[tc::CHAIN_MAX_DEPS]; int ndeps = 0;
  bool need_flush = h->chain.njobs >= tc::CHAIN_MAX_JOBS;
  for (const void* r : reads) {
    const char* p = reinterpret_cast<const char*>(r);
    if (!p || need_flush) continue;
    for (const auto& w : h->chain_writers) {
      if (p < w.lo || p >= w.hi) continue;
      const tc::ChainJob& Pj = h->chain.jobs[w.job];
      if (p != w.lo || Pj.sig_base < 0) { need_flush = true; break; }
      bool dup = false;
      for (int d = 0; d < ndeps; ++d) dup = dup || deps[d].base == Pj.sig_base;
      if (dup) continue;
      if (ndeps == tc::CHAIN_MAX_DEPS) { need_flush = true; break; }
      deps[ndeps++] = tc::ChainDep{Pj.sig_base, tc::EPI_WARPS * Pj.tiles_n * Pj.num_splits, 0, (Pj.M + tc::BLOCK_M - 1) / tc::BLOCK_M, 0};
    }
  }
  if (need_flush) { GM_TRY(chain_flush(h, st)); ndeps = 0; }
  tc::ChainJob& J = h->chain.jobs[h->chain.njobs];
  memset(&J, 0, sizeof(J));
  J.M = M; J.N = 0; J.kind = kind; J.num_splits = 1;
  // row tiles are dealt to single CTAs also in pair mode, where chain_tiles counts pair tiles
  J.tiles_n = sub; J.tiles_mn = tiles_m * sub; J.total_tiles = tiles_m * sub; J.tile_base = (h->chain_quad ? 4 : h->chain_pair ? 2 : 1) * h->chain_tiles;
  {
    const int cl = h->chain_quad ? 4 : h->chain_pair ? 2 : 1;
    const int part = h->part_on ? h->cur_part : 0;
    J.wfirst = part == 2 ? h->part_chain_walkers : 0;
    J.wcount = part == 1 ? h->part_chain_walkers : part == 2 ? h->part_walkers - h->part_chain_walkers : 0;
    if (part != 0) J.tile_base = cl * h->part_tiles[part];
    h->part_tiles[part] += (tiles_m * sub + cl - 1) / cl;
  }
  J.ndeps = ndeps; J.epi_dep = -1;
  for (int d = 0; d < ndeps; ++d) J.deps[d] = deps[d];
  J.sig_base = -1;
  if (h->chain_counter_next + tiles_m <= h->chain_counter_cap) {
    J.sig_base = h->chain_counter_next; h->chain_counter_next += tiles_m;
  } else {
    h->chain_flush_after = true;
  }
  for (const auto& w : writes)
    if (w.first) h->chain_writers.push_back({reinterpret_cast<const char*>(w.first), reinterpret_cast<const char*>(w.first) + w.second, h->chain.njobs});
  memcpy(J.epi, &prm, sizeof(P));
  { const int cl = h->chain_quad ? 4 : h->chain_pair ? 2 : 1; h->chain_tiles += (J.total_tiles + cl - 1) / cl; }
  h->chain.njobs++;
  if (h->chain_flush_after) GM_TRY(chain_flush(h, st));
  return 0;
}
template <class Epi> struct chainable { static constexpr bool value = tc::epi_kind<Epi>::value != tc::EK_NONE; };

template <class Epi, bool B_MN = false>
static int tc_dispatch_kk(gmvae_handle* h, const tc::Operand& A, const tc::Operand& B, const tc::Operand* A2,
                          const tc::Operand* B2, int M, int N, const Epi& epi, cudaStream_t st) {
  int r;
  if constexpr (chainable<Epi>::value) {
    if (h->chain_on && chain_io(epi).ok) {
      // outputs staged for TMA stores use tiles that are whole 32-column groups; MN-major B comes in 64-column slabs
      const bool f32 = tc::epi_kind<Epi>::value == tc::EK_STORE_F32;
      int bn = (!B_MN && f32 && N <= 16) ? 16 : (!B_MN && f32 && N <= 32) ? 32 : N <= 64 ? 64 : (N <= 128 || (h->debug_flags & DBG_BN128)) ? 128 : 256;
      if (bn == 256 && h->wide_bn > 0 && N > h->wide_bn) bn = h->wide_bn;       // tile width of the wide layers (GMVAE_CHAIN_BN)
      return chain_add(h, A, B, A2, B2, M, N, bn, false, B_MN, 1, epi, st);
    }
  }
  GM_TRY(chain_flush(h, st));
  if constexpr (B_MN) {
    if (N <= 64) r = tc::launch_gemm_tc<64, false, true, Epi>(A, B, A2, B2, M, N, 1, epi, st);
    else if (N <= 128 || (h->debug_flags & DBG_BN128)) r = tc::launch_gemm_tc<128, false, true, Epi>(A, B, A2, B2, M, N, 1, epi, st);
    else r = tc::launch_gemm_tc<256, false, true, Epi>(A, B, A2, B2, M, N, 1, epi, st);
  } else {
    if (N <= 16) r = tc::launch_gemm_tc<16, false, false, Epi>(A, B, A2, B2, M, N, 1, epi, st);
    else if (N <= 32) r = tc::launch_gemm_tc<32, false, false, Epi>(A, B, A2, B2, M, N, 1, epi, st);
    else if (N <= 64) r = tc::launch_gemm_tc<64, false, false, Epi>(A, B, A2, B2, M, N, 1, epi, st);
    else if (N <= 128 || (h->debug_flags & DBG_BN128)) r = tc::launch_gemm_tc<128, false, false, Epi>(A, B, A2, B2, M, N, 1, epi, st);
    else r = tc::launch_gemm_tc<256, false, false, Epi>(A, B, A2, B2, M, N, 1, epi, st);
  }
  if (r == 0) GM_LAUNCHED(h, st, PC_TC_GEMM);
  return r;
}

// C[M,out] = A[M,in] * W (+ A2[M,in2] * W2)        forward through a linear layer
template <typename TA, class Epi, bool ALLOW_TC = true>
static int lin_fwd(gmvae_handle* h, const TA* A, int64_t lda, int M, const LinView& L, const Epi& epi, cudaStream_t st,
                   const TA* A2 = nullptr, int64_t lda2 = 0, const LinView* L2 = nullptr) {
  if constexpr (ALLOW_TC && std::is_same<TA, bf16>::value) {
    bool ok = tc_ok_fwd<TA>(h, A, lda, L);
    if (L2) ok = ok && lda2 % 8 == 0 && aligned16(A2) && aligned16(L2->w_bf16);
    if (ok) {
      // K extents are rounded up to the (zero-filled) 16-byte padding of the buffers.
      // B = W[in, out] as stored (row-major, the contraction index is the row): an MN-major operand.  Rows of W
      // beyond `in` are outside the tensor map (read as zero); A's zero padding covers the rounded-up K extent.
      tc::Operand a{A, lda, M, kpad(L.in, lda)}, b{L.w_bf16, L.ld_w, L.out, L.in};
      if (L2) {
        tc::Operand a2{A2, lda2, M, kpad(L2->in, lda2)}, b2{L2->w_bf16, L2->ld_w, L2->out, L2->in};
        return tc_dispatch_kk<Epi, true>(h, a, b, &a2, &b2, M, L.out, epi, st);
      }
      return tc_dispatch_kk<Epi, true>(h, a, b, nullptr, nullptr, M, L.out, epi, st);
    }
  }
  GM_REQUIRE(L2 == nullptr, "two-segment forward requires the tensor-core path");
  GM_TRY(chain_flush(h, st));
  GM_CHECK_CUDA((launch_gemm_simt<TA, float, Epi>(A, lda, 1, L.w, L.ldw32, 1, M, L.out, L.in, 1, epi, st)));
  GM_LAUNCHED(h, st, PC_SIMT_GEMM);
  return 0;
}

// dX[M,in] = dY[M,out] * W^T  (+ dY2[M,out2] * W2^T: two layers reading the same input, one accumulator)
template <typename TD, class Epi>
static int lin_dgrad(gmvae_handle* h, const TD* dY, int64_t ldy, int M, const LinView& L, const Epi& epi, cudaStream_t st,
                     const TD* dY2 = nullptr, int64_t ldy2 = 0, const LinView* L2 = nullptr) {
  if constexpr (std::is_same<TD, bf16>::value) {
    bool ok = tc_ok_dgrad<TD>(h, dY, ldy, L);
    if (L2) ok = ok && tc_ok_dgrad<TD>(h, dY2, ldy2, *L2) && L2->in == L.in;
    if (ok) {
      tc::Operand a{dY, ldy, M, kpad(L.out, ldy)}, b{L.w_bf16, L.ld_w, L.in, kpad(L.out, L.ld_w)};
      if (L2) {
        tc::Operand a2{dY2, ldy2, M, kpad(L2->out, ldy2)}, b2{L2->w_bf16, L2->ld_w, L2->in, kpad(L2->out, L2->ld_w)};
        return tc_dispatch_kk(h, a, b, &a2, &b2, M, L.in, epi, st);
      }
      return tc_dispatch_kk(h, a, b, nullptr, nullptr, M, L.in, epi, st);
    }
  }
  GM_REQUIRE(L2 == nullptr, "two-segment data gradient requires the tensor-core path");
  GM_TRY(chain_flush(h, st));
  GM_CHECK_CUDA((launch_gemm_simt<TD, float, Epi>(dY, ldy, 1, L.w, 1, L.ldw32, M, L.in, L.out, 1, epi, st)));
  GM_LAUNCHED(h, st, PC_SIMT_GEMM);
  return 0;
}

// Tile width and k-split of a weight-gradient GEMM on the tensor cores: one wave of persistent CTAs (CTA pairs): split the batch
// so that tiles * split ~ number of SMs (pairs), keeping at least 4 k-blocks (256 samples) per split.
// (with the walker partition a job is two rounds of the weight-gradient pairs: same tiles, same split)
// (measured at cfg4, tiles x splits as a multiple of the walkers: 0.34 / 0.5 / 0.75 / 1 / 2 / 3 / 4 -> 0.386 / 0.356 / 0.348 / 0.347 / 0.376 /
// 0.395 / 0.419 ms: shorter tiles pay the reduce-add epilogue more often, longer ones leave pairs without a tile)
static int wgrad_bn(const gmvae_handle* h, int out) { return out <= 64 ? 64 : (out <= 128 || (h->debug_flags & DBG_BN128)) ? 128 : 256; }
static int wgrad_split(const gmvae_handle* h, int in, int out, int M, bool pair, bool quad) {
  const int bn = wgrad_bn(h, out);
  const int tiles = pair ? ((in + 255) / 256) * ((out + bn - 1) / bn) : ((in + 127) / 128) * ((out + bn - 1) / bn);
  const int kb = (M + tc::BLOCK_K - 1) / tc::BLOCK_K;
  const int walkers = quad ? h->max_quads : pair ? tc::num_sms() / 2 : tc::num_sms(), units = quad ? (tiles + 1) / 2 : tiles;   // quad: 4-CTA clusters, double tiles
  return std::max(1, std::min(std::max(1, kb / 4), walkers / units));
}

// dW[in,out] += A^T[in,M] * dY[M,out]   (grads pre-zeroed; split over the batch, fp32 atomics; deterministic mode: k-split slices)
template <typename TA, typename TD>
static int lin_wgrad(gmvae_handle* h, const TA* A, int64_t lda, const TD* dY, int64_t ldy, int M, const LinView& L,
                     cudaStream_t st) {
  EpiAtomicAdd epi{L.dw, (int64_t)L.ldw32};
  if constexpr (std::is_same<TA, bf16>::value && std::is_same<TD, bf16>::value) {
    bool ok = h->bf16_mode() && !(h->debug_flags & (DBG_NO_TC | DBG_NO_TC_WGRAD)) && lda % 8 == 0 && ldy % 8 == 0 &&
              aligned16(A) && aligned16(dY);
    if (ok) {
      tc::Operand a{A, lda, kpad(L.in, lda), M}, b{dY, ldy, kpad(L.out, ldy), M};
      const int bn = wgrad_bn(h, L.out);
      const bool pair = h->chain_on && h->chain_pair;
      const int split = wgrad_split(h, L.in, L.out, M, pair, pair && h->chain_quad);
      if (h->chain_on) {
        EpiAtomicAdd e = epi;
        if (h->det) {
          // the k-splits store their partials into slices of this job's buffer (chain_add: a 3-D tensor map); the reduction step
          // adds slices 0 .. S-1 of every element in that order
          const int kb = (M + tc::BLOCK_K - 1) / tc::BLOCK_K, per = (kb + split - 1) / split, S = (kb + per - 1) / per;
          const int ld = tc::det_slice_ld(L.out);
          const int64_t need = round_up((int)std::min<int64_t>((int64_t)S * L.in * ld, 1LL << 30), 64);
          GM_REQUIRE(h->det_wg_next + need <= h->det_wg_cap && (int)h->det_segs.size() < DET_MAX_SEGS,
                     "deterministic mode: out of weight-gradient partial space");
          float* part = h->buf<float>("det.wg") + h->det_wg_next;
          h->det_wg_next += need;
          e = EpiAtomicAdd{part, (int64_t)ld};
          h->det_segs.push_back(DetSeg{L.dw, part, nullptr, (long long)L.in * ld, L.in, L.out, S, L.ldw32, ld, 0});
        }
        const int saved_part = h->cur_part;
        if (saved_part == 1) h->cur_part = h->part_tail ? 0 : 2;      // weight gradients: their own walkers (the tail: everybody)
        const int r = chain_add(h, a, b, nullptr, nullptr, L.in, L.out, bn, true, true, split, e, st);
        h->cur_part = saved_part;
        return r;
      }
      GM_REQUIRE(!h->det, "deterministic mode: weight gradients outside the chained kernel");   // (bf16 always chains there)
      GM_TRY(chain_flush(h, st));
      int r = bn == 64    ? tc::launch_gemm_tc<64, true, true, EpiAtomicAdd>(a, b, nullptr, nullptr, L.in, L.out, split, epi, st)
              : bn == 128 ? tc::launch_gemm_tc<128, true, true, EpiAtomicAdd>(a, b, nullptr, nullptr, L.in, L.out, split, epi, st)
                          : tc::launch_gemm_tc<256, true, true, EpiAtomicAdd>(a, b, nullptr, nullptr, L.in, L.out, split, epi, st);
      if (r == 0) GM_LAUNCHED(h, st, PC_TC_WGRAD);
      return r;
    }
  }
  GM_TRY(chain_flush(h, st));
  const int tiles = ((L.in + SIMT_BM - 1) / SIMT_BM) * ((L.out + SIMT_BN - 1) / SIMT_BN);
  int split = std::max(1, std::min((M + 255) / 256, (4 * 148 + tiles - 1) / tiles));
  if (h->det) split = 1;
  GM_CHECK_CUDA((launch_gemm_simt<TA, TD, EpiAtomicAdd>(A, 1, lda, dY, ldy, 1, L.in, L.out, M, split, epi, st)));
  GM_LAUNCHED(h, st, PC_SIMT_GEMM);
  return 0;
}

template <typename T>
static int bias_grad(gmvae_handle* h, const T* dY, int64_t ldy, int M, int N, float* db, cudaStream_t st) {
  const int col_blocks = (N + 255) / 256;
  int rows_per_block = std::max(64, (M * col_blocks + 2 * 148 - 1) / (2 * 148));
  float* part = nullptr;
  if (h->det) {
    // DET_ROW_BLOCKS partial rows (row blocks beyond M store zeros), summed in order by the reduction step
    rows_per_block = std::max(8, (M + DET_ROW_BLOCKS - 1) / DET_ROW_BLOCKS);
    GM_REQUIRE(h->det_part_next + (int64_t)N * DET_ROW_BLOCKS <= h->det_part_cap && (int)h->det_segs.size() < DET_MAX_SEGS,
               "deterministic mode: out of partial-sum space");
    part = h->buf<float>("det.part") + h->det_part_next;
    h->det_part_next += (int64_t)N * DET_ROW_BLOCKS;
    h->det_segs.push_back(DetSeg{db, part, nullptr, N, 1, N, DET_ROW_BLOCKS, 0, N, 0});
    // run after the step's last chained launch (dY stays untouched until the step ends): the chain is not cut here
    const int rpb = round_up(rows_per_block, 8);
    h->det_colsums.push_back([=]() -> int {
      GM_CHECK_CUDA(launch_k(colsum_kernel<T>, dim3(col_blocks, DET_ROW_BLOCKS), dim3(256), 0, st, true, dY, ldy, M, N, rpb, db, part));
      GM_LAUNCHED(h, st, PC_BIAS_GRAD);
      return 0;
    });
    return 0;
  }
  rows_per_block = round_up(rows_per_block, 8);
  dim3 grid(col_blocks, (M + rows_per_block - 1) / rows_per_block);
  GM_TRY(chain_flush(h, st));
  GM_CHECK_CUDA(launch_k(colsum_kernel<T>, grid, dim3(256), 0, st, true, dY, ldy, M, N, rows_per_block, db, part));
  GM_LAUNCHED(h, st, PC_BIAS_GRAD);
  return 0;
}

// ============================================================================ MLP passes
// Every GEMM-operand activation buffer has its row stride rounded up to 8 elements (16 bytes, the
// TMA requirement); the padding columns are never written and stay zero from allocation.
static inline int ldp(int n) { return round_up(n, 8); }

template <typename A> struct MlpBufs { std::vector<A*> hid, dhid; std::vector<uint32_t*> bits; };

template <typename A>
static MlpBufs<A> mlp_bufs(const gmvae_handle* h, const Mlp& m) {
  MlpBufs<A> b;
  for (size_t i = 0; i + 1 < m.layers.size(); ++i) {
    b.hid.push_back(h->buf<A>(m.name + ".h" + std::to_string(i)));
    b.dhid.push_back(h->buf<A>(m.name + ".dh" + std::to_string(i)));
    b.bits.push_back(h->buf<uint32_t>(m.name + ".bits" + std::to_string(i)));
  }
  return b;
}

// Hidden layers i >= first of an MLP: h[i] = relu(h[i-1] W_i + b_i). Layer 0's input is `in0`
// (row stride ld0) and multiplies the first `in0_cols` rows of W_0.
template <typename A>
static int mlp_hidden_fwd(gmvae_handle* h, const Mlp& m, const MlpBufs<A>& b, const A* in0, int64_t ld0, int in0_cols, int M,
                          int first, cudaStream_t st) {
  const int nh = (int)m.layers.size() - 1;
  for (int i = first; i < nh; ++i) {
    const A* in = i == 0 ? in0 : b.hid[i - 1];
    int64_t ld = i == 0 ? ld0 : ldp(m.layers[i - 1].out);
    LinView L = view(h, m.layers[i], 0, i == 0 ? in0_cols : -1);
    EpiStore<A> epi{b.hid[i], (int64_t)ldp(m.layers[i].out), L.b, nullptr, 0, 1, 1.f};
    if (tc::CHAIN_RELU_BITS && h->chain_on && h->row_jobs && !(h->debug_flags & DBG_NO_RELU_BITS)) { epi.relu_bits = b.bits[i]; epi.ld_bits = round_up(M, 32); }
    GM_TRY(lin_fwd<A>(h, in, ld, M, L, epi, st));
    h->relu_bits_valid[b.hid[i]] = epi.relu_bits != nullptr && h->last_gemm_chained;
  }
  return 0;
}

// Backward through the whole MLP given dOut = d loss / d (last layer output).
// Computes every dW, db and the hidden gradients down to dh[0]; the gradient w.r.t. the MLP
// input is left to the caller (it is only needed for z and y, never for the image x).
// `in0_cols` = how many leading rows of W_0 multiply `in0` (encoder_gmm: D of D+K).
// On the tensor-core path the dgrad epilogue that writes dh[i-1] also reduces its columns, which
// is the bias gradient of layer i-1 (no separate pass over dh).
template <typename A, typename TD>
static int mlp_backward(gmvae_handle* h, const Mlp& m, const MlpBufs<A>& b, const A* in0, int64_t ld0, int in0_cols,
                        const TD* dOut, int64_t ld_dout, int M, cudaStream_t st, bool dout_bias_done = false, int min_layer = 0,
                        std::vector<std::function<int()>>* defer = nullptr, int defer_below = 0) {
  // `defer`: the weight-gradient GEMMs of layers < defer_below (off the critical path of the backward pass) are not
  // issued here but returned, upper layer first, so that the caller can place them where the chain of dependent
  // jobs needs filler work.
  const int nl = (int)m.layers.size();
  const bool fuse = !(h->debug_flags & DBG_NO_FUSED_COLSUM) && !h->det;   // deterministic mode: column sums by bias_grad
  bool bias_done = dout_bias_done;   // bias gradient of the layer whose output gradient we hold
  // Per layer, top down: first the data gradient (the next layer's input, so the chain of dependent
  // GEMMs keeps moving), then the weight gradient of the same layer (its operands are complete by then).
  for (int i = nl - 1; i >= min_layer; --i) {
    const Linear& l = m.layers[i];
    const bool first = i == 0;
    LinView L = view(h, l, 0, first ? in0_cols : -1);
    const A* in = first ? in0 : b.hid[i - 1];
    const int64_t ld = first ? ld0 : ldp(m.layers[i - 1].out);
    const bool top = i == nl - 1;
    const A* dA = top ? nullptr : b.dhid[i];
    const int64_t ldd = top ? ld_dout : ldp(l.out);
    bool next_bias_done = false;
    if (!first) {
      LinView Lf = view(h, l);
      const int64_t ldh = ldp(m.layers[i - 1].out);
      // (layers below min_layer get their bias gradient from the caller)
      const bool ok = top ? tc_ok_dgrad<TD>(h, dOut, ld_dout, Lf) : tc_ok_dgrad<A>(h, dA, ldd, Lf);
      float* cs = (fuse && i - 1 >= min_layer && ok) ? h->grads + m.layers[i - 1].b_off : nullptr;
      EpiReluMask<A, A> epi{b.dhid[i - 1], ldh, b.hid[i - 1], ldh, cs};
      {
        auto it = h->relu_bits_valid.find(b.hid[i - 1]);
        if (h->chain_on && it != h->relu_bits_valid.end() && it->second) { epi.relu_bits = b.bits[i - 1]; epi.ld_bits = round_up(M, 32); }
      }
      if (top) GM_TRY((lin_dgrad<TD>(h, dOut, ld_dout, M, Lf, epi, st)));
      else GM_TRY((lin_dgrad<A>(h, dA, ldd, M, Lf, epi, st)));
      next_bias_done = cs != nullptr;
      if (h->part_last_mlp && i == 1) h->part_tail = true;      // that was the last job of the dependent chain
    }
    const bool need_bias = !bias_done;
    const int out_cols = l.out;
    std::function<int()> wg;
    if (top) {
      wg = [=]() -> int {
        GM_TRY((lin_wgrad<A, TD>(h, in, ld, dOut, ld_dout, M, L, st)));
        if (need_bias) GM_TRY(bias_grad<TD>(h, dOut, ld_dout, M, out_cols, L.db, st));
        return 0;
      };
    } else {
      wg = [=]() -> int {
        GM_TRY((lin_wgrad<A, A>(h, in, ld, dA, ldd, M, L, st)));
        if (need_bias) GM_TRY(bias_grad<A>(h, dA, ldd, M, out_cols, L.db, st));
        return 0;
      };
    }
    if (h->wg_late) h->wg_late->push_back(wg);
    else if (defer && i < defer_below) defer->push_back(wg); else GM_TRY(wg());
    bias_done = next_bias_done;
  }
  return 0;
}

// ============================================================================ the step
// Input conversion, noise and the encoder side of the forward pass (q(y|x), the relaxed sample y,
// p(z|y), q(z|x,y) / q(z|x)) up to the encoder's [mu|raw] output.  Shared by the training step and by
// gmvae_encode (reconstruct_images / transform of the model classes).
template <typename A>
static int forward_encoder(gmvae_handle* h, const uint8_t* x_u8, int B, float inv_bg, const float*& eps, const float*& u, float* acc,
                           cudaStream_t st) {
  const gmvae_config& c = h->cfg;
  const int D = h->D, Z = h->Z, K = h->K, nl = h->L;
  const int Dp = ldp(D), Kp = ldp(K);
  const bool gm = c.model == GMVAE_MODEL_GMVAE;
  A* x_act = h->buf<A>("x_act");
  {
    const int64_t n = (int64_t)B * D;
    const bool need_noise = !eps || (gm && !u);
    const uint64_t draw = (need_noise && !h->in_train_step) ? ++h->draws : 0;
    float* e = h->buf<float>("eps"); float* uu = gm ? h->buf<float>("u") : nullptr;
    const int64_t ne = eps ? 0 : (int64_t)B * Z, nu = (gm && !u) ? (int64_t)B * K : 0;
    const int64_t q = (ne + 3) / 4 + (nu + 3) / 4;
    // first kernel of the step: follows a memset node, launched with a full dependency
    if (D % 16 == 0 && need_noise) {      // image conversion and noise in one launch
      const unsigned xb = (unsigned)((n / 16 + 255) / 256), nb = (unsigned)((q + 255) / 256);
      GM_CHECK_CUDA(launch_k(prologue_kernel<A>, dim3(xb + nb), dim3(256), 0, st, false, x_u8, x_act, n, (int)xb, e, ne, uu, nu,
                             (const DeviceState*)h->state, (uint64_t)h->rank, draw));
      GM_LAUNCHED(h, st, PC_MISC);
    } else {
      if (D % 16 == 0) GM_CHECK_CUDA(launch_k(convert_x_kernel<A>, dim3((unsigned)((n / 16 + 255) / 256)), dim3(256), 0, st, false, x_u8, x_act, n));
      else GM_CHECK_CUDA(launch_k(convert_x_rows_kernel<A>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, false, x_u8, x_act, B, D, Dp));
      GM_LAUNCHED(h, st, PC_MISC);
      if (need_noise) {
        GM_CHECK_CUDA(launch_k(fill_noise_kernel, dim3((unsigned)((q + 255) / 256)), dim3(256), 0, st, true, e, ne, uu, nu,
                               (const DeviceState*)h->state, (uint64_t)h->rank, 1, draw));
        GM_LAUNCHED(h, st, PC_MISC);
      }
    }
    // The q(y|x) head consumes Gumbel noise g = -log(-log u): drawn that way above, converted here when u was injected.
    if (gm && u) {
      const int64_t nuu = (int64_t)B * K;
      GM_CHECK_CUDA(launch_k(gumbel_from_u_kernel, dim3((unsigned)((nuu + 255) / 256)), dim3(256), 0, st, true, u, uu, nuu));
      GM_LAUNCHED(h, st, PC_MISC);
      u = uu;
    }
    if (!eps) eps = e;
    if (gm && !u) u = uu;
  }
  MlpBufs<A> enc = mlp_bufs<A>(h, h->encoder);
  float* enc_out = h->buf<float>("enc_out");
  const Linear& enc_l0 = h->encoder.layers[0];
  const Linear& enc_last = h->encoder.layers[nl - 1];
  auto hid_ld = [&](int i) { return (int64_t)ldp(h->hidden[i]); };
  if (gm) {
    MlpBufs<A> ey = mlp_bufs<A>(h, h->encoder_y);
    float* logits_y = h->buf<float>("logits_y"); float* y_f32 = h->buf<float>("y_f32"); A* y_act = h->buf<A>("y_act");
    float* prior_out = h->buf<float>("prior_out");
    // q(y|x): encoder_y MLP, logits in fp32 (gmvae.py:238)
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder_y, ey, x_act, Dp, D, B, 0, st));
    const bool rows_ok = h->chain_on && h->row_jobs;
    bool y_fused = false;
    {
      const Linear& l = h->encoder_y.layers[nl - 1];
      EpiStore<float> epi{logits_y, (int64_t)K, h->params + l.b_off, nullptr, 0, 0, 1.f};
      if (rows_ok && K <= 16 && Kp <= 16 && u && !(h->debug_flags & DBG_NO_FUSE_HEADS)) {
        // the q(y|x) head runs in the epilogue of this GEMM (the lane holds the whole row of K logits)
        tc::RowsYFwd prm{logits_y, u, K, 1.f / c.temperature, inv_bg, y_f32, reinterpret_cast<bf16*>(y_act), Kp, acc};
        h->fuse_next = gmvae_handle::FuseReq();
        h->fuse_next.kind = tc::EK_ROWS_Y_FWD;
        memcpy(h->fuse_next.prm, &prm, sizeof(prm));
        h->fuse_next.writes = {{y_f32, (size_t)B * K * 4}, {y_act, (size_t)B * Kp * 2}};
      }
      GM_TRY(lin_fwd<A>(h, nl == 1 ? x_act : ey.hid[nl - 2], nl == 1 ? Dp : hid_ld(nl - 2), B, view(h, l), epi, st));
      y_fused = h->fuse_next.consumed;
      h->fuse_next = gmvae_handle::FuseReq();
    }
    if (y_fused) {
      // nothing to do: y, its bf16 operand row and the entropy term were produced by the logits job
    } else if (rows_ok && K <= 16 && Kp <= 16 && u) {
      // q(y|x) head as a job of the chain: no launch, no pipeline drain between encoder_y and encoder_gmm
      tc::RowsYFwd prm{logits_y, u, K, 1.f / c.temperature, inv_bg, y_f32, reinterpret_cast<bf16*>(y_act), Kp, acc};
      GM_TRY(chain_add_rows(h, tc::EK_ROWS_Y_FWD, prm, B, {logits_y, u},
                            {{y_f32, (size_t)B * K * 4}, {y_act, (size_t)B * Kp * 2}}, st));
    } else {
    GM_TRY(chain_flush(h, st));
    if (std::is_same<A, bf16>::value && K <= 16 && Kp <= 16) {
      GM_CHECK_CUDA(launch_k(head_y_fwd_row_kernel, dim3((B + 127) / 128), dim3(128), 0, st, true, (const float*)logits_y, u, B, K,
                             1.f / c.temperature, inv_bg, y_f32, reinterpret_cast<bf16*>(y_act), Kp, acc));
    } else {
      GM_CHECK_CUDA(launch_k(head_y_fwd_kernel<A>, dim3((B + 7) / 8), dim3(256), 0, st, true, (const float*)logits_y, u, B, K,
                             1.f / c.temperature, inv_bg, y_f32, y_act, Kp, acc));
    }
    GM_LAUNCHED(h, st, PC_HEADS);
    }
    // q(z|x,y) layer 0: [x,y] W = x W[:D] + y W[D:]  (no concat, base.py:66)
    LinView Lx = view(h, enc_l0, 0, D), Ly = view(h, enc_l0, D, K);
    const bool last0 = nl == 1;
    const bool two_seg = tc_ok_fwd<A>(h, x_act, Dp, Lx) && tc_ok_fwd<A>(h, y_act, Kp, Ly) && !(h->debug_flags & DBG_NO_TWO_SEG);
    if (two_seg) {
      if (last0) {
        EpiStore<float> epi{enc_out, (int64_t)2 * Z, Lx.b, nullptr, 0, 0, 1.f};
        GM_TRY(lin_fwd<A>(h, x_act, Dp, B, Lx, epi, st, y_act, Kp, &Ly));
      } else {
        EpiStore<A> epi{enc.hid[0], hid_ld(0), Lx.b, nullptr, 0, 1, 1.f};
        if (tc::CHAIN_RELU_BITS && h->chain_on && h->row_jobs && !(h->debug_flags & DBG_NO_RELU_BITS)) { epi.relu_bits = enc.bits[0]; epi.ld_bits = round_up(B, 32); }
        GM_TRY(lin_fwd<A>(h, x_act, Dp, B, Lx, epi, st, y_act, Kp, &Ly));
        h->relu_bits_valid[enc.hid[0]] = epi.relu_bits != nullptr && h->last_gemm_chained;
      }
    } else {   // fp32 validation mode: pre = y W[D:] + b, then relu(x W[:D] + pre)   (CUDA-core GEMMs)
      float* pre = h->buf<float>("pre_y");
      EpiStore<float> e0{pre, (int64_t)enc_l0.out, Lx.b, nullptr, 0, 0, 1.f};
      GM_TRY((lin_fwd<A, EpiStore<float>, false>(h, y_act, Kp, B, Ly, e0, st)));
      if (last0) {
        EpiStore<float, EPI_ADDEND> epi{enc_out, (int64_t)2 * Z, nullptr, pre, (int64_t)enc_l0.out, 0, 1.f};
        GM_TRY((lin_fwd<A, EpiStore<float, EPI_ADDEND>, false>(h, x_act, Dp, B, Lx, epi, st)));
      } else {
        EpiStore<A, EPI_ADDEND> epi{enc.hid[0], hid_ld(0), nullptr, pre, (int64_t)enc_l0.out, 1, 1.f};
        GM_TRY((lin_fwd<A, EpiStore<A, EPI_ADDEND>, false>(h, x_act, Dp, B, Lx, epi, st)));
      }
    }
    // p(z|y): one linear K -> 2Z (gmvae.py:243, 321-327).  Issued after encoder_gmm's first layer: in the chained kernel that
    // layer starts on its x segment while the y head is still finishing, and y is complete by the time this thin job runs.
    {
      const Linear& l = h->prior_gmm.layers[0];
      EpiStore<float> epi{prior_out, (int64_t)2 * Z, h->params + l.b_off, nullptr, 0, 0, 1.f};
      GM_TRY(lin_fwd<A>(h, y_act, Kp, B, view(h, l), epi, st));
    }
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder, enc, x_act, Dp, D, B, 1, st));
  } else {
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder, enc, x_act, Dp, D, B, 0, st));
  }
  if (nl > 1 || !gm) {   // last encoder layer -> enc_out (fp32)
    EpiStore<float> epi{enc_out, (int64_t)2 * Z, h->params + enc_last.b_off, nullptr, 0, 0, 1.f};
    GM_TRY(lin_fwd<A>(h, nl == 1 ? x_act : enc.hid[nl - 2], nl == 1 ? Dp : hid_ld(nl - 2), B, view(h, enc_last, 0, nl == 1 ? D : -1),
                      epi, st));
  }
  return 0;
}

template <typename A>
static int forward_backward_body(gmvae_handle* h, const uint8_t* x_u8, int B, int Bg, const float* eps_in, const float* u_in, cudaStream_t st);

// Deterministic mode: the step's final sums in a fixed order (det_reduce_kernel), into the bias entries of the gradient buffer,
// the VAE_GMP prior's gradients and slot 0 of every loss term of the tail -- where the atomics of the default mode put them.
static int det_reduce(gmvae_handle* h, cudaStream_t st) {
  DetSegs segs;
  segs.nseg = (int)h->det_segs.size();
  long long nmax = 1;
  for (int i = 0; i < segs.nseg; ++i) { segs.s[i] = h->det_segs[i]; nmax = std::max(nmax, (long long)segs.s[i].rows * segs.s[i].cols); }
  GM_CHECK_CUDA(launch_k(det_reduce_kernel, dim3((unsigned)std::min(1024LL, (nmax + 255) / 256), segs.nseg), dim3(256), 0, st, true, segs));
  GM_LAUNCHED(h, st, PC_BIAS_GRAD);
  return 0;
}

// Records the tensor-core GEMMs between two head kernels as one chained launch (gemm_chain.cuh).
template <typename A>
static int forward_backward_impl(gmvae_handle* h, const uint8_t* x_u8, int B, int Bg, const float* eps_in,
                                 const float* u_in, cudaStream_t st) {
  h->chain.njobs = 0; h->chain.nmaps = 0; h->chain_tiles = 0; h->chain_writers.clear(); h->chain_counter_next = 0; h->chain_launch_idx = 0;
  h->relu_bits_valid.clear();
  h->chain_counters = h->buf<int>("chain.counters");
  h->chain_on = std::is_same<A, bf16>::value && h->bf16_mode() && h->chain_counters && !(h->debug_flags & (DBG_NO_TC | DBG_NO_CHAIN));
  // Heads as row jobs (one launch for the whole pass) pay off once there are enough 128-row blocks to keep the SMs busy
  // across the dependent thin jobs; below that the heads run as separate kernels between chained launches.
  h->row_jobs = h->chain_on && !(h->debug_flags & DBG_NO_ROW_JOBS) && (B >= 32 * tc::BLOCK_M || (h->debug_flags & DBG_ROW_JOBS));
  // CTA pairs (256-row tiles) where the one-launch plan runs: large batches, every SM available
  h->chain_pair = h->row_jobs && !(h->debug_flags & DBG_NO_PAIR) && !(h->comm && h->world > 1 && h->overlap_comm) && tc::g_reserved_sms == 0;
  h->chain_quad = false;
  // Measured slower than plain pairs so far (0.379 vs 0.348 ms at cfg4: the two pairs of a cluster advance in lock-step through the
  // shared ring slots, and the multicast halves the L2 reads of A but not what each SM receives): opt-in, GMVAE_CHAIN_QUAD=1.
  if (h->chain_pair && h->quad_opt_in && !(h->debug_flags & DBG_NO_QUAD)) {
    // clusters of 4: how many the device can co-schedule (a GPC with an odd number of TPCs leaves one idle); cached per device
    static int max_quads_by_dev[64] = {};
    int& mq = max_quads_by_dev[tc::current_device()];
    if (mq == 0) {
      GM_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_chain_kernel<tc::ChainParams, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::CHAIN_SMEM_BYTES));
      cudaLaunchConfig_t qc = {};
      qc.gridDim = dim3(tc::num_sms() & ~3); qc.blockDim = dim3(tc::NUM_THREADS2); qc.dynamicSmemBytes = tc::CHAIN_SMEM_BYTES;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension; qa[0].val.clusterDim.x = 4; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      qc.attrs = qa; qc.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, tc::gemm_chain_kernel<tc::ChainParams, 4>, &qc) != cudaSuccess) { cudaGetLastError(); n = 0; }
      mq = n > 0 ? std::min(n, tc::num_sms() / 4) : -1;
      if (getenv("GMVAE_VERBOSE")) fprintf(stderr, "[gmvae] 4-CTA clusters of the chained kernel co-resident on this device: %d\n", n);
    }
    h->max_quads = mq;
    h->chain_quad = mq >= 28;                    // fewer than 112 of the SMs in clusters: stay with pairs
  }
  h->part_on = false; h->cur_part = 0; h->part_tail = false; h->part_last_mlp = false;
  h->part_tiles[0] = h->part_tiles[1] = h->part_tiles[2] = 0;
  if (h->chain_pair && !h->chain_quad && !(h->debug_flags & DBG_NO_PARTITION)) {
    int mc = 0;
    GM_TRY(pair_max_clusters(h, &mc));
    const int W = std::min(tc::num_sms() / 2, mc);
    const int split_env = h->chain_split_opt;
    // Measured at cfg4: 0.458 / 0.415 / 0.387 / 0.358 / 0.405 ms with 24 / 30 / 37 / 44 / 52 of the 74 pairs on the chain against 0.354 ms
    // without a partition (the chain's tiles are paced by their epilogues, fewer pairs stretch every stage): off unless asked for.
    const int x = split_env;
    if (x >= 4 && W - x >= 4) { h->part_on = true; h->part_walkers = W; h->part_chain_walkers = x; }
  }
  if (h->chain_on) GM_CHECK_CUDA(cudaMemsetAsync(h->chain_counters, 0, (size_t)h->chain_counter_cap * 4, st));
  int r = forward_backward_body<A>(h, x_u8, B, Bg, eps_in, u_in, st);
  if (r == 0) r = chain_flush(h, st);
  if (h->det) {
    for (auto& f : h->det_colsums) if (r == 0) r = f();
    h->det_colsums.clear();
    if (r == 0) r = det_reduce(h, st);
  }
  h->chain_on = false; h->chain_pair = false; h->chain_quad = false; h->chain.njobs = 0; h->chain.nmaps = 0;
  return r;
}

template <typename A>
static int forward_backward_body(gmvae_handle* h, const uint8_t* x_u8, int B, int Bg, const float* eps_in,
                                 const float* u_in, cudaStream_t st) {
  const gmvae_config& c = h->cfg;
  const int D = h->D, Z = h->Z, K = h->K, nl = h->L;
  const int Dp = ldp(D), Zp = ldp(Z), Z2p = ldp(2 * Z), Kp = ldp(K);
  const float inv_bg = 1.f / (float)Bg;
  const bool gm = c.model == GMVAE_MODEL_GMVAE;
  float* acc = h->grads + h->n_params;
  if (h->profiling) GM_TRY(profile_mark(h, st, PC_START));
  // gradients accumulate (split-K weight gradients, column sums, loss terms): start from zeros -- left behind by the previous
  // training step's Adam kernel, or cleared here
  if (!h->grads_clean) GM_CHECK_CUDA(cudaMemsetAsync(h->grads, 0, (size_t)(h->n_params + ACC_SLOTS) * 4, st));
  h->grads_clean = false;
  h->reduced_upto = 0;
  unsigned long long* fx = h->det ? h->buf<unsigned long long>("det.fx") : nullptr;
  if (h->det) {
    const int nfx = 3 + (c.model == GMVAE_MODEL_VAE_GMP ? K + 2 * K * Z : 0);
    GM_CHECK_CUDA(cudaMemsetAsync(fx, 0, (size_t)nfx * 16, st));
    acc = acc_fixed_tag(fx);
    h->det_segs.clear(); h->det_colsums.clear(); h->det_part_next = 0; h->det_wg_next = 0;
    h->det_segs.push_back(DetSeg{h->grads + h->n_params, nullptr, fx, 0, 3, 1, 0, ACC_PER_TERM, 0, 0});   // slot 0 of each term
    if (c.model == GMVAE_MODEL_VAE_GMP) {   // fx sums 3 ..: [K mixture logits | K*Z loc | K*Z raw_scale_diag] (gmp_prior_kernel)
      h->det_segs.push_back(DetSeg{h->grads + h->mix_off, nullptr, fx + 2 * 3, 0, 1, K, 0, 0, 0, 0});
      h->det_segs.push_back(DetSeg{h->grads + h->loc_off, nullptr, fx + 2 * (3 + K), 0, 1, K * Z, 0, 0, 0, 0});
      h->det_segs.push_back(DetSeg{h->grads + h->raw_scale_off, nullptr, fx + 2 * (3 + K + K * Z), 0, 1, K * Z, 0, 0, 0, 0});
    }
  }

  const float* eps = eps_in; const float* u = u_in;
  GM_TRY(forward_encoder<A>(h, x_u8, B, inv_bg, eps, u, acc, st));

  A* x_act = h->buf<A>("x_act");
  MlpBufs<A> dec = mlp_bufs<A>(h, h->decoder), enc = mlp_bufs<A>(h, h->encoder);
  float* enc_out = h->buf<float>("enc_out");
  A* d_enc_out = h->buf<A>("d_enc_out");
  A* z_act = h->buf<A>("z_act");
  float* dz = h->buf<float>("dz");
  A* dlogits_x = h->buf<A>("dec.dlogits");
  const Linear& enc_l0 = h->encoder.layers[0];
  const Linear& enc_last = h->encoder.layers[nl - 1];
  auto hid_ld = [&](int i) { return (int64_t)ldp(h->hidden[i]); };
  MlpBufs<A> ey; float *logits_y = nullptr, *y_f32 = nullptr, *prior_out = nullptr; A* y_act = nullptr;
  if (gm) {
    ey = mlp_bufs<A>(h, h->encoder_y);
    logits_y = h->buf<float>("logits_y"); y_f32 = h->buf<float>("y_f32"); y_act = h->buf<A>("y_act");
    prior_out = h->buf<float>("prior_out");
  }
  // z head
  const int prior_mode = gm ? 2 : (c.model == GMVAE_MODEL_VAE_GMP ? 1 : 0);
  float* z_f32 = h->buf<float>("z_f32");
  {
    int64_t n = (int64_t)B * Z;
    const bool v4 = std::is_same<A, bf16>::value && Z % 4 == 0 && Z <= 256 && aligned16(eps) && aligned16(enc_out) &&
                    (prior_mode != 2 || aligned16(prior_out));
    const bool rows_ok = h->chain_on && h->row_jobs && v4 && prior_mode != 1 && z_f32 == nullptr;
    if (rows_ok) {
      tc::RowsZFwd prm{enc_out, eps, prior_out, prior_mode, Z, c.raw_sigma_bias, c.sigma_min, inv_bg, reinterpret_cast<bf16*>(z_act), Zp, acc};
      GM_TRY(chain_add_rows(h, tc::EK_ROWS_Z_FWD, prm, B, {enc_out, eps, prior_out}, {{z_act, (size_t)B * Zp * 2}}, st, 4));
    } else {
    GM_TRY(chain_flush(h, st));
    if (v4) {
      const int blocks = (int)std::min<int64_t>((n / 4 + 255) / 256, 8 * tc::num_sms());
      GM_CHECK_CUDA(launch_k(head_z_fwd_v4_kernel, dim3(blocks), dim3(256), 0, st, true, (const float*)enc_out, eps, (const float*)prior_out,
                             prior_mode, B, Z, c.raw_sigma_bias, c.sigma_min, inv_bg, reinterpret_cast<bf16*>(z_act), Zp, z_f32, acc));
    } else {
      GM_CHECK_CUDA(launch_k(head_z_fwd_kernel<A>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, true, (const float*)enc_out, eps,
                             (const float*)prior_out, prior_mode, B, Z, c.raw_sigma_bias, c.sigma_min, inv_bg, z_act, Zp, z_f32, acc));
    }
    GM_LAUNCHED(h, st, PC_HEADS);
    }
  }
  float* dz_prior = h->buf<float>("dz_prior");
  if (prior_mode == 1) {
    const int warps = 4;
    GM_TRY(chain_flush(h, st));
    GM_CHECK_CUDA(launch_k(gmp_prior_kernel, dim3((B + warps - 1) / warps), dim3(warps * 32), warps * K * sizeof(float), st, true,
                           (const float*)z_f32, (const float*)(h->params + h->loc_off), (const float*)(h->params + h->raw_scale_off),
                           (const float*)(h->params + h->mix_off), B, K, Z, inv_bg, dz_prior, h->grads + h->loc_off,
                           h->grads + h->raw_scale_off, h->grads + h->mix_off, acc, fx ? fx + 2 * 3 : nullptr));
    GM_LAUNCHED(h, st, PC_HEADS);
  }
  // decoder: hidden layers, then logits fused with the Bernoulli log-likelihood (and db of that layer)
  bool dec_bias_fused = false;
  GM_TRY(mlp_hidden_fwd<A>(h, h->decoder, dec, z_act, Zp, Z, B, 0, st));
  {
    const Linear& l = h->decoder.layers[nl - 1];
    const A* in = nl == 1 ? z_act : dec.hid[nl - 2];
    const int64_t ldin = nl == 1 ? Zp : hid_ld(nl - 2);
    LinView Ld = view(h, l);
    dec_bias_fused = !(h->debug_flags & DBG_NO_FUSED_COLSUM) && !h->det && tc_ok_fwd<A>(h, in, ldin, Ld);
    EpiBCE<A> epi{dlogits_x, (int64_t)Dp, h->params + l.b_off, c.gen_bias_init, x_u8, (int64_t)D, 1, nullptr, (double*)nullptr,
                  acc, inv_bg, 0.f, dec_bias_fused ? h->grads + l.b_off : nullptr, h->bf16_mode() ? 1 : 0};
    GM_TRY(lin_fwd<A>(h, in, ldin, B, Ld, epi, st));
  }

  // -------------------------------------------------------------------------- backward
  // Order of the jobs: the data gradients form the critical path (each depends on the one before); the weight
  // gradients only read finished tensors, so in the chained kernel they are placed where that path has bubbles:
  // right after the thin jobs (dz, dy, the heads), whose dependants would otherwise wait out a full tile latency.
  const bool spread = h->chain_on && h->row_jobs && !(h->debug_flags & DBG_NO_SPREAD) && !(h->comm && h->world > 1 && h->overlap_comm);
  // In-order CTAs cannot step over a weight-gradient tile (28 k-blocks, 9-15 us, and waiting for a whole batch slice of its operands)
  // to the data-gradient tile behind it: interleaved, every stage of the dependent chain paid for one (20.8 us per stage against 9.3
  // in the forward pass).  In the one-launch plan all weight gradients therefore follow the chain, where nothing waits for them.
  std::vector<std::function<int()>> wg_late;
  struct WgLateGuard { gmvae_handle* h; ~WgLateGuard() { h->wg_late = nullptr; } } wg_late_guard{h};
  if (spread && (h->debug_flags & DBG_WG_LATE)) h->wg_late = &wg_late;
  // Walker partition: from here on the chain jobs are dealt to the first part_chain_walkers CTA pairs and the weight-gradient jobs
  // to the others (the tail after the last data gradient to everybody again).
  struct PartGuard { gmvae_handle* h; ~PartGuard() { h->cur_part = 0; h->part_tail = false; h->part_last_mlp = false; } } part_guard{h};
  if (h->part_on && spread && !h->wg_late) h->cur_part = 1;
  std::vector<std::function<int()>> wg_dec;          // weight gradients of the two lowest decoder layers
  GM_TRY((mlp_backward<A, A>(h, h->decoder, dec, z_act, Zp, Z, dlogits_x, Dp, B, st, dec_bias_fused, 0, spread ? &wg_dec : nullptr,
                             std::min(2, nl - 1))));
  {  // dz = d(first decoder layer input)
    const Linear& l0 = h->decoder.layers[0];
    EpiStore<float> epi{dz, (int64_t)Z, nullptr, nullptr, 0, 0, 1.f};
    if (nl == 1) GM_TRY((lin_dgrad<A>(h, dlogits_x, Dp, B, view(h, l0), epi, st)));
    else GM_TRY((lin_dgrad<A>(h, dec.dhid[0], hid_ld(0), B, view(h, l0), epi, st)));
  }
  size_t wg_dec_next = 0;
  if (wg_dec.size() > 1) GM_TRY(wg_dec[wg_dec_next++]());   // filler between dz and the z head that consumes it
  GM_TRY(comm_bucket(h, st, h->bucket_end[0]));     // decoder gradients are final
  A* d_prior_out = h->buf<A>("d_prior_out");
  bool enc_bias_fused = false;
  {
    int64_t n = (int64_t)B * Z;
    const bool z_cs_ok = Z <= 256 && !(h->debug_flags & DBG_NO_FUSED_COLSUM);
    enc_bias_fused = z_cs_ok && !h->det;         // deterministic mode: the row job / kernel leaves the column sums to bias_grad
    const bool rows_ok = h->chain_on && h->row_jobs && z_cs_ok && prior_mode != 1 &&
                         (Z == 4 || Z == 8 || Z == 16 || Z == 32 || Z == 64) && aligned16(eps) && aligned16(enc_out) && aligned16(dz) &&
                         (prior_mode != 2 || aligned16(prior_out));
    if (rows_ok) {
      tc::RowsZBwd prm{enc_out, eps, prior_out, dz, prior_mode, Z, c.raw_sigma_bias, c.sigma_min, inv_bg, reinterpret_cast<bf16*>(d_enc_out),
                       reinterpret_cast<bf16*>(d_prior_out), Z2p, enc_bias_fused ? h->grads + enc_last.b_off : (float*)nullptr,
                       (gm && enc_bias_fused) ? h->grads + h->prior_gmm.layers[0].b_off : (float*)nullptr};
      GM_TRY(chain_add_rows(h, tc::EK_ROWS_Z_BWD, prm, B, {dz, enc_out, prior_out, eps},
                            {{d_enc_out, (size_t)B * Z2p * 2}, {gm ? d_prior_out : nullptr, (size_t)B * Z2p * 2}}, st, 4));
    } else {
    GM_TRY(chain_flush(h, st));
    const bool v4 = std::is_same<A, bf16>::value && enc_bias_fused && Z % 4 == 0 && aligned16(eps) && aligned16(enc_out) && aligned16(dz) &&
                    (prior_mode != 2 || aligned16(prior_out)) && (prior_mode != 1 || aligned16(dz_prior));
    if (v4) {
      // rows are spread over 4 CTAs per SM: every thread sees 1-2 rows, the column sums cost 4Z atomics per CTA
      const int rpi = 256 / (Z / 4);
      const int blocks = std::max(1, std::min(4 * tc::num_sms(), (B + rpi - 1) / rpi));
      GM_CHECK_CUDA(launch_k(head_z_bwd_v4_kernel, dim3(blocks), dim3(256), (size_t)16 * 256 * sizeof(float), st, true, (const float*)enc_out,
                             eps, (const float*)prior_out, (const float*)dz, (const float*)dz_prior, prior_mode, B, Z, c.raw_sigma_bias,
                             c.sigma_min, inv_bg, reinterpret_cast<bf16*>(d_enc_out), reinterpret_cast<bf16*>(d_prior_out), Z2p,
                             h->grads + enc_last.b_off, gm ? h->grads + h->prior_gmm.layers[0].b_off : (float*)nullptr));
    } else if (enc_bias_fused) {
      // also reduces db of the last encoder layer and of prior_gmm over the batch
      const int lanes = 256 / Z;
      const int blocks = std::max(1, std::min(2 * tc::num_sms(), (B + lanes - 1) / lanes));
      GM_CHECK_CUDA(launch_k(head_z_bwd_cs_kernel<A>, dim3(blocks), dim3(256), 4 * 256 * sizeof(float), st, true, (const float*)enc_out, eps,
                             (const float*)prior_out, (const float*)dz, (const float*)dz_prior, prior_mode, B, Z, c.raw_sigma_bias,
                             c.sigma_min, inv_bg, d_enc_out, d_prior_out, Z2p, h->grads + enc_last.b_off,
                             gm ? h->grads + h->prior_gmm.layers[0].b_off : (float*)nullptr));
    } else {
      GM_CHECK_CUDA(launch_k(head_z_bwd_kernel<A>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, true, (const float*)enc_out, eps,
                             (const float*)prior_out, (const float*)dz, (const float*)dz_prior, prior_mode, B, Z, c.raw_sigma_bias,
                             c.sigma_min, inv_bg, d_enc_out, d_prior_out, Z2p));
    }
    GM_LAUNCHED(h, st, PC_HEADS);
    }
  }
  for (; wg_dec_next < wg_dec.size(); ++wg_dec_next) GM_TRY(wg_dec[wg_dec_next]());   // filler between the z head and the encoder's data gradients
  std::vector<std::function<int()>> wg_enc;          // weight gradient of the encoder's first layer (x part)
  if (!gm) { h->part_last_mlp = true; if (h->encoder.layers.size() < 2) h->part_tail = true; }
  GM_TRY((mlp_backward<A, A>(h, h->encoder, enc, x_act, Dp, D, d_enc_out, Z2p, B, st, enc_bias_fused, 0, (spread && gm) ? &wg_enc : nullptr, 1)));
  if (gm) {
    float* dy = h->buf<float>("dy"); A* dlogits_y = h->buf<A>("dlogits_y");
    LinView Ly = view(h, enc_l0, D, K);
    // y-columns of encoder_gmm layer 0: dW[D:] = y^T dh0 ; dy = dh0 W[D:]^T
    const A* dh0 = nl == 1 ? d_enc_out : enc.dhid[0];
    const int64_t ld_dh0 = nl == 1 ? Z2p : hid_ld(0);
    // dy = dh0 W[D:]^T + d_prior_out Wp^T : two K segments of one data-gradient GEMM (one accumulator)
    const Linear& lp = h->prior_gmm.layers[0];
    LinView Lp = view(h, lp);
    const bool dy_two_seg = tc_ok_dgrad<A>(h, dh0, ld_dh0, Ly) && tc_ok_dgrad<A>(h, d_prior_out, Z2p, Lp) && !(h->debug_flags & DBG_NO_TWO_SEG);
    const bool y_cs_ok = !(h->debug_flags & DBG_NO_FUSED_COLSUM);
    const bool ey_bias_fused = y_cs_ok && !h->det;
    bool yb_fused = false;
    {
      EpiStore<float> e{dy, (int64_t)K, nullptr, nullptr, 0, 0, 1.f};
      if (dy_two_seg && h->chain_on && h->row_jobs && K <= 16 && Kp <= 16 && y_cs_ok && !(h->debug_flags & DBG_NO_FUSE_HEADS)) {
        // the backward of the q(y|x) head runs in the epilogue of the dy GEMM; dy itself never reaches memory
        tc::RowsYBwd prm{logits_y, y_f32, nullptr, K, 1.f / c.temperature, inv_bg, reinterpret_cast<bf16*>(dlogits_y), Kp,
                         ey_bias_fused ? h->grads + h->encoder_y.layers[nl - 1].b_off : (float*)nullptr};
        h->fuse_next = gmvae_handle::FuseReq();
        h->fuse_next.kind = tc::EK_ROWS_Y_BWD;
        memcpy(h->fuse_next.prm, &prm, sizeof(prm));
        h->fuse_next.writes = {{dlogits_y, (size_t)B * Kp * 2}};
      }
      if (dy_two_seg) GM_TRY((lin_dgrad<A>(h, dh0, ld_dh0, B, Ly, e, st, d_prior_out, Z2p, &Lp)));
      else GM_TRY((lin_dgrad<A>(h, dh0, ld_dh0, B, Ly, e, st)));
      yb_fused = h->fuse_next.consumed;
      h->fuse_next = gmvae_handle::FuseReq();
    }
    if (!dy_two_seg) {
      EpiStore<float, EPI_ACCUM> e{dy, (int64_t)K, nullptr, nullptr, 0, 0, 1.f};
      GM_TRY((lin_dgrad<A>(h, d_prior_out, Z2p, B, Lp, e, st)));
    }
    for (auto& f : wg_enc) GM_TRY(f());               // dW[:D] = x^T dh0: filler between dy and the y head that consumes it
    auto wg_y = [&]() -> int {
      GM_TRY((lin_wgrad<A, A>(h, y_act, Kp, dh0, ld_dh0, B, Ly, st)));
      // prior_gmm: dWp = y^T d_prior_out ; dbp
      GM_TRY((lin_wgrad<A, A>(h, y_act, Kp, d_prior_out, Z2p, B, Lp, st)));
      if (!enc_bias_fused) GM_TRY(bias_grad<A>(h, d_prior_out, Z2p, B, 2 * Z, Lp.db, st));
      return 0;
    };
    if (h->wg_late) h->wg_late->push_back(wg_y);
    else if (!spread) GM_TRY(wg_y());
    GM_TRY(comm_bucket(h, st, h->bucket_end[1]));   // encoder_gmm and prior_gmm gradients are final
    if (yb_fused) {
      // dlogits_y and encoder_y's last bias gradient were produced by the dy job
    } else if (h->chain_on && h->row_jobs && K <= 16 && Kp <= 16) {
      tc::RowsYBwd prm{logits_y, y_f32, dy, K, 1.f / c.temperature, inv_bg, reinterpret_cast<bf16*>(dlogits_y), Kp,
                       ey_bias_fused ? h->grads + h->encoder_y.layers[nl - 1].b_off : (float*)nullptr};
      GM_TRY(chain_add_rows(h, tc::EK_ROWS_Y_BWD, prm, B, {dy, logits_y, y_f32}, {{dlogits_y, (size_t)B * Kp * 2}}, st));
    } else {
    GM_TRY(chain_flush(h, st));
    if (std::is_same<A, bf16>::value && K <= 16 && Kp <= 16) {
      GM_CHECK_CUDA(launch_k(head_y_bwd_row_kernel, dim3(std::max(1, std::min(tc::num_sms(), (B + 127) / 128))), dim3(128), 0, st, true,
                             (const float*)logits_y, (const float*)y_f32, (const float*)dy, B, K, 1.f / c.temperature, inv_bg,
                             reinterpret_cast<bf16*>(dlogits_y), Kp, ey_bias_fused ? h->grads + h->encoder_y.layers[nl - 1].b_off : (float*)nullptr));
    } else {
      GM_CHECK_CUDA(launch_k(head_y_bwd_kernel<A>, dim3(std::max(1, std::min(2 * tc::num_sms(), (B + 7) / 8))), dim3(256), 0, st, true,
                             (const float*)logits_y, (const float*)y_f32, (const float*)dy, B, K, 1.f / c.temperature, inv_bg, dlogits_y, Kp,
                             ey_bias_fused ? h->grads + h->encoder_y.layers[nl - 1].b_off : (float*)nullptr));
    }
    GM_LAUNCHED(h, st, PC_HEADS);
    }
    if (spread && !h->wg_late) GM_TRY(wg_y());        // filler between the y head and encoder_y's data gradients
    h->part_last_mlp = true;
    if (h->encoder_y.layers.size() < 2) h->part_tail = true;
    GM_TRY((mlp_backward<A, A>(h, h->encoder_y, ey, x_act, Dp, D, dlogits_y, Kp, B, st, ey_bias_fused)));
    if (h->wg_late) {                                 // (wg_y captures this scope by reference: run here)
      h->wg_late = nullptr;
      for (auto& f : wg_late) GM_TRY(f());
      wg_late.clear();
    }
  }
  if (h->wg_late) {
    h->wg_late = nullptr;
    for (auto& f : wg_late) GM_TRY(f());
  }
  return 0;
}


// ============================================================================ objective M
// K-way marginalised ELBO (north_star (1)-(2); SURVEY.md Appendix A.3):
//   pi = softmax(encoder_y(x));  for every component k (y = e_k):
//     h1_k = relu(x W1[:D] + W1[D+k] + b1)   -- x-projection computed ONCE per sample, broadcast over k
//     (mu_q, s_q)_k = rest of encoder_gmm;  z_k = mu_q + s_q eps_k;  rec_k = log p(x | z_k)
//     KL_k = KL(N(mu_q, s_q) || prior_gmm(e_k))  (analytic)
//   loss = mean_b sum_k pi_k (KL_k - rec_k) + mean_b sum_k pi_k log pi_k
// The per-component rows (r = b*K + k) run through the SAME GEMM kernels as objective R, in
// chunks of whole samples; weight gradients accumulate across chunks in the flat gradient buffer.
template <typename A>
static int forward_backward_marginal(gmvae_handle* h, const uint8_t* x_u8, int B, int Bg, const float* eps_in, cudaStream_t st) {
  const gmvae_config& c = h->cfg;
  const int D = h->D, Z = h->Z, K = h->K, nl = h->L;
  const int Dp = ldp(D), Zp = ldp(Z), Z2p = ldp(2 * Z), Kp = ldp(K);
  const float inv_bg = 1.f / (float)Bg;
  float* acc = h->grads + h->n_params;
  if (h->profiling) GM_TRY(profile_mark(h, st, PC_START));
  if (!h->grads_clean) GM_CHECK_CUDA(cudaMemsetAsync(h->grads, 0, (size_t)(h->n_params + ACC_SLOTS) * 4, st));
  h->grads_clean = false;
  h->reduced_upto = 0;
  double* rec = h->buf<double>("rec"); float* klrow = h->buf<float>("klrow");
  float* tab = h->buf<float>("tab"); float* dtab = h->buf<float>("dtab");
  GM_CHECK_CUDA(cudaMemsetAsync(rec, 0, (size_t)B * K * 8, st));
  GM_CHECK_CUDA(cudaMemsetAsync(dtab, 0, (size_t)K * 2 * Z * 4, st));

  A* x_act = h->buf<A>("x_act");
  {
    const int64_t n = (int64_t)B * D;
    if (D % 16 == 0) GM_CHECK_CUDA(launch_k(convert_x_kernel<A>, dim3((unsigned)((n / 16 + 255) / 256)), dim3(256), 0, st, false, x_u8, x_act, n));
    else GM_CHECK_CUDA(launch_k(convert_x_rows_kernel<A>, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, false, x_u8, x_act, B, D, Dp));
    GM_LAUNCHED(h, st, PC_MISC);
  }
  const float* eps = eps_in;
  if (!eps) {
    float* e = h->buf<float>("eps");
    const int64_t ne = (int64_t)B * K * Z, q = (ne + 3) / 4;
    GM_CHECK_CUDA(launch_k(fill_noise_kernel, dim3((unsigned)((q + 255) / 256)), dim3(256), 0, st, true, e, ne, (float*)nullptr, (int64_t)0,
                           (const DeviceState*)h->state, (uint64_t)h->rank, 0, h->in_train_step ? (uint64_t)0 : ++h->draws));
    GM_LAUNCHED(h, st, PC_MISC);
    eps = e;
  }
  MlpBufs<A> dec = mlp_bufs<A>(h, h->decoder), enc = mlp_bufs<A>(h, h->encoder), ey = mlp_bufs<A>(h, h->encoder_y);
  float* enc_out = h->buf<float>("enc_out"); A* d_enc_out = h->buf<A>("d_enc_out");
  A* z_act = h->buf<A>("z_act"); float* dz = h->buf<float>("dz"); A* dlogits_x = h->buf<A>("dec.dlogits");
  float* logits_y = h->buf<float>("logits_y"); float* pi = h->buf<float>("y_f32"); A* y_act = h->buf<A>("y_act");
  float* xproj = h->buf<float>("xproj"); A* dxproj = h->buf<A>("dxproj"); A* dlogits_y = h->buf<A>("dlogits_y");
  const Linear& enc_l0 = h->encoder.layers[0];
  const Linear& enc_last = h->encoder.layers[nl - 1];
  const Linear& prior = h->prior_gmm.layers[0];
  const int H0 = enc_l0.out, H0p = ldp(H0);
  auto hid_ld = [&](int i) { return (int64_t)ldp(h->hidden[i]); };

  // ---- q(y|x) on the whole batch: pi = softmax(logits), nent
  GM_TRY(mlp_hidden_fwd<A>(h, h->encoder_y, ey, x_act, Dp, D, B, 0, st));
  {
    const Linear& l = h->encoder_y.layers[nl - 1];
    EpiStore<float> epi{logits_y, (int64_t)K, h->params + l.b_off, nullptr, 0, 0, 1.f};
    GM_TRY(lin_fwd<A>(h, ey.hid[nl - 2], hid_ld(nl - 2), B, view(h, l), epi, st));
  }
  GM_CHECK_CUDA(launch_k(head_y_fwd_kernel<A>, dim3((B + 7) / 8), dim3(256), 0, st, true, (const float*)logits_y, (const float*)nullptr, B, K,
                         1.f, inv_bg, pi, y_act, Kp, acc));
  GM_LAUNCHED(h, st, PC_HEADS);
  // ---- prior table p(z | y = e_k), k = 0..K-1
  GM_CHECK_CUDA(launch_k(prior_table_kernel, dim3((K * 2 * Z + 255) / 256), dim3(256), 0, st, true, (const float*)(h->params + prior.w_off),
                         (const float*)(h->params + prior.b_off), K, 2 * Z, tab));
  GM_LAUNCHED(h, st, PC_HEADS);
  // ---- shared x-projection of encoder_gmm layer 0 (no bias, no activation), fp32
  {
    EpiStore<float> epi{xproj, (int64_t)H0, nullptr, nullptr, 0, 0, 1.f};
    GM_TRY(lin_fwd<A>(h, x_act, Dp, B, view(h, enc_l0, 0, D), epi, st));
  }
  const float* Wy = h->params + enc_l0.w_off + (int64_t)D * H0;     // rows D..D+K-1 of W1

  for (int b0 = 0; b0 < B; b0 += h->chunk_samples) {
    const int nb = std::min(h->chunk_samples, B - b0), R = nb * K, row0 = b0 * K;
    // h1 for all components of the chunk
    {
      const int64_t work = (int64_t)R * (H0 / 4);
      GM_REQUIRE(H0 % 4 == 0, "objective=marginal needs hidden sizes that are multiples of 4");
      const int blocks = (int)std::min<int64_t>((work + 255) / 256, 16 * tc::num_sms());
      GM_CHECK_CUDA(launch_k(expand_h1_kernel<A>, dim3(blocks), dim3(256), 0, st, true, (const float*)(xproj + (int64_t)b0 * H0), (int64_t)H0, Wy,
                             (const float*)(h->params + enc_l0.b_off), R, K, H0, enc.hid[0], (int64_t)H0p));
      GM_LAUNCHED(h, st, PC_HEADS);
    }
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder, enc, x_act, Dp, D, R, 1, st));
    {
      EpiStore<float> epi{enc_out, (int64_t)2 * Z, h->params + enc_last.b_off, nullptr, 0, 0, 1.f};
      GM_TRY(lin_fwd<A>(h, enc.hid[nl - 2], hid_ld(nl - 2), R, view(h, enc_last), epi, st));
    }
    GM_CHECK_CUDA(launch_k(head_z_m_fwd_kernel<A>, dim3(std::max(1, std::min(4 * tc::num_sms(), (R + 7) / 8))), dim3(256), 0, st, true,
                           (const float*)enc_out, eps, (const float*)tab, (const float*)pi, row0, R, K, Z, c.raw_sigma_bias, c.sigma_min,
                           inv_bg, z_act, Zp, klrow, acc));
    GM_LAUNCHED(h, st, PC_HEADS);
    // decoder on every component row; Bernoulli log-likelihood weighted by pi, rec[r] kept for d/d pi
    GM_TRY(mlp_hidden_fwd<A>(h, h->decoder, dec, z_act, Zp, Z, R, 0, st));
    bool dec_bias_fused = false;
    {
      const Linear& l = h->decoder.layers[nl - 1];
      LinView Ld = view(h, l);
      dec_bias_fused = !(h->debug_flags & DBG_NO_FUSED_COLSUM) && tc_ok_fwd<A>(h, dec.hid[nl - 2], hid_ld(nl - 2), Ld);
      EpiBCE<A> epi{dlogits_x, (int64_t)Dp, h->params + l.b_off, c.gen_bias_init, x_u8 + (int64_t)b0 * D, (int64_t)D, K, pi + row0, rec + row0,
                    acc, inv_bg, 0.f, dec_bias_fused ? h->grads + l.b_off : nullptr, h->bf16_mode() ? 1 : 0};
      GM_TRY(lin_fwd<A>(h, dec.hid[nl - 2], hid_ld(nl - 2), R, Ld, epi, st));
    }
    GM_TRY((mlp_backward<A, A>(h, h->decoder, dec, z_act, Zp, Z, dlogits_x, Dp, R, st, dec_bias_fused)));
    {
      const Linear& l0 = h->decoder.layers[0];
      EpiStore<float> epi{dz, (int64_t)Z, nullptr, nullptr, 0, 0, 1.f};
      GM_TRY((lin_dgrad<A>(h, dec.dhid[0], hid_ld(0), R, view(h, l0), epi, st)));
    }
    {
      const int lanes = 256 / Z;
      const int blocks = std::max(1, std::min(2 * tc::num_sms(), (R + lanes - 1) / lanes));
      const size_t smem = (size_t)(2 * 256 + K * 2 * Z) * sizeof(float);
      GM_REQUIRE(smem <= 200 * 1024, "objective=marginal: mixture_components * latent_size too large for the prior-table gradient tile");
      static size_t smem_set_by_dev[64] = {};
      size_t& smem_set = smem_set_by_dev[tc::current_device()];
      if (smem > smem_set) {
        GM_CHECK_CUDA(cudaFuncSetAttribute(head_z_m_bwd_kernel<A>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = smem;
      }
      GM_CHECK_CUDA(launch_k(head_z_m_bwd_kernel<A>, dim3(blocks), dim3(256), smem, st, true, (const float*)enc_out, eps, (const float*)tab,
                             (const float*)pi, (const float*)dz, row0, R, K, Z, c.raw_sigma_bias, c.sigma_min, inv_bg, d_enc_out, Z2p,
                             h->grads + enc_last.b_off, dtab));
      GM_LAUNCHED(h, st, PC_HEADS);
    }
    // encoder_gmm layers >= 1 backward (layer 0 is handled through the shared x-projection)
    GM_TRY((mlp_backward<A, A>(h, h->encoder, enc, x_act, Dp, D, d_enc_out, Z2p, R, st, true, 1)));
    {
      const int col_blocks = (H0 + 63) / 64;
      int spb = std::max(4, (nb * col_blocks + 2 * tc::num_sms() - 1) / (2 * tc::num_sms()));
      dim3 grid(col_blocks, (nb + spb - 1) / spb);
      static bool attr_by_dev[64] = {};
      bool& attr = attr_by_dev[tc::current_device()];
      if (!attr) {
        GM_CHECK_CUDA(cudaFuncSetAttribute(reduce_k_kernel<A>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * HEAD_MAXK * 64 * (int)sizeof(float)));
        attr = true;
      }
      GM_CHECK_CUDA(launch_k(reduce_k_kernel<A>, grid, dim3(256), (size_t)4 * K * 64 * sizeof(float), st, true, (const A*)enc.dhid[0], (int64_t)H0p,
                             b0, nb, K, H0, dxproj, (int64_t)H0p, h->grads + enc_l0.w_off + (int64_t)D * H0, h->grads + enc_l0.b_off, spb));
      GM_LAUNCHED(h, st, PC_BIAS_GRAD);
    }
  }
  GM_TRY(comm_bucket(h, st, h->bucket_end[0]));     // decoder gradients are final
  // x-part of encoder_gmm layer 0: dW1[:D] = x^T dxproj over the whole batch
  GM_TRY((lin_wgrad<A, A>(h, x_act, Dp, dxproj, H0p, B, view(h, enc_l0, 0, D), st)));
  GM_CHECK_CUDA(launch_k(prior_table_bwd_kernel, dim3((2 * Z + 127) / 128), dim3(128), 0, st, true, (const float*)dtab, K, 2 * Z,
                         h->grads + prior.w_off, h->grads + prior.b_off));
  GM_LAUNCHED(h, st, PC_HEADS);
  GM_TRY(comm_bucket(h, st, h->bucket_end[1]));     // encoder_gmm and prior_gmm gradients are final
  const bool ey_bias_fused = !(h->debug_flags & DBG_NO_FUSED_COLSUM);
  GM_CHECK_CUDA(launch_k(head_y_m_bwd_kernel<A>, dim3(std::max(1, std::min(2 * tc::num_sms(), (B + 7) / 8))), dim3(256), 0, st, true,
                         (const float*)logits_y, (const float*)pi, (const double*)rec, (const float*)klrow, B, K, inv_bg, dlogits_y, Kp,
                         ey_bias_fused ? h->grads + h->encoder_y.layers[nl - 1].b_off : (float*)nullptr));
  GM_LAUNCHED(h, st, PC_HEADS);
  GM_TRY((mlp_backward<A, A>(h, h->encoder_y, ey, x_act, Dp, D, dlogits_y, Kp, B, st, ey_bias_fused)));
  return 0;
}

// bf16 operand copies of every weight matrix after the parameters were written from outside
// (initialisation, checkpoint restore).  During training the Adam kernel keeps them current itself.
static int refresh_shadows(gmvae_handle* h, cudaStream_t st) {
  if (h->shadow_tiles > 0) {
    GM_CHECK_CUDA(launch_k(refresh_shadows_kernel, dim3(h->shadow_tiles), dim3(32, 8), 0, st, true, (const ShadowEntry*)h->shadow_dev,
                           (int)h->shadow_host.size())); GM_LAUNCHED(h, st, PC_ADAM);
  }
  return 0;
}

// Every entry point that enqueues work makes the handle's device current for the duration of the call and restores the
// caller's afterwards (a process may hold handles on several GPUs).
struct DeviceGuard {
  int prev = -1, want = -1;
  explicit DeviceGuard(const gmvae_handle* h) {
    if (!h) return;
    want = h->cfg.device;
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != want) cudaSetDevice(want);
  }
  ~DeviceGuard() { if (prev >= 0 && prev != want) cudaSetDevice(prev); }
};

static int check_ready(const gmvae_handle* h) {
  GM_REQUIRE(h != nullptr, "null handle");
  GM_REQUIRE(h->params != nullptr, "gmvae_bind has not been called");
  return 0;
}

}  // namespace gmvae

// ================================================================================ C ABI
extern "C" {

const char* gmvae_last_error(void) { return g_last_error.c_str(); }
const char* gmvae_build_info(void) { return "gmvae_b200 sm_100a (tcgen05/TMA bf16 + fp32 SIMT validation) abi=1 " __DATE__ " " __TIME__; }

int gmvae_create(const gmvae_config* cfg, gmvae_handle** out) {
  GM_REQUIRE(cfg && out, "null argument");
  GM_REQUIRE(cfg->abi_version == GMVAE_ABI_VERSION, "ABI version mismatch");
  GM_REQUIRE(cfg->model >= 0 && cfg->model <= 2, "unknown model");
  GM_REQUIRE(cfg->precision == GMVAE_PRECISION_FP32 || cfg->precision == GMVAE_PRECISION_BF16, "unknown precision");
  GM_REQUIRE(cfg->num_hidden >= 0 && cfg->num_hidden <= GMVAE_MAX_HIDDEN_LAYERS, "num_hidden out of range");
  GM_REQUIRE(cfg->data_size > 0 && cfg->latent_size > 0 && cfg->max_batch > 0, "sizes must be positive");
  for (int i = 0; i < cfg->num_hidden; ++i) GM_REQUIRE(cfg->hidden_sizes[i] > 0, "hidden sizes must be positive");
  if (cfg->model != GMVAE_MODEL_VAE)
    GM_REQUIRE(cfg->mixture_components >= 1 && cfg->mixture_components <= HEAD_MAXK, "mixture_components must be in [1,128]");
  GM_REQUIRE(cfg->objective == GMVAE_OBJECTIVE_REFERENCE || cfg->model == GMVAE_MODEL_GMVAE, "objective applies to GMVAE only");
  if (cfg->objective == GMVAE_OBJECTIVE_MARGINAL)
    GM_REQUIRE(cfg->num_hidden >= 1 && cfg->latent_size <= 256, "objective=marginal needs at least one hidden layer and latent_size <= 256");
  GM_REQUIRE(cfg->deterministic == 0 || cfg->deterministic == 1, "deterministic must be 0 or 1");
  if (cfg->deterministic) {
    GM_REQUIRE(cfg->objective == GMVAE_OBJECTIVE_REFERENCE, "deterministic mode supports objective=reference only");
    // the opt-in launch plans are not covered by the guarantee
    for (const char* v : {"GMVAE_DEBUG_FLAGS", "GMVAE_CHAIN_SPLIT", "GMVAE_CHAIN_QUAD"}) {
      const char* e = getenv(v);
      GM_REQUIRE(!e || atoi(e) == 0, std::string("deterministic mode cannot be combined with ") + v);
    }
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error("no CUDA device: libgmvae_b200 has no CPU fallback");
    return -4;
  }
  GM_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "device ordinal out of range");
  cudaDeviceProp prop;
  GM_CHECK_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  GM_REQUIRE(prop.major == 10, "libgmvae_b200 is built for sm_100a (B200) only");
  gmvae_handle* h = new gmvae_handle();
  h->cfg = *cfg;
  DeviceGuard dev_guard(h);
  const char* dbg = getenv("GMVAE_DEBUG_FLAGS");
  h->debug_flags = dbg ? atoi(dbg) : 0;
  h->det = cfg->deterministic == 1;
  g_use_pdl = !(h->debug_flags & DBG_NO_PDL);
  if (const char* q = getenv("GMVAE_CHAIN_QUAD")) h->quad_opt_in = atoi(q) != 0;
  if (const char* q = getenv("GMVAE_CHAIN_SPLIT")) h->chain_split_opt = atoi(q);
  if (const char* bnv = getenv("GMVAE_CHAIN_BN")) { const int v = atoi(bnv); if (v == 128 || v == 192) h->wide_bn = v; }
  plan(h);
  GM_CHECK_CUDA(cudaMalloc(&h->state, sizeof(DeviceState)));
  DeviceState s0; s0.step = 0; s0.seed = 0x243F6A8885A308D3ull; s0.adam_blocks = 0; s0.pad = 0; s0.beta1_power = 1.0; s0.beta2_power = 1.0;
  h->seed_host = s0.seed;
  GM_CHECK_CUDA(cudaMemcpy(h->state, &s0, sizeof(s0), cudaMemcpyHostToDevice));
  *out = h;
  return 0;
}

void gmvae_destroy(gmvae_handle* h) {
  if (!h) return;
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  for (void* m : h->peer_mapped) if (m) cudaIpcCloseMemHandle(m);
  if (h->peer_region) cudaFree(h->peer_region);
  if (h->comm) ncclCommDestroy(h->comm);
  if (h->comm_stream) cudaStreamDestroy(h->comm_stream);
  for (auto& e : h->comm_ev) if (e) cudaEventDestroy(e);
  if (h->shadow_dev) cudaFree(h->shadow_dev);
  if (h->state) cudaFree(h->state);
  delete h;
}

int64_t gmvae_param_count(const gmvae_handle* h) { return h ? h->n_params : -1; }
int64_t gmvae_grad_count(const gmvae_handle* h) { return h ? h->n_params + ACC_SLOTS : -1; }
int gmvae_num_params(const gmvae_handle* h) { return h ? (int)h->table.size() : -1; }
int gmvae_param_table(const gmvae_handle* h, gmvae_param_desc* out, int cap) {
  GM_REQUIRE(h && out, "null argument");
  int n = std::min(cap, (int)h->table.size());
  for (int i = 0; i < n; ++i) out[i] = h->table[i];
  return n;
}
size_t gmvae_workspace_bytes(const gmvae_handle* h) { return h ? h->ws_needed : 0; }
int64_t gmvae_launch_count(const gmvae_handle* h) { return h ? h->launches : -1; }

int gmvae_bind(gmvae_handle* h, float* params, float* grads, float* adam_m, float* adam_v, void* workspace, size_t workspace_bytes) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && params && grads && adam_m && adam_v && workspace, "null argument");
  GM_REQUIRE(workspace_bytes >= h->ws_needed, "workspace too small");
  GM_REQUIRE(aligned16(params) && aligned16(grads) && aligned16(adam_m) && aligned16(adam_v), "buffers must be 16-byte aligned");
  GM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "workspace must be 256-byte aligned");
  GM_REQUIRE(!h->peer_ready, "gmvae_bind after gmvae_peer_attach is not supported");
  h->params = params; h->grads = grads; h->grads_bound = grads; h->adam_m = adam_m; h->adam_v = adam_v;
  h->ws = reinterpret_cast<uint8_t*>(workspace); h->ws_bytes = workspace_bytes;
  h->shadow_host.clear(); h->shadow_tiles = 0;
  if (h->bf16_mode()) {
    Mlp* mlps[4] = {&h->decoder, &h->encoder, &h->encoder_y, &h->prior_gmm};
    for (Mlp* m : mlps)
      for (auto& l : m->layers) {
        l.w_bf16 = h->buf<bf16>("shadow.w." + std::to_string(l.w_off));
        ShadowEntry e;
        e.w = params + l.w_off; e.w_bf16 = l.w_bf16;
        e.off = l.w_off; e.rows = l.in; e.cols = l.out; e.ld_w = l.ld_w;
        e.tiles_x = (l.ld_w + 31) / 32;
        int tiles_y = (l.in + 31) / 32;
        e.tile_begin = h->shadow_tiles;
        h->shadow_tiles += e.tiles_x * tiles_y;
        h->shadow_host.push_back(e);
      }
    // sorted by flat offset: the Adam kernel finds the matrix an element belongs to by bisection
    std::sort(h->shadow_host.begin(), h->shadow_host.end(), [](const ShadowEntry& a, const ShadowEntry& b) { return a.off < b.off; });
    h->shadow_tiles = 0;
    for (auto& e : h->shadow_host) { e.tile_begin = h->shadow_tiles; h->shadow_tiles += e.tiles_x * ((e.rows + 31) / 32); }
    if (h->shadow_dev) cudaFree(h->shadow_dev);
    GM_CHECK_CUDA(cudaMalloc(&h->shadow_dev, sizeof(ShadowEntry) * h->shadow_host.size()));
    GM_CHECK_CUDA(cudaMemcpy(h->shadow_dev, h->shadow_host.data(), sizeof(ShadowEntry) * h->shadow_host.size(), cudaMemcpyHostToDevice));
  }
  return 0;
}

int gmvae_params_updated(gmvae_handle* h, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  return refresh_shadows(h, (cudaStream_t)stream);
}

int gmvae_forward_backward(gmvae_handle* h, const uint8_t* x_u8, int batch, int global_batch, const float* eps,
                           const float* gumbel_u, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  GM_REQUIRE(x_u8 != nullptr, "null input");
  GM_REQUIRE(batch > 0 && batch <= h->cfg.max_batch, "batch must be in [1, max_batch]");
  GM_REQUIRE(global_batch >= batch, "global_batch must be >= batch");
  GM_REQUIRE(aligned16(x_u8), "x must be 16-byte aligned");
  if (h->cfg.objective == GMVAE_OBJECTIVE_MARGINAL) {
    if (h->bf16_mode()) return forward_backward_marginal<bf16>(h, x_u8, batch, global_batch, eps, (cudaStream_t)stream);
    return forward_backward_marginal<float>(h, x_u8, batch, global_batch, eps, (cudaStream_t)stream);
  }
  if (h->bf16_mode()) return forward_backward_impl<bf16>(h, x_u8, batch, global_batch, eps, gumbel_u, (cudaStream_t)stream);
  return forward_backward_impl<float>(h, x_u8, batch, global_batch, eps, gumbel_u, (cudaStream_t)stream);
}

int gmvae_finalize_loss(gmvae_handle* h, float* loss_terms, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  GM_REQUIRE(loss_terms != nullptr, "null loss_terms");
  GM_CHECK_CUDA(launch_k(finalize_loss_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream, false, (const float*)(h->grads + h->n_params), loss_terms)); GM_LAUNCHED(h, (cudaStream_t)stream, PC_MISC);
  return 0;
}

// Adam (+ optionally the loss-term finalisation, folded into the same launch by gmvae_train_step)
static int adam_step_impl(gmvae_handle* h, float* loss_terms, cudaStream_t st, bool zero_grads, bool fused_exchange = false) {
  const gmvae_config& c = h->cfg;
  int64_t n = h->n_params;
  // after a cross-stream join (data-parallel all-reduce) the kernel is launched with a full dependency
  const bool pdl = !(h->comm && h->world > 1 && (h->debug_flags & DBG_COMM_OVERLAP));
  // one launch: parameter update, the bf16 operand copies of the weight matrices, global_step += 1, (training step) gradients cleared
  const int64_t per_block = (int64_t)ADAM_THREADS * 4 * ADAM_VEC;
  AdamPeer ap = {nullptr, nullptr, nullptr, 0, 0};
  float* g_src = h->grads;
  if (fused_exchange) {
    // last phase of the peer-memory all-reduce (peer.cuh): read the reduced gradients the shard owners pushed into this rank's
    // `red` buffer once all of them have landed, clear this rank's own gradient buffer
    const peer::Layout& L = h->peer_layout;
    char* base = static_cast<char*>(h->peer_region);
    g_src = reinterpret_cast<float*>(base + L.red_off);
    ap.flags = reinterpret_cast<const unsigned long long*>(base + L.flags_off) + peer::MAX_WORLD;
    ap.epoch = &reinterpret_cast<peer::Local*>(base + L.local_off)->epoch;
    ap.own_grads = h->grads; ap.world = L.world; ap.timeout_cycles = h->peer_timeout_cycles;
    zero_grads = true;
  }
  GM_CHECK_CUDA(launch_k(adam_kernel, dim3((unsigned)((n + per_block - 1) / per_block)), dim3(ADAM_THREADS), 0, st, pdl && !fused_exchange, h->params, g_src,
                         h->adam_m, h->adam_v, n, c.learning_rate, c.beta1, c.beta2, c.epsilon, h->state,
                         g_src + h->n_params, loss_terms, (const ShadowEntry*)h->shadow_dev,
                         h->bf16_mode() ? (int)h->shadow_host.size() : 0, zero_grads ? 1 : 0, ap));
  GM_LAUNCHED(h, st, PC_ADAM);
  h->grads_clean = zero_grads;
  return 0;
}

int gmvae_adam_step(gmvae_handle* h, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  return adam_step_impl(h, nullptr, (cudaStream_t)stream, false);     // stand-alone: the gradients stay readable
}

int gmvae_get_step(gmvae_handle* h, int64_t* step, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && step, "null argument");
  DeviceState s;
  GM_CHECK_CUDA(cudaMemcpyAsync(&s, h->state, sizeof(s), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  GM_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  *step = s.step;
  return 0;
}
int gmvae_set_step(gmvae_handle* h, int64_t step, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h, "null argument");
  long long v = step;
  const double pw[2] = {pow((double)h->cfg.beta1, (double)step), pow((double)h->cfg.beta2, (double)step)};   // the beta-power accumulators follow the step
  GM_CHECK_CUDA(cudaMemcpyAsync(&h->state->step, &v, sizeof(v), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  GM_CHECK_CUDA(cudaMemcpyAsync(&h->state->beta1_power, pw, sizeof(pw), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  GM_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}
int gmvae_set_seed(gmvae_handle* h, uint64_t seed) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h, "null argument");
  unsigned long long v = seed;
  GM_CHECK_CUDA(cudaMemcpy(&h->state->seed, &v, sizeof(v), cudaMemcpyHostToDevice));
  h->seed_host = seed;
  return 0;
}

int gmvae_nccl_unique_id(char out[128]) {
  GM_REQUIRE(out, "null argument");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  ncclUniqueId id;
  ncclResult_t r = ncclGetUniqueId(&id);
  if (r != ncclSuccess) { set_error(std::string("ncclGetUniqueId: ") + ncclGetErrorString(r)); return -5; }
  memcpy(out, &id, 128);
  return 0;
}
int gmvae_nccl_init(gmvae_handle* h, const char id[128], int world_size, int rank) {
  GM_REQUIRE(h && id, "null argument");
  GM_REQUIRE(world_size >= 1 && rank >= 0 && rank < world_size, "bad world_size / rank");
  ncclUniqueId uid; memcpy(&uid, id, 128);
  GM_CHECK_CUDA(cudaSetDevice(h->cfg.device));
  // The persistent GEMM kernels occupy every SM they are given (one ~210 KB CTA each), which would
  // starve the all-reduce running on the side stream.  Under data parallelism a few SMs are left to
  // NCCL and NCCL is told to use no more channels (= CTAs) than that.
  if (world_size > 1 && (h->debug_flags & DBG_COMM_OVERLAP)) {
    const char* env = getenv("GMVAE_COMM_SMS");
    int reserve = env ? atoi(env) : 8;
    tc::g_reserved_sms = std::max(0, std::min(64, reserve));
    if (tc::g_reserved_sms > 0) {
      std::string v = std::to_string(tc::g_reserved_sms);
      setenv("NCCL_MAX_NCHANNELS", v.c_str(), 0);
      setenv("NCCL_MAX_CTAS", v.c_str(), 0);
    }
  }
  ncclResult_t r = ncclCommInitRank(&h->comm, world_size, uid, rank);
  if (r != ncclSuccess) { set_error(std::string("ncclCommInitRank: ") + ncclGetErrorString(r)); return -5; }
  h->world = world_size; h->rank = rank;
  GM_CHECK_CUDA(cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking));
  for (auto& e : h->comm_ev) GM_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return 0;
}
// ---- the exchange step over NVLink peer memory (peer.cuh).  export: allocate this rank's symmetric region (gradient buffer,
// reduced-gradient buffer, flags) and hand out its cudaIpc handle; attach: map every rank's region (handles in rank order, own
// included) and MOVE the handle's gradient buffer into the region (gmvae_peer_grads returns it; the caller's buffer is no longer
// used).  The caller puts a barrier between attach and the first step.
int gmvae_peer_export(gmvae_handle* h, int world_size, int rank, char out[64]) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && out, "null argument");
  GM_TRY(check_ready(h));
  GM_REQUIRE(world_size >= 2 && world_size <= peer::MAX_WORLD && rank >= 0 && rank < world_size, "bad world_size / rank");
  GM_REQUIRE(!h->peer_region, "peer region already exported");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
  const int64_t total = h->n_params + ACC_SLOTS;
  GM_REQUIRE(total % 4 == 0, "gradient buffer length must be a multiple of 4 floats");
  h->peer_layout = peer::make_layout(world_size, total);
  GM_CHECK_CUDA(cudaMalloc(&h->peer_region, h->peer_layout.bytes));
  GM_CHECK_CUDA(cudaMemset(h->peer_region, 0, h->peer_layout.bytes));
  GM_CHECK_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t ipc;
  GM_CHECK_CUDA(cudaIpcGetMemHandle(&ipc, h->peer_region));
  memcpy(out, &ipc, 64);
  if (h->world == 1) { h->world = world_size; h->rank = rank; }
  GM_REQUIRE(h->world == world_size && h->rank == rank, "world_size / rank differ from the NCCL communicator's");
  return 0;
}
int gmvae_peer_attach(gmvae_handle* h, const char* handles) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && handles, "null argument");
  GM_REQUIRE(h->peer_region && !h->peer_ready, "call gmvae_peer_export first (once)");
  const peer::Layout& L = h->peer_layout;
  for (int r = 0; r < L.world; ++r) {
    void* base = h->peer_region;
    if (r != h->rank) {
      cudaIpcMemHandle_t ipc;
      memcpy(&ipc, handles + 64 * r, 64);
      GM_CHECK_CUDA(cudaIpcOpenMemHandle(&base, ipc, cudaIpcMemLazyEnablePeerAccess));
      h->peer_mapped[r] = base;
    }
    char* b = static_cast<char*>(base);
    h->peer_ptrs.grad[r] = reinterpret_cast<float4*>(b + L.grad_off);
    h->peer_ptrs.red[r] = reinterpret_cast<float4*>(b + L.red_off);
    h->peer_ptrs.flags[r] = reinterpret_cast<unsigned long long*>(b + L.flags_off);
  }
  const char* ts = getenv("GMVAE_PEER_TIMEOUT_S");
  const double secs = ts ? std::max(1.0, atof(ts)) : 120.0;
  int khz = 0;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->cfg.device);
  h->peer_timeout_cycles = (long long)(secs * 1e3 * (double)std::max(khz, 1000000));
  // the backward pass now accumulates straight into the symmetric region (zero from the memset at export)
  h->grads_bound = h->grads;
  h->grads = reinterpret_cast<float*>(static_cast<char*>(h->peer_region) + L.grad_off);
  h->grads_clean = true;
  if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }   // captured with the old pointers
  h->peer_ready = true;
  return 0;
}
// The gradient buffer after gmvae_peer_attach (float[grad_count] inside the symmetric region), or the bound one.
float* gmvae_peer_grads(gmvae_handle* h) { return h ? h->grads : nullptr; }

static int peer_exchange(gmvae_handle* h, cudaStream_t st) {
  const peer::Layout& L = h->peer_layout;
  peer::Local* loc = reinterpret_cast<peer::Local*>(static_cast<char*>(h->peer_region) + L.local_off);
  const int per_block = peer::exchange_block_items(L.world);
  const unsigned blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>((L.cap4 + per_block - 1) / per_block, 8 * tc::num_sms()));
  auto kern = L.world == 2 ? peer::exchange_kernel<2> : L.world == 4 ? peer::exchange_kernel<4> : L.world == 8 ? peer::exchange_kernel<8>
            : L.world == 16 ? peer::exchange_kernel<16> : peer::exchange_kernel<0>;
  GM_CHECK_CUDA(launch_k(kern, dim3(blocks), dim3(peer::THREADS), 0, st, false, L, h->rank, h->peer_ptrs, loc, h->peer_timeout_cycles));
  GM_LAUNCHED(h, st, PC_COMM);
  return 0;
}

int gmvae_allreduce_grads(gmvae_handle* h, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  if (h->peer_ready && h->world > 1) {
    // stand-alone form: exchange, then the reduced gradients are copied back over this rank's gradient buffer
    GM_TRY(peer_exchange(h, (cudaStream_t)stream));
    const peer::Layout& L = h->peer_layout;
    peer::Local* loc = reinterpret_cast<peer::Local*>(static_cast<char*>(h->peer_region) + L.local_off);
    const unsigned blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>((L.n4 + peer::THREADS - 1) / peer::THREADS, 4 * tc::num_sms()));
    GM_CHECK_CUDA(launch_k(peer::gather_kernel, dim3(blocks), dim3(peer::THREADS), 0, (cudaStream_t)stream, false, L, h->rank, h->peer_ptrs, loc,
                           h->peer_timeout_cycles));
    GM_LAUNCHED(h, (cudaStream_t)stream, PC_COMM);
    return 0;
  }
  if (!h->comm || h->world == 1) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = h->n_params + ACC_SLOTS;
  if (h->overlap_comm) {
    // the buckets issued during the backward pass cover [0, reduced_upto); finish the rest on the
    // side stream and join it back into the caller's stream
    GM_TRY(comm_bucket(h, st, total));
    cudaEvent_t ev = h->comm_ev[h->comm_ev_next++ % 8];
    GM_CHECK_CUDA(cudaEventRecord(ev, h->comm_stream));
    GM_CHECK_CUDA(cudaStreamWaitEvent(st, ev, 0));
    return 0;
  }
  ncclResult_t r = ncclAllReduce(h->grads, h->grads, (size_t)total, ncclFloat, ncclSum, h->comm, st);
  if (r != ncclSuccess) { set_error(std::string("ncclAllReduce: ") + ncclGetErrorString(r)); return -5; }
  GM_LAUNCHED(h, st, PC_COMM);                               // the exchange step is in-stream: its interval is the exposed communication
  return 0;
}

int gmvae_train_step(gmvae_handle* h, const uint8_t* x_u8, int batch, int global_batch, const float* eps, const float* gumbel_u,
                     float* loss_terms, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h != nullptr, "null handle");
  h->overlap_comm = h->comm != nullptr && h->world > 1 && (h->debug_flags & DBG_COMM_OVERLAP);
  h->in_train_step = true;
  int r = gmvae_forward_backward(h, x_u8, batch, global_batch, eps, gumbel_u, stream);
  h->in_train_step = false;
  const bool fused = h->peer_ready && h->world > 1;             // exchange kernel + Adam as the all-reduce's last phase (peer.cuh)
  if (r == 0) r = fused ? peer_exchange(h, (cudaStream_t)stream) : gmvae_allreduce_grads(h, stream);
  h->overlap_comm = false;
  GM_TRY(r);
  return adam_step_impl(h, loss_terms, (cudaStream_t)stream, true, fused);
}

int gmvae_step_graph_capture(gmvae_handle* h, const uint8_t* x_u8, int batch, int global_batch, const float* eps,
                             const float* gumbel_u, float* loss_terms, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  cudaStream_t st = (cudaStream_t)stream;
  GM_REQUIRE(st != nullptr, "graph capture needs a non-default stream");
  if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
  // Warm every kernel once outside capture (function attributes, tensor-map cache, lazy module load).
  int saved = h->debug_flags; h->debug_flags &= ~DBG_SYNC_EACH;
  h->graph_has_memset = !h->grads_clean;                     // the step clears the gradients itself only when they are not already zero
  GM_CHECK_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  int r = gmvae_train_step(h, x_u8, batch, global_batch, eps, gumbel_u, loss_terms, stream);
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(st, &graph);
  h->debug_flags = saved;
  if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
  GM_CHECK_CUDA(e);
  // nothing ran during capture: the buffer is in the state it was in before
  h->grads_clean = !h->graph_has_memset;
  e = cudaGraphInstantiate(&h->graph_exec, graph, 0);
  cudaGraphDestroy(graph);
  GM_CHECK_CUDA(e);
  return 0;
}
int gmvae_step_graph_launch(gmvae_handle* h, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && h->graph_exec, "no captured graph");
  // a graph captured without the clearing memset relies on the previous step's Adam kernel; after an eager forward_backward in
  // between the gradients are cleared here
  if (!h->graph_has_memset && !h->grads_clean)
    GM_CHECK_CUDA(cudaMemsetAsync(h->grads, 0, (size_t)(h->n_params + ACC_SLOTS) * 4, (cudaStream_t)stream));
  GM_CHECK_CUDA(cudaGraphLaunch(h->graph_exec, (cudaStream_t)stream));
  h->grads_clean = true;
  return 0;
}

}  // extern "C"

template <typename A>
static int encode_impl(gmvae_handle* h, const uint8_t* x_u8, int B, const float* eps, const float* u, float* logits_y_out, float* z_mean,
                       float* z_sample, cudaStream_t st) {
  const int Z = h->Z, K = h->K;
  float* acc = h->buf<float>("infer.acc");
  GM_CHECK_CUDA(cudaMemsetAsync(acc, 0, ACC_SLOTS * 4, st));
  GM_TRY(forward_encoder<A>(h, x_u8, B, 1.f / (float)B, eps, u, acc, st));
  if (logits_y_out && h->cfg.model == GMVAE_MODEL_GMVAE)
    GM_CHECK_CUDA(cudaMemcpyAsync(logits_y_out, h->buf<float>("logits_y"), (size_t)B * K * 4, cudaMemcpyDeviceToDevice, st));
  const int64_t n = (int64_t)B * Z;
  GM_CHECK_CUDA(launch_k(encode_out_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, st, false, (const float*)h->buf<float>("enc_out"), eps, B, Z,
                         h->cfg.raw_sigma_bias, h->cfg.sigma_min, z_mean, z_sample));
  GM_LAUNCHED(h, st, PC_HEADS);
  return 0;
}

template <typename A>
static int decode_impl(gmvae_handle* h, const float* z, int n, float* x_mean, cudaStream_t st) {
  const int D = h->D, Z = h->Z, nl = h->L, Zp = ldp(Z);
  A* z_act = h->buf<A>("z_act");
  MlpBufs<A> dec = mlp_bufs<A>(h, h->decoder);
  const int64_t cnt = (int64_t)n * Z;
  GM_CHECK_CUDA(launch_k(to_act_kernel<A>, dim3((unsigned)((cnt + 255) / 256)), dim3(256), 0, st, false, z, n, Z, z_act, Zp));
  GM_LAUNCHED(h, st, PC_MISC);
  GM_TRY(mlp_hidden_fwd<A>(h, h->decoder, dec, z_act, Zp, Z, n, 0, st));
  const Linear& l = h->decoder.layers[nl - 1];
  // Bernoulli mean = sigmoid(logits), logits = MLP(z) + gen_bias_init (base.py:135,138-146)
  EpiStore<float> epi{x_mean, (int64_t)D, h->params + l.b_off, nullptr, 0, 2, 1.f, h->cfg.gen_bias_init};
  GM_TRY(lin_fwd<A>(h, nl == 1 ? z_act : dec.hid[nl - 2], nl == 1 ? (int64_t)Zp : (int64_t)ldp(h->hidden[nl - 2]), n, view(h, l), epi, st));
  return 0;
}

// ConditionalNormal / ConditionalBernoulli / ConditionalCategorical .condition(tensor_list) (base.py:63-72, 130-135, 193-198):
// concat(inputs) -> MLP -> distribution parameters, on caller tensors, through the same GEMM kernels as the step.
template <typename A>
static int condition_impl(gmvae_handle* h, int which, const float* in1, const float* in2, int n, float* out_a, float* out_b, cudaStream_t st) {
  const gmvae_config& c = h->cfg;
  const int D = h->D, Z = h->Z, K = h->K, nl = h->L;
  const int Dp = ldp(D), Zp = ldp(Z), Kp = ldp(K);
  const bool gm = c.model == GMVAE_MODEL_GMVAE;
  auto hid_ld = [&](int i) { return (int64_t)ldp(h->hidden[i]); };
  auto to_act = [&](const float* src, int cols, A* dst, int ld) -> int {
    const int64_t cnt = (int64_t)n * cols;
    GM_CHECK_CUDA(launch_k(to_act_kernel<A>, dim3((unsigned)((cnt + 255) / 256)), dim3(256), 0, st, false, src, n, cols, dst, ld));
    GM_LAUNCHED(h, st, PC_MISC);
    return 0;
  };
  auto normal_out = [&](const float* outs) -> int {
    const int64_t cnt = (int64_t)n * Z;
    GM_CHECK_CUDA(launch_k(normal_params_kernel, dim3((unsigned)((cnt + 255) / 256)), dim3(256), 0, st, true, outs, n, Z, c.raw_sigma_bias,
                           c.sigma_min, out_a, out_b));
    GM_LAUNCHED(h, st, PC_HEADS);
    return 0;
  };
  // last layer of an MLP into an fp32 matrix
  auto last_layer = [&](const Mlp& m, const MlpBufs<A>& b, const A* in0, int64_t ld0, int in0_cols, float* out, int out_cols) -> int {
    const Linear& l = m.layers[nl - 1];
    EpiStore<float> epi{out, (int64_t)out_cols, h->params + l.b_off, nullptr, 0, 0, 1.f};
    return lin_fwd<A>(h, nl == 1 ? in0 : b.hid[nl - 2], nl == 1 ? ld0 : hid_ld(nl - 2), n, view(h, l, 0, nl == 1 ? in0_cols : -1), epi, st);
  };
  if (which == GMVAE_COND_DECODER) {                          // logits = MLP(z) + bias_init
    A* z_act = h->buf<A>("z_act");
    MlpBufs<A> dec = mlp_bufs<A>(h, h->decoder);
    GM_TRY(to_act(in1, Z, z_act, Zp));
    GM_TRY(mlp_hidden_fwd<A>(h, h->decoder, dec, z_act, Zp, Z, n, 0, st));
    GM_TRY(last_layer(h->decoder, dec, z_act, Zp, Z, out_a, D));
    if (c.gen_bias_init != 0.f) {
      const int64_t cnt = (int64_t)n * D;
      GM_CHECK_CUDA(launch_k(add_scalar_kernel, dim3((unsigned)((cnt + 255) / 256)), dim3(256), 0, st, true, out_a, cnt, c.gen_bias_init));
      GM_LAUNCHED(h, st, PC_MISC);
    }
    return 0;
  }
  A* x_act = h->buf<A>("x_act");
  if (which == GMVAE_COND_ENCODER_Y) {                        // logits of q(y|x)
    GM_REQUIRE(gm, "encoder_y exists in the GMVAE only");
    MlpBufs<A> ey = mlp_bufs<A>(h, h->encoder_y);
    GM_TRY(to_act(in1, D, x_act, Dp));
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder_y, ey, x_act, Dp, D, n, 0, st));
    return last_layer(h->encoder_y, ey, x_act, Dp, D, out_a, K);
  }
  if (which == GMVAE_COND_PRIOR_GMM) {                        // p(z|y): one linear K -> 2Z
    GM_REQUIRE(gm, "prior_gmm exists in the GMVAE only");
    A* y_act = h->buf<A>("y_act"); float* prior_out = h->buf<float>("prior_out");
    GM_REQUIRE(prior_out != nullptr, "gmvae_condition(prior_gmm) needs a handle created with objective=reference");
    GM_TRY(to_act(in1, K, y_act, Kp));
    const Linear& l = h->prior_gmm.layers[0];
    EpiStore<float> epi{prior_out, (int64_t)2 * Z, h->params + l.b_off, nullptr, 0, 0, 1.f};
    GM_TRY(lin_fwd<A>(h, y_act, Kp, n, view(h, l), epi, st));
    return normal_out(prior_out);
  }
  GM_REQUIRE(which == GMVAE_COND_ENCODER, "unknown conditional distribution");
  MlpBufs<A> enc = mlp_bufs<A>(h, h->encoder);
  float* enc_out = h->buf<float>("enc_out");
  GM_TRY(to_act(in1, D, x_act, Dp));
  if (!gm) {                                                  // q(z|x)
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder, enc, x_act, Dp, D, n, 0, st));
    GM_TRY(last_layer(h->encoder, enc, x_act, Dp, D, enc_out, 2 * Z));
    return normal_out(enc_out);
  }
  // q(z|x,y): [x,y] W = x W[:D] + y W[D:]  (no concat, base.py:66)
  GM_REQUIRE(in2 != nullptr, "encoder_gmm takes (x, y)");
  GM_REQUIRE(c.objective == GMVAE_OBJECTIVE_REFERENCE, "gmvae_condition(encoder_gmm) needs a handle created with objective=reference");
  A* y_act = h->buf<A>("y_act");
  GM_TRY(to_act(in2, K, y_act, Kp));
  const Linear& enc_l0 = h->encoder.layers[0];
  LinView Lx = view(h, enc_l0, 0, D), Ly = view(h, enc_l0, D, K);
  const bool last0 = nl == 1;
  const bool two_seg = tc_ok_fwd<A>(h, x_act, Dp, Lx) && tc_ok_fwd<A>(h, y_act, Kp, Ly) && !(h->debug_flags & DBG_NO_TWO_SEG);
  if (two_seg) {
    if (last0) {
      EpiStore<float> epi{enc_out, (int64_t)2 * Z, Lx.b, nullptr, 0, 0, 1.f};
      GM_TRY(lin_fwd<A>(h, x_act, Dp, n, Lx, epi, st, y_act, Kp, &Ly));
    } else {
      EpiStore<A> epi{enc.hid[0], hid_ld(0), Lx.b, nullptr, 0, 1, 1.f};
      GM_TRY(lin_fwd<A>(h, x_act, Dp, n, Lx, epi, st, y_act, Kp, &Ly));
    }
  } else {
    float* pre = h->buf<float>("pre_y");
    EpiStore<float> e0{pre, (int64_t)enc_l0.out, Lx.b, nullptr, 0, 0, 1.f};
    GM_TRY((lin_fwd<A, EpiStore<float>, false>(h, y_act, Kp, n, Ly, e0, st)));
    if (last0) {
      EpiStore<float, EPI_ADDEND> epi{enc_out, (int64_t)2 * Z, nullptr, pre, (int64_t)enc_l0.out, 0, 1.f};
      GM_TRY((lin_fwd<A, EpiStore<float, EPI_ADDEND>, false>(h, x_act, Dp, n, Lx, epi, st)));
    } else {
      EpiStore<A, EPI_ADDEND> epi{enc.hid[0], hid_ld(0), nullptr, pre, (int64_t)enc_l0.out, 1, 1.f};
      GM_TRY((lin_fwd<A, EpiStore<A, EPI_ADDEND>, false>(h, x_act, Dp, n, Lx, epi, st)));
    }
  }
  if (!last0) {
    GM_TRY(mlp_hidden_fwd<A>(h, h->encoder, enc, x_act, Dp, D, n, 1, st));
    GM_TRY(last_layer(h->encoder, enc, x_act, Dp, D, enc_out, 2 * Z));
  }
  return normal_out(enc_out);
}

extern "C" {

int gmvae_encode(gmvae_handle* h, const uint8_t* x_u8, int batch, const float* eps, const float* gumbel_u, float* logits_y, float* z_mean,
                 float* z_sample, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  GM_REQUIRE(x_u8 && z_mean && z_sample, "null argument");
  GM_REQUIRE(batch > 0 && batch <= h->cfg.max_batch, "batch must be in [1, max_batch]");
  GM_REQUIRE(h->cfg.objective == GMVAE_OBJECTIVE_REFERENCE, "gmvae_encode needs a handle created with objective=reference");
  if (h->bf16_mode()) return encode_impl<bf16>(h, x_u8, batch, eps, gumbel_u, logits_y, z_mean, z_sample, (cudaStream_t)stream);
  return encode_impl<float>(h, x_u8, batch, eps, gumbel_u, logits_y, z_mean, z_sample, (cudaStream_t)stream);
}
int gmvae_condition(gmvae_handle* h, int which, const float* in1, const float* in2, int n, float* out_a, float* out_b, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  GM_REQUIRE(in1 && out_a, "null argument");
  GM_REQUIRE(n > 0 && n <= h->cfg.max_batch, "n must be in [1, max_batch]");
  GM_REQUIRE(which >= 0 && which <= 3, "unknown conditional distribution");
  GM_REQUIRE(out_b || which == GMVAE_COND_DECODER || which == GMVAE_COND_ENCODER_Y, "a ConditionalNormal returns (mu, sigma): out_b is null");
  if (h->bf16_mode()) return condition_impl<bf16>(h, which, in1, in2, n, out_a, out_b, (cudaStream_t)stream);
  return condition_impl<float>(h, which, in1, in2, n, out_a, out_b, (cudaStream_t)stream);
}
// sample / log_prob / mean of the distribution objects the Conditional* classes return (TFP semantics, SURVEY Appendix B.3-B.5)
int gmvae_dist_normal_sample(const float* mu, const float* sigma, const float* eps, int64_t n, float* out, void* stream) {
  GM_REQUIRE(mu && sigma && eps && out && n > 0, "bad argument");
  GM_CHECK_CUDA(launch_k(dist_map_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, false, 0, mu, sigma, eps, n, out));
  return 0;
}
int gmvae_dist_normal_log_prob(const float* mu, const float* sigma, const float* z, int n, int d, float* out, void* stream) {
  GM_REQUIRE(mu && sigma && z && out && n > 0 && d > 0, "bad argument");
  GM_CHECK_CUDA(launch_k(dist_row_kernel, dim3((unsigned)((n + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, false, 0, mu, sigma, z, n, d, 1.f, out));
  return 0;
}
int gmvae_dist_bernoulli_log_prob(const float* logits, const float* x, int n, int d, float* out, void* stream) {
  GM_REQUIRE(logits && x && out && n > 0 && d > 0, "bad argument");
  GM_CHECK_CUDA(launch_k(dist_row_kernel, dim3((unsigned)((n + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, false, 1, logits, (const float*)nullptr, x, n, d, 1.f, out));
  return 0;
}
int gmvae_dist_bernoulli_mean(const float* logits, int64_t n, float* out, void* stream) {
  GM_REQUIRE(logits && out && n > 0, "bad argument");
  GM_CHECK_CUDA(launch_k(dist_map_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, false, 1, logits, (const float*)nullptr,
                         (const float*)nullptr, n, out));
  return 0;
}
int gmvae_dist_relaxed_sample(const float* logits, const float* u, int n, int k, float temperature, float* out, void* stream) {
  GM_REQUIRE(logits && u && out && n > 0 && k > 0 && temperature > 0.f, "bad argument");
  GM_CHECK_CUDA(launch_k(dist_row_kernel, dim3((unsigned)((n + 7) / 8)), dim3(256), 0, (cudaStream_t)stream, false, 2, logits, (const float*)nullptr, u, n, k,
                         1.f / temperature, out));
  return 0;
}
int gmvae_decode(gmvae_handle* h, const float* z, int n, float* x_mean, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  GM_REQUIRE(z && x_mean, "null argument");
  const int cap = h->cfg.objective == GMVAE_OBJECTIVE_MARGINAL ? h->chunk_samples * h->K : h->cfg.max_batch;
  GM_REQUIRE(n > 0 && n <= cap, "n must be in [1, max_batch]");
  if (h->bf16_mode()) return decode_impl<bf16>(h, z, n, x_mean, (cudaStream_t)stream);
  return decode_impl<float>(h, z, n, x_mean, (cudaStream_t)stream);
}
int gmvae_prior_table(gmvae_handle* h, float* mu, float* sigma, void* stream) {
  DeviceGuard dev_guard(h);
  GM_TRY(check_ready(h));
  GM_REQUIRE(mu && sigma, "null argument");
  const int K = h->K, Z = h->Z;
  const float* a = nullptr; const float* b = nullptr; int mode = 0;
  if (h->cfg.model == GMVAE_MODEL_GMVAE) { a = h->params + h->prior_gmm.layers[0].w_off; b = h->params + h->prior_gmm.layers[0].b_off; mode = 2; }
  else if (h->cfg.model == GMVAE_MODEL_VAE_GMP) { a = h->params + h->loc_off; b = h->params + h->raw_scale_off; mode = 1; }
  GM_CHECK_CUDA(launch_k(prior_params_kernel, dim3((K * Z + 255) / 256), dim3(256), 0, (cudaStream_t)stream, false, a, b, mode, K, Z,
                         h->cfg.raw_sigma_bias, h->cfg.sigma_min, mu, sigma));
  return 0;
}

int gmvae_debug_noise(gmvae_handle* h, float* eps, int64_t n_eps, float* u, int64_t n_u, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h, "null argument");
  if (!eps) n_eps = 0;
  if (!u) n_u = 0;
  int64_t q = (n_eps + 3) / 4 + (n_u + 3) / 4;
  if (q == 0) return 0;
  GM_CHECK_CUDA(launch_k(fill_noise_kernel, dim3((unsigned)((q + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, false, eps, n_eps, u, n_u,
                         (const DeviceState*)h->state, (uint64_t)h->rank, 0, ++h->draws));
  return 0;
}

// runners.create_dataset._preprocess (runners.py:44-47) on the device: x = (intensity / 255 < uniform).
// `intensities` [n_rows, D] bytes resident in HBM; output row r comes from row row_index[r] (device int64[batch],
// each in [0, n_rows)) or, without an index, from row r.  Uniforms: Philox keyed by (seed, draw, rank, element).
int gmvae_binarize(gmvae_handle* h, const uint8_t* intensities, int64_t n_rows, const int64_t* row_index, int batch, uint64_t draw,
                   uint8_t* x_u8, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && h->state, "null handle");
  GM_REQUIRE(batch >= 0 && n_rows >= 0, "negative size");
  if (batch == 0) return 0;
  GM_REQUIRE(intensities && x_u8, "null argument");
  GM_REQUIRE(row_index || batch <= n_rows, "batch exceeds the number of intensity rows");
  const int D = h->cfg.data_size;
  const uint8_t* lo = intensities; const uint8_t* hi = intensities + n_rows * D;
  GM_REQUIRE(x_u8 + (int64_t)batch * D <= lo || x_u8 >= hi, "x_u8 must not overlap the intensities");
  const int64_t n_out = (int64_t)batch * D;
  const int mode = binarize_mode(intensities, x_u8, D);
  const int64_t units = mode == BINARIZE_VEC16 ? n_out / 16 : (n_out + 3) / 4;      // work items of one thread-iteration
  static int blocks_per_sm = 0;
  if (blocks_per_sm == 0) {
    GM_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, binarize_kernel, BINARIZE_THREADS, 0));
    blocks_per_sm = std::max(1, blocks_per_sm);
  }
  const int blocks = (int)std::min<int64_t>((units + BINARIZE_THREADS - 1) / BINARIZE_THREADS, (int64_t)blocks_per_sm * tc::num_sms());
  PhiloxKeys rk;                                                                       // uniforms keyed by (seed, draw, rank, element)
  philox_schedule(binarize_key(h->seed_host, draw), rk);
  GM_CHECK_CUDA(launch_k(binarize_kernel, dim3(blocks), dim3(BINARIZE_THREADS), 0, (cudaStream_t)stream, false, intensities, row_index, D,
                         n_out, rk, (uint64_t)h->rank, mode, x_u8));
  h->launches++;
  return 0;
}

// Bit-packed binary images (numpy.packbits order, ceil(D/8) bytes per row) -> the [batch, D] {0,1} bytes the step reads.
int gmvae_unpack_bits(gmvae_handle* h, const uint8_t* packed, int batch, uint8_t* x_u8, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && packed && x_u8, "null argument");
  GM_REQUIRE(batch > 0, "batch must be positive");
  const int D = h->cfg.data_size, row_bytes = (D + 7) / 8;
  const int64_t n = (int64_t)batch * row_bytes;
  GM_CHECK_CUDA(launch_k(unpack_bits_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, false, packed, n, row_bytes, D, x_u8));
  h->launches++;
  return 0;
}

// Test hook: clock64 stamps of CTA `cta` of every chained-GEMM launch of the following steps are written to
// `trace` (device, 8 launches x 64 tiles x 16 int64; see gemm_chain.cuh).  Null switches it off.
int gmvae_debug_chain_trace(gmvae_handle* h, long long* trace, int cta) {
  GM_REQUIRE(h, "null handle");
  h->chain_trace = trace; h->chain_trace_cta = cta;
  return 0;
}

// Test hook: per-job counters (8 x uint64 per job, gemm_chain.cuh ChainParamsT::jobstat) of the first chained launch of the
// following steps; `stat` = device buffer of 8 * 40 uint64 pre-set by the caller ([0] of every job to ~0, the rest 0).
int gmvae_debug_chain_jobstat(gmvae_handle* h, unsigned long long* stat) {
  GM_REQUIRE(h, "null handle");
  h->chain_jobstat = stat;
  return 0;
}
// Descriptions of the jobs of that launch: 8 ints per job (kind, M, N, k-blocks, tiles, splits, block_n, ndeps); returns the job count.
int gmvae_debug_chain_jobs(gmvae_handle* h, int* out, int cap_jobs) {
  GM_REQUIRE(h && out, "null argument");
  const int n = std::min(cap_jobs, (int)h->chain_jobdesc.size() / 8);
  for (int i = 0; i < 8 * n; ++i) out[i] = h->chain_jobdesc[i];
  return n;
}

int gmvae_profile_enable(gmvae_handle* h, int on) {
  GM_REQUIRE(h, "null argument");
  for (auto& m : h->marks) cudaEventDestroy(m.first);
  h->marks.clear();
  h->profiling = on != 0;
  return 0;
}
int gmvae_profile_read(gmvae_handle* h, double* ms_by_class, int64_t* launches_by_class, int n_classes) {
  GM_REQUIRE(h && ms_by_class && launches_by_class, "null argument");
  GM_REQUIRE(n_classes >= PC_COUNT, "need room for 8 classes");
  for (int i = 0; i < n_classes; ++i) { ms_by_class[i] = 0; launches_by_class[i] = 0; }
  if (h->marks.empty()) return 0;
  GM_CHECK_CUDA(cudaEventSynchronize(h->marks.back().first));
  for (size_t i = 1; i < h->marks.size(); ++i) {
    int cls = h->marks[i].second;
    if (cls < 0) continue;
    float ms = 0.f;
    GM_CHECK_CUDA(cudaEventElapsedTime(&ms, h->marks[i - 1].first, h->marks[i].first));
    ms_by_class[cls] += ms; launches_by_class[cls] += 1;
  }
  return PC_COUNT;
}

// ---- kernel-level test hook ------------------------------------------------------------------
__global__ void dbg_to_bf16(const float* in, bf16* out, int64_t rows, int64_t cols, int64_t ld) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * ld) {
    int64_t r = i / ld, c = i % ld;
    out[i] = __float2bfloat16_rn(c < cols ? in[r * cols + c] : 0.f);
  }
}

int gmvae_debug_gemm(gmvae_handle* h, int impl, int transA, int transB, int M, int N, int K, const float* A, const float* B,
                     float* C, int split_k, void* stream) {
  DeviceGuard dev_guard(h);
  GM_REQUIRE(h && A && B && C, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  GM_CHECK_CUDA(cudaMemsetAsync(C, 0, (size_t)M * N * 4, st));
  EpiAtomicAdd epi{C, (int64_t)N};
  if (impl == 0) {
    int64_t sAm = transA ? 1 : K, sAk = transA ? M : 1, sBk = transB ? 1 : N, sBn = transB ? K : 1;
    GM_CHECK_CUDA((launch_gemm_simt<float, float, EpiAtomicAdd>(A, sAm, sAk, B, sBk, sBn, M, N, K, split_k, epi, st)));
    return 0;
  }
  // tcgen05 path: operands converted to bf16 scratch, rows padded to 16 bytes (test hook only).
  // A stored [M,K] (transA=0 -> K-major) or [K,M] (transA=1 -> MN-major);
  // B stored [K,N] (transB=0 -> MN-major) or [N,K] (transB=1 -> K-major).
  const bool a_mn = transA != 0, b_mn = transB == 0;
  GM_REQUIRE(a_mn == b_mn, "debug hook covers K-major x K-major and MN-major x MN-major");
  const int64_t a_rows = a_mn ? K : M, a_cols = a_mn ? M : K, b_rows = b_mn ? K : N, b_cols = b_mn ? N : K;
  const int64_t lda = round_up((int)a_cols, 8), ldb = round_up((int)b_cols, 8);
  bf16 *a16 = nullptr, *b16 = nullptr;
  GM_CHECK_CUDA(cudaMalloc(&a16, (size_t)a_rows * lda * 2));
  GM_CHECK_CUDA(cudaMalloc(&b16, (size_t)b_rows * ldb * 2));
  dbg_to_bf16<<<(unsigned)((a_rows * lda + 255) / 256), 256, 0, st>>>(A, a16, a_rows, a_cols, lda);
  dbg_to_bf16<<<(unsigned)((b_rows * ldb + 255) / 256), 256, 0, st>>>(B, b16, b_rows, b_cols, ldb);
  int r;
  if (impl >= 2) {
    // traced run of a forward-style layer: out = relu(A B^T + bias) in bf16; the first 4096 int64 of C
    // receive CTA 0's clock64 stamps (16 per tile: see gemm_tc.cuh)
    GM_REQUIRE(!a_mn && (size_t)M * N * 4 >= 4096 * 8, "trace needs K-major operands and a large enough C");
    bf16* o16 = nullptr; float* bias = nullptr; long long* tr = nullptr;
    GM_CHECK_CUDA(cudaMalloc(&o16, (size_t)M * round_up(N, 8) * 2));
    GM_CHECK_CUDA(cudaMalloc(&bias, (size_t)N * 4));
    GM_CHECK_CUDA(cudaMalloc(&tr, 4096 * 8));
    GM_CHECK_CUDA(cudaMemsetAsync(bias, 0, (size_t)N * 4, st));
    GM_CHECK_CUDA(cudaMemsetAsync(tr, 0, 4096 * 8, st));
    tc::Operand a{a16, lda, M, kpad(K, lda)}, b{b16, ldb, N, kpad(K, ldb)};
    tc::g_trace = tr;
    if (impl == 2) {
      EpiStore<bf16> e2{o16, (int64_t)round_up(N, 8), bias, nullptr, 0, 1, 1.f};
      r = tc_dispatch_kk(h, a, b, nullptr, nullptr, M, N, e2, st);
    } else {
      EpiReluMask<bf16, bf16> e3{o16, (int64_t)round_up(N, 8), a16, lda, impl == 4 ? bias : nullptr};
      r = tc_dispatch_kk(h, a, b, nullptr, nullptr, M, N, e3, st);
    }
    tc::g_trace = nullptr;
    GM_CHECK_CUDA(cudaMemcpyAsync(C, tr, 4096 * 8, cudaMemcpyDeviceToDevice, st));
    cudaError_t e = cudaStreamSynchronize(st);
    cudaFree(o16); cudaFree(bias); cudaFree(tr); cudaFree(a16); cudaFree(b16);
    if (r != 0) return r;
    GM_CHECK_CUDA(e);
    return 0;
  }
  if (!a_mn) {
    tc::Operand a{a16, lda, M, kpad(K, lda)}, b{b16, ldb, N, kpad(K, ldb)};
    r = tc_dispatch_kk(h, a, b, nullptr, nullptr, M, N, epi, st);
  } else {
    tc::Operand a{a16, lda, kpad(M, lda), K}, b{b16, ldb, kpad(N, ldb), K};
    r = N <= 64    ? tc::launch_gemm_tc<64, true, true, EpiAtomicAdd>(a, b, nullptr, nullptr, M, N, split_k, epi, st)
        : N <= 128 ? tc::launch_gemm_tc<128, true, true, EpiAtomicAdd>(a, b, nullptr, nullptr, M, N, split_k, epi, st)
                   : tc::launch_gemm_tc<256, true, true, EpiAtomicAdd>(a, b, nullptr, nullptr, M, N, split_k, epi, st);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(a16); cudaFree(b16);
  if (r != 0) return r;
  GM_CHECK_CUDA(e);
  return 0;
}

}  // extern "C"

// chain_sched.cuh -- the schedule arithmetic of the chained kernel (gemm_chain.cuh): the job record, which walker takes which tile, and
// which rows / columns a tile covers.  Free of device-only code so that tests/native/host_chain_sched.cu compiles THESE functions for
// the host and checks them exhaustively (every tile taken exactly once in every mode) without a GPU.
#pragma once

#if defined(__CUDACC__)
#define GMVAE_SCHED_FN __host__ __device__ __forceinline__
#else
#define GMVAE_SCHED_FN inline
#endif

namespace gmvae {
namespace tc {

constexpr int CHAIN_MAX_DEPS = 4;
constexpr int CHAIN_EPI_BYTES = 128;
constexpr int CHAIN_EPI2_BYTES = 64;
constexpr int SCHED_BLOCK_M = 128;      // rows of a CTA's tile (= BLOCK_M of gemm_tc.cuh)

// counters[base + row_block] >= target.  by_k = 0: the row block of the consumer's own tile;
// by_k = 1 (weight gradients: the contraction runs over the batch): every row block its k-range covers.
struct ChainDep { int base, target, by_k, nblocks, seg2; };   // seg2: only the second K segment reads it (checked when that segment starts)

struct alignas(16) ChainJob {
  int a1, b1, a2, b2;                // indices into ChainParams::maps
  int c;                             // epilogue operand read by TMA (ReLU-mask source), box = one patch
  int d;                             // output written by TMA store / reduce-add, box = one patch
  int gw;                            // 16-column chunks per 64-byte patch row: 2 (bf16), 1 (fp32), 0: per-row stores
  int M, N, kb1, kb2, kb_per_split, num_splits;
  int block_n, a_mn, b_mn, kind;
  int tiles_n, tiles_mn, total_tiles, tile_base;
  int sig_base;                      // counters[sig_base + m_block] += 1 per epilogue warp per finished tile; -1: nobody waits
  int ndeps;
  int epi_dep;                       // index into deps of the job that wrote the epilogue's own operand (ReLU mask source), or -1
  ChainDep deps[CHAIN_MAX_DEPS];
  alignas(16) unsigned char epi[CHAIN_EPI_BYTES];
  int rot;                           // 1: the n-tile index is rotated by the row block (see chain_tile)
  int walk_total;                    // steps of a walker (CTA, CTA pair, 4-CTA cluster) through the job: total_tiles, or tiles_mn2 * num_splits (quad mode)
  int tiles_mn2;                     // quad mode: double tiles (two adjacent pair tiles) per k-split = ceil(tiles_mn / 2)
  int wfirst, wcount;                // the walkers [wfirst, wfirst + wcount) take the job's tiles (wcount 0: all of them).  The backward pass
                                     // gives the chain of dependent data-gradient jobs and the weight-gradient jobs disjoint sets of CTA pairs:
                                     // an in-order walker cannot step over a long weight-gradient tile to the chain tile queued behind it
  int share;                         // quad mode: the two pair tiles of a double tile cover the same rows (tiles_n even): A is loaded once, multicast
  int fuse;                          // EK_STORE_F32 jobs with N <= 16: a y head applied to the row in the epilogue (EK_ROWS_Y_FWD / _BWD), 0 = none
  int zslice;                        // EK_ATOMIC, deterministic mode: tile of k-split z STORES its partial into slice z of the 3-D map d
                                     // ([splits][M][ld], det_slice_index) instead of reduce-adding into the gradient buffer
  alignas(16) unsigned char epi2[CHAIN_EPI2_BYTES];   // its parameters (RowsYFwd / RowsYBwd)
};
// Tile l of a job -> (k-split z, row block mb, first column n0).  n fastest, then m, then k-split.  With J.rot the n-tile index
// is rotated by the row block: a job whose last n-tile is ragged (784 = 3 x 256 + 16) has cheap and expensive tiles, and since
// the CTAs walk the tile sequence with a stride (148) that is a multiple of tiles_n, every CTA would otherwise see one n-tile
// index only -- a quarter of the CTAs all the cheap tiles, the rest all the expensive ones.
// PAIR: the job's tile space is in PAIR tiles of 256 rows (J.tiles_mn = ceil(row blocks / 2) * tiles_n); CTA `rank` of the pair owns
// row block 2 * pm + rank (possibly beyond M: a phantom half whose loads read zeros and whose stores are clipped).
// QUAD (CL = 4): a walker is a cluster of two CTA pairs and `l` counts DOUBLE tiles -- the pair tiles 2d and 2d + 1 of a k-split, taken
// by pair h = crank >> 1.  With an even number of n-tiles both lie in the same row block: the pairs share the A rows (J.share, TMA
// multicast).  An odd per-split tile count leaves the last double tile's second half a phantom (rows beyond M).
template <int CL>
GMVAE_SCHED_FN void chain_tile(const ChainJob& J, int l, int crank, int& z, int& mb, int& n0) {
  int mn;
  if (CL == 4) {
    z = l / J.tiles_mn2;
    mn = 2 * (l - z * J.tiles_mn2) + (crank >> 1);
  } else {
    z = l / J.tiles_mn;
    mn = l - z * J.tiles_mn;
  }
  int pm = mn / J.tiles_n;
  int nt = mn - pm * J.tiles_n;
  if (CL == 4 && mn >= J.tiles_mn) { pm = J.tiles_mn / J.tiles_n; nt = 0; }     // phantom pair tile
  if (J.rot) { nt += pm % J.tiles_n; if (nt >= J.tiles_n) nt -= J.tiles_n; }
  n0 = nt * J.block_n;
  mb = CL >= 2 ? 2 * pm + (crank & 1) : pm;
}

// Which tiles of job J walker c (of G) takes: first index and stride; false: none.  MUL: walker units per entry of J.wfirst / J.wcount
// (row jobs are dealt to single CTAs).
template <int MUL>
GMVAE_SCHED_FN bool chain_walk(const ChainJob& J, int c, int G, int& first, int& stride) {
  int wf = J.wfirst * MUL, wc = J.wcount * MUL;
  if (wc <= 0 || wf + wc > G) { wf = 0; wc = G; }          // everybody (also when the grid came out smaller than planned)
  const int cj = c - wf;
  if (cj < 0 || cj >= wc) return false;
  stride = wc;
  first = ((cj - J.tile_base) % wc + wc) % wc;
  return true;
}

// Host side: tile space of a GEMM job.  cl = CTAs per walker (1: single CTAs, 128-row tiles; 2: CTA pairs, 256-row pair tiles; 4: clusters
// of two pairs walking double tiles).  `split_k` is a request: the k-blocks are cut into equal runs and the number of runs recomputed.
inline void chain_job_geometry(ChainJob& J, int M, int N, int block_n, int split_k, int kb_total, bool a_mn, int cl) {
  const int tiles_m = (M + SCHED_BLOCK_M - 1) / SCHED_BLOCK_M, tiles_n = (N + block_n - 1) / block_n;
  const int tiles_m_walk = cl >= 2 ? (tiles_m + 1) / 2 : tiles_m;      // pair modes: tiles of 256 rows, one row block per CTA of the pair
  if (split_k < 1) split_k = 1;
  const int per = (kb_total + split_k - 1) / split_k;
  split_k = (kb_total + per - 1) / per;
  J.M = M; J.N = N; J.kb_per_split = per; J.num_splits = split_k;
  J.block_n = block_n; J.a_mn = a_mn ? 1 : 0;
  J.tiles_n = tiles_n; J.tiles_mn = tiles_m_walk * tiles_n; J.total_tiles = J.tiles_mn * split_k;
  J.tiles_mn2 = (J.tiles_mn + 1) / 2;
  J.walk_total = cl == 4 ? J.tiles_mn2 * split_k : J.total_tiles;
  J.share = (cl == 4 && tiles_n % 2 == 0) ? 1 : 0;
  J.rot = (tiles_n > 1 && N % block_n != 0 && !a_mn) ? 1 : 0;
}
// Deterministic mode: where element (m, n) of k-split z of a weight-gradient job lives in its partial buffer, slices of M rows x ld
// floats (ld = N rounded up to 4: 16-byte rows for TMA).  The tiles store through a 3-D tensor map of this layout (a ragged row block
// is clipped at M within its own slice); det_reduce_kernel adds slices 0 .. splits-1 of every element in that order.
GMVAE_SCHED_FN int det_slice_ld(int N) { return (N + 3) / 4 * 4; }
GMVAE_SCHED_FN long long det_slice_index(int z, int m, int n, int M, int ld) { return ((long long)z * M + m) * ld + n; }
// The rows / columns tile (z, mb, n0) of a weight-gradient job writes: [r0, r1) x [c0, c1) of slice z (empty for a phantom half)
GMVAE_SCHED_FN void det_tile_region(const ChainJob& J, int mb, int n0, int& r0, int& r1, int& c0, int& c1) {
  r0 = mb * SCHED_BLOCK_M; r1 = r0 + SCHED_BLOCK_M < J.M ? r0 + SCHED_BLOCK_M : J.M;
  c0 = n0; c1 = n0 + J.block_n < J.N ? n0 + J.block_n : J.N;
  if (r1 < r0) r1 = r0;
}

// Row-block counters a job's tiles signal (phantom halves / phantom pair tiles signal counters nobody waits for)
inline int chain_job_counters(int M, int cl) {
  const int tiles_m = (M + SCHED_BLOCK_M - 1) / SCHED_BLOCK_M;
  return cl >= 2 ? 2 * ((tiles_m + 1) / 2) + (cl == 4 ? 2 : 0) : tiles_m;
}

}  // namespace tc
}  // namespace gmvae

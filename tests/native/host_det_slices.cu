// Host build of the deterministic mode's weight-gradient slice arithmetic (gmvae_b200/csrc/chain_sched.cuh): simulates every walker
// and CTA of a weight-gradient job of the chained kernel and checks that every (k-split, element) of the partial buffer is written by
// exactly one tile, and that the reduction (det_reduce_kernel's addressing) reads every split of every element exactly once, in
// increasing split order.
#include <vector>

#include "../../gmvae_b200/csrc/chain_sched.cuh"

using namespace gmvae::tc;

template <int CL>
static int check(int M, int N, int block_n, int split_k, int kb, int G) {
  ChainJob J = {};
  chain_job_geometry(J, M, N, block_n, split_k, kb, true, CL);
  const int S = J.num_splits, ld = det_slice_ld(N);
  if (ld < N || ld % 4 != 0) return 1;
  std::vector<unsigned char> written((size_t)S * M * ld, 0);
  for (int c = 0; c < G; ++c) {
    int first = -1, stride = -1;
    if (!chain_walk<1>(J, c, G, first, stride)) continue;
    for (int l = first; l < J.walk_total; l += stride)
      for (int r = 0; r < CL; ++r) {
        int z, mb, n0, r0, r1, c0, c1;
        chain_tile<CL>(J, l, r, z, mb, n0);
        if (z < 0 || z >= S) return 2;
        det_tile_region(J, mb, n0, r0, r1, c0, c1);     // a phantom half (rows beyond M) writes nothing
        for (int m = r0; m < r1; ++m)
          for (int n = c0; n < c1; ++n) {
            const long long i = det_slice_index(z, m, n, M, ld);
            if (i < 0 || i >= (long long)S * M * ld) return 3;
            if (written[i]++) return 4;                // two tiles on one element of one slice
          }
      }
  }
  // the reduction: element (m, n) reads part + m * ld + n + s * (M * ld) for s = 0 .. S-1
  std::vector<unsigned char> read((size_t)S * M * ld, 0);
  for (int m = 0; m < M; ++m)
    for (int n = 0; n < N; ++n) {
      long long prev = -1;
      for (int s = 0; s < S; ++s) {
        const long long i = (long long)m * ld + n + (long long)s * ((long long)M * ld);
        if (i != det_slice_index(s, m, n, M, ld)) return 5;
        if (i <= prev) return 6;                          // increasing split order
        if (!written[i]) return 7;                        // a split nobody wrote
        if (read[i]++) return 8;
        prev = i;
      }
    }
  for (size_t i = 0; i < written.size(); ++i)
    if (written[i] && !read[i]) return 9;                 // written but never reduced
  return 0;
}

extern "C" int host_det_check(int M, int N, int block_n, int split_k, int kb, int cl, int G) {
  return cl == 2 ? check<2>(M, N, block_n, split_k, kb, G) : check<1>(M, N, block_n, split_k, kb, G);
}

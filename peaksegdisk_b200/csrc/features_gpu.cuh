// features_gpu.cuh -- per-problem coverage statistics on the device (psd_features).
//
// The features penalty learning uses (PeakSegPipeline's problem.features: quartiles, mean, sd, bases,
// rows) are statistics of the per-base vector x of a problem: row i contributes w_i = chromEnd_i -
// chromStart_i copies of its count c_i.  The kernels never expand the rows.  They return exact
// integers only -- S1 = sum w c, S2 = sum w c^2 (128 bits), min, max and x[k] (the sorted vector) at the
// at most PSD_FEAT_SEL ranks the interior quartiles need -- and the host does the fp64 arithmetic.
//
// x[k] comes from a weighted radix select over the 31-bit counts, four 8-bit digits from the top:
//   * features_hist_kernel<FIRST> (one pass over the rows, the tiling of rle_encode_kernel: 8,192-row
//     tiles that never straddle two problems): each block adds the weights of the rows whose higher
//     digits equal a selection's prefix into shared 64-bit bins of the row's current digit, one set of
//     256 bins per distinct prefix of the tile's problem, and flushes the non-zero bins with global
//     atomics.  A thread keeps a run (digit, weight) per selection and adds to shared memory only when
//     the digit changes, so the common long runs of one digit (the top digits of small counts) cost one
//     shared atomic per thread.  The first pass also accumulates S1, S2 (two u64 words, explicit carry),
//     min and max.
//   * features_select_kernel (one warp per problem) walks each selection's histogram to the bucket
//     that holds its remaining rank, appends the digit to the prefix, zeroes the histograms for the
//     next pass, and re-points selections with equal prefixes at one shared histogram.
// Traffic: 8 B per row per pass (int32 weight and count), four passes.
#pragma once
#include <cuda_runtime.h>
#include "rle_gpu.cuh"

#define PSD_FEAT_SEL 6   // x[lo] and x[lo + 1] of the quartiles at p = .25, .5, .75

struct FeatProblem {
  long long row_off;   // first row in the packed weight / count arrays
  int n_rows;
  int tile0;           // id of the problem's first tile
  int sel0, n_sel;     // its selections, [sel0, sel0 + n_sel)
};

struct FeatSel {
  unsigned long long rank;   // rank of the wanted base among those whose count starts with `prefix`
  unsigned prefix;           // the digits selected so far (bits below the current digit are 0)
  int rep;                   // first selection of the problem with the same prefix: it owns the histogram
};

struct FeatSums {
  unsigned long long s1, s2_lo, s2_hi;   // sum w c; sum w c^2 as 128 bits
  unsigned min, max;                     // the host sets min = 0xffffffff, max = 0
};

struct FeatHistParams {
  const FeatProblem* probs;
  const int* tile_prob;   // tile -> problem
  int n_tiles;
  const int* weight; const int* count;
  const FeatSel* sel;
  unsigned long long* hist;   // [selection][256], zero before each pass
  FeatSums* sums;
  int shift;                  // the digit of this pass: bits [shift + 7 : shift]
  unsigned mask;              // the bits above it
};

struct FeatSelectParams {
  const FeatProblem* probs;
  int n_probs;
  FeatSel* sel;
  unsigned long long* hist;
  int shift;
  int* error;   // set to 1 if a rank is not inside its histogram (never expected)
};

template <bool FIRST>
__global__ void __launch_bounds__(PSD_RLE_WARPS * 32) features_hist_kernel(const FeatHistParams P) {
  __shared__ unsigned long long s_bin[PSD_FEAT_SEL][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x;
  const int pi = P.tile_prob[tile];
  const FeatProblem Q = P.probs[pi];
  bool act[PSD_FEAT_SEL]; unsigned pre[PSD_FEAT_SEL];
#pragma unroll
  for (int j = 0; j < PSD_FEAT_SEL; j++) {
    act[j] = false; pre[j] = 0;
    if (j < Q.n_sel) {
      const FeatSel S = P.sel[Q.sel0 + j];
      act[j] = S.rep == Q.sel0 + j;
      pre[j] = S.prefix;
    }
  }
  for (int i = threadIdx.x; i < PSD_FEAT_SEL * 256; i += blockDim.x) (&s_bin[0][0])[i] = 0ull;
  __syncthreads();

  const int* __restrict__ wv = P.weight + Q.row_off;
  const int* __restrict__ cv = P.count + Q.row_off;
  const int n = Q.n_rows;
  const int wbase = (tile - Q.tile0) * PSD_RLE_TILE + warp * (32 * PSD_RLE_STRIPES);
  int rd[PSD_FEAT_SEL]; unsigned long long rw[PSD_FEAT_SEL];   // the thread's current run per selection
#pragma unroll
  for (int j = 0; j < PSD_FEAT_SEL; j++) { rd[j] = -1; rw[j] = 0; }
  unsigned long long s1 = 0, s2lo = 0, s2hi = 0;
  unsigned mn = 0xffffffffu, mx = 0;
#pragma unroll 8
  for (int s = 0; s < PSD_RLE_STRIPES; s++) {
    const int i = wbase + 32 * s + lane;
    if (i >= n) break;
    const unsigned c = (unsigned)__ldcs(cv + i);
    const unsigned long long w = (unsigned)__ldcs(wv + i);
    if (FIRST) {
      s1 += w * c;
      const unsigned long long c2 = (unsigned long long)c * c, lo = c2 * w;
      s2hi += __umul64hi(c2, w);
      s2lo += lo;
      s2hi += s2lo < lo;
      mn = min(mn, c); mx = max(mx, c);
    }
    const int d = (int)((c >> P.shift) & 255u);
#pragma unroll
    for (int j = 0; j < PSD_FEAT_SEL; j++) {
      if (act[j] && (c & P.mask) == pre[j]) {
        if (d == rd[j]) rw[j] += w;
        else {
          if (rd[j] >= 0) atomicAdd(&s_bin[j][rd[j]], rw[j]);
          rd[j] = d; rw[j] = w;
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < PSD_FEAT_SEL; j++)
    if (rd[j] >= 0) atomicAdd(&s_bin[j][rd[j]], rw[j]);

  if (FIRST) {   // warp totals, then one set of global atomics per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_down_sync(0xffffffffu, s1, o);
      const unsigned long long lo = __shfl_down_sync(0xffffffffu, s2lo, o);
      s2hi += __shfl_down_sync(0xffffffffu, s2hi, o);
      s2lo += lo;
      s2hi += s2lo < lo;
      mn = min(mn, __shfl_down_sync(0xffffffffu, mn, o));
      mx = max(mx, __shfl_down_sync(0xffffffffu, mx, o));
    }
    if (lane == 0 && wbase < n) {
      FeatSums* S = P.sums + pi;
      atomicAdd(&S->s1, s1);
      const unsigned long long old = atomicAdd(&S->s2_lo, s2lo);
      atomicAdd(&S->s2_hi, s2hi + (old + s2lo < old ? 1ull : 0ull));   // the carry out of the low word
      atomicMin(&S->min, mn);
      atomicMax(&S->max, mx);
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < PSD_FEAT_SEL; j++) {
    if (!act[j]) continue;
    for (int b = threadIdx.x; b < 256; b += blockDim.x) {
      const unsigned long long v = s_bin[j][b];
      if (v) atomicAdd(P.hist + (size_t)(Q.sel0 + j) * 256 + b, v);
    }
  }
}

__global__ void __launch_bounds__(256) features_select_kernel(const FeatSelectParams P) {
  const int pi = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (pi >= P.n_probs) return;
  const FeatProblem Q = P.probs[pi];
  // lane j < n_sel holds selection j
  FeatSel S{0ull, 0u, -1};
  if (lane < Q.n_sel) S = P.sel[Q.sel0 + lane];
  const int old_rep = S.rep;
  for (int j = 0; j < Q.n_sel; j++) {
    const int rep = __shfl_sync(0xffffffffu, S.rep, j);
    const unsigned long long rank = __shfl_sync(0xffffffffu, S.rank, j);
    const unsigned long long* h = P.hist + (size_t)rep * 256 + lane * 8;
    unsigned long long v[8], tot = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) { v[k] = h[k]; tot += v[k]; }
    unsigned long long incl = tot;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    unsigned long long below = incl - tot;   // weight of the bins before this lane's
    const bool mine = below <= rank && rank < incl;
    int d = -1;
    if (mine) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        if (d < 0 && rank < below + v[k]) d = lane * 8 + k;
        else if (d < 0) below += v[k];
      }
    }
    const unsigned who = __ballot_sync(0xffffffffu, mine);
    if (!who) { if (lane == 0) *P.error = 1; continue; }
    const int src = __ffs(who) - 1;
    d = __shfl_sync(0xffffffffu, d, src);
    below = __shfl_sync(0xffffffffu, below, src);
    if (lane == j) { S.prefix |= (unsigned)d << P.shift; S.rank = rank - below; }
  }
  __syncwarp();
  // zero the histograms of this pass, then share one histogram among selections with equal prefixes
  for (int j = 0; j < Q.n_sel; j++) {
    const int rep = __shfl_sync(0xffffffffu, old_rep, j);
    if (rep == Q.sel0 + j) {
      unsigned long long* h = P.hist + (size_t)rep * 256;
      for (int b = lane; b < 256; b += 32) h[b] = 0ull;
    }
  }
  int rep = Q.sel0 + lane;
  for (int j = Q.n_sel - 1; j >= 0; j--) {
    const unsigned pj = __shfl_sync(0xffffffffu, S.prefix, j);
    if (j < lane && pj == S.prefix) rep = Q.sel0 + j;
  }
  if (lane < Q.n_sel) { S.rep = rep; P.sel[Q.sel0 + lane] = S; }
}

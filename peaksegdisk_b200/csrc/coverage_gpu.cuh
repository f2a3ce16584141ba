// coverage_gpu.cuh -- per-base coverage of aligned reads on the device (psd_coverage_from_reads).
//
// Front half of the reads -> segmentation workflow the reference's Spatial_correlation vignette does
// with R or bedtools (`genomecov -bga`): the coverage of base b of a region is the number of reads
// [start, end) with start <= b < end, and the output rows are the maximal runs of equal coverage that
// tile the region.  Three steps per wave of problems, all HBM-bound integer work, no sort:
//   1. the dense int32 delta buffer (one entry per base of every region, packed back to back) is
//      zeroed with cudaMemsetAsync;
//   2. reads_scatter_kernel: one thread per read (grid-stride), clipped to its problem's region,
//      +1 at its first base and -1 at the base after its last one (when that is inside the region);
//   3. coverage_scan_kernel: an in-place inclusive prefix sum per problem turns deltas into per-base
//      coverage, with the tiling, ticket order and decoupled look-back of rle_encode_kernel
//      (rle_gpu.cuh: 8,192-base tiles that never straddle two problems, the same RleVec / tile_vec
//      descriptors);
// then rle_encode_kernel, unchanged, turns the coverage into rows.  Traffic: 4 B per base zeroed,
// 8 B per base scanned (read + write), 4 B per base encoded, 12 B per row and ~8 B per read.
#pragma once
#include <cuda_runtime.h>
#include "rle_gpu.cuh"

struct CovScatterParams {
  const int* read_start; const int* read_end;   // all reads of the wave, problem after problem
  long long n_reads;
  const long long* read_off;                    // [n_probs + 1]: first read of each problem
  const int* region_start;                      // [n_probs]
  const RleVec* vecs;                           // [n_probs]: raw_off = first base in `delta`, n_pos = region length
  int n_probs;
  int* delta;
};

struct CovScanParams {
  const RleVec* vecs;
  const int* tile_vec;              // tile -> problem
  int n_tiles;
  int* cov;                         // in place: deltas in, coverage out
  unsigned long long* tile_state;   // zeroed before the launch; see cov_pack()
  unsigned int* ticket;             // zeroed before the launch
  int* error;                       // set to 1 if a look-back ever gave up (never expected)
};

__global__ void __launch_bounds__(256) reads_scatter_kernel(const CovScatterParams P) {
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < P.n_reads; r += (long long)gridDim.x * blockDim.x) {
    int lo = 0, hi = P.n_probs - 1;   // the last problem whose first read is <= r (problems may have no reads)
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (__ldg(P.read_off + mid) <= r) lo = mid; else hi = mid - 1;
    }
    const int n = P.vecs[lo].n_pos;
    const long long a = (long long)__ldcs(P.read_start + r) - __ldg(P.region_start + lo);
    const long long b = (long long)__ldcs(P.read_end + r) - __ldg(P.region_start + lo);
    if (b <= 0 || a >= n) continue;   // wholly outside the region
    int* d = P.delta + P.vecs[lo].raw_off;
    atomicAdd(d + (a > 0 ? a : 0), 1);
    if (b < n) atomicAdd(d + b, -1);
  }
}

// tile state word: [63:62] flag (0 empty, 1 aggregate of this tile, 2 inclusive prefix), [31:0] the
// signed sum (a tile's aggregate is negative when it holds more read ends than starts)
__device__ __forceinline__ unsigned long long cov_pack(unsigned flag, int sum) {
  return ((unsigned long long)flag << 62) | (unsigned long long)(unsigned)sum;
}

__global__ void __launch_bounds__(PSD_RLE_WARPS * 32) coverage_scan_kernel(const CovScanParams P) {
  __shared__ int s_tile;
  __shared__ int s_wtot[PSD_RLE_WARPS];
  __shared__ int s_excl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) s_tile = (int)atomicAdd(P.ticket, 1u);
  __syncthreads();
  const int tile = s_tile;
  if (tile >= P.n_tiles) return;
  const RleVec V = P.vecs[P.tile_vec[tile]];
  int* __restrict__ v = P.cov + V.raw_off;
  const int n_pos = V.n_pos;
  const int wbase = (tile - V.tile0) * PSD_RLE_TILE + warp * (32 * PSD_RLE_STRIPES);

  // ---- inclusive scan of the warp's 32 stripes (all 32 loads in flight first) ---------------------
  int val[PSD_RLE_STRIPES];
#pragma unroll
  for (int s = 0; s < PSD_RLE_STRIPES; s++) {
    const int i = wbase + 32 * s + lane;
    val[s] = (i < n_pos) ? v[i] : 0;
  }
  int run = 0;   // sum of the warp's earlier stripes
#pragma unroll
  for (int s = 0; s < PSD_RLE_STRIPES; s++) {
    int x = val[s];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    val[s] = run + x;
    run += __shfl_sync(0xffffffffu, x, 31);
  }
  if (lane == 0) s_wtot[warp] = run;
  __syncthreads();

  // ---- tile prefix by decoupled look-back (thread 0) -------------------------------------------------
  if (threadIdx.x == 0) {
    int t_sum = 0;
#pragma unroll
    for (int w = 0; w < PSD_RLE_WARPS; w++) t_sum += s_wtot[w];
    int e_sum = 0;
    if (tile > V.tile0) {
      atomicExch(P.tile_state + tile, cov_pack(1u, t_sum));
      for (int t = tile - 1; t >= V.tile0; t--) {
        unsigned long long w = 0;
        long long spins = 0;
        do {
          w = atomicAdd(P.tile_state + t, 0ull);
          if (++spins > (1ll << 22)) { *P.error = 1; break; }
        } while ((w >> 62) == 0);
        e_sum += (int)(unsigned)(w & 0xffffffffull);
        if ((w >> 62) != 1) break;   // an inclusive prefix ends the walk
      }
    }
    atomicExch(P.tile_state + tile, cov_pack(2u, e_sum + t_sum));
    s_excl = e_sum;
  }
  __syncthreads();

  int base = s_excl;
#pragma unroll
  for (int w = 0; w < PSD_RLE_WARPS; w++) {
    if (w < warp) base += s_wtot[w];
  }
#pragma unroll
  for (int s = 0; s < PSD_RLE_STRIPES; s++) {
    const int i = wbase + 32 * s + lane;
    if (i < n_pos) v[i] = base + val[s];
  }
}

// joint_gpu.cuh -- exact joint single-peak models over many samples on the device (psd_joint_models).
//
// The model (include/peaksegdisk_b200.h documents it; joint.cpp restates it on the host):  a problem has S
// samples over a grid of N bins; a peak (a, b), 1 <= a < b <= N - 1, is shared by position, and sample s can
// carry it only if its peak mean is strictly above both flank means.  The reduction r_s = L1_s - L3_s of the
// feasible samples, sorted by (r desc, s asc), gives R_k, the sequential sum of the first k, and
// loss_k(a, b) = flat - R_k.  For every k the device finds the minimum over all peaks, ties to the smaller
// (a, b), which is the smaller flattened pair index t.
//
// Arrays of one problem are [grid index][sample] ((N + 1) * S elements from grid_off), so that the lanes of
// a warp, which hold consecutive samples, load consecutive words:
//   pref   int64 C_s(0, i), exact (the host bins the rows);
//   lleft  L_s(0, i) and lright L_s(i, N) (joint_flank_kernel); L1_s = lleft at i = N.
// Kernels:
//   joint_flank_kernel   one thread per (grid index, sample), 1,024-element tiles that never straddle problems.
//   joint_flat_kernel    one thread per problem: flat = sum of L1_s in sample order.
//   joint_pair_kernel<J> the hot path.  The (a, b) triangle of every problem is cut into chunks of
//                        consecutive pair indices, one chunk per warp.  Per pair, lane l holds samples
//                        l + 32 j (j < J): one psd_log and the two 128-bit feasibility tests each; then a
//                        bitonic sort of the 32 J (r, s) keys across the warp (position lane * J + j), the
//                        sequential prefix of the sorted reductions lane by lane, and a running (loss, t)
//                        minimum per k in registers (k = lane * J + j + 1).  The chunk's minima go to the
//                        candidate arrays [k - 1][chunk].
//   joint_reduce_kernel  one warp per (problem, k): the minimum (loss, t) over the problem's chunks.
#pragma once
#include <cuda_runtime.h>
#include "psd_math.h"

#define PSD_JOINT_WARPS 8           // warps per block of the pair kernel
#define PSD_JOINT_FLANK_TILE 1024   // elements per block of the flank kernel

struct JointProblem {
  long long grid_off;   // first element of the [grid index][sample] arrays
  long long cand_off;   // first candidate ([k - 1][chunk], S * n_chunks of them)
  int S, N, bin, len;   // samples, bins, bin width, region length (g_N - g_0)
  int chunk0, n_chunks; // the problem's chunks in the chunk table
  int tile0;            // its first flank tile
};

struct JointChunk {
  int prob;
  int a, b;             // the first pair of the chunk
  int t0, count;        // its flattened index and the number of pairs
};

struct JointItem { int prob, k; };

struct JointParams {
  const JointProblem* probs;
  const long long* pref;
  double* lleft; double* lright;
  double* flat;                        // per problem
  const int* tile_prob; int n_tiles;   // flank tiles
  int n_probs;
  const JointChunk* chunks; int chunk_begin, chunk_end;   // pair kernel: the chunks of one J
  double* cand_loss; int* cand_t;
  const JointItem* items; int n_items;
  double* out_loss; int* out_t;        // per item
};

__device__ __forceinline__ long long joint_g(int i, int N, int bin, int len) { return i == N ? (long long)len : (long long)i * bin; }

// L = C - C log(C / W), 0 when C == 0
__device__ __forceinline__ double joint_seg_loss(long long c, long long w, const uint64_t* T) {
  if (c == 0) return 0.0;
  const double C = (double)c;
  return C - C * psd_log(C / (double)w, T);
}

// (r desc, s asc): the order in which samples are added to the peak
__device__ __forceinline__ bool joint_first(double r1, int s1, double r2, int s2) { return r1 > r2 || (r1 == r2 && s1 < s2); }

__global__ void __launch_bounds__(256) joint_flank_kernel(const JointParams P) {
  __shared__ uint64_t tab[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = d_log_tab[i];
  __syncthreads();
  const int pi = P.tile_prob[blockIdx.x];
  const JointProblem Q = P.probs[pi];
  const long long n = (long long)(Q.N + 1) * Q.S;
  const long long* pref = P.pref + Q.grid_off;
  for (long long e = (long long)(blockIdx.x - Q.tile0) * PSD_JOINT_FLANK_TILE + threadIdx.x;
       e < n && e < (long long)(blockIdx.x - Q.tile0 + 1) * PSD_JOINT_FLANK_TILE; e += blockDim.x) {
    const int i = (int)(e / Q.S), s = (int)(e - (long long)i * Q.S);
    const long long c0i = pref[e], tot = pref[(long long)Q.N * Q.S + s];
    const long long g = joint_g(i, Q.N, Q.bin, Q.len);
    P.lleft[Q.grid_off + e] = i == 0 ? 0.0 : joint_seg_loss(c0i, g, tab);
    P.lright[Q.grid_off + e] = i == Q.N ? 0.0 : joint_seg_loss(tot - c0i, Q.len - g, tab);
  }
}

__global__ void __launch_bounds__(128) joint_flat_kernel(const JointParams P) {
  const int pi = blockIdx.x * blockDim.x + threadIdx.x;
  if (pi >= P.n_probs) return;
  const JointProblem Q = P.probs[pi];
  const double* l1 = P.lleft + Q.grid_off + (long long)Q.N * Q.S;
  double f = 0.0;
  for (int s = 0; s < Q.S; s++) f += l1[s];
  P.flat[pi] = f;
}

template <int J>
__global__ void __launch_bounds__(PSD_JOINT_WARPS * 32) joint_pair_kernel(const JointParams P) {
  __shared__ uint64_t tab[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = d_log_tab[i];
  __syncthreads();
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int c = P.chunk_begin + blockIdx.x * PSD_JOINT_WARPS + (threadIdx.x >> 5);
  if (c >= P.chunk_end) return;
  const JointChunk K = P.chunks[c];
  const JointProblem Q = P.probs[K.prob];
  const int S = Q.S, N = Q.N;
  const long long* __restrict__ pref = P.pref + Q.grid_off;
  const double* __restrict__ ll = P.lleft + Q.grid_off;
  const double* __restrict__ lr = P.lright + Q.grid_off;
  const double flat = P.flat[K.prob];
  long long tot[J], pa[J];
  double l1[J], la[J], best[J];
  int bt[J];
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int s = j * 32 + lane;
    tot[j] = s < S ? pref[(long long)N * S + s] : 0;
    l1[j] = s < S ? ll[(long long)N * S + s] : 0.0;
    best[j] = PSD_INF; bt[j] = -1;
  }
  int a = K.a, b = K.b;
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int s = j * 32 + lane;
    pa[j] = s < S ? pref[(long long)a * S + s] : 0;
    la[j] = s < S ? ll[(long long)a * S + s] : 0.0;
  }
  for (int q = 0; q < K.count; q++) {
    const long long ga = joint_g(a, N, Q.bin, Q.len), gb = joint_g(b, N, Q.bin, Q.len);
    const unsigned long long w0a = (unsigned long long)ga, wab = (unsigned long long)(gb - ga), wbn = (unsigned long long)(Q.len - gb);
    double kr[J]; int ks[J];
    int nf = 0;
#pragma unroll
    for (int j = 0; j < J; j++) {
      const int s = j * 32 + lane;
      kr[j] = -PSD_INF; ks[j] = s;
      if (s < S) {
        const long long pb = pref[(long long)b * S + s];
        const unsigned long long cab = (unsigned long long)(pb - pa[j]), c0a = (unsigned long long)pa[j], cbn = (unsigned long long)(tot[j] - pb);
        const bool feasible = (unsigned __int128)cab * w0a > (unsigned __int128)c0a * wab &&
                              (unsigned __int128)cab * wbn > (unsigned __int128)cbn * wab;
        if (feasible) {
          const double l3 = (la[j] + joint_seg_loss((long long)cab, (long long)wab, tab)) + lr[(long long)b * S + s];
          kr[j] = l1[j] - l3;
          nf++;
        }
      }
    }
    nf = __reduce_add_sync(FULL, nf);
    if (nf > 0) {
      // bitonic sort, position lane * J + j, first keys first
#pragma unroll
      for (int k = 2; k <= 32 * J; k <<= 1) {
#pragma unroll
        for (int st = k >> 1; st > 0; st >>= 1) {
          if (st >= J) {
#pragma unroll
            for (int j = 0; j < J; j++) {
              const int i = lane * J + j;
              const double orr = __shfl_xor_sync(FULL, kr[j], st / J);
              const int os = __shfl_xor_sync(FULL, ks[j], st / J);
              const bool up = (i & k) == 0, lower = (i & st) == 0;
              const bool me_first = joint_first(kr[j], ks[j], orr, os);
              if ((lower == up) != me_first) { kr[j] = orr; ks[j] = os; }
            }
          } else {
#pragma unroll
            for (int j = 0; j < J; j++) {
              const int jp = j ^ st;
              if (jp > j) {
                const bool up = ((lane * J + j) & k) == 0;
                const bool sw = up ? joint_first(kr[jp], ks[jp], kr[j], ks[j]) : joint_first(kr[j], ks[j], kr[jp], ks[jp]);
                if (sw) {
                  const double tr = kr[j]; kr[j] = kr[jp]; kr[jp] = tr;
                  const int ts = ks[j]; ks[j] = ks[jp]; ks[jp] = ts;
                }
              }
            }
          }
        }
      }
      // R_k, the sequential sum of the first k sorted reductions, lane after lane
      double R[J];
      double run = 0.0;
      const int nl = (nf + J - 1) / J;
      for (int l = 0; l < nl; l++) {
        if (lane == l) {
#pragma unroll
          for (int j = 0; j < J; j++) { run = run + kr[j]; R[j] = run; }
        }
        run = __shfl_sync(FULL, run, l);
      }
      const int t = K.t0 + q;
#pragma unroll
      for (int j = 0; j < J; j++) {
        if (kr[j] != -PSD_INF) {
          const double loss = flat - R[j];
          if (loss < best[j]) { best[j] = loss; bt[j] = t; }   // pairs come in increasing t: ties keep the first
        }
      }
    }
    if (++b == N) {
      a++; b = a + 1;
#pragma unroll
      for (int j = 0; j < J; j++) {
        const int s = j * 32 + lane;
        pa[j] = s < S ? pref[(long long)a * S + s] : 0;
        la[j] = s < S ? ll[(long long)a * S + s] : 0.0;
      }
    }
  }
  const int local = c - Q.chunk0;
#pragma unroll
  for (int j = 0; j < J; j++) {
    const int k = lane * J + j + 1;
    if (k <= S) {
      const long long o = Q.cand_off + (long long)(k - 1) * Q.n_chunks + local;
      P.cand_loss[o] = best[j]; P.cand_t[o] = bt[j];
    }
  }
}

__global__ void __launch_bounds__(256) joint_reduce_kernel(const JointParams P) {
  const int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (w >= P.n_items) return;
  const JointItem it = P.items[w];
  const JointProblem Q = P.probs[it.prob];
  const double* cl = P.cand_loss + Q.cand_off + (long long)(it.k - 1) * Q.n_chunks;
  const int* ct = P.cand_t + Q.cand_off + (long long)(it.k - 1) * Q.n_chunks;
  double bl = PSD_INF; int bt = -1;
  for (int c = lane; c < Q.n_chunks; c += 32) {
    const int t = ct[c];
    const double l = cl[c];
    if (t >= 0 && (bt < 0 || l < bl || (l == bl && t < bt))) { bl = l; bt = t; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double l = __shfl_xor_sync(0xffffffffu, bl, o);
    const int t = __shfl_xor_sync(0xffffffffu, bt, o);
    if (t >= 0 && (bt < 0 || l < bl || (l == bl && t < bt))) { bl = l; bt = t; }
  }
  if (lane == 0) { P.out_loss[w] = bl; P.out_t[w] = bt; }
}

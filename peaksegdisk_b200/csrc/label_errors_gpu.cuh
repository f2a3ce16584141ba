// label_errors_gpu.cuh -- label errors of the segmentations a wave has just backtracked (PeakError
// semantics, include/peaksegdisk_b200.h "label errors").
//
// One warp per solved problem, one lane per label (lanes stride over the labels).  The problem's
// compacted segments stay where fpop_backtrack_kernel wrote them (seg_row from seg_offset, last segment
// first): segment s is a peak when s is odd, so peak j starts at boundary seg_row[2j + 1] and ends at
// boundary seg_row[2j], and both sequences decrease with j.  A lane finds its label's o / a / b counts
// with five binary searches over them; nothing is downloaded but the per-label fp / fn and the
// problem's totals.
//
// Units: a boundary in seg_row is a row number r (the segment starts at chromEnd[r]) for row problems
// and a coordinate for count-vector problems.  The host converts each label end x once into a code in
// doubled units of the same grid: 2r when x == chromEnd[r] (2x for count problems), 2r - 1 when x lies
// strictly between chromEnd[r - 1] and chromEnd[r].  A boundary b has the code 2b, so comparing codes
// compares coordinates exactly, on and between the grid points alike.
#pragma once
#include <cuda_runtime.h>

#define PSD_LABEL_WARPS_PER_BLOCK 4

struct LabelDesc { long long off; int n; int pad_; };   // labels [off, off + n) of one GPU problem

struct LabelParams {
  const DpResult* results;
  const int* order;       // the wave's GPU problems
  int n_order;
  const int* seg_row;     // compacted segment boundaries (fpop_backtrack_kernel)
  const LabelDesc* desc;  // per GPU problem
  const int4* labels;     // (start code, end code, kind, 0)
  int* fp; int* fn;       // per label
  int* totals;            // 5 per GPU problem: fp, fn, possible_fp, possible_fn, errors
};

// peaks j in [0, np) whose boundary (which = 1: start, 0: end) has a code below x
__device__ __forceinline__ int peaks_below(const int* seg, int np, int which, long long x) {
  int lo = 0, hi = np;   // first j with 2 * seg[2j + which] < x: the codes decrease with j
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (2ll * seg[2 * mid + which] < x) hi = mid; else lo = mid + 1;
  }
  return np - lo;
}

__global__ void __launch_bounds__(PSD_LABEL_WARPS_PER_BLOCK * 32)
label_errors_kernel(const LabelParams P) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= P.n_order) return;
  const int id = P.order[warp];
  const LabelDesc d = P.desc[id];
  const DpResult* res = &P.results[id];
  if (d.n == 0 || res->status != PSD_ST_OK) return;
  const int* seg = P.seg_row + res->seg_offset;
  const int np = (res->n_segments - 1) / 2;
  int fp = 0, fn = 0, pfp = 0, pfn = 0;
  for (int k = lane; k < d.n; k += 32) {
    const int4 L = P.labels[d.off + k];
    const long long ls = L.x, le = L.y;
    int lfp = 0, lfn = 0;
    if (L.z <= 1) {
      const int o = max(0, peaks_below(seg, np, 1, le) - peaks_below(seg, np, 0, ls + 1));   // ps < le and pe > ls
      if (L.z == 0) lfp = o > 0; else lfn = o == 0;
    } else {
      const int c = L.z == 2 ? peaks_below(seg, np, 1, le) - peaks_below(seg, np, 1, ls)            // ls <= ps < le
                             : peaks_below(seg, np, 0, le + 1) - peaks_below(seg, np, 0, ls + 1);   // ls < pe <= le
      lfp = c > 1; lfn = c == 0;
    }
    P.fp[d.off + k] = lfp; P.fn[d.off + k] = lfn;
    fp += lfp; fn += lfn; pfp += L.z != 1; pfn += L.z != 0;
  }
  fp = __reduce_add_sync(0xffffffffu, fp); fn = __reduce_add_sync(0xffffffffu, fn);
  pfp = __reduce_add_sync(0xffffffffu, pfp); pfn = __reduce_add_sync(0xffffffffu, pfn);
  if (lane == 0) {
    int* t = P.totals + 5ll * id;
    t[0] = fp; t[1] = fn; t[2] = pfp; t[3] = pfn; t[4] = fp + fn;
  }
}

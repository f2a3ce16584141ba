// fpop_warp.cuh -- the PeakSegFPOP dynamic program as warp-cooperative device code (sm_100a).
//
// The two cost functions of the up-down-constrained optimal-partitioning DP are piecewise
// Poisson-loss functions of the log-mean; each is a structure-of-arrays piece list in shared memory
// (a global-memory workspace when a function outgrows it), one lane per piece.  Per bedGraph row
//     up_t   = rescale( min_env( min_less(down_{t-1}) + penalty/W_{t-1}, up_{t-1} ) )
//     down_t = rescale( min_env( min_more(up_{t-1}),                     down_{t-1} ) )
// and the breakpoints/back-pointers of both functions are appended to the cost-function store
// (HBM; spilling through an HBM ring and cudaMemcpyAsync to pinned host memory).  The two
// recursions are independent given row t-1.  This source is compiled TWICE:
//   * fpop_gpu.cu (operator group = 16 lanes): the THROUGHPUT kernel.  One warp owns one problem, its two
//     half-warps run the two recursions side by side through the same code; 14 warps per SM march in
//     phase lock (dp_run_queue).
//   * fpop_lat.cu (-DPSD_G32, operator group = 32 lanes): the LATENCY kernel.  One block owns one
//     problem, one warp per recursion, two helper warps for the second Newton solve and for the
//     second half of wide passes (dp_run_latency, lat_helper_loop).
//
// Reference behaviour being reproduced (file:line into tdhock/PeakSegDisk):
//   piece algebra, Newton roots     src/funPieceListLog.cpp:29-234
//   set_to_min_less_of              src/funPieceListLog.cpp:236-437   -> min_mono_op (dir 0)
//   set_to_min_more_of              src/funPieceListLog.cpp:439-616   -> min_mono_op (dir 1)
//   set_to_min_env_of / push_min_pieces / push_piece
//                                   src/funPieceListLog.cpp:832-1285  -> min_env_op (+ pair_rule)
//   add / multiply / set_prev_seg_end  :618-641  -> fused into the operators' output writes
//   Minimize / findMean             :689-712 / :643-653  -> best_piece / backtrack_problem
//   DP loop, decode                 src/PeakSegFPOPLog.cpp:258-442  -> dp_run_queue, dp_run_latency / backtrack_problem
//   per-row store                   src/PeakSegFPOPLog.cpp:12-141   -> StorePool, StoreRing, store_write (HBM chunk arena)
// Every floating-point expression keeps the reference's operand order and rounding (build with
// -fmad=false); exp/log are psd_math.h, bit-identical to the libm the reference links.
//
// How the sequential operators map onto a warp:
//   * min_less / min_more (one routine, direction = data): lanes evaluate everything that depends on
//     one piece only (end costs, argmin, argmin cost); the scan-order state machine then advances by
//     ballots: "first piece that starts a flat stretch", then "first piece that ends it", the
//     Newton solves of the second question running speculatively in all candidate lanes.
//   * min_env: the overlap intervals of the two breakpoint lists are enumerated with a per-lane
//     binary search + warp scan (a merge path), one lane then owns one interval and applies the
//     crossing rule (0/1/2 roots) independently; the resulting candidate pieces are compacted with
//     a scan and adjacent equal pieces are merged by a run-head pass that reproduces push_piece.
//
// This header is compiled by nvcc for the product and, unmodified, by g++ against
// tests/emu/warp_emu.h (PSD_EMU) where fibers stand in for the lanes of one or several warps -- a test
// tool only.
// Builds: PSD_G32 the latency kernel (above); PSD_TIMING the cycle-counter build (`make timing`, read
// by tools/prof_timing*.py, prof_tail.py, prof_newton_rounds.py); PSD_EMU the emulator, PSD_EMU_STATS
// its operator-size histograms (tools/emu_stats.py).
#pragma once
#include "psd_math.h"

#if defined(PSD_EMU)
#include "warp_emu.h"
#else
#define PSD_DEV __device__ __forceinline__
#define PSD_DEVNI static __device__ __noinline__
PSD_DEV int psd_lane() { return (int)(threadIdx.x & 31u); }
#if defined(PSD_G32)
// latency kernel (fpop_lat.cu): one operator group per WARP -- the up chain and the down chain of a
// problem run on two warps of 32 lanes each, so the group collectives are whole-warp collectives
PSD_DEV int psd_glane() { return (int)(threadIdx.x & 31u); }
PSD_DEV double psd_g_shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
PSD_DEV int psd_g_shfl_i(int v, int src) { return __shfl_sync(0xffffffffu, v, src); }
PSD_DEV double psd_g_shfl_up_d(double v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
PSD_DEV double psd_g_shfl_down_d(double v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
PSD_DEV int psd_g_shfl_up_i(int v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
PSD_DEV unsigned psd_g_ballot(int p) { return __ballot_sync(0xffffffffu, p); }
PSD_DEV void psd_g_sync() { __syncwarp(); }
PSD_DEV void psd_cta_sync() { __syncthreads(); }
PSD_DEV int psd_warp_in_block() { return (int)(threadIdx.x >> 5); }
// named barriers: sync = arrive and wait, arrive = arrive and go on (n = threads of all participating warps)
PSD_DEV void psd_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(n) : "memory"); }
PSD_DEV void psd_bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(n) : "memory"); }
#else
// 16-lane groups: the two half-warps of a problem's warp run the up- and the down-recursion
PSD_DEV int psd_glane() { return (int)(threadIdx.x & 15u); }
PSD_DEV unsigned psd_gmask_() { return 0xffffu << (threadIdx.x & 16u); }
PSD_DEV double psd_g_shfl_d(double v, int src) { return __shfl_sync(psd_gmask_(), v, src, 16); }
PSD_DEV int psd_g_shfl_i(int v, int src) { return __shfl_sync(psd_gmask_(), v, src, 16); }
PSD_DEV double psd_g_shfl_up_d(double v, int d) { return __shfl_up_sync(psd_gmask_(), v, d, 16); }
PSD_DEV double psd_g_shfl_down_d(double v, int d) { return __shfl_down_sync(psd_gmask_(), v, d, 16); }
PSD_DEV int psd_g_shfl_up_i(int v, int d) { return __shfl_up_sync(psd_gmask_(), v, d, 16); }
PSD_DEV unsigned psd_g_ballot(int p) { return (__ballot_sync(psd_gmask_(), p) >> (threadIdx.x & 16u)) & 0xffffu; }
PSD_DEV void psd_g_sync() { __syncwarp(psd_gmask_()); }
#endif
PSD_DEV double psd_shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
PSD_DEV int psd_shfl_i(int v, int src) { return __shfl_sync(0xffffffffu, v, src); }
PSD_DEV unsigned long long psd_shfl_u64(unsigned long long v, int src) { return __shfl_sync(0xffffffffu, v, src); }
PSD_DEV double psd_shfl_up_d(double v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
PSD_DEV double psd_shfl_down_d(double v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
PSD_DEV int psd_shfl_up_i(int v, int d) { return __shfl_up_sync(0xffffffffu, v, d); }
PSD_DEV double psd_shfl_xor_d(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
PSD_DEV int psd_shfl_xor_i(int v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
PSD_DEV unsigned psd_ballot(int p) { return __ballot_sync(0xffffffffu, p); }
PSD_DEV void psd_syncwarp() { __syncwarp(); }
PSD_DEV int psd_ffs(unsigned m) { return __ffs((int)m); }
PSD_DEV int psd_clz(unsigned m) { return __clz((int)m); }
PSD_DEV int psd_popc(unsigned m) { return __popc(m); }
PSD_DEV unsigned long long psd_atomic_add_ull(unsigned long long* p, unsigned long long v) { return atomicAdd(p, v); }
PSD_DEV int psd_atomic_add_int(int* p, int v) { return atomicAdd(p, v); }
// the cost-function store is written once and read (sparsely) once: evict-first streaming stores
PSD_DEV void psd_st_cs_i(int* p, int v) { __stcs(p, v); }
PSD_DEV void psd_st_cs_u64(unsigned long long* p, unsigned long long v) { __stcs(p, v); }
PSD_DEV void psd_st_cs_u4(unsigned* p, unsigned a, unsigned b, unsigned c, unsigned d) { __stcs((uint4*)p, make_uint4(a, b, c, d)); }
PSD_DEV void psd_fence_system() { __threadfence_system(); }
PSD_DEV void psd_fence_device() { __threadfence(); }
// Bulk asynchronous copies shared -> global (the copy engine of the SM moves the bytes; the issuing
// lane goes on).  Sizes are multiples of 16 bytes, both addresses 16-byte aligned.  One lane issues
// the copies of a record as one bulk group and later waits until the engine has READ the sources.
PSD_DEV void psd_bulk_s2g(void* dst_global, const void* src_shared, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               :: "l"(dst_global), "r"((unsigned)__cvta_generic_to_shared(src_shared)), "r"(bytes) : "memory");
}
PSD_DEV void psd_bulk_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }   // lanes' shared-memory writes -> visible to the copy engine
PSD_DEV void psd_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
PSD_DEV void psd_bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }   // all but the newest group have read their sources
PSD_DEV void psd_bulk_wait_read_0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
PSD_DEV void psd_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }           // ... and written their destinations
// a warp waits (one lane spinning) until the host has handed back a ring slot for free-queue position pos
// (gives up after ~10 s without a slot -- a dead host thread must not hang the GPU; the problem then reports status 102)
#define PSD_RING_WAIT(sp, pos) do { unsigned ns_ = 64, spins_ = 0; while (*(sp).ring.free_tail <= (pos) && spins_ < (1u << 20)) { __nanosleep(ns_); if (ns_ < 8192) ns_ <<= 1; spins_++; } } while (0)
#endif

// PSD_TIMING (experiment builds only): per-section cycle counters, accumulated by lane 0 / lane 16
#if defined(PSD_TIMING) && !defined(PSD_EMU)
__device__ unsigned long long psd_dbg[32];
__device__ unsigned long long psd_hist[4][64];   // phase durations per warp and row, 2,048-cycle buckets: [0] min_less/min_more, [1] min_env (<= 32 intervals), [2] min_env (> 32), [3] barrier-to-barrier row time
#define PSD_HIST(slot, cyc) do { if ((threadIdx.x & 31u) == 0) { long long b_ = (long long)(cyc) >> 11; atomicAdd(&psd_hist[slot][b_ < 0 ? 0 : (b_ > 63 ? 63 : b_)], 1ull); } } while (0)
#define PSD_T0(v) const long long v = clock64()
#if defined(PSD_G32)
#define PSD_T1(v, slot) do { if ((threadIdx.x & 31u) == 0) atomicAdd(&psd_dbg[slot], (unsigned long long)(clock64() - v)); } while (0)
#else
#define PSD_T1(v, slot) do { if ((threadIdx.x & 15u) == 0) atomicAdd(&psd_dbg[slot], (unsigned long long)(clock64() - v)); } while (0)
#endif
#else
#define PSD_T0(v) do {} while (0)
#define PSD_T1(v, slot) do {} while (0)
#define PSD_HIST(slot, cyc) do {} while (0)
#endif
// PSD_EMU_STATS (emulator only, tools/emu_stats.py): histograms of the sizes that decide how many
// 16- or 32-lane passes an operator takes -- the source of the waiting at the phase barriers
#if defined(PSD_EMU) && defined(PSD_EMU_STATS)
extern unsigned long long psd_emu_stats[8][65];
#define PSD_STAT(slot, leader, v) do { if (leader) { const int v_ = (v); psd_emu_stats[slot][v_ < 0 ? 0 : (v_ > 64 ? 64 : v_)]++; } } while (0)
#else
#define PSD_STAT(slot, leader, v) do {} while (0)
#endif
#if defined(PSD_G32)
#define PSD_G 32             /* lanes per operator group: a whole warp (latency kernel) */
#else
#define PSD_G 16             /* lanes per operator group (half a warp) */
#endif
#define PSD_EPS 1e-12        /* NEWTON_EPSILON, src/funPieceListLog.cpp:9 */
#define PSD_MAX_STEPS 100    /* NEWTON_STEPS,   src/funPieceListLog.cpp:10 */

// status words a warp can raise for its problem (0 = ok)
#define PSD_ST_OK 0
#define PSD_ST_PIECE_OVERFLOW 101   /* a piece list outgrew the current tier's capacity */
#define PSD_ST_STORE_EXHAUSTED 102  /* the HBM cost-function store ran out of chunks */
#define PSD_ST_BACKTRACK_LOST 103   /* backtrack found no piece containing the mean */
#define PSD_ST_INTERNAL 104         /* a "should never happen" branch of the reference was reached */

// ---- piece list: structure of arrays behind one base pointer --------------------------------------
// doubles [0,cap): a (coef of e^x)  [cap,2cap): b (coef of x)  [2cap,3cap): c (constant)
//         [3cap,4cap): hi (right end of the piece, log-mean)   [4cap,5cap): back_x (prev_log_mean)
// ints at byte offset 40*cap: back_i (data_i).  The left end of piece k is hi[k-1] (domain min for k=0).
struct PList { double* base; int n; };
// Shared-memory tier: the operators are instantiated a second time with the promise that every list
// and scratch pointer is a shared-memory address (32-bit LDS/STS instead of generic 64-bit LD/ST).
#if defined(PSD_EMU)
#define PSD_ASSUME_SHARED(p) do {} while (0)
#else
#define PSD_ASSUME_SHARED(p) __builtin_assume(__isShared((const void*)(p)))
#endif
#define PL_A(L, i) ((L).base[(i)])
#define PL_B(L, i) ((L).base[cap + (i)])
#define PL_C(L, i) ((L).base[2 * cap + (i)])
#define PL_X(L, i) ((L).base[3 * cap + (i)])
#define PL_P(L, i) ((L).base[4 * cap + (i)])
#define PL_I(L, i) (((int*)((L).base + 5 * cap))[(i)])
#define PSD_LIST_BYTES(cap) ((size_t)(cap) * 44)

// Per-warp workspace (shared memory in the fast tier, global memory in the overflow tier):
//   [0,16)  header: int flags (bit 0 = a capacity was exceeded, bit 1 = an impossible branch taken)
//   6 piece lists of `cap` pieces: up_{t-1}, down_{t-1}, up_t, down_t, min-less result, min-more result
//   2 x scratch (one per half-warp group): candidate right ends (ccap doubles), interval codes
//   (2*cap ints: i_f | i_g << 16), candidate sources (ccap ints: bit 30 = from g | piece index).
// The handle is passed BY VALUE (`scratch` already points at the calling group's scratch).
struct WarpWs { unsigned char* base; unsigned char* scratch; int* flags; int cap; int ccap; void* help; };   // help: the chain's LatHelp (latency kernel with helper warps) or null
#define PSD_WS_HDR 16
#define PSD_WS_LISTS 6
#define PSD_FLAG_OVERFLOW 1
#define PSD_FLAG_INTERNAL 2
// one group's scratch: candidate right ends (ccap doubles), interval codes (2*cap ints), candidate
// sources (ccap ints)
#define PSD_WS_SCRATCH_BYTES(cap, ccap) (12ull * (unsigned)(ccap) + 8ull * (unsigned)(cap))
#define PSD_WS_BYTES(cap, ccap) ((PSD_WS_HDR + (unsigned long long)PSD_WS_LISTS * 44ull * (unsigned)(cap) + 2ull * PSD_WS_SCRATCH_BYTES(cap, ccap) + 15ull) & ~15ull)
PSD_DEV double* ws_list(const WarpWs w, int k) { return (double*)(w.base + PSD_WS_HDR + (unsigned long long)k * 44ull * (unsigned)w.cap); }
PSD_DEV unsigned char* ws_scratch0(const WarpWs w) { return w.base + PSD_WS_HDR + (unsigned long long)PSD_WS_LISTS * 44ull * (unsigned)w.cap; }
PSD_DEV double* ws_cand_x(const WarpWs w) { return (double*)w.scratch; }
PSD_DEV int* ws_ivl(const WarpWs w) { return (int*)(ws_cand_x(w) + w.ccap); }
PSD_DEV int* ws_cand_s(const WarpWs w) { return ws_ivl(w) + 2 * w.cap; }
PSD_DEV volatile int* ws_flags(const WarpWs w) { return (volatile int*)w.flags; }
PSD_DEV void ws_raise(const WarpWs w, int flag) { *ws_flags(w) = *ws_flags(w) | flag; }

// exp/log tables: first 4 KB of the block's dynamic shared memory (host arrays under the emulator)
#if defined(PSD_EMU)
#define PSD_ETAB psd_exp_tab_host
#define PSD_LTAB psd_log_tab_host
#else
extern __shared__ __align__(16) unsigned char psd_smem[];
#define PSD_ETAB ((const uint64_t*)psd_smem)
#define PSD_LTAB (((const uint64_t*)psd_smem) + 256)
#endif
PSD_DEVNI double w_exp(double x) { return psd_exp(x, PSD_ETAB); }
PSD_DEVNI double w_log(double x) { return psd_log(x, PSD_LTAB); }

// rescale applied while writing an operator's output:  ((v * mul) + add) * inv  per coefficient,
// i.e. multiply(W_{t-1}); add(w, -z*w, 0); multiply(1/W_t)   (src/PeakSegFPOPLog.cpp:316-321)
struct Rescale { double mul, add_a, add_b, inv; };

PSD_DEV double pc_cost(double a, double b, double c, double x) {
  const double et = (x == -PSD_INF) ? 0.0 : a * w_exp(x);
  const double lt = (b == 0) ? 0.0 : b * x;
  return et + lt + c;
}
// same, when e^x is already known
PSD_DEV double pc_cost_e(double a, double b, double c, double x, double ex) {
  const double et = (x == -PSD_INF) ? 0.0 : a * ex;
  const double lt = (b == 0) ? 0.0 : b * x;
  return et + lt + c;
}
// loss in mean space given log(m) (PoissonLoss, :52-61)
PSD_DEV double pc_cost_m(double a, double b, double c, double m, double logm) {
  const double base = a * m + c;
  if (b == 0) return base;
  const double prod = logm * b;
  return base + prod;
}
PSD_DEV double pc_abs(double v) { return v < 0 ? -v : v; }

// The two big operators are inlined into the kernel body, each at its single call site per tier
// (the executed footprint per phase is unchanged, argument passing through local memory and 320 B of
// spills go away: +1-2 %).  Real functions mattered only before the phase lock, when the warps of
// an SM were at unrelated program counters.  exp/log stay real functions (w_exp / w_log above;
// inlining those loses 3-4 %: they have ~20 call sites).
// The two Newton solvers are inlined into their three call sites (the code per phase stays the same
// size, the 8-double argument shuffle of a call disappears: +4 % on config 2, +6 % on short
// problems, profiles/README.md).
// get_smaller_root (:129-190): Newton in log space from argmin-1.
// x0 = argmin, c0 = cost(x0), cl = cost(lo) are passed in (the reference recomputes the same values).
PSD_DEV double root_left(double a, double b, double c, double lo, double level,
                          double x0, double c0, double cl) {
  if ((level < cl && cl < c0) || (level > cl && cl > c0)) return lo - 1;
  double x = x0 - 1;
  double f, pos_f = PSD_INF, pos_x = PSD_INF, neg_f = -PSD_INF, neg_x = PSD_INF;
  if (c0 < 0) { neg_f = c0; neg_x = x0; } else { pos_f = c0; pos_x = x0; }
  int step = 0;
  do {
    const double et = (x == -PSD_INF) ? 0.0 : a * w_exp(x);
    f = (et + b * x + c) - level;
    if (0 < f && f < pos_f) { pos_f = f; pos_x = x; }
    if (neg_f < f && f < 0) { neg_f = f; neg_x = x; }
    if (PSD_MAX_STEPS <= ++step) {
      const double mid = (pos_x + neg_x) / 2;
      const double em = (mid == -PSD_INF) ? 0.0 : a * w_exp(mid);
      const double fm = (em + b * mid + c) - level;
      return (pc_abs(fm) < pc_abs(f)) ? mid : x;
    }
    const double d = et + b;
    const double off = f / d;
    x = x - off;
  } while (PSD_EPS < pc_abs(f));
  return x;
}

// get_larger_root (:69-127): Newton in mean space from argmin_mean+1; returns log(root).
// m0 = argmin_mean, c0 = PoissonLoss(m0), cr = cost(hi) are passed in.
PSD_DEV double root_right(double a, double b, double c, double hi, double level,
                           double m0, double c0, double cr) {
  if ((c0 < cr && cr < level) || (c0 > cr && cr > level)) return hi + 1;
  double m = m0 + 1;
  double f, pos_f = PSD_INF, pos_m = PSD_INF, neg_f = -PSD_INF, neg_m = PSD_INF;
  if (c0 < 0) { neg_f = c0; neg_m = m0; } else { pos_f = c0; pos_m = m0; }
  int step = 0;
  do {
    f = ((a * m + c) + w_log(m) * b) - level;
    if (0 < f && f < pos_f) { pos_f = f; pos_m = m; }
    if (neg_f < f && f < 0) { neg_f = f; neg_m = m; }
    if (PSD_MAX_STEPS <= ++step) {
      const double mid = (pos_m + neg_m) / 2;
      const double fm = ((a * mid + c) + w_log(mid) * b) - level;
      return (pc_abs(fm) < pc_abs(f)) ? w_log(mid) : w_log(m);
    }
    const double d = a + b / m;
    m = m - f / d;
  } while (PSD_EPS < pc_abs(f));
  return w_log(m);
}

// has_two_roots (:29-50) from the precomputed optimum costs (log-space c1, mean-space c2)
PSD_DEV bool two_roots(double a, double c1, double c2, double level) {
  if (0 < a) return c1 + PSD_EPS < level && c2 + PSD_EPS < level;
  return level + PSD_EPS < c1 && level + PSD_EPS < c2;
}

PSD_DEV bool same_coefs(double a1, double b1, double c1, double a2, double b2, double c2) {  // sameFuns :862-868
  return a1 == a2 && b1 == b2 && pc_abs(c1 - c2) < PSD_EPS;
}

PSD_DEV void pl_emit(const WarpWs ws, const PList out, int k, double a, double b, double c, double hi, double bx, int bi) {
  const int cap = ws.cap;
  if (k < cap) {
    PL_A(out, k) = a; PL_B(out, k) = b; PL_C(out, k) = c; PL_X(out, k) = hi; PL_P(out, k) = bx; PL_I(out, k) = bi;
  } else {
    ws_raise(ws, PSD_FLAG_OVERFLOW);
  }
}

// ---- set_to_min_less_of (dir 0) / set_to_min_more_of (dir 1), one routine --------------------------
// Both are the same scan, mirrored: min_less walks the pieces left to right and keeps the running
// minimum from the left; min_more walks right to left.  In SCAN ORDER (u = 0 is the first piece
// visited) a piece has an entry edge and an exit edge (less: lo/hi, more: hi/lo), the neighbour
// test looks at the next piece's cost at ITS entry edge, a flat stretch opens at the entry edge or
// at the interior argmin and is closed by a root or at an exit edge.  The two half-warps of a warp
// call this routine TOGETHER (dir is group-uniform data), so everything except the root solvers is
// one converged instruction stream.  The reference's asymmetries are kept by selects on dir:
//   * degenerate pieces (b == 0): less may open a flat stretch at one and never closes one on it
//     (:256-308, :376-384); more always copies it and intersects it in closed form (:458-467, :561-564)
//   * less opens at the entry edge only if the cost also rises towards the exit and the next piece
//     (:327-336); more only needs the cost to fall across the piece (:484-510)
//   * less stamps back_i, adds the penalty to c and +0.0 to a and b (add(0,0,c), :618-625); more only stamps
// Output pieces are produced in scan order and, for dir 1, reversed at the end.
template <bool SH>
PSD_DEV int min_mono_op(const WarpWs ws, const PList in, const PList out, double dmin, int stamp, double cshift, int dir) {
  if (SH) { PSD_ASSUME_SHARED(in.base); PSD_ASSUME_SHARED(out.base); PSD_ASSUME_SHARED(ws.scratch); PSD_ASSUME_SHARED(ws.flags); }
  const int lane = psd_glane();   // lane within this 16-lane group
  const int cap = ws.cap;
  const int n = in.n;
  double level = PSD_INF;                             // cost of the pending flat piece; +inf while following the input
  double edge = dir ? PL_X(in, n - 1) : dmin;         // where the next output piece starts (scan order)
  double arg_at = PSD_INF;                            // where the flat piece's minimum is attained
  int out_n = 0;
  int stat_windows = 0;
  PSD_STAT(0, lane == 0, n);
  for (int base = 0; base < n; base += PSD_G) {
    const int u = base + lane;                        // scan position
    const bool valid = u < n;
    const int i = dir ? n - 1 - u : u;                // piece index
    const int end = (n - base < PSD_G) ? n : base + PSD_G;
    double a = 0, b = 0, c = 0, hi = 0, lo = 0;
    double cl = 0, cr = 0, m = 0, mu = 0, cmu = 0, c2 = 0;
    if (valid) {
      a = PL_A(in, i); b = PL_B(in, i); c = PL_C(in, i); hi = PL_X(in, i);
      lo = (i == 0) ? dmin : PL_X(in, i - 1);
      cl = pc_cost(a, b, c, lo);
      cr = pc_cost(a, b, c, hi);
      if (b != 0) {
        m = -b / a;
        mu = w_log(m);
        cmu = pc_cost(a, b, c, mu);
        c2 = pc_cost_m(a, b, c, m, mu);
      }
    }
    const double ein = dir ? hi : lo, eout = dir ? lo : hi;      // entry / exit edge
    const double cin = dir ? cr : cl, cout = dir ? cl : cr;      // cost there
    // cost of the next piece (scan order) at its entry edge, which is my exit edge
    double nxt = psd_g_shfl_down_d(cin, 1);
    const bool has_nxt = u + 1 < n;
    if (lane == PSD_G - 1 && has_nxt) {
      const int j = dir ? i - 1 : i + 1;
      nxt = pc_cost(PL_A(in, j), PL_B(in, j), PL_C(in, j), eout);
    }
    // what this piece does when reached while following the input:
    // 0 = copied whole, 1 = a flat stretch starts at its entry edge, 2 = its minimum is interior
    int kind = 0;
    if (valid) {
      if (b == 0) {
        if (!dir) {
          const bool flat = (cout - cin) < PSD_EPS;
          const bool next_above = !has_nxt || PSD_EPS < nxt - cin;
          kind = (next_above && !flat) ? 1 : 0;
        }
      } else {
        const bool next_ok = !has_nxt || PSD_EPS < nxt - cmu;
        if (!dir) {
          const bool ok = PSD_EPS < cout - cmu && next_ok;
          kind = (mu <= ein && ok) ? 1 : ((mu < eout && ok) ? 2 : 0);
        } else {
          if (ein <= mu) kind = (PSD_EPS < cout - cin) ? 1 : 0;
          else if (eout < mu && PSD_EPS < cout - cmu && next_ok) kind = 2;
        }
      }
    }
    // coefficients of a copied piece
    const double ea = dir ? a : a + 0.0, eb = dir ? b : b + 0.0, ec = dir ? c : c + cshift;
    int pos = base;
    while (pos < end) {
      if (level == PSD_INF) {
        const unsigned mask = psd_g_ballot(valid && u >= pos && kind != 0);
        const int first = mask ? base + psd_ffs(mask) - 1 : end;
        if (valid && u >= pos && u < first) pl_emit(ws, out, out_n + (u - pos), ea, eb, ec, (dir && u == pos) ? edge : hi, PSD_INF, stamp);
        const int src = (first < end) ? first - base : 0;
        const int kf = psd_g_shfl_i(kind, src);
        const double ein_f = psd_g_shfl_d(ein, src), cin_f = psd_g_shfl_d(cin, src);
        const double mu_f = psd_g_shfl_d(mu, src), cmu_f = psd_g_shfl_d(cmu, src);
        const double eout_last = psd_g_shfl_d(eout, end - 1 - base);
        if (first > pos) edge = (first < end) ? ein_f : eout_last;
        out_n += first - pos;
        if (first >= end) { pos = end; break; }
        if (kf == 1) { level = cin_f; arg_at = ein_f; }
        else {
          if (dir ? (mu_f < edge) : (edge < mu_f)) {
            if (lane == src) pl_emit(ws, out, out_n, ea, eb, ec, dir ? edge : mu_f, PSD_INF, stamp);
            out_n++;
          }
          edge = mu_f; arg_at = mu_f; level = cmu_f;
        }
        pos = first + 1;
      } else {
        stat_windows++;
        int flag = 0;
        double r = PSD_INF;   // no root: fails the interval test below
        if (valid && u >= pos && u < pos + PSD_G) {
          if (b == 0) {
            if (dir) r = w_log((level - c) / a);
            else if (a < 0) flag = 3;   // the reference throws here ("should never happen")
          } else if (two_roots(a, cmu, c2, level)) {
            r = dir ? root_right(a, b, c, hi, level, m, c2, cr) : root_left(a, b, c, lo, level, mu, cmu, cl);
          }
          if (flag == 0 && (dir || b != 0)) {
            if (lo < r && r < hi) flag = 1;
            else if (cout <= level + PSD_EPS) flag = 2;
          }
        }
        const unsigned mask = psd_g_ballot(flag != 0);
        if (!mask) { pos = (pos + PSD_G < end) ? pos + PSD_G : end; continue; }   // still flat: next window
        const int src = psd_ffs(mask) - 1;
        const int fl = psd_g_shfl_i(flag, src);
        const double r_s = psd_g_shfl_d(r, src), eout_s = psd_g_shfl_d(eout, src);
        if (fl == 3) { ws_raise(ws, PSD_FLAG_INTERNAL); pos = end; level = PSD_INF; break; }
        const double xe = (fl == 1) ? r_s : eout_s;
        if (lane == 0) pl_emit(ws, out, out_n, dir ? 0.0 : 0.0 + 0.0, dir ? 0.0 : 0.0 + 0.0, dir ? level : level + cshift, dir ? edge : xe, arg_at, stamp);
        out_n++;
        level = PSD_INF; edge = xe;
        pos = base + src + (fl == 1 ? 0 : 1);
      }
    }
  }
  if (level < PSD_INF) {
    if (lane == 0) pl_emit(ws, out, out_n, dir ? 0.0 : 0.0 + 0.0, dir ? 0.0 : 0.0 + 0.0, dir ? level : level + cshift, dir ? edge : PL_X(in, n - 1), arg_at, stamp);
    out_n++;
  }
  PSD_STAT(1, lane == 0, stat_windows);
  psd_g_sync();
  if (dir && out_n <= cap) {   // pieces were produced right to left
    for (int k = lane; k < (out_n >> 1); k += PSD_G) {
      const int j = out_n - 1 - k;
      double t;
      t = PL_A(out, k); PL_A(out, k) = PL_A(out, j); PL_A(out, j) = t;
      t = PL_B(out, k); PL_B(out, k) = PL_B(out, j); PL_B(out, j) = t;
      t = PL_C(out, k); PL_C(out, k) = PL_C(out, j); PL_C(out, j) = t;
      t = PL_X(out, k); PL_X(out, k) = PL_X(out, j); PL_X(out, j) = t;
      t = PL_P(out, k); PL_P(out, k) = PL_P(out, j); PL_P(out, j) = t;
      const int ti = PL_I(out, k); PL_I(out, k) = PL_I(out, j); PL_I(out, j) = ti;
    }
  }
  psd_g_sync();
  return out_n;
}

// ---- push_min_pieces (:870-1259) for one overlap interval, one lane --------------------------------
// Result: nc candidate pieces.  Candidate 0 comes from f if s0 == 0 else from g; candidates
// alternate sources; split points x1 (and x2).   [s0] | x1 | [!s0] | x2 | [s0]
struct PairOut {
  int nc; int s0; double x1, x2;
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
  int two;   // statistics only: this interval ran the two Newton solves
  int heavy; // statistics only: this interval needed more than loads and comparisons
#endif
};

PSD_DEV PairOut pair_rule(const int cap, const PList f, const PList g, int i, int j, double dmin,
                          double* lo_out, double* hi_out) {
  PSD_T0(q0);
  PairOut o; o.nc = 1; o.s0 = 0; o.x1 = 0; o.x2 = 0;
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
  o.two = 0; o.heavy = 0;
#endif
  const double pa = PL_A(f, i), pb = PL_B(f, i), pcst = PL_C(f, i);
  const double qa = PL_A(g, j), qb = PL_B(g, j), qcst = PL_C(g, j);
  const double plo = (i == 0) ? dmin : PL_X(f, i - 1), phi = PL_X(f, i);
  const double qlo = (j == 0) ? dmin : PL_X(g, j - 1), qhi = PL_X(g, j);
  bool eq_left, eq_right;
  double lo, hi;
  if (plo < qlo) { eq_left = same_coefs(PL_A(g, j - 1), PL_B(g, j - 1), PL_C(g, j - 1), pa, pb, pcst); lo = qlo; }
  else {
    lo = plo;
    if (qlo < plo) eq_left = same_coefs(PL_A(f, i - 1), PL_B(f, i - 1), PL_C(f, i - 1), qa, qb, qcst);
    else eq_left = (i == 0 || j == 0) ? false
                   : same_coefs(PL_A(f, i - 1), PL_B(f, i - 1), PL_C(f, i - 1), PL_A(g, j - 1), PL_B(g, j - 1), PL_C(g, j - 1));
  }
  if (phi < qhi) { eq_right = same_coefs(PL_A(f, i + 1), PL_B(f, i + 1), PL_C(f, i + 1), qa, qb, qcst); hi = phi; }
  else {
    hi = qhi;
    if (qhi < phi) eq_right = same_coefs(pa, pb, pcst, PL_A(g, j + 1), PL_B(g, j + 1), PL_C(g, j + 1));
    else eq_right = (i + 1 == f.n || j + 1 == g.n) ? false
                    : same_coefs(PL_A(f, i + 1), PL_B(f, i + 1), PL_C(f, i + 1), PL_A(g, j + 1), PL_B(g, j + 1), PL_C(g, j + 1));
  }
  *lo_out = lo; *hi_out = hi;
  PSD_T1(q0, 16);
  PSD_T0(q1);
  if (lo == hi) { o.nc = 0; return o; }
  if (same_coefs(pa, pb, pcst, qa, qb, qcst)) { o.s0 = 0; return o; }
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
  o.heavy = 1;
#endif
  const double da = pa - qa, db = pb - qb, dc = pcst - qcst;
  const double ehi = w_exp(hi), elo = w_exp(lo);
  const double mid_m = (ehi + elo) / 2;
  const double dmid = pc_cost(da, db, dc, w_log(mid_m));
  const int by_mid = (dmid < 0) ? 0 : 1;
  PSD_T1(q1, 17);
  PSD_T0(q2);
  if (eq_left && eq_right) { o.s0 = by_mid; return o; }
  if (db == 0) {
    if (da == 0) { o.s0 = (dc < 0) ? 0 : 1; return o; }
    if (dc == 0) { o.s0 = (da < 0) ? 0 : 1; return o; }
    const double x = w_log(-dc / da);
    if (lo < x && x < hi) { o.nc = 2; o.x1 = x; o.s0 = (0 < da) ? 0 : 1; return o; }
    o.s0 = by_mid; return o;
  }
  const double dl = pc_cost_e(da, db, dc, lo, elo), dr = pc_cost_e(da, db, dc, hi, ehi);
  const double m = -db / da;
  const double xo = w_log(m);
  const double c1 = pc_cost(da, db, dc, xo);
  const double c2 = pc_cost_m(da, db, dc, m, xo);
  const bool two = two_roots(da, c1, c2, 0.0);
  PSD_T1(q2, 18);
  // Both crossings are always solved, as in the reference (:1024-1027).  Skipping the one a branch
  // below does not read (exact, the solvers are pure) was measured 10 % SLOWER: it splits the lanes
  // of a Newton round into two differently-predicated regions.
  double rs = PSD_INF, rl = PSD_INF;
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
  o.two = two ? 1 : 0;
#endif
  if (two) {
    PSD_T0(tn);
    rs = root_left(da, db, dc, lo, 0.0, xo, c1, dl);
    PSD_T1(tn, 12);
    PSD_T0(tm);
    rl = root_right(da, db, dc, hi, 0.0, m, c2, dr);
    PSD_T1(tm, 13);
  }
  PSD_T0(q3);
  if (eq_right) {
    if (two) {
      if (lo < rs && rs < xo && xo < hi) { o.nc = 2; o.x1 = rs; o.s0 = (dl < 0) ? 0 : 1; return o; }
      const bool f_low_at_zero = 0 < db;
      if (rs < lo) o.s0 = f_low_at_zero ? 1 : 0;
      else o.s0 = f_low_at_zero ? 0 : 1;
      return o;
    }
    o.s0 = by_mid; return o;
  }
  if (eq_left) {
    if (two) {
      if (lo < xo && xo < rl && rl < hi) { o.nc = 2; o.x1 = rl; o.s0 = (dr < 0) ? 1 : 0; return o; }
    }
    o.s0 = by_mid; return o;
  }
  double x1 = PSD_INF, x2 = PSD_INF;
  if (two) {
    const bool l_in = lo < rl && rl < hi;
    const bool s_in = lo < rs && 0 < w_exp(rs) && rs < hi;
    if (l_in) { if (s_in && rs < rl) { x1 = rs; x2 = rl; } else x1 = rl; }
    else if (s_in) x1 = rs;
  }
  if (x2 != PSD_INF) {
    bool f_first;
    if (x2 - x1 < x1 - lo) {
      const double bm = (elo + w_exp(x1)) / 2;
      f_first = pc_cost(da, db, dc, w_log(bm)) < 0;
    } else {
      f_first = !(pc_cost(da, db, dc, (x1 + x2) / 2) < 0);
    }
    o.nc = 3; o.x1 = x1; o.x2 = x2; o.s0 = f_first ? 0 : 1;
  } else if (x1 != PSD_INF) {
    const double bm = (elo + w_exp(x1)) / 2;
    const double before = pc_cost(da, db, dc, w_log(bm));
    const double after = pc_cost(da, db, dc, (hi + x1) / 2);
    if (before < 0) {
      if (after < 0) o.s0 = 0;
      else { o.nc = 2; o.x1 = x1; o.s0 = 0; }
    } else {
      if (after < 0) { o.nc = 2; o.x1 = x1; o.s0 = 1; }
      else o.s0 = 1;
    }
  } else {
    const double v = (pc_abs(dmid) < PSD_EPS) ? dr : dmid;
    o.s0 = (v < 0) ? 0 : 1;
  }
  PSD_T1(q3, 19);
  return o;
}

#define PSD_SRC_G 0x40000000   /* candidate source code: bit 30 = the piece comes from g, low bits = piece index */

#if defined(PSD_G32)
// ---- pair_rule split at the has_two_roots decision (latency kernel) ---------------------------------
// pair_pre() finishes every interval that does not need the two Newton solves and otherwise returns
// the state the solves and the rule's tail need; pair_post() is the tail given both roots.  In
// between, the chain's main warp solves the smaller roots while its HELPER warp solves the larger
// ones (LatHelp): the two Newton loops of an interval run on two warps instead of back to back.
struct PairJob { double da, db, dc, lo, hi, xo, m, c1, c2, dl, dr, elo, dmid; int flags; };   // flags: eq_left | eq_right << 1 | by_mid << 2

PSD_DEV bool pair_pre(const int cap, const PList f, const PList g, int i, int j, double dmin, double* hi_out, PairOut* op, PairJob* job) {
  PairOut o; o.nc = 1; o.s0 = 0; o.x1 = 0; o.x2 = 0;
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
  o.two = 0; o.heavy = 0;
#endif
  const double pa = PL_A(f, i), pb = PL_B(f, i), pcst = PL_C(f, i);
  const double qa = PL_A(g, j), qb = PL_B(g, j), qcst = PL_C(g, j);
  const double plo = (i == 0) ? dmin : PL_X(f, i - 1), phi = PL_X(f, i);
  const double qlo = (j == 0) ? dmin : PL_X(g, j - 1), qhi = PL_X(g, j);
  bool eq_left, eq_right;
  double lo, hi;
  if (plo < qlo) { eq_left = same_coefs(PL_A(g, j - 1), PL_B(g, j - 1), PL_C(g, j - 1), pa, pb, pcst); lo = qlo; }
  else {
    lo = plo;
    if (qlo < plo) eq_left = same_coefs(PL_A(f, i - 1), PL_B(f, i - 1), PL_C(f, i - 1), qa, qb, qcst);
    else eq_left = (i == 0 || j == 0) ? false
                   : same_coefs(PL_A(f, i - 1), PL_B(f, i - 1), PL_C(f, i - 1), PL_A(g, j - 1), PL_B(g, j - 1), PL_C(g, j - 1));
  }
  if (phi < qhi) { eq_right = same_coefs(PL_A(f, i + 1), PL_B(f, i + 1), PL_C(f, i + 1), qa, qb, qcst); hi = phi; }
  else {
    hi = qhi;
    if (qhi < phi) eq_right = same_coefs(pa, pb, pcst, PL_A(g, j + 1), PL_B(g, j + 1), PL_C(g, j + 1));
    else eq_right = (i + 1 == f.n || j + 1 == g.n) ? false
                    : same_coefs(PL_A(f, i + 1), PL_B(f, i + 1), PL_C(f, i + 1), PL_A(g, j + 1), PL_B(g, j + 1), PL_C(g, j + 1));
  }
  *hi_out = hi;
  if (lo == hi) { o.nc = 0; *op = o; return false; }
  if (same_coefs(pa, pb, pcst, qa, qb, qcst)) { o.s0 = 0; *op = o; return false; }
  const double da = pa - qa, db = pb - qb, dc = pcst - qcst;
  const double ehi = w_exp(hi), elo = w_exp(lo);
  const double mid_m = (ehi + elo) / 2;
  const double dmid = pc_cost(da, db, dc, w_log(mid_m));
  const int by_mid = (dmid < 0) ? 0 : 1;
  if (eq_left && eq_right) { o.s0 = by_mid; *op = o; return false; }
  if (db == 0) {
    if (da == 0) { o.s0 = (dc < 0) ? 0 : 1; *op = o; return false; }
    if (dc == 0) { o.s0 = (da < 0) ? 0 : 1; *op = o; return false; }
    const double x = w_log(-dc / da);
    if (lo < x && x < hi) { o.nc = 2; o.x1 = x; o.s0 = (0 < da) ? 0 : 1; *op = o; return false; }
    o.s0 = by_mid; *op = o; return false;
  }
  const double dl = pc_cost_e(da, db, dc, lo, elo), dr = pc_cost_e(da, db, dc, hi, ehi);
  const double m = -db / da;
  const double xo = w_log(m);
  const double c1 = pc_cost(da, db, dc, xo);
  const double c2 = pc_cost_m(da, db, dc, m, xo);
  const bool two = two_roots(da, c1, c2, 0.0);
  if (!two) {   // the rule's tail without roots (:536-582 of pair_rule with two == false)
    if (eq_right || eq_left) o.s0 = by_mid;
    else { const double v = (pc_abs(dmid) < PSD_EPS) ? dr : dmid; o.s0 = (v < 0) ? 0 : 1; }
    *op = o; return false;
  }
  job->da = da; job->db = db; job->dc = dc; job->lo = lo; job->hi = hi; job->xo = xo; job->m = m; job->c1 = c1; job->c2 = c2;
  job->dl = dl; job->dr = dr; job->elo = elo; job->dmid = dmid;
  job->flags = (eq_left ? 1 : 0) | (eq_right ? 2 : 0) | (by_mid ? 4 : 0);
  *op = o;
  return true;
}

// the two Newton solves and the rule's tail for an interval whose difference has two roots
PSD_DEV PairOut pair_post(const PairJob jb, const double rs, const double rl) {
  PairOut o; o.nc = 1; o.s0 = 0; o.x1 = 0; o.x2 = 0;
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
  o.two = 1; o.heavy = 1;
#endif
  const double da = jb.da, db = jb.db, dc = jb.dc, lo = jb.lo, hi = jb.hi, xo = jb.xo, dl = jb.dl, dr = jb.dr, elo = jb.elo;
  const bool eq_left = (jb.flags & 1) != 0, eq_right = (jb.flags & 2) != 0;
  if (eq_right) {
    if (lo < rs && rs < xo && xo < hi) { o.nc = 2; o.x1 = rs; o.s0 = (dl < 0) ? 0 : 1; return o; }
    const bool f_low_at_zero = 0 < db;
    if (rs < lo) o.s0 = f_low_at_zero ? 1 : 0;
    else o.s0 = f_low_at_zero ? 0 : 1;
    return o;
  }
  if (eq_left) {
    if (lo < xo && xo < rl && rl < hi) { o.nc = 2; o.x1 = rl; o.s0 = (dr < 0) ? 1 : 0; return o; }
    o.s0 = (jb.flags & 4) ? 1 : 0; return o;
  }
  double x1 = PSD_INF, x2 = PSD_INF;
  {
    const bool l_in = lo < rl && rl < hi;
    const bool s_in = lo < rs && 0 < w_exp(rs) && rs < hi;
    if (l_in) { if (s_in && rs < rl) { x1 = rs; x2 = rl; } else x1 = rl; }
    else if (s_in) x1 = rs;
  }
  if (x2 != PSD_INF) {
    bool f_first;
    if (x2 - x1 < x1 - lo) {
      const double bm = (elo + w_exp(x1)) / 2;
      f_first = pc_cost(da, db, dc, w_log(bm)) < 0;
    } else {
      f_first = !(pc_cost(da, db, dc, (x1 + x2) / 2) < 0);
    }
    o.nc = 3; o.x1 = x1; o.x2 = x2; o.s0 = f_first ? 0 : 1;
  } else if (x1 != PSD_INF) {
    const double bm = (elo + w_exp(x1)) / 2;
    const double before = pc_cost(da, db, dc, w_log(bm));
    const double after = pc_cost(da, db, dc, (hi + x1) / 2);
    if (before < 0) {
      if (after < 0) o.s0 = 0;
      else { o.nc = 2; o.x1 = x1; o.s0 = 0; }
    } else {
      if (after < 0) { o.nc = 2; o.x1 = x1; o.s0 = 1; }
      else o.s0 = 1;
    }
  } else {
    const double v = (pc_abs(jb.dmid) < PSD_EPS) ? dr : jb.dmid;
    o.s0 = (v < 0) ? 0 : 1;
  }
  return o;
}


// mailbox between a chain's main warp and its helper warp (shared memory)
struct LatHelp {
  int cmd;                 // 1: solve the posted jobs, 2: exit, 3: a wide pass (below)
  unsigned mask;           // lanes that posted a job
  double job[32][8];       // da, db, dc, hi, m, c2, dr of the interval's difference function
  double rl[32];           // the helper's answer: get_larger_root
  // wide pass: a call with more than 32 overlap intervals left hands the second 32 to the helper,
  // which applies the whole crossing rule to them while the main warp does the first 32
  double* f_base; double* g_base; int nf, ng;     // the two functions of the call
  int* ivl; double* cand_x; int* cand_s; int* flags;
  int cap, ccap, K, base, T_in;                   // helper's intervals: [base + 32, base + 64) ∩ [0, K); candidates written so far
  int tot_main, tot_help;                         // candidates of the main warp's / of the helper's 32 intervals
  double dmin;
};
#define PSD_BAR_PAIR 1          /* named barriers of a latency block: the two main warps of the problem */
#define psd_pair_sync() psd_bar_sync(PSD_BAR_PAIR, 64)
#define PSD_BAR_JOBS(g) (2 + (g))   /* chain g: jobs posted (main arrives, helper waits) */
#define PSD_BAR_DONE(g) (4 + (g))   /* chain g: helper's results ready (helper arrives, main waits) */
#define PSD_BAR_MID(g) (6 + (g))    /* chain g, wide pass: the main warp's candidate count is known (main arrives, helper waits) */

PSD_DEV void lat_helper_loop(LatHelp* H, int g) {
  const int lane = psd_lane();
  for (;;) {
    psd_bar_sync(PSD_BAR_JOBS(g), 64);
    const int cmd = *(volatile int*)&H->cmd;
    if (cmd == 2) break;
    if (cmd == 3) {
      // the second 32 intervals of a wide pass: whole crossing rule, candidates appended after the main warp's
      const int cap = H->cap, ccap = H->ccap;
      PList F, G;
      F.base = H->f_base; F.n = H->nf; G.base = H->g_base; G.n = H->ng;
      const int q = H->base + 32 + lane;
      const bool valid = q < H->K;
      PairOut o; o.nc = 0; o.s0 = 0; o.x1 = 0; o.x2 = 0;
      double lo = 0, hi = 0;
      int i = 0, j = 0;
      if (valid) {
        const int code = H->ivl[q];
        i = code & 0xffff; j = code >> 16;
        o = pair_rule(cap, F, G, i, j, H->dmin, &lo, &hi);
      }
      const int nc = valid ? o.nc : 0;
      int incl = nc;
      for (int d = 1; d < 32; d <<= 1) { const int t = psd_g_shfl_up_i(incl, d); if (lane >= d) incl += t; }
      const int tot = psd_g_shfl_i(incl, 31);
      psd_bar_sync(PSD_BAR_MID(g), 64);       // the main warp's count is in the mailbox
      const int off = H->T_in + *(volatile int*)&H->tot_main + incl - nc;
      if (nc > 0) {
        const int sf = i, sg = j | PSD_SRC_G;
        const int c0 = o.s0 ? sg : sf, c1 = o.s0 ? sf : sg;
        if (off + nc <= ccap) {
          H->cand_s[off] = c0; H->cand_x[off] = (nc > 1) ? o.x1 : hi;
          if (nc > 1) { H->cand_s[off + 1] = c1; H->cand_x[off + 1] = (nc > 2) ? o.x2 : hi; }
          if (nc > 2) { H->cand_s[off + 2] = c0; H->cand_x[off + 2] = hi; }
        } else *(volatile int*)H->flags = *(volatile int*)H->flags | PSD_FLAG_OVERFLOW;
      }
      if (lane == 0) H->tot_help = tot;
      psd_syncwarp();
      psd_bar_arrive(PSD_BAR_DONE(g), 64);
      continue;
    }
    const unsigned m = *(volatile unsigned*)&H->mask;
    if ((m >> lane) & 1u) {
      const double* J = H->job[lane];
      H->rl[lane] = root_right(J[0], J[1], J[2], J[3], 0.0, J[4], J[5], J[6]);
    }
    psd_bar_arrive(PSD_BAR_DONE(g), 64);
  }
}
#endif



// ---- set_to_min_env_of(f, g) followed by the row rescale -------------------------------------------
// f is the freshly built min-less/min-more function, g the previous cost function; of / og are the
// same two lists of the OTHER chain (the call is converged over both half-warps and stage 2 pools
// the intervals of both chains over all 32 lanes).
template <bool SH>
PSD_DEV int min_env_op(const WarpWs ws, const PList f, const PList g, const PList of, const PList og, const PList out,
                       double dmin, const Rescale rs) {
  if (SH) {
    PSD_ASSUME_SHARED(f.base); PSD_ASSUME_SHARED(g.base); PSD_ASSUME_SHARED(of.base); PSD_ASSUME_SHARED(og.base);
    PSD_ASSUME_SHARED(out.base); PSD_ASSUME_SHARED(ws.scratch); PSD_ASSUME_SHARED(ws.flags);
  }
  const int lane = psd_glane();   // lane within this 16-lane group
  const int cap = ws.cap, ccap = ws.ccap;
  int* const ivl = ws_ivl(ws);
  double* const cand_x = ws_cand_x(ws);
  int* const cand_s = ws_cand_s(ws);
  const int nf = f.n, ng = g.n;
  PSD_T0(t1);
  // 1. enumerate overlap intervals, one g piece per lane: f pieces s..e overlap g[j]
  int K = 0;
  {
    int carry_next = 0;   // first f piece that can overlap the next g piece
    for (int base = 0; base < ng; base += PSD_G) {
      const int j = base + lane;
      const bool valid = j < ng;
      int e = 0, tie = 0;
      if (valid) {
        const double v = PL_X(g, j);
        int lo_i = 0, hi_i = nf - 1;    // lower_bound: first f piece whose right end >= v
        while (lo_i < hi_i) {
          const int mid = (lo_i + hi_i) >> 1;
          if (PL_X(f, mid) < v) lo_i = mid + 1; else hi_i = mid;
        }
        e = lo_i;
        tie = (PL_X(f, e) == v) ? 1 : 0;
      }
      int s = psd_g_shfl_up_i(e + tie, 1);
      if (lane == 0) s = carry_next;
      int cnt = valid ? (e - s + 1) : 0;
      if (cnt < 0) cnt = 0;
      // exclusive scan of cnt
      int incl = cnt;
      for (int d = 1; d < PSD_G; d <<= 1) { const int t = psd_g_shfl_up_i(incl, d); if (lane >= d) incl += t; }
      const int off = K + incl - cnt;
      for (int q = 0; q < cnt; q++) {
        if (off + q < 2 * cap) ivl[off + q] = (s + q) | (j << 16); else ws_raise(ws, PSD_FLAG_OVERFLOW);
      }
      K += psd_g_shfl_i(incl, PSD_G - 1);
      carry_next = psd_g_shfl_i(e + tie, (ng - base < PSD_G) ? ng - base - 1 : PSD_G - 1);
    }
  }
  if (K > 2 * cap) { K = 2 * cap; }
  PSD_STAT(2, lane == 0, ng);
  PSD_STAT(3, lane == 0, K);
  psd_syncwarp();   // both chains' interval lists are visible to the whole warp
  PSD_T1(t1, 8);
  PSD_T0(t2);
#if defined(PSD_G32)
  // 2. crossing rule per interval -> candidate pieces: one lane per interval of THIS chain (the
  // chain has the whole warp to itself in the latency kernel; of / og are unused).  Intervals whose
  // difference function has two roots post their get_larger_root to the chain's helper warp and
  // solve get_smaller_root themselves meanwhile.
  int T = 0;
  LatHelp* const H = (LatHelp*)ws.help;
  const int chain = psd_warp_in_block() & 1;
  for (int base = 0; base < K; base += 32) {
    if (H && K - base > 32) {
      // WIDE pass: more than 32 intervals left (functions of more than ~16 pieces: high penalties,
      // the worst-case sequences).  The helper warp takes intervals [base + 32, base + 64) with the whole
      // crossing rule while this warp does [base, base + 32): 64 intervals per pass.
      if (lane == 0) {
        H->f_base = f.base; H->g_base = g.base; H->nf = nf; H->ng = ng; H->ivl = ivl; H->cand_x = cand_x; H->cand_s = cand_s;
        H->flags = (int*)ws.flags; H->cap = cap; H->ccap = ccap; H->K = K; H->base = base; H->T_in = T; H->dmin = dmin; H->cmd = 3;
      }
      psd_syncwarp();
      psd_bar_arrive(PSD_BAR_JOBS(chain), 64);
      const int code = ivl[base + lane];
      const int i = code & 0xffff, j = code >> 16;
      double lo = 0, hi = 0;
      const PairOut o = pair_rule(cap, f, g, i, j, dmin, &lo, &hi);
      int incl = o.nc;
      for (int d = 1; d < 32; d <<= 1) { const int t = psd_g_shfl_up_i(incl, d); if (lane >= d) incl += t; }
      const int tot = psd_g_shfl_i(incl, 31);
      if (lane == 0) H->tot_main = tot;
      psd_syncwarp();
      psd_bar_arrive(PSD_BAR_MID(chain), 64);
      const int off = T + incl - o.nc;
      if (o.nc > 0) {
        const int sf = i, sg = j | PSD_SRC_G;
        const int c0 = o.s0 ? sg : sf, c1 = o.s0 ? sf : sg;
        if (off + o.nc <= ccap) {
          cand_s[off] = c0; cand_x[off] = (o.nc > 1) ? o.x1 : hi;
          if (o.nc > 1) { cand_s[off + 1] = c1; cand_x[off + 1] = (o.nc > 2) ? o.x2 : hi; }
          if (o.nc > 2) { cand_s[off + 2] = c0; cand_x[off + 2] = hi; }
        } else ws_raise(ws, PSD_FLAG_OVERFLOW);
      }
      psd_bar_sync(PSD_BAR_DONE(chain), 64);
      T += tot + *(volatile int*)&H->tot_help;
      base += 32;       // (the loop adds the other 32)
      continue;
    }
    const int q = base + lane;
    const bool valid = q < K;
    PairOut o; o.nc = 0; o.s0 = 0; o.x1 = 0; o.x2 = 0;
#if defined(PSD_TIMING) || defined(PSD_EMU_STATS)
    o.two = 0; o.heavy = 0;
#endif
    PairJob jb; jb.da = jb.db = jb.dc = jb.lo = jb.hi = jb.xo = jb.m = jb.c1 = jb.c2 = jb.dl = jb.dr = jb.elo = jb.dmid = 0; jb.flags = 0;
    double hi = 0;
    int i = 0, j = 0;
    bool need = false;
    if (valid) {
      const int code = ivl[q];
      i = code & 0xffff; j = code >> 16;
      need = pair_pre(cap, f, g, i, j, dmin, &hi, &o, &jb);
    }
    if (H) {
      const unsigned nm = psd_g_ballot(need);
      if (nm) {
        if (need) { double* J = H->job[lane]; J[0] = jb.da; J[1] = jb.db; J[2] = jb.dc; J[3] = jb.hi; J[4] = jb.m; J[5] = jb.c2; J[6] = jb.dr; }
        psd_syncwarp();
        if (lane == 0) { H->mask = nm; H->cmd = 1; }
        psd_bar_arrive(PSD_BAR_JOBS(chain), 64);
        double rs = 0;
        if (need) rs = root_left(jb.da, jb.db, jb.dc, jb.lo, 0.0, jb.xo, jb.c1, jb.dl);
        psd_bar_sync(PSD_BAR_DONE(chain), 64);
        if (need) o = pair_post(jb, rs, H->rl[lane]);
      }
    } else if (need) {
      const double rs = root_left(jb.da, jb.db, jb.dc, jb.lo, 0.0, jb.xo, jb.c1, jb.dl);
      const double rl = root_right(jb.da, jb.db, jb.dc, jb.hi, 0.0, jb.m, jb.c2, jb.dr);
      o = pair_post(jb, rs, rl);
    }
    const int mine_nc = valid ? o.nc : 0;
    int incl = mine_nc;
    for (int d = 1; d < 32; d <<= 1) { const int t = psd_g_shfl_up_i(incl, d); if (lane >= d) incl += t; }
    const int tot = psd_g_shfl_i(incl, 31);
    const int off = T + incl - mine_nc;
    if (o.nc > 0) {
      const int sf = i, sg = j | PSD_SRC_G;
      const int c0 = o.s0 ? sg : sf, c1 = o.s0 ? sf : sg;
      if (off + o.nc <= ccap) {
        cand_s[off] = c0; cand_x[off] = (o.nc > 1) ? o.x1 : hi;
        if (o.nc > 1) { cand_s[off + 1] = c1; cand_x[off + 1] = (o.nc > 2) ? o.x2 : hi; }
        if (o.nc > 2) { cand_s[off + 2] = c0; cand_x[off + 2] = hi; }
      } else ws_raise(ws, PSD_FLAG_OVERFLOW);
    }
    T += tot;
  }
#else
  // 2. crossing rule per interval -> candidate pieces.  The intervals of BOTH chains (this call is
  // converged: lanes 0-15 hold the up chain's arguments, lanes 16-31 the down chain's) are pooled
  // over the 32 lanes: a chain with 20 intervals next to one with 10 takes one pass, not two, and
  // the other warps of the block wait at the phase barrier for one pass less (profiles/README.md).
  int T = 0;
  {
    const int wl = psd_lane();
    const int grp = wl >> 4;
    // the other chain's scratch: same layout, the neighbouring scratch block
    double* const of_base = of.base;
    double* const og_base = og.base;
    const int onf = of.n, ong = og.n, oK = psd_shfl_i(K, wl ^ 16);
    WarpWs ows = ws;
    ows.scratch = grp ? ws.scratch - PSD_WS_SCRATCH_BYTES(cap, ccap) : ws.scratch + PSD_WS_SCRATCH_BYTES(cap, ccap);
    int* const oivl = ws_ivl(ows);
    double* const ocand_x = ws_cand_x(ows);
    int* const ocand_s = ws_cand_s(ows);
    // NOTE: no PSD_ASSUME_SHARED(ows.scratch) here.  With that assumption on the derived pointer nvcc
    // 12.9 generated code that read the wrong scratch block (every min_env came out with one piece;
    // the emulator build was fine, bisected on the GPU).  The few cross-chain accesses stay generic.
    const int K0 = grp ? oK : K, K1 = grp ? K : oK;     // intervals of the up / of the down chain
    const int total = K0 + K1;
    PSD_STAT(4, wl == 0, total);
    int T0 = 0, T1 = 0;
#if defined(PSD_TIMING) && !defined(PSD_EMU)
    int stat_jobs = 0, stat_rounds = 0;
#endif
#if defined(PSD_EMU_STATS)
    int stat_heavy = 0, stat_two = 0;
#endif
    for (int base = 0; base < total; base += 32) {
      const int q = base + wl;
      const bool valid = q < total;
      const int c = (valid && q >= K0) ? 1 : 0;           // which chain this lane works for in this pass
      const int qi = c ? q - K0 : q;
      const bool mine = (c == grp);
      PList F, G;
      F.base = mine ? f.base : of_base; F.n = mine ? nf : onf;
      G.base = mine ? g.base : og_base; G.n = mine ? ng : ong;
      if (SH) { PSD_ASSUME_SHARED(F.base); PSD_ASSUME_SHARED(G.base); }
      PairOut o; o.nc = 0; o.s0 = 0; o.x1 = 0; o.x2 = 0;
      double lo = 0, hi = 0;
      int i = 0, j = 0;
#if defined(PSD_EMU_STATS)
      o.two = 0; o.heavy = 0;
#endif
#if defined(PSD_TIMING) && !defined(PSD_EMU)
      o.two = 0;
      if (wl == 0) atomicAdd(&psd_dbg[20], 1ull);
      if (valid) atomicAdd(&psd_dbg[21], 1ull);
#endif
      if (valid) {
        const int code = (mine ? ivl : oivl)[qi];
        i = code & 0xffff; j = code >> 16;
        o = pair_rule(cap, F, G, i, j, dmin, &lo, &hi);
      }
#if defined(PSD_TIMING) && !defined(PSD_EMU)
      {
        const unsigned tw = psd_ballot(valid && o.two);
        stat_jobs += psd_popc(tw); stat_rounds += tw ? 1 : 0;
      }
#endif
#if defined(PSD_EMU_STATS)
      stat_heavy += psd_popc(psd_ballot(valid && o.heavy)); stat_two += psd_popc(psd_ballot(valid && o.two));
#endif
      // exclusive scan of the candidate counts, per chain: both counts ride in one int (<= 96 each)
      const int mine_nc = valid ? o.nc : 0;
      int incl = c ? (mine_nc << 16) : mine_nc;
      for (int d = 1; d < 32; d <<= 1) { const int t = psd_shfl_up_i(incl, d); if (wl >= d) incl += t; }
      const int tot = psd_shfl_i(incl, 31);
      const int off = c ? T1 + (incl >> 16) - mine_nc : T0 + (incl & 0xffff) - mine_nc;
      if (o.nc > 0) {
        double* const CX = mine ? cand_x : ocand_x;
        int* const CS = mine ? cand_s : ocand_s;
        const int sf = i, sg = j | PSD_SRC_G;
        const int c0 = o.s0 ? sg : sf, c1 = o.s0 ? sf : sg;
        if (off + o.nc <= ccap) {
          CS[off] = c0; CX[off] = (o.nc > 1) ? o.x1 : hi;
          if (o.nc > 1) { CS[off + 1] = c1; CX[off + 1] = (o.nc > 2) ? o.x2 : hi; }
          if (o.nc > 2) { CS[off + 2] = c0; CX[off + 2] = hi; }
        } else ws_raise(ws, PSD_FLAG_OVERFLOW);
      }
      T0 += tot & 0xffff; T1 += tot >> 16;
    }
    T = grp ? T1 : T0;
#if defined(PSD_EMU_STATS)
    PSD_STAT(6, wl == 0, stat_heavy);
    PSD_STAT(7, wl == 0, stat_two);
#endif
#if defined(PSD_TIMING) && !defined(PSD_EMU)
    if (wl == 0) {
      atomicAdd(&psd_dbg[22], (unsigned long long)stat_jobs);
      atomicAdd(&psd_dbg[23], (unsigned long long)stat_rounds);
      atomicAdd(&psd_dbg[24], 1ull);
      if (stat_rounds) atomicAdd(&psd_dbg[25], 1ull);
      atomicAdd(&psd_dbg[26], (unsigned long long)((stat_jobs + 31) / 32));   // rounds a compacted job list needs
      if (total > 32) atomicAdd(&psd_dbg[27], 1ull);
    }
#endif
  }
#endif
  psd_syncwarp();   // every candidate of my chain is in place, whichever half-warp wrote it
  PSD_T1(t2, 9);
  PSD_T0(t3);
  if (T > ccap) T = ccap;
  PSD_STAT(5, lane == 0, T);
  // 3. push_piece: merge each candidate into the current run when it equals the run's head
  int out_n = 0;
  bool carry_ok = false;
  double ha = 0, hb = 0, hc = 0, hp = 0; int hi_i = 0;   // head of the run open at the chunk boundary
  int carry_slot = 0;
  for (int base = 0; base < T; base += PSD_G) {
    const int q = base + lane;
    const bool valid = q < T;
    double a = 0, b = 0, c = 0, p = 0, x = 0; int bi = 0;
    if (valid) {
      const int code = cand_s[q];
      x = cand_x[q];
      const int k = code & 0xffffff;
      if (code & PSD_SRC_G) { a = PL_A(g, k); b = PL_B(g, k); c = PL_C(g, k); p = PL_P(g, k); bi = PL_I(g, k); }
      else { a = PL_A(f, k); b = PL_B(f, k); c = PL_C(f, k); p = PL_P(f, k); bi = PL_I(f, k); }
    }
    // first guess: a candidate continues the run iff it equals its immediate predecessor
    double pa_ = psd_g_shfl_up_d(a, 1), pb_ = psd_g_shfl_up_d(b, 1), pc_ = psd_g_shfl_up_d(c, 1), pp_ = psd_g_shfl_up_d(p, 1);
    int pi_ = psd_g_shfl_up_i(bi, 1);
    bool pv = lane > 0;
    if (lane == 0) { pa_ = ha; pb_ = hb; pc_ = hc; pp_ = hp; pi_ = hi_i; pv = carry_ok; }
    bool head = valid && !(pv && same_coefs(pa_, pb_, pc_, a, b, c) && p == pp_ && bi == pi_);
    // verify against the true run heads (push_piece compares with the list's last piece, whose
    // coefficients are those of the run's first member); repair the first disagreement and retry
    for (;;) {
      const unsigned hm = psd_g_ballot(head);
      const unsigned below = hm & ((1u << lane) - 1u);
      const int hl = below ? 31 - psd_clz(below) : -1;   // head of the run candidate q-1 belongs to
      double ra = psd_g_shfl_d(a, hl < 0 ? 0 : hl), rb = psd_g_shfl_d(b, hl < 0 ? 0 : hl), rc = psd_g_shfl_d(c, hl < 0 ? 0 : hl);
      double rp = psd_g_shfl_d(p, hl < 0 ? 0 : hl);
      int ri = psd_g_shfl_i(bi, hl < 0 ? 0 : hl);
      bool rv = true;
      if (hl < 0) { ra = ha; rb = hb; rc = hc; rp = hp; ri = hi_i; rv = carry_ok; }
      const bool want_head = valid && !(rv && same_coefs(ra, rb, rc, a, b, c) && p == rp && bi == ri);
      const unsigned bad = psd_g_ballot(valid && want_head != head);
      if (!bad) break;
      if (lane == psd_ffs(bad) - 1) head = want_head;
    }
    const unsigned hm = psd_g_ballot(head);
    const unsigned vm = psd_g_ballot(valid);
    const int rank = psd_popc(hm & ((1u << lane) - 1u));
    const unsigned upto = hm & ((2u << lane) - 1u);       // heads at or below this lane
    const int my_head = upto ? 31 - psd_clz(upto) : -1;
    const int slot = (my_head < 0) ? carry_slot : out_n + psd_popc(hm & ((1u << my_head) - 1u));
    if (head) {
      const double na = ((a * rs.mul) + rs.add_a) * rs.inv;
      const double nb = ((b * rs.mul) + rs.add_b) * rs.inv;
      const double nc = ((c * rs.mul) + 0.0) * rs.inv;
      if (out_n + rank < cap) {
        const PList o = out;
        PL_A(o, out_n + rank) = na; PL_B(o, out_n + rank) = nb; PL_C(o, out_n + rank) = nc;
        PL_P(o, out_n + rank) = p; PL_I(o, out_n + rank) = bi;
      } else ws_raise(ws, PSD_FLAG_OVERFLOW);
    }
    // the last member of every run (within this chunk) sets the run's right end
    const bool last_valid = valid && (lane == PSD_G - 1 || !((vm >> (lane + 1)) & 1u));
    const bool next_is_head = (lane < PSD_G - 1) && ((hm >> (lane + 1)) & 1u);
    if (valid && (last_valid || next_is_head)) { if (slot < cap) PL_X(out, slot) = x; }
    // carry the open run into the next chunk
    const int n_heads = psd_popc(hm);
    if (n_heads) {
      const int last_head = 31 - psd_clz(hm);
      ha = psd_g_shfl_d(a, last_head); hb = psd_g_shfl_d(b, last_head); hc = psd_g_shfl_d(c, last_head);
      hp = psd_g_shfl_d(p, last_head); hi_i = psd_g_shfl_i(bi, last_head);
      carry_slot = out_n + n_heads - 1;
      carry_ok = true;
    }
    out_n += n_heads;
  }
  psd_g_sync();
  PSD_T1(t3, 10);
  return out_n;
}

// copy with rescale (rows 0/1 of the DP, src/PeakSegFPOPLog.cpp:297-299, 324-328)
template <bool SH>
PSD_DEVNI int copy_rescale_op(const WarpWs ws, const PList in, const PList out, const Rescale rs) {
  if (SH) { PSD_ASSUME_SHARED(in.base); PSD_ASSUME_SHARED(out.base); }
  const int lane = psd_glane();   // lane within this 16-lane group
  const int cap = ws.cap;
  for (int k = lane; k < in.n; k += PSD_G) {
    PL_A(out, k) = ((PL_A(in, k) * rs.mul) + rs.add_a) * rs.inv;
    PL_B(out, k) = ((PL_B(in, k) * rs.mul) + rs.add_b) * rs.inv;
    PL_C(out, k) = ((PL_C(in, k) * rs.mul) + 0.0) * rs.inv;
    PL_X(out, k) = PL_X(in, k); PL_P(out, k) = PL_P(in, k); PL_I(out, k) = PL_I(in, k);
  }
  psd_g_sync();
  return in.n;
}

// ---- Minimize (:689-712): first piece with the strictly smallest clamped-argmin cost ---------------
PSD_DEVNI void best_piece(const WarpWs ws, const PList f, double dmin, double* best_c, double* best_x, int* back_i, double* back_x) {
  const int lane = psd_lane();
  const int cap = ws.cap;
  double bc = PSD_INF, bx = 0, bpx = 0; int bbi = 0; int bidx = 0x7fffffff;
  for (int base = 0; base < f.n; base += 32) {
    const int i = base + lane;
    double cc = PSD_INF, x = 0;
    if (i < f.n) {
      const double a = PL_A(f, i), b = PL_B(f, i), c = PL_C(f, i), hi = PL_X(f, i);
      const double lo = (i == 0) ? dmin : PL_X(f, i - 1);
      x = w_log(-b / a);
      if (x < lo) x = lo; else if (hi < x) x = hi;
      cc = pc_cost(a, b, c, x);
      if (!(cc < PSD_INF)) cc = PSD_INF;   // NaN/inf are never selected
    }
    if (cc < bc) { bc = cc; bx = x; bidx = i; bbi = PL_I(f, i); bpx = PL_P(f, i); }
  }
  for (int d = 16; d >= 1; d >>= 1) {
    const double oc = psd_shfl_xor_d(bc, d), ox = psd_shfl_xor_d(bx, d), op = psd_shfl_xor_d(bpx, d);
    const int oi = psd_shfl_xor_i(bidx, d), ob = psd_shfl_xor_i(bbi, d);
    if (oc < bc || (oc == bc && oi < bidx)) { bc = oc; bx = ox; bpx = op; bidx = oi; bbi = ob; }
  }
  *best_c = bc; *best_x = bx; *back_i = bbi; *back_x = bpx;
}

// ---- HBM cost-function store ------------------------------------------------------------------------
// A pool of fixed-size chunks; a warp appends its rows' records to its current chunk and takes a new
// one (atomicAdd on the pool cursor) when the next record does not fit.  Record of row t, 16-byte
// aligned, every array padded to a multiple of 16 bytes (U = n_up rounded up to 2, Ui = to 4; D, Di alike):
//   u32 n_up | u32 n_down | u32 row | u32 0
//   f64 up.hi[U] | f64 up.back_x[U] | f64 down.hi[D] | f64 down.back_x[D] | i32 up.back_i[Ui] | i32 down.back_i[Di]
// These are the arrays of the shared-memory piece lists as they lie there, so a record is written by
// SIX BULK COPIES shared -> global (cp.async.bulk) issued by one lane; the lists are not overwritten
// before row t+2, by which time the copy engine has read them.  (Lists in the global-memory tier and
// records that go to host memory through the mapping are written by the lanes instead.)
// index[t] = byte offset of the record in the pool.  The reference's record
// (src/PeakSegFPOPLog.cpp:12-34) carries the same fields at 8 + 20 bytes per piece per function.
// When the HBM pool is exhausted and a pinned host region is configured the store SPILLS: chunk numbers
// past the HBM region address the host region (the backtrack reads the few records it needs through
// the mapping).  How the records get there:
//   * DMA drain (default): such a chunk is written into a slot of an HBM RING; when the warp leaves
//     the chunk it publishes (host chunk, slot) in a pinned done-queue, a host thread copies the slot
//     to its place in the host region with cudaMemcpyAsync on a side stream and hands the slot back
//     through a pinned free-queue.  The DP's stores stay HBM stores; PCIe sees 64 KB DMA transfers.
//   * zero-copy (ring off, or records larger than a chunk): the lanes' stores go through the mapping.
struct StoreRing {
  unsigned char* base;                      // HBM ring: n_slots slots of chunk_bytes (n_slots = 0: ring off)
  unsigned long long n_slots;
  unsigned long long* head;                 // device counter: next free-queue position to take
  unsigned long long* done_head;            // device counter: next done-queue position to fill
  volatile unsigned long long* free_tail;   // pinned, written by the host: free-queue positions below this are valid
  volatile unsigned int* free_q;            // pinned, written by the host: slot ids
  volatile unsigned long long* done_q;      // pinned, written by the device: { position + 1, host chunk << 32 | slot }
  unsigned int q_mask;
};
struct StorePool {
  unsigned char* base;            // HBM region
  unsigned long long* cursor;     // next free HBM chunk
  unsigned long long n_chunks;
  unsigned long long chunk_bytes;
  unsigned char* host_base;       // device-visible pinned host region (null: no spill)
  unsigned long long* host_cursor;   // zero-copy chunks handed out (from the top of the host region when the ring is on)
  unsigned long long host_chunks;
  StoreRing ring;
};
struct StoreWriter { unsigned long long cur, end; long long slot; };   // slot: ring slot of the open chunk, -1 = none

struct RecLayout { unsigned hi[2], bx[2], bi[2]; };   // byte offsets of the six arrays inside a record
PSD_HD RecLayout rec_layout(int n_up, int n_down) {
  const unsigned U = (unsigned)(n_up + 1) & ~1u, D = (unsigned)(n_down + 1) & ~1u, Ui = (unsigned)(n_up + 3) & ~3u;
  RecLayout L;
  L.hi[0] = 16u; L.bx[0] = 16u + 8u * U; L.hi[1] = 16u + 16u * U; L.bx[1] = 16u + 16u * U + 8u * D;
  L.bi[0] = 16u + 16u * (U + D); L.bi[1] = L.bi[0] + 4u * Ui;
  return L;
}
PSD_DEV unsigned long long store_record_bytes(int n_up, int n_down) {
  const unsigned long long U = (unsigned long long)((n_up + 1) & ~1), D = (unsigned long long)((n_down + 1) & ~1);
  const unsigned long long Ui = (unsigned long long)((n_up + 3) & ~3), Di = (unsigned long long)((n_down + 3) & ~3);
  return 16ull + 16ull * (U + D) + 4ull * (Ui + Di);
}

// ONE thread: publish the ring chunk a writer is leaving (its stores must already be visible system-wide)
PSD_DEV void store_ring_publish(const StorePool& sp, unsigned long long host_chunk, long long slot) {
  const unsigned long long pos = psd_atomic_add_ull(sp.ring.done_head, 1ull);
  volatile unsigned long long* e = sp.ring.done_q + 2ull * (pos & sp.ring.q_mask);
  e[1] = (host_chunk << 32) | (unsigned long long)slot;
  psd_fence_system();
  e[0] = pos + 1ull;
}

// ONE thread: take `need` contiguous chunks.  Returns the first chunk number (~0: exhausted); *slot
// receives the ring slot when the chunk has to be written through the ring.
PSD_DEV unsigned long long store_take(const StorePool& sp, unsigned long long need, long long* slot) {
  *slot = -1;
  const unsigned long long first = psd_atomic_add_ull(sp.cursor, need);
  if (first + need <= sp.n_chunks) return first;
  if (sp.host_chunks == 0) return ~0ull;
  if (sp.ring.n_slots != 0 && need == 1) {
    const unsigned long long pos = psd_atomic_add_ull(sp.ring.head, 1ull);
    // host chunks: ring positions from the bottom, zero-copy allocations from the top.  Each side bumps
    // its own counter, fences, then reads the other's: of two allocations racing for the last chunks at
    // least one sees the other and gives up, so they can never be handed the same chunk.
    psd_fence_device();
    if (pos + 1ull + *(volatile unsigned long long*)sp.host_cursor > sp.host_chunks) return ~0ull;
    PSD_RING_WAIT(sp, pos);
    if (*sp.ring.free_tail <= pos) return ~0ull;
    psd_fence_system();   // the slot id was written before free_tail was advanced
    *slot = (long long)sp.ring.free_q[pos & sp.ring.q_mask];
    return sp.n_chunks + pos;
  }
  const unsigned long long h = psd_atomic_add_ull(sp.host_cursor, need);
  if (sp.ring.n_slots == 0) return (h + need > sp.host_chunks) ? ~0ull : sp.n_chunks + h;
  psd_fence_device();
  if (h + need + *(volatile unsigned long long*)sp.ring.head > sp.host_chunks) return ~0ull;
  return sp.n_chunks + sp.host_chunks - h - need;
}

// the writer's open chunk, if it is a ring chunk, is complete: make the warp's stores visible, publish
PSD_DEV void store_close(const StorePool& sp, StoreWriter& w) {
  if (w.slot < 0) return;
  if (psd_lane() == 0) psd_bulk_wait_all();   // bulk copies into the chunk have landed
  psd_fence_system();
  psd_syncwarp();
  if (psd_lane() == 0) store_ring_publish(sp, w.end / sp.chunk_bytes - 1ull - sp.n_chunks, w.slot);
  w.slot = -1;
}

// returns the record offset or ~0 when the pool is exhausted
PSD_DEV unsigned long long store_alloc(const StorePool& sp, StoreWriter& w, unsigned long long bytes) {
  if (w.cur + bytes > w.end) {
    const unsigned long long need = (bytes + sp.chunk_bytes - 1) / sp.chunk_bytes;
    store_close(sp, w);
    unsigned long long first = 0; long long slot = -1;
    if (psd_lane() == 0) first = store_take(sp, need, &slot);
    first = psd_shfl_u64(first, 0);
    slot = (long long)psd_shfl_u64((unsigned long long)slot, 0);
    if (first == ~0ull) return ~0ull;
    w.slot = slot;
    w.cur = first * sp.chunk_bytes;
    w.end = w.cur + need * sp.chunk_bytes;
  }
  const unsigned long long off = w.cur;
  w.cur += bytes;
  return off;
}

// where a record at offset `off` is READ (backtrack, inspection): HBM or the pinned host region
PSD_DEV unsigned char* store_ptr(const StorePool& sp, unsigned long long off) {
  const unsigned long long hbm = sp.n_chunks * sp.chunk_bytes;
  return off < hbm ? sp.base + off : sp.host_base + (off - hbm);
}
// where the writer WRITES the record it just allocated: its ring slot while the chunk is open
PSD_DEV unsigned char* store_wptr(const StorePool& sp, const StoreWriter& w, unsigned long long off) {
  if (w.slot >= 0) return sp.ring.base + (unsigned long long)w.slot * sp.chunk_bytes + (off - (w.end - sp.chunk_bytes));
  return store_ptr(sp, off);
}

// one function of a record written by lanes (global-tier lists, or a destination in host memory)
template <bool SH>
PSD_DEV void store_fn_lanes(const WarpWs ws, unsigned char* rec, const RecLayout R, const PList L, int which, int lane, int n_lanes) {
  if (SH) PSD_ASSUME_SHARED(L.base);
  const int cap = ws.cap;
  double* hi = (double*)(rec + R.hi[which]); double* bx = (double*)(rec + R.bx[which]); int* bi = (int*)(rec + R.bi[which]);
  for (int k = lane; k < L.n; k += n_lanes) { hi[k] = PL_X(L, k); bx[k] = PL_P(L, k); psd_st_cs_i(bi + k, PL_I(L, k)); }
}
// ... and by three bulk copies shared -> global (issued by ONE lane, after psd_bulk_fence)
PSD_DEV void store_fn_bulk(const WarpWs ws, unsigned char* rec, const RecLayout R, const PList L, int which) {
  const int cap = ws.cap;
  if (L.n == 0) return;
  const unsigned nd = 8u * ((unsigned)(L.n + 1) & ~1u), ni = 4u * ((unsigned)(L.n + 3) & ~3u);
  psd_bulk_s2g(rec + R.hi[which], &PL_X(L, 0), nd);
  psd_bulk_s2g(rec + R.bx[which], &PL_P(L, 0), nd);
  psd_bulk_s2g(rec + R.bi[which], &PL_I(L, 0), ni);
}

#if !defined(PSD_G32)
// bulk: the lists are in shared memory and the record in device memory
template <bool SH>
PSD_DEV void store_write(const WarpWs ws, unsigned char* rec, int row, const PList up, const PList down, bool bulk) {
  const int lane = psd_lane();
  const RecLayout R = rec_layout(up.n, down.n);
  if (lane == 0) psd_st_cs_u4((unsigned*)rec, (unsigned)up.n, (unsigned)down.n, (unsigned)row, 0u);
  if (SH && bulk) {
    // the lists were completed before the phase barrier; one lane hands them to the copy engine
    if (lane == 0) {
      psd_bulk_fence();
      store_fn_bulk(ws, rec, R, up, 0);
      store_fn_bulk(ws, rec, R, down, 1);
      psd_bulk_commit();
      psd_bulk_wait_read_1();   // the record of row t-1 has left its lists (they are written again in row t+1)
    }
    return;
  }
  // lanes 0-15 write the up function, lanes 16-31 the down function
  store_fn_lanes<SH>(ws, rec, R, (lane >> 4) ? down : up, lane >> 4, lane & 15, 16);
}
#endif

// per-problem result of the DP (device -> host), and of the backtrack
struct DpResult {
  int status;
  int back_i;                 // Minimize(): last row of the previous segment
  double best_cost;           // mean penalized cost
  double best_x;              // log-mean of the last segment
  double back_x;
  unsigned long long total_intervals;
  int max_intervals;
  int n_segments;
  int n_equality;
  int pad_;
  unsigned long long seg_offset;   // where the backtrack kernel put this problem's segments
  unsigned long long bt_bytes;     // record + index bytes the backtrack read (8 + 16 + 20 per piece of the function used)
};

// optional per-row trace for tests (null in production): called by lane 0 after every row
#if defined(PSD_EMU)
typedef void (*psd_trace_fn)(void* user, int row, int which, int n, int cap, const double* base);
#endif

struct DpProblem {
  const int* weight;          // chromEnd - chromStart per row
  const int* coverage;
  int n_rows;
  double penalty;
  double dmin, dmax;          // log(min coverage), log(max coverage)
  unsigned long long* index;  // n_rows record offsets
};

// ---- the DP driver: a block of warps works through a queue of problems in PHASE LOCK ----------------
// Each warp owns one problem at a time (src/PeakSegFPOPLog.cpp:258-397 + Minimize at :404) and pops
// the next one from an atomic queue when it finishes.
//
// Inside a row the two recursions are independent given row t-1:
//     up_t   = rescale(min_env(min_less(down_{t-1}) + penalty/W, up_{t-1}))      lanes  0-15
//     down_t = rescale(min_env(min_more(up_{t-1}),               down_{t-1}))    lanes 16-31
// so the warp's two 16-lane groups run them side by side: the min_env calls of both groups are ONE
// converged call (same code, different lists), which halves the issue slots and the latency of the
// most expensive operator; min_less / min_more are different code and overlap only in latency.
//
// The warps of a block are independent, but they cross a block barrier between the phases of a row
// so that at any moment all warps of the SM execute the SAME operators: the DP's code (~110 KB of
// SASS) is several times the instruction cache, and without the phase lock 84 % of all stall
// samples were instruction fetch (profiles/README.md).  Rows need not be aligned, only phases.
#if defined(PSD_EMU)
#define psd_block_sync() do {} while (0)
#define psd_block_or(x) (x)
#else
#define psd_block_sync() __syncthreads()
#define psd_block_or(x) __syncthreads_or(x)
#endif

// Copies list `src` (n pieces, capacity scap) into list `dst` (capacity dcap); all 32 lanes.
PSD_DEV void pl_move(const double* src, int scap, double* dst, int dcap, int n) {
  for (int k = psd_lane(); k < n; k += 32) {
    for (int a = 0; a < 5; a++) dst[a * dcap + k] = src[a * scap + k];
    ((int*)(dst + 5 * dcap))[k] = ((const int*)(src + 5 * scap))[k];
  }
}

// A problem running from its global workspace (in_g) returns to shared memory (capacity cap_s,
// 0 = disabled) once both functions fill at most half of it.
PSD_DEV bool back_to_shared(bool in_g, int n_up, int n_down, int cap_s) {
  return in_g && cap_s > 0 && 2 * n_up <= cap_s && 2 * n_down <= cap_s;
}

#if !defined(PSD_G32)
// order[] lists problem ids longest first.  Slot q = warp_in_block * n_blocks + block is taken
// statically by that warp (so the longest problems land one per SM and a small batch spreads over
// all SMs instead of filling a few blocks); the rest are popped from the atomic cursor, which the
// host initialises to n_blocks * warps_per_block.
struct DpQueue {
  const DpProblem* problems;
  const int* order;
  int n_order;
  int* cursor;
  DpResult* results;
  int first_slot;        // this warp's static slot
};

// ws_s: the warp's shared-memory workspace (cap 0 = disabled), ws_g: its global-memory workspace
// (cap 0 = none).  A problem runs from shared memory; when a row's functions outgrow it the warp
// moves the two previous functions to the global workspace and REPEATS THAT ROW there (the
// operators never write their inputs), and moves back once both functions fit comfortably again.
// NOTE: the aggregates are taken by const reference on purpose.  Taken by value, nvcc 12.9 handed this
// (force-inlined) function a DpQueue whose last member was garbage once StorePool grew to 56 bytes
// (the caller's copy was intact); found with device printf, see profiles/README.md.
PSD_DEV void dp_run_queue(const WarpWs& ws_s, const WarpWs& ws_g, const DpQueue& Q, const StorePool& sp
#if defined(PSD_EMU)
                          , psd_trace_fn trace, void* trace_user
#endif
) {
  const int lane = psd_lane();
  const int grp = lane >> 4;          // 0: up chain (min_less), 1: down chain (min_more)
  // per-warp state (uniform across lanes)
  int have = 0, id = 0, t = 0, N = 0, status = PSD_ST_OK, max_iv = 0, w_l = 0, z_l = 0, n_spill = 0;
  const int* weight = nullptr; const int* coverage = nullptr; unsigned long long* index = nullptr;
  double penalty = 0, dmin = 0, dmax = 0, cw = 0, cw_done = 0.0;
  unsigned long long total_iv = 0, my_off = 0;
  bool in_g = ws_s.cap == 0;          // current tier
  WarpWs ws = in_g ? ws_g : ws_s;
  WarpWs wg = ws;                     // this group's view: its own scratch
  PList upP, downP, upN, downN, tmp;
  upP.n = downP.n = upN.n = downN.n = tmp.n = 0;
#define PSD_BIND_TIER()                                                                              \
  do {                                                                                               \
    ws = in_g ? ws_g : ws_s;                                                                         \
    wg = ws;                                                                                         \
    wg.scratch = ws_scratch0(ws) + (unsigned long long)grp * PSD_WS_SCRATCH_BYTES(ws.cap, ws.ccap);  \
    upP.base = ws_list(ws, 0); downP.base = ws_list(ws, 1); upN.base = ws_list(ws, 2);               \
    downN.base = ws_list(ws, 3); tmp.base = ws_list(ws, 4 + grp);                                    \
  } while (0)
  PSD_BIND_TIER();
  StoreWriter sw; sw.cur = 0; sw.end = 0; sw.slot = -1;
  Rescale rs; rs.mul = rs.add_a = rs.add_b = rs.inv = 0;
  bool fetch = true;
  int first_q = Q.first_slot;
  for (;;) {
    // ---- phase A: (next problem,) next row; min_less on group 0 | min_more on group 1 -----------------
    if (fetch) {
      int q = first_q;   // the first problem of every warp is assigned statically (see DpQueue)
      first_q = -1;
      if (q < 0) {
        if (lane == 0) q = psd_atomic_add_int(Q.cursor, 1);
        q = psd_shfl_i(q, 0);
      }
      have = q < Q.n_order;
      fetch = false;
      if (have) {
        id = Q.order[q];
        const DpProblem pb = Q.problems[id];
        weight = pb.weight; coverage = pb.coverage; index = pb.index; N = pb.n_rows;
        penalty = pb.penalty; dmin = pb.dmin; dmax = pb.dmax;
        t = 0; status = PSD_ST_OK; max_iv = 0; total_iv = 0; cw = 0.0; cw_done = 0.0; n_spill = 0;
        in_g = ws_s.cap == 0;
        PSD_BIND_TIER();
        upP.n = downP.n = upN.n = downN.n = tmp.n = 0;
        if (lane == 0) *ws_flags(ws) = 0;
        psd_syncwarp();
      }
    }
    if (have) {
      if ((t & 31) == 0) {   // coalesced load of the next 32 rows
        const int r = t + lane;
        w_l = (r < N) ? weight[r] : 0;
        z_l = (r < N) ? coverage[r] : 0;
      }
      const int wi = psd_shfl_i(w_l, t & 31), z = psd_shfl_i(z_l, t & 31);
      const double w = (double)wi;
      cw = cw_done + w;
      rs.mul = cw_done; rs.add_a = w; rs.add_b = (double)(-z) * w; rs.inv = 1 / cw;
      if (t == 0) {
        if (lane == 0) pl_emit(ws, downP, 0, 1.0, (double)(-z), 0.0, dmax, -5.0, -1);
        downP.n = 1; upP.n = 0;
        psd_syncwarp();
      } else if (grp == 0 || t >= 2) {
        // min_less(down_{t-1}) on group 0 and min_more(up_{t-1}) on group 1: one converged call
        PSD_T0(ta);
        tmp.n = in_g ? min_mono_op<false>(wg, grp ? upP : downP, tmp, dmin, t - 1, penalty / cw_done, grp)
                     : min_mono_op<true>(wg, grp ? upP : downP, tmp, dmin, t - 1, penalty / cw_done, grp);
        PSD_T1(ta, grp);
#if defined(PSD_TIMING) && !defined(PSD_EMU)
        PSD_HIST(0, clock64() - ta);
#endif
      }
    }
    // block barrier 1 of 2; it doubles as the block's termination vote (a warp that just saw an empty
    // queue has have == 0; the block leaves when every warp has)
    PSD_T0(tw1);
    const int any_have = psd_block_or(have);
    PSD_T1(tw1, 5);     // wait at barrier 1 (after min_less / min_more)
    if (!any_have) break;
    // ---- phase B: both min_env's as one converged call --------------------------------------------------
    int n_out = 0;
    if (have && t >= 1) {
      const PList prev = grp ? downP : upP;     // previous cost function of my chain
      const PList dst = grp ? downN : upN;
      if (t == 1) n_out = in_g ? copy_rescale_op<false>(wg, grp ? downP : tmp, dst, rs) : copy_rescale_op<true>(wg, grp ? downP : tmp, dst, rs);   // :297-299, :324-328
      else {
        PSD_T0(tb);
        PList otmp; otmp.base = ws_list(ws, 4 + (grp ^ 1)); otmp.n = psd_shfl_i(tmp.n, lane ^ 16);   // the other chain's lists
        const PList oprev = grp ? upP : downP;
        n_out = in_g ? min_env_op<false>(wg, tmp, prev, otmp, oprev, dst, dmin, rs)
                     : min_env_op<true>(wg, tmp, prev, otmp, oprev, dst, dmin, rs);
        PSD_T1(tb, 2 + grp);
#if defined(PSD_TIMING) && !defined(PSD_EMU)
        PSD_HIST((tmp.n + prev.n + otmp.n + oprev.n > 36) ? 2 : 1, clock64() - tb);   // (pieces of the four lists: a proxy for > 32 overlap intervals)
#endif
      }
      psd_syncwarp();   // both chains done; their lists are visible to the whole warp
    }
    PSD_T0(tw2);
    psd_block_sync();   // block barrier 2 of 2
    PSD_T1(tw2, 6);     // wait at barrier 2 (after min_env)
    // ---- phase C: tier switch or: counters, store record, end of problem --------------------------------
    PSD_T0(tc);
    if (have) {
      const int flags = *ws_flags(ws);
      bool redo = false;
      if (flags) {
        if ((flags & PSD_FLAG_OVERFLOW) && !(flags & PSD_FLAG_INTERNAL) && !in_g && ws_g.cap > 0) {
          // this row does not fit the shared-memory tier: repeat it from the global workspace
          if (lane == 0) psd_bulk_wait_read_0();   // no record copy is still reading the shared-memory lists
          psd_syncwarp();
          pl_move(upP.base, ws_s.cap, ws_list(ws_g, 0), ws_g.cap, upP.n);
          pl_move(downP.base, ws_s.cap, ws_list(ws_g, 1), ws_g.cap, downP.n);
          if (lane == 0) *ws_flags(ws) = 0;
          in_g = true; n_spill++;
          PSD_BIND_TIER();
          psd_syncwarp();
          redo = true;
        } else {
          status = (flags & PSD_FLAG_INTERNAL) ? PSD_ST_INTERNAL : PSD_ST_PIECE_OVERFLOW;
        }
      }
      if (!redo) {
        if (status == PSD_ST_OK) {
          if (t >= 1) {   // the new functions become the previous ones
            upN.n = psd_shfl_i(n_out, 0);
            downN.n = psd_shfl_i(n_out, 16);
            const PList u = upP, d = downP;
            upP = upN; downP = downN; upN = u; downN = d;
          }
          cw_done = cw;
          total_iv += (unsigned long long)(upP.n + downP.n);
          if (max_iv < upP.n) max_iv = upP.n;
          if (max_iv < downP.n) max_iv = downP.n;
#if defined(PSD_EMU)
          if (trace && lane == 0) { trace(trace_user, t, 0, upP.n, ws.cap, upP.base); trace(trace_user, t, 1, downP.n, ws.cap, downP.base); }
#endif
          const unsigned long long off = store_alloc(sp, sw, store_record_bytes(upP.n, downP.n));
          if (off == ~0ull) status = PSD_ST_STORE_EXHAUSTED;
          else {
            // bulk copies need a device-memory destination: HBM, or the writer's ring slot
            const bool dev_dst = sw.slot >= 0 || off < sp.n_chunks * sp.chunk_bytes;
            if (in_g) store_write<false>(ws, store_wptr(sp, sw, off), t, upP, downP, false);
            else store_write<true>(ws, store_wptr(sp, sw, off), t, upP, downP, dev_dst);
            if (lane == (t & 31)) my_off = off;
            if ((t & 31) == 31 || t == N - 1) {
              const int r = (t & ~31) + lane;
              if (r <= t) psd_st_cs_u64(index + r, my_off);
            }
          }
        }
        t++;
        if (status != PSD_ST_OK || t == N) {
          double bc = 0, bx = 0, bpx = 0; int bbi = -1;
          if (status == PSD_ST_OK) best_piece(ws, downP, dmin, &bc, &bx, &bbi, &bpx);
          if (lane == 0) psd_bulk_wait_read_0();   // the next problem starts in the same lists
          if (lane == 0) {
            DpResult* res = &Q.results[id];
            res->status = status; res->back_i = bbi; res->best_cost = bc; res->best_x = bx; res->back_x = bpx;
            res->total_intervals = total_iv; res->max_intervals = max_iv; res->n_segments = 0; res->n_equality = 0;
            res->pad_ = n_spill;
          }
          fetch = true;
        } else if (back_to_shared(in_g, upP.n, downP.n, ws_s.cap)) {
          // both functions fit comfortably again: move back to shared memory
          psd_syncwarp();
          pl_move(upP.base, ws_g.cap, ws_list(ws_s, 0), ws_s.cap, upP.n);
          pl_move(downP.base, ws_g.cap, ws_list(ws_s, 1), ws_s.cap, downP.n);
          in_g = false;
          PSD_BIND_TIER();
          psd_syncwarp();
        }
      }
    }
    PSD_T1(tc, 4);

  }
  store_close(sp, sw);   // a ring chunk still open when the warp retires goes to the host like the others
#undef PSD_BIND_TIER
}
#endif   // !PSD_G32

#if defined(PSD_G32)
// ---- latency mode: one problem per thread block, one chain per warp ---------------------------------
// When a batch has fewer problems than the GPU has warp slots (one long chromosome, a sequential
// search, the worst-case sequences), one warp per problem leaves the chip idle and the problem's
// rows are a single chain of dependent fp64 instructions.  Here a block of two warps owns the
// problem: warp 0 runs the up recursion (min_less, min_env), warp 1 the down recursion (min_more,
// min_env), each with all 32 lanes (functions of up to 32 pieces / 32 overlap intervals take one
// pass), their Newton solves overlap instead of serialising on two half-warps, and the piece lists
// have the block's whole shared memory (hundreds of pieces before the global tier is needed).
// A chain reads the other chain's PREVIOUS function only in min_less / min_more, so the two warps
// meet at ONE block barrier per row.  Same operators, same arithmetic, same record format.
struct LatShared {
  int n_out[2][2];                  // [row parity][chain]: pieces of the new function
  unsigned long long chunk_first;   // store chunk handed out by warp 0 to both warps
  long long chunk_slot;             // its ring slot (-1: none)
  LatHelp help[2];                  // mailboxes of the two helper warps (warps 2 and 3 of the block)
};

// store chunk allocation for the block: both warps keep identical StoreWriter state; the chunk is
// taken (and a ring chunk being left is published) once, by warp 0, and the result passed through
// shared memory.  Both warps write into the open chunk, so both make their stores visible first.
PSD_DEV unsigned long long store_alloc_cta(const StorePool& sp, StoreWriter& w, unsigned long long bytes, LatShared* sh, int grp) {
  if (w.cur + bytes > w.end) {
    const unsigned long long need = (bytes + sp.chunk_bytes - 1) / sp.chunk_bytes;
    if (w.slot >= 0) { if (psd_lane() == 0) psd_bulk_wait_all(); psd_fence_system(); psd_pair_sync(); }
    if (grp == 0 && psd_lane() == 0) {
      if (w.slot >= 0) store_ring_publish(sp, w.end / sp.chunk_bytes - 1ull - sp.n_chunks, w.slot);
      long long slot = -1;
      sh->chunk_first = store_take(sp, need, &slot);
      sh->chunk_slot = slot;
    }
    psd_pair_sync();
    const unsigned long long first = *(volatile unsigned long long*)&sh->chunk_first;
    w.slot = *(volatile long long*)&sh->chunk_slot;
    if (first == ~0ull) { w.slot = -1; return ~0ull; }
    w.cur = first * sp.chunk_bytes;
    w.end = w.cur + need * sp.chunk_bytes;
  }
  const unsigned long long off = w.cur;
  w.cur += bytes;
  return off;
}

// one function's part of a row's record, written by that chain's warp (layout: see StorePool)
template <bool SH>
PSD_DEV void store_write_fn(const WarpWs ws, unsigned char* rec, int row, const PList L, int which, int n_up, int n_down, bool bulk) {
  const int lane = psd_lane();
  const RecLayout R = rec_layout(n_up, n_down);
  if (which == 0 && lane == 0) psd_st_cs_u4((unsigned*)rec, (unsigned)n_up, (unsigned)n_down, (unsigned)row, 0u);
  if (SH && bulk) {
    if (lane == 0) {
      psd_bulk_fence();
      store_fn_bulk(ws, rec, R, L, which);
      psd_bulk_commit();
      psd_bulk_wait_read_1();
    }
    return;
  }
  store_fn_lanes<SH>(ws, rec, R, L, which, lane, 32);
}

// use_help: warps 2 and 3 of the block run lat_helper_loop() for chains 0 and 1
PSD_DEV void dp_run_latency(const WarpWs& ws_s, const WarpWs& ws_g, const DpProblem& pb, DpResult* res, const StorePool& sp, LatShared* sh, const bool use_help
#if defined(PSD_EMU)
                            , psd_trace_fn trace, void* trace_user
#endif
) {
  const int lane = psd_lane();
  const int grp = psd_warp_in_block();   // 0: up chain (min_less), 1: down chain (min_more)
  const int N = pb.n_rows;
  const int* weight = pb.weight; const int* coverage = pb.coverage; unsigned long long* index = pb.index;
  const double penalty = pb.penalty, dmin = pb.dmin, dmax = pb.dmax;
  int t = 0, status = PSD_ST_OK, max_iv = 0, w_l = 0, z_l = 0, n_spill = 0;
  double cw = 0, cw_done = 0.0;
  unsigned long long total_iv = 0, my_off = 0;
  bool in_g = ws_s.cap == 0;
  WarpWs ws, wg;
  PList upP, downP, upN, downN, tmp;
  upP.n = downP.n = upN.n = downN.n = tmp.n = 0;
  // four flag words (the workspace header): [2 * row parity + chain].  A warp only ever writes its own
  // words; the words of row t are read by both warps after row t's barrier and zeroed by their
  // owner at the start of row t + 2, one barrier later.
  int* const flag_words = ws_s.flags;
#define PSD_BIND_TIER()                                                                              \
  do {                                                                                               \
    ws = in_g ? ws_g : ws_s;                                                                         \
    wg = ws;                                                                                         \
    wg.scratch = ws_scratch0(ws) + (unsigned long long)grp * PSD_WS_SCRATCH_BYTES(ws.cap, ws.ccap);  \
    wg.flags = flag_words + 2 * (t & 1) + grp;                                                       \
    wg.help = use_help ? (void*)&sh->help[grp] : nullptr;                                            \
    upP.base = ws_list(ws, 0); downP.base = ws_list(ws, 1); upN.base = ws_list(ws, 2);               \
    downN.base = ws_list(ws, 3); tmp.base = ws_list(ws, 4 + grp);                                    \
  } while (0)
  PSD_BIND_TIER();
  StoreWriter sw; sw.cur = 0; sw.end = 0; sw.slot = -1;
  Rescale rs; rs.mul = rs.add_a = rs.add_b = rs.inv = 0;
  for (;;) {
    wg.flags = flag_words + 2 * (t & 1) + grp;
    if (lane == 0) *wg.flags = 0;
    psd_syncwarp();
    if ((t & 31) == 0) {   // coalesced load of the next 32 rows (both warps keep their own copy)
      const int r = t + lane;
      w_l = (r < N) ? weight[r] : 0;
      z_l = (r < N) ? coverage[r] : 0;
    }
    const int wi = psd_shfl_i(w_l, t & 31), z = psd_shfl_i(z_l, t & 31);
    const double w = (double)wi;
    cw = cw_done + w;
    rs.mul = cw_done; rs.add_a = w; rs.add_b = (double)(-z) * w; rs.inv = 1 / cw;
    int n_out = 0;
    if (t == 0) {
      if (grp == 1 && lane == 0) pl_emit(wg, downP, 0, 1.0, (double)(-z), 0.0, dmax, -5.0, -1);
      downP.n = 1; upP.n = 0;
    } else {
      // my chain of row t: min_less(down_{t-1}) / min_more(up_{t-1}), then the envelope with my own
      // previous function; nothing here depends on what the other warp computes for row t
      PSD_T0(ta);
      if (grp == 0 || t >= 2)
        tmp.n = in_g ? min_mono_op<false>(wg, grp ? upP : downP, tmp, dmin, t - 1, penalty / cw_done, grp)
                     : min_mono_op<true>(wg, grp ? upP : downP, tmp, dmin, t - 1, penalty / cw_done, grp);
      PSD_T1(ta, grp);
      const PList prev = grp ? downP : upP;
      const PList dst = grp ? downN : upN;
      PSD_T0(tb);
      if (t == 1) n_out = in_g ? copy_rescale_op<false>(wg, grp ? downP : tmp, dst, rs) : copy_rescale_op<true>(wg, grp ? downP : tmp, dst, rs);
      else n_out = in_g ? min_env_op<false>(wg, tmp, prev, tmp, prev, dst, dmin, rs) : min_env_op<true>(wg, tmp, prev, tmp, prev, dst, dmin, rs);
      PSD_T1(tb, 2 + grp);
      if (lane == 0) sh->n_out[t & 1][grp] = n_out;
    }
    PSD_T0(tw);
    psd_pair_sync();   // the row's one barrier: both new functions are complete and visible
    PSD_T1(tw, 5);
    PSD_T0(tc);
    const int flags = ((volatile int*)flag_words)[2 * (t & 1)] | ((volatile int*)flag_words)[2 * (t & 1) + 1];
    bool redo = false;
    if (flags) {
      if ((flags & PSD_FLAG_OVERFLOW) && !(flags & PSD_FLAG_INTERNAL) && !in_g && ws_g.cap > 0) {
        // this row does not fit the shared-memory tier: repeat it from the global workspace
        if (lane == 0) psd_bulk_wait_read_0();   // no record copy is still reading the shared-memory lists
        if (grp == 0) pl_move(upP.base, ws_s.cap, ws_list(ws_g, 0), ws_g.cap, upP.n);
        else pl_move(downP.base, ws_s.cap, ws_list(ws_g, 1), ws_g.cap, downP.n);
        in_g = true; n_spill++;
        PSD_BIND_TIER();
        psd_pair_sync();   // both warps have read the flag words and moved their function
        redo = true;
      } else {
        status = (flags & PSD_FLAG_INTERNAL) ? PSD_ST_INTERNAL : PSD_ST_PIECE_OVERFLOW;
      }
    }
    if (redo) continue;
    if (status == PSD_ST_OK) {
      if (t >= 1) {   // the new functions become the previous ones
        upN.n = ((volatile int*)sh->n_out[t & 1])[0];
        downN.n = ((volatile int*)sh->n_out[t & 1])[1];
        const PList u = upP, d = downP;
        upP = upN; downP = downN; upN = u; downN = d;
      }
      cw_done = cw;
      total_iv += (unsigned long long)(upP.n + downP.n);
      if (max_iv < upP.n) max_iv = upP.n;
      if (max_iv < downP.n) max_iv = downP.n;
#if defined(PSD_EMU)
      if (trace && lane == 0 && grp == 0) { trace(trace_user, t, 0, upP.n, ws.cap, upP.base); trace(trace_user, t, 1, downP.n, ws.cap, downP.base); }
#endif
      const unsigned long long off = store_alloc_cta(sp, sw, store_record_bytes(upP.n, downP.n), sh, grp);
      if (off == ~0ull) status = PSD_ST_STORE_EXHAUSTED;
      else {
        const bool dev_dst = sw.slot >= 0 || off < sp.n_chunks * sp.chunk_bytes;
        if (in_g) store_write_fn<false>(ws, store_wptr(sp, sw, off), t, grp ? downP : upP, grp, upP.n, downP.n, false);
        else store_write_fn<true>(ws, store_wptr(sp, sw, off), t, grp ? downP : upP, grp, upP.n, downP.n, dev_dst);
        if (grp == 0) {
          if (lane == (t & 31)) my_off = off;
          if ((t & 31) == 31 || t == N - 1) {
            const int r = (t & ~31) + lane;
            if (r <= t) psd_st_cs_u64(index + r, my_off);
          }
        }
      }
    }
    PSD_T1(tc, 4);
    t++;
    if (status != PSD_ST_OK || t == N) {
      if (grp == 0) {
        double bc = 0, bx = 0, bpx = 0; int bbi = -1;
        if (status == PSD_ST_OK) best_piece(ws, downP, dmin, &bc, &bx, &bbi, &bpx);
        if (lane == 0) {
          res->status = status; res->back_i = bbi; res->best_cost = bc; res->best_x = bx; res->back_x = bpx;
          res->total_intervals = total_iv; res->max_intervals = max_iv; res->n_segments = 0; res->n_equality = 0;
          res->pad_ = n_spill;
        }
      }
      break;
    }
    if (back_to_shared(in_g, upP.n, downP.n, ws_s.cap)) {
      // both functions fit comfortably again: move back to shared memory
      if (grp == 0) pl_move(upP.base, ws_g.cap, ws_list(ws_s, 0), ws_s.cap, upP.n);
      else pl_move(downP.base, ws_g.cap, ws_list(ws_s, 1), ws_s.cap, downP.n);
      in_g = false;
      PSD_BIND_TIER();
      psd_pair_sync();
    }
  }
  if (lane == 0) psd_bulk_wait_all();   // no bulk copy may outlive the block's shared memory
  if (sw.slot >= 0) {   // the ring chunk still open at the end goes to the host like the others
    psd_fence_system();
    psd_pair_sync();
    if (grp == 0 && lane == 0) store_ring_publish(sp, sw.end / sp.chunk_bytes - 1ull - sp.n_chunks, sw.slot);
  }
  if (use_help) {       // release this chain's helper warp
    if (lane == 0) sh->help[grp].cmd = 2;
    psd_syncwarp();
    psd_bar_arrive(PSD_BAR_JOBS(grp), 64);
  }
#undef PSD_BIND_TIER
}
#endif   // PSD_G32

// ---- decode (src/PeakSegFPOPLog.cpp:400-442 + findMean :643-653) ------------------------------------
// Walks the stored functions from the last row back.  Output, last segment first:
//   seg_x[s]   = log-mean of segment s            (s = 0 .. n_segments-1)
//   seg_row[s] = last row of the segment before s (s = 0 .. n_segments-2)
PSD_DEV void backtrack_problem(const StorePool& sp, const unsigned long long* index, int n_rows,
                               DpResult* res, int* seg_row, double* seg_x) {
  const int lane = psd_lane();
  if (res->status != PSD_ST_OK) return;
  double best_x = res->best_x, back_x = res->back_x;
  int back_i = res->back_i;
  int use_down = 0;   // the last segment is "down"; the function read first is an "up" one
  int n_seg = 1, n_eq = 0, status = PSD_ST_OK;
  unsigned long long bytes = 0;
  while (0 <= back_i) {
    if (n_seg > n_rows) { status = PSD_ST_BACKTRACK_LOST; break; }
    const unsigned char* rec = store_ptr(sp, index[back_i]);
    const unsigned* hdr = (const unsigned*)rec;
    const int n_up = (int)hdr[0], n_down = (int)hdr[1];
    const int n = use_down ? n_down : n_up;
    bytes += 24ull + 20ull * (unsigned)n;
    const RecLayout R = rec_layout(n_up, n_down);
    const double* his = (const double*)(rec + R.hi[use_down]);
    const double* bxs = (const double*)(rec + R.bx[use_down]);
    const int* bis = (const int*)(rec + R.bi[use_down]);
    if (lane == 0) { seg_row[n_seg - 1] = back_i; seg_x[n_seg - 1] = best_x; }
    n_seg++;
    use_down ^= 1;
    if (back_x != PSD_INF) best_x = back_x; else n_eq++;
    // findMean: first piece k with lo_k <= x <= hi_k, lo_0 = -inf, lo_k = hi_{k-1}
    int found = 0;
    for (int base = 0; base < n && !found; base += 32) {
      const int k = base + lane;
      double hi = 0, lo = -PSD_INF;
      if (k < n) { hi = his[k]; if (k > 0) lo = his[k - 1]; }
      const unsigned mask = psd_ballot(k < n && lo <= best_x && best_x <= hi);
      if (mask) {
        const int kk = base + psd_ffs(mask) - 1;
        back_i = bis[kk];
        back_x = bxs[kk];
        found = 1;
      }
    }
    if (!found) { status = PSD_ST_BACKTRACK_LOST; break; }
  }
  if (lane == 0) {
    seg_x[n_seg - 1] = best_x;
    res->n_segments = n_seg; res->n_equality = n_eq; res->bt_bytes = bytes;
    if (status != PSD_ST_OK) res->status = status;
  }
}

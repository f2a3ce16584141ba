// fpop_gpu.cu -- sm_100a kernels and the batched plan behind the C ABI (include/peaksegdisk_b200.h).
//
// Launch structure (one CUDA stream, no host sync between kernels):
//   rle_encode_kernel      (upload, count-vector problems only) run-length encodes raw count vectors
//                          into the DP's rows (rle_gpu.cuh).
//   reads_scatter_kernel, coverage_scan_kernel, then rle_encode_kernel
//                          (psd_coverage_from_reads only, not part of a plan) per-base coverage of
//                          aligned reads and its rows (coverage_gpu.cuh).
//   features_hist_kernel, features_select_kernel (x 4)
//                          (psd_features only, not part of a plan) per-problem coverage statistics by
//                          a weighted radix select over the rows (features_gpu.cuh).
//   joint_flank_kernel, joint_flat_kernel, joint_pair_kernel<J>, joint_reduce_kernel
//                          (psd_joint_models only, not part of a plan) exact joint single-peak models
//                          of many samples (joint_gpu.cuh).
//   fpop_dp_kernel<W,B>    persistent warps; each warp takes problems (longest first) from an atomic
//                          queue and runs dp_run_queue() (fpop_warp.cuh): the whole DP of one
//                          (bedGraph x penalty), piece lists in shared memory (moving to a per-warp
//                          global workspace and back when a row's functions outgrow it), cost-function
//                          records streamed to the HBM chunk pool.  Two builds: <16,1> one block of
//                          14 warps per SM (default), <14,2> two blocks (waves of short problems,
//                          choose_config()).
//   fpop_backtrack_kernel  one warp per problem: backtrack_problem() walks the stored records,
//                          then compacts the segments into one array for a single D2H copy.
//   label_errors_kernel    (plans with labels only) one warp per problem: label errors of the
//                          compacted segments (label_errors_gpu.cuh).
// Problems whose functions outgrow even the per-warp workspace (status 101) are re-run by the same
// kernel with larger piece lists in global memory; when the store pool is exhausted (status 102)
// it is grown, then overflows into mapped pinned host memory, and only then are the remaining
// problems re-run in a later wave after the pool is recycled.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <atomic>
#include <mutex>
#include <queue>
#include <thread>
#include <string>
#include <unordered_map>
#include <vector>
#include "dp_params.h"
#include "label_errors_gpu.cuh"
#include "rle_gpu.cuh"
#include "coverage_gpu.cuh"
#include "features_gpu.cuh"
#include "plan_internal.h"

#define PSD_MAX_WARPS_PER_BLOCK 16   /* __launch_bounds__(512): 128 registers per thread (fewer registers only add spills; 14-16 warps fit shared memory) */
#define PSD_BT_WARPS_PER_BLOCK 4

#if defined(PSD_TIMING)
__device__ unsigned long long psd_blk_end[160];
#endif
__device__ const uint64_t d_exp_tab[256] = PSD_EXP_TAB_INIT;
__device__ const uint64_t d_log_tab[256] = PSD_LOG_TAB_INIT;
#include "joint_gpu.cuh"   // after d_log_tab: its kernels copy the table to shared memory

static inline unsigned long long psd_ws_bytes(int cap, int ccap) { return cap > 0 ? PSD_WS_BYTES(cap, ccap) : PSD_WS_HDR; }

// Two builds of the same kernel: <16,1> one phase-locked block per SM at 128 registers (the default:
// lowest per-row latency), <14,2> two blocks per SM at 72 registers (28 warps/SM: +18 % on batches of
// many short problems, -25 % when a long problem sets the critical path; see choose_config()).
template <int MAXW, int MINB>
__global__ void __launch_bounds__(MAXW * 32, MINB)
fpop_dp_kernel(const DpKernelParams P) {
  uint64_t* etab = (uint64_t*)psd_smem;     // psd_smem: the block's dynamic shared memory (fpop_warp.cuh)
  uint64_t* ltab = etab + 256;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) { etab[i] = d_exp_tab[i]; ltab[i] = d_log_tab[i]; }
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  const int wpb = blockDim.x >> 5;
  WarpWs ws_s, ws_g;
  ws_s.base = psd_smem + PSD_TAB_BYTES + (unsigned long long)warp * P.ws_s_bytes;
  ws_s.scratch = nullptr; ws_s.flags = (int*)ws_s.base; ws_s.cap = P.cap_s; ws_s.ccap = P.ccap_s; ws_s.help = nullptr;
  ws_g.base = P.gws ? P.gws + ((unsigned long long)blockIdx.x * wpb + warp) * P.ws_g_bytes : nullptr;
  ws_g.scratch = nullptr; ws_g.flags = ws_s.flags; ws_g.cap = P.gws ? P.cap_g : 0; ws_g.ccap = P.ccap_g; ws_g.help = nullptr;
  DpQueue Q;
  Q.problems = P.problems; Q.order = P.order; Q.n_order = P.n_order; Q.cursor = P.queue; Q.results = P.results;
  Q.first_slot = warp * (int)gridDim.x + (int)blockIdx.x;
  dp_run_queue(ws_s, ws_g, Q, P.pool);
#if defined(PSD_TIMING)
  if (threadIdx.x == 0 && blockIdx.x < 160) {   // when did this block run out of work? (ns since kernel start is derived on the host)
    unsigned long long tns; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tns));
    psd_blk_end[blockIdx.x] = tns;
  }
#endif
}

struct BtKernelParams {
  const DpProblem* problems;
  const int* order;
  int n_order;
  DpResult* results;
  StorePool pool;
  const unsigned long long* seg_scratch_off;   // per problem: offset of its scratch segment arrays
  int* scratch_row; double* scratch_x;         // n_rows + 1 entries per problem
  int* seg_row; double* seg_x;                 // compacted output
  unsigned long long* seg_cursor;
  const int* end_base;                         // count-vector problems: chromEnd rows made by rle_gpu.cuh
  const long long* end_off;                    // per problem: offset into end_base, -1 = a row problem
};

__global__ void __launch_bounds__(PSD_BT_WARPS_PER_BLOCK * 32)
fpop_backtrack_kernel(const BtKernelParams P) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= P.n_order) return;
  const int id = P.order[warp];
  DpResult* res = &P.results[id];
  if (res->status != PSD_ST_OK) return;
  const DpProblem pb = P.problems[id];
  int* srow = P.scratch_row + P.seg_scratch_off[id];
  double* sx = P.scratch_x + P.seg_scratch_off[id];
  backtrack_problem(P.pool, pb.index, pb.n_rows, res, srow, sx);
  __syncwarp();
  __threadfence_block();
  const int ns = __shfl_sync(0xffffffffu, (lane == 0) ? res->n_segments : 0, 0);
  const int st = __shfl_sync(0xffffffffu, (lane == 0) ? res->status : 0, 0);
  if (st != PSD_ST_OK) return;
  unsigned long long off = 0;
  if (lane == 0) { off = atomicAdd(P.seg_cursor, (unsigned long long)ns); res->seg_offset = off; }
  off = __shfl_sync(0xffffffffu, off, 0);
  const long long eo = P.end_base ? P.end_off[id] : -1;
  for (int s = lane; s < ns; s += 32) {
    P.seg_x[off + s] = sx[s];
    int r = (s < ns - 1) ? srow[s] : -1;
    if (eo >= 0 && r >= 0) r = P.end_base[eo + r];   // row number -> coordinate (the host has no rows)
    P.seg_row[off + s] = r;
  }
}

// ---- plan ---------------------------------------------------------------------------------------
namespace {
thread_local std::string g_last_error;
std::mutex g_opt_mutex;
struct Options { int piece_cap = 48; int overflow_cap = 8192; double store_gb = 0; int chunk_kb = 64; int spill_cap = 512; double host_spill_gb = -1; int occupancy_mode = 0; int devices = 1; int latency_mode = 0; int latency_max_blocks = 16; int spill_mode = 0; double ring_gb = 0; double coverage_gb = 0; } g_opt;

bool cuda_ok(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
  return false;
}
#define CK(call) do { if (!cuda_ok((call), #call)) return PSD_ERR_CUDA; } while (0)

template <class T> void dfree(T*& p) { if (p) cudaFree(p); p = nullptr; }

}  // namespace

void psd_set_last_error(const std::string& s) { g_last_error = s; }
const std::string& psd_get_last_error() { return g_last_error; }

int psd_set_option_impl(const char* name, double value) {
  std::lock_guard<std::mutex> lk(g_opt_mutex);
  std::string n(name);
  if (n == "piece_cap") g_opt.piece_cap = (int)value;
  else if (n == "overflow_cap") g_opt.overflow_cap = (int)value;
  else if (n == "store_gb") g_opt.store_gb = value;
  else if (n == "chunk_kb") g_opt.chunk_kb = (int)value;
  else if (n == "spill_cap") g_opt.spill_cap = std::max(0, (int)value);
  else if (n == "host_spill_gb") g_opt.host_spill_gb = value;
  else if (n == "occupancy_mode") g_opt.occupancy_mode = (int)value;   // 0 auto, 1 one block/SM, 2 two blocks/SM
  else if (n == "latency_mode") g_opt.latency_mode = (int)value;       // 0 auto (small waves), 1 always the latency kernel, 2 never
  else if (n == "latency_max_blocks") g_opt.latency_max_blocks = std::max(1, (int)value);   // auto: waves of up to this many problems per SM
  else if (n == "spill_mode") g_opt.spill_mode = (int)value;           // 0 DMA drain of an HBM ring (cudaMemcpyAsync on a side stream), 1 zero-copy stores
  else if (n == "ring_gb") g_opt.ring_gb = value;                      // HBM ring of the DMA drain (0 = automatic)
  else if (n == "devices") g_opt.devices = (int)value;                 // 1 current device only, k first k GPUs, <= 0 all
  else if (n == "coverage_gb") g_opt.coverage_gb = value;              // psd_coverage_from_reads / psd_features / psd_joint_models wave budget (0 = half of free HBM)
  else return PSD_ERR_ARG;
  return 0;
}

struct psd_plan {
  int device = 0;
  Options opt;
  cudaDeviceProp prop;
  // host side
  std::vector<HostProblem> probs;
  std::vector<int32_t> h_weight, h_cov;        // packed rows of the non-trivial problems
  // device side
  int *d_weight = nullptr, *d_cov = nullptr;
  unsigned long long* d_index = nullptr;
  DpProblem* d_problems = nullptr;
  DpResult* d_results = nullptr;
  int* d_order = nullptr;
  int* d_queue = nullptr;                      // the atomic cursor of the throughput kernel's problem queue
  unsigned long long* d_cursors = nullptr;     // [0] store chunk cursor, [1] segment cursor
  unsigned long long* d_seg_scratch_off = nullptr;
  int *d_scratch_row = nullptr, *d_seg_row = nullptr;
  double *d_scratch_x = nullptr, *d_seg_x = nullptr;
  unsigned char* d_pool = nullptr; unsigned long long pool_bytes = 0, pool_chunk = 0;
  size_t d_rows_cap = 0, d_index_cap = 0, d_prob_cap = 0, d_seg_cap = 0;
  std::vector<std::pair<const RowData*, int64_t>> row_sets;   // distinct row sets of the uploaded problems and their device offsets
  std::vector<std::pair<const RowData*, int64_t>> packed_row_sets;   // the row sets the pinned staging holds
  unsigned char* d_gws = nullptr; unsigned long long gws_bytes = 0;
  // count-vector problems: raw counts, chromEnd rows, run-length-encoding descriptors
  int *d_raw = nullptr, *d_end = nullptr; size_t d_raw_cap = 0, d_end_cap = 0;
  long long* d_end_off = nullptr;
  RleVec* d_rle_vecs = nullptr; int *d_tile_vec = nullptr, *d_rle_nrows = nullptr;
  unsigned long long* d_tile_state = nullptr;   // [n_tiles] look-back words, then ticket (4 B) and error flag (4 B)
  size_t d_rle_vec_cap = 0, d_tile_cap = 0;
  int32_t* p_raw = nullptr; size_t p_raw_cap = 0;
  int* p_rle_nrows = nullptr; size_t p_rle_nrows_cap = 0;
  int64_t rows_plain = 0, total_pos = 0; size_t n_count_problems = 0;
  unsigned char* h_spill = nullptr; unsigned char* d_spill = nullptr; unsigned long long spill_bytes = 0;   // mapped pinned host region
  // DMA drain of the spill (StoreRing): HBM ring, pinned queues, side stream
  unsigned char* d_ring = nullptr; unsigned long long ring_slots = 0, ring_chunk = 0;
  unsigned char* h_ringq = nullptr; unsigned char* d_ringq = nullptr; unsigned int ring_qlen = 0;   // [free_tail 64 B | free_q | done_q]
  cudaStream_t drain_stream = nullptr;
  // labels of the GPU problems (label_errors_gpu.cuh); n_labels == 0: the plan launches no label kernel
  int4* d_labels = nullptr; LabelDesc* d_label_desc = nullptr; int *d_label_fp = nullptr, *d_label_fn = nullptr, *d_label_tot = nullptr;
  int *p_label_fp = nullptr, *p_label_fn = nullptr, *p_label_tot = nullptr;
  size_t d_label_cap = 0, d_label_prob_cap = 0, p_label_cap = 0, p_label_prob_cap = 0;
  std::vector<LabelDesc> label_desc;
  int64_t n_labels = 0;
  double label_ms = 0;
  int64_t solve_h2d_bytes = 0, solve_d2h_bytes = 0;   // descriptors, order and status words of the last solve
  // pinned staging
  int32_t *p_weight = nullptr, *p_cov = nullptr;
  DpResult* p_results = nullptr;
  int* p_seg_row = nullptr; double* p_seg_x = nullptr;
  unsigned long long* p_cursors = nullptr;
  int* p_queue_init = nullptr;
  size_t p_rows_cap = 0, p_res_cap = 0, p_seg_cap = 0;
  // bookkeeping
  std::vector<int> gpu_ids;                    // problem ids that go to the GPU
  int64_t total_rows = 0, total_index = 0;
  bool uploaded = false, solved = false, packed = false;
  std::vector<DpResult> results;               // per gpu problem (indexed like gpu_ids)
  std::vector<int> result_wave;                // the store wave that produced each result (the pool holds only the last wave's records)
  unsigned long long last_hbm_bytes = 0;       // HBM part of the store in the last wave (offsets beyond it address the host region)
  std::vector<int> seg_row; std::vector<double> seg_x;
  unsigned long long n_seg_total = 0;
  psd_stats stats;
  cudaEvent_t ev[8];
  bool ev_ok = false;
  struct LaunchCfg { bool ok = false; int blocks = 1, wpb = 0, cap = 0, ccap = 0; size_t smem = 0; } cfg[2];
  bool configured = false;
  double last_mean_intervals = 0;   // of the previous solve of this plan (0: unknown)

  ~psd_plan() { release(); }
  void release_device() {
    dfree(d_weight); dfree(d_cov); dfree(d_index); dfree(d_problems); dfree(d_results); dfree(d_order);
    dfree(d_queue); dfree(d_cursors); dfree(d_seg_scratch_off); dfree(d_scratch_row); dfree(d_seg_row);
    dfree(d_scratch_x); dfree(d_seg_x); dfree(d_pool); dfree(d_gws); dfree(d_ring); ring_slots = 0;
    dfree(d_labels); dfree(d_label_desc); dfree(d_label_fp); dfree(d_label_fn); dfree(d_label_tot); d_label_cap = d_label_prob_cap = 0;
    dfree(d_raw); dfree(d_end); dfree(d_end_off); dfree(d_rle_vecs); dfree(d_tile_vec); dfree(d_tile_state); dfree(d_rle_nrows);
    d_raw_cap = d_end_cap = d_rle_vec_cap = d_tile_cap = 0;
    d_rows_cap = d_index_cap = d_prob_cap = d_seg_cap = 0; pool_bytes = 0; gws_bytes = 0;
    uploaded = false;
  }
  void release() {
    release_device();
    if (p_weight) cudaFreeHost(p_weight); if (p_cov) cudaFreeHost(p_cov);
    if (p_results) cudaFreeHost(p_results); if (p_seg_row) cudaFreeHost(p_seg_row);
    if (p_seg_x) cudaFreeHost(p_seg_x); if (p_cursors) cudaFreeHost(p_cursors); if (p_queue_init) cudaFreeHost(p_queue_init);
    if (h_spill) cudaFreeHost(h_spill);
    if (h_ringq) cudaFreeHost(h_ringq);
    h_ringq = d_ringq = nullptr; ring_qlen = 0;
    if (drain_stream) { cudaStreamDestroy(drain_stream); drain_stream = nullptr; }
    if (p_raw) cudaFreeHost(p_raw); if (p_rle_nrows) cudaFreeHost(p_rle_nrows);
    if (p_label_fp) cudaFreeHost(p_label_fp); if (p_label_fn) cudaFreeHost(p_label_fn); if (p_label_tot) cudaFreeHost(p_label_tot);
    p_label_fp = p_label_fn = p_label_tot = nullptr; p_label_cap = p_label_prob_cap = 0;
    p_raw = nullptr; p_rle_nrows = nullptr; p_raw_cap = p_rle_nrows_cap = 0;
    h_spill = d_spill = nullptr; spill_bytes = 0;
    p_queue_init = nullptr;
    p_weight = p_cov = nullptr; p_results = nullptr; p_seg_row = nullptr; p_seg_x = nullptr; p_cursors = nullptr;
    if (ev_ok) { for (auto& e : ev) cudaEventDestroy(e); ev_ok = false; }
  }
};

int psd_option_devices() {
  if (const char* e = getenv("PSD_DEVICES")) return atoi(e);
  std::lock_guard<std::mutex> lk(g_opt_mutex);
  return g_opt.devices;
}

static Options current_options() {
  Options o;
  { std::lock_guard<std::mutex> lk(g_opt_mutex); o = g_opt; }
  // environment overrides (tuning experiments)
  if (const char* e = getenv("PSD_PIECE_CAP")) o.piece_cap = atoi(e);
  if (const char* e = getenv("PSD_STORE_GB")) o.store_gb = atof(e);
  if (const char* e = getenv("PSD_SPILL_CAP")) o.spill_cap = std::max(0, atoi(e));
  if (const char* e = getenv("PSD_HOST_SPILL_GB")) o.host_spill_gb = atof(e);
  if (const char* e = getenv("PSD_OCCUPANCY_MODE")) o.occupancy_mode = atoi(e);
  if (const char* e = getenv("PSD_SPILL_MODE")) o.spill_mode = atoi(e);
  if (const char* e = getenv("PSD_LATENCY_MODE")) o.latency_mode = atoi(e);
  if (const char* e = getenv("PSD_LATENCY_MAX_BLOCKS")) o.latency_max_blocks = std::max(1, atoi(e));
  return o;
}

static bool same_options(const Options& a, const Options& b) {
  return a.piece_cap == b.piece_cap && a.overflow_cap == b.overflow_cap && a.store_gb == b.store_gb && a.chunk_kb == b.chunk_kb &&
         a.spill_cap == b.spill_cap && a.host_spill_gb == b.host_spill_gb && a.occupancy_mode == b.occupancy_mode &&
         a.latency_mode == b.latency_mode && a.latency_max_blocks == b.latency_max_blocks && a.spill_mode == b.spill_mode && a.ring_gb == b.ring_gb;
}

psd_plan* psd_plan_create_impl(int device) {
  // No CUDA call here: a plan holding only one-segment (trivial) problems never needs the device.
  psd_plan* p = new psd_plan();
  p->device = device;
  p->opt = current_options();
  memset(&p->stats, 0, sizeof p->stats);
  return p;
}

// First use of the device by this plan.  Fails loudly when there is no GPU: there is no CPU path.
static int ensure_device(psd_plan* p) {
  if (p->ev_ok) return cuda_ok(cudaSetDevice(p->device), "cudaSetDevice") ? 0 : PSD_ERR_CUDA;
  int ndev = 0;
  if (!cuda_ok(cudaGetDeviceCount(&ndev), "cudaGetDeviceCount")) return PSD_ERR_CUDA;
  if (ndev == 0) { g_last_error = "no CUDA device"; return PSD_ERR_CUDA; }
  if (p->device < 0) CK(cudaGetDevice(&p->device));
  CK(cudaSetDevice(p->device));
  CK(cudaGetDeviceProperties(&p->prop, p->device));
  if (p->prop.major < 10) { g_last_error = "peaksegdisk_b200 is built for sm_100a only"; return PSD_ERR_CUDA; }
  for (auto& e : p->ev) CK(cudaEventCreate(&e));
  p->ev_ok = true;
  return 0;
}

// ---- one recycled plan for the file entry points ------------------------------------------------------
// PeakSegFPOP_disk is called once per (file, penalty) by the reference's R code; creating and
// destroying the device buffers, the pinned staging and the store pool on every call costs 10-50 ms
// (much more on a box with slow allocation) next to a ~100 ms solve.  The file entry points
// therefore park their plan here when its footprint is small and take it back on the next call:
// its buffers are grow-only.  The parked plan is never freed at process exit on purpose (static
// destructors may run after the CUDA runtime is gone).
namespace {
std::mutex g_park_mutex;
psd_plan* g_parked = nullptr;
}

psd_plan* psd_plan_acquire_parked() {
  psd_plan* p = nullptr;
  { std::lock_guard<std::mutex> lk(g_park_mutex); p = g_parked; g_parked = nullptr; }
  if (p) {
    int dev = -1;
    const bool ok = cudaGetDevice(&dev) == cudaSuccess && dev == p->device && same_options(p->opt, current_options());
    if (ok) return p;
    psd_plan_destroy_impl(p);
  }
  return psd_plan_create_impl(-1);
}

// frees the parked plan (device buffers, store pool, pinned staging), if any
void psd_plan_drop_parked() {
  psd_plan* p = nullptr;
  { std::lock_guard<std::mutex> lk(g_park_mutex); p = g_parked; g_parked = nullptr; }
  if (p) psd_plan_destroy_impl(p);
}

void psd_plan_release_parked(psd_plan* p) {
  if (!p) return;
  const unsigned long long pinned = (unsigned long long)(p->p_rows_cap * 8 + p->p_raw_cap * 4 + p->p_seg_cap * 12 + p->p_res_cap * sizeof(DpResult));
  // freeing a multi-GB store pool and unpinning the staging costs 0.5-0.9 s per call (measured), far
  // more than keeping them for the next call of the same process; only very large plans are let go
  const bool small = p->ev_ok && p->pool_bytes <= (100ull << 30) && pinned <= (8ull << 30) && p->spill_bytes == 0 &&
                     p->gws_bytes <= (4ull << 30);
  if (small) {
    p->probs.clear(); p->gpu_ids.clear(); p->results.clear(); p->seg_row.clear(); p->seg_x.clear();
    p->uploaded = p->solved = p->packed = false; p->last_mean_intervals = 0;
    std::lock_guard<std::mutex> lk(g_park_mutex);
    if (!g_parked) { g_parked = p; return; }
  }
  psd_plan_destroy_impl(p);
}

void psd_plan_destroy_impl(psd_plan* p) { if (p) { if (p->ev_ok) cudaSetDevice(p->device); delete p; } }

std::vector<HostProblem>& psd_plan_problems(psd_plan* p) { return p->probs; }
const std::vector<HostProblem>& psd_plan_problems_c(const psd_plan* p) { return p->probs; }
void psd_plan_invalidate(psd_plan* p) { p->uploaded = false; p->solved = false; p->packed = false; }
void psd_plan_mark_penalty_changed(psd_plan* p) { p->solved = false; }
void psd_plan_mark_labels_changed(psd_plan* p) { p->uploaded = false; p->solved = false; }
const psd_stats& psd_plan_stats_ref(const psd_plan* p) { return p->stats; }

// Predicted store bytes per row (record + index): 16 B header + 8 B index + 40 B per piece pair; 520 B
// (12 pieces per function) until a solve of this plan has measured the mean piece count.  The pool is
// sized with it and the wave planner uses the same number, so a batch is split only when HBM is short.
static double psd_est_row_bytes(const psd_plan* p) {
  return p->last_mean_intervals > 0 ? std::max(520.0, 1.15 * (64.0 + 40.0 * p->last_mean_intervals)) : 520.0;
}

// H2D: pack the rows of the non-trivial problems, allocate index / result / segment buffers.
int psd_plan_upload_impl(psd_plan* p, void* stream_v) {
  cudaStream_t st = (cudaStream_t)stream_v;
  Trace tr;
  if (p->ev_ok) CK(cudaSetDevice(p->device));
  p->gpu_ids.clear();
  int64_t total = 0, total_pos = 0;
  size_t n_counts = 0;
  // row problems first: their (weight, coverage) rows are copied from the host, ONCE per RowData (the
  // penalties of one file share their rows on the host and on the device); the rows of count-vector
  // problems are produced on the device and only their raw counts are copied.  The record index is
  // per problem.
  int64_t total_index = 0;
  std::unordered_map<const RowData*, int64_t> off_of;
  p->row_sets.clear();
  for (int pass = 0; pass < 2; pass++)
    for (size_t i = 0; i < p->probs.size(); i++) {
      HostProblem& hp = p->probs[i];
      if (hp.status != 0 || hp.trivial || (int)hp.from_counts != pass) continue;
      hp.index_off = total_index; total_index += hp.n_rows;
      if (pass == 0) {
        auto it = off_of.find(hp.rows.get());
        if (it == off_of.end()) { it = off_of.emplace(hp.rows.get(), total).first; p->row_sets.push_back({hp.rows.get(), total}); total += hp.n_rows; }
        hp.row_off = it->second;
      } else {
        hp.row_off = total; total += hp.n_rows;
        hp.raw_off = total_pos; total_pos += hp.n_pos; n_counts++;
      }
    }
  if (p->row_sets != p->packed_row_sets) p->packed = false;
  p->rows_plain = 0;
  for (const auto& rs : p->row_sets) p->rows_plain += (int64_t)rs.first->coverage.size();
  for (size_t i = 0; i < p->probs.size(); i++) {
    const HostProblem& hp = p->probs[i];
    if (hp.status == 0 && !hp.trivial) p->gpu_ids.push_back((int)i);
  }
  p->total_rows = total; p->total_index = total_index; p->total_pos = total_pos; p->n_count_problems = n_counts;
  p->stats.h2d_bytes = 0; p->stats.h2d_ms = 0;
  const size_t ng = p->gpu_ids.size();
  if (ng == 0) { p->uploaded = true; p->solved = false; return 0; }
  { const int rc = ensure_device(p); if (rc) return rc; }
  tr.mark("upload: ensure_device");
  const int64_t plain = p->rows_plain;
  if ((size_t)plain > p->p_rows_cap) {
    if (p->p_weight) cudaFreeHost(p->p_weight); if (p->p_cov) cudaFreeHost(p->p_cov);
    p->p_weight = p->p_cov = nullptr; p->p_rows_cap = 0;
    CK(cudaMallocHost(&p->p_weight, sizeof(int32_t) * plain));
    CK(cudaMallocHost(&p->p_cov, sizeof(int32_t) * plain));
    p->p_rows_cap = plain; p->packed = false;
  }
  if ((size_t)total_pos > p->p_raw_cap) {
    if (p->p_raw) cudaFreeHost(p->p_raw);
    p->p_raw = nullptr; p->p_raw_cap = 0;
    CK(cudaMallocHost(&p->p_raw, sizeof(int32_t) * total_pos));
    p->p_raw_cap = total_pos; p->packed = false;
  }
  tr.mark("upload: pinned row staging");
  // rows are packed into the pinned staging buffers once per change of the problem set; a repeated
  // upload of the same plan is then a pure pinned-host -> device copy
  if (!p->packed) {
    for (int id : p->gpu_ids) {
      const HostProblem& hp = p->probs[id];
      if (hp.from_counts) memcpy(p->p_raw + hp.raw_off, hp.counts.data(), sizeof(int32_t) * hp.n_pos);
    }
    // row sets are laid out first and in order, so the device offset equals the staging offset; a big
    // batch is packed on all host cores (240 MB for config 2)
    auto pack_one = [&](int k) {
      const auto& rs = p->row_sets[k];
      memcpy(p->p_weight + rs.second, rs.first->weight.data(), sizeof(int32_t) * rs.first->weight.size());
      memcpy(p->p_cov + rs.second, rs.first->coverage.data(), sizeof(int32_t) * rs.first->coverage.size());
    };
    if (p->rows_plain > (1 << 22)) parallel_for((int)p->row_sets.size(), pack_one);
    else for (int k = 0; k < (int)p->row_sets.size(); k++) pack_one(k);
    p->packed = true; p->packed_row_sets = p->row_sets;
  }
  tr.mark("upload: pack rows");
  // device buffers are grow-only: a plan that is re-uploaded with the same shapes allocates nothing
  if ((size_t)total > p->d_rows_cap) {
    dfree(p->d_weight); dfree(p->d_cov); p->d_rows_cap = 0;
    CK(cudaMalloc(&p->d_weight, sizeof(int) * total));
    CK(cudaMalloc(&p->d_cov, sizeof(int) * total));
    p->d_rows_cap = total;
  }
  if ((size_t)total_index > p->d_index_cap) {
    dfree(p->d_index); p->d_index_cap = 0;
    CK(cudaMalloc(&p->d_index, sizeof(unsigned long long) * total_index));
    p->d_index_cap = total_index;
  }
  if (ng > p->d_prob_cap) {
    dfree(p->d_problems); dfree(p->d_results); dfree(p->d_order); dfree(p->d_seg_scratch_off); dfree(p->d_end_off);
    CK(cudaMalloc(&p->d_end_off, sizeof(long long) * ng));
    CK(cudaMalloc(&p->d_problems, sizeof(DpProblem) * ng));
    CK(cudaMalloc(&p->d_results, sizeof(DpResult) * ng));
    CK(cudaMalloc(&p->d_order, sizeof(int) * ng));
    CK(cudaMalloc(&p->d_seg_scratch_off, sizeof(unsigned long long) * ng));
    p->d_prob_cap = ng;
  }
  if (!p->d_cursors) CK(cudaMalloc(&p->d_cursors, sizeof(unsigned long long) * 8));   // [0] HBM chunk cursor [1] segment cursor [2] zero-copy host chunks [4] ring head [5] ring done head
  if ((size_t)(total_index + ng) > p->d_seg_cap) {
    dfree(p->d_scratch_row); dfree(p->d_scratch_x); dfree(p->d_seg_row); dfree(p->d_seg_x); p->d_seg_cap = 0;
    CK(cudaMalloc(&p->d_scratch_row, sizeof(int) * (total_index + ng)));
    CK(cudaMalloc(&p->d_scratch_x, sizeof(double) * (total_index + ng)));
    CK(cudaMalloc(&p->d_seg_row, sizeof(int) * (total_index + ng)));
    CK(cudaMalloc(&p->d_seg_x, sizeof(double) * (total_index + ng)));
    p->d_seg_cap = total_index + ng;
  }
  // count-vector problems: raw counts in, rows made on the device
  std::vector<RleVec> rvecs; std::vector<int> tile_vec;
  if (n_counts) {
    if ((size_t)total_pos > p->d_raw_cap) { dfree(p->d_raw); p->d_raw_cap = 0; CK(cudaMalloc(&p->d_raw, sizeof(int) * total_pos)); p->d_raw_cap = total_pos; }
    if ((size_t)total > p->d_end_cap) { dfree(p->d_end); p->d_end_cap = 0; CK(cudaMalloc(&p->d_end, sizeof(int) * total)); p->d_end_cap = total; }
    rvecs.reserve(n_counts);
    for (int id : p->gpu_ids) {
      const HostProblem& h = p->probs[id];
      if (!h.from_counts) continue;
      RleVec v; v.raw_off = h.raw_off; v.row_off = h.row_off; v.n_pos = (int)h.n_pos; v.tile0 = (int)tile_vec.size();
      const int nt = (int)((h.n_pos + PSD_RLE_TILE - 1) / PSD_RLE_TILE);
      tile_vec.insert(tile_vec.end(), (size_t)nt, (int)rvecs.size());
      rvecs.push_back(v);
    }
    if (rvecs.size() > p->d_rle_vec_cap) {
      dfree(p->d_rle_vecs); dfree(p->d_rle_nrows); p->d_rle_vec_cap = 0;
      CK(cudaMalloc(&p->d_rle_vecs, sizeof(RleVec) * rvecs.size()));
      CK(cudaMalloc(&p->d_rle_nrows, sizeof(int) * rvecs.size()));
      p->d_rle_vec_cap = rvecs.size();
    }
    if (tile_vec.size() > p->d_tile_cap) {
      dfree(p->d_tile_vec); dfree(p->d_tile_state); p->d_tile_cap = 0;
      CK(cudaMalloc(&p->d_tile_vec, sizeof(int) * tile_vec.size()));
      CK(cudaMalloc(&p->d_tile_state, sizeof(unsigned long long) * (tile_vec.size() + 1)));
      p->d_tile_cap = tile_vec.size();
    }
    if (rvecs.size() + 1 > p->p_rle_nrows_cap) {   // + the kernel's error flag
      if (p->p_rle_nrows) cudaFreeHost(p->p_rle_nrows);
      p->p_rle_nrows = nullptr; p->p_rle_nrows_cap = 0;
      CK(cudaMallocHost(&p->p_rle_nrows, sizeof(int) * (rvecs.size() + 1)));
      p->p_rle_nrows_cap = rvecs.size() + 1;
    }
  }
  tr.mark("upload: device buffers");
  if (ng > p->p_res_cap) {
    if (p->p_results) cudaFreeHost(p->p_results);
    p->p_results = nullptr; p->p_res_cap = 0;
    CK(cudaMallocHost(&p->p_results, sizeof(DpResult) * ng));
    p->p_res_cap = ng;
  }
  // (the pinned staging of the segments is sized at download, from the number of segments found:
  // pinning the worst case of one segment per row cost more than the whole D2H copy)
  if (!p->p_cursors) CK(cudaMallocHost(&p->p_cursors, sizeof(unsigned long long) * 8));
  if (!p->p_queue_init) CK(cudaMallocHost(&p->p_queue_init, sizeof(int)));   // initial value of the queue cursor
  tr.mark("upload: pinned result staging");
  // store pool: sized from free memory unless the option pins it
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  unsigned long long want;
  if (p->opt.store_gb > 0) want = (unsigned long long)(p->opt.store_gb * (double)(1ull << 30));
  else {
    // estimate: 16 B header + 8 B index + 20 B x 2 functions x ~11 pieces per row (config 2 writes 380 B
    // per row, Mono27ac 300-560); a wave that still runs out grows the pool x4 and repeats; clamp to 80% of free memory
    want = (unsigned long long)((double)total_index * psd_est_row_bytes(p)) + (64ull << 20);
    const unsigned long long lim = (unsigned long long)((double)free_b * 0.80);
    if (want > lim) want = lim;
  }
  const unsigned long long chunk = (unsigned long long)p->opt.chunk_kb << 10;
  want = (want / chunk) * chunk;
  if (want < chunk * 16) want = chunk * 16;
  if (want > p->pool_bytes || p->pool_chunk != chunk) {
    dfree(p->d_pool); p->pool_bytes = 0;
    if (p->opt.store_gb <= 0) {   // re-evaluate the clamp now that the old pool is gone
      CK(cudaMemGetInfo(&free_b, &total_b));
      const unsigned long long lim = ((unsigned long long)((double)free_b * 0.80) / chunk) * chunk;
      if (want > lim) want = lim;
    }
    CK(cudaMalloc(&p->d_pool, want));
    p->pool_bytes = want; p->pool_chunk = chunk;
  }
  tr.mark("upload: store pool");
  // device problem descriptors
  std::vector<DpProblem> hp(ng);
  std::vector<unsigned long long> soff(ng);
  std::vector<long long> eoff(ng);
  // backtrack scratch: n_rows + 1 entries per problem, handed out in gpu_ids order (independent of
  // the row_off order, which puts count-vector problems after row problems)
  unsigned long long scratch_cursor = 0;
  for (size_t g = 0; g < ng; g++) {
    const HostProblem& h = p->probs[p->gpu_ids[g]];
    hp[g].weight = p->d_weight + h.row_off; hp[g].coverage = p->d_cov + h.row_off;
    hp[g].n_rows = (int)h.n_rows; hp[g].penalty = h.penalty; hp[g].dmin = h.dmin; hp[g].dmax = h.dmax;
    hp[g].index = p->d_index + h.index_off;
    soff[g] = scratch_cursor; scratch_cursor += (unsigned long long)h.n_rows + 1ull;
    eoff[g] = h.from_counts ? (long long)h.row_off : -1;
  }
  // labels: codes (start, end, kind) packed per GPU problem, in gpu_ids order
  std::vector<int4> labs;
  p->label_desc.assign(ng, LabelDesc{0, 0, 0});
  for (size_t g = 0; g < ng; g++) {
    const HostProblem& h = p->probs[p->gpu_ids[g]];
    if (!h.labels) continue;
    const LabelSet& L = *h.labels;
    p->label_desc[g].off = (long long)labs.size(); p->label_desc[g].n = (int)L.kind.size();
    for (size_t k = 0; k < L.kind.size(); k++) labs.push_back(make_int4(L.code_start[k], L.code_end[k], L.kind[k], 0));
  }
  p->n_labels = (int64_t)labs.size();
  if (p->n_labels) {
    if (labs.size() > p->d_label_cap) {
      dfree(p->d_labels); dfree(p->d_label_fp); dfree(p->d_label_fn); p->d_label_cap = 0;
      CK(cudaMalloc(&p->d_labels, sizeof(int4) * labs.size()));
      CK(cudaMalloc(&p->d_label_fp, sizeof(int) * labs.size()));
      CK(cudaMalloc(&p->d_label_fn, sizeof(int) * labs.size()));
      p->d_label_cap = labs.size();
    }
    if (ng > p->d_label_prob_cap) {
      dfree(p->d_label_desc); dfree(p->d_label_tot); p->d_label_prob_cap = 0;
      CK(cudaMalloc(&p->d_label_desc, sizeof(LabelDesc) * ng));
      CK(cudaMalloc(&p->d_label_tot, sizeof(int) * 5 * ng));
      p->d_label_prob_cap = ng;
    }
    if (labs.size() > p->p_label_cap) {
      if (p->p_label_fp) cudaFreeHost(p->p_label_fp); if (p->p_label_fn) cudaFreeHost(p->p_label_fn);
      p->p_label_fp = p->p_label_fn = nullptr; p->p_label_cap = 0;
      CK(cudaMallocHost(&p->p_label_fp, sizeof(int) * labs.size()));
      CK(cudaMallocHost(&p->p_label_fn, sizeof(int) * labs.size()));
      p->p_label_cap = labs.size();
    }
    if (ng > p->p_label_prob_cap) {
      if (p->p_label_tot) cudaFreeHost(p->p_label_tot);
      p->p_label_tot = nullptr; p->p_label_prob_cap = 0;
      CK(cudaMallocHost(&p->p_label_tot, sizeof(int) * 5 * ng));
      p->p_label_prob_cap = ng;
    }
  }
  CK(cudaEventRecord(p->ev[0], st));
  if (p->n_labels) {
    CK(cudaMemcpyAsync(p->d_labels, labs.data(), sizeof(int4) * labs.size(), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(p->d_label_desc, p->label_desc.data(), sizeof(LabelDesc) * ng, cudaMemcpyHostToDevice, st));
  }
  if (plain) {
    CK(cudaMemcpyAsync(p->d_weight, p->p_weight, sizeof(int) * plain, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(p->d_cov, p->p_cov, sizeof(int) * plain, cudaMemcpyHostToDevice, st));
  }
  if (n_counts) {
    CK(cudaMemcpyAsync(p->d_raw, p->p_raw, sizeof(int) * total_pos, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(p->d_rle_vecs, rvecs.data(), sizeof(RleVec) * rvecs.size(), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(p->d_tile_vec, tile_vec.data(), sizeof(int) * tile_vec.size(), cudaMemcpyHostToDevice, st));
  }
  CK(cudaMemcpyAsync(p->d_problems, hp.data(), sizeof(DpProblem) * ng, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(p->d_seg_scratch_off, soff.data(), sizeof(unsigned long long) * ng, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(p->d_end_off, eoff.data(), sizeof(long long) * ng, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(p->ev[1], st));
  p->stats.rle_ms = 0; p->stats.rle_bytes_algorithmic = 0; p->stats.rle_positions = 0; p->stats.n_rle_launches = n_counts ? 1 : 0;
  if (n_counts) {
    // run-length encode on the device (rle_gpu.cuh): one single-pass kernel on the plan's stream
    RleParams R;
    R.vecs = p->d_rle_vecs; R.tile_vec = p->d_tile_vec; R.n_tiles = (int)tile_vec.size(); R.n_vecs = (int)rvecs.size();
    R.raw = p->d_raw; R.coverage = p->d_cov; R.chrom_end = p->d_end; R.weight = p->d_weight;
    R.tile_state = p->d_tile_state; R.n_rows = p->d_rle_nrows;
    R.ticket = (unsigned int*)(p->d_tile_state + R.n_tiles); R.error = (int*)(R.ticket + 1);
    CK(cudaMemsetAsync(p->d_tile_state, 0, sizeof(unsigned long long) * ((size_t)R.n_tiles + 1), st));
    CK(cudaEventRecord(p->ev[5], st));
    rle_encode_kernel<<<R.n_tiles, PSD_RLE_WARPS * 32, 0, st>>>(R);
    CK(cudaGetLastError());
    CK(cudaEventRecord(p->ev[6], st));
    CK(cudaMemcpyAsync(p->p_rle_nrows, p->d_rle_nrows, sizeof(int) * rvecs.size(), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(p->p_rle_nrows + rvecs.size(), R.error, sizeof(int), cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));   // hp/soff/... are pageable temporaries
  tr.mark("upload: H2D + RLE + sync");
  float ms = 0; cudaEventElapsedTime(&ms, p->ev[0], p->ev[1]);
  p->stats.h2d_ms = ms;
  p->stats.h2d_bytes = (int64_t)(2 * sizeof(int) * plain + sizeof(int) * total_pos + (sizeof(DpProblem) + 16) * ng +
                                 sizeof(RleVec) * rvecs.size() + sizeof(int) * tile_vec.size() +
                                 (p->n_labels ? sizeof(int4) * labs.size() + sizeof(LabelDesc) * ng : 0));
  if (n_counts) {
    cudaEventElapsedTime(&ms, p->ev[5], p->ev[6]);
    p->stats.rle_ms = ms; p->stats.rle_positions = total_pos;
    p->stats.rle_bytes_algorithmic = (int64_t)(4 * total_pos + 12 * (total - plain));
    if (p->p_rle_nrows[rvecs.size()] != 0) { g_last_error = "device run-length encoding: look-back gave up"; return PSD_ERR_INTERNAL; }
    size_t k = 0;
    for (int id : p->gpu_ids) {
      const HostProblem& h = p->probs[id];
      if (!h.from_counts) continue;
      if (p->p_rle_nrows[k] != (int)h.n_rows) { g_last_error = "device run-length encoding disagrees with the host's run count"; return PSD_ERR_INTERNAL; }
      k++;
    }
  }
  p->uploaded = true; p->solved = false;
  return 0;
}

template <int MAXW, int MINB>
static int configure_one(psd_plan* p, psd_plan::LaunchCfg& L, int cap0) {
  int cap = cap0;
  if (cap < 8) cap = 8;
  cap = (cap + 3) & ~3;   // multiples of 4 keep every list array 16-byte aligned (bulk copies of the record store)
  for (;;) {
    const int ccap = 2 * cap;
    const size_t per_warp = psd_ws_bytes(cap, ccap);
    // each block also costs ~1 KB of reserved shared memory
    int w = (int)((((size_t)p->prop.sharedMemPerMultiprocessor / MINB) - 1024 - PSD_TAB_BYTES) / per_warp);
    w = std::min(w, (int)(((size_t)p->prop.sharedMemPerBlockOptin - PSD_TAB_BYTES) / per_warp));
    w = std::min(w, MAXW);
    for (; w >= 1; w--) {   // registers may allow fewer warps than shared memory does
      const size_t smem = PSD_TAB_BYTES + (size_t)w * per_warp;
      CK(cudaFuncSetAttribute(fpop_dp_kernel<MAXW, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int nb = 0;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fpop_dp_kernel<MAXW, MINB>, w * 32, smem));
      if (nb >= MINB) { L.ok = true; L.blocks = MINB; L.wpb = w; L.cap = cap; L.ccap = ccap; L.smem = smem; return 0; }
    }
    cap = ((cap / 2) + 3) & ~3;
    if (cap < 8) { L.ok = false; return 0; }
  }
}

static int configure_kernel(psd_plan* p) {
  if (p->configured) return 0;
  int rc = configure_one<PSD_MAX_WARPS_PER_BLOCK, 1>(p, p->cfg[0], p->opt.piece_cap);
  if (rc) return rc;
  if (!p->cfg[0].ok) { g_last_error = "cannot fit the DP kernel's shared memory"; return PSD_ERR_CUDA; }
  rc = configure_one<14, 2>(p, p->cfg[1], p->opt.piece_cap / 2);
  if (rc) return rc;
  p->configured = true;
  return 0;
}

// Makespan, in rows, of the persistent-warp queue: problems (longest first) go to the slot that frees
// up first.  This is what the kernel's static first assignment + atomic queue does when every slot
// advances at the same rows per second.
static double queue_makespan(const psd_plan* p, const std::vector<int>& todo, size_t slots) {
  if (todo.size() <= slots) return todo.empty() ? 0.0 : (double)p->probs[p->gpu_ids[todo[0]]].n_rows;
  std::priority_queue<double, std::vector<double>, std::greater<double>> free_at;
  for (size_t k = 0; k < slots; k++) free_at.push((double)p->probs[p->gpu_ids[todo[k]]].n_rows);
  double last = 0;
  for (size_t k = slots; k < todo.size(); k++) {
    const double t = free_at.top() + (double)p->probs[p->gpu_ids[todo[k]]].n_rows;
    free_at.pop(); free_at.push(t);
  }
  while (!free_at.empty()) { last = free_at.top(); free_at.pop(); }
  return last;
}

// Picks the launch configuration for one wave (todo is sorted longest first).  Measured on B200
// (profiles/README.md): with twice the warps per SM, cfg[1] moves 1.2x the rows per second per SM,
// so each of its warps advances at 1.2/2 of a cfg[0] warp's rate.  Both makespans are simulated;
// cfg[1] must win by 5 %, the functions must be small enough for its 24-piece shared-memory tier
// (when known from a previous solve of the same plan) and the problems must be short.
static int choose_config(psd_plan* p, const std::vector<int>& todo) {
  if (p->opt.occupancy_mode == 1 || !p->cfg[1].ok) return 0;
  if (p->opt.occupancy_mode == 2) return 1;
  if (todo.empty()) return 0;
  const double longest = (double)p->probs[p->gpu_ids[todo[0]]].n_rows;
  if (p->last_mean_intervals > 9.0) return 0;
  // Measured (profiles/README.md): the two-block build wins on batches of problems up to ~15 k rows
  // (+16...+25 %), loses 32 % on 30 k-row problems and 17 % on 7.5 k-75 k-row problems even when their
  // functions are small and the long problems get the SM to themselves: only short problems qualify.
  if (longest > 16000) return 0;
  const size_t n_sm = (size_t)p->prop.multiProcessorCount;
  const size_t slots0 = n_sm * (size_t)(p->cfg[0].wpb * p->cfg[0].blocks), slots1 = n_sm * (size_t)(p->cfg[1].wpb * p->cfg[1].blocks);
  if (todo.size() <= slots0) return 0;                            // every problem already has its own warp
  const double t0 = queue_makespan(p, todo, slots0) * (double)slots0;            // rows / (rows per second per SM), up to a constant
  const double t1 = queue_makespan(p, todo, slots1) * (double)slots1 / 1.2;
  return t1 < 0.95 * t0 ? 1 : 0;
}

// ---- DMA drain of the store spill (host side of StoreRing, fpop_warp.cuh) --------------------------
// While the DP kernel runs, a host thread polls the pinned done-queue; every published ring slot is
// copied to its place in the pinned host region by cudaMemcpyAsync on a side stream, and once a batch
// of copies has completed the slots go back to the device through the pinned free-queue.
struct RingDrain {
  psd_plan* p = nullptr;
  unsigned long long chunk = 0;
  std::atomic<unsigned long long> final_count{~0ull};   // set when the kernel has finished: total chunks published
  std::atomic<int> error{0};
  unsigned long long drained = 0;
  std::thread th;
  volatile unsigned long long* free_tail() const { return (volatile unsigned long long*)p->h_ringq; }
  volatile unsigned int* free_q() const { return (volatile unsigned int*)(p->h_ringq + 64); }
  volatile unsigned long long* done_q() const { return (volatile unsigned long long*)(p->h_ringq + 64 + 4ull * p->ring_qlen); }
  void run() {
    if (cudaSetDevice(p->device) != cudaSuccess) { error = 1; return; }
    const unsigned mask = p->ring_qlen - 1;
    unsigned long long next = 0, ftail = p->ring_slots;
    std::vector<unsigned> batch;
    int idle = 0;
    for (;;) {
      volatile unsigned long long* e = done_q() + 2ull * (next & mask);
      if (e[0] == next + 1ull && batch.size() < 256) {
        const unsigned long long payload = e[1];
        const unsigned long long host_chunk = payload >> 32, slot = payload & 0xffffffffull;
        if (cudaMemcpyAsync(p->h_spill + host_chunk * chunk, p->d_ring + slot * chunk, chunk, cudaMemcpyDeviceToHost, p->drain_stream) != cudaSuccess) error = 2;
        batch.push_back((unsigned)slot);
        next++; idle = 0;
        continue;
      }
      if (!batch.empty()) {
        if (cudaStreamSynchronize(p->drain_stream) != cudaSuccess) error = 3;
        for (unsigned slot : batch) { free_q()[ftail & mask] = slot; ftail++; }
        std::atomic_thread_fence(std::memory_order_release);
        *free_tail() = ftail;
        batch.clear();
        continue;
      }
      const unsigned long long fin = final_count.load(std::memory_order_acquire);
      if (fin != ~0ull && next >= fin) break;
      if (++idle > 64) std::this_thread::sleep_for(std::chrono::microseconds(20)); else std::this_thread::yield();
    }
    drained = next;
  }
};

// (re)creates the ring for a launch of `n_warps` writers; returns 0 when the ring is ready
static int ring_prepare(psd_plan* p, unsigned long long chunk, unsigned long long n_writers) {
  // every writer can hold one open ring chunk while it waits at a phase barrier for a warp that is
  // waiting for a free slot: the ring must be larger than the number of writers (fpop_warp.cuh)
  unsigned long long want_slots = 4ull * n_writers + 64ull;
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  unsigned long long auto_bytes = p->opt.ring_gb > 0 ? (unsigned long long)(p->opt.ring_gb * (double)(1ull << 30)) : std::min<unsigned long long>(2ull << 30, (free_b + p->ring_slots * p->ring_chunk) / 8);
  want_slots = std::max(want_slots, auto_bytes / chunk);
  if (want_slots > 0xfffffff0ull) want_slots = 0xfffffff0ull;
  if (p->ring_slots < want_slots || p->ring_chunk != chunk) {
    dfree(p->d_ring); p->ring_slots = 0;
    CK(cudaMalloc(&p->d_ring, want_slots * chunk));
    p->ring_slots = want_slots; p->ring_chunk = chunk;
  }
  unsigned qlen = 64; while ((unsigned long long)qlen < 4ull * p->ring_slots) qlen <<= 1;
  if (qlen != p->ring_qlen) {
    if (p->h_ringq) cudaFreeHost(p->h_ringq);
    p->h_ringq = p->d_ringq = nullptr; p->ring_qlen = 0;
    CK(cudaHostAlloc((void**)&p->h_ringq, 64 + 20ull * qlen, cudaHostAllocMapped | cudaHostAllocPortable));
    CK(cudaHostGetDevicePointer((void**)&p->d_ringq, p->h_ringq, 0));
    p->ring_qlen = qlen;
  }
  if (!p->drain_stream) CK(cudaStreamCreateWithFlags(&p->drain_stream, cudaStreamNonBlocking));
  return 0;
}

// Which kernel for a wave?  Makespan model from measurements on B200 (profiles/README.md, round 2):
//   throughput kernel (one problem per warp, 14 per SM): 53 M rows/s when all 2,072 slots are busy, but a
//   row of ONE problem takes 17.6 us with <= 148 problems in flight and 38 us at full load;
//   latency kernel (one problem per block): 12.3 / 15.2 / 19 / 24 us per row with 1 / 2 / 3 / 4 blocks per
//   SM, no gain beyond 4 resident blocks (instruction cache), further blocks queue behind them.
// Both makespans = max(work bound, critical path of the longest problem); todo is sorted longest first.
static bool choose_latency_kernel(const psd_plan* p, const std::vector<int>& todo) {
  if (p->opt.latency_mode == 1) return true;
  if (p->opt.latency_mode == 2 || todo.empty()) return false;
  const double n_sm = (double)p->prop.multiProcessorCount, n = (double)todo.size();
  const int b = (int)((todo.size() + (size_t)n_sm - 1) / (size_t)n_sm);
  if (b <= 2) return true;
  if (b > p->opt.latency_max_blocks) return false;
  double total = 0;
  for (int g : todo) total += (double)p->probs[p->gpu_ids[g]].n_rows;
  const double longest = (double)p->probs[p->gpu_ids[todo[0]]].n_rows;
  const double L = b == 3 ? 19.0 : 24.0;                                   // us per row of one problem
  const double t_lat = std::max(total * L / (n_sm * std::min(b, 4)), longest * L);
  static const double xs[] = {148, 296, 592, 1184, 2072}, ys[] = {17.6, 21.1, 28.4, 30.5, 38.0};
  const double load = n * 148.0 / n_sm;                                    // problems in flight, scaled to 148 SMs
  double l_thr = ys[4];
  if (load <= xs[0]) l_thr = ys[0];
  else for (int k = 1; k < 5; k++) if (load <= xs[k]) { l_thr = ys[k - 1] + (ys[k] - ys[k - 1]) * (load - xs[k - 1]) / (xs[k] - xs[k - 1]); break; }
  const double t_thr = std::max(total / (53.0 * n_sm / 148.0), longest * l_thr);
  return t_lat < 0.9 * t_thr;
}

// Pinned host region of the store spill (mapped: the backtrack reads it, zero-copy writers write it).
// want_gb <= 0: nothing.  Pinning costs ~0.3 s per GB, so callers ask for what the records need.
static bool alloc_host_spill(psd_plan* p, double want_gb, unsigned long long chunk) {
  if (p->d_spill || want_gb <= 0) return p->d_spill != nullptr;
  const unsigned long long want = ((unsigned long long)(want_gb * (double)(1ull << 30)) / chunk) * chunk;
  if (want < chunk * 16) return false;
  if (cudaHostAlloc((void**)&p->h_spill, want, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
    cudaGetLastError();   // no pinned memory to be had
    p->h_spill = nullptr;
    return false;
  }
  if (cudaHostGetDevicePointer((void**)&p->d_spill, p->h_spill, 0) != cudaSuccess) { cudaFreeHost(p->h_spill); p->h_spill = p->d_spill = nullptr; return false; }
  p->spill_bytes = want;
  return true;
}

// the automatic size limit of the host region: a quarter of the host's available memory, at most 64 GB
static double host_spill_limit_gb(const psd_plan* p) {
  if (p->opt.host_spill_gb >= 0) return p->opt.host_spill_gb;
  double gb = 8;
  if (FILE* mf = fopen("/proc/meminfo", "r")) {
    char line[256];
    while (fgets(line, sizeof line, mf)) { unsigned long long kb; if (sscanf(line, "MemAvailable: %llu kB", &kb) == 1) gb = (double)kb / (1024.0 * 1024.0) * 0.25; }
    fclose(mf);
  }
  return gb > 64 ? 64 : gb;
}

// DP + backtrack for every uploaded problem.  Device-only: no host<->device row traffic.
int psd_plan_solve_impl(psd_plan* p, void* stream_v) {
  cudaStream_t st = (cudaStream_t)stream_v;
  Trace tr;
  if (!p->uploaded) { g_last_error = "psd_plan_solve before psd_plan_upload"; return PSD_ERR_ARG; }
  const size_t ng = p->gpu_ids.size();
  if (ng) CK(cudaSetDevice(p->device));
  psd_stats& S = p->stats;
  S.dp_ms = S.backtrack_ms = 0; S.n_launches = 0; S.n_waves = 0; S.n_overflow_tier = 0; S.n_latency_waves = 0;
  S.rows_solved = 0; S.store_bytes_algorithmic = 0; S.store_bytes_written = 0; S.backtrack_bytes_read = 0; S.store_bytes_spilled_host = 0; S.store_bytes_drained_dma = 0;
  p->results.assign(ng, DpResult());
  p->result_wave.assign(ng, -1);
  p->n_seg_total = 0;
  p->label_ms = 0; p->solve_h2d_bytes = 0; p->solve_d2h_bytes = 0;
  if (ng == 0) { p->solved = true; return 0; }
  int rc = configure_kernel(p);
  if (rc) return rc;
  tr.mark("solve: configure_kernel");
  S.piece_cap = p->cfg[0].cap; S.warps_per_sm = p->cfg[0].wpb * p->cfg[0].blocks; S.n_sm = p->prop.multiProcessorCount;
  // penalties may have changed since upload (sequential search): refresh the descriptors' penalty
  {
    std::vector<DpProblem> hp(ng);
    for (size_t g = 0; g < ng; g++) {
      const HostProblem& h = p->probs[p->gpu_ids[g]];
      hp[g].weight = p->d_weight + h.row_off; hp[g].coverage = p->d_cov + h.row_off;
      hp[g].n_rows = (int)h.n_rows; hp[g].penalty = h.penalty; hp[g].dmin = h.dmin; hp[g].dmax = h.dmax;
      hp[g].index = p->d_index + h.index_off;
    }
    CK(cudaMemcpyAsync(p->d_problems, hp.data(), sizeof(DpProblem) * ng, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    p->solve_h2d_bytes += (int64_t)(sizeof(DpProblem) * ng);
  }
  const unsigned long long chunk = (unsigned long long)p->opt.chunk_kb << 10;
  std::vector<int> todo(ng);            // problems of the wave about to run (current tier)
  for (size_t g = 0; g < ng; g++) todo[g] = (int)g;
  std::sort(todo.begin(), todo.end(), [&](int a, int b) {
    const int64_t na = p->probs[p->gpu_ids[a]].n_rows, nb = p->probs[p->gpu_ids[b]].n_rows;
    return na != nb ? na > nb : a < b;
  });
  std::vector<int> deferred;            // same tier, waiting for the store pool to be recycled
  std::vector<int> overflow_acc;        // need the next piece-list tier
  // Store planning from a PREDICTION of the record bytes (16 B header + 8 B index + 40 B per piece pair
  // per row; the mean piece count of the plan's previous solve when there was one, else 12), so that a
  // batch larger than the store is not discovered by running out half way:
  //   * problems are dealt into waves whose predicted records fit the store (each wave recycles it);
  //   * a single problem larger than the HBM pool gets its pinned host region (spill) before it starts.
  double est_row_bytes = psd_est_row_bytes(p);
  auto plan_wave = [&](std::vector<int>& wave, std::vector<int>& later) {
    // (the automatic pool is sized with the same 520 B per row: a batch is only split when HBM could not hold the prediction)
    const double cap_bytes = (double)(p->pool_bytes + p->spill_bytes);
    double sum = 0;
    size_t keep = 0;
    for (; keep < wave.size(); keep++) {
      const double b = est_row_bytes * (double)p->probs[p->gpu_ids[wave[keep]]].n_rows;
      if (keep > 0 && sum + b > cap_bytes) break;
      sum += b;
    }
    later.insert(later.end(), wave.begin() + keep, wave.end());
    wave.resize(keep);
  };
  if (!todo.empty() && p->opt.host_spill_gb != 0 && !p->d_spill) {
    const double first = est_row_bytes * (double)p->probs[p->gpu_ids[todo[0]]].n_rows;
    if (first > (double)p->pool_bytes) {
      const double gb = std::min(host_spill_limit_gb(p), 1.3 * (first - 0.8 * (double)p->pool_bytes) / (double)(1ull << 30) + 0.05);
      alloc_host_spill(p, gb, chunk);
      tr.mark("solve: pinned host region for the spill");
    }
  }
  plan_wave(todo, deferred);
  if (!deferred.empty() && p->opt.host_spill_gb != 0 && !p->d_spill) {
    // A second wave costs at least the critical path of its longest problem (~15 us per row); pinned
    // host memory for the same records costs ~0.33 s per GB.  Spill instead of waiting when that is cheaper.
    double later_bytes = 0, later_longest = 0;
    for (int g : deferred) {
      const double r = (double)p->probs[p->gpu_ids[g]].n_rows;
      later_bytes += est_row_bytes * r; later_longest = std::max(later_longest, r);
    }
    const double need_gb = 1.15 * later_bytes / (double)(1ull << 30) + 0.05;
    if (need_gb <= host_spill_limit_gb(p) && 0.33 * need_gb < later_longest * 15e-6 && alloc_host_spill(p, need_gb, chunk)) {
      todo.insert(todo.end(), deferred.begin(), deferred.end());
      deferred.clear();
      plan_wave(todo, deferred);
      tr.mark("solve: pinned host region instead of a second wave");
    }
  }
  CK(cudaMemsetAsync(p->d_cursors, 0, sizeof(unsigned long long) * 8, st));
  bool global_tier = false;
  int gcap = p->opt.overflow_cap;
  if (gcap > 32768) gcap = 32768;
  for (int guard = 0;; guard++) {
    if (guard > 4096) { g_last_error = "solve did not converge"; return PSD_ERR_INTERNAL; }
    if (todo.empty()) {
      if (!deferred.empty()) {
        todo.swap(deferred);
        std::sort(todo.begin(), todo.end(), [&](int a, int b) {
          const int64_t na = p->probs[p->gpu_ids[a]].n_rows, nb = p->probs[p->gpu_ids[b]].n_rows;
          return na != nb ? na > nb : a < b;
        });
        plan_wave(todo, deferred);
      } else if (!overflow_acc.empty()) {
        if (global_tier) {
          if (gcap >= 32768) {   // largest tier exhausted: report status 101 for these problems
            for (int g : overflow_acc) { p->results[g] = DpResult(); p->results[g].status = PSD_ST_PIECE_OVERFLOW; }
            overflow_acc.clear();
            continue;
          }
          gcap *= 2;
        }
        global_tier = true;
        todo.swap(overflow_acc);
      } else break;
    }
    const int n = (int)todo.size();
    DpKernelParams K;
    K.problems = p->d_problems; K.order = p->d_order; K.n_order = n; K.queue = p->d_queue; K.results = p->d_results;
    K.pool.base = p->d_pool; K.pool.cursor = p->d_cursors; K.pool.n_chunks = p->pool_bytes / chunk; K.pool.chunk_bytes = chunk;
    K.pool.host_base = p->d_spill; K.pool.host_cursor = p->d_cursors + 2; K.pool.host_chunks = p->spill_bytes / chunk;
    memset(&K.pool.ring, 0, sizeof K.pool.ring);
    K.lat_help = 0;
    int grid; size_t smem; int wpb; int which = 0; int blocks = 1;
    // Few problems (a sequential search on one chromosome, the worst-case sequences, single calls):
    // the latency kernel, one problem per block and one chain per warp (fpop_lat.cu)
    const int n_sm = p->prop.multiProcessorCount;
    const int per_sm = (n + n_sm - 1) / n_sm;
    const bool lat = choose_latency_kernel(p, todo);
    if (lat) {
      wpb = PSD_LAT_WARPS;
      if (!global_tier) {
        const int resident = std::max(1, std::min(per_sm, 4));   // more than 4 resident blocks per SM gain nothing (measured)
        const size_t per_block = std::min((size_t)p->prop.sharedMemPerMultiprocessor / resident - 1024, (size_t)p->prop.sharedMemPerBlockOptin);
        long cap = ((long)per_block - PSD_TAB_BYTES - PSD_LAT_SHARED_BYTES - 32) / 328;   // PSD_WS_BYTES(cap, 2 cap) = 16 + 328 cap
        cap = std::min(640L, cap) & ~3L;
        if (p->opt.piece_cap < 48) cap = std::min(cap, (long)((p->opt.piece_cap + 3) & ~3));   // a tier below the default is a request (tests force the global tier with it)
        if (cap < 8) cap = 8;
        K.cap_s = (int)cap; K.ccap_s = 2 * K.cap_s; K.ws_s_bytes = psd_ws_bytes(K.cap_s, K.ccap_s);
        // the block's global workspace takes what outgrows shared memory: with one block per SM it is
        // sized for the worst-case sequences (config 5) so that no host-level re-run is needed
        K.cap_g = (n <= n_sm) ? std::max(p->opt.spill_cap, std::min(p->opt.overflow_cap, 32768)) : p->opt.spill_cap;
        K.ccap_g = 3 * K.cap_g; K.ws_g_bytes = psd_ws_bytes(K.cap_g, K.ccap_g);
      } else {
        K.cap_s = 0; K.ccap_s = 0; K.ws_s_bytes = psd_ws_bytes(0, 0);
        K.cap_g = gcap; K.ccap_g = 3 * gcap; K.ws_g_bytes = psd_ws_bytes(K.cap_g, K.ccap_g);
      }
      smem = PSD_TAB_BYTES + PSD_LAT_SHARED_BYTES + (size_t)K.ws_s_bytes;
      grid = n;
      // helper warps pay with one block per SM (-9 % per row); with more resident blocks they cost more than they give (measured)
      K.lat_help = per_sm <= 1 ? 1 : 0;
      S.piece_cap = K.cap_s; S.warps_per_sm = (K.lat_help ? 4 : PSD_LAT_WARPS) * std::min(per_sm, std::max(1, psd_lat_resident_blocks(smem, K.lat_help)));
    } else if (!global_tier) {
      // shared-memory tier, with a per-warp global workspace the kernel moves to (and back from)
      // when a row's functions outgrow shared memory
      which = choose_config(p, todo);
      const psd_plan::LaunchCfg& L = p->cfg[which];
      K.cap_s = L.cap; K.ccap_s = L.ccap; K.ws_s_bytes = psd_ws_bytes(K.cap_s, K.ccap_s);
      K.cap_g = p->opt.spill_cap; K.ccap_g = 3 * K.cap_g; K.ws_g_bytes = psd_ws_bytes(K.cap_g, K.ccap_g);
      smem = L.smem; wpb = L.wpb; blocks = L.blocks;
      S.piece_cap = L.cap; S.warps_per_sm = L.wpb * L.blocks;
    } else {
      // host-level re-run of problems that outgrew even that: global lists only
      K.cap_s = 0; K.ccap_s = 0; K.ws_s_bytes = psd_ws_bytes(0, 0);
      K.cap_g = gcap; K.ccap_g = 3 * gcap; K.ws_g_bytes = psd_ws_bytes(K.cap_g, K.ccap_g);
      wpb = std::min(8, PSD_MAX_WARPS_PER_BLOCK);
      smem = PSD_TAB_BYTES + (size_t)wpb * K.ws_s_bytes;
    }
    if (!lat) grid = std::max(1, std::min(p->prop.multiProcessorCount * blocks, n));   // a small batch spreads one warp per SM
    K.gws = nullptr;
    if (K.cap_g > 0) {
      const unsigned long long need = (unsigned long long)grid * (lat ? 1 : wpb) * K.ws_g_bytes;
      if (need > p->gws_bytes) { dfree(p->d_gws); p->gws_bytes = 0; CK(cudaMalloc(&p->d_gws, need)); p->gws_bytes = need; }
      K.gws = p->d_gws;
    }
    tr.mark("solve: descriptors + workspace");
    if (!p->d_queue) CK(cudaMalloc(&p->d_queue, sizeof(int)));
    CK(cudaMemcpyAsync(p->d_order, todo.data(), sizeof(int) * n, cudaMemcpyHostToDevice, st));
    *p->p_queue_init = grid * wpb;   // slots below this are assigned statically
    CK(cudaMemcpyAsync(p->d_queue, p->p_queue_init, sizeof(int), cudaMemcpyHostToDevice, st));
    p->solve_h2d_bytes += (int64_t)(sizeof(int) * (n + 1));
    K.queue = p->d_queue;
    CK(cudaMemsetAsync(p->d_cursors, 0, sizeof(unsigned long long), st));   // recycle the store pool
    CK(cudaMemsetAsync(p->d_cursors + 2, 0, sizeof(unsigned long long), st));
    // spill through the DMA drain: an HBM ring that a host thread empties into the pinned host region
    const bool use_ring = p->d_spill != nullptr && p->opt.spill_mode == 0 && K.pool.host_chunks > 0;
    RingDrain drain;
    if (use_ring) {
      rc = ring_prepare(p, chunk, (unsigned long long)grid * (unsigned long long)(lat ? 1 : wpb));
      if (rc) return rc;
      const unsigned qlen = p->ring_qlen;
      memset(p->h_ringq, 0, 64 + 20ull * qlen);
      unsigned int* fq = (unsigned int*)(p->h_ringq + 64);
      for (unsigned long long i = 0; i < p->ring_slots; i++) fq[i] = (unsigned int)i;
      *(volatile unsigned long long*)p->h_ringq = p->ring_slots;
      CK(cudaMemsetAsync(p->d_cursors + 4, 0, 2 * sizeof(unsigned long long), st));
      K.pool.ring.base = p->d_ring; K.pool.ring.n_slots = p->ring_slots;
      K.pool.ring.head = p->d_cursors + 4; K.pool.ring.done_head = p->d_cursors + 5;
      K.pool.ring.free_tail = (volatile unsigned long long*)p->d_ringq;
      K.pool.ring.free_q = (volatile unsigned int*)(p->d_ringq + 64);
      K.pool.ring.done_q = (volatile unsigned long long*)(p->d_ringq + 64 + 4ull * qlen);
      K.pool.ring.q_mask = qlen - 1;
      drain.p = p; drain.chunk = chunk;
    }
    CK(cudaEventRecord(p->ev[2], st));
    if (lat) {
      CK((cudaError_t)psd_lat_set_smem(smem));
      CK((cudaError_t)psd_lat_launch(K, grid, smem, st));
      S.n_latency_waves++;
    } else {
      if (which == 1) fpop_dp_kernel<14, 2><<<grid, wpb * 32, smem, st>>>(K);
      else fpop_dp_kernel<PSD_MAX_WARPS_PER_BLOCK, 1><<<grid, wpb * 32, smem, st>>>(K);
      CK(cudaGetLastError());
    }
    CK(cudaEventRecord(p->ev[3], st));
    if (use_ring) {
      // the drain runs while the kernel does; the backtrack may only start when every published chunk is on the host
      drain.th = std::thread([&drain]() { drain.run(); });
      const cudaError_t e1 = cudaEventSynchronize(p->ev[3]);
      unsigned long long done_total = 0;
      const cudaError_t e2 = (e1 == cudaSuccess) ? cudaMemcpyAsync(&done_total, p->d_cursors + 5, sizeof done_total, cudaMemcpyDeviceToHost, p->drain_stream) : e1;
      const cudaError_t e3 = (e2 == cudaSuccess) ? cudaStreamSynchronize(p->drain_stream) : e2;
      drain.final_count.store(e3 == cudaSuccess ? done_total : 0ull, std::memory_order_release);
      drain.th.join();
      CK(e3);
      if (drain.error.load()) { g_last_error = "store drain: a DMA copy failed"; return PSD_ERR_CUDA; }
      S.store_bytes_drained_dma += (int64_t)(drain.drained * chunk);
    }
    BtKernelParams B;
    B.problems = p->d_problems; B.order = p->d_order; B.n_order = n; B.results = p->d_results; B.pool = K.pool;
    B.seg_scratch_off = p->d_seg_scratch_off; B.scratch_row = p->d_scratch_row; B.scratch_x = p->d_scratch_x;
    B.seg_row = p->d_seg_row; B.seg_x = p->d_seg_x; B.seg_cursor = p->d_cursors + 1;
    B.end_base = p->n_count_problems ? p->d_end : nullptr; B.end_off = p->d_end_off;
    fpop_backtrack_kernel<<<(n + PSD_BT_WARPS_PER_BLOCK - 1) / PSD_BT_WARPS_PER_BLOCK, PSD_BT_WARPS_PER_BLOCK * 32, 0, st>>>(B);
    CK(cudaGetLastError());
    CK(cudaEventRecord(p->ev[4], st));
    S.n_launches += 2; S.n_waves++;
    if (p->n_labels) {
      LabelParams L;
      L.results = p->d_results; L.order = p->d_order; L.n_order = n; L.seg_row = p->d_seg_row; L.desc = p->d_label_desc;
      L.labels = p->d_labels; L.fp = p->d_label_fp; L.fn = p->d_label_fn; L.totals = p->d_label_tot;
      label_errors_kernel<<<(n + PSD_LABEL_WARPS_PER_BLOCK - 1) / PSD_LABEL_WARPS_PER_BLOCK, PSD_LABEL_WARPS_PER_BLOCK * 32, 0, st>>>(L);
      CK(cudaGetLastError());
      CK(cudaEventRecord(p->ev[7], st));
      S.n_launches++;
    }
    p->last_hbm_bytes = K.pool.n_chunks * chunk;
    // the wave's status words decide what (if anything) has to be re-run
    CK(cudaMemcpyAsync(p->p_results, p->d_results, sizeof(DpResult) * ng, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(p->p_cursors, p->d_cursors, sizeof(unsigned long long) * 8, cudaMemcpyDeviceToHost, st));
    p->solve_d2h_bytes += (int64_t)(sizeof(DpResult) * ng + sizeof(unsigned long long) * 8);
    if (p->n_labels) {   // the label results come back with the status words
      CK(cudaMemcpyAsync(p->p_label_tot, p->d_label_tot, sizeof(int) * 5 * ng, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(p->p_label_fp, p->d_label_fp, sizeof(int) * p->n_labels, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(p->p_label_fn, p->d_label_fn, sizeof(int) * p->n_labels, cudaMemcpyDeviceToHost, st));
      p->solve_d2h_bytes += (int64_t)(sizeof(int) * (5 * ng + 2 * p->n_labels));
    }
    tr.mark("solve: launches enqueued");
    CK(cudaStreamSynchronize(st));
    tr.mark("solve: kernels + status D2H");
    float ms = 0;
    cudaEventElapsedTime(&ms, p->ev[2], p->ev[3]); S.dp_ms += ms;
    cudaEventElapsedTime(&ms, p->ev[3], p->ev[4]); S.backtrack_ms += ms;
    if (p->n_labels) { cudaEventElapsedTime(&ms, p->ev[4], p->ev[7]); p->label_ms += ms; }
    S.store_bytes_written += (int64_t)(std::min<unsigned long long>(p->p_cursors[0], K.pool.n_chunks) * chunk);
    S.store_bytes_spilled_host += (int64_t)(std::min<unsigned long long>(p->p_cursors[2] + (use_ring ? p->p_cursors[5] : 0ull), K.pool.host_chunks) * chunk);
    std::vector<int> exhausted;
    for (int g : todo) {
      const DpResult& r = p->p_results[g];
      if (r.status == PSD_ST_PIECE_OVERFLOW) overflow_acc.push_back(g);
      else if (r.status == PSD_ST_STORE_EXHAUSTED) exhausted.push_back(g);
      else { p->results[g] = r; p->result_wave[g] = S.n_waves; if (r.pad_ > 0) S.n_overflow_tier++; }
    }
    if (!exhausted.empty()) {
      // Some problems ran out of store.  In order of preference: a bigger HBM pool (the automatic
      // size is only an estimate of ~1 KB per row), then overflow into mapped pinned host memory,
      // and only then smaller waves that recycle the pool.
      size_t free_b = 0, total_b = 0;
      CK(cudaMemGetInfo(&free_b, &total_b));
      const unsigned long long lim = (((unsigned long long)((double)(free_b + p->pool_bytes) * 0.80)) / chunk) * chunk;
      bool retry_bigger = false;
      if (p->opt.store_gb <= 0 && p->pool_bytes * 2 <= lim) {
        const unsigned long long want = std::min(lim, p->pool_bytes * 4);
        dfree(p->d_pool); p->pool_bytes = 0;
        CK(cudaMalloc(&p->d_pool, want));
        p->pool_bytes = want;
        retry_bigger = true;
      } else {
        // The prediction was too low for these problems.  They are re-run in later waves (each
        // recycles the store) unless the largest of them cannot fit the store at all: only then is
        // pinned host memory added (pinning costs ~0.3 s per GB), sized for that problem.
        est_row_bytes *= 1.3;
        double largest = 0;
        for (int g : exhausted) largest = std::max(largest, est_row_bytes * (double)p->probs[p->gpu_ids[g]].n_rows);
        if (largest > (double)(p->pool_bytes + p->spill_bytes) && !p->d_spill && p->opt.host_spill_gb != 0) {
          const double gb = std::min(host_spill_limit_gb(p), 1.3 * (largest - 0.8 * (double)p->pool_bytes) / (double)(1ull << 30) + 0.25);
          retry_bigger = alloc_host_spill(p, gb, chunk);
        }
        if (!retry_bigger && (int)exhausted.size() < n) {   // part of the wave fitted: the rest goes into planned later waves
          std::vector<int> later;
          plan_wave(exhausted, later);
          deferred.insert(deferred.end(), later.begin(), later.end());
        }
      }
      if (!retry_bigger && (int)exhausted.size() == n) {   // same store, and it held none of them
        if (n == 1) { p->results[exhausted[0]] = p->p_results[exhausted[0]]; exhausted.clear(); }
        else {
          const int h = (n + 1) / 2;
          deferred.insert(deferred.end(), exhausted.begin() + h, exhausted.end());
          exhausted.resize(h);
        }
      }
    }
    todo.swap(exhausted);
  }
  // algorithmic bytes (SURVEY.md 8d): per problem N*24 + 20*total_intervals
  double sum_iv = 0, sum_rows = 0;
  for (size_t g = 0; g < ng; g++) {
    const DpResult& r = p->results[g];
    const HostProblem& h = p->probs[p->gpu_ids[g]];
    if (r.status == 0) {
      S.rows_solved += h.n_rows;
      S.store_bytes_algorithmic += h.n_rows * 24 + 20 * (int64_t)r.total_intervals;
      S.backtrack_bytes_read += (int64_t)r.bt_bytes;
      sum_iv += (double)r.total_intervals; sum_rows += (double)h.n_rows;
    }
  }
  if (sum_rows > 0) p->last_mean_intervals = sum_iv / (2.0 * sum_rows);
  p->n_seg_total = p->p_cursors[1];
  for (size_t g = 0; g < ng; g++) {   // label errors of the GPU problems
    HostProblem& h = p->probs[p->gpu_ids[g]];
    h.label_status = -1; h.label_fp.clear(); h.label_fn.clear();
    if (!h.labels) continue;
    h.label_status = p->results[g].status;
    if (h.label_status != 0) continue;
    const int* t = p->p_label_tot + 5 * g;
    h.label_total = psd_label_errors{t[0], t[1], t[2], t[3], t[4]};
    const LabelDesc& d = p->label_desc[g];
    h.label_fp.assign(p->p_label_fp + d.off, p->p_label_fp + d.off + d.n);
    h.label_fn.assign(p->p_label_fn + d.off, p->p_label_fn + d.off + d.n);
  }
  p->solved = true;
  return 0;
}

void psd_plan_collect_results(psd_plan* p) {
  for (size_t g = 0; g < p->gpu_ids.size(); g++) {
    HostProblem& h = p->probs[p->gpu_ids[g]];
    const DpResult& r = p->results[g];
    h.result_status = r.status;
    if (r.status != 0) continue;
    h.n_segments = r.n_segments; h.n_equality = r.n_equality;
    h.best_cost = r.best_cost; h.total_intervals = (double)r.total_intervals; h.max_intervals = r.max_intervals;
  }
}

PlanSolveTotals psd_plan_solve_totals(const psd_plan* p) {
  const psd_stats& S = p->stats;
  return PlanSolveTotals{S.dp_ms, S.backtrack_ms, p->label_ms, S.rows_solved, S.h2d_bytes + p->solve_h2d_bytes, p->solve_d2h_bytes};
}

int psd_plan_download_impl(psd_plan* p, void* stream_v) {
  cudaStream_t st = (cudaStream_t)stream_v;
  if (!p->solved) { g_last_error = "psd_plan_download before psd_plan_solve"; return PSD_ERR_ARG; }
  const size_t ng = p->gpu_ids.size();
  if (ng) CK(cudaSetDevice(p->device));
  p->stats.d2h_bytes = 0; p->stats.d2h_ms = 0;
  if (ng) {
    const unsigned long long ns = p->n_seg_total;
    if (ns > p->p_seg_cap) {
      if (p->p_seg_row) cudaFreeHost(p->p_seg_row); if (p->p_seg_x) cudaFreeHost(p->p_seg_x);
      p->p_seg_row = nullptr; p->p_seg_x = nullptr; p->p_seg_cap = 0;
      const size_t want = (size_t)(ns + ns / 4 + 1024);
      CK(cudaMallocHost(&p->p_seg_row, sizeof(int) * want));
      CK(cudaMallocHost(&p->p_seg_x, sizeof(double) * want));
      p->p_seg_cap = want;
    }
    CK(cudaEventRecord(p->ev[5], st));
    if (ns) {
      CK(cudaMemcpyAsync(p->p_seg_row, p->d_seg_row, sizeof(int) * ns, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(p->p_seg_x, p->d_seg_x, sizeof(double) * ns, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaEventRecord(p->ev[6], st));
    CK(cudaStreamSynchronize(st));
    float ms = 0; cudaEventElapsedTime(&ms, p->ev[5], p->ev[6]);
    p->stats.d2h_ms = ms;
    p->stats.d2h_bytes = (int64_t)(12 * ns + sizeof(DpResult) * ng);
  }
  // fill the host problems' results
  for (size_t g = 0; g < ng; g++) {
    HostProblem& h = p->probs[p->gpu_ids[g]];
    const DpResult& r = p->results[g];
    h.seg_row.clear(); h.seg_x.clear();
    if (r.status != 0) { h.result_status = r.status; continue; }
    h.result_status = 0;
    h.n_segments = r.n_segments; h.n_equality = r.n_equality;
    h.best_cost = r.best_cost; h.total_intervals = (double)r.total_intervals; h.max_intervals = r.max_intervals;
    h.seg_row.assign(p->p_seg_row + r.seg_offset, p->p_seg_row + r.seg_offset + r.n_segments);
    h.seg_x.assign(p->p_seg_x + r.seg_offset, p->p_seg_x + r.seg_offset + r.n_segments);
  }
  return 0;
}

// Reads one stored cost function back (what DiskVector::read does in the reference,
// src/PeakSegFPOPLog.cpp:103-117): the record of `row`, function `which` (0 up, 1 down), as the
// reference's record fields max_log_mean / data_i / prev_log_mean.  Valid after a solve that needed
// a single store wave (the pool then still holds every record).  A few small D2H copies per call:
// an inspection path for tests and tools, not a hot path.
int psd_plan_store_function_impl(psd_plan* p, int id, int row, int which, int cap, int* n_out, double* hi, int* back_i, double* back_x) {
  if (!p->solved) { g_last_error = "store inspection needs a solved plan"; return PSD_ERR_ARG; }
  if (id < 0 || id >= (int)p->probs.size() || which < 0 || which > 1 || !n_out) return PSD_ERR_ARG;
  const HostProblem& h = p->probs[id];
  if (h.status != 0 || h.trivial || h.result_status != 0 || row < 0 || row >= h.n_rows) return PSD_ERR_ARG;
  {
    const auto it = std::find(p->gpu_ids.begin(), p->gpu_ids.end(), id);
    if (it == p->gpu_ids.end() || p->result_wave[it - p->gpu_ids.begin()] != p->stats.n_waves) {
      g_last_error = "store inspection: this problem was solved in an earlier store wave, its records have been recycled";
      return PSD_ERR_ARG;
    }
  }
  CK(cudaSetDevice(p->device));
  unsigned long long off = 0;
  CK(cudaMemcpy(&off, p->d_index + h.index_off + row, sizeof off, cudaMemcpyDeviceToHost));
  auto fetch = [&](void* dst, unsigned long long o, size_t bytes) -> cudaError_t {
    if (o < p->last_hbm_bytes) return cudaMemcpy(dst, p->d_pool + o, bytes, cudaMemcpyDeviceToHost);
    memcpy(dst, p->h_spill + (o - p->last_hbm_bytes), bytes);     // spilled record: already in pinned host memory
    return cudaSuccess;
  };
  unsigned hdr[4];
  CK(fetch(hdr, off, sizeof hdr));
  if ((int)hdr[2] != row) { g_last_error = "store record does not belong to the requested row"; return PSD_ERR_INTERNAL; }
  const int n_up = (int)hdr[0], n_down = (int)hdr[1];
  const int n = which ? n_down : n_up;
  *n_out = n;
  if (n > cap) return PSD_ERR_ARG;
  if (n == 0) return 0;
  const RecLayout R = rec_layout(n_up, n_down);
  CK(fetch(hi, off + R.hi[which], 8ull * n));
  CK(fetch(back_x, off + R.bx[which], 8ull * n));
  CK(fetch(back_i, off + R.bi[which], 4ull * n));
  return 0;
}

// ---- coverage from aligned reads (psd_coverage_from_reads, coverage_gpu.cuh) -------------------------
namespace {
// Device arena, pinned staging and events of one psd_coverage_from_reads call, freed on every return.
struct CovScratch {
  unsigned char* d_arena = nullptr; size_t arena_bytes = 0;
  int32_t *p_start = nullptr, *p_end = nullptr; size_t p_reads_cap = 0;   // reads of a wave
  int32_t *p_cov = nullptr, *p_rend = nullptr; size_t p_rows_cap = 0;     // rows of a wave
  int* p_small = nullptr;                                                 // n_rows of a wave's problems + 2 error flags
  cudaEvent_t ev[6]; bool ev_ok = false;
  ~CovScratch() {
    if (d_arena) cudaFree(d_arena);
    if (p_start) cudaFreeHost(p_start); if (p_end) cudaFreeHost(p_end);
    if (p_cov) cudaFreeHost(p_cov); if (p_rend) cudaFreeHost(p_rend); if (p_small) cudaFreeHost(p_small);
    if (ev_ok) for (auto& e : ev) cudaEventDestroy(e);
  }
};

struct CovJob {
  int prob;
  int64_t n_reads, n_bases, row_bound, n_tiles;
};

inline size_t cov_align(size_t b) { return (b + 255) & ~(size_t)255; }

// device bytes of a wave (the arena is carved in this order, see psd_coverage_from_reads_impl)
size_t cov_wave_bytes(int64_t n_probs, int64_t bases, int64_t rows, int64_t reads, int64_t tiles) {
  return cov_align(4 * bases) + 2 * cov_align(4 * reads) + 3 * cov_align(4 * rows) + cov_align(sizeof(RleVec) * n_probs) +
         cov_align(8 * (n_probs + 1)) + 2 * cov_align(4 * n_probs) + cov_align(4 * tiles) + 2 * cov_align(8 * (tiles + 1));
}
}  // namespace

// Host checks (before any device work), then waves of problems whose device footprint fits the
// "coverage_gb" budget: H2D of the reads, zero-fill, scatter, scan, RLE, D2H of the rows.  Problems
// without a read inside their region never reach the device: their one zero row is made here.
int psd_coverage_from_reads_impl(int device, int n, const psd_reads* P, psd_coverage** out) {
  if (!out) { g_last_error = "psd_coverage_from_reads: out is null"; return PSD_ERR_ARG; }
  *out = nullptr;
  if (n < 0 || (n > 0 && !P)) { g_last_error = "psd_coverage_from_reads: n_problems < 0 or problems is null"; return PSD_ERR_ARG; }
  std::vector<int64_t> inside(n, 0);   // reads that overlap the region
  std::vector<std::string> err(n);
  auto check = [&](int k) {
    const psd_reads& q = P[k];
    char msg[192];
    if (q.n_reads < 0 || q.n_reads >= (1ll << 31)) snprintf(msg, sizeof msg, "n_reads %lld is outside [0, 2^31)", (long long)q.n_reads);
    else if (q.n_reads > 0 && (!q.read_start || !q.read_end)) snprintf(msg, sizeof msg, "read_start or read_end is null with n_reads %lld", (long long)q.n_reads);
    else if (q.region_start < 0) snprintf(msg, sizeof msg, "region_start %d < 0", q.region_start);
    else if (q.region_end <= q.region_start) snprintf(msg, sizeof msg, "region_end %d <= region_start %d", q.region_end, q.region_start);
    else if ((int64_t)q.region_end - q.region_start > 0x3fffffff) snprintf(msg, sizeof msg, "region of %lld bases is longer than 0x3fffffff", (long long)q.region_end - q.region_start);
    else {
      int64_t m = 0;
      for (int64_t r = 0; r < q.n_reads; r++) {
        const int32_t s = q.read_start[r], e = q.read_end[r];
        if (s < 0) { snprintf(msg, sizeof msg, "read %lld: start %d < 0", (long long)r, s); err[k] = msg; return; }
        if (e <= s) { snprintf(msg, sizeof msg, "read %lld: end %d <= start %d", (long long)r, e, s); err[k] = msg; return; }
        m += (e > q.region_start && s < q.region_end);
      }
      inside[k] = m;
      return;
    }
    err[k] = msg;
  };
  int64_t all_reads = 0;
  for (int k = 0; k < n; k++) all_reads += P[k].n_reads > 0 ? P[k].n_reads : 0;
  if (all_reads > (1 << 22)) parallel_for(n, check);
  else for (int k = 0; k < n; k++) check(k);
  for (int k = 0; k < n; k++)
    if (!err[k].empty()) { g_last_error = "psd_coverage_from_reads: problem " + std::to_string(k) + ": " + err[k]; return PSD_ERR_ARG; }

  std::unique_ptr<psd_coverage> C(new psd_coverage());
  psd_coverage_stats& S = C->stats;
  memset(&S, 0, sizeof S);
  S.n_problems = n;
  C->row_off.assign(1, 0);
  auto emit = [&](int32_t s, int32_t e, int32_t c) { C->chrom_start.push_back(s); C->chrom_end.push_back(e); C->count.push_back(c); };
  int next_emit = 0;
  auto emit_empty_until = [&](int k_end) {   // problems before k_end that have no read in their region: one zero row
    for (; next_emit < k_end; next_emit++) {
      emit(P[next_emit].region_start, P[next_emit].region_end, 0);
      C->row_off.push_back((int64_t)C->count.size());
    }
  };
  std::vector<CovJob> jobs;
  for (int k = 0; k < n; k++) {
    if (!inside[k]) continue;
    const int64_t nb = (int64_t)P[k].region_end - P[k].region_start;
    jobs.push_back({k, P[k].n_reads, nb, std::min(nb, 2 * inside[k] + 1), (nb + PSD_RLE_TILE - 1) / PSD_RLE_TILE});
  }
  if (!jobs.empty()) {
    int ndev = 0;
    if (!cuda_ok(cudaGetDeviceCount(&ndev), "cudaGetDeviceCount")) return PSD_ERR_CUDA;
    if (ndev == 0) { g_last_error = "no CUDA device"; return PSD_ERR_CUDA; }
    if (device < 0) CK(cudaGetDevice(&device));
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { g_last_error = "peaksegdisk_b200 is built for sm_100a only"; return PSD_ERR_CUDA; }
    CovScratch X;
    for (auto& e : X.ev) CK(cudaEventCreate(&e));
    X.ev_ok = true;
    // waves: consecutive jobs while their footprint fits the budget (a job larger than it runs alone)
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const double gb = current_options().coverage_gb;
    const size_t budget = gb > 0 ? (size_t)(gb * (double)(1ull << 30)) : free_b / 2;
    std::vector<std::pair<size_t, size_t>> waves;   // [first job, end job)
    size_t arena = 0, max_reads = 0;
    for (size_t j0 = 0; j0 < jobs.size();) {
      size_t j1 = j0;
      int64_t bases = 0, rows = 0, reads = 0, tiles = 0;
      size_t bytes = 0;
      for (; j1 < jobs.size(); j1++) {
        const CovJob& J = jobs[j1];
        const size_t b = cov_wave_bytes((int64_t)(j1 - j0 + 1), bases + J.n_bases, rows + J.row_bound, reads + J.n_reads, tiles + J.n_tiles);
        if (j1 > j0 && b > budget) break;
        bases += J.n_bases; rows += J.row_bound; reads += J.n_reads; tiles += J.n_tiles; bytes = b;
      }
      waves.push_back({j0, j1});
      arena = std::max(arena, bytes); max_reads = std::max(max_reads, (size_t)reads);
      j0 = j1;
    }
    CK(cudaMalloc(&X.d_arena, arena));
    X.arena_bytes = arena;
    CK(cudaMallocHost(&X.p_start, 4 * max_reads));
    CK(cudaMallocHost(&X.p_end, 4 * max_reads));
    X.p_reads_cap = max_reads;
    size_t max_probs = 0;
    for (const auto& w : waves) max_probs = std::max(max_probs, w.second - w.first);
    CK(cudaMallocHost(&X.p_small, sizeof(int) * (max_probs + 2)));
    const cudaStream_t st = 0;
    for (const auto& w : waves) {
      const int np = (int)(w.second - w.first);
      std::vector<RleVec> vecs(np);
      std::vector<long long> read_off(np + 1, 0);
      std::vector<int> region(np), tile_vec;
      int64_t bases = 0, rows = 0, reads = 0;
      for (int j = 0; j < np; j++) {
        const CovJob& J = jobs[w.first + j];
        RleVec& v = vecs[j];
        v.raw_off = bases; v.row_off = rows; v.n_pos = (int)J.n_bases; v.tile0 = (int)tile_vec.size();
        tile_vec.insert(tile_vec.end(), (size_t)J.n_tiles, j);
        region[j] = P[J.prob].region_start;
        read_off[j] = reads;
        bases += J.n_bases; rows += J.row_bound; reads += J.n_reads;
      }
      read_off[np] = reads;
      const int n_tiles = (int)tile_vec.size();
      auto stage = [&](int j) {
        const psd_reads& q = P[jobs[w.first + j].prob];
        memcpy(X.p_start + read_off[j], q.read_start, 4 * (size_t)q.n_reads);
        memcpy(X.p_end + read_off[j], q.read_end, 4 * (size_t)q.n_reads);
      };
      if (reads > (1 << 22)) parallel_for(np, stage);
      else for (int j = 0; j < np; j++) stage(j);
      // carve the arena (the order cov_wave_bytes() counts)
      unsigned char* a = X.d_arena;
      auto carve = [&](size_t b) { unsigned char* r = a; a += cov_align(b); return r; };
      int* d_cov = (int*)carve(4 * bases);
      int* d_start = (int*)carve(4 * reads);
      int* d_end = (int*)carve(4 * reads);
      int* d_rcov = (int*)carve(4 * rows);
      int* d_rend = (int*)carve(4 * rows);
      int* d_rw = (int*)carve(4 * rows);
      RleVec* d_vecs = (RleVec*)carve(sizeof(RleVec) * np);
      long long* d_read_off = (long long*)carve(8 * (np + 1));
      int* d_region = (int*)carve(4 * np);
      int* d_nrows = (int*)carve(4 * np);
      int* d_tile_vec = (int*)carve(4 * n_tiles);
      unsigned long long* d_scan_state = (unsigned long long*)carve(8 * (n_tiles + 1));   // look-back words, then ticket and error flag
      unsigned long long* d_rle_state = (unsigned long long*)carve(8 * (n_tiles + 1));
      CK(cudaEventRecord(X.ev[0], st));
      CK(cudaMemcpyAsync(d_start, X.p_start, 4 * reads, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(d_end, X.p_end, 4 * reads, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(d_vecs, vecs.data(), sizeof(RleVec) * np, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(d_read_off, read_off.data(), 8 * (np + 1), cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(d_region, region.data(), 4 * np, cudaMemcpyHostToDevice, st));
      CK(cudaMemcpyAsync(d_tile_vec, tile_vec.data(), 4 * (size_t)n_tiles, cudaMemcpyHostToDevice, st));
      CK(cudaEventRecord(X.ev[1], st));
      CK(cudaMemsetAsync(d_cov, 0, 4 * bases, st));
      CK(cudaMemsetAsync(d_scan_state, 0, 8 * (n_tiles + 1), st));
      CK(cudaMemsetAsync(d_rle_state, 0, 8 * (n_tiles + 1), st));
      CovScatterParams A;
      A.read_start = d_start; A.read_end = d_end; A.n_reads = reads; A.read_off = d_read_off; A.region_start = d_region;
      A.vecs = d_vecs; A.n_probs = np; A.delta = d_cov;
      const long long want_blocks = (reads + 255) / 256;
      reads_scatter_kernel<<<(int)std::min<long long>(want_blocks, 16ll * prop.multiProcessorCount), 256, 0, st>>>(A);
      CK(cudaGetLastError());
      CovScanParams B;
      B.vecs = d_vecs; B.tile_vec = d_tile_vec; B.n_tiles = n_tiles; B.cov = d_cov;
      B.tile_state = d_scan_state; B.ticket = (unsigned int*)(d_scan_state + n_tiles); B.error = (int*)(B.ticket + 1);
      coverage_scan_kernel<<<n_tiles, PSD_RLE_WARPS * 32, 0, st>>>(B);
      CK(cudaGetLastError());
      RleParams R;
      R.vecs = d_vecs; R.tile_vec = d_tile_vec; R.n_tiles = n_tiles; R.n_vecs = np;
      R.raw = d_cov; R.coverage = d_rcov; R.chrom_end = d_rend; R.weight = d_rw;
      R.tile_state = d_rle_state; R.n_rows = d_nrows;
      R.ticket = (unsigned int*)(d_rle_state + n_tiles); R.error = (int*)(R.ticket + 1);
      rle_encode_kernel<<<n_tiles, PSD_RLE_WARPS * 32, 0, st>>>(R);
      CK(cudaGetLastError());
      CK(cudaEventRecord(X.ev[2], st));
      CK(cudaMemcpyAsync(X.p_small, d_nrows, 4 * np, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(X.p_small + np, B.error, 4, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(X.p_small + np + 1, R.error, 4, cudaMemcpyDeviceToHost, st));
      CK(cudaEventRecord(X.ev[3], st));
      CK(cudaStreamSynchronize(st));
      if (X.p_small[np] || X.p_small[np + 1]) { g_last_error = "device coverage: look-back gave up"; return PSD_ERR_INTERNAL; }
      int64_t got = 0;
      for (int j = 0; j < np; j++) {
        const int nr = X.p_small[j];
        if (nr < 1 || nr > jobs[w.first + j].row_bound) { g_last_error = "device coverage: row count outside its bound"; return PSD_ERR_INTERNAL; }
        got += nr;
      }
      if ((size_t)got > X.p_rows_cap) {
        if (X.p_cov) cudaFreeHost(X.p_cov); if (X.p_rend) cudaFreeHost(X.p_rend);
        X.p_cov = X.p_rend = nullptr; X.p_rows_cap = 0;
        CK(cudaMallocHost(&X.p_cov, 4 * got));
        CK(cudaMallocHost(&X.p_rend, 4 * got));
        X.p_rows_cap = got;
      }
      // rows: exact counts per problem, packed into the staging
      CK(cudaEventRecord(X.ev[4], st));
      int64_t o = 0;
      for (int j = 0; j < np; j++) {
        const int nr = X.p_small[j];
        CK(cudaMemcpyAsync(X.p_cov + o, d_rcov + vecs[j].row_off, 4 * (size_t)nr, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(X.p_rend + o, d_rend + vecs[j].row_off, 4 * (size_t)nr, cudaMemcpyDeviceToHost, st));
        o += nr;
      }
      CK(cudaEventRecord(X.ev[5], st));
      CK(cudaStreamSynchronize(st));
      float t01 = 0, t13 = 0, t45 = 0, t12 = 0;
      cudaEventElapsedTime(&t01, X.ev[0], X.ev[1]); cudaEventElapsedTime(&t13, X.ev[1], X.ev[3]);
      cudaEventElapsedTime(&t45, X.ev[4], X.ev[5]); cudaEventElapsedTime(&t12, X.ev[1], X.ev[2]);
      S.device_ms += t01 + t13 + t45; S.kernel_ms += t12;
      S.reads += reads; S.bases += bases; S.n_waves++;
      S.h2d_bytes += 8 * reads + (int64_t)(sizeof(RleVec) + 12) * np + 8 + 4 * (int64_t)n_tiles;
      S.d2h_bytes += 4 * (np + 2) + 8 * got;
      o = 0;
      for (int j = 0; j < np; j++) {
        const int k = jobs[w.first + j].prob;
        emit_empty_until(k);
        const int nr = X.p_small[j], r0 = P[k].region_start;
        int prev = r0;
        for (int r = 0; r < nr; r++) {
          const int e = X.p_rend[o + r] + r0;
          emit(prev, e, X.p_cov[o + r]);
          prev = e;
        }
        o += nr;
        C->row_off.push_back((int64_t)C->count.size());
        next_emit = k + 1;
      }
    }
  }
  emit_empty_until(n);
  S.rows = (int64_t)C->count.size();
  *out = C.release();
  return 0;
}

// ---- per-problem coverage statistics (psd_features, features_gpu.cuh) ---------------------------------
namespace {
struct FeatScratch {
  unsigned char* d_arena = nullptr;
  int32_t *p_w = nullptr, *p_c = nullptr;   // weight and count rows of a wave
  cudaEvent_t ev[4]; bool ev_ok = false;
  ~FeatScratch() {
    if (d_arena) cudaFree(d_arena);
    if (p_w) cudaFreeHost(p_w); if (p_c) cudaFreeHost(p_c);
    if (ev_ok) for (auto& e : ev) cudaEventDestroy(e);
  }
};

struct FeatJob {
  int64_t bases;
  int64_t rank[PSD_FEAT_SEL];   // the distinct ranks of x the interior quartiles need, ascending
  int n_sel;
  int64_t n_tiles;
};

// device bytes of a wave (the arena is carved in this order, see psd_features_impl)
size_t feat_wave_bytes(int64_t n_probs, int64_t rows, int64_t tiles, int64_t sels) {
  return 2 * cov_align(4 * rows) + cov_align(sizeof(FeatProblem) * n_probs) + cov_align(4 * tiles) +
         cov_align(sizeof(FeatSel) * sels) + cov_align(2048 * sels) + cov_align(sizeof(FeatSums) * n_probs) + cov_align(4);
}

// R's type-7 quantile at p from x[lo] and x[lo + 1] (h = (B - 1) p, lo = floor(h), g = h - lo); every
// step is exact in fp64 for int32 counts and B < 2^32
void feat_type7(int64_t B, double p, double* h, int64_t* lo, double* g) {
  *h = (double)(B - 1) * p;
  *lo = (int64_t)std::floor(*h);
  *g = *h - (double)*lo;
}
}  // namespace

// Host checks (check_rows, before any device work), then waves of consecutive problems that fit the
// "coverage_gb" budget: H2D of weight and count, four histogram + select passes, D2H of the sums and
// the selected counts; the host turns the integers into the features.
int psd_features_impl(int device, int n, const psd_rows* P, psd_problem_features* out, psd_features_stats* stats) {
  psd_features_stats S;
  memset(&S, 0, sizeof S);
  if (stats) *stats = S;
  if (n < 0 || (n > 0 && (!P || !out))) { g_last_error = "psd_features: n_problems < 0, or problems or out is null"; return PSD_ERR_ARG; }
  std::vector<std::string> err(n);
  std::vector<int> code(n, 0);
  auto check = [&](int k) { code[k] = check_rows(P[k].n_rows, P[k].chromStart, P[k].chromEnd, P[k].coverage, &err[k]); };
  int64_t all_rows = 0;
  for (int k = 0; k < n; k++) all_rows += P[k].n_rows > 0 ? P[k].n_rows : 0;
  if (all_rows > (1 << 22)) parallel_for(n, check);
  else for (int k = 0; k < n; k++) check(k);
  for (int k = 0; k < n; k++)
    if (code[k]) { g_last_error = "psd_features: problem " + std::to_string(k) + ": " + err[k]; return code[k]; }
  if (n == 0) return 0;
  S.n_problems = n;

  std::vector<FeatJob> jobs(n);
  for (int k = 0; k < n; k++) {
    FeatJob& J = jobs[k];
    J.bases = (int64_t)P[k].chromEnd[P[k].n_rows - 1] - P[k].chromStart[0];
    J.n_tiles = (P[k].n_rows + PSD_RLE_TILE - 1) / PSD_RLE_TILE;
    J.n_sel = 0;
    for (double p : {0.25, 0.5, 0.75}) {
      double h, g; int64_t lo;
      feat_type7(J.bases, p, &h, &lo, &g);
      for (int64_t r : {lo, g != 0 ? lo + 1 : lo})
        if (std::find(J.rank, J.rank + J.n_sel, r) == J.rank + J.n_sel) J.rank[J.n_sel++] = r;
    }
    std::sort(J.rank, J.rank + J.n_sel);
  }
  int ndev = 0;
  if (!cuda_ok(cudaGetDeviceCount(&ndev), "cudaGetDeviceCount")) return PSD_ERR_CUDA;
  if (ndev == 0) { g_last_error = "no CUDA device"; return PSD_ERR_CUDA; }
  if (device < 0) CK(cudaGetDevice(&device));
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) { g_last_error = "peaksegdisk_b200 is built for sm_100a only"; return PSD_ERR_CUDA; }
  FeatScratch X;
  for (auto& e : X.ev) CK(cudaEventCreate(&e));
  X.ev_ok = true;
  // waves: consecutive problems while their footprint fits the budget (a problem larger than it runs alone)
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  const double gb = current_options().coverage_gb;
  const size_t budget = gb > 0 ? (size_t)(gb * (double)(1ull << 30)) : free_b / 2;
  std::vector<std::pair<int, int>> waves;   // [first problem, end problem)
  size_t arena = 0, max_rows = 0;
  for (int k0 = 0; k0 < n;) {
    int k1 = k0;
    int64_t rows = 0, tiles = 0, sels = 0;
    size_t bytes = 0;
    for (; k1 < n; k1++) {
      const size_t b = feat_wave_bytes(k1 - k0 + 1, rows + P[k1].n_rows, tiles + jobs[k1].n_tiles, sels + jobs[k1].n_sel);
      if (k1 > k0 && b > budget) break;
      rows += P[k1].n_rows; tiles += jobs[k1].n_tiles; sels += jobs[k1].n_sel; bytes = b;
    }
    waves.push_back({k0, k1});
    arena = std::max(arena, bytes); max_rows = std::max(max_rows, (size_t)rows);
    k0 = k1;
  }
  CK(cudaMalloc(&X.d_arena, arena));
  CK(cudaMallocHost(&X.p_w, 4 * max_rows));
  CK(cudaMallocHost(&X.p_c, 4 * max_rows));
  const cudaStream_t st = 0;
  for (const auto& w : waves) {
    const int np = w.second - w.first;
    std::vector<FeatProblem> probs(np);
    std::vector<FeatSel> sel;
    std::vector<int> tile_prob;
    int64_t rows = 0;
    for (int j = 0; j < np; j++) {
      const FeatJob& J = jobs[w.first + j];
      FeatProblem& q = probs[j];
      q.row_off = rows; q.n_rows = (int)P[w.first + j].n_rows; q.tile0 = (int)tile_prob.size();
      q.sel0 = (int)sel.size(); q.n_sel = J.n_sel;
      tile_prob.insert(tile_prob.end(), (size_t)J.n_tiles, j);
      for (int s = 0; s < J.n_sel; s++) sel.push_back(FeatSel{(unsigned long long)J.rank[s], 0u, q.sel0});
      rows += q.n_rows;
    }
    const int n_tiles = (int)tile_prob.size(), n_sel = (int)sel.size();
    auto stage = [&](int j) {
      const psd_rows& q = P[w.first + j];
      int32_t* pw = X.p_w + probs[j].row_off;
      for (int64_t i = 0; i < q.n_rows; i++) pw[i] = q.chromEnd[i] - q.chromStart[i];
      memcpy(X.p_c + probs[j].row_off, q.coverage, 4 * (size_t)q.n_rows);
    };
    if (rows > (1 << 22)) parallel_for(np, stage);
    else for (int j = 0; j < np; j++) stage(j);
    std::vector<FeatSums> sums(np, FeatSums{0ull, 0ull, 0ull, 0xffffffffu, 0u});
    // carve the arena (the order feat_wave_bytes() counts)
    unsigned char* a = X.d_arena;
    auto carve = [&](size_t b) { unsigned char* r = a; a += cov_align(b); return r; };
    int* d_w = (int*)carve(4 * rows);
    int* d_c = (int*)carve(4 * rows);
    FeatProblem* d_probs = (FeatProblem*)carve(sizeof(FeatProblem) * np);
    int* d_tile_prob = (int*)carve(4 * (size_t)n_tiles);
    FeatSel* d_sel = (FeatSel*)carve(sizeof(FeatSel) * n_sel);
    unsigned long long* d_hist = (unsigned long long*)carve(2048 * (size_t)n_sel);
    FeatSums* d_sums = (FeatSums*)carve(sizeof(FeatSums) * np);
    int* d_err = (int*)carve(4);
    CK(cudaEventRecord(X.ev[0], st));
    CK(cudaMemcpyAsync(d_w, X.p_w, 4 * rows, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_c, X.p_c, 4 * rows, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_probs, probs.data(), sizeof(FeatProblem) * np, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_tile_prob, tile_prob.data(), 4 * (size_t)n_tiles, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_sel, sel.data(), sizeof(FeatSel) * n_sel, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_sums, sums.data(), sizeof(FeatSums) * np, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(X.ev[1], st));
    CK(cudaMemsetAsync(d_hist, 0, 2048 * (size_t)n_sel, st));
    CK(cudaMemsetAsync(d_err, 0, 4, st));
    for (int pass = 0; pass < 4; pass++) {
      FeatHistParams H;
      H.probs = d_probs; H.tile_prob = d_tile_prob; H.n_tiles = n_tiles; H.weight = d_w; H.count = d_c;
      H.sel = d_sel; H.hist = d_hist; H.sums = d_sums;
      H.shift = 24 - 8 * pass; H.mask = pass == 0 ? 0u : 0xffffffffu << (H.shift + 8);
      if (pass == 0) features_hist_kernel<true><<<n_tiles, PSD_RLE_WARPS * 32, 0, st>>>(H);
      else features_hist_kernel<false><<<n_tiles, PSD_RLE_WARPS * 32, 0, st>>>(H);
      CK(cudaGetLastError());
      FeatSelectParams Z;
      Z.probs = d_probs; Z.n_probs = np; Z.sel = d_sel; Z.hist = d_hist; Z.shift = H.shift; Z.error = d_err;
      features_select_kernel<<<(np + 7) / 8, 256, 0, st>>>(Z);
      CK(cudaGetLastError());
      S.n_launches += 2;
    }
    CK(cudaEventRecord(X.ev[2], st));
    int h_err = 0;
    CK(cudaMemcpyAsync(sums.data(), d_sums, sizeof(FeatSums) * np, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(sel.data(), d_sel, sizeof(FeatSel) * n_sel, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h_err, d_err, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(X.ev[3], st));
    CK(cudaStreamSynchronize(st));
    if (h_err) { g_last_error = "device features: a rank fell outside its histogram"; return PSD_ERR_INTERNAL; }
    float t03 = 0, t12 = 0;
    cudaEventElapsedTime(&t03, X.ev[0], X.ev[3]); cudaEventElapsedTime(&t12, X.ev[1], X.ev[2]);
    S.device_ms += t03; S.kernel_ms += t12;
    S.rows += rows; S.n_waves++;
    S.h2d_bytes += 8 * rows + (int64_t)(sizeof(FeatProblem) + sizeof(FeatSums)) * np + 4 * (int64_t)n_tiles + (int64_t)sizeof(FeatSel) * n_sel;
    S.d2h_bytes += (int64_t)sizeof(FeatSums) * np + (int64_t)sizeof(FeatSel) * n_sel + 4;
    for (int j = 0; j < np; j++) {
      const FeatJob& J = jobs[w.first + j];
      const FeatSums& U = sums[j];
      auto x_at = [&](int64_t r) { return (double)sel[probs[j].sel0 + (std::find(J.rank, J.rank + J.n_sel, r) - J.rank)].prefix; };
      psd_problem_features& F = out[w.first + j];
      const int64_t B = J.bases;
      F.quartile[0] = (double)U.min;
      F.quartile[4] = (double)U.max;
      const double ps[3] = {0.25, 0.5, 0.75};
      for (int t = 0; t < 3; t++) {
        double h, g; int64_t lo;
        feat_type7(B, ps[t], &h, &lo, &g);
        const double x0 = x_at(lo);
        if (g == 0) { F.quartile[t + 1] = x0; continue; }
        const double x1 = x_at(lo + 1);
        F.quartile[t + 1] = x1 == x0 ? x0 : (1 - g) * x0 + g * x1;
      }
      F.mean = (double)(int64_t)U.s1 / (double)B;
      const unsigned __int128 s2 = ((unsigned __int128)U.s2_hi << 64) | U.s2_lo;
      const unsigned __int128 V = (unsigned __int128)(uint64_t)B * s2 - (unsigned __int128)U.s1 * U.s1;
      F.sd = B == 1 ? NAN : std::sqrt((double)V / ((double)B * (double)(B - 1)));
      F.bases = B;
      F.rows = P[w.first + j].n_rows;
    }
  }
  if (stats) *stats = S;
  return 0;
}

// ---- joint single-peak models (psd_joint_models, joint_gpu.cuh) -------------------------------------
namespace {
struct JointScratch {
  unsigned char* d_arena = nullptr;
  int64_t* p_pref = nullptr;   // prefix sums of a wave, pinned
  cudaEvent_t ev[4]; bool ev_ok = false;
  ~JointScratch() {
    if (d_arena) cudaFree(d_arena);
    if (p_pref) cudaFreeHost(p_pref);
    if (ev_ok) for (auto& e : ev) cudaEventDestroy(e);
  }
};

int joint_lanes(int S) { int j = 1; while (32 * j < S) j <<= 1; return j; }   // J: keys per lane

// device bytes of a wave (the arena is carved in this order, see psd_joint_device)
size_t joint_wave_bytes(int64_t n_probs, int64_t elems, int64_t tiles, int64_t chunks, int64_t cands, int64_t items) {
  return cov_align(8 * elems) * 3 + cov_align(sizeof(JointProblem) * n_probs) + cov_align(8 * n_probs) + cov_align(4 * tiles) +
         cov_align(sizeof(JointChunk) * chunks) + cov_align(8 * cands) + cov_align(4 * cands) + cov_align(sizeof(JointItem) * items) +
         cov_align(8 * items) + cov_align(4 * items);
}
}  // namespace

// Waves of consecutive problems that fit the "coverage_gb" budget: H2D of the prefix sums and the tables,
// the flank, flat, pair (one launch per J present) and reduce kernels, D2H of one (loss, t) per (problem, k).
int psd_joint_device(int device, const std::vector<JointDeviceProblem>& P, double* out_loss, int32_t* out_t, psd_joint_stats* S) {
  const int n = (int)P.size();
  if (n == 0) return 0;
  int ndev = 0;
  if (!cuda_ok(cudaGetDeviceCount(&ndev), "cudaGetDeviceCount")) return PSD_ERR_CUDA;
  if (ndev == 0) { g_last_error = "no CUDA device"; return PSD_ERR_CUDA; }
  if (device < 0) CK(cudaGetDevice(&device));
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) { g_last_error = "peaksegdisk_b200 is built for sm_100a only"; return PSD_ERR_CUDA; }
  // one chunk size for the call: about 64 chunks per warp slot of the device, at least 8 pairs
  std::vector<int64_t> pairs(n), chunks(n), tiles(n), elems(n);
  int64_t all_pairs = 0;
  for (int k = 0; k < n; k++) {
    const int64_t N = P[k].N;
    pairs[k] = (N - 1) * (N - 2) / 2;
    all_pairs += pairs[k];
  }
  const int64_t target = (int64_t)prop.multiProcessorCount * 64 * 64;
  const int64_t cp = std::max<int64_t>(8, (all_pairs + target - 1) / target);
  for (int k = 0; k < n; k++) {
    chunks[k] = (pairs[k] + cp - 1) / cp;
    elems[k] = (int64_t)(P[k].N + 1) * P[k].S;
    tiles[k] = (elems[k] + PSD_JOINT_FLANK_TILE - 1) / PSD_JOINT_FLANK_TILE;
  }
  JointScratch X;
  for (auto& e : X.ev) CK(cudaEventCreate(&e));
  X.ev_ok = true;
  size_t free_b = 0, total_b = 0;
  CK(cudaMemGetInfo(&free_b, &total_b));
  const double gb = current_options().coverage_gb;
  const size_t budget = gb > 0 ? (size_t)(gb * (double)(1ull << 30)) : free_b / 2;
  std::vector<std::pair<int, int>> waves;   // [first problem, end problem)
  size_t arena = 0, max_elems = 0;
  for (int k0 = 0; k0 < n;) {
    int k1 = k0;
    int64_t e = 0, t = 0, c = 0, cd = 0, it = 0;
    size_t bytes = 0;
    for (; k1 < n; k1++) {
      const size_t b = joint_wave_bytes(k1 - k0 + 1, e + elems[k1], t + tiles[k1], c + chunks[k1], cd + chunks[k1] * P[k1].S, it + P[k1].S);
      if (k1 > k0 && b > budget) break;
      e += elems[k1]; t += tiles[k1]; c += chunks[k1]; cd += chunks[k1] * P[k1].S; it += P[k1].S; bytes = b;
    }
    waves.push_back({k0, k1});
    arena = std::max(arena, bytes); max_elems = std::max(max_elems, (size_t)e);
    k0 = k1;
  }
  CK(cudaMalloc(&X.d_arena, arena));
  CK(cudaMallocHost(&X.p_pref, 8 * max_elems));
  const cudaStream_t st = 0;
  for (const auto& w : waves) {
    const int np = w.second - w.first;
    std::vector<JointProblem> probs(np);
    std::vector<int> tile_prob;
    std::vector<JointItem> items;
    std::vector<JointChunk> chunk_tab;
    std::vector<std::pair<int, int>> j_range;   // per J present: [first chunk, end chunk)
    int64_t e = 0, cd = 0;
    for (int j = 0; j < np; j++) {
      const JointDeviceProblem& D = P[w.first + j];
      JointProblem& q = probs[j];
      q.grid_off = e; q.cand_off = cd; q.S = D.S; q.N = D.N; q.bin = D.bin; q.len = D.len;
      q.n_chunks = (int)chunks[w.first + j]; q.tile0 = (int)tile_prob.size();
      tile_prob.insert(tile_prob.end(), (size_t)tiles[w.first + j], j);
      for (int k = 1; k <= D.S; k++) items.push_back({j, k});
      memcpy(X.p_pref + e, D.pref, 8 * (size_t)elems[w.first + j]);
      e += elems[w.first + j]; cd += (int64_t)q.n_chunks * D.S;
    }
    for (int J = 1; J <= 8; J <<= 1) {   // the chunks grouped by J, one pair-kernel launch per group
      const int c0 = (int)chunk_tab.size();
      for (int j = 0; j < np; j++) {
        JointProblem& q = probs[j];
        if (joint_lanes(q.S) != J) continue;
        q.chunk0 = (int)chunk_tab.size();
        int a = 1, b = 2;
        for (int64_t t0 = 0; t0 < pairs[w.first + j]; t0 += cp) {
          const int cnt = (int)std::min<int64_t>(cp, pairs[w.first + j] - t0);
          chunk_tab.push_back({j, a, b, (int)t0, cnt});
          for (int r = cnt; r > 0;) {   // advance (a, b) by cnt pairs
            const int left = q.N - b;   // pairs left in row a, b included
            if (r < left) { b += r; r = 0; } else { r -= left; a++; b = a + 1; }
          }
        }
      }
      if ((int)chunk_tab.size() > c0) j_range.push_back({c0, (int)chunk_tab.size()});
      else j_range.push_back({c0, c0});
    }
    const int n_tiles = (int)tile_prob.size(), n_chunks = (int)chunk_tab.size(), n_items = (int)items.size();
    unsigned char* ar = X.d_arena;
    auto carve = [&](size_t b) { unsigned char* r = ar; ar += cov_align(b); return r; };
    JointParams K;
    memset(&K, 0, sizeof K);
    long long* d_pref = (long long*)carve(8 * e);
    K.pref = d_pref;
    K.lleft = (double*)carve(8 * e);
    K.lright = (double*)carve(8 * e);
    JointProblem* d_probs = (JointProblem*)carve(sizeof(JointProblem) * np);
    K.probs = d_probs;
    K.flat = (double*)carve(8 * np);
    int* d_tile = (int*)carve(4 * (size_t)n_tiles);
    K.tile_prob = d_tile; K.n_tiles = n_tiles; K.n_probs = np;
    JointChunk* d_chunks = (JointChunk*)carve(sizeof(JointChunk) * n_chunks);
    K.chunks = d_chunks;
    K.cand_loss = (double*)carve(8 * cd);
    K.cand_t = (int*)carve(4 * cd);
    JointItem* d_items = (JointItem*)carve(sizeof(JointItem) * n_items);
    K.items = d_items; K.n_items = n_items;
    K.out_loss = (double*)carve(8 * (size_t)n_items);
    K.out_t = (int*)carve(4 * (size_t)n_items);
    CK(cudaEventRecord(X.ev[0], st));
    CK(cudaMemcpyAsync(d_pref, X.p_pref, 8 * e, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_probs, probs.data(), sizeof(JointProblem) * np, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_tile, tile_prob.data(), 4 * (size_t)n_tiles, cudaMemcpyHostToDevice, st));
    if (n_chunks) CK(cudaMemcpyAsync(d_chunks, chunk_tab.data(), sizeof(JointChunk) * n_chunks, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_items, items.data(), sizeof(JointItem) * n_items, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(X.ev[1], st));
    joint_flank_kernel<<<n_tiles, 256, 0, st>>>(K);
    CK(cudaGetLastError());
    joint_flat_kernel<<<(np + 127) / 128, 128, 0, st>>>(K);
    CK(cudaGetLastError());
    S->n_launches += 3;
    for (int g = 0; g < 4; g++) {
      K.chunk_begin = j_range[g].first; K.chunk_end = j_range[g].second;
      const int nc = K.chunk_end - K.chunk_begin;
      if (nc == 0) continue;
      const int blocks = (nc + PSD_JOINT_WARPS - 1) / PSD_JOINT_WARPS;
      if (g == 0) joint_pair_kernel<1><<<blocks, PSD_JOINT_WARPS * 32, 0, st>>>(K);
      else if (g == 1) joint_pair_kernel<2><<<blocks, PSD_JOINT_WARPS * 32, 0, st>>>(K);
      else if (g == 2) joint_pair_kernel<4><<<blocks, PSD_JOINT_WARPS * 32, 0, st>>>(K);
      else joint_pair_kernel<8><<<blocks, PSD_JOINT_WARPS * 32, 0, st>>>(K);
      CK(cudaGetLastError());
      S->n_launches++;
    }
    joint_reduce_kernel<<<(n_items + 7) / 8, 256, 0, st>>>(K);
    CK(cudaGetLastError());
    CK(cudaEventRecord(X.ev[2], st));
    std::vector<double> loss(n_items);
    std::vector<int> tt(n_items);
    CK(cudaMemcpyAsync(loss.data(), K.out_loss, 8 * (size_t)n_items, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(tt.data(), K.out_t, 4 * (size_t)n_items, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(X.ev[3], st));
    CK(cudaStreamSynchronize(st));
    float t03 = 0, t12 = 0;
    cudaEventElapsedTime(&t03, X.ev[0], X.ev[3]); cudaEventElapsedTime(&t12, X.ev[1], X.ev[2]);
    S->device_ms += t03; S->kernel_ms += t12;
    S->n_waves++;
    S->h2d_bytes += 8 * e + (int64_t)sizeof(JointProblem) * np + 4 * (int64_t)n_tiles + (int64_t)sizeof(JointChunk) * n_chunks +
                    (int64_t)sizeof(JointItem) * n_items;
    S->d2h_bytes += 12 * (int64_t)n_items;
    int o = 0;
    for (int j = 0; j < np; j++) {
      const JointDeviceProblem& D = P[w.first + j];
      S->pair_sample_evals += pairs[w.first + j] * D.S;
      for (int k = 0; k < D.S; k++, o++) { out_loss[D.out_off + k] = loss[o]; out_t[D.out_off + k] = tt[o]; }
    }
  }
  return 0;
}

int psd_device_count_impl() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

#if defined(PSD_TIMING)
extern "C" int psd_debug_block_ends(unsigned long long* out) {
  return cudaMemcpyFromSymbol(out, psd_blk_end, sizeof(unsigned long long) * 160) == cudaSuccess ? 0 : -1;
}
extern "C" int psd_debug_hist(unsigned long long* out256, int reset) {
  if (cudaMemcpyFromSymbol(out256, psd_hist, sizeof(unsigned long long) * 256) != cudaSuccess) return -1;
  if (reset) { unsigned long long z[256]; memset(z, 0, sizeof z); cudaMemcpyToSymbol(psd_hist, z, sizeof z); }
  return 0;
}
extern "C" int psd_debug_read(unsigned long long* out, int n, int reset) {
  unsigned long long tmp[32];
  if (cudaMemcpyFromSymbol(tmp, psd_dbg, sizeof tmp) != cudaSuccess) return -1;
  for (int i = 0; i < n && i < 32; i++) out[i] = tmp[i];
  if (reset) { memset(tmp, 0, sizeof tmp); cudaMemcpyToSymbol(psd_dbg, tmp, sizeof tmp); }
  return 0;
}
#endif

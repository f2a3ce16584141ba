// plan_internal.h -- host-side types shared by fpop_gpu.cu (device plan) and host_api.cpp (C ABI,
// bedGraph text I/O).  Not installed; the public surface is include/peaksegdisk_b200.h.
#pragma once
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <memory>
#include <thread>
#include <string>
#include <vector>
#include "../../include/peaksegdisk_b200.h"

// The rows of one bedGraph (or one psd_plan_add call) and their pass-1 totals.  Problems that solve
// the same file at different penalties share one RowData: it is parsed, summed, packed and copied to
// the device once.
struct RowData {
  std::vector<int32_t> chrom_start, chrom_end, coverage, weight;
  double bases = 0, sum_wz = 0;   // pass-1 totals (src/PeakSegFPOPLog.cpp:187-189)
  double dmin = 0, dmax = 0;      // log(min coverage), log(max coverage)
};

// Labels of one problem (psd_plan_set_labels), as given and as codes in the units of the problem's
// seg_row (label_errors_gpu.cuh).  Shared by the solves of one problem at different penalties.
struct LabelSet {
  std::vector<int32_t> start, end, kind;
  std::vector<int32_t> code_start, code_end;
};

struct HostProblem {
  int status = 0;                 // reference-style input status (0 ok)
  bool trivial = false;           // one-segment model: penalty Inf or constant coverage
  bool penalty_is_inf = false;
  double penalty = 0;
  int64_t n_rows = 0;
  std::shared_ptr<RowData> rows;  // row problems (null for count-vector problems)
  // count-vector problems (psd_plan_add_counts): no row arrays on the host, the device run-length
  // encodes `counts`; positions are 0..n_pos and seg_row then holds coordinates, not row numbers
  bool from_counts = false;
  int64_t n_pos = 0;
  std::vector<int32_t> counts;
  int64_t raw_off = 0;            // offset into the packed device count buffer
  double bases = 0, sum_wz = 0;   // pass-1 totals (src/PeakSegFPOPLog.cpp:187-189)
  double dmin = 0, dmax = 0;      // log(min coverage), log(max coverage)
  int64_t row_off = 0;            // offset into the packed device row arrays (shared by the problems of one RowData)
  int64_t index_off = 0;          // offset into the device record-index array (one entry per row per PROBLEM)
  // results
  int result_status = -1;         // -1 not solved yet
  int n_segments = 0, n_equality = 0;
  double best_cost = 0, total_intervals = 0, max_intervals = 0;
  std::vector<int> seg_row;       // last row of the previous segment, last segment first (-1 for the first)
  std::vector<double> seg_x;      // log-mean per segment
  // labels and their errors (filled by psd_plan_solve for GPU problems)
  std::shared_ptr<const LabelSet> labels;
  int label_status = -1;          // -1 not scored yet, else the solve's status
  psd_label_errors label_total{};
  std::vector<int32_t> label_fp, label_fn;
};

inline int hp_first_start(const HostProblem& h) { return h.from_counts ? 0 : h.rows->chrom_start[0]; }
inline int hp_last_end(const HostProblem& h) { return h.from_counts ? (int)h.n_pos : h.rows->chrom_end[h.n_rows - 1]; }
// chromStart of segment s (segments are stored last first; s < n_segments - 1)
inline int hp_seg_start(const HostProblem& h, int s) { return h.from_counts ? h.seg_row[s] : h.rows->chrom_end[h.seg_row[s]]; }

// PSD_TRACE=1: wall-clock stage marks on stderr (where does a small solve's latency go?)
struct Trace {
  bool on; std::chrono::steady_clock::time_point t;
  Trace() : on(getenv("PSD_TRACE") != nullptr), t(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    fprintf(stderr, "[psd trace] %-34s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
    t = n;
  }
};

// Runs fn(i) for i in [0,n) on up to hardware_concurrency host threads.
template <class F> void parallel_for(int n, F fn) {
  int nt = (int)std::thread::hardware_concurrency();
  if (nt < 1) nt = 1;
  if (nt > n) nt = n;
  if (nt <= 1) { for (int i = 0; i < n; i++) fn(i); return; }
  std::atomic<int> next(0);
  std::vector<std::thread> pool;
  for (int t = 0; t < nt; t++) pool.emplace_back([&]() { for (;;) { const int i = next.fetch_add(1); if (i >= n) break; fn(i); } });
  for (auto& th : pool) th.join();
}

// Result of psd_coverage_from_reads: the rows of problem i are [row_off[i], row_off[i + 1]).
struct psd_coverage {
  std::vector<int64_t> row_off;
  std::vector<int32_t> chrom_start, chrom_end, count;
  psd_coverage_stats stats;
};
int psd_coverage_from_reads_impl(int device, int n_problems, const psd_reads* problems, psd_coverage** out);
int psd_features_impl(int device, int n_problems, const psd_rows* problems, psd_problem_features* out, psd_features_stats* stats);

struct psd_plan;
psd_plan* psd_plan_create_impl(int device);
void psd_plan_destroy_impl(psd_plan* p);
psd_plan* psd_plan_acquire_parked();          // file entry points: reuse the previous call's buffers
void psd_plan_release_parked(psd_plan* p);
void psd_plan_drop_parked();
std::vector<HostProblem>& psd_plan_problems(psd_plan* p);
const std::vector<HostProblem>& psd_plan_problems_c(const psd_plan* p);
void psd_plan_invalidate(psd_plan* p);
void psd_plan_mark_penalty_changed(psd_plan* p);
const psd_stats& psd_plan_stats_ref(const psd_plan* p);
int psd_plan_upload_impl(psd_plan* p, void* stream);
int psd_plan_solve_impl(psd_plan* p, void* stream);
int psd_plan_download_impl(psd_plan* p, void* stream);
// what the model-path driver reads back from a solve (model_path.cpp)
struct PlanSolveTotals { double dp_ms, backtrack_ms, label_ms; int64_t rows_solved, h2d_bytes, d2h_bytes; };
PlanSolveTotals psd_plan_solve_totals(const psd_plan* p);
// fills the loss fields of the GPU problems' HostProblem (psd_plan_result) from the solve's status
// words, without downloading segments
void psd_plan_collect_results(psd_plan* p);
void psd_plan_mark_labels_changed(psd_plan* p);
int psd_plan_store_function_impl(psd_plan* p, int id, int row, int which, int cap, int* n_out, double* hi, int* back_i, double* back_x);
int psd_device_count_impl();
int psd_set_option_impl(const char* name, double value);
int psd_option_devices();                      // option "devices" / env PSD_DEVICES: GPUs one batched file call may use
void psd_set_last_error(const std::string& s);
// host_api.cpp: the row and label rules shared by psd_plan_add / psd_plan_set_labels and psd_model_path
int check_rows(int64_t n_rows, const int32_t* chromStart, const int32_t* chromEnd, const int32_t* coverage, std::string* why);
HostProblem make_row_problem(int64_t n_rows, const int32_t* chromStart, const int32_t* chromEnd, const int32_t* coverage);
int make_label_set(const HostProblem& h, int64_t n, const int32_t* start, const int32_t* end, const int32_t* kind,
                   std::shared_ptr<const LabelSet>* out, std::string* why);
const std::string& psd_get_last_error();
// the target interval of psd_model_path and psd_joint_models (host_api.cpp): models sorted by peaks ascending
void target_interval(const std::vector<psd_path_model>& m, double* lo, double* hi, int* errors);

// joint.cpp -> fpop_gpu.cu: one problem of psd_joint_models as the device sees it (problems with N >= 3)
struct JointDeviceProblem {
  int S, N, bin, len;      // samples, bins, bin width, region length
  const int64_t* pref;     // C_s(0, i), (N + 1) * S entries, [grid index][sample]
  int64_t out_off;         // its S results (k = 1..S) in out_loss / out_t
};
// For every problem and k = 1..S the minimum of loss_k over all peaks (joint_gpu.cuh): out_loss, and out_t the
// flattened pair index (-1: no pair has k feasible samples).  Adds device time, waves, launches, copies and
// pair x sample evaluations to *stats.
int psd_joint_device(int device, const std::vector<JointDeviceProblem>& probs, double* out_loss, int32_t* out_t, psd_joint_stats* stats);

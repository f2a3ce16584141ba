// host_api.cpp -- the C ABI (include/peaksegdisk_b200.h): penalty / bedGraph text front end with the
// reference's validation order and status codes, the result writers reproducing the reference's
// iostream formatting, and the thin glue onto the device plan (fpop_gpu.cu).
//
// Reference behaviour mirrored here (file:line into tdhock/PeakSegDisk):
//   penalty parsing and its error order      src/PeakSegFPOPLog.cpp:145-159
//   bedGraph pass 1 (validation + totals)    src/PeakSegFPOPLog.cpp:160-209
//   output file creation before any solve    src/PeakSegFPOPLog.cpp:212-223
//   trivial one-segment model                src/PeakSegFPOPLog.cpp:224-243
//   segments / loss lines                    src/PeakSegFPOPLog.cpp:419-454
//   output failure checks                    src/PeakSegFPOPLog.cpp:456-461
//   status -> message                        src/interface.cpp:16-55
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <algorithm>
#include <atomic>
#include <vector>
#include "psd_math.h"
#include "plan_internal.h"

namespace {

inline double hlog(double x) { return psd_log(x, psd_log_tab_host); }
inline double hexp(double x) { return psd_exp(x, psd_exp_tab_host); }

int parse_penalty(const char* s, double* pen, bool* is_inf) {
  *is_inf = strcmp(s, "Inf") == 0;
  try { *pen = std::stod(s); }
  catch (const std::invalid_argument&) { return PSD_ERR_PENALTY_NOT_NUMERIC; }
  catch (const std::out_of_range&) { return PSD_ERR_PENALTY_NOT_FINITE; }  // the reference aborts (uncaught); documented deviation
  if (*is_inf) return 0;
  if (!std::isfinite(*pen)) return PSD_ERR_PENALTY_NOT_FINITE;
  if (*pen < 0) return PSD_ERR_PENALTY_NEGATIVE;
  return 0;
}

inline bool is_ws(unsigned char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

// One integer field with sscanf("%d") semantics: optional whitespace, optional sign, decimal digits,
// value clamped to long then truncated to int.  Returns false on a matching failure.
inline bool scan_int(const char*& p, const char* end, int* out) {
  while (p < end && is_ws((unsigned char)*p)) p++;
  if (p >= end) return false;
  bool neg = false;
  const char* q = p;
  if (*q == '+' || *q == '-') { neg = (*q == '-'); q++; }
  if (q >= end || *q < '0' || *q > '9') return false;
  unsigned long long v = 0;
  bool over = false;
  while (q < end && *q >= '0' && *q <= '9') {
    if (v > (0x7fffffffffffffffULL - 9) / 10) over = true; else v = v * 10 + (unsigned)(*q - '0');
    q++;
  }
  long long sv;
  if (over) sv = neg ? (long long)0x8000000000000000ULL : 0x7fffffffffffffffLL;
  else sv = neg ? -(long long)v : (long long)v;
  *out = (int)sv;
  p = q;
  return true;
}

struct Parsed {
  int status = 0;
  int bad_items = 0, bad_line = 0;
  std::string chrom;
  std::shared_ptr<RowData> rows = std::make_shared<RowData>();   // shared by every penalty solved on this file
};

// Pass 1 of the reference with its first-error semantics; the text is scanned once.
void parse_bedgraph(const char* path, Parsed& P) {
  FILE* f = fopen(path, "rb");
  if (!f) { P.status = PSD_ERR_UNABLE_TO_OPEN_BEDGRAPH; return; }
  std::vector<char> buf;
  {
    // regular files: one read of the whole size; anything else (pipes, /proc): 64 KB at a time
    long size = -1;
    if (fseek(f, 0, SEEK_END) == 0) { size = ftell(f); if (fseek(f, 0, SEEK_SET) != 0) size = -1; }
    if (size > 0) {
      buf.resize((size_t)size);
      const size_t got = fread(buf.data(), 1, (size_t)size, f);
      buf.resize(got);
    }
    char tmp[1 << 16];
    size_t n;
    while ((n = fread(tmp, 1, sizeof tmp, f)) > 0) buf.insert(buf.end(), tmp, tmp + n);
  }
  const bool rd_err = ferror(f) != 0;
  fclose(f);
  if (rd_err && buf.empty()) { P.status = PSD_ERR_UNABLE_TO_OPEN_BEDGRAPH; return; }
  const char* p = buf.data();
  const char* const fend = p + buf.size();
  int line_i = 0, prev_end = -1;
  const char* chrom_b = nullptr; const char* chrom_e = nullptr;
  {   // typical rows are 20-30 bytes: one allocation instead of a dozen doublings
    const size_t guess = buf.size() / 16 + 16;
    P.rows->chrom_start.reserve(guess); P.rows->chrom_end.reserve(guess); P.rows->coverage.reserve(guess);
  }
  while (p < fend) {
    const char* nl = (const char*)memchr(p, '\n', (size_t)(fend - p));
    const char* const e = nl ? nl : fend;        // sscanf works on a C string: a NUL inside the line ends it (checked below)
    line_i++;
    const char* q = p;
    int items = 0;
    int cs = 0, ce = 0, cv = 0;
    while (q < e && is_ws((unsigned char)*q)) q++;
    if (q >= e || *q == '\0') items = -1;   // sscanf returns EOF on an empty line
    else {
      chrom_b = q;
      while (q < e && *q != '\0' && !is_ws((unsigned char)*q)) q++;
      chrom_e = q;
      items = 1;
      if (scan_int(q, e, &cs)) { items = 2; if (scan_int(q, e, &ce)) { items = 3; if (scan_int(q, e, &cv)) items = 4; } }
    }
    if (items < 4) { P.status = PSD_ERR_NOT_ENOUGH_COLUMNS; P.bad_items = items; P.bad_line = line_i; return; }
    while (q < e && is_ws((unsigned char)*q)) q++;
    if (q < e && *q != '\0') { P.status = PSD_ERR_NON_INTEGER_DATA; return; }   // "%d%s": trailing text after the 4th column
    if (line_i > 1 && cs != prev_end) { P.status = PSD_ERR_INCONSISTENT_CHROMSTART_CHROMEND; return; }
    prev_end = ce;
    P.rows->chrom_start.push_back(cs); P.rows->chrom_end.push_back(ce); P.rows->coverage.push_back(cv);
    p = nl ? nl + 1 : fend;
  }
  if (line_i == 0) { P.status = PSD_ERR_NO_DATA; return; }
  size_t len = (size_t)(chrom_e - chrom_b);
  P.chrom.assign(chrom_b, len);
}

// Pass-1 totals of a row set: weights, sum of weights, sum of weight x coverage, log range.
// The reference takes log(coverage) of every row and keeps the smallest and the largest
// (src/PeakSegFPOPLog.cpp:190-197); log is monotone on the integers, so these are the logs of the
// smallest and the largest coverage: two log calls instead of one per row.
void finish_rows(RowData& r) {
  const int64_t n = (int64_t)r.coverage.size();
  r.weight.resize(n);
  double W = 0, SWZ = 0;
  int32_t zmin = n ? r.coverage[0] : 0, zmax = zmin;
  for (int64_t t = 0; t < n; t++) {
    const int32_t wi = r.chrom_end[t] - r.chrom_start[t];
    r.weight[t] = wi;
    const double w = (double)wi;
    const int32_t z = r.coverage[t];
    W += w;
    SWZ += w * z;
    zmin = z < zmin ? z : zmin; zmax = z > zmax ? z : zmax;
  }
  r.bases = W; r.sum_wz = SWZ;
  if (zmin < 0) {
    // negative coverage (the reference accepts it): log gives NaN, and NaN never replaces the running
    // min / max in the reference's comparisons -- keep its exact row-by-row semantics for this corner
    double xmin = INFINITY, xmax = -INFINITY;
    for (int64_t t = 0; t < n; t++) {
      const double lx = hlog((double)r.coverage[t]);
      if (lx < xmin) xmin = lx;
      if (xmax < lx) xmax = lx;
    }
    r.dmin = xmin; r.dmax = xmax;
  } else {
    r.dmin = n ? hlog((double)zmin) : INFINITY; r.dmax = n ? hlog((double)zmax) : -INFINITY;
  }
}

// Fills the derived fields of a problem from its (finished) rows.
void finish_problem(HostProblem& h) {
  const RowData& r = *h.rows;
  h.bases = r.bases; h.sum_wz = r.sum_wz; h.dmin = r.dmin; h.dmax = r.dmax;
  h.trivial = h.penalty_is_inf || r.dmin == r.dmax;
}

void format_g(std::string& out, const char* fmt, double v) {
  char b[64];
  snprintf(b, sizeof b, fmt, v);
  out += b;
}

// text of <prefix>_segments.bed and <prefix>_loss.tsv for a solved problem
void render(const HostProblem& h, const std::string& chrom, const char* penalty_str,
            std::string& seg_txt, std::string& loss_txt) {
  char ib[64];
  const int64_t n = h.n_rows;
  if (h.trivial) {
    const double SWZ = h.sum_wz, W = h.bases;
    const double bc = (SWZ != 0) ? SWZ * (1 - hlog(SWZ) + hlog(W)) : 0;
    seg_txt = chrom; seg_txt += "\t";
    snprintf(ib, sizeof ib, "%d\t%d\tbackground\t", hp_first_start(h), hp_last_end(h)); seg_txt += ib;
    format_g(seg_txt, "%g", SWZ / W); seg_txt += "\n";
    loss_txt = penalty_str;
    snprintf(ib, sizeof ib, "\t1\t0\t%d\t%d\t", (int)W, (int)n); loss_txt += ib;
    format_g(loss_txt, "%.20g", bc / W); loss_txt += "\t";
    format_g(loss_txt, "%.20g", bc); loss_txt += "\t0\t0\t0\n";
    return;
  }
  const int ns = h.n_segments;
  int prev_end = hp_last_end(h);
  seg_txt.clear();
  for (int s = 0; s < ns; s++) {
    const int st = (s < ns - 1) ? hp_seg_start(h, s) : hp_first_start(h);
    seg_txt += chrom;
    snprintf(ib, sizeof ib, "\t%d\t%d\t%s\t", st, prev_end, (s & 1) ? "peak" : "background"); seg_txt += ib;
    format_g(seg_txt, "%g", hexp(h.seg_x[s])); seg_txt += "\n";
    prev_end = st;
  }
  const int n_peaks = (ns - 1) / 2;
  loss_txt.clear();
  format_g(loss_txt, "%.20g", h.penalty);
  snprintf(ib, sizeof ib, "\t%d\t%d\t%d\t%d\t", ns, n_peaks, (int)h.bases, (int)n); loss_txt += ib;
  format_g(loss_txt, "%.20g", h.best_cost); loss_txt += "\t";
  format_g(loss_txt, "%.20g", h.best_cost * h.bases - h.penalty * n_peaks);
  snprintf(ib, sizeof ib, "\t%d\t", h.n_equality); loss_txt += ib;
  format_g(loss_txt, "%.20g", h.total_intervals / (double)((int)n * 2)); loss_txt += "\t";
  format_g(loss_txt, "%.20g", h.max_intervals); loss_txt += "\n";
}

bool write_all(FILE* f, const std::string& s) {
  if (!f) return false;
  bool ok = s.empty() || fwrite(s.data(), 1, s.size(), f) == s.size();
  if (fflush(f) != 0) ok = false;
  return ok;
}

// wall-clock stages of the last file batch of this process (psd_last_batch_stats)
std::mutex g_batch_stats_mutex;
psd_batch_stats g_batch_stats;
struct StageClock {
  std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
  double lap() {
    const auto n = std::chrono::steady_clock::now();
    const double ms = std::chrono::duration<double, std::milli>(n - t).count();
    t = n;
    return ms;
  }
};

struct FileJob {
  std::string bedgraph, penalty_str, db;
  int status = 0;
  double penalty = 0; bool is_inf = false;
  std::shared_ptr<Parsed> parsed;
  bool loss_created = false, seg_created = false;
  int plan_id = -1;
  int dev_slot = 0;          // which of the batch's plans (one per GPU in use) owns this problem
};

// creates / truncates a file and closes it again (outputs exist, empty, before the solve)
bool touch(const std::string& path) {
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) return false;
  return fclose(f) == 0;
}

bool write_file(const std::string& path, const std::string& text) {
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) return false;
  const bool ok = write_all(f, text);
  return (fclose(f) == 0) && ok;
}

int run_file_batch(int n, const char* const* bedgraphs, const char* const* penalties, const char* const* dbs, int* status_out) {
  std::vector<FileJob> jobs(n);
  Trace tr;
  StageClock clk;
  psd_batch_stats BS;
  memset(&BS, 0, sizeof BS);
  BS.n_problems = n;
  // several penalties on one bedGraph parse it once; distinct files are parsed on all host cores
  std::map<std::string, std::shared_ptr<Parsed>> cache;
  std::vector<std::shared_ptr<Parsed>> to_parse;
  std::vector<std::string> to_parse_name;
  for (int i = 0; i < n; i++) {
    FileJob& j = jobs[i];
    j.bedgraph = bedgraphs[i]; j.penalty_str = penalties[i]; j.db = dbs[i];
    j.status = parse_penalty(penalties[i], &j.penalty, &j.is_inf);
    if (j.status) continue;   // penalty errors come before any file access (:152-159)
    auto it = cache.find(j.bedgraph);
    if (it == cache.end()) {
      it = cache.emplace(j.bedgraph, std::make_shared<Parsed>()).first;
      to_parse.push_back(it->second); to_parse_name.push_back(j.bedgraph);
    }
    j.parsed = it->second;
  }
  parallel_for((int)to_parse.size(), [&](int k) {
    parse_bedgraph(to_parse_name[k].c_str(), *to_parse[k]);
    if (to_parse[k]->status == 0) finish_rows(*to_parse[k]->rows);
  });
  tr.mark("files: parse");
  BS.parse_ms = clk.lap();
  BS.n_files_parsed = (int)to_parse.size();
  for (const auto& P : to_parse) BS.rows_parsed += (int64_t)P->rows->coverage.size();
  int fatal = 0;
  for (int i = 0; i < n; i++) {
    FileJob& j = jobs[i];
    if (j.status) continue;
    j.status = j.parsed->status;
    if (j.status == PSD_ERR_NOT_ENOUGH_COLUMNS)
      printf("problem: %d items on line %d\n", j.parsed->bad_items, j.parsed->bad_line);
    if (j.status) continue;
    // outputs are created (empty) before anything else can fail, as the reference does (:222-223)
    const std::string prefix = j.bedgraph + "_penalty=" + j.penalty_str;
    j.loss_created = touch(prefix + "_loss.tsv");
    j.seg_created = touch(prefix + "_segments.bed");
  }
  // Multi-GPU inside one call (option "devices" > 1; SURVEY 8e): the problems are independent, so
  // they are dealt to the GPUs longest-first onto the least loaded one, each GPU gets its own plan
  // and host thread, and there is no exchange between them.
  int n_dev = psd_option_devices();
  if (n_dev != 1) {
    const int have = psd_device_count_impl();
    n_dev = (n_dev <= 0 || n_dev > have) ? have : n_dev;
    if (n_dev < 1) n_dev = 1;
  }
  if (n_dev > 1) {
    std::vector<int> order;
    for (int i = 0; i < n; i++) if (!jobs[i].status) order.push_back(i);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return jobs[a].parsed->rows->coverage.size() > jobs[b].parsed->rows->coverage.size(); });
    std::vector<double> load(n_dev, 0.0);
    for (int i : order) {
      int best = 0;
      for (int d = 1; d < n_dev; d++) if (load[d] < load[best]) best = d;
      jobs[i].dev_slot = best; load[best] += (double)jobs[i].parsed->rows->coverage.size();
    }
  }
  tr.mark("files: create outputs");
  std::vector<psd_plan*> plans(n_dev, nullptr);
  // build the plans: slots first (serial, cheap), then rows / pass-1 totals / scratch db on all host cores
  for (int i = 0; i < n; i++) {
    FileJob& j = jobs[i];
    if (j.status) continue;
    psd_plan*& plan = plans[j.dev_slot];
    if (!plan) {
      plan = (n_dev == 1) ? psd_plan_acquire_parked() : psd_plan_create_impl(j.dev_slot);
      if (!plan) { fatal = PSD_ERR_CUDA; break; }
    }
    const Parsed& P = *j.parsed;
    if (P.rows->coverage.empty() || P.rows->coverage.size() > 0x3fffffff) { j.status = PSD_ERR_ARG; continue; }
    std::vector<HostProblem>& v = psd_plan_problems(plan);
    j.plan_id = (int)v.size();
    v.emplace_back();
  }
  if (!fatal) {
    parallel_for(n, [&](int i) {
      FileJob& j = jobs[i];
      if (j.status || j.plan_id < 0) return;
      const Parsed& P = *j.parsed;
      HostProblem& h = psd_plan_problems(plans[j.dev_slot])[j.plan_id];
      h.n_rows = (int64_t)P.rows->coverage.size(); h.penalty = j.penalty; h.penalty_is_inf = j.is_inf;
      h.rows = P.rows;          // shared, not copied: parsed, summed and uploaded once per file
      finish_problem(h);
      if (!h.trivial) {
        // the reference creates its scratch db here; keep that contract (error 7 when unwritable)
        FILE* d = fopen(j.db.c_str(), "wb");
        bool ok = d != nullptr;
        if (ok) {
          char hdr[64];
          memset(hdr, 0, sizeof hdr);
          snprintf(hdr, sizeof hdr, "PSD-B200 cost functions live in HBM; rows=%lld", (long long)h.n_rows);
          ok = fwrite(hdr, 1, sizeof hdr, d) == sizeof hdr;
          if (fclose(d) != 0) ok = false;
        }
        if (!ok) { j.status = PSD_ERR_WRITING_COST_FUNCTIONS; h.status = j.status; }
      }
    });
    for (psd_plan* plan : plans) if (plan) psd_plan_invalidate(plan);
  }
  tr.mark("files: build plan");
  BS.build_ms = clk.lap();
  if (!fatal) {
    if (n_dev == 1) {
      if (plans[0]) fatal = psd_plan_run(plans[0], nullptr);
    } else {
      std::vector<int> rcs(n_dev, 0);
      std::vector<std::string> errs(n_dev);
      std::vector<std::thread> pool;
      for (int d = 0; d < n_dev; d++)
        if (plans[d]) pool.emplace_back([&, d]() { rcs[d] = psd_plan_run(plans[d], nullptr); if (rcs[d]) errs[d] = psd_get_last_error(); });
      for (auto& th : pool) th.join();
      for (int d = 0; d < n_dev; d++) if (rcs[d] && !fatal) { fatal = rcs[d]; psd_set_last_error(errs[d]); }
    }
  }
  tr.mark("files: upload + solve + download");
  BS.run_ms = clk.lap();
  BS.n_devices = 0;
  for (psd_plan* plan : plans) {
    if (!plan) continue;
    const psd_stats& d = psd_plan_stats_ref(plan);
    BS.n_devices++;
    BS.dp_ms = std::max(BS.dp_ms, d.dp_ms); BS.backtrack_ms = std::max(BS.backtrack_ms, d.backtrack_ms);
    BS.h2d_bytes += d.h2d_bytes; BS.d2h_bytes += d.d2h_bytes; BS.rows_solved += d.rows_solved;
    BS.n_launches += d.n_launches; BS.n_waves += d.n_waves; BS.n_latency_waves += d.n_latency_waves;
    BS.store_bytes_algorithmic += d.store_bytes_algorithmic;
  }
  // render and write the result files on all host cores
  parallel_for(n, [&](int i) {
    FileJob& j = jobs[i];
    if (!j.status && fatal) j.status = fatal;
    if (!j.status) {
      const HostProblem& h = psd_plan_problems(plans[j.dev_slot])[j.plan_id];
      if (!h.trivial && h.result_status != 0) j.status = (h.result_status < 0) ? PSD_ERR_INTERNAL : h.result_status;
      else {
        std::string seg_txt, loss_txt;
        render(h, j.parsed->chrom, j.penalty_str.c_str(), seg_txt, loss_txt);
        const std::string prefix = j.bedgraph + "_penalty=" + j.penalty_str;
        const bool seg_ok = j.seg_created && write_file(prefix + "_segments.bed", seg_txt);
        const bool loss_ok = j.loss_created && write_file(prefix + "_loss.tsv", loss_txt);
        if (!loss_ok) j.status = PSD_ERR_WRITING_LOSS_OUTPUT;
        else if (!seg_ok) j.status = PSD_ERR_WRITING_SEGMENTS_OUTPUT;
      }
    }
    status_out[i] = j.status;
  });
  tr.mark("files: render + write");
  BS.write_ms = clk.lap();
  for (psd_plan* plan : plans)
    if (plan) { if (fatal || n_dev > 1) psd_plan_destroy_impl(plan); else psd_plan_release_parked(plan); }
  tr.mark("files: park / release the plan");
  BS.release_ms = clk.lap();
  { std::lock_guard<std::mutex> lk(g_batch_stats_mutex); g_batch_stats = BS; }
  return fatal;
}

}  // namespace

// The rows rule of psd_plan_add and psd_model_path.  Returns 0 or the status, *why says which row.
int check_rows(int64_t n_rows, const int32_t* chromStart, const int32_t* chromEnd, const int32_t* coverage, std::string* why) {
  char msg[160];
  if (n_rows <= 0 || n_rows > 0x3fffffff) { snprintf(msg, sizeof msg, "n_rows %lld is outside [1, 0x3fffffff]", (long long)n_rows); *why = msg; return PSD_ERR_ARG; }
  if (!chromStart || !chromEnd || !coverage) { *why = "a row array is null"; return PSD_ERR_ARG; }
  // the file path's contract (src/PeakSegFPOPLog.cpp:180-186): rows are contiguous; in addition the
  // in-memory entry insists on positive widths and non-negative coverage (a zero first width makes
  // penalty / cumulative weight infinite in the kernel; psd_plan_add_counts rejects negatives too)
  for (int64_t i = 0; i < n_rows; i++) {
    if (i > 0 && chromStart[i] != chromEnd[i - 1]) {
      snprintf(msg, sizeof msg, "row %lld: chromStart %d != chromEnd %d of the row before", (long long)i, chromStart[i], chromEnd[i - 1]);
      *why = msg; return PSD_ERR_INCONSISTENT_CHROMSTART_CHROMEND;
    }
    if (chromEnd[i] <= chromStart[i] || coverage[i] < 0) {
      snprintf(msg, sizeof msg, "row %lld: empty or negative width, or negative coverage", (long long)i);
      *why = msg; return PSD_ERR_ARG;
    }
  }
  return 0;
}

// A row problem (penalty 0) on its own copy of the rows; the rows must have passed check_rows.
HostProblem make_row_problem(int64_t n_rows, const int32_t* chromStart, const int32_t* chromEnd, const int32_t* coverage) {
  HostProblem h;
  h.n_rows = n_rows;
  h.rows = std::make_shared<RowData>();
  h.rows->chrom_start.assign(chromStart, chromStart + n_rows);
  h.rows->chrom_end.assign(chromEnd, chromEnd + n_rows);
  h.rows->coverage.assign(coverage, coverage + n_rows);
  finish_rows(*h.rows);
  finish_problem(h);
  return h;
}

// Checks n labels of problem h and converts their ends into codes of h's seg_row units
// (label_errors_gpu.cuh): 2r for chromEnd[r], 2r - 1 between chromEnd[r - 1] and chromEnd[r]; 2x for
// count-vector problems.  n == 0 gives no label set.  Returns 0 or PSD_ERR_ARG, *why names the label.
int make_label_set(const HostProblem& h, int64_t n, const int32_t* start, const int32_t* end, const int32_t* kind,
                   std::shared_ptr<const LabelSet>* out, std::string* why) {
  out->reset();
  char msg[160];
  if (n < 0 || n > 0x3fffffff) { snprintf(msg, sizeof msg, "n_labels %lld is outside [0, 0x3fffffff]", (long long)n); *why = msg; return PSD_ERR_ARG; }
  if (n == 0) return 0;
  if (!start || !end || !kind) { *why = "a label array is null"; return PSD_ERR_ARG; }
  const int lo = hp_first_start(h), hi = hp_last_end(h);
  auto L = std::make_shared<LabelSet>();
  L->start.assign(start, start + n); L->end.assign(end, end + n); L->kind.assign(kind, kind + n);
  L->code_start.resize(n); L->code_end.resize(n);
  auto code = [&](int32_t x) -> int32_t {
    if (h.from_counts) return 2 * x;
    const std::vector<int32_t>& ce = h.rows->chrom_end;
    const int32_t r = (int32_t)(std::lower_bound(ce.begin(), ce.end(), x) - ce.begin());
    return ce[r] == x ? 2 * r : 2 * r - 1;
  };
  for (int64_t k = 0; k < n; k++) {
    if (kind[k] < 0 || kind[k] > 3) { snprintf(msg, sizeof msg, "label %lld: kind %d is not 0..3", (long long)k, kind[k]); *why = msg; return PSD_ERR_ARG; }
    if (start[k] >= end[k]) { snprintf(msg, sizeof msg, "label %lld: chromStart %d >= chromEnd %d", (long long)k, start[k], end[k]); *why = msg; return PSD_ERR_ARG; }
    if (start[k] < lo || end[k] > hi) {
      snprintf(msg, sizeof msg, "label %lld: [%d, %d) is not inside the problem's [%d, %d)", (long long)k, start[k], end[k], lo, hi);
      *why = msg; return PSD_ERR_ARG;
    }
    L->code_start[k] = code(start[k]); L->code_end[k] = code(end[k]);
  }
  *out = L;
  return 0;
}

// Target interval: the widest run (in log penalty) of consecutive models with the fewest errors; a run
// that reaches 0 or infinity is infinitely wide; ties go to the smaller min_lambda.
void target_interval(const std::vector<psd_path_model>& m, double* lo, double* hi, int* errors) {
  int best = m[0].errors;
  for (const auto& x : m) best = std::min(best, x.errors);
  double best_w = -1, best_lo = NAN, best_hi = NAN;
  for (size_t a = 0; a < m.size();) {
    if (m[a].errors != best) { a++; continue; }
    size_t b = a;
    while (b + 1 < m.size() && m[b + 1].errors == best) b++;
    // models are sorted by peaks ascending, so lambda decreases from a to b
    const double r_hi = m[a].max_lambda, r_lo = m[b].min_lambda;
    const double w = (r_lo == 0 || std::isinf(r_hi)) ? INFINITY : std::log(r_hi) - std::log(r_lo);
    if (best_w < 0 || w > best_w || (w == best_w && r_lo < best_lo)) { best_w = w; best_lo = r_lo; best_hi = r_hi; }
    a = b + 1;
  }
  *lo = best_lo; *hi = best_hi; *errors = best;
}

extern "C" {

int psd_fpop_disk_batch(int n, const char* const* bedGraph_file_names, const char* const* penalty_strs,
                        const char* const* db_file_names, int* status_out) {
  if (n < 0 || (n > 0 && (!bedGraph_file_names || !penalty_strs || !db_file_names || !status_out))) return PSD_ERR_ARG;
  if (n == 0) return 0;
  return run_file_batch(n, bedGraph_file_names, penalty_strs, db_file_names, status_out);
}

int psd_fpop_disk(const char* bedGraph_file_name, const char* penalty_str, const char* db_file_name) {
  if (!bedGraph_file_name || !penalty_str || !db_file_name) return PSD_ERR_ARG;
  int st = -1;
  const int rc = run_file_batch(1, &bedGraph_file_name, &penalty_str, &db_file_name, &st);
  return st >= 0 ? st : rc;
}

const char* psd_status_message(int status) {
  switch (status) {
    case 0: return "ok";
    case 1: return "penalty=%s but must be finite";
    case 2: return "penalty=%s must be non-negative";
    case 3: return "unable to open input file for reading %s";
    case 4: return "each line of input data file %s should have exactly four columns";
    case 5: return "fourth column of input data file %s should be integer";
    case 6: return "there should be no gaps (columns 2-3) in input data file %s";
    case 7: return "unable to write to cost function database file %s";
    case 8: return "unable to write to loss output file %s_penalty=%s_loss.tsv";
    case 9: return "input file %s contains no data";
    case 10: return "penalty string '%s' is not numeric; it should be convertible to double";
    case 11: return "unable to write to segments output file %s_penalty=%s_segments.bed";
    case PSD_ERR_PIECE_OVERFLOW: return "a cost function outgrew the largest piece-list tier";
    case PSD_ERR_STORE_EXHAUSTED: return "the HBM cost-function store cannot hold this problem";
    case PSD_ERR_BACKTRACK: return "backtrack lost the optimal mean";
    case PSD_ERR_INTERNAL: return "internal solver error";
    case PSD_ERR_CUDA: return "CUDA error (no device, driver failure or kernel fault)";
    case PSD_ERR_ARG: return "invalid argument";
    default: return "error code %d";
  }
}

const char* psd_last_error(void) { return psd_get_last_error().c_str(); }

psd_plan* psd_plan_create(int device) { return psd_plan_create_impl(device); }
void psd_plan_destroy(psd_plan* plan) { psd_plan_destroy_impl(plan); }

int psd_plan_add(psd_plan* plan, int64_t n_rows, const int32_t* chromStart, const int32_t* chromEnd,
                 const int32_t* coverage, double penalty, int penalty_is_inf) {
  if (!plan || n_rows <= 0 || n_rows > 0x3fffffff || !chromStart || !chromEnd || !coverage) return -PSD_ERR_ARG;
  if (!penalty_is_inf) {
    if (!std::isfinite(penalty)) return -PSD_ERR_PENALTY_NOT_FINITE;
    if (penalty < 0) return -PSD_ERR_PENALTY_NEGATIVE;
  }
  std::string why;
  const int rc = check_rows(n_rows, chromStart, chromEnd, coverage, &why);
  if (rc) return -rc;
  std::vector<HostProblem>& v = psd_plan_problems(plan);
  v.push_back(make_row_problem(n_rows, chromStart, chromEnd, coverage));
  HostProblem& h = v.back();
  h.penalty = penalty; h.penalty_is_inf = penalty_is_inf != 0;
  finish_problem(h);
  psd_plan_invalidate(plan);
  return (int)v.size() - 1;
}

// In-memory front end for a count vector (R/PeakSegFPOP_vec.R:18-25 does rle() + cumsum on the host
// and goes through a bedGraph file): position i of `counts` is the base [i, i+1).  One host pass
// for the totals the loss line needs (bases, sum of counts, runs = bedGraph.lines, log range); the
// run-length encoding itself happens on the device at upload (rle_gpu.cuh).
int psd_plan_add_counts(psd_plan* plan, int64_t n, const int32_t* counts, double penalty, int penalty_is_inf) {
  if (!plan || n <= 0 || n > 0x3fffffff || !counts) return -PSD_ERR_ARG;
  if (!penalty_is_inf) {
    if (!std::isfinite(penalty)) return -PSD_ERR_PENALTY_NOT_FINITE;
    if (penalty < 0) return -PSD_ERR_PENALTY_NEGATIVE;
  }
  int32_t lo = counts[0], hi = counts[0];
  int64_t runs = 1; double sum = (double)counts[0];
  for (int64_t i = 1; i < n; i++) {
    const int32_t z = counts[i];
    runs += (z != counts[i - 1]);
    sum += (double)z;            // exact: integers below 2^53, like the reference's running double total
    lo = z < lo ? z : lo; hi = z > hi ? z : hi;
  }
  if (lo < 0) return -PSD_ERR_ARG;
  std::vector<HostProblem>& v = psd_plan_problems(plan);
  v.emplace_back();
  HostProblem& h = v.back();
  h.from_counts = true; h.n_pos = n; h.n_rows = runs;
  h.penalty = penalty; h.penalty_is_inf = penalty_is_inf != 0;
  h.counts.assign(counts, counts + n);
  h.bases = (double)n; h.sum_wz = sum; h.dmin = hlog((double)lo); h.dmax = hlog((double)hi);
  h.trivial = h.penalty_is_inf || lo == hi;
  psd_plan_invalidate(plan);
  return (int)v.size() - 1;
}

int psd_plan_set_labels(psd_plan* plan, int id, int64_t n, const int32_t* chromStart, const int32_t* chromEnd, const int32_t* kind) {
  if (!plan) { psd_set_last_error("psd_plan_set_labels: plan is null"); return PSD_ERR_ARG; }
  std::vector<HostProblem>& v = psd_plan_problems(plan);
  if (id < 0 || id >= (int)v.size()) { psd_set_last_error("psd_plan_set_labels: no problem " + std::to_string(id)); return PSD_ERR_ARG; }
  std::string why;
  std::shared_ptr<const LabelSet> L;
  if (make_label_set(v[id], n, chromStart, chromEnd, kind, &L, &why)) {
    psd_set_last_error("psd_plan_set_labels: problem " + std::to_string(id) + ": " + why);
    return PSD_ERR_ARG;
  }
  v[id].labels = L;
  v[id].label_status = -1;
  psd_plan_mark_labels_changed(plan);
  return 0;
}

int psd_plan_label_errors(const psd_plan* plan, int id, psd_label_errors* total, int32_t* fp, int32_t* fn) {
  if (!plan) return PSD_ERR_ARG;
  const std::vector<HostProblem>& v = psd_plan_problems_c(plan);
  if (id < 0 || id >= (int)v.size()) return PSD_ERR_ARG;
  const HostProblem& h = v[id];
  if (!h.labels) { psd_set_last_error("psd_plan_label_errors: problem " + std::to_string(id) + " has no labels"); return PSD_ERR_ARG; }
  if (h.status) return h.status;
  const LabelSet& L = *h.labels;
  const size_t n = L.kind.size();
  if (h.trivial) {   // one segment, no peak: every label that needs a peak misses it
    psd_label_errors t{};
    for (size_t k = 0; k < n; k++) {
      const int miss = L.kind[k] != 0;
      if (fp) fp[k] = 0;
      if (fn) fn[k] = miss;
      t.fn += miss; t.possible_fp += L.kind[k] != 1; t.possible_fn += L.kind[k] != 0;
    }
    t.errors = t.fn;
    if (total) *total = t;
    return 0;
  }
  if (h.label_status != 0) {
    if (h.label_status < 0) psd_set_last_error("psd_plan_label_errors: problem " + std::to_string(id) + " is not solved");
    return h.label_status < 0 ? PSD_ERR_ARG : h.label_status;
  }
  if (total) *total = h.label_total;
  if (fp) memcpy(fp, h.label_fp.data(), sizeof(int32_t) * n);
  if (fn) memcpy(fn, h.label_fn.data(), sizeof(int32_t) * n);
  return 0;
}

int psd_plan_size(const psd_plan* plan) { return plan ? (int)psd_plan_problems_c(plan).size() : 0; }

int psd_plan_set_penalty(psd_plan* plan, int id, double penalty, int penalty_is_inf) {
  if (!plan) return PSD_ERR_ARG;
  std::vector<HostProblem>& v = psd_plan_problems(plan);
  if (id < 0 || id >= (int)v.size()) return PSD_ERR_ARG;
  if (!penalty_is_inf) {
    if (!std::isfinite(penalty)) return PSD_ERR_PENALTY_NOT_FINITE;
    if (penalty < 0) return PSD_ERR_PENALTY_NEGATIVE;
  }
  HostProblem& h = v[id];
  const bool was_trivial = h.trivial;
  h.penalty = penalty; h.penalty_is_inf = penalty_is_inf != 0;
  h.trivial = h.penalty_is_inf || h.dmin == h.dmax;
  h.result_status = -1;
  if (was_trivial != h.trivial) psd_plan_invalidate(plan);   // the set of GPU problems changed
  else psd_plan_mark_penalty_changed(plan);
  return 0;
}

int psd_plan_upload(psd_plan* plan, void* stream) { return plan ? psd_plan_upload_impl(plan, stream) : PSD_ERR_ARG; }
int psd_plan_solve(psd_plan* plan, void* stream) { return plan ? psd_plan_solve_impl(plan, stream) : PSD_ERR_ARG; }
int psd_plan_download(psd_plan* plan, void* stream) { return plan ? psd_plan_download_impl(plan, stream) : PSD_ERR_ARG; }

int psd_plan_run(psd_plan* plan, void* stream) {
  if (!plan) return PSD_ERR_ARG;
  int rc = psd_plan_upload_impl(plan, stream);
  if (!rc) rc = psd_plan_solve_impl(plan, stream);
  if (!rc) rc = psd_plan_download_impl(plan, stream);
  return rc;
}

int psd_plan_result(const psd_plan* plan, int id, psd_result* out) {
  if (!plan || !out) return PSD_ERR_ARG;
  const std::vector<HostProblem>& v = psd_plan_problems_c(plan);
  if (id < 0 || id >= (int)v.size()) return PSD_ERR_ARG;
  const HostProblem& h = v[id];
  memset(out, 0, sizeof *out);
  out->n_rows = (int32_t)h.n_rows; out->penalty = h.penalty; out->bases = h.bases; out->trivial = h.trivial ? 1 : 0;
  if (h.status) { out->status = h.status; return 0; }
  if (h.trivial) {
    const double SWZ = h.sum_wz, W = h.bases;
    const double bc = (SWZ != 0) ? SWZ * (1 - hlog(SWZ) + hlog(W)) : 0;
    out->status = 0; out->n_segments = 1; out->n_peaks = 0; out->mean_pen_cost = bc / W; out->total_loss = bc;
    if (h.penalty_is_inf) out->penalty = INFINITY;
    return 0;
  }
  if (h.result_status != 0) { out->status = h.result_status < 0 ? PSD_ERR_ARG : h.result_status; return 0; }
  const int np = (h.n_segments - 1) / 2;
  out->n_segments = h.n_segments; out->n_peaks = np; out->n_equality = h.n_equality;
  out->mean_pen_cost = h.best_cost; out->total_loss = h.best_cost * h.bases - h.penalty * np;
  out->mean_intervals = h.total_intervals / (double)((int)h.n_rows * 2); out->max_intervals = h.max_intervals;
  return 0;
}

int psd_plan_segments(const psd_plan* plan, int id, int32_t* chromStart, int32_t* chromEnd, int32_t* is_peak, double* mean) {
  if (!plan) return PSD_ERR_ARG;
  const std::vector<HostProblem>& v = psd_plan_problems_c(plan);
  if (id < 0 || id >= (int)v.size()) return PSD_ERR_ARG;
  const HostProblem& h = v[id];
  if (h.status) return h.status;
  if (h.trivial) {
    chromStart[0] = hp_first_start(h); chromEnd[0] = hp_last_end(h); is_peak[0] = 0; mean[0] = h.sum_wz / h.bases;
    return 0;
  }
  if (h.result_status != 0) return h.result_status < 0 ? PSD_ERR_ARG : h.result_status;
  int prev_end = hp_last_end(h);
  for (int s = 0; s < h.n_segments; s++) {
    const int st = (s < h.n_segments - 1) ? hp_seg_start(h, s) : hp_first_start(h);
    chromStart[s] = st; chromEnd[s] = prev_end; is_peak[s] = s & 1; mean[s] = hexp(h.seg_x[s]);
    prev_end = st;
  }
  return 0;
}

int psd_plan_get_stats(const psd_plan* plan, psd_stats* out) {
  if (!plan || !out) return PSD_ERR_ARG;
  *out = psd_plan_stats_ref(plan);
  return 0;
}

int psd_plan_store_function(psd_plan* plan, int id, int row, int which, int cap, int* n_pieces, double* max_log_mean,
                            int* data_i, double* prev_log_mean) {
  if (!plan) return PSD_ERR_ARG;
  return psd_plan_store_function_impl(plan, id, row, which, cap, n_pieces, max_log_mean, data_i, prev_log_mean);
}

// The text R/writeBedGraph.R:35-37 produces (data.table::fwrite, tab separated, no header), written
// with a hand-rolled integer formatter: ~1 GB/s instead of the tens of MB/s of formatted I/O.
int psd_write_bedgraph(const char* path, const char* chrom, int64_t n_rows, const int32_t* chromStart,
                       const int32_t* chromEnd, const int32_t* count) {
  if (!path || !chrom || n_rows < 0 || (n_rows > 0 && (!chromStart || !chromEnd || !count))) return PSD_ERR_ARG;
  FILE* f = fopen(path, "wb");
  if (!f) return PSD_ERR_ARG;
  const size_t clen = strlen(chrom);
  std::vector<char> buf;
  buf.reserve((1u << 20) + clen + 64);
  auto put_int = [&](int32_t v) {
    char tmp[16]; int k = 0;
    unsigned u = v < 0 ? 0u - (unsigned)v : (unsigned)v;
    do { tmp[k++] = (char)('0' + u % 10); u /= 10; } while (u);
    if (v < 0) buf.push_back('-');
    while (k) buf.push_back(tmp[--k]);
  };
  bool ok = true;
  for (int64_t i = 0; i < n_rows; i++) {
    buf.insert(buf.end(), chrom, chrom + clen);
    buf.push_back('\t'); put_int(chromStart[i]); buf.push_back('\t'); put_int(chromEnd[i]); buf.push_back('\t'); put_int(count[i]); buf.push_back('\n');
    if (buf.size() >= (1u << 20)) { ok = ok && fwrite(buf.data(), 1, buf.size(), f) == buf.size(); buf.clear(); }
  }
  if (!buf.empty()) ok = ok && fwrite(buf.data(), 1, buf.size(), f) == buf.size();
  if (fclose(f) != 0) ok = false;
  return ok ? 0 : PSD_ERR_ARG;
}

int psd_last_batch_stats(psd_batch_stats* out) {
  if (!out) return PSD_ERR_ARG;
  std::lock_guard<std::mutex> lk(g_batch_stats_mutex);
  *out = g_batch_stats;
  return 0;
}

int psd_coverage_from_reads(int device, int n_problems, const psd_reads* problems, psd_coverage** out) {
  return psd_coverage_from_reads_impl(device, n_problems, problems, out);
}

int64_t psd_coverage_n_rows(const psd_coverage* cov, int i) {
  if (!cov || i < 0 || i + 1 >= (int64_t)cov->row_off.size()) return -1;
  return cov->row_off[i + 1] - cov->row_off[i];
}

int psd_coverage_rows(const psd_coverage* cov, int i, int32_t* chromStart, int32_t* chromEnd, int32_t* count) {
  const int64_t n = psd_coverage_n_rows(cov, i);
  if (n < 0 || !chromStart || !chromEnd || !count) return PSD_ERR_ARG;
  const int64_t o = cov->row_off[i];
  memcpy(chromStart, cov->chrom_start.data() + o, sizeof(int32_t) * n);
  memcpy(chromEnd, cov->chrom_end.data() + o, sizeof(int32_t) * n);
  memcpy(count, cov->count.data() + o, sizeof(int32_t) * n);
  return 0;
}

int psd_coverage_get_stats(const psd_coverage* cov, psd_coverage_stats* out) {
  if (!cov || !out) return PSD_ERR_ARG;
  *out = cov->stats;
  return 0;
}

void psd_coverage_free(psd_coverage* cov) { delete cov; }

int psd_features(int device, int n_problems, const psd_rows* problems, psd_problem_features* out, psd_features_stats* stats) {
  return psd_features_impl(device, n_problems, problems, out, stats);
}

int psd_set_option(const char* name, double value) { return name ? psd_set_option_impl(name, value) : PSD_ERR_ARG; }
int psd_device_count(void) { return psd_device_count_impl(); }
void psd_release_cache(void) { psd_plan_drop_parked(); }

}  // extern "C"

// The reference's own entry point, with its C++ linkage (src/PeakSegFPOPLog.h:15 declares it without
// extern "C"), so an unmodified src/interface.cpp links against this library.
int PeakSegFPOP_disk(char* bedGraph_file_name, char* penalty_str, char* db_file_name) {
  return psd_fpop_disk(bedGraph_file_name, penalty_str, db_file_name);
}

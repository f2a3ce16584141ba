// joint.cpp -- psd_joint_models: exact joint single-peak models of many samples (include/peaksegdisk_b200.h
// documents the model), with model selection, label errors and the target interval.
//
// The host checks every input, bins each sample's rows into int64 prefix sums at the grid points, and hands
// the problems with at least one peak (N >= 3) to the device (psd_joint_device, joint_gpu.cuh), which returns
// the minimum of loss_k and its pair for every k.  The host then recomputes, for each winning pair, the
// feasible samples, their sort and R_k with the same arithmetic (psd_log, bit-equal to the device's) and
// requires the device's loss bit for bit, so the peaked samples never come back from the device.  Model
// selection and label errors are a few hundred host operations per problem.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include "psd_math.h"
#include "plan_internal.h"

struct psd_joint {
  std::vector<int> S;
  std::vector<std::vector<psd_joint_model>> models;   // k ascending
  std::vector<std::vector<std::vector<uint8_t>>> in_peak;   // per model, S flags
  std::vector<double> target_min, target_max;
  std::vector<int> target_errors;                     // -1: no target
  psd_joint_stats stats;
};

namespace {

inline double hlog(double x) { return psd_log(x, psd_log_tab_host); }

double seg_loss(int64_t c, int64_t w) {
  if (c == 0) return 0.0;
  const double C = (double)c;
  return C - C * hlog(C / (double)w);
}

struct Prob {
  int S = 0, N = 0, bin = 0, len = 0, start = 0;
  std::vector<int64_t> pref;                                  // [grid index][sample]
  std::vector<std::shared_ptr<const LabelSet>> labels;        // per sample (null: none)
  bool any_labels = false;
};

int64_t grid(const Prob& p, int i) { return i == p.N ? (int64_t)p.len : (int64_t)i * p.bin; }

// r_s of every sample at (a, b), -inf when s cannot carry the peak (joint_pair_kernel's arithmetic)
void reductions(const Prob& p, const std::vector<double>& l1, int a, int b, std::vector<double>* r) {
  const int S = p.S, N = p.N;
  const uint64_t w0a = (uint64_t)grid(p, a), wab = (uint64_t)(grid(p, b) - grid(p, a)), wbn = (uint64_t)(p.len - grid(p, b));
  r->assign(S, -INFINITY);
  for (int s = 0; s < S; s++) {
    const int64_t c0a = p.pref[(size_t)a * S + s], c0b = p.pref[(size_t)b * S + s], tot = p.pref[(size_t)N * S + s];
    const uint64_t cab = (uint64_t)(c0b - c0a), cbn = (uint64_t)(tot - c0b);
    if (!((unsigned __int128)cab * w0a > (unsigned __int128)(uint64_t)c0a * wab && (unsigned __int128)cab * wbn > (unsigned __int128)cbn * wab)) continue;
    const double l3 = (seg_loss(c0a, (int64_t)w0a) + seg_loss((int64_t)cab, (int64_t)wab)) + seg_loss((int64_t)cbn, (int64_t)wbn);
    (*r)[s] = l1[s] - l3;
  }
}

// PeakError's fp / fn of the labels of one sample against at most one peak [ps, pe) (has_peak)
void add_label_errors(const LabelSet& L, bool has_peak, int ps, int pe, psd_joint_model* m) {
  for (size_t q = 0; q < L.kind.size(); q++) {
    const int ls = L.start[q], le = L.end[q], kind = L.kind[q];
    const int o = has_peak && ps < le && ls < pe;
    const int na = has_peak && ls <= ps && ps < le;
    const int nb = has_peak && ls < pe && pe <= le;
    int fp = 0, fn = 0;
    if (kind == 0) fp = o > 0;
    else if (kind == 1) fn = o == 0;
    else { const int c = kind == 2 ? na : nb; fp = c > 1; fn = c == 0; }
    m->fp += fp; m->fn += fn; m->possible_fp += kind != 1; m->possible_fn += kind != 0;
  }
  m->errors = m->fp + m->fn;
}

}  // namespace

static int joint_impl(int device, int n, const psd_joint_problem* P, psd_joint** out) {
  auto fail = [](const std::string& m) { psd_set_last_error("psd_joint_models: " + m); return PSD_ERR_ARG; };
  if (!out) return fail("out is null");
  *out = nullptr;
  if (n < 0 || (n > 0 && !P)) return fail("n_problems < 0 or problems is null");
  std::vector<Prob> probs(n);
  for (int k = 0; k < n; k++) {
    const psd_joint_problem& q = P[k];
    const std::string where = "problem " + std::to_string(k) + ": ";
    if (q.n_samples < 1 || q.n_samples > PSD_JOINT_MAX_SAMPLES) return fail(where + "n_samples " + std::to_string(q.n_samples) + " is outside [1, 256]");
    if (!q.samples) return fail(where + "samples is null");
    if (q.bin_bases < 1) return fail(where + "bin_bases " + std::to_string(q.bin_bases) + " < 1");
    if (q.region_end <= q.region_start) return fail(where + "region_end <= region_start");
    const int64_t len = (int64_t)q.region_end - q.region_start;
    const int64_t N = (len + q.bin_bases - 1) / q.bin_bases;
    if (N > PSD_JOINT_MAX_BINS) return fail(where + std::to_string(N) + " bins, more than PSD_JOINT_MAX_BINS (32768)");
    Prob& p = probs[k];
    p.S = q.n_samples; p.N = (int)N; p.bin = q.bin_bases; p.len = (int)len; p.start = q.region_start;
    p.pref.assign((size_t)(N + 1) * p.S, 0);
    p.labels.resize(p.S);
    for (int s = 0; s < p.S; s++) {
      const psd_joint_sample& x = q.samples[s];
      const std::string ws = where + "sample " + std::to_string(s) + ": ";
      std::string why;
      if (check_rows(x.n_rows, x.chromStart, x.chromEnd, x.coverage, &why)) return fail(ws + why);
      if (x.chromStart[0] != q.region_start || x.chromEnd[x.n_rows - 1] != q.region_end)
        return fail(ws + "rows cover [" + std::to_string(x.chromStart[0]) + ", " + std::to_string(x.chromEnd[x.n_rows - 1]) +
                    "), not the region [" + std::to_string(q.region_start) + ", " + std::to_string(q.region_end) + ")");
      HostProblem h;   // the row bounds make_label_set checks labels against
      h.n_rows = x.n_rows;
      h.rows = std::make_shared<RowData>();
      h.rows->chrom_start.assign(x.chromStart, x.chromStart + x.n_rows);
      h.rows->chrom_end.assign(x.chromEnd, x.chromEnd + x.n_rows);
      if (make_label_set(h, x.n_labels, x.label_start, x.label_end, x.label_kind, &p.labels[s], &why)) return fail(ws + why);
      p.any_labels |= (bool)p.labels[s];
      // prefix sums at the grid points: C_s(0, i) = the counts of the bases before g_i
      int64_t acc = 0;
      int64_t r = 0;
      for (int i = 1; i <= N; i++) {
        const int64_t g = i == N ? q.region_end : (int64_t)q.region_start + (int64_t)i * q.bin_bases;
        const int64_t g0 = (int64_t)q.region_start + (int64_t)(i - 1) * q.bin_bases;
        int64_t x0 = g0;
        while (x0 < g) {   // rows overlapping [g0, g)
          while (x.chromEnd[r] <= x0) r++;
          const int64_t e = std::min<int64_t>(x.chromEnd[r], g);
          acc += (int64_t)x.coverage[r] * (e - x0);
          x0 = e;
        }
        p.pref[(size_t)i * p.S + s] = acc;
      }
    }
  }

  std::unique_ptr<psd_joint> R(new psd_joint());
  psd_joint_stats& st = R->stats;
  memset(&st, 0, sizeof st);
  st.n_problems = n;
  std::vector<JointDeviceProblem> dev;
  std::vector<int64_t> off(n, -1);
  int64_t n_out = 0;
  for (int k = 0; k < n; k++) {
    st.samples += probs[k].S;
    if (probs[k].N < 3) continue;   // no peak fits
    off[k] = n_out;
    dev.push_back({probs[k].S, probs[k].N, probs[k].bin, probs[k].len, probs[k].pref.data(), n_out});
    n_out += probs[k].S;
  }
  std::vector<double> best_loss(n_out);
  std::vector<int32_t> best_t(n_out);
  if (!dev.empty()) {
    const int rc = psd_joint_device(device, dev, best_loss.data(), best_t.data(), &st);
    if (rc) return rc;
  }

  R->S.resize(n); R->models.resize(n); R->in_peak.resize(n);
  R->target_min.assign(n, NAN); R->target_max.assign(n, NAN); R->target_errors.assign(n, -1);
  for (int k = 0; k < n; k++) {
    const Prob& p = probs[k];
    const int S = p.S;
    R->S[k] = S;
    std::vector<double> l1(S);
    double flat = 0.0;
    for (int s = 0; s < S; s++) { l1[s] = seg_loss(p.pref[(size_t)p.N * S + s], p.len); flat += l1[s]; }
    std::vector<psd_joint_model>& M = R->models[k];
    std::vector<std::vector<uint8_t>>& F = R->in_peak[k];
    psd_joint_model m0;
    memset(&m0, 0, sizeof m0);
    m0.total_loss = flat; m0.peaks = 0; m0.peak_start = m0.peak_end = -1;
    M.push_back(m0);
    F.push_back(std::vector<uint8_t>(S, 0));
    std::vector<double> r;
    std::vector<int> order(S);
    int cached_t = -1;
    for (int kk = 1; off[k] >= 0 && kk <= S; kk++) {
      const int t = best_t[off[k] + kk - 1];
      if (t < 0) continue;
      // the pair of flattened index t: row a holds N - 1 - a pairs
      int a = 1, tt = t;
      while (a < p.N - 1 && tt >= p.N - 1 - a) { tt -= p.N - 1 - a; a++; }
      const int b = a + 1 + tt;
      if (a >= p.N - 1 || b > p.N - 1) { psd_set_last_error("psd_joint_models: device returned pair index " + std::to_string(t) + " outside problem " + std::to_string(k)); return PSD_ERR_INTERNAL; }
      if (t != cached_t) {
        reductions(p, l1, a, b, &r);
        for (int s = 0; s < S; s++) order[s] = s;
        std::sort(order.begin(), order.end(), [&](int x, int y) { return r[x] > r[y] || (r[x] == r[y] && x < y); });
        cached_t = t;
      }
      double Rk = 0.0;
      for (int j = 0; j < kk; j++) Rk = Rk + r[order[j]];
      const double loss = flat - Rk;
      if (r[order[kk - 1]] == -INFINITY || PSD_D2U(loss) != PSD_D2U(best_loss[off[k] + kk - 1])) {
        char msg[256];
        snprintf(msg, sizeof msg, "psd_joint_models: problem %d, k %d: the device's loss %.17g at pair (%d, %d) is not the host's %.17g",
                 k, kk, best_loss[off[k] + kk - 1], a, b, loss);
        psd_set_last_error(msg);
        return PSD_ERR_INTERNAL;
      }
      psd_joint_model m;
      memset(&m, 0, sizeof m);
      m.total_loss = loss; m.peaks = kk;
      m.peak_start = p.start + (int)grid(p, a); m.peak_end = p.start + (int)grid(p, b);
      M.push_back(m);
      std::vector<uint8_t> f(S, 0);
      for (int j = 0; j < kk; j++) f[order[j]] = 1;
      F.push_back(std::move(f));
    }
    // selectable models: corners of the lower convex hull of (k, loss_k) with positive breakpoints
    auto lam = [&](int i, int j) { return (M[i].total_loss - M[j].total_loss) / (double)(M[j].peaks - M[i].peaks); };
    std::vector<int> hull{0};
    for (int j = 1; j < (int)M.size(); j++) {
      while (hull.size() >= 2 && !(lam(hull[hull.size() - 2], hull.back()) > lam(hull.back(), j))) hull.pop_back();
      hull.push_back(j);
    }
    while (hull.size() >= 2 && !(lam(hull[hull.size() - 2], hull.back()) > 0)) hull.pop_back();
    for (auto& m : M) { m.min_lambda = NAN; m.max_lambda = NAN; }
    for (size_t h = 0; h < hull.size(); h++) {
      psd_joint_model& m = M[hull[h]];
      m.selectable = 1;
      m.max_lambda = h == 0 ? INFINITY : lam(hull[h - 1], hull[h]);
      m.min_lambda = h + 1 == hull.size() ? 0.0 : lam(hull[h], hull[h + 1]);
    }
    if (p.any_labels) {
      for (size_t i = 0; i < M.size(); i++)
        for (int s = 0; s < S; s++)
          if (p.labels[s]) add_label_errors(*p.labels[s], F[i][s] != 0, M[i].peak_start, M[i].peak_end, &M[i]);
      std::vector<psd_path_model> sel;
      for (int h : hull) {
        psd_path_model x;
        memset(&x, 0, sizeof x);
        x.min_lambda = M[h].min_lambda; x.max_lambda = M[h].max_lambda; x.peaks = M[h].peaks; x.errors = M[h].errors;
        sel.push_back(x);
      }
      target_interval(sel, &R->target_min[k], &R->target_max[k], &R->target_errors[k]);
    }
  }
  *out = R.release();
  return 0;
}

extern "C" {

int psd_joint_models(int device, int n_problems, const psd_joint_problem* problems, psd_joint** out) {
  return joint_impl(device, n_problems, problems, out);
}

int psd_joint_n_models(const psd_joint* h, int i) {
  if (!h || i < 0 || i >= (int)h->models.size()) return -1;
  return (int)h->models[i].size();
}

int psd_joint_model_table(const psd_joint* h, int i, psd_joint_model* models) {
  if (!h || i < 0 || i >= (int)h->models.size() || !models) return PSD_ERR_ARG;
  std::copy(h->models[i].begin(), h->models[i].end(), models);
  return 0;
}

int psd_joint_samples(const psd_joint* h, int i, int k, uint8_t* in_peak) {
  if (!h || i < 0 || i >= (int)h->models.size() || !in_peak) return PSD_ERR_ARG;
  const auto& M = h->models[i];
  for (size_t j = 0; j < M.size(); j++)
    if (M[j].peaks == k) { std::copy(h->in_peak[i][j].begin(), h->in_peak[i][j].end(), in_peak); return 0; }
  return PSD_ERR_ARG;
}

int psd_joint_target(const psd_joint* h, int i, double* min_lambda, double* max_lambda, int32_t* errors) {
  if (!h || i < 0 || i >= (int)h->models.size() || !min_lambda || !max_lambda || !errors) return PSD_ERR_ARG;
  *min_lambda = h->target_min[i]; *max_lambda = h->target_max[i]; *errors = h->target_errors[i];
  return 0;
}

int psd_joint_get_stats(const psd_joint* h, psd_joint_stats* out) {
  if (!h || !out) return PSD_ERR_ARG;
  *out = h->stats;
  return 0;
}

void psd_joint_free(psd_joint* h) { delete h; }

}  // extern "C"

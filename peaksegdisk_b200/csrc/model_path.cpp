// model_path.cpp -- psd_model_path: every model that is optimal for some penalty in [pen_min, pen_max]
// (CROPS, Haynes, Eckley and Fearnhead 2017), for many problems at once, with label errors and the
// target interval (include/peaksegdisk_b200.h).
//
// The optimal model is a piecewise-constant function of the penalty; its breakpoints are the corners of
// the lower convex hull of (peaks, total.loss).  Rules (the tests re-implement them and compare bit for bit):
//   1. round 1 solves at pen_min and pen_max (pen_min alone when they are equal); the same peaks at both
//      make a one-model path, found at pen_min;
//   2. a model keeps (peaks, total.loss, segments, penalty) of the solve that found it, total.loss being
//      psd_plan_result's value at that penalty;
//   3. a pending pair i, j with peaks_i > peaks_j is solved at lambda = (loss_j - loss_i) / (peaks_i - peaks_j)
//      unless lambda is not finite or outside [pen_min, pen_max] (rounding only): then the pair closes at
//      lambda clamped.  A result k with peaks_j < peaks_k < peaks_i and loss_k + lambda peaks_k <
//      loss_i + lambda peaks_i is inserted and (i, k), (k, j) become pending; anything else (ties
//      included) makes lambda the boundary of i and j;
//   4. the pending pairs of all problems are solved in one batched plan solve per round.
// One plan serves all rounds: each problem's rows (one RowData) and labels (one LabelSet) are shared by
// its solves, so they are neither copied on the host nor re-packed while the set of unfinished problems
// stays the same.  Only the status words and the label totals come back from the device; no segments.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include "plan_internal.h"

struct psd_path {
  std::vector<int> status;
  std::vector<std::vector<psd_path_model>> models;   // sorted by peaks ascending
  std::vector<double> target_min, target_max;
  std::vector<int> target_errors;                    // -1: no target
  psd_path_stats stats;
};

namespace {

struct Pair { int i, j; double lambda; };   // indices into Problem::found, peaks_i > peaks_j
struct Boundary { int i, j; double lambda; };

struct Problem {
  HostProblem tmpl;                 // rows and labels, shared by every solve of this problem
  int status = 0;
  std::vector<psd_path_model> found;
  std::vector<Pair> pending;        // solved this round (jobs index it)
  std::vector<Pair> fresh;          // pending for the next round
  std::vector<Boundary> closed;
};

struct Job { int prob; int pair; double penalty; };   // pair -1: a round-1 solve

}  // namespace

static int model_path_impl(int device, int n, const psd_path_problem* P, double pen_min, double pen_max, psd_path** out) {
  auto fail = [](const std::string& m) { psd_set_last_error("psd_model_path: " + m); return PSD_ERR_ARG; };
  if (!out) return fail("out is null");
  *out = nullptr;
  if (n < 0 || (n > 0 && !P)) return fail("n_problems < 0 or problems is null");
  if (std::isnan(pen_min) || pen_min < 0) return fail("pen_min must be a non-negative number");
  if (std::isnan(pen_max)) return fail("pen_max is NaN");
  if (std::isinf(pen_min) && !std::isinf(pen_max)) return fail("pen_min is infinite and pen_max is not");
  if (pen_min > pen_max) return fail("pen_min > pen_max");
  std::vector<Problem> probs(n);
  for (int k = 0; k < n; k++) {
    const psd_path_problem& q = P[k];
    std::string why;
    if (check_rows(q.n_rows, q.chromStart, q.chromEnd, q.coverage, &why)) return fail("problem " + std::to_string(k) + ": " + why);
    probs[k].tmpl = make_row_problem(q.n_rows, q.chromStart, q.chromEnd, q.coverage);
    if (make_label_set(probs[k].tmpl, q.n_labels, q.label_start, q.label_end, q.label_kind, &probs[k].tmpl.labels, &why))
      return fail("problem " + std::to_string(k) + ": " + why);
  }

  std::unique_ptr<psd_path> R(new psd_path());
  psd_path_stats& S = R->stats;
  memset(&S, 0, sizeof S);
  S.n_problems = n;
  std::unique_ptr<psd_plan, void (*)(psd_plan*)> plan(psd_plan_create_impl(device), psd_plan_destroy_impl);
  std::vector<Job> jobs;
  for (int k = 0; k < n; k++) {
    jobs.push_back({k, -1, pen_min});
    if (pen_max != pen_min) jobs.push_back({k, -1, pen_max});
  }
  auto add_pair = [&](Problem& pb, int i, int j) {
    const psd_path_model &mi = pb.found[i], &mj = pb.found[j];
    const double lam = (mj.total_loss - mi.total_loss) / (double)(mi.peaks - mj.peaks);
    if (!std::isfinite(lam) || lam < pen_min || lam > pen_max) pb.closed.push_back({i, j, std::min(std::max(lam, pen_min), pen_max)});
    else pb.fresh.push_back({i, j, lam});
  };
  while (!jobs.empty()) {
    std::vector<HostProblem>& v = psd_plan_problems(plan.get());
    v.clear();
    for (const Job& J : jobs) {
      v.push_back(probs[J.prob].tmpl);
      HostProblem& h = v.back();
      h.penalty_is_inf = std::isinf(J.penalty);
      h.penalty = h.penalty_is_inf ? 0.0 : J.penalty;
      h.trivial = h.penalty_is_inf || h.dmin == h.dmax;
    }
    int rc = psd_plan_upload_impl(plan.get(), nullptr);
    if (!rc) rc = psd_plan_solve_impl(plan.get(), nullptr);
    if (rc) return rc;
    psd_plan_collect_results(plan.get());
    const PlanSolveTotals T = psd_plan_solve_totals(plan.get());
    S.dp_ms += T.dp_ms; S.backtrack_ms += T.backtrack_ms; S.label_ms += T.label_ms;
    S.rows_solved += T.rows_solved; S.h2d_bytes += T.h2d_bytes; S.d2h_bytes += T.d2h_bytes;
    S.rounds++; S.solves += (int32_t)jobs.size();
    // the models the solves found, in job order (a problem's round-1 pair is two consecutive jobs)
    std::vector<psd_path_model> got(jobs.size());
    for (size_t t = 0; t < jobs.size(); t++) {
      Problem& pb = probs[jobs[t].prob];
      psd_result r;
      psd_plan_result(plan.get(), (int)t, &r);
      psd_label_errors e{};
      if (!r.status && pb.tmpl.labels) r.status = psd_plan_label_errors(plan.get(), (int)t, &e, nullptr, nullptr);
      if (r.status) { if (!pb.status) pb.status = r.status; continue; }
      psd_path_model& m = got[t];
      memset(&m, 0, sizeof m);
      m.penalty = jobs[t].penalty; m.total_loss = r.total_loss; m.peaks = r.n_peaks; m.segments = r.n_segments;
      m.fp = e.fp; m.fn = e.fn; m.possible_fp = e.possible_fp; m.possible_fn = e.possible_fn; m.errors = e.errors;
    }
    std::vector<Job> next;
    for (size_t t = 0; t < jobs.size(); t++) {
      const Job& J = jobs[t];
      Problem& pb = probs[J.prob];
      if (J.pair < 0) {
        const bool two = t + 1 < jobs.size() && jobs[t + 1].prob == J.prob && jobs[t + 1].pair < 0;
        if (!pb.status) {
          const psd_path_model &a = got[t], &b = got[two ? t + 1 : t];
          pb.found.push_back(a);
          if (two && a.peaks != b.peaks) {
            pb.found.push_back(b);
            if (a.peaks > b.peaks) add_pair(pb, 0, 1); else add_pair(pb, 1, 0);
          }
        }
        if (two) t++;
      } else if (!pb.status) {
        const Pair pr = pb.pending[J.pair];
        const psd_path_model &k = got[t], &mi = pb.found[pr.i], &mj = pb.found[pr.j];
        if (mj.peaks < k.peaks && k.peaks < mi.peaks && k.total_loss + pr.lambda * k.peaks < mi.total_loss + pr.lambda * mi.peaks) {
          pb.found.push_back(k);
          const int ki = (int)pb.found.size() - 1;
          add_pair(pb, pr.i, ki);
          add_pair(pb, ki, pr.j);
        } else {
          pb.closed.push_back({pr.i, pr.j, pr.lambda});
        }
      }
    }
    for (int k = 0; k < n; k++) {
      Problem& pb = probs[k];
      pb.pending.clear();
      pb.pending.swap(pb.fresh);
      if (pb.status) pb.pending.clear();
      for (size_t q = 0; q < pb.pending.size(); q++) next.push_back({k, (int)q, pb.pending[q].lambda});
    }
    jobs.swap(next);
  }

  R->status.resize(n); R->models.resize(n);
  R->target_min.assign(n, NAN); R->target_max.assign(n, NAN); R->target_errors.assign(n, -1);
  for (int k = 0; k < n; k++) {
    Problem& pb = probs[k];
    R->status[k] = pb.status;
    if (pb.status) continue;
    std::vector<psd_path_model>& f = pb.found;
    for (const Boundary& b : pb.closed) { f[b.i].max_lambda = b.lambda; f[b.j].min_lambda = b.lambda; }
    // the model with the most peaks reaches pen_min, the one with the fewest pen_max
    auto most = std::max_element(f.begin(), f.end(), [](const psd_path_model& a, const psd_path_model& b) { return a.peaks < b.peaks; });
    auto fewest = std::min_element(f.begin(), f.end(), [](const psd_path_model& a, const psd_path_model& b) { return a.peaks < b.peaks; });
    most->min_lambda = pen_min; fewest->max_lambda = pen_max;
    std::sort(f.begin(), f.end(), [](const psd_path_model& a, const psd_path_model& b) { return a.peaks < b.peaks; });
    S.models += (int32_t)f.size();
    if (pb.tmpl.labels) target_interval(f, &R->target_min[k], &R->target_max[k], &R->target_errors[k]);
    R->models[k] = std::move(f);
  }
  *out = R.release();
  return 0;
}

extern "C" {

int psd_model_path(int device, int n_problems, const psd_path_problem* problems, double pen_min, double pen_max, psd_path** out) {
  return model_path_impl(device, n_problems, problems, pen_min, pen_max, out);
}

int psd_path_status(const psd_path* path, int i) {
  if (!path || i < 0 || i >= (int)path->status.size()) return PSD_ERR_ARG;
  return path->status[i];
}

int psd_path_n_models(const psd_path* path, int i) {
  if (!path || i < 0 || i >= (int)path->models.size()) return -1;
  return (int)path->models[i].size();
}

int psd_path_models(const psd_path* path, int i, psd_path_model* models) {
  if (!path || i < 0 || i >= (int)path->models.size() || !models) return PSD_ERR_ARG;
  std::copy(path->models[i].begin(), path->models[i].end(), models);
  return 0;
}

int psd_path_target(const psd_path* path, int i, double* min_lambda, double* max_lambda, int32_t* errors) {
  if (!path || i < 0 || i >= (int)path->models.size() || !min_lambda || !max_lambda || !errors) return PSD_ERR_ARG;
  *min_lambda = path->target_min[i]; *max_lambda = path->target_max[i]; *errors = path->target_errors[i];
  return 0;
}

int psd_path_get_stats(const psd_path* path, psd_path_stats* out) {
  if (!path || !out) return PSD_ERR_ARG;
  *out = path->stats;
  return 0;
}

void psd_path_free(psd_path* path) { delete path; }

}  // extern "C"

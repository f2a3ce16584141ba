// Test oracle: a plain C restatement of psd_joint_models' model (include/peaksegdisk_b200.h) with libm's log.
// Build: gcc -O2 -ffp-contract=off -shared -fPIC -o joint_oracle.so joint_oracle.c -lm
//
// joint_oracle() scores every peak (a, b) with a_lo <= a < a_hi (all of them for a_lo = 1, a_hi = N - 1) of one
// problem given its prefix sums pref[i * S + s] = C_s(0, i), i = 0..N.  For k = 0..S it writes loss[k] (INFINITY
// when no peak of the range reaches k), the pair a_out[k], b_out[k] (-1 for k = 0 or none) and the peaked
// samples in_peak[k * S + s].  Ranges can be scored apart and merged: the smaller loss wins, ties go to the
// smaller (a, b).
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static double seg_loss(int64_t c, int64_t w) {
  if (c == 0) return 0.0;
  const double C = (double)c;
  return C - C * log(C / (double)w);
}

static int64_t grid(int i, int N, int bin, int len) { return i == N ? (int64_t)len : (int64_t)i * bin; }

typedef struct { double r; int s; } key;

static int first(const void* x, const void* y) {   // (r desc, s asc)
  const key *a = (const key*)x, *b = (const key*)y;
  if (a->r > b->r) return -1;
  if (a->r < b->r) return 1;
  return a->s < b->s ? -1 : a->s > b->s;
}

// the feasible samples of (a, b), sorted; returns their number
static int sorted_reductions(int S, int N, int bin, int len, const int64_t* pref, const double* l1, int a, int b, key* K) {
  const uint64_t w0a = (uint64_t)grid(a, N, bin, len), wab = (uint64_t)(grid(b, N, bin, len) - grid(a, N, bin, len));
  const uint64_t wbn = (uint64_t)(len - grid(b, N, bin, len));
  int nf = 0;
  for (int s = 0; s < S; s++) {
    const int64_t c0a = pref[(int64_t)a * S + s], c0b = pref[(int64_t)b * S + s], tot = pref[(int64_t)N * S + s];
    const uint64_t cab = (uint64_t)(c0b - c0a), cbn = (uint64_t)(tot - c0b);
    if ((unsigned __int128)cab * w0a > (unsigned __int128)(uint64_t)c0a * wab && (unsigned __int128)cab * wbn > (unsigned __int128)cbn * wab) {
      const double l3 = (seg_loss(c0a, (int64_t)w0a) + seg_loss((int64_t)cab, (int64_t)wab)) + seg_loss((int64_t)cbn, (int64_t)wbn);
      K[nf].r = l1[s] - l3; K[nf].s = s; nf++;
    }
  }
  qsort(K, (size_t)nf, sizeof(key), first);
  return nf;
}

int joint_oracle(int S, int N, int bin, int len, const int64_t* pref, int a_lo, int a_hi, double* loss, int* a_out,
                 int* b_out, unsigned char* in_peak) {
  double* l1 = (double*)malloc(sizeof(double) * S);
  key* K = (key*)malloc(sizeof(key) * S);
  double flat = 0.0;
  for (int s = 0; s < S; s++) { l1[s] = seg_loss(pref[(int64_t)N * S + s], len); flat += l1[s]; }
  memset(in_peak, 0, (size_t)(S + 1) * S);
  loss[0] = flat; a_out[0] = b_out[0] = -1;
  for (int k = 1; k <= S; k++) { loss[k] = INFINITY; a_out[k] = b_out[k] = -1; }
  for (int a = a_lo; a < a_hi && a < N - 1; a++) {
    for (int b = a + 1; b <= N - 1; b++) {
      const int nf = sorted_reductions(S, N, bin, len, pref, l1, a, b, K);
      double R = 0.0;
      for (int k = 1; k <= nf; k++) {
        R = R + K[k - 1].r;
        const double l = flat - R;
        if (l < loss[k]) { loss[k] = l; a_out[k] = a; b_out[k] = b; }   // pairs come in increasing (a, b)
      }
    }
  }
  for (int k = 1; k <= S; k++) {
    if (a_out[k] < 0) continue;
    sorted_reductions(S, N, bin, len, pref, l1, a_out[k], b_out[k], K);
    for (int j = 0; j < k; j++) in_peak[(int64_t)k * S + K[j].s] = 1;
  }
  free(l1); free(K);
  return 0;
}

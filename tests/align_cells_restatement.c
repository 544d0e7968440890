/*
 * align_cells_restatement.c -- the Viterbi alignment of oracle/ctc_oracle.c (align_utterance, CTC lattice) restated
 * so that it also returns what the N-best aligner adds: the best path's cell index at every frame and the value of
 * the final cell the backtrace starts from.  The recursion, the window, the comparison order and the backtrace are
 * the oracle's, line for line; the labels it writes are the oracle's (tests/test_gpu_align_nbest.py checks that on
 * every alignment golden file).  N lattices per utterance: lattice r aligns hypothesis row r against the frames of
 * utterance utt[r], so the log-probabilities are never replicated.
 *
 * Values of the early exits, as the aligner defines them: the empty hypothesis scores sum_t lp[t][blank] in frame
 * order (every cell 0); one frame and one label scores lp[0][label] (cell 1); one frame and more labels is
 * infeasible: -inf, cell -1.  Built by the test module into a temporary directory (gcc -O2 -fopenmp).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define NEG_INF (-INFINITY)

static int imax(int a, int b) { return a > b ? a : b; }
static int imin(int a, int b) { return a < b ? a : b; }

/* lp: [T][V]; out: [T] labels; cell: [T] path cells; *value: the final cell's value */
static void align_cells(const double* lp, int V, const int64_t* targets, int T, int L, int blank, int64_t* out,
                        int64_t* cell, double* value) {
  for (int k = 0; k < T; k++) { out[k] = 0; cell[k] = 0; }
  *value = NAN;
  if (T == 0) return;
  const int S = 2 * L + 1;
  if (S == 1) {
    double acc = lp[blank];
    for (int k = 1; k < T; k++) acc += lp[(size_t)k * V + blank];
    *value = acc;
    return;
  }
  if (T == 1) {
    out[0] = targets[0];
    cell[0] = L == 1 ? 1 : -1;
    *value = L == 1 ? lp[targets[0]] : NEG_INF;
    return;
  }
  int64_t* ext = (int64_t*)malloc(sizeof(int64_t) * (size_t)S);
  for (int i = 0; i < S; i++) ext[i] = (i & 1) ? targets[i / 2] : (int64_t)blank;
  double* alpha = (double*)malloc(sizeof(double) * (size_t)S * (size_t)T);
  int* path = (int*)calloc((size_t)S * (size_t)T, sizeof(int));
  for (size_t q = 0; q < (size_t)S * (size_t)T; q++) alpha[q] = NEG_INF;
#define A(i, k) alpha[(size_t)(i) * T + (k)]
#define P(i, k) path[(size_t)(i) * T + (k)]
  A(0, 0) = lp[ext[0]];
  A(1, 0) = lp[ext[1]];
  for (int k = 1; k < T; k++) {
    const int start = imax(0, S - 2 * (T - k)), end = imin(k * 2 + 2, S);
    for (int i = start; i < end; i++) { A(i, k) = A(i, k - 1); P(i, k) = i; }
    for (int i = start; i < end; i++) {
      const int64_t cur = ext[i];
      if (i > 0) {
        if (A(i - 1, k - 1) > A(i, k)) { A(i, k) = A(i - 1, k - 1); P(i, k) = i - 1; }
        if (cur != blank && i - 2 > 0 && ext[i - 2] != cur && A(i - 2, k - 1) > A(i, k)) { A(i, k) = A(i - 2, k - 1); P(i, k) = i - 2; }
      }
      A(i, k) += lp[(size_t)k * V + cur];
    }
  }
  int i = S - 1;
  if (A(i - 1, T - 1) > A(i, T - 1)) i = i - 1;
  *value = A(i, T - 1);
  for (int k = T - 1; k >= 0; k--) { out[k] = ext[i]; cell[k] = i; i = P(i, k); }
#undef A
#undef P
  free(ext); free(alpha); free(path);
}

/* lp [B][T][V]; R lattices: targets [R][Lmax], tgt_len [R], utt [R]; in_len [B].
 * out, cells [R][T] (-100 / -1 past the utterance's frames); value [R]. */
void ctc_restatement_align_cells(const double* lp, int B, int T, int V, int R, const int64_t* utt, const int64_t* targets,
                                 int Lmax, const int64_t* in_len, const int64_t* tgt_len, int blank, int64_t* out,
                                 int64_t* cells, double* value) {
  (void)B;
#pragma omp parallel for schedule(dynamic)
  for (int r = 0; r < R; r++) {
    const int b = (int)utt[r];
    int64_t* o = out + (size_t)r * T;
    int64_t* c = cells + (size_t)r * T;
    for (int k = 0; k < T; k++) { o[k] = -100; c[k] = -1; }
    align_cells(lp + (size_t)b * T * V, V, targets + (size_t)r * Lmax, (int)in_len[b], (int)tgt_len[r], blank, o, c,
                value + r);
  }
}

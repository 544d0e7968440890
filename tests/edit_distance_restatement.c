/* Restatement of the edit-distance counts of include/e2e_ctc.h (e2e_ctc_edit_distance_device) for the tests: the
 * textbook Levenshtein table over pairs (errors, substitutions), compared as "fewer errors, then more substitutions",
 * with words compared token by token.  It shares no code and no key packing with csrc/edit_distance.cu.
 *
 * hyps [B * N, hyp_width], refs [B, ref_width] (dense int64), hyp_len [B * N], ref_len [B]; separator < 0: token level,
 * else word level.  A length outside [0, width] gives -1 in every output of its pairs, as the kernel does. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct { int start, len; } unit_t;

/* the units of row[0:n): every token, or the maximal runs of tokens != sep */
static int units_of(const int64_t* row, int n, int64_t sep, unit_t* out) {
  int k = 0;
  for (int i = 0; i < n; ++i) {
    if (sep < 0) { out[k].start = i; out[k].len = 1; ++k; continue; }
    if (row[i] == sep) continue;
    if (i == 0 || row[i - 1] == sep) { out[k].start = i; out[k].len = 0; ++k; }
    out[k - 1].len++;
  }
  return k;
}

static int same(const int64_t* a, unit_t ua, const int64_t* b, unit_t ub) {
  return ua.len == ub.len && memcmp(a + ua.start, b + ub.start, (size_t)ua.len * sizeof(int64_t)) == 0;
}

/* (e1, s1) better than (e2, s2) */
static int better(int64_t e1, int64_t s1, int64_t e2, int64_t s2) { return e1 < e2 || (e1 == e2 && s1 > s2); }

/* counts of one pair: out = errors, substitutions, insertions, deletions; returns the reference units */
int64_t edit_restatement_pair(const int64_t* hyp, int n, const int64_t* ref, int m, int64_t sep, int64_t* out) {
  unit_t* hu = (unit_t*)malloc(sizeof(unit_t) * (size_t)(n + 1));
  unit_t* ru = (unit_t*)malloc(sizeof(unit_t) * (size_t)(m + 1));
  const int nh = units_of(hyp, n, sep, hu), nr = units_of(ref, m, sep, ru);
  /* E[i][j], S[i][j], I[i][j]: hypothesis units [0, i) against reference units [0, j) */
  const size_t cells = (size_t)(nh + 1) * (size_t)(nr + 1);
  int64_t* E = (int64_t*)malloc(cells * sizeof(int64_t));
  int64_t* S = (int64_t*)malloc(cells * sizeof(int64_t));
  int64_t* I = (int64_t*)malloc(cells * sizeof(int64_t));
#define AT(i, j) ((size_t)(i) * (size_t)(nr + 1) + (size_t)(j))
  for (int i = 0; i <= nh; ++i) {
    for (int j = 0; j <= nr; ++j) {
      if (i == 0) { E[AT(i, j)] = j; S[AT(i, j)] = 0; I[AT(i, j)] = 0; continue; }
      if (j == 0) { E[AT(i, j)] = i; S[AT(i, j)] = 0; I[AT(i, j)] = i; continue; }
      const int eq = same(hyp, hu[i - 1], ref, ru[j - 1]);
      int64_t be = E[AT(i - 1, j - 1)] + !eq, bs = S[AT(i - 1, j - 1)] + !eq, bi = I[AT(i - 1, j - 1)];
      /* insertion: hypothesis unit i - 1 has no reference counterpart */
      if (better(E[AT(i - 1, j)] + 1, S[AT(i - 1, j)], be, bs)) { be = E[AT(i - 1, j)] + 1; bs = S[AT(i - 1, j)]; bi = I[AT(i - 1, j)] + 1; }
      /* deletion: reference unit j - 1 is missing */
      if (better(E[AT(i, j - 1)] + 1, S[AT(i, j - 1)], be, bs)) { be = E[AT(i, j - 1)] + 1; bs = S[AT(i, j - 1)]; bi = I[AT(i, j - 1)]; }
      E[AT(i, j)] = be; S[AT(i, j)] = bs; I[AT(i, j)] = bi;
    }
  }
  out[0] = E[AT(nh, nr)];
  out[1] = S[AT(nh, nr)];
  out[2] = I[AT(nh, nr)];
  out[3] = out[0] - out[1] - out[2];
#undef AT
  free(E); free(S); free(I); free(hu); free(ru);
  return nr;
}

void edit_restatement(int B, int N, const int64_t* hyps, int hyp_width, const int64_t* hyp_len, const int64_t* refs,
                      int ref_width, const int64_t* ref_len, int64_t sep, int64_t* errors, int64_t* subs, int64_t* ins,
                      int64_t* dels, int64_t* ref_units) {
  for (int b = 0; b < B; ++b) {
    const int64_t m = ref_len[b];
    const int bad_ref = m < 0 || m > ref_width;
    ref_units[b] = -1;
    for (int n = 0; n < N; ++n) {
      const int64_t r = (int64_t)b * N + n, h = hyp_len[r];
      int64_t out[4] = {-1, -1, -1, -1};
      if (!bad_ref && h >= 0 && h <= hyp_width) {
        edit_restatement_pair(hyps + r * hyp_width, (int)h, refs + (int64_t)b * ref_width, (int)m, sep, out);
      }
      errors[r] = out[0]; subs[r] = out[1]; ins[r] = out[2]; dels[r] = out[3];
    }
    if (!bad_ref) {
      unit_t* ru = (unit_t*)malloc(sizeof(unit_t) * (size_t)(m + 1));
      ref_units[b] = units_of(refs + (int64_t)b * ref_width, (int)m, sep, ru);
      free(ru);
    }
  }
}

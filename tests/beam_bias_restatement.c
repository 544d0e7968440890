/*
 * TEST INFRASTRUCTURE ONLY -- the N best prefixes of the prefix beam search with phrase biasing, over sub-word labels
 * with a word n-gram language model fused in, restated in plain C.
 *
 * The search is tests/beam_lm_tokens_restatement.c's (kept as it is below) with the bias of include/e2e_ctc.h,
 * e2e_ctc_bias, added last to every score the search ranks with: committed + phi of the prefix's label sequence.  Both
 * are computed by brute force from the definition, with no automaton: committed is the left fold over the positions of
 * out_i, out_i found by testing every phrase for being a suffix of the first i labels (so a node stores the fold up to
 * its own position), and phi by testing every suffix length against every phrase.  The final ranking and the returned
 * scores add committed only.  With lmwt = 0, oov_penalty = 0 and a character alphabet written as kinds the search is
 * the LM-free one.  tests/test_gpu_beam_bias.py compiles this file into a temporary directory.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NEG_INF (-INFINITY)
#define MAXO 6
#define NCTX (MAXO - 1)

typedef struct {
  int order, n_ngrams, n_vocab, bos, eos, unk;
  const int32_t* ng_ids;     /* [n_ngrams][6], oldest word first */
  const int32_t* ng_n;       /* [n_ngrams] */
  const double *ng_prob, *ng_bow;
  const int32_t* voc_off;    /* [n_vocab + 1]: spelling of word i = voc_chars[voc_off[i] .. voc_off[i + 1]); */
  const int32_t* voc_chars;  /*   a word that cannot be spelled (<s>, </s>, <unk>) has voc_off[i + 1] < voc_off[i] + 1 and is skipped */
  const int32_t* voc_ok;     /* [n_vocab]: 1 if the word can be spelled */
  const int32_t* label_kind; /* [V]: 0 continuation, 1 word start, 2 boundary (the blank's entry is not read) */
  const int32_t* label_off;  /* [V + 1]: label c spells label_chars[label_off[c] .. label_off[c + 1]) */
  const int32_t* label_chars;
  double lmwt, oov_penalty;
  int n_phrases;
  const int32_t* ph_off;     /* [n_phrases + 1]: phrase i is ph_labels[ph_off[i] .. ph_off[i + 1]) */
  const int32_t* ph_labels;
  const double* ph_w;        /* [n_phrases]: per-token weight */
  int ph_max;                /* the longest phrase's length */
} LM;

/* out of the sequence y[0..n): the phrases that are a suffix of it, in ascending phrase index, w * k summed */
static double bias_out(const LM* m, const int* y, int n) {
  double acc = 0.0;
  for (int i = 0; i < m->n_phrases; i++) {
    const int k = m->ph_off[i + 1] - m->ph_off[i];
    if (k > n || memcmp(y + n - k, m->ph_labels + m->ph_off[i], sizeof(int) * (size_t)k) != 0) continue;
    acc = acc + m->ph_w[i] * (double)k;
  }
  return acc;
}

/* phi of y[0..n): d times the largest weight of the phrases whose proper prefix is y's suffix of length d, d the longest
 * such suffix length */
static double bias_phi(const LM* m, const int* y, int n) {
  for (int d = n < m->ph_max - 1 ? n : m->ph_max - 1; d >= 1; d--) {   /* a proper prefix is shorter than its phrase */
    double best = -1.0;
    for (int i = 0; i < m->n_phrases; i++) {
      const int k = m->ph_off[i + 1] - m->ph_off[i];
      if (k <= d || memcmp(y + n - d, m->ph_labels + m->ph_off[i], sizeof(int) * (size_t)d) != 0) continue;
      if (m->ph_w[i] > best) best = m->ph_w[i];
    }
    if (best > 0.0) return (double)d * best;
  }
  return 0.0;
}

/* index of the n-gram w[0..n) or -1 */
static int ng_find(const LM* m, const int* w, int n) {
  for (int i = 0; i < m->n_ngrams; i++) {
    if (m->ng_n[i] != n) continue;
    int k = 0;
    while (k < n && m->ng_ids[(size_t)i * MAXO + k] == w[k]) k++;
    if (k == n) return i;
  }
  return -1;
}

/* ln10 * log10 P(w | history h[0..NCTX), h[NCTX-1] the most recent word, -1 before the start) with ARPA backoff */
static double lm_term(const LM* m, const int* h, int w) {
  int nctx = 0;
  while (nctx < NCTX && nctx < m->order - 1 && h[NCTX - 1 - nctx] >= 0) nctx++;
  double t = 0.0;
  for (int j = nctx; j >= 0; j--) {
    int key[MAXO];
    for (int i = 0; i < j; i++) key[i] = h[NCTX - j + i];
    key[j] = w;
    const int e = ng_find(m, key, j + 1);
    if (e >= 0) { t = t + m->ng_prob[e]; break; }
    if (j > 0) { const int c = ng_find(m, key, j); if (c >= 0) t = t + m->ng_bow[c]; }
  }
  return t * M_LN10;
}

/* the word id of a spelling, or -1 (out of vocabulary) */
static int word_of(const LM* m, const int* sp, int n) {
  for (int i = 0; i < m->n_vocab; i++) {
    if (!m->voc_ok[i] || m->voc_off[i + 1] - m->voc_off[i] != n) continue;
    if (n == 0 || memcmp(m->voc_chars + m->voc_off[i], sp, sizeof(int) * (size_t)n) == 0) return i;
  }
  return -1;
}

/* the LM state of a prefix: current word's spelling, history, LM sum, OOV count */
typedef struct { int* word; int wlen; int h[NCTX]; double lm; int oov; } LMState;

/* the state after completing the current word (if any) */
static LMState lm_complete(const LM* m, const LMState* s) {
  LMState r = *s;
  r.word = NULL; r.wlen = 0;
  if (s->wlen == 0) return r;
  int w = word_of(m, s->word, s->wlen);
  if (w < 0) { w = m->unk; r.oov++; }
  r.lm = s->lm + lm_term(m, s->h, w);
  for (int i = 0; i < NCTX - 1; i++) r.h[i] = s->h[i + 1];
  r.h[NCTX - 1] = w;
  return r;
}

/* the state of the prefix extended with label c (the word is copied) */
static LMState lm_extend(const LM* m, const LMState* s, int c) {
  const int kind = m->label_kind[c];
  LMState r = kind == 0 ? *s : lm_complete(m, s);
  if (kind == 2) return r;
  const int n = m->label_off[c + 1] - m->label_off[c], base = kind == 0 ? s->wlen : 0;
  r.word = (int*)malloc(sizeof(int) * (size_t)(base + n + 1));
  if (base) memcpy(r.word, s->word, sizeof(int) * (size_t)base);
  if (n) memcpy(r.word + base, m->label_chars + m->label_off[c], sizeof(int) * (size_t)n);
  r.wlen = base + n;
  return r;
}

/* the word count of the prefix extended with label c */
static int words_after(const LM* m, const LMState* s, int nw, int c) {
  const int kind = m->label_kind[c];
  if (kind == 1) return nw + 1;
  if (kind == 2) return nw;
  return nw + (s->wlen == 0 ? 1 : 0);
}

static double lm_score(const LM* m, double full, const LMState* s, int num_words, double wip) {
  return ((full + m->lmwt * s->lm) - num_words * wip) + s->oov * m->oov_penalty;
}

static double lse2(double a, double b) {
  if (a == NEG_INF) return b;
  if (b == NEG_INF) return a;
  if (a > b) return a + log(1.0 + exp(b - a));
  return b + log(1.0 + exp(a - b));
}

/*
 * LM-free prefix beam search, one utterance: src/decoders/ctc_decoder.cpp:353-441 (decode_sentence) with
 * get_next_prefix (:241-309, the lm_model == nullptr branch), Prefix::next_step / get_prev_full_prob (:331-340),
 * get_prev_full_prob_with_lmwt (:311-315) and Prefix::get_sentence (:225-239).
 *
 * The reference keeps prefixes as shared_ptr objects; a child is found through a weak_ptr in its parent's
 * `next_data`.  What that ownership model DOES is restated with explicit reference counts (BNode.refs: one for
 * membership of the beam + one per living child, exactly the shared_ptr holders `prefixes` and `Prefix::parent`):
 *   - a child that is still in the beam is found and accumulates (is_new == false, :244-246),
 *   - a child that was pruned but is kept alive by a descendant in the beam is ALSO found, is not in the list,
 *     and therefore swallows the extension: that prefix cannot re-enter the beam while the descendant lives
 *     (a property of the reference, reproduced on purpose),
 *   - a child whose last owner went away has expired: a fresh prefix is made (:248-308).
 * The V-1 fresh prefixes every beam member makes per frame (:377-378) are records in a flat array here; only
 * those that survive the prune become nodes (the others are created and destroyed within the frame in the
 * reference, unobserved).  Scores: get_prev_full_prob() + lm_score*lmwt - num_words*wip + num_oov_words*oov_penalty
 * with lm_score = 0, lmwt = 0 (ctc_decoder.cpp:76), num_oov_words = 0.
 * Prune (:399-410) keeps the beam_width best; std::nth_element / std::sort leave the choice among EQUAL scores to
 * the library -- here ties go to the lower position (beam members in beam order, then fresh prefixes by
 * (member, symbol)), and the surviving list keeps that order.
 * Result: the symbols of the n_best best prefixes of the final sorted list (:413-419); the EMPTY prefix yields the
 * single symbol -1 with length 1 (get_sentence pushes last_char = -1 of the root), as the compiled reference returns.
 */
typedef struct BNode {
  struct BNode *parent, *first_child, *next_sib;
  int chr, refs, slot;
  LMState st;
  double committed;   /* the bias fold up to this node's position */
} BNode;

/* the label sequence of a node (the root's empty), into y; its length */
static int node_labels(const BNode* n, int* y) {
  int len = 0;
  for (const BNode* p = n; p->parent; p = p->parent) len++;
  int k = len;
  for (const BNode* p = n; p->parent; p = p->parent) y[--k] = p->chr;
  return len;
}

static void bnode_unref(BNode* n) {
  while (n && --n->refs == 0) {
    BNode* p = n->parent;
    if (p) {  /* weak_ptr in the parent's next_data expires */
      BNode** q = &p->first_child;
      while (*q != n) q = &(*q)->next_sib;
      *q = n->next_sib;
    }
    free(n->st.word);
    free(n);
    n = p;
  }
}

typedef struct { double score; int idx; } BKey;
static int bkey_cmp(const void* a, const void* b) {
  const BKey *x = (const BKey*)a, *y = (const BKey*)b;
  if (x->score > y->score) return -1;
  if (x->score < y->score) return 1;
  return x->idx < y->idx ? -1 : (x->idx > y->idx ? 1 : 0);
}


static void beam_utterance(const LM* m, const double* lp, int V, int T, int blank, int beam_width, int n_best, double wip, int64_t* out, int Tw, int64_t* out_len, double* scores, double* log_probs,
                           double* lm_scores, int64_t* oov_words, double* bias_scores, int64_t* ties) {
  const size_t cap = (size_t)beam_width + 1;
  int64_t n_ties = 0;   /* prunes (and the final pick) where EQUAL scores straddle the cut: the reference's choice is libstdc++'s */
  BNode** node = (BNode**)malloc(sizeof(BNode*) * cap);
  BNode** node2 = (BNode**)malloc(sizeof(BNode*) * cap);
  double *pb = (double*)malloc(sizeof(double) * cap), *pnb = (double*)malloc(sizeof(double) * cap);
  double *pb2 = (double*)malloc(sizeof(double) * cap), *pnb2 = (double*)malloc(sizeof(double) * cap);
  double *npb = (double*)malloc(sizeof(double) * cap), *npnb = (double*)malloc(sizeof(double) * cap), *full = (double*)malloc(sizeof(double) * cap);
  int *nw = (int*)malloc(sizeof(int) * cap), *nw2 = (int*)malloc(sizeof(int) * cap);
  /* fresh prefixes of this frame, indexed member * V + symbol */
  const size_t fcap = cap * (size_t)V;
  double* f_pnb = (double*)malloc(sizeof(double) * fcap);
  int* f_nw = (int*)malloc(sizeof(int) * fcap);
  char* f_made = (char*)malloc(fcap);
  LMState* f_st = (LMState*)malloc(sizeof(LMState) * fcap);
  LMState* comp = (LMState*)malloc(sizeof(LMState) * cap);   /* per member: the state after completing its word */
  char* alive = (char*)malloc(cap + fcap);
  BKey* keys = (BKey*)malloc(sizeof(BKey) * (fcap + cap));
  double* f_com = (double*)malloc(sizeof(double) * fcap);   /* committed of a fresh prefix */
  double* f_bias = (double*)malloc(sizeof(double) * fcap);  /* its committed + phi */
  double* m_bias = (double*)malloc(sizeof(double) * cap);   /* a member's committed + phi */
  int* ybuf = (int*)malloc(sizeof(int) * ((size_t)T + 2));

  BNode* root = (BNode*)calloc(1, sizeof(BNode));   /* get_initial_prefix (:201-209) */
  root->chr = -1; root->refs = 1; root->slot = 0;
  for (int i = 0; i < NCTX; i++) root->st.h[i] = i == NCTX - 1 ? m->bos : -1;
  int W = 1;
  node[0] = root; pb[0] = 0.0; pnb[0] = NEG_INF; nw[0] = 0;

  for (int t = 0; t < T; t++) {
    const double* row = lp + (size_t)t * V;
    for (int s = 0; s < W; s++) { full[s] = lse2(pnb[s], pb[s]); npb[s] = NEG_INF; npnb[s] = NEG_INF; comp[s] = lm_complete(m, &node[s]->st); }
    memset(f_made, 0, (size_t)W * V);
    for (int s = 0; s < W; s++) {   /* the bias of every member and of its extension by every label */
      const int n = node_labels(node[s], ybuf);
      m_bias[s] = node[s]->committed + bias_phi(m, ybuf, n);
      for (int c = 0; c < V; c++) {
        if (c == blank) continue;
        ybuf[n] = c;
        const size_t f = (size_t)s * V + c;
        f_com[f] = node[s]->committed + bias_out(m, ybuf, n + 1);
        f_bias[f] = f_com[f] + bias_phi(m, ybuf, n + 1);
      }
    }
    for (int c = 0; c < V; c++) {          /* for every character (:368) */
      const double cur = row[c];
      for (int s = 0; s < W; s++) {        /* for every prefix (:371) */
        if (c == blank) { npb[s] = lse2(npb[s], cur + full[s]); continue; }
        BNode* ch = node[s]->first_child;  /* get_next_prefix (:244-246): a living child is found */
        while (ch && ch->chr != c) ch = ch->next_sib;
        double sink = NEG_INF, *target;
        if (ch) target = ch->slot >= 0 ? &npnb[ch->slot] : &sink;   /* in the beam, or kept alive by a descendant */
        else {
          const size_t f = (size_t)s * V + c;
          f_made[f] = 1; f_pnb[f] = NEG_INF;
          f_nw[f] = words_after(m, &node[s]->st, nw[s], c);
          if (m->label_kind[c] != 0) f_st[f] = comp[s];   /* the new word of a word start is spelled when the node is made */
          else { f_st[f] = node[s]->st; f_st[f].word = NULL; }   /* the grown word is spelled when the node is made */
          target = &f_pnb[f];
        }
        if (c == node[s]->chr) {   /* repeated character (:381-385) */
          *target = lse2(*target, cur + pb[s]);
          npnb[s] = lse2(npnb[s], cur + pnb[s]);
        } else {
          *target = lse2(*target, cur + full[s]);
        }
      }
    }
    /* next_step for everybody (:397), then the prune (:399-410) */
    int total = 0;
    for (int s = 0; s < W; s++) { keys[total].score = lm_score(m, lse2(npnb[s], npb[s]), &node[s]->st, nw[s], wip) + m_bias[s]; keys[total++].idx = s; }
    for (size_t f = 0; f < (size_t)W * V; f++)
      if (f_made[f]) { keys[total].score = lm_score(m, lse2(f_pnb[f], NEG_INF), &f_st[f], f_nw[f], wip) + f_bias[f]; keys[total++].idx = W + (int)f; }
    int keep = total;
    if (total > beam_width) {
      qsort(keys, (size_t)total, sizeof(BKey), bkey_cmp);
      keep = beam_width;
      if (keys[keep - 1].score == keys[keep].score) n_ties++;
    }
    memset(alive, 0, (size_t)W + (size_t)W * V);
    for (int i = 0; i < keep; i++) alive[keys[i].idx] = 1;
    int W2 = 0;   /* the surviving list, in position order */
    for (int s = 0; s < W; s++)
      if (alive[s]) { node2[W2] = node[s]; pb2[W2] = npb[s]; pnb2[W2] = npnb[s]; nw2[W2] = nw[s]; W2++; }
    for (int s = 0; s < W; s++)
      for (int c = 0; c < V; c++) {
        const size_t f = (size_t)s * V + c;
        if (!f_made[f] || !alive[W + f]) continue;
        BNode* n = (BNode*)calloc(1, sizeof(BNode));
        n->chr = c; n->refs = 1; n->parent = node[s]; node[s]->refs++;
        n->st = lm_extend(m, &node[s]->st, c);
        n->committed = f_com[f];
        n->next_sib = node[s]->first_child; node[s]->first_child = n;
        node2[W2] = n; pb2[W2] = NEG_INF; pnb2[W2] = f_pnb[f]; nw2[W2] = f_nw[f]; W2++;
      }
    for (int s = 0; s < W; s++) if (!alive[s]) { node[s]->slot = -1; bnode_unref(node[s]); }
    W = W2;
    for (int s = 0; s < W; s++) { node[s] = node2[s]; node[s]->slot = s; pb[s] = pb2[s]; pnb[s] = pnb2[s]; nw[s] = nw2[s]; }
  }

  /* std::sort (:413-419): the final list in score order, equal scores by position; prefixes[0] is decode's result */
  LMState* fin = comp;   /* end of the utterance: the trailing word is completed, then </s> is scored */
  for (int s = 0; s < W; s++) {
    fin[s] = lm_complete(m, &node[s]->st);
    fin[s].lm = fin[s].lm + lm_term(m, fin[s].h, m->eos);
    keys[s].score = lm_score(m, lse2(pnb[s], pb[s]), &fin[s], nw[s], wip) + node[s]->committed; keys[s].idx = s;
  }
  qsort(keys, (size_t)W, sizeof(BKey), bkey_cmp);
  for (int r = 0; r < n_best && r + 1 < W; r++)   /* a returned prefix shares its score with another one */
    if (keys[r].score == keys[r + 1].score) { n_ties++; break; }
  if (ties) *ties = n_ties;
  for (int r = 0; r < n_best; r++) {
    if (r >= W) { out_len[r] = 0; scores[r] = log_probs[r] = lm_scores[r] = bias_scores[r] = NEG_INF; oov_words[r] = 0; continue; }
    const int s = keys[r].idx;
    scores[r] = keys[r].score;
    bias_scores[r] = node[s]->committed;
    lm_scores[r] = fin[s].lm; oov_words[r] = fin[s].oov;
    log_probs[r] = lse2(pnb[s], pb[s]);
    /* get_sentence (:225-239): last_char of the prefix, then of every ancestor except the root */
    int n = 0;
    for (BNode* p = node[s]; p; p = p->parent) if (p == node[s] || p->parent) n++;
    int k = n;
    int64_t* o = out + (size_t)r * Tw;
    for (BNode* p = node[s]; p; p = p->parent) if (p == node[s] || p->parent) o[--k] = p->chr;
    out_len[r] = n;
  }
  for (int s = 0; s < W; s++) bnode_unref(node[s]);
  free(node); free(node2); free(pb); free(pnb); free(pb2); free(pnb2); free(npb); free(npnb); free(full); free(nw); free(nw2);
  free(f_pnb); free(f_nw); free(f_made); free(alive); free(keys); free(f_st); free(comp);
  free(f_com); free(f_bias); free(m_bias); free(ybuf);
}

/* The n_best best prefixes of the final beam with the language model and the phrases: out [B][n_best][Tw] zero-filled,
 * Tw = max(T, 1); out_len, scores, log_probs, lm_scores, oov_words, bias_scores [B][n_best]; ties [B] (optional),
 * counted as in beam_nbest_restatement.c.  Slots past the final beam: length 0, scores = log_probs = lm_scores =
 * bias_scores = -inf, oov_words 0. */
void ctc_beam_bias_nbest(const double* lp, int B, int T, int V, const int64_t* in_len, int blank, int beam_width,
                              int n_best, double wip, double lmwt, double oov_penalty, int order, int n_ngrams,
                              const int32_t* ng_ids, const int32_t* ng_n, const double* ng_prob, const double* ng_bow,
                              int n_vocab, const int32_t* voc_off, const int32_t* voc_chars, const int32_t* voc_ok,
                              const int32_t* label_kind, const int32_t* label_off, const int32_t* label_chars, int bos,
                              int eos, int unk, int n_phrases, const int32_t* ph_off, const int32_t* ph_labels,
                              const double* ph_w, int64_t* out, int64_t* out_len, double* scores, double* log_probs,
                              double* lm_scores, int64_t* oov_words, double* bias_scores, int64_t* ties) {
  LM m = {order, n_ngrams, n_vocab, bos, eos, unk, ng_ids, ng_n, ng_prob, ng_bow, voc_off, voc_chars, voc_ok, label_kind,
          label_off, label_chars, lmwt, oov_penalty, n_phrases, ph_off, ph_labels, ph_w, 0};
  for (int i = 0; i < n_phrases; i++) if (ph_off[i + 1] - ph_off[i] > m.ph_max) m.ph_max = ph_off[i + 1] - ph_off[i];
  const int Tw = T > 1 ? T : 1;
  memset(out, 0, sizeof(int64_t) * (size_t)B * n_best * Tw);
#pragma omp parallel for schedule(dynamic)
  for (int b = 0; b < B; b++) {
    int Ti = (int)in_len[b];
    if (Ti > T) Ti = T;
    if (Ti < 0) Ti = 0;
    const size_t o = (size_t)b * n_best;
    beam_utterance(&m, lp + (size_t)b * T * V, V, Ti, blank, beam_width, n_best, wip, out + o * Tw, Tw,
                   out_len + o, scores + o, log_probs + o, lm_scores + o, oov_words + o, bias_scores + o, ties ? ties + b : NULL);
  }
}

// K8 -- LM-free CTC prefix beam search (SURVEY.md 8(f3)).
//
// Replaces src/decoders/ctc_decoder.cpp: decode (:153-198), decode_sentence (:353-441), get_next_prefix (:241-309, the
// branch without a language model), Prefix::next_step / get_prev_full_prob (:331-340), get_prev_full_prob_with_lmwt
// (:311-315) and Prefix::get_sentence (:225-239), plus the F.log_softmax of decoders/ctc_decoder.py:95-97 when the
// input is raw logits.
//
// One CTA per utterance; the frames are a dependent chain, the work inside a frame is parallel:
//   * the beam (<= beam_width prefixes: trie node, last symbol, word count, log p(blank), log p(not blank)) lives in
//     shared memory, double buffered;
//   * the reference makes a Prefix object for each of the beam x (V-1) extensions of a frame and throws all but
//     beam_width of them away (std::nth_element).  Here an extension is never materialised: its score is one add of
//     the frame's log-probability to a per-member base, recomputed wherever it is needed;
//   * the beam_width best of the beam members + extensions are found on an order-preserving 64-bit image of the fp64
//     score (kept in shared memory when beam x V fits): normally by ONE 256-bin histogram over the keys within +-3 nats of
//     the predicted cut (the cut moves slowly relative to the frame's best score; keys above the window are only counted)
//     and an exact ranking of the boundary bin's few keys; otherwise (first frames, cut outside the window, keys not
//     cached) by an MSB-first radix select (8-bit digits from the highest byte in which the keys differ, stopping as soon
//     as a digit bin holds exactly what is still needed).  Both select the same set;
//   * large alphabets (beam x V beyond the key cache): for one member the extensions with an ordinary symbol rank by the
//     symbol's log-probability alone, so only the beam_width + 2 most probable symbols of the frame (ties included; the
//     member's own last symbol and the space score differently) plus the space can reach the beam_width best.  Their
//     threshold comes from a radix select over the row, and every member is extended with that list only (c4, V = 1024:
//     104 of 1023 symbols, 73 -> 14 ms); same results as without the filter;
//   * survivors are compacted in position order (members in beam order, then extensions by (member, symbol)) with
//     ballot / popc ranks and one scan over the per-member counts: bitwise reproducible.
//
// The reference finds an existing child through a weak_ptr in its parent (:244-246).  What that does is kept exactly:
// the prefix trie lives in the caller's workspace with a reference count per node (one for membership of the beam, one per
// living child = the shared_ptr holders `prefixes` and `Prefix::parent`); the slot of every member's parent and the pruned
// prefixes that still block an extension of a member (at most one per member, see DESIGN.md) are kept in shared memory, so
// the frame loop follows no pointers, and
//   - an extension whose node is in the beam adds its mass to that member (is_new == false),
//   - an extension whose node was pruned but is still referenced by a descendant in the beam is swallowed: that prefix
//     cannot re-enter the beam while the descendant lives (a property of the reference, reproduced on purpose),
//   - otherwise the extension is a fresh prefix.
// Equal scores on both sides of the prune cut are resolved by libstdc++'s introselect in the reference; here the lower
// position wins and the utterance's tie counter is raised, so a caller can tell when the result depended on that.
//
// Arithmetic: fp64 log-space with the reference's two-argument log_sum_exp (src/utils/math_utils.h:8-16) and the score
// expression of :311-315 evaluated in its order without fused multiply-adds.
//
// The LM template parameter fuses a word n-gram language model into the same search (include/e2e_ctc.h, e2e_ctc_ngram and
// e2e_ctc_ngram_tokens).  Every label has a kind: a continuation grows the current word, a word start or a boundary
// completes it (characters: the space is the boundary, every other label a continuation).  For one member the
// extensions of one kind differ only by the label's log-probability (BeamExt), so the symbol filter ranks each kind on
// its own, and the select and the trie are as above.  Each new member walks the lexicon through its label's characters
// and looks up what completing its current word would add once, right after the write phase; LM = false compiles to the
// LM-free kernel unchanged.
//
// The BIAS template parameter boosts caller-given phrases (include/e2e_ctc.h, e2e_ctc_bias), with or without the LM: every
// member carries its node of an Aho-Corasick automaton over labels and its committed bonus, and every key adds committed
// + partial credit of the extended prefix.  A label in no phrase moves to the root and adds the member's committed
// bonus alone, so the symbol filter ranks those labels as before and extends every member with every phrase label as
// well; BIAS = false compiles to the kernel without it unchanged.
#include <cstdio>
#include <cstdlib>

#include "common.cuh"

namespace e2e {
namespace {

struct __align__(16) BeamNode {   // 16 bytes
  int parent, chr, refs, depth;
};

struct BeamParams {
  const void* logits; int dtype; long long sb, st;
  const void* in_len; int len_is64;
  long long* decoded;        // [B, n_best, T] zero padded
  long long* decoded_len;    // [B, n_best]
  double* scores;            // [B, n_best] or null: the ranking score
  double* log_probs;         // [B, n_best] or null: log p of the prefix, without the word penalty
  long long* ties;           // [B] or null
  BeamNode* nodes;           // [B][node_cap]
  long long node_cap;
  int B, T, V, blank, beam, space, from_logits, n_best;
  int prefilter;             // large alphabets: only the beam+2 most probable symbols of a frame (and the space) are extended
  int kc_cap;                // keys the shared-memory cache holds (0: none)
  double wip;
};

// ---- word n-gram language model (the LM variant, e2e_ctc_beam_lm_nbest_device) ----------------------------------------
struct __align__(16) NGramEntry {   // 48 bytes: one n-gram of the open-addressing table (n == 0: empty slot)
  int n, w[6], pad;
  double prob, bow;                 // log10 probability and backoff weight, as the ARPA file gives them
};
struct BeamLMParams {
  const NGramEntry* table; unsigned long long mask;   // slots - 1 (a power of two)
  const int* lex_child;      // [lex_nodes][n_chars]: child of a lexicon node for a character, -1: no word spelled so
  const int* lex_word;       // [lex_nodes]: the word a node spells, -1: none
  // the labels' text: label c spells label_chars[label_off[c] .. label_off[c + 1]) (character ids; a word start's marker
  // stripped) and is of kind label_kind[c] (0 continuation, 1 word start, 2 boundary).  Character alphabets pass null
  // label_kind and label_off: label_chars[c] is the one character of label c, the space is the boundary, every other
  // label a continuation.
  const signed char* label_kind;
  const int* label_off;
  const int* label_chars;
  int n_chars, order, bos, eos, unk;
  double lmwt, oov_penalty;
  double* lm_scores;         // [B, n_best]: lm of the returned prefixes, end-of-utterance terms included
  long long* oov_words;      // [B, n_best]
};
constexpr int kLMMaxOrder = 6, kLMCtx = kLMMaxOrder - 1;

// ---- phrase biasing (the BIAS variant, e2e_ctc_beam_bias_nbest_device): an Aho-Corasick automaton over labels ----------
struct BeamBiasParams {
  const int* label_col;      // [V]: column of a phrase label in next, -1 for every other label (those go to the root)
  const int* next;           // [nodes][n_cols]: the full transition function over the phrase labels
  const double* partial;     // [nodes]: phi of the node's label string (withdrawn at the end)
  const double* complete;    // [nodes]: what reaching the node adds to committed (the phrases that end there)
  int n_cols;
  double* bias_scores;       // [B, n_best]: committed of the returned prefixes
};

__device__ __forceinline__ unsigned long long ngram_hash(const int* w, int n) {   // n is a compile-time constant at the call sites
  unsigned long long h = 0x9e3779b97f4a7c15ull * (unsigned long long)(n + 1);
#pragma unroll
  for (int i = 0; i < kLMMaxOrder; i++) {
    if (i < n) { h ^= (unsigned)w[i]; h *= 0xff51afd7ed558ccdull; h ^= h >> 33; }
  }
  return h;
}

// the table entry of the n-gram w[0..n) or null
__device__ __forceinline__ const NGramEntry* ngram_find(const NGramEntry* table, unsigned long long mask, const int* w, int n) {
  unsigned long long slot = ngram_hash(w, n) & mask;
  while (true) {
    const NGramEntry* e = table + slot;
    const int en = __ldg(&e->n);
    if (en == 0) return nullptr;
    if (en == n) {
      bool eq = true;
#pragma unroll
      for (int i = 0; i < kLMMaxOrder; i++) if (i < n) eq = eq && __ldg(&e->w[i]) == w[i];
      if (eq) return e;
    }
    slot = (slot + 1) & mask;
  }
}

// ln10 * log10 P(w | history) with ARPA backoff: from the longest context down, either (context, w) is an n-gram (add its
// probability, stop) or it is not (add the context's backoff weight, 0 if it is no n-gram, and drop its oldest word).
// h4 is the most recent word of the history, h0 the oldest; -1 marks its start.  The context is at most order - 1 words.
// (out of line: it is called once per new member and once per final prefix, and the frame loop must fit the instruction
// cache)
__device__ __noinline__ double lm_term(const NGramEntry* table, unsigned long long mask, int order, int h0, int h1, int h2,
                                       int h3, int h4, int w) {
  const int h[kLMCtx] = {h0, h1, h2, h3, h4};
  int nctx = 0;
#pragma unroll
  for (int i = kLMCtx - 1; i >= 0; i--) if (h[i] >= 0 && nctx == kLMCtx - 1 - i && nctx < order - 1) nctx++;
  double t = 0.0;
#pragma unroll
  for (int j = kLMCtx; j >= 0; j--) {   // context length j
    if (j > nctx) continue;
    int key[kLMMaxOrder];
#pragma unroll
    for (int i = 0; i < kLMMaxOrder; i++) key[i] = i < j ? h[kLMCtx - j + i] : (i == j ? w : -1);
    const NGramEntry* e = ngram_find(table, mask, key, j + 1);
    if (e) { t = __dadd_rn(t, __ldg(&e->prob)); break; }
    if (j > 0) { const NGramEntry* c = ngram_find(table, mask, key, j); if (c) t = __dadd_rn(t, __ldg(&c->bow)); }
  }
  return __dmul_rn(t, 2.302585092994045684);   // M_LN10
}

__global__ void ngram_build_kernel(NGramEntry* table, unsigned long long mask, long long count, const int* ids,
                                   const int* orders, const double* probs, const double* bows) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  int w[kLMMaxOrder];
#pragma unroll
  for (int k = 0; k < kLMMaxOrder; k++) w[k] = ids[i * kLMMaxOrder + k];
  const int n = orders[i];
  unsigned long long slot = ngram_hash(w, n) & mask;
  while (atomicCAS(&table[slot].n, 0, n) != 0) slot = (slot + 1) & mask;   // the n-grams are distinct: no key to compare
#pragma unroll
  for (int k = 0; k < kLMMaxOrder; k++) table[slot].w[k] = k < n ? w[k] : -1;
  table[slot].prob = probs[i]; table[slot].bow = bows[i];
}

#ifndef E2E_BEAM_DIGIT
#define E2E_BEAM_DIGIT 8
#endif
constexpr int kBeamMaxWidth = 256;     // beam members are handled one per thread by the first 256 threads
constexpr int kBeamDigit = E2E_BEAM_DIGIT;          // radix-select digit, bits
constexpr int kBeamBins = 1 << kBeamDigit;
constexpr int kBeamTopShift = (63 / kBeamDigit) * kBeamDigit;
static_assert(kBeamBins % 32 == 0 && kBeamBins <= 2048, "digit width");
constexpr int kBeamPre = 4;        // symbols per thread of the next frame's row kept in flight (V <= 4 x threads)
constexpr int kBeamKeyCache = 19200;   // extensions (beam x alphabet) whose keys are kept in shared memory (150 KB)

// (out of line on purpose: fp64 exp + log are ~400 instructions, and the frame loop must fit the instruction cache)
__device__ __noinline__ double beam_lse(double a, double b) {   // math_utils.h:8-16
  if (a == -INFINITY) return b;
  if (b == -INFINITY) return a;
  if (a > b) return __dadd_rn(a, log(__dadd_rn(1.0, exp(__dsub_rn(b, a)))));
  return __dadd_rn(b, log(__dadd_rn(1.0, exp(__dsub_rn(a, b)))));
}

// get_prev_full_prob_with_lmwt (:311-315) without a language model: lm_score = 0, lmwt = 0, num_oov_words = 0
__device__ __forceinline__ double beam_score(double full, int num_words, double wip) {
  return __dsub_rn(__dadd_rn(full, 0.0), __dmul_rn((double)num_words, wip));
}

// order-preserving image of a double, never 0 (0 marks "no candidate"); +0 and -0 coincide, NaN sorts below everything
__device__ __forceinline__ unsigned long long beam_key(double x) {
  if (x != x) return 1ull;
  x = __dadd_rn(x, 0.0);
  const unsigned long long u = (unsigned long long)__double_as_longlong(x);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

__device__ __forceinline__ double beam_unkey(unsigned long long k) {   // the score behind a key (k > 1)
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

struct BeamBuf {          // one copy of the beam (+ the pruned prefixes that still block an extension of a member)
  double *pb, *pnb;
  int *node, *par, *last, *nw, *dep, *pslot;   // trie node, parent node, last symbol, words, length, parent's slot or -1
  int *zn, *zp, *zc;                           // blocked extensions: node, parent's slot, symbol
  // LM variant: lexicon node of the current word (-1: no word is spelled so), the word its completion scores (-1: the
  // current word is empty; the <unk> id when out of vocabulary), OOV words so far, the last words (h[kLMCtx - 1] the most
  // recent, -1 before the start), the LM sum and what completing the current word adds to it
  int *lex, *cw, *oov, *h[kLMCtx];
  double *lm, *sd;
  int* bn;                 // BIAS variant: automaton node of the prefix
  double* bc;              //   and its committed bias
};
struct BeamSmem {
  double* lp;            // [Vp]
  double *full, *npb, *npnb;
  unsigned long long* mkey;
  int *nwx;              // word count of an extension with a symbol other than space
  int *cgt, *ceq;        // per position group: survivors above the cut / in the cut class (members: [0,W), rows: [W,2W))
  unsigned* bitmap;      // [W][VW] extensions that are not fresh prefixes
  unsigned* hist;        // [kBeamBins]
  double *penx, *pens;   // word penalty of an extension with a symbol other than space / with the space
  unsigned long long* kc;   // [W][nR] keys of the extensions (0: none) when they fit
  int* rc;               // [nR] the symbols a member is extended with this frame, ascending (never the blank)
  unsigned* rmask;       // [VW] the same set as a bit mask
  double *lmx, *lms, *oox, *oos;   // LM variant: lmwt * lm and oov * oov_penalty of a continuation / of an extension that
                                   // completes the current word (word start or boundary)
  // LM variant, at the start of the dynamic shared memory (no register holds the table's address across the frame loop):
  unsigned char* kind;   // [V] kind of every label (0 continuation, 1 word start, 2 boundary)
  double* pen1;          // word penalty of a word-start extension
  int* col;              // BIAS variant, there as well: [V] column of every label in the automaton, -1: no phrase label
  double* bcom;          // BIAS variant: a member's committed bias this frame (what a non-phrase label extends it with)
  int* bnode;            //   and its automaton node
};

// get_prev_full_prob_with_lmwt (:311-315) with a language model: ((log p + lmwt * lm) - words * wip) + oov * oov_penalty
__device__ __forceinline__ double beam_score_lm(double full, double lmw, int num_words, double wip, double oovw) {
  return __dadd_rn(__dsub_rn(__dadd_rn(full, lmw), __dmul_rn((double)num_words, wip)), oovw);
}

// What an extension of one member adds to its value besides the frame's log-probability; one key expression for every
// site that builds an extension key.  Without the LM only the space scores differently (it adds no word).  With the LM
// the label's kind decides: a word start or a boundary completes the current word (lms, oos), a word start adds a word.
// So for one member the extensions of one kind rank by the label's log-probability alone.  With BIAS the bias of the
// extended prefix is added last; every label that is not a phrase label gives the member's committed bias, so the
// extensions of one kind by non-phrase labels still rank by the label's log-probability alone.
template <bool LM, bool BIAS>
struct BeamExt {
  double penx, pens, pen1, lmx, lms, oox, oos, com;
  const int* row;   // BIAS: the member's row of the automaton's transitions
  __device__ __forceinline__ BeamExt(const BeamSmem& S, int s, const BeamBiasParams& z)
      : penx(S.penx[s]), pens(S.pens[s]), pen1(LM ? S.pen1[s] : 0.0), lmx(LM ? S.lmx[s] : 0.0), lms(LM ? S.lms[s] : 0.0),
        oox(LM ? S.oox[s] : 0.0), oos(LM ? S.oos[s] : 0.0), com(BIAS ? S.bcom[s] : 0.0),
        row(BIAS ? z.next + (long long)S.bnode[s] * z.n_cols : nullptr) {}
  // the automaton node the label moves the member to (the root for a label in no phrase)
  __device__ __forceinline__ int bias_node(int c, const BeamSmem& S) const {
    const int col = S.col[c];
    return col < 0 ? 0 : __ldg(&row[col]);
  }
  // committed + phi of the extended prefix, (committed + complete) + partial
  __device__ __forceinline__ double bias(int c, const BeamSmem& S, const BeamBiasParams& z) const {
    const int col = S.col[c];
    if (col < 0) return com;
    const int n = __ldg(&row[col]);
    return __dadd_rn(__dadd_rn(com, __ldg(&z.complete[n])), __ldg(&z.partial[n]));
  }
  __device__ __forceinline__ unsigned long long key(double v, int c, const BeamSmem& S, int space,
                                                    const BeamBiasParams& z) const {
    if (BIAS) {
      double e;
      if (!LM) e = __dsub_rn(__dadd_rn(v, 0.0), c == space ? pens : penx);
      else if (S.kind[c] == 0) e = __dadd_rn(__dsub_rn(__dadd_rn(v, lmx), penx), oox);
      else e = __dadd_rn(__dsub_rn(__dadd_rn(v, lms), S.kind[c] == 1 ? pen1 : pens), oos);
      return beam_key(__dadd_rn(e, bias(c, S, z)));
    }
    if (!LM) return beam_key(__dsub_rn(__dadd_rn(v, 0.0), c == space ? pens : penx));
    const int k = S.kind[c];
    if (k == 0) return beam_key(__dadd_rn(__dsub_rn(__dadd_rn(v, lmx), penx), oox));
    return beam_key(__dadd_rn(__dsub_rn(__dadd_rn(v, lms), k == 1 ? pen1 : pens), oos));
  }
};

// :381-390: a repeated character extends from the blank-ending mass only
#define BEAM_EXT_VALUE(c, last_s, pb_s, full_s) __dadd_rn(S.lp[c], (c) == (last_s) ? (pb_s) : (full_s))

// NT threads per CTA: 512 when every utterance has an SM to itself (the frame chain is latency-bound: more warps hide more
// of it), 256 for larger batches (several CTAs per SM)
#ifdef BEAM_PROF
__device__ long long g_beam_prof[16];
#define BEAM_T(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) { const long long now_ = clock64(); g_beam_prof[k] += now_ - prof_t; prof_t = now_; } } while (0)
#else
#define BEAM_T(k) do { } while (0)
#endif
template <typename T, bool CACHE, int NT, bool LM, bool BIAS>
__global__ void __launch_bounds__(NT, 1) ctc_beam_kernel(const BeamParams p, const BeamLMParams q, const BeamBiasParams z) {
#ifdef BEAM_PROF
  long long prof_t = clock64();
#endif
  constexpr int kBeamThreads = NT, kBeamWarps = NT / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ unsigned long long s_thr, s_kmax, s_kmin;
  __shared__ int s_need, s_ties, s_excl, s_done, s_nz2, s_ovf, s_nR, s_wcnt[8], s_above, s_tie_now;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int V = p.V, WB = p.beam, VW = (V + 31) >> 5, Vp = (V + 1) & ~1;
  using raw_t = typename Elem<T>::acc_t;   // float for 32/16-bit inputs, double for f64

  BeamSmem S;
  BeamBuf C, N;
  raw_t* raw;
  {
    unsigned char* q = smem_raw;
    auto take = [&](size_t bytes) { unsigned char* r = q; q += (bytes + 15) & ~(size_t)15; return r; };
    if (LM || BIAS) {   // padded to 128 bytes: every array after it is aligned as in the LM-free layout
      if (LM) { S.kind = take((size_t)V); S.pen1 = reinterpret_cast<double*>(take(8 * WB)); }
      if (BIAS) S.col = reinterpret_cast<int*>(take(4 * (size_t)V));
      q = smem_raw + ((q - smem_raw + 127) & ~(ptrdiff_t)127);
    }
    S.lp = reinterpret_cast<double*>(take(sizeof(double) * Vp));
    raw = reinterpret_cast<raw_t*>(take(sizeof(double) * Vp));
    C.pb = reinterpret_cast<double*>(take(8 * WB)); C.pnb = reinterpret_cast<double*>(take(8 * WB));
    N.pb = reinterpret_cast<double*>(take(8 * WB)); N.pnb = reinterpret_cast<double*>(take(8 * WB));
    S.full = reinterpret_cast<double*>(take(8 * WB));
    S.npb = reinterpret_cast<double*>(take(8 * WB));
    S.npnb = reinterpret_cast<double*>(take(8 * WB));
    S.mkey = reinterpret_cast<unsigned long long*>(take(8 * WB));
    int** cf[9] = {&C.node, &C.par, &C.last, &C.nw, &C.dep, &C.pslot, &C.zn, &C.zp, &C.zc};
    int** nf[9] = {&N.node, &N.par, &N.last, &N.nw, &N.dep, &N.pslot, &N.zn, &N.zp, &N.zc};
#pragma unroll
    for (int k = 0; k < 9; k++) { *cf[k] = reinterpret_cast<int*>(take(4 * WB)); *nf[k] = reinterpret_cast<int*>(take(4 * WB)); }
    S.nwx = reinterpret_cast<int*>(take(4 * WB));
    S.cgt = reinterpret_cast<int*>(take(4 * (2 * WB + 4)));
    S.ceq = reinterpret_cast<int*>(take(4 * (2 * WB + 4)));
    S.bitmap = reinterpret_cast<unsigned*>(take((size_t)4 * WB * VW));
    S.hist = reinterpret_cast<unsigned*>(take(4 * kBeamBins));
    S.penx = reinterpret_cast<double*>(take(8 * WB)); S.pens = reinterpret_cast<double*>(take(8 * WB));
    S.rc = reinterpret_cast<int*>(take(4 * (size_t)V));
    S.rmask = reinterpret_cast<unsigned*>(take(4 * (size_t)VW));
    S.kc = reinterpret_cast<unsigned long long*>(take(CACHE ? (size_t)8 * p.kc_cap : 0));
    if (LM) {
      BeamBuf* bufs[2] = {&C, &N};
#pragma unroll
      for (int k = 0; k < 2; k++) {
        BeamBuf& u = *bufs[k];
        u.lm = reinterpret_cast<double*>(take(8 * WB)); u.sd = reinterpret_cast<double*>(take(8 * WB));
        u.lex = reinterpret_cast<int*>(take(4 * WB)); u.cw = reinterpret_cast<int*>(take(4 * WB));
        u.oov = reinterpret_cast<int*>(take(4 * WB));
#pragma unroll
        for (int i = 0; i < kLMCtx; i++) u.h[i] = reinterpret_cast<int*>(take(4 * WB));
      }
      S.lmx = reinterpret_cast<double*>(take(8 * WB)); S.lms = reinterpret_cast<double*>(take(8 * WB));
      S.oox = reinterpret_cast<double*>(take(8 * WB)); S.oos = reinterpret_cast<double*>(take(8 * WB));
    }
    if (BIAS) {
      C.bc = reinterpret_cast<double*>(take(8 * WB)); N.bc = reinterpret_cast<double*>(take(8 * WB));
      S.bcom = reinterpret_cast<double*>(take(8 * WB));
      C.bn = reinterpret_cast<int*>(take(4 * WB)); N.bn = reinterpret_cast<int*>(take(4 * WB));
      S.bnode = reinterpret_cast<int*>(take(4 * WB));
    }
  }

  long long Ti_ll = p.in_len ? load_index(p.in_len, p.len_is64, b) : (long long)p.T;
  const int Ti = (int)max(0LL, min(Ti_ll, (long long)p.T));
  BeamNode* nodes = p.nodes + (long long)b * p.node_cap;
  const T* x = reinterpret_cast<const T*>(p.logits) + (long long)b * p.sb;
  const bool use_pre = V <= kBeamThreads * kBeamPre;

  if (tid == 0) {   // get_initial_prefix (:201-209): the empty prefix with log p(blank) = 0
    BeamNode r; r.parent = -1; r.chr = -1; r.refs = 1; r.depth = 0;
    nodes[0] = r;
    C.node[0] = 0; C.par[0] = -1; C.last[0] = -1; C.nw[0] = 0; C.dep[0] = 0; C.pslot[0] = -1; C.pb[0] = 0.0; C.pnb[0] = -INFINITY;
    s_ties = 0; s_ovf = 0; s_nz2 = 0; s_tie_now = 0;
    if (LM) {   // the empty prefix: no word yet, the history is <s>
      C.lex[0] = 0; C.cw[0] = -1; C.oov[0] = 0; C.lm[0] = 0.0; C.sd[0] = 0.0;
#pragma unroll
      for (int i = 0; i < kLMCtx; i++) C.h[i][0] = i == kLMCtx - 1 ? q.bos : -1;
    }
    if (BIAS) { C.bn[0] = 0; C.bc[0] = 0.0; }   // the automaton's root, nothing committed
  }
  // The first kFront threads (8 warps) run the head of a frame -- staging the row, the log-softmax, the members' own
  // updates -- synchronising among themselves on a named barrier.  With 512 threads the other half spends that time
  // releasing the trie nodes of the members the PREVIOUS frame pruned (dependent atomics to L2: a fifth of the frame when
  // it sat on the critical path); the two halves meet at one CTA-wide barrier before the blocked-extension list is rebuilt.
  constexpr int kFront = 256;
  constexpr int kCascOff = kBeamThreads >= 2 * kBeamMaxWidth ? kBeamMaxWidth : 0;   // thread kCascOff + u releases member u
  auto front_sync = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(kFront) : "memory"); };
  __shared__ int s_ncls[2];   // LM / BIAS variants: labels of kind 0 / kind 1 (the blank and the phrase labels aside)
  if (LM || BIAS) {
    if (tid < 2) s_ncls[tid] = 0;
    __syncthreads();
    int n0 = 0, n1 = 0;
    for (int c = tid; c < V; c += kBeamThreads) {
      const int k = !LM ? 0 : q.label_kind ? (int)__ldg(&q.label_kind[c]) : (c == p.space ? 2 : 0);
      if (LM) S.kind[c] = (unsigned char)k;
      bool ranked = c != p.blank;
      if (BIAS) { const int col = __ldg(&z.label_col[c]); S.col[c] = col; ranked = ranked && col < 0; }
      if (ranked) { n0 += k == 0; n1 += k == 1; }
    }
    n0 = warp_sum(n0); n1 = warp_sum(n1);
    if (lane == 0) { if (n0) atomicAdd(&s_ncls[0], n0); if (n1) atomicAdd(&s_ncls[1], n1); }
  }
  if (!p.prefilter) {   // every symbol but the blank, in order
    for (int i = tid; i < VW; i += kBeamThreads) {
      unsigned m = (32 * i + 32 <= V) ? 0xffffffffu : ((1u << (V - 32 * i)) - 1u);
      if ((p.blank >> 5) == i) m &= ~(1u << (p.blank & 31));
      S.rmask[i] = m;
    }
  }
  raw_t pre[kBeamPre];
#pragma unroll
  for (int k = 0; k < kBeamPre; k++) {
    const int c = tid + k * kFront;
    pre[k] = (use_pre && Ti > 0 && tid < kFront && c < V) ? (raw_t)Elem<T>::load(x + c) : (raw_t)0;
  }
  __syncthreads();

  int W = 1, n_nodes = 1, nz_prev = 0, W_prev = 0;
  int casc_n = -1, casc_par = -1;                 // the node this thread releases at the top of the next frame
  double cut_depth = -1.0;                        // how far below the best score the last frame's cut was (< 0: unknown)
  unsigned long long ptcls = 0ull; int psh = 0, pneed = 0;   // last frame's cut: slot of a member after that prune
  auto prev_slot = [&](int q) -> int {
    const unsigned long long kq = S.mkey[q] >> psh;
    const int eb = S.ceq[q];
    return (kq > ptcls || (kq == ptcls && eb < pneed)) ? S.cgt[q] + min(eb, pneed) : -1;
  };
  for (int t = 0; t < Ti; t++) {
    BEAM_T(8);
    // ---- members that left the beam last frame release their node; a node nobody holds releases its parent (off the
    //      critical path: see above) ----------------------------------------------------------------------------------------
    if (casc_n >= 0) {
      int n = casc_n, par = casc_par;
      while (true) {
        const int r = atomicSub(&nodes[n].refs, 1) - 1;
        if (r > 0 || par < 0) break;
        n = par;
        par = __ldcg(&nodes[n].parent);
      }
    }
    if (tid < kFront) {
      // ---- the frame's row: staged from the registers it was prefetched into; the next frame's row is requested now ----
      const T* row = x + (long long)t * p.st;
      if (use_pre) {
#pragma unroll
        for (int k = 0; k < kBeamPre; k++) { const int c = tid + k * kFront; if (c < V) raw[c] = pre[k]; }
        if (t + 1 < Ti) {
#pragma unroll
          for (int k = 0; k < kBeamPre; k++) { const int c = tid + k * kFront; if (c < V) pre[k] = (raw_t)Elem<T>::load(row + p.st + c); }
        }
      } else {
        for (int c = tid; c < V; c += kFront) raw[c] = (raw_t)Elem<T>::load(row + c);
      }
      for (int i = tid; i < W * VW; i += kFront) S.bitmap[i] = 0u;
      if (tid == 0) { s_excl = 0; s_done = 0; s_kmax = 0ull; s_kmin = ~0ull; s_nz2 = 0; }
      front_sync();
    // ---- log-probabilities (decoders/ctc_decoder.py:95-97 when the input is raw logits): every warp reduces the whole row
    //      on its own (same order, same result) so that no block-wide reduction sits on the chain -------------------------------
    if (p.from_logits) {
      raw_t m = -INFINITY;
      for (int c = lane; c < V; c += 32) m = raw[c] > m ? raw[c] : m;
      m = warp_max(m);
      raw_t sum = 0;
      if (sizeof(raw_t) == 8) { for (int c = lane; c < V; c += 32) sum += (raw_t)exp((double)raw[c] - (double)m); }
      else { for (int c = lane; c < V; c += 32) sum += (raw_t)expf((float)raw[c] - (float)m); }
      sum = warp_sum(sum);
      const raw_t ls = sizeof(raw_t) == 8 ? (raw_t)log((double)sum) : (raw_t)logf((float)sum);
      for (int c = tid; c < V; c += kFront) {
        raw_t v = (raw[c] - m) - ls;   // torch's operation order
        if (sizeof(T) == 2) { T r; Elem<T>::store(&r, (float)v); v = (raw_t)Elem<T>::get(r); }   // torch returns the input dtype
        S.lp[c] = (double)v;
      }
    } else {
      for (int c = tid; c < V; c += kFront) S.lp[c] = (double)raw[c];
    }
    front_sync();
    if (p.prefilter) {
      // ---- large alphabets: for a given member the extensions with an ordinary symbol rank by the symbol's log-probability,
      //      so only the beam_width + 2 most probable symbols (the member's own last symbol and the space score differently)
      //      plus the space can be among the beam_width best prefixes.  Their threshold by radix select over the row.
      //      With the LM the same holds within each kind of label (BeamExt): the beam_width + 2 most probable continuations,
      //      the beam_width + 2 most probable word starts, each class by its own select, and every boundary.
      //      With BIAS the selects rank the labels of no phrase only, and every phrase label is extended. ------------------
      constexpr int kCls = LM ? 2 : 1;
      unsigned long long rcls0 = ~0ull, rcls1 = ~0ull;
      int shr0 = 56, shr1 = 56;
      for (int i = tid; i < VW; i += kFront) S.rmask[i] = 0u;
#pragma unroll
      for (int cl = 0; cl < kCls; cl++) {
        const int kR = (LM || BIAS) ? min(WB + 2, s_ncls[cl]) : min(WB + 2, V - 1);
        unsigned long long rprefix = 0ull;
        int rremaining = kR, shr = 56;
        for (; (!(LM || BIAS) || kR > 0) && shr >= 0; shr -= 8) {
          for (int i = tid; i < kBeamBins; i += kFront) S.hist[i] = 0u;
          front_sync();
          const unsigned long long pm = shr == 56 ? 0ull : (~0ull << (shr + 8));
          for (int c = tid; c < V; c += kFront) {
            if (c == p.blank || (LM && S.kind[c] != cl) || (BIAS && S.col[c] >= 0)) continue;
            const unsigned long long k = beam_key(S.lp[c]);
            if ((k & pm) == (rprefix & pm)) atomicAdd(&S.hist[(unsigned)(k >> shr) & 255u], 1u);
          }
          front_sync();
          // every warp finds the bin on its own: the same registers everywhere, nothing to broadcast through shared memory
          unsigned h[8], mine = 0;
#pragma unroll
          for (int j = 0; j < 8; j++) { h[j] = S.hist[lane * 8 + j]; mine += h[j]; }
          unsigned above = mine;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) { const unsigned u = __shfl_down_sync(0xffffffffu, above, o); if (lane + o < 32) above += u; }
          above -= mine;
          const bool here = above < (unsigned)rremaining && above + mine >= (unsigned)rremaining;
          unsigned acc = above, hd = h[0]; int d = 0;
#pragma unroll
          for (int j = 7; j > 0; j--) {
            if (d == 0) { if (acc + h[j] >= (unsigned)rremaining) { d = j; hd = h[j]; } else acc += h[j]; }
          }
          const int src = __ffs(__ballot_sync(0xffffffffu, here)) - 1;
          const int bin = __shfl_sync(0xffffffffu, lane * 8 + d, src);
          const int need_r = __shfl_sync(0xffffffffu, rremaining - (int)acc, src);
          const int cnt_r = __shfl_sync(0xffffffffu, (int)hd, src);
          rprefix |= (unsigned long long)bin << shr;
          rremaining = need_r;
          front_sync();                       // the histogram is cleared again at the top
          if (cnt_r == need_r || shr == 0) break;
        }
        if (!(LM || BIAS) || kR > 0) { if (cl == 0) { rcls0 = rprefix >> shr; shr0 = shr; } else { rcls1 = rprefix >> shr; shr1 = shr; } }
      }
      int nlist = 0;
      for (int c0 = 0; c0 < V; c0 += kFront) {   // the list, in symbol order
        const int c = c0 + tid;
        bool in = c < V && c != p.blank;
        if (LM) {
          if (in) {
            const int kd = S.kind[c];
            const unsigned long long k = beam_key(S.lp[c]);
            in = kd == 2 || (kd == 0 ? (k >> shr0) >= rcls0 : (k >> shr1) >= rcls1);
          }
        } else {
          in = in && ((beam_key(S.lp[c]) >> shr0) >= rcls0 || c == p.space);
        }
        if (BIAS) in = in || (c < V && c != p.blank && S.col[c] >= 0);
        const unsigned m = __ballot_sync(0xffffffffu, in);
        if (lane == 0) s_wcnt[warp] = __popc(m);
        front_sync();
        int off = nlist, tot = 0;
#pragma unroll
        for (int q = 0; q < kFront / 32; q++) { const int n = s_wcnt[q]; if (q < warp) off += n; tot += n; }
        if (in) { S.rc[off + __popc(m & ((1u << lane) - 1u))] = c; atomicOr(&S.rmask[c >> 5], 1u << (c & 31)); }
        nlist += tot;
        front_sync();
      }
      if (tid == 0) s_nR = nlist;
    }

    // ---- phase A: every member's own update (:372-376, :383-385) ----------------------------------------------
    if (tid < W) {
      const int s = tid;
      const double pbv = C.pb[s], pnbv = C.pnb[s];
      const double full = beam_lse(pnbv, pbv);                       // get_prev_full_prob (:331-333)
      S.full[s] = full;
      S.npb[s] = __dadd_rn(S.lp[p.blank], full);                     // log_sum_exp(-inf, x) = x
      const int last = C.last[s];
      S.npnb[s] = last >= 0 ? __dadd_rn(S.lp[last], pnbv) : -INFINITY;
      const int nws = C.nw[s];
      // :252-257 for a symbol other than space; with the LM, for a continuation (the current word is empty after a boundary)
      const int nwx = nws + ((nws == 0 || (LM ? S.kind[last] == 2 : last == p.space)) ? 1 : 0);
      S.nwx[s] = nwx;
      S.penx[s] = __dmul_rn((double)nwx, p.wip); S.pens[s] = __dmul_rn((double)nws, p.wip);
      if (LM) {   // a word start or a boundary completes the current word (if any): its LM term and OOV count join the score
        S.pen1[s] = __dmul_rn((double)(nws + 1), p.wip);
        const double lm = C.lm[s];
        const int oov = C.oov[s], cw = C.cw[s];
        const double lmx = __dmul_rn(q.lmwt, lm), oox = __dmul_rn((double)oov, q.oov_penalty);
        S.lmx[s] = lmx; S.oox[s] = oox;
        S.lms[s] = cw >= 0 ? __dmul_rn(q.lmwt, __dadd_rn(lm, C.sd[s])) : lmx;
        S.oos[s] = cw >= 0 ? __dmul_rn((double)(oov + (cw == q.unk ? 1 : 0)), q.oov_penalty) : oox;
      }
      if (BIAS) { S.bcom[s] = C.bc[s]; S.bnode[s] = C.bn[s]; }   // a label in no phrase extends it with this bias
    }
    }   // front threads
    __syncthreads();   // the members' updates are done; so are last frame's releases
    BEAM_T(0);
    // ---- the pruned prefixes that block an extension of a member THIS frame: pruned last frame or earlier, still alive
    //      (a descendant in the beam holds them), parent still in the beam.  N holds last frame's beam and list. ------------
    for (int i = tid; i < nz_prev; i += kBeamThreads) {
      const int np = prev_slot(N.zp[i]);
      if (np >= 0 && __ldcg(&nodes[N.zn[i]].refs) > 0) {
        const int o = atomicAdd(&s_nz2, 1);
        if (o < WB) { C.zn[o] = N.zn[i]; C.zp[o] = np; C.zc[o] = N.zc[i]; } else s_ovf = 1;
      }
    }
    for (int u = tid; u < W_prev; u += kBeamThreads) {
      if (prev_slot(u) >= 0) continue;
      const int sp = N.pslot[u];
      const int np = sp >= 0 ? prev_slot(sp) : -1;
      if (np >= 0 && __ldcg(&nodes[N.node[u]].refs) > 0) {
        const int o = atomicAdd(&s_nz2, 1);
        if (o < WB) { C.zn[o] = N.node[u]; C.zp[o] = np; C.zc[o] = N.last[u]; } else s_ovf = 1;
      }
    }
    __syncthreads();
    BEAM_T(1);
    const int nz = min(s_nz2, WB);
    const int nR = p.prefilter ? s_nR : V - 1;                      // symbols every member is extended with
    const bool use_cache = CACHE && (long long)W * nR <= (long long)p.kc_cap;
    auto sym = [&](int j) -> int { return p.prefilter ? S.rc[j] : j + (j >= p.blank ? 1 : 0); };   // j-th extended symbol
    // ---- phase B: extensions that find a living prefix (:244-246): a member of the beam takes the mass, a pruned prefix
    //      that a descendant keeps alive swallows it ---------------------------------------------------------------------------
    if (tid < W) {
      const int sp = C.pslot[tid];
      if (sp >= 0) {
        const int c = C.last[tid];
        atomicOr(&S.bitmap[sp * VW + (c >> 5)], 1u << (c & 31));
        S.npnb[tid] = beam_lse(S.npnb[tid], BEAM_EXT_VALUE(c, C.last[sp], C.pb[sp], S.full[sp]));
      }
    }
    for (int i = tid; i < nz; i += kBeamThreads) atomicOr(&S.bitmap[C.zp[i] * VW + (C.zc[i] >> 5)], 1u << (C.zc[i] & 31));
    __syncthreads();
    BEAM_T(2);
    // ---- phase C: scores of the members and of the fresh extensions; how many prefixes are there now (:392-399) ------
    if (tid < W) {
      if (BIAS) {   // the member's bias: committed + phi of its automaton node
        const double e = LM ? beam_score_lm(beam_lse(S.npnb[tid], S.npb[tid]), S.lmx[tid], C.nw[tid], p.wip, S.oox[tid])
                            : beam_score(beam_lse(S.npnb[tid], S.npb[tid]), C.nw[tid], p.wip);
        S.mkey[tid] = beam_key(__dadd_rn(e, __dadd_rn(C.bc[tid], __ldg(&z.partial[C.bn[tid]]))));
      }
      else if (LM) S.mkey[tid] = beam_key(beam_score_lm(beam_lse(S.npnb[tid], S.npb[tid]), S.lmx[tid], C.nw[tid], p.wip, S.oox[tid]));
      else S.mkey[tid] = beam_key(beam_score(beam_lse(S.npnb[tid], S.npb[tid]), C.nw[tid], p.wip));
    }
    {
      int excl = 0;
      for (int i = tid; i < W * VW; i += kBeamThreads) excl += __popc(S.bitmap[i] & S.rmask[i % VW]);
      excl = warp_sum(excl);
      if (lane == 0 && excl) atomicAdd(&s_excl, excl);
    }
    if (use_cache) {
      unsigned long long kmax = 0ull, kmin = ~0ull;
      if (tid < W) {
        // members take part in the range as well (mkey is this thread's own value)
        kmax = S.mkey[tid]; kmin = kmax;
      }
      // the warps that hold members have just spent a log-sum-exp (fp64 exp + log) on the member keys: with 16 warps
      // the rows go to the other warps only
      const int mw = kBeamWarps >= 16 ? min((W + 31) >> 5, kBeamWarps - 8) : 0;
            for (int s = warp - mw; s < W && s >= 0; s += kBeamWarps - mw) {
        const int last = C.last[s];
        const double base = S.full[s], baseb = C.pb[s];
        const BeamExt<LM, BIAS> ex(S, s, z);
                      for (int j0 = 0; j0 < nR; j0 += 32) {
          const int j = j0 + lane;
          if (j < nR) {
            const int c = sym(j);
            unsigned long long k = 0ull;
            if (!((S.bitmap[s * VW + (c >> 5)] >> (c & 31)) & 1u)) {
              const double v = BEAM_EXT_VALUE(c, last, baseb, base);
              k = ex.key(v, c, S, p.space, z);
              kmax = k > kmax ? k : kmax; kmin = k < kmin ? k : kmin;
            }
            S.kc[s * nR + j] = k;
          }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long a = __shfl_xor_sync(0xffffffffu, kmax, o), bq = __shfl_xor_sync(0xffffffffu, kmin, o);
        kmax = a > kmax ? a : kmax; kmin = bq < kmin ? bq : kmin;
      }
      if (lane == 0) { atomicMax(&s_kmax, kmax); atomicMin(&s_kmin, kmin); }
    }
    __syncthreads();
    BEAM_T(3);
    const int total = W + W * nR - s_excl;
    // ---- phase D: radix select of the beam_width best (8-bit digits from the highest byte in which the keys differ) -------
    unsigned long long thr = 0ull;
    int sh = 0, need = total;
    bool selected = false;
    if (use_cache && total > WB && kBeamBins == 256 && cut_depth >= 0.0) {
      // Fast path.  Shared-memory atomics retire about one per cycle per SM, so a histogram over all beam x V keys costs
      // as many cycles as there are keys (measured: 5.4k of a 25k-cycle frame on c2).  The cut moves slowly relative to
      // the best score, so only the keys within +-kWin of the PREDICTED cut (best score - last frame's depth) go into a
      // 256-bin histogram (bins by integer key distance: monotone in the score); keys above the window are merely
      // counted (ballots), keys below it ignored; the few keys of the boundary bin are then ranked exactly.  A wrong
      // prediction (cut outside the window, boundary bin too full) falls back to the radix passes below: same result.
      constexpr int kSelCap = 128;                          // 128 keys = the histogram's 1 KB, reused as the list
      constexpr double kWin = 3.0;
      const double smax = beam_unkey(s_kmax);
      const unsigned long long hi_key = beam_key(smax - cut_depth + kWin), lo_key = beam_key(smax - cut_depth - kWin);
      const unsigned long long span = hi_key - lo_key;
      const int bshift = (span >> 8) ? (64 - __clzll((long long)span)) - 8 : 0;
      for (int i = tid; i < 256; i += kBeamThreads) S.hist[i] = 0u;
      if (tid == 0) { s_need = 0; s_done = 0; s_above = 0; }
      __syncthreads();
      if (hi_key > lo_key && lo_key > 1ull) {
        int above = 0;
        if (tid < W) {
          const unsigned long long k = S.mkey[tid];
          if (k > hi_key) above++; else if (k >= lo_key) atomicAdd(&S.hist[(unsigned)((hi_key - k) >> bshift)], 1u);
        }
        for (int i = tid; i < W * nR; i += kBeamThreads) {
          const unsigned long long k = S.kc[i];
          if (k > hi_key) above++; else if (k >= lo_key) atomicAdd(&S.hist[(unsigned)((hi_key - k) >> bshift)], 1u);
        }
        above = warp_sum(above);
        if (lane == 0 && above) atomicAdd(&s_above, above);
      }
      __syncthreads();
      BEAM_T(11);
      if (warp == 0 && s_above < WB && hi_key > lo_key && lo_key > 1ull) {   // the bin that holds the beam_width-th best (bin 0 is the best)
        const unsigned want = (unsigned)(WB - s_above);
        unsigned h[8], mine = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { h[j] = S.hist[lane * 8 + j]; mine += h[j]; }
        unsigned incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += u; }
        const unsigned before = incl - mine;
        if (before < want && incl >= want) {
          unsigned run = before, acc = before, hd = 0; int d = -1;
#pragma unroll
          for (int j = 0; j < 8; j++) {     // first bin of this lane whose running count reaches what is wanted
            if (d < 0 && run + h[j] >= want) { d = j; hd = h[j]; acc = run; }
            run += h[j];
          }
          s_thr = (unsigned long long)(lane * 8 + d);       // boundary bin
          s_need = (int)(want - acc);                        // how many of its keys survive
          s_done = hd <= (unsigned)kSelCap ? 1 : 0;
        }
      }
      __syncthreads();
      BEAM_T(12);
      if (s_done) {
        const unsigned bbin = (unsigned)s_thr; const int bneed = s_need;
        unsigned long long* sel = reinterpret_cast<unsigned long long*>(S.hist);
        __syncthreads();                                    // everybody has read the verdict: the histogram becomes the list
        if (tid == 0) s_above = 0;                          // (now the list length)
        __syncthreads();
        if (tid < W) {
          const unsigned long long k = S.mkey[tid];
          if (k <= hi_key && k >= lo_key && (unsigned)((hi_key - k) >> bshift) == bbin) sel[atomicAdd(&s_above, 1)] = k;
        }
                for (int i = tid; i < W * nR; i += kBeamThreads) {
          const unsigned long long k = S.kc[i];
          if (k <= hi_key && k >= lo_key && (unsigned)((hi_key - k) >> bshift) == bbin) sel[atomicAdd(&s_above, 1)] = k;
        }
        __syncthreads();
        BEAM_T(13);
        const int nsel = s_above;
#ifdef BEAM_PROF
        if (blockIdx.x == 0 && tid == 0) g_beam_prof[15] += nsel;
#endif
        if (tid < nsel) {   // exact rank inside the boundary bin
          const unsigned long long k = sel[tid];
          int gt = 0, eq = 0;
          for (int j = 0; j < nsel; j++) { const unsigned long long o = sel[j]; gt += o > k; eq += o == k; }
          if (gt < bneed && gt + eq >= bneed) {   // the bneed-th largest (threads holding an equal key agree)
            s_thr = k; s_need = bneed - gt;
            if (eq > bneed - gt) s_tie_now = 1;   // equal scores on both sides of the cut
          }
        }
        __syncthreads();
        BEAM_T(14);
        thr = s_thr; sh = 0; need = s_need;
        if (tid == 0 && s_tie_now) { s_ties++; s_tie_now = 0; }
        selected = true;
#ifdef BEAM_PROF
        if (blockIdx.x == 0 && tid == 0) g_beam_prof[9] += 1;
#endif
      }
    }
    if (total > WB && !selected) {
#ifdef BEAM_PROF
      if (blockIdx.x == 0 && tid == 0) g_beam_prof[10] += 1;
#endif
      int remaining = WB;
      unsigned long long prefix = 0ull;
      int sh0 = kBeamTopShift;
      if (use_cache) {
        const unsigned long long diff = s_kmax ^ s_kmin;
        sh0 = diff ? ((63 - __clzll((long long)diff)) / kBeamDigit) * kBeamDigit : 0;
        prefix = sh0 + kBeamDigit >= 64 ? 0ull : (s_kmax & (~0ull << (sh0 + kBeamDigit)));
      }
      for (sh = sh0; sh >= 0; sh -= kBeamDigit) {
        for (int i = tid; i < kBeamBins; i += kBeamThreads) S.hist[i] = 0u;
        __syncthreads();
        const unsigned long long pm = sh + kBeamDigit >= 64 ? 0ull : (~0ull << (sh + kBeamDigit));
        if (tid < W) {
          const unsigned long long k = S.mkey[tid];
          if ((k & pm) == (prefix & pm)) atomicAdd(&S.hist[(unsigned)(k >> sh) & (kBeamBins - 1)], 1u);
        }
        if (use_cache) {
                            for (int i = tid; i < W * nR; i += kBeamThreads) {
            const unsigned long long k = S.kc[i];
            if (k && (k & pm) == (prefix & pm)) atomicAdd(&S.hist[(unsigned)(k >> sh) & (kBeamBins - 1)], 1u);
          }
        } else {
                        for (int s = warp; s < W; s += kBeamWarps) {
            const int last = C.last[s];
            const double base = S.full[s], baseb = C.pb[s];
            const BeamExt<LM, BIAS> ex(S, s, z);
                          for (int j0 = 0; j0 < nR; j0 += 32) {
              const int j = j0 + lane;
              const int c = j < nR ? sym(j) : 0;
              bool valid = j < nR && !((S.bitmap[s * VW + (c >> 5)] >> (c & 31)) & 1u);
              unsigned long long k = 0ull;
              if (valid) {
                const double v = BEAM_EXT_VALUE(c, last, baseb, base);
                k = ex.key(v, c, S, p.space, z);
                valid = (k & pm) == (prefix & pm);
              }
              const unsigned d = (unsigned)(k >> sh) & (kBeamBins - 1);
              const unsigned act = __ballot_sync(0xffffffffu, valid);
              if (valid) {
                const unsigned m = __match_any_sync(act, d);
                if (lane == __ffs(m) - 1) atomicAdd(&S.hist[d], (unsigned)__popc(m));
              }
            }
          }
        }
        __syncthreads();
        if (warp == 0) {                          // the bin that holds the remaining-th largest
          constexpr int BPL = kBeamBins / 32;   // bins per lane
          unsigned h[BPL]; unsigned mine = 0;
#pragma unroll
          for (int j = 0; j < BPL; j++) { h[j] = S.hist[lane * BPL + j]; mine += h[j]; }
          unsigned above = 0;                     // entries in bins of higher lanes
          {
            unsigned v = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned u = __shfl_down_sync(0xffffffffu, v, o); if (lane + o < 32) v += u; }
            above = v - mine;
          }
          const bool here = above < (unsigned)remaining && above + mine >= (unsigned)remaining;
          if (here) {
            unsigned acc = above, hd = h[0]; int d = 0;
#pragma unroll
            for (int j = BPL - 1; j > 0; j--) {     // no dynamic indexing of h[]: it stays in registers
              if (d == 0) { if (acc + h[j] >= (unsigned)remaining) { d = j; hd = h[j]; } else acc += h[j]; }
            }
            s_need = remaining - (int)acc;
            s_thr = prefix | ((unsigned long long)(lane * BPL + d) << sh);
            s_done = (hd == (unsigned)(remaining - (int)acc)) ? 1 : 0;
            if (sh == 0 && !s_done) s_ties++;    // equal scores on both sides of the cut
          }
        }
        __syncthreads();
        prefix = s_thr; remaining = s_need;
        if (s_done || sh == 0) break;
      }
      thr = prefix; need = remaining;
    }
    if (use_cache && total > WB) {   // the prediction for the next frame's fast path
      const double depth = beam_unkey(s_kmax) - beam_unkey(thr > 1ull ? thr : 2ull);
      cut_depth = (depth == depth && depth < 1e300) ? depth : -1.0;
    }
    const unsigned long long tcls = thr >> sh;
    BEAM_T(4);
    // ---- phase E: survivors per position group ---------------------------------------------------------------
    if (tid < W) {
      const unsigned long long kq = S.mkey[tid] >> sh;
      S.cgt[tid] = kq > tcls; S.ceq[tid] = kq == tcls;
    }
        for (int s = warp; s < W; s += kBeamWarps) {
      const int last = C.last[s];
      const double base = S.full[s], baseb = C.pb[s];
      const BeamExt<LM, BIAS> ex(S, s, z);
      int ngt = 0, neq = 0;
            for (int j0 = 0; j0 < nR; j0 += 32) {
        const int j = j0 + lane;
        const int c = j < nR ? sym(j) : 0;
        unsigned long long k = 0ull;
        if (use_cache) { if (j < nR) k = S.kc[s * nR + j]; }
        else if (j < nR && !((S.bitmap[s * VW + (c >> 5)] >> (c & 31)) & 1u)) {
          const double v = BEAM_EXT_VALUE(c, last, baseb, base);
          k = ex.key(v, c, S, p.space, z);
        }
        const unsigned long long kq = k >> sh;
        ngt += __popc(__ballot_sync(0xffffffffu, k != 0ull && kq > tcls));
        neq += __popc(__ballot_sync(0xffffffffu, k != 0ull && kq == tcls));
      }
      if (lane == 0) { S.cgt[W + s] = ngt; S.ceq[W + s] = neq; }
    }
    __syncthreads();
    BEAM_T(5);
    if (warp < 2) {   // exclusive scans over the 2W position groups (members, then member rows): warp 0 the counts above
      int* a = warp == 0 ? S.cgt : S.ceq;   // the cut, warp 1 those in the cut class; the totals go to entry 2W
      int run = 0;
            for (int i0 = 0; i0 < 2 * W; i0 += 32) {
        const int i = i0 + lane;
        const int g = i < 2 * W ? a[i] : 0;
        int sg = g;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, sg, o); if (lane >= o) sg += u; }
        if (i < 2 * W) a[i] = run + sg - g;
        run += __shfl_sync(0xffffffffu, sg, 31);
      }
      if (lane == 0) a[2 * W] = run;
    }
    __syncthreads();
    BEAM_T(6);
    // surviving members = everything before entry W; survivors in all = the totals
    const int keepm = S.cgt[W] + min(S.ceq[W], need), keepall = S.cgt[2 * W] + min(S.ceq[2 * W], need), node0 = n_nodes;
    // slot of member q after this frame's prune, -1 when it leaves the beam
    auto new_slot = [&](int q) -> int {
      const unsigned long long kq = S.mkey[q] >> sh;
      const int eb = S.ceq[q];
      return (kq > tcls || (kq == tcls && eb < need)) ? S.cgt[q] + min(eb, need) : -1;
    };
    // ---- phase F: write the surviving list (next_step, :397) --------------------------------------------------
    if (tid < W) {
      const int s = tid;
      const int ns = new_slot(s);
      if (ns >= 0) {
        N.node[ns] = C.node[s]; N.par[ns] = C.par[s]; N.last[ns] = C.last[s]; N.nw[ns] = C.nw[s]; N.dep[ns] = C.dep[s];
        N.pb[ns] = S.npb[s]; N.pnb[ns] = S.npnb[s];
        const int sp = C.pslot[s];
        N.pslot[ns] = sp >= 0 ? new_slot(sp) : -1;
        if (LM) {
          N.lex[ns] = C.lex[s]; N.cw[ns] = C.cw[s]; N.oov[ns] = C.oov[s]; N.lm[ns] = C.lm[s]; N.sd[ns] = C.sd[s];
#pragma unroll
          for (int i = 0; i < kLMCtx; i++) N.h[i][ns] = C.h[i][s];
        }
        if (BIAS) { N.bn[ns] = C.bn[s]; N.bc[ns] = C.bc[s]; }
      }
    }
        for (int s = warp; s < W; s += kBeamWarps) {
      const int last = C.last[s];
      const double base = S.full[s], baseb = C.pb[s];
      const BeamExt<LM, BIAS> ex(S, s, z);
      int gb = S.cgt[W + s], eb = S.ceq[W + s];
      const int pn = C.node[s], pd = C.dep[s];
      const int psl = new_slot(s);
            for (int j0 = 0; j0 < nR; j0 += 32) {
        const int j = j0 + lane;
        const int c = j < nR ? sym(j) : 0;
        unsigned long long k = 0ull;
        if (use_cache) { if (j < nR) k = S.kc[s * nR + j]; }
        else if (j < nR && !((S.bitmap[s * VW + (c >> 5)] >> (c & 31)) & 1u)) {
          const double v = BEAM_EXT_VALUE(c, last, baseb, base);
          k = ex.key(v, c, S, p.space, z);
        }
        const unsigned long long kq = k >> sh;
        const bool isgt = k != 0ull && kq > tcls, iseq = k != 0ull && kq == tcls;
        const unsigned mg = __ballot_sync(0xffffffffu, isgt), me = __ballot_sync(0xffffffffu, iseq);
        const unsigned below = (1u << lane) - 1u;
        const int g = gb + __popc(mg & below), e = eb + __popc(me & below);
        if (isgt || (iseq && e < need)) {
          const int ns = g + min(e, need);
          const int id = node0 + (ns - keepm);
          N.node[ns] = id; N.par[ns] = pn; N.last[ns] = c; N.dep[ns] = pd + 1; N.pslot[ns] = psl;
          if (LM) { const int kd = S.kind[c]; N.nw[ns] = kd == 0 ? S.nwx[s] : C.nw[s] + (kd == 1 ? 1 : 0); }
          else N.nw[ns] = c == p.space ? C.nw[s] : S.nwx[s];
          N.pb[ns] = -INFINITY; N.pnb[ns] = BEAM_EXT_VALUE(c, last, baseb, base);
          BeamNode r; r.parent = pn; r.chr = c; r.refs = 1; r.depth = pd + 1;
          nodes[id] = r;
          atomicAdd(&nodes[pn].refs, 1);
          if (BIAS) {   // the automaton moves by the label; committed takes what the phrases ending there add
            const int bn = ex.bias_node(c, S);
            N.bn[ns] = bn; N.bc[ns] = S.col[c] < 0 ? ex.com : __dadd_rn(ex.com, __ldg(&z.complete[bn]));
          }
          if (LM) {
            const int cw = C.cw[s];
            if (S.kind[c] != 0) {   // completes the current word, if there is one; the next word starts at the lexicon's root
              const bool done = cw >= 0;
              N.lm[ns] = done ? __dadd_rn(C.lm[s], C.sd[s]) : C.lm[s];
              N.oov[ns] = C.oov[s] + (done && cw == q.unk ? 1 : 0);
#pragma unroll
              for (int i = 0; i < kLMCtx; i++) N.h[i][ns] = done ? (i == kLMCtx - 1 ? cw : C.h[i + 1][s]) : C.h[i][s];
              N.lex[ns] = 0; N.cw[ns] = -1; N.sd[ns] = 0.0;
            } else {                // the word grows; its spelling is walked below, once per new member
              N.lex[ns] = C.lex[s];
              N.lm[ns] = C.lm[s]; N.oov[ns] = C.oov[s];
#pragma unroll
              for (int i = 0; i < kLMCtx; i++) N.h[i][ns] = C.h[i][s];
            }
          }
        }
        gb += __popc(mg); eb += __popc(me);
      }
    }
    __syncthreads();
    if (LM) {   // the new members whose label spells characters: walk the lexicon through them (it stops as soon as no word
                //  is spelled so), then the word a completion would score and its LM term
      for (int ns = keepm + tid; ns < keepall; ns += kBeamThreads) {
        const int c = N.last[ns];
        if (S.kind[c] == 2) continue;
        int lx = N.lex[ns];
        const int i0 = q.label_off ? __ldg(&q.label_off[c]) : c, i1 = q.label_off ? __ldg(&q.label_off[c + 1]) : c + 1;
        for (int i = i0; i < i1 && lx >= 0; i++) lx = __ldg(&q.lex_child[(long long)lx * q.n_chars + __ldg(&q.label_chars[i])]);
        N.lex[ns] = lx;
        int w = lx >= 0 ? __ldg(&q.lex_word[lx]) : -1;
        if (w < 0) w = q.unk;
        N.cw[ns] = w;
        N.sd[ns] = lm_term(q.table, q.mask, q.order, N.h[0][ns], N.h[1][ns], N.h[2][ns], N.h[3][ns], N.h[4][ns], w);
      }
      __syncthreads();
    }
    BEAM_T(7);
    // ---- carried into the next frame: the nodes to release, this frame's cut (slot of a member after the prune) ------
    {
      const int u = tid - kCascOff;
      casc_n = -1;
      if (u >= 0 && u < W && new_slot(u) < 0) { casc_n = C.node[u]; casc_par = C.par[u]; }
    }
    ptcls = tcls; psh = sh; pneed = need; nz_prev = nz; W_prev = W;
    W = keepall; n_nodes = node0 + (keepall - keepm);
    { const BeamBuf tmp = C; C = N; N = tmp; }
  }

  // ---- the n_best best prefixes (:413-419: the reference sorts the final list) and their symbols (get_sentence, :225-239).
  //      Every member ranks itself by counting over the keys: rank = keys above + equal keys at lower positions, so rank 0
  //      is the member the reference's prefixes[0] is when no two scores are equal. ----------------------------------------
  __syncthreads();   // the last frame's tail still reads the member keys
  if (tid < W) {
    if (LM) {   // end of the utterance: a trailing word is completed, then </s> is scored
      const int cw = C.cw[tid];
      const bool done = cw >= 0;
      int h[kLMCtx];
#pragma unroll
      for (int i = 0; i < kLMCtx; i++) h[i] = done ? (i == kLMCtx - 1 ? cw : C.h[i + 1][tid]) : C.h[i][tid];
      double lm = done ? __dadd_rn(C.lm[tid], C.sd[tid]) : C.lm[tid];
      const int oov = C.oov[tid] + (done && cw == q.unk ? 1 : 0);
      lm = __dadd_rn(lm, lm_term(q.table, q.mask, q.order, h[0], h[1], h[2], h[3], h[4], q.eos));
      S.lms[tid] = lm; S.nwx[tid] = oov;
      const double e = beam_score_lm(beam_lse(C.pnb[tid], C.pb[tid]), __dmul_rn(q.lmwt, lm), C.nw[tid], p.wip,
                                     __dmul_rn((double)oov, q.oov_penalty));
      S.mkey[tid] = beam_key(BIAS ? __dadd_rn(e, C.bc[tid]) : e);   // partial credit is withdrawn: committed only
    } else {
      const double e = beam_score(beam_lse(C.pnb[tid], C.pb[tid]), C.nw[tid], p.wip);
      S.mkey[tid] = beam_key(BIAS ? __dadd_rn(e, C.bc[tid]) : e);
    }
  }
  if (tid == 0) s_tie_now = 0;
  __syncthreads();
  const int NB = p.n_best;
  long long* out = p.decoded + (long long)b * NB * p.T;
  if (tid < W) {
    const unsigned long long k = S.mkey[tid];
    int rank = 0, same = 0;
    for (int j = 0; j < W; j++) { const unsigned long long o = S.mkey[j]; rank += o > k || (o == k && j < tid); same += o == k; }
    if (rank < NB) {
      if (same > 1) s_tie_now = 1;                       // the returned list depends on equal final scores
      const int depth = C.dep[tid];
      long long* row = out + (long long)rank * p.T;
      int len;
      if (depth == 0) { row[0] = -1; len = 1; }          // the empty prefix: get_sentence pushes the root's last_char = -1
      else {
        len = depth;
        int n = C.node[tid];
        for (int i = depth - 1; i >= 0; i--) { const BeamNode q = nodes[n]; row[i] = q.chr; n = q.parent; }
      }
      const long long o = (long long)b * NB + rank;
      p.decoded_len[o] = len;
      if (p.scores) {
        const double lp = beam_lse(C.pnb[tid], C.pb[tid]);
        if (LM) {
          const double lm = S.lms[tid];
          const int oov = S.nwx[tid];
          p.scores[o] = beam_score_lm(lp, __dmul_rn(q.lmwt, lm), C.nw[tid], p.wip, __dmul_rn((double)oov, q.oov_penalty));
          q.lm_scores[o] = lm; q.oov_words[o] = oov;
        } else {
          p.scores[o] = beam_score(lp, C.nw[tid], p.wip);
        }
        if (BIAS) { p.scores[o] = __dadd_rn(p.scores[o], C.bc[tid]); z.bias_scores[o] = C.bc[tid]; }
        if (p.log_probs) p.log_probs[o] = lp;
      }
      S.cgt[rank] = len;
    }
  } else if (tid < NB) {                                 // fewer members than asked for: empty slots
    const long long o = (long long)b * NB + tid;
    p.decoded_len[o] = 0;
    if (p.scores) { p.scores[o] = -INFINITY; if (p.log_probs) p.log_probs[o] = -INFINITY; }
    if (LM) { q.lm_scores[o] = -INFINITY; q.oov_words[o] = 0; }
    if (BIAS) z.bias_scores[o] = -INFINITY;
    S.cgt[tid] = 0;
  }
  __syncthreads();
  if (tid == 0 && p.ties) p.ties[b] = s_ovf ? -1 : s_ties + s_tie_now;
  for (int i = tid; i < NB * p.T; i += kBeamThreads) {
    const int r = i / p.T;
    if (i - r * p.T >= S.cgt[r]) out[i] = 0;
  }
}

size_t beam_smem_bytes(int V, int WB, size_t kc_cap, bool lm, bool bias) {
  auto a16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const int VW = (V + 31) >> 5, Vp = (V + 1) & ~1;
  size_t n = 2 * a16(sizeof(double) * Vp);   // lp, raw
  n += 4 * a16(8 * (size_t)WB);        // pb, pnb x 2
  n += 4 * a16(8 * (size_t)WB);        // full, npb, npnb, mkey
  n += 18 * a16(4 * (size_t)WB);       // node, par, last, nw, dep, pslot, zn, zp, zc x 2
  n += a16(4 * (size_t)WB);            // nwx
  n += 2 * a16(4 * (2 * (size_t)WB + 4));    // cgt, ceq (+ the totals)
  n += a16((size_t)4 * WB * VW);
  n += a16(4 * (size_t)kBeamBins) + 2 * a16(8 * (size_t)WB);   // hist, penx, pens
  n += a16(4 * (size_t)V) + a16(4 * (size_t)VW);               // rc, rmask
  n += a16(8 * kc_cap);
  // kind, pen1 (LM), col (BIAS), padded to 128 bytes
  if (lm || bias) n += ((lm ? a16((size_t)V) + a16(8 * (size_t)WB) : 0) + (bias ? a16(4 * (size_t)V) : 0) + 127) & ~(size_t)127;
  if (lm) n += 8 * a16(8 * (size_t)WB) + (2 * (3 + kLMCtx)) * a16(4 * (size_t)WB);   // lm, sd x 2, lmx, lms, oox, oos; lex, cw, oov, h x 2
  if (bias) n += 3 * a16(8 * (size_t)WB) + 3 * a16(4 * (size_t)WB);                   // bc x 2, bcom; bn x 2, bnode
  return n;
}

constexpr size_t kBeamSmemLimit = 200 * 1024;
// How a shape runs: the symbols extended per frame (all, or the beam_width + 2 most probable + the space for large alphabets)
// and how many extension keys are cached in shared memory (0: recomputed in every pass).
struct BeamMode { int prefilter; int kc_cap; size_t smem; bool ok; };
BeamMode beam_mode(int V, int WB, bool lm, bool bias) {
  BeamMode m{0, 0, 0, false};
  const long long all = (long long)V * WB;
  if (all <= kBeamKeyCache) { m.kc_cap = (int)all; }
  else if (V - 1 >= WB + 3) { m.prefilter = 1; m.kc_cap = kBeamKeyCache; }
  m.smem = beam_smem_bytes(V, WB, (size_t)m.kc_cap, lm, bias);
  if (m.smem > kBeamSmemLimit && m.kc_cap) { m.kc_cap = 0; m.smem = beam_smem_bytes(V, WB, 0, lm, bias); }   // no room for the cache
  m.ok = m.smem <= kBeamSmemLimit;
  return m;
}

}  // namespace

size_t beam_workspace_bytes(const e2e_ctc_desc& d, int beam_width) {
  const size_t cap = (size_t)d.max_frames * (size_t)beam_width + 1;
  return (size_t)d.batch * cap * sizeof(BeamNode);
}

bool beam_supported(const e2e_ctc_desc& d, int beam_width, bool lm, bool bias) {
  return beam_width >= 1 && beam_width <= kBeamMaxWidth && beam_mode(d.alphabet, beam_width, lm, bias).ok;
}

size_t ngram_table_bytes(long long slots) { return (size_t)slots * sizeof(NGramEntry); }

int launch_ngram_build(void* table, long long slots, long long count, const int* ids, const int* orders, const double* probs,
                       const double* bows, cudaStream_t s) {
  E2E_CUDA_TRY(cudaMemsetAsync(table, 0, ngram_table_bytes(slots), s));
  if (count > 0) {
    KernelTimer timer(kKernelNGramBuild, s);
    ngram_build_kernel<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(reinterpret_cast<NGramEntry*>(table),
                                                                         (unsigned long long)slots - 1ull, count, ids, orders,
                                                                         probs, bows);
  }
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

static int launch_beam_impl(const e2e_ctc_desc& d, int beam_width, int n_best, int space_idx, double wip, const void* logits,
                            const void* in_len, int64_t* decoded, int64_t* decoded_len, double* scores, double* log_probs,
                            int64_t* ties, char* ws, cudaStream_t s, const BeamLMParams* lmp,
                            const BeamBiasParams* zp) {
  BeamParams p;
  p.logits = logits; p.dtype = d.dtype; p.sb = d.logits_stride_b; p.st = d.logits_stride_t;
  p.in_len = in_len; p.len_is64 = d.lengths_itype == E2E_I64;
  p.decoded = reinterpret_cast<long long*>(decoded); p.decoded_len = reinterpret_cast<long long*>(decoded_len);
  p.scores = scores; p.log_probs = scores ? log_probs : nullptr; p.n_best = n_best;
  p.ties = reinterpret_cast<long long*>(ties);
  p.nodes = reinterpret_cast<BeamNode*>(ws);
  p.node_cap = (long long)d.max_frames * beam_width + 1;
  p.B = d.batch; p.T = d.max_frames; p.V = d.alphabet; p.blank = d.blank_idx; p.beam = beam_width; p.space = space_idx;
  p.from_logits = d.from_logits; p.wip = wip;
  const bool lm = lmp != nullptr;
  BeamLMParams q{};
  if (lm) q = *lmp;
  const bool bias = zp != nullptr;
  BeamBiasParams z{};
  if (bias) z = *zp;
  const BeamMode md = beam_mode(d.alphabet, beam_width, lm, bias);
  static const int no_pref = []() { const char* v = getenv("E2E_CTC_BEAM_NOPREFILTER"); return (v && *v) ? atoi(v) : 0; }();   // tests / experiments
  p.prefilter = no_pref ? 0 : md.prefilter;
  p.kc_cap = (no_pref && md.prefilter) ? 0 : md.kc_cap;
  const bool cache = p.kc_cap > 0;
  const size_t smem = beam_smem_bytes(d.alphabet, beam_width, (size_t)p.kc_cap, lm, bias);
  int dev = 0, sms = 148;
  E2E_CUDA_TRY(cudaGetDevice(&dev));
  E2E_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  static const int force_wide = []() { const char* v = getenv("E2E_CTC_BEAM_WIDE"); return (v && *v) ? atoi(v) : -1; }();   // experiments only
  const bool wide = force_wide >= 0 ? force_wide != 0 : d.batch <= sms;
  KernelTimer timer(bias ? kKernelBeamBias : lm ? kKernelBeamLM : kKernelBeam, s);
#define E2E_K8_(TYPE, CACHE_, NT_, LM_, BIAS_)                                                               \
  do {                                                                                                       \
    E2E_CUDA_TRY(cudaFuncSetAttribute(ctc_beam_kernel<TYPE, CACHE_, NT_, LM_, BIAS_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    ctc_beam_kernel<TYPE, CACHE_, NT_, LM_, BIAS_><<<(unsigned)d.batch, NT_, smem, s>>>(p, q, z);            \
  } while (0)
#define E2E_K8L(TYPE, LM_, BIAS_)                                                                            \
  do {                                                                                                       \
    if (cache) { if (wide) E2E_K8_(TYPE, true, 512, LM_, BIAS_); else E2E_K8_(TYPE, true, 256, LM_, BIAS_); } \
    else { if (wide) E2E_K8_(TYPE, false, 512, LM_, BIAS_); else E2E_K8_(TYPE, false, 256, LM_, BIAS_); }     \
  } while (0)
#define E2E_K8(TYPE)                                                                                         \
  do {                                                                                                       \
    if (bias) { if (lm) E2E_K8L(TYPE, true, true); else E2E_K8L(TYPE, false, true); }                        \
    else { if (lm) E2E_K8L(TYPE, true, false); else E2E_K8L(TYPE, false, false); }                           \
  } while (0)
  switch (d.dtype) {
    case E2E_F32: E2E_K8(float); break;
    case E2E_BF16: E2E_K8(__nv_bfloat16); break;
    case E2E_F16: E2E_K8(__half); break;
    case E2E_F64: E2E_K8(double); break;
    default: set_error("beam: unsupported dtype %d", d.dtype); return E2E_ERR_INVALID_ARGUMENT;
  }
#undef E2E_K8
#undef E2E_K8L
#undef E2E_K8_
#ifdef BEAM_PROF
  {
    long long h[16];
    cudaStreamSynchronize(s);
    cudaMemcpyFromSymbol(h, g_beam_prof, sizeof(h));
    fprintf(stderr, "[beam prof] cycles of CTA 0: head %lld | blocked-list %lld | B %lld | C %lld | select %lld | count %lld | scan %lld | write %lld | tail %lld | fast selects %lld, radix selects %lld | fast path: histogram %lld, boundary %lld, collect %lld, rank %lld, keys in the boundary bins %lld\n", h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7], h[8], h[9], h[10], h[11], h[12], h[13], h[14], h[15]);
    long long z[16] = {0};
    cudaMemcpyToSymbol(g_beam_prof, z, sizeof(z));
  }
#endif
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

int launch_beam(const e2e_ctc_desc& d, int beam_width, int n_best, int space_idx, double wip, const void* logits,
                const void* in_len, int64_t* decoded, int64_t* decoded_len, double* scores, double* log_probs, int64_t* ties,
                char* ws, cudaStream_t s) {
  return launch_beam_impl(d, beam_width, n_best, space_idx, wip, logits, in_len, decoded, decoded_len, scores, log_probs,
                          ties, ws, s, nullptr, nullptr);
}

static BeamLMParams beam_lm_params(const e2e_ctc_ngram& lm, const e2e_ctc_ngram_tokens* tokens, double lmwt,
                                   double oov_penalty, double* lm_scores, int64_t* oov_words) {
  BeamLMParams q;
  q.table = reinterpret_cast<const NGramEntry*>(lm.table); q.mask = (unsigned long long)lm.table_slots - 1ull;
  q.lex_child = lm.lex_child; q.lex_word = lm.lex_word;
  q.label_kind = tokens ? reinterpret_cast<const signed char*>(tokens->label_kind) : nullptr;
  q.label_off = tokens ? tokens->label_off : nullptr;
  q.label_chars = tokens ? tokens->label_chars : lm.label_char;
  q.n_chars = lm.n_chars; q.order = lm.order; q.bos = lm.bos_id; q.eos = lm.eos_id; q.unk = lm.unk_id;
  q.lmwt = lmwt; q.oov_penalty = oov_penalty;
  q.lm_scores = lm_scores; q.oov_words = reinterpret_cast<long long*>(oov_words);
  return q;
}

int launch_beam_lm(const e2e_ctc_desc& d, const e2e_ctc_ngram& lm, const e2e_ctc_ngram_tokens* tokens, int beam_width,
                   int n_best, int space_idx, double wip, double lmwt, double oov_penalty, const void* logits,
                   const void* in_len, int64_t* decoded, int64_t* decoded_len, double* scores, double* log_probs,
                   double* lm_scores, int64_t* oov_words, int64_t* ties, char* ws, cudaStream_t s) {
  const BeamLMParams q = beam_lm_params(lm, tokens, lmwt, oov_penalty, lm_scores, oov_words);
  return launch_beam_impl(d, beam_width, n_best, space_idx, wip, logits, in_len, decoded, decoded_len, scores, log_probs,
                          ties, ws, s, &q, nullptr);
}

int launch_beam_bias(const e2e_ctc_desc& d, const e2e_ctc_ngram* lm, const e2e_ctc_ngram_tokens* tokens,
                     const e2e_ctc_bias& bias, int beam_width, int n_best, int space_idx, double wip, double lmwt,
                     double oov_penalty, const void* logits, const void* in_len, int64_t* decoded, int64_t* decoded_len,
                     double* scores, double* log_probs, double* lm_scores, int64_t* oov_words, double* bias_scores,
                     int64_t* ties, char* ws, cudaStream_t s) {
  BeamBiasParams z;
  z.label_col = bias.label_col; z.next = bias.next; z.partial = bias.partial; z.complete = bias.complete;
  z.n_cols = bias.n_cols; z.bias_scores = bias_scores;
  BeamLMParams q{};
  if (lm) q = beam_lm_params(*lm, tokens, lmwt, oov_penalty, lm_scores, oov_words);
  return launch_beam_impl(d, beam_width, n_best, space_idx, wip, logits, in_len, decoded, decoded_len, scores, log_probs,
                          ties, ws, s, lm ? &q : nullptr, &z);
}

}  // namespace e2e

// K9: CTC log-likelihood of N hypotheses per utterance, forward only (minus the loss of src/losses/ctc_loss.cpp:15-118
// with each hypothesis as the target).  One CTA serves one utterance and kScoreWarps of its hypotheses, one warp per
// hypothesis.  The CTA stages a block of frames once -- normalised once when the input is raw logits -- and every warp
// runs its alpha recursion over the block from shared memory: the rows of an utterance are read ceil(N / kScoreWarps)
// times, not N times, and nothing is stashed for a backward.
//
// Numerics: fp64 log domain with the reference's chained two-argument log-sum-exp (math_utils.h:8-16), the
// same lattice, skip rule and window.  Cell s of a lattice lives in lane s % 32, register s / 32: a warp skips every
// 32-cell group outside the frame's window [max(0, S - 2(T - t)), min(2t + 2, S)), so a short hypothesis costs what
// its own lattice costs, whatever the launch's Lmax.
#include <algorithm>

#include "common.cuh"

namespace e2e {

namespace {

constexpr int kScoreWarps = 8;                 // hypotheses per CTA
constexpr int kScoreMaxFB = 32;                // frames per staged block
constexpr int kScoreSmemBudget = 160 * 1024;   // staging + labels + row statistics
constexpr int kScoreDenseBytes = 64 * 1024;    // dense mode: the block of rows the CTA aims at

struct ScoreParams {
  const void* x;          // logits / log-probs [B, T, V] (element strides sb, st, 1)
  const void* hyps;       // [B * N, Lmax] (row stride hs)
  const void* in_len;     // [B] or null (T)
  const void* hyp_len;    // [B * N]
  double* out;            // [B * N]
  long long sb, st, hs;
  int T, V, Lmax, N, G, blank, from_logits, t_is64, l_is64;
  int dense;              // 1: whole rows staged, indexed by symbol; 0: per warp, blank + the hypothesis's labels
  int FB;                 // frames per staged block
};

struct ScoreMode { int dense, FB; size_t smem; };

__host__ __device__ __forceinline__ size_t a16(size_t x) { return (x + 15) & ~(size_t)15; }

// shared memory: labels [kScoreWarps][Lmax + 1] int | row statistics [kScoreMaxFB][2] double | `extra` bytes (K10's
// label chains and per-warp state) | staged emissions
ScoreMode score_mode(const e2e_ctc_desc& d, size_t extra = 0) {
  ScoreMode m;
  const size_t head = a16((size_t)kScoreWarps * (d.max_targets + 1) * 4) + 2 * kScoreMaxFB * sizeof(double) + extra;
  const size_t row = (size_t)d.alphabet * sizeof(double);
  const size_t fb_dense = std::min<size_t>(kScoreMaxFB, std::max<size_t>(8, kScoreDenseBytes / row));
  if (head + fb_dense * row <= (size_t)kScoreSmemBudget) {
    m.dense = 1;
    m.FB = (int)fb_dense;
    m.smem = head + fb_dense * row;
  } else {
    const size_t frame = (size_t)kScoreWarps * (d.max_targets + 1) * sizeof(double);
    m.dense = 0;
    m.FB = (int)std::min<size_t>(kScoreMaxFB, (kScoreSmemBudget - head) / frame);
    m.smem = head + (size_t)m.FB * frame;
  }
  return m;
}

// the reference's log_sum_exp (math_utils.h:8-16), argument order and -inf rules included
__device__ __forceinline__ double lse2(double a, double b) {
  if (a == -INFINITY) return b;
  if (b == -INFINITY) return a;
  return a > b ? a + log(1.0 + exp(b - a)) : b + log(1.0 + exp(a - b));
}

// max and log sum exp of one row, reduced by one warp
template <typename T>
__device__ __forceinline__ void row_stats(const T* r, int V, int lane, typename Elem<T>::acc_t* m_out,
                                          typename Elem<T>::acc_t* ls_out) {
  using raw_t = typename Elem<T>::acc_t;
  raw_t m = -INFINITY;
  for (int c = lane; c < V; c += 32) { const raw_t v = (raw_t)Elem<T>::load(r + c); m = v > m ? v : m; }
  m = warp_max(m);
  raw_t sum = 0;
  if (sizeof(raw_t) == 8) { for (int c = lane; c < V; c += 32) sum += (raw_t)exp((double)Elem<T>::load(r + c) - (double)m); }
  else { for (int c = lane; c < V; c += 32) sum += (raw_t)expf((float)Elem<T>::load(r + c) - (float)m); }
  sum = warp_sum(sum);
  *m_out = m;
  *ls_out = sizeof(raw_t) == 8 ? (raw_t)log((double)sum) : (raw_t)logf((float)sum);
}

// Stages frames [t0, t0 + nf) of utterance xb for the CTA.  Dense mode: whole rows by symbol, shared by every warp;
// gathered mode: each `gather` warp's blank and labels, frame by frame (row statistics first, for raw logits).  Every
// thread of the CTA calls it; it starts behind a barrier and ends with the block ready for every warp.
template <typename T>
__device__ __forceinline__ void stage_block(const ScoreParams& p, const T* xb, double* E, double* stat, const int* lab,
                                            int L, int Lp, int t0, int nf, int warp, int lane, bool gather) {
  using raw_t = typename Elem<T>::acc_t;
  __syncthreads();                                    // every warp is done with the previous block
  if (p.dense) {
    for (int f = warp; f < nf; f += kScoreWarps) {
      const T* r = xb + (long long)(t0 + f) * p.st;
      double* er = E + (size_t)f * p.V;
      if (p.from_logits) {
        raw_t m, ls;
        row_stats<T>(r, p.V, lane, &m, &ls);
        for (int c = lane; c < p.V; c += 32) er[c] = normalise<T>((raw_t)Elem<T>::load(r + c), m, ls);
      } else {
        for (int c = lane; c < p.V; c += 32) er[c] = (double)Elem<T>::load(r + c);
      }
    }
    __syncthreads();
  } else {
    if (p.from_logits) {
      for (int f = warp; f < nf; f += kScoreWarps) {
        raw_t m, ls;
        row_stats<T>(xb + (long long)(t0 + f) * p.st, p.V, lane, &m, &ls);
        if (lane == 0) { stat[2 * f] = (double)m; stat[2 * f + 1] = (double)ls; }
      }
      __syncthreads();
    }
    if (gather) {                                   // gather blank + this hypothesis's labels, frame by frame
      double* ew = E + (size_t)warp * p.FB * Lp;
      const int w = L + 1;
      for (int i = lane; i < nf * w; i += 32) {
        const int f = i / w, k = i - f * w;
        const raw_t v = (raw_t)Elem<T>::load(xb + (long long)(t0 + f) * p.st + (k ? lab[k - 1] : p.blank));
        ew[f * Lp + k] = p.from_logits ? normalise<T>(v, (raw_t)stat[2 * f], (raw_t)stat[2 * f + 1]) : (double)v;
      }
      __syncwarp();
    }
  }
}

// alpha at frame t from alpha at t - 1 (A in place); e: the frame's staged emissions, indexed by idx
template <int K>
__device__ __forceinline__ void alpha_frame(double (&A)[K], const double* e, const int (&idx)[K], unsigned long long skip,
                                            int t, int Tu, int S, int lane) {
  if (t == 0) {                                       // ctc_loss.cpp:39-41
#pragma unroll
    for (int c = 0; c < K; c++) {
      const int s = c * 32 + lane;
      A[c] = ((s == 0 && (Tu > 1 || S == 1)) || (s == 1 && S > 1)) ? e[idx[c]] : -INFINITY;
    }
    return;
  }
  const int lo = max(0, S - 2 * (Tu - t)), hi = min(2 * t + 2, S);
#pragma unroll
  for (int c = K - 1; c >= 0; c--) {                 // falling c: cell groups read their left neighbours' old values
    if (c * 32 >= hi || c * 32 + 32 <= lo) continue;
    const double a0 = A[c];
    const double pm = c > 0 ? A[c - 1] : -INFINITY;
    const double a1 = __shfl_sync(0xffffffffu, lane == 31 ? pm : a0, (lane + 31) & 31);   // cell s - 1
    const double a2 = __shfl_sync(0xffffffffu, lane >= 30 ? pm : a0, (lane + 30) & 31);   // cell s - 2
    const int s = c * 32 + lane;
    double a = a0;
    if (s > 0) {
      a = lse2(a, a1);
      if ((skip >> c) & 1ull) a = lse2(a, a2);
    }
    A[c] = (s >= lo && s < hi) ? a + e[idx[c]] : -INFINITY;
  }
}

template <typename T, int K>
__global__ void __launch_bounds__(kScoreWarps * 32) ctc_score_kernel(const ScoreParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / p.G;
  const int n = (blockIdx.x - b * p.G) * kScoreWarps + warp;
  const bool live = n < p.N;                          // the last group of an utterance may be partial
  const long long row = (long long)b * p.N + n;
  const int Lp = p.Lmax + 1;
  int* lab = reinterpret_cast<int*>(smem) + warp * Lp;
  double* stat = reinterpret_cast<double*>(smem + a16((size_t)kScoreWarps * Lp * 4));
  double* E = stat + 2 * kScoreMaxFB;
  const T* xb = reinterpret_cast<const T*>(p.x) + (long long)b * p.sb;

  // ---- arguments: out of range gives NaN (the utterance's or the hypothesis's), never an out-of-bounds read ----
  const int Ti = p.in_len ? (int)max(-1LL, min((long long)INT_MAX, load_index(p.in_len, p.l_is64, b))) : p.T;
  const bool bad_utt = Ti < 1 || Ti > p.T;
  const int Tu = bad_utt ? 0 : Ti;                    // every warp of the CTA runs the same frames
  bool bad = false;
  int L = 0;
  if (live) {
    const long long Lr = load_index(p.hyp_len, p.l_is64, row);
    bad = Lr < 0 || Lr > p.Lmax;
    L = bad ? 0 : (int)Lr;
    bool lbad = false;
    for (int k = lane; k < L; k += 32) {
      const long long v = load_index(p.hyps, p.t_is64, row * p.hs + k);
      const bool ok = v >= 0 && v < p.V;
      lab[k] = ok ? (int)v : 0;
      lbad |= !ok;
    }
    bad |= __any_sync(0xffffffffu, lbad);
    if (bad) L = 0;                                   // the lattice runs empty; the result is replaced by NaN
  }
  __syncwarp();
  const int S = 2 * L + 1;
  int idx[K];                                         // the cell's column in the staged rows
  unsigned long long skip = 0ull;                     // bit c: cell c * 32 + lane may be entered from s - 2
  double A[K];
#pragma unroll
  for (int c = 0; c < K; c++) {
    const int s = c * 32 + lane;
    const bool is_lab = (s & 1) && s < S;
    const int sym = is_lab ? lab[s >> 1] : p.blank;
    idx[c] = p.dense ? sym : (is_lab ? (s + 1) >> 1 : 0);
    if (is_lab && s >= 3 && sym != p.blank && sym != lab[(s >> 1) - 1]) skip |= 1ull << c;
    A[c] = -INFINITY;
  }
  const int es = p.dense ? p.V : Lp;                  // doubles per staged frame
  const double* Ew = p.dense ? E : E + (size_t)warp * p.FB * Lp;

  for (int t0 = 0; t0 < Tu; t0 += p.FB) {
    const int nf = min(p.FB, Tu - t0);
    stage_block<T>(p, xb, E, stat, lab, L, Lp, t0, nf, warp, lane, live);
    if (!live) continue;
    for (int f = 0; f < nf; f++) alpha_frame<K>(A, Ew + (size_t)f * es, idx, skip, t0 + f, Tu, S, lane);
  }
  if (!live) return;
  // ---- -loss, ctc_loss.cpp:63-70 ----
  double v1 = -INFINITY, v2 = -INFINITY;
#pragma unroll
  for (int c = 0; c < K; c++) {
    const int s = c * 32 + lane;
    if (s == S - 1) v1 = A[c];
    if (s == S - 2) v2 = A[c];
  }
  v1 = __shfl_sync(0xffffffffu, v1, (S - 1) & 31);
  v2 = __shfl_sync(0xffffffffu, v2, (S - 2) & 31);
  if (lane == 0) p.out[row] = (bad || bad_utt) ? __longlong_as_double(0x7ff8000000000000LL) : (S > 1 ? lse2(v1, v2) : v1);
}


// ------------------------------------------------------------------ K10: the scorer's backward ----------------------
// d score[b, n] / d input: per group of kScoreWarps hypotheses, the occupancies gamma_bn(t, v) scaled by g[b, n] and summed
// into one partial row per (utterance, group, frame); the row kernel below sums the groups and writes the dtype.
//
// One kernel body, three passes chosen at compile time.  K10 runs pass 1 (alpha, checkpoints, log p) and pass 2 (beta,
// g * gamma) in one launch.  MWER splits them at that seam: K12a is pass 1 alone, for every in-list hypothesis, and keeps
// the checkpoints and log p in the loss's state; K12c is pass 2 alone, from that state, with g = w_b * weight[b, n].
enum : int { kPassBoth = 0, kPassAlpha = 1, kPassBeta = 2 };

struct ScoreBwdParams {
  ScoreParams f;
  const double* g;        // [B * N] upstream gradient of the scores (K12c: the MWER weights of K12b)
  const double* utt;      // K12c: [B] upstream gradient of each utterance's loss, w_b
  const unsigned char* mask;   // K12a: [B * N] the slots in the list, or null (all)
  double* logp;           // K12a writes, K12c reads: [B * N] log p of every slot (-inf: masked or infeasible; NaN: bad)
  double* ckpt;           // [B * N][nblk][Kc][32] alpha at the last frame of every staged block; then beta's carry
  double* scr;            // [B * N][FB][Kc][32] one block's alpha, overwritten by g * gamma
  double* part;           // [B][G][T][V] the group's partial rows (frames < T_b)
  double* coef;           // [B * G] sum over the group of g * [score > -inf]; NaN: a bad argument in the group
  int* used;              // [B * G] 1: the group wrote its partial rows
  int Kc, nblk;           // 32-cell groups that cover 2 Lmax + 1 cells; staged blocks of max_frames
};

// K10's shared memory beyond K9's head: label chains [kScoreWarps][Lmax + 1] int | per warp {L, active, coefficient}
size_t bwd_extra(const e2e_ctc_desc& d) { return a16((size_t)kScoreWarps * (d.max_targets + 1) * 4) + kScoreWarps * 16; }

template <typename T, int K, int PASS>
__global__ void __launch_bounds__(kScoreWarps * 32, 1) ctc_score_bwd_kernel(const ScoreBwdParams q) {
  const ScoreParams& p = q.f;
  extern __shared__ __align__(16) unsigned char smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / p.G, grp = blockIdx.x - b * p.G;
  const int n = grp * kScoreWarps + warp;
  const bool live = n < p.N;
  const long long row0 = (long long)b * p.N + grp * kScoreWarps, row = row0 + warp;
  const int Lp = p.Lmax + 1;
  size_t off = a16((size_t)kScoreWarps * Lp * 4);
  int* const lab0 = reinterpret_cast<int*>(smem);
  int* const lab = lab0 + warp * Lp;
  double* const stat = reinterpret_cast<double*>(smem + off);
  off += 2 * kScoreMaxFB * sizeof(double);
  int* const chain0 = reinterpret_cast<int*>(smem + off);
  int* const chain = chain0 + warp * Lp;
  off += a16((size_t)kScoreWarps * Lp * 4);
  int* const wL = reinterpret_cast<int*>(smem + off);
  int* const wAct = wL + kScoreWarps;
  double* const wCf = reinterpret_cast<double*>(wAct + kScoreWarps);
  double* const E = wCf + kScoreWarps;
  const T* xb = reinterpret_cast<const T*>(p.x) + (long long)b * p.sb;

  // ---- arguments, as K9 reads them ----
  const int Ti = p.in_len ? (int)max(-1LL, min((long long)INT_MAX, load_index(p.in_len, p.l_is64, b))) : p.T;
  const bool bad_utt = Ti < 1 || Ti > p.T;
  const int Tu = bad_utt ? 0 : Ti;
  const double gv = !live || PASS == kPassAlpha ? 0.0 : PASS == kPassBeta ? q.utt[b] * q.g[row] : q.g[row];
  const bool in_list = live && (PASS != kPassAlpha || !q.mask || q.mask[row]);
  bool bad = false;
  int L = 0;
  if (live) {
    const long long Lr = load_index(p.hyp_len, p.l_is64, row);
    bad = Lr < 0 || Lr > p.Lmax;
    L = bad ? 0 : (int)Lr;
    bool lbad = false;
    for (int k = lane; k < L; k += 32) {
      const long long v = load_index(p.hyps, p.t_is64, row * p.hs + k);
      const bool ok = v >= 0 && v < p.V;
      lab[k] = ok ? (int)v : 0;
      lbad |= !ok;
    }
    bad |= __any_sync(0xffffffffu, lbad);
    if (bad) L = 0;
  }
  __syncwarp();
  // a zero upstream gradient costs no sweep, and so does a masked-out slot; K12c leaves a NaN weight (a bad utterance)
  // to the coefficient below
  bool act = live && !bad && !bad_utt &&
             (PASS == kPassAlpha ? in_list : gv != 0.0 && (PASS == kPassBoth || gv == gv));
  if (act && PASS != kPassAlpha) {
    // the labels grouped by symbol: chain[k] - 1 is the next position with label lab[k] (-1: none); bit 30 marks the
    // first position of every symbol other than the blank, whose lane sums the chain in position order
    for (int k = lane; k < L; k += 32) {
      const int v = lab[k];
      int nx = -1;
      for (int j = k + 1; j < L; j++) if (lab[j] == v) { nx = j; break; }
      bool head = v != p.blank;
      for (int j = 0; j < k && head; j++) head = lab[j] != v;
      chain[k] = (nx + 1) | (head ? 1 << 30 : 0);
    }
  }
  const int S = 2 * L + 1;
  int idx[K];
  unsigned long long skip = 0ull, bskip = 0ull;        // bskip bit c: cell c * 32 + lane takes beta from s + 2
  double A[K];
#pragma unroll
  for (int c = 0; c < K; c++) {
    const int s = c * 32 + lane;
    const bool is_lab = (s & 1) && s < S;
    const int sym = is_lab ? lab[s >> 1] : p.blank;
    idx[c] = p.dense ? sym : (is_lab ? (s + 1) >> 1 : 0);
    if (is_lab && s >= 3 && sym != p.blank && sym != lab[(s >> 1) - 1]) skip |= 1ull << c;
    // the transpose of alpha's edge s -> s + 2, so that gamma is the derivative of the forward's score
    const int s2 = s + 2;
    if ((s2 & 1) && s2 < S && s2 >= 3) {
      const int sy2 = lab[s2 >> 1];
      if (sy2 != p.blank && sy2 != lab[(s2 >> 1) - 1]) bskip |= 1ull << c;
    }
    A[c] = -INFINITY;
  }
  const int es = p.dense ? p.V : Lp;
  const double* Ew = p.dense ? E : E + (size_t)warp * p.FB * Lp;
  double* const ck = q.ckpt + (size_t)(live ? row : 0) * q.nblk * q.Kc * 32;
  double* const sc = q.scr + (size_t)(live ? row : 0) * p.FB * q.Kc * 32;

  // ---- pass 1: alpha, a checkpoint at the end of every staged block but the last, log p ----
  double logp = -INFINITY;
  if (PASS != kPassBeta && __syncthreads_or(act)) {
    for (int t0 = 0, blk = 0; t0 < Tu; t0 += p.FB, blk++) {
      const int nf = min(p.FB, Tu - t0);
      stage_block<T>(p, xb, E, stat, lab, L, Lp, t0, nf, warp, lane, act);
      if (!act) continue;
      for (int f = 0; f < nf; f++) alpha_frame<K>(A, Ew + (size_t)f * es, idx, skip, t0 + f, Tu, S, lane);
      if (t0 + nf < Tu) {
#pragma unroll
        for (int c = 0; c < K; c++) if (c < q.Kc) ck[((size_t)blk * q.Kc + c) * 32 + lane] = A[c];
      }
    }
    if (act) {
      double v1 = -INFINITY, v2 = -INFINITY;
#pragma unroll
      for (int c = 0; c < K; c++) {
        const int s = c * 32 + lane;
        if (s == S - 1) v1 = A[c];
        if (s == S - 2) v2 = A[c];
      }
      v1 = __shfl_sync(0xffffffffu, v1, (S - 1) & 31);
      v2 = __shfl_sync(0xffffffffu, v2, (S - 2) & 31);
      logp = S > 1 ? lse2(v1, v2) : v1;
      bad |= logp != logp;                            // NaN input
      act = logp > -INFINITY;                         // an infeasible hypothesis contributes exactly 0
    }
  }
  if (PASS == kPassAlpha) {                           // K12a: K9's score of every in-list slot, -inf for the others
    if (live && lane == 0)
      q.logp[row] = bad_utt ? (double)NAN : !in_list ? -INFINITY : bad ? (double)NAN : logp;
    return;
  }
  if (PASS == kPassBeta) {                            // K12c: log p from K12a, through the state
    logp = live ? q.logp[row] : -INFINITY;
    act = act && logp > -INFINITY;
  }
  // K12c: a NaN weight marks a bad utterance; a bad slot with weight 0 is one K12a left out of the list
  const bool nan_cf = PASS == kPassBeta ? gv != gv || (bad && gv != 0.0) : bad;
  if (lane == 0) {
    wL[warp] = L;
    wAct[warp] = act;
    wCf[warp] = !live ? 0.0 : nan_cf ? (double)NAN : act ? gv : 0.0;
  }
  const bool any = __syncthreads_or(act);
  if (threadIdx.x == 0) {
    double c = 0.0;
    for (int w = 0; w < kScoreWarps; w++) c += wCf[w];   // warp order
    q.coef[blockIdx.x] = bad_utt ? (double)NAN : c;
    q.used[blockIdx.x] = any;
  }
  if (!any) return;

  // ---- pass 2, block by block from the last: alpha again from the checkpoint, then beta down the block ----
  // X[c]: beta(t, s) + e_t(s) of the frame above, beta excluding the emission at t (ctc_loss.cpp:72-100)
  const int nb = (Tu + p.FB - 1) / p.FB;
  for (int blk = nb - 1; blk >= 0; blk--) {
    const int t0 = blk * p.FB, nf = min(p.FB, Tu - t0);
    stage_block<T>(p, xb, E, stat, lab, L, Lp, t0, nf, warp, lane, act);
    if (act) {
#pragma unroll
      for (int c = 0; c < K; c++) A[c] = (blk > 0 && c < q.Kc) ? ck[((size_t)(blk - 1) * q.Kc + c) * 32 + lane] : -INFINITY;
      for (int f = 0; f < nf; f++) {
        alpha_frame<K>(A, Ew + (size_t)f * es, idx, skip, t0 + f, Tu, S, lane);
#pragma unroll
        for (int c = 0; c < K; c++) if (c < q.Kc) sc[((size_t)f * q.Kc + c) * 32 + lane] = A[c];
      }
      double X[K];
#pragma unroll
      for (int c = 0; c < K; c++) X[c] = (blk + 1 < nb && c < q.Kc) ? ck[((size_t)(blk + 1) * q.Kc + c) * 32 + lane] : -INFINITY;
      for (int f = nf - 1; f >= 0; f--) {
        const int t = t0 + f;
        const double* e = Ew + (size_t)f * es;
        if (t == Tu - 1) {                            // ctc_loss.cpp:72-74
#pragma unroll
          for (int c = 0; c < K; c++) {
            const int s = c * 32 + lane;
            X[c] = ((s == S - 1 && (Tu > 1 || S == 1)) || (s == S - 2 && S > 1)) ? 0.0 : -INFINITY;
          }
        } else {
          const int lo = max(0, S - 2 * (Tu - t)), hi = min(2 * t + 2, S);
#pragma unroll
          for (int c = 0; c < K; c++) {               // rising c: cell groups read their right neighbours' old values
            if (c * 32 >= hi || c * 32 + 32 <= lo) { X[c] = -INFINITY; continue; }
            const double x0 = X[c];
            const double nx = c + 1 < K ? X[c + 1] : -INFINITY;
            // lanes 0 and 1 hand the next group's cells to lanes 31 and 30, 31
            const double x1 = __shfl_sync(0xffffffffu, lane == 0 ? nx : x0, (lane + 1) & 31);    // cell s + 1
            const double x2 = __shfl_sync(0xffffffffu, lane <= 1 ? nx : x0, (lane + 2) & 31);    // cell s + 2
            const int s = c * 32 + lane;
            double v = x0;
            if (s < S - 1) {
              v = lse2(v, x1);
              if ((bskip >> c) & 1ull) v = lse2(v, x2);
            }
            X[c] = (s >= lo && s < hi) ? v : -INFINITY;
          }
        }
        // g * gamma(t, s) = g * exp(alpha + beta - log p) over the alpha slot; then the carry for frame t - 1
#pragma unroll
        for (int c = 0; c < K; c++) {
          const int s = c * 32 + lane;
          if (c < q.Kc) {
            double* slot = sc + ((size_t)f * q.Kc + c) * 32 + lane;
            *slot = s < S ? gv * exp(*slot + X[c] - logp) : 0.0;
          }
          X[c] += e[idx[c]];
        }
      }
      if (blk > 0) {
#pragma unroll
        for (int c = 0; c < K; c++) if (c < q.Kc) ck[((size_t)blk * q.Kc + c) * 32 + lane] = X[c];
      }
    }
    __syncthreads();                                  // every warp's g * gamma of the block is in scr
    // ---- the block's partial rows: warps over frames, the group's hypotheses summed in warp order ----
    for (int f = warp; f < nf; f += kScoreWarps) {
      double* pr = q.part + (((size_t)b * p.G + grp) * p.T + t0 + f) * p.V;
      for (int v = lane; v < p.V; v += 32) pr[v] = 0.0;
      __syncwarp();
      for (int w = 0; w < kScoreWarps; w++) {
        if (!wAct[w]) continue;
        const int Lw = wL[w], Sw = 2 * Lw + 1;
        const int* lw = lab0 + w * Lp;
        const int* cw = chain0 + w * Lp;
        const double* gw = q.scr + ((size_t)(row0 + w) * p.FB + f) * q.Kc * 32;
        // the blank's column: blank cells and blank-valued labels, lanes over cells, then the warp's fixed tree
        double sb = 0.0;
        for (int s = lane; s < Sw; s += 32) if (!(s & 1) || lw[s >> 1] == p.blank) sb += gw[s];
        sb = warp_sum(sb);
        if (lane == 0) pr[p.blank] += sb;
        for (int k = lane; k < Lw; k += 32) {       // every other symbol: its chain, in position order
          if (!(cw[k] >> 30)) continue;
          double sum = 0.0;
          for (int j = k; j >= 0; j = (cw[j] & 0x3fffffff) - 1) sum += gw[2 * j + 1];
          pr[lw[k]] += sum;
        }
        __syncwarp();
      }
    }
  }
}

struct ScoreRowsParams {
  const void* x;
  const void* in_len;
  const double* part;
  const double* coef;
  const int* used;
  void* grads;
  long long sb, st, gsb, gst;
  int B, T, V, G, from_logits, l_is64;
};

// One warp per (b, t) row: the groups' partial rows summed in group order, minus (sum_n g [finite]) * softmax for raw
// logits; 0 past the utterance's frames; NaN rows for a bad argument (every row when the logits length is bad).
template <typename T>
__global__ void __launch_bounds__(256) ctc_score_rows_kernel(const ScoreRowsParams r) {
  using raw_t = typename Elem<T>::acc_t;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long gr = (long long)blockIdx.x * 8 + warp;
  if (gr >= (long long)r.B * r.T) return;
  const int b = (int)(gr / r.T), t = (int)(gr - (long long)b * r.T);
  const int Ti = r.in_len ? (int)max(-1LL, min((long long)INT_MAX, load_index(r.in_len, r.l_is64, b))) : r.T;
  const bool bad_utt = Ti < 1 || Ti > r.T;
  T* out = reinterpret_cast<T*>(r.grads) + (long long)b * r.gsb + (long long)t * r.gst;
  if (!bad_utt && t >= Ti) {
    for (int v = lane; v < r.V; v += 32) Elem<T>::store(out + v, (raw_t)0);
    return;
  }
  double c = 0.0;
  for (int g = 0; g < r.G; g++) c += r.coef[(size_t)b * r.G + g];
  if (bad_utt || c != c) {
    for (int v = lane; v < r.V; v += 32) Elem<T>::store(out + v, (raw_t)NAN);
    return;
  }
  const T* x = reinterpret_cast<const T*>(r.x) + (long long)b * r.sb + (long long)t * r.st;
  raw_t m = 0, ls = 0;
  if (r.from_logits) row_stats<T>(x, r.V, lane, &m, &ls);
  for (int v = lane; v < r.V; v += 32) {
    double acc = 0.0;
    for (int g = 0; g < r.G; g++)
      if (r.used[(size_t)b * r.G + g]) acc += r.part[(((size_t)b * r.G + g) * r.T + t) * r.V + v];
    if (r.from_logits) acc -= c * exp(normalise<T>((raw_t)Elem<T>::load(x + v), m, ls));
    Elem<T>::store(out + v, (raw_t)acc);
  }
}

// ------------------------------------------------------------------ K12b: MWER weights ------------------------------
// One warp per utterance.  The list U_b: slots in the mask whose score is finite.  p = softmax(lambda s) over U_b (fp64,
// max subtracted), loss_b = R_b = sum_U p r, weight = lambda p (r - R_b) in U_b and 0 elsewhere.  A NaN score or a
// negative / NaN in-list risk: NaN loss and NaN weights for the utterance.  An empty list: loss 0.  Equal in-list risks
// (one slot included): loss = that risk and weights exactly 0.  Lane-strided partial sums, then the butterfly: every
// lane holds the same bits and every run gives them.
struct MwerWeightsParams {
  const double* s;           // [B * N] K12a's scores
  const double* risk;        // [B * N]
  const unsigned char* mask; // [B * N] or null
  double* loss;              // [B]
  double* w;                 // [B * N] lambda p (r - R)
  double* scores;            // [B * N] copy of s for the caller, or null
  double lam;
  int B, N;
};

__global__ void __launch_bounds__(256) ctc_mwer_weights_kernel(const MwerWeightsParams k) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + warp;
  if (b >= k.B) return;
  const size_t r0 = (size_t)b * k.N;
  bool bad = false;
  double mx = -INFINITY, rlo = INFINITY, rhi = -INFINITY;
  for (int n = lane; n < k.N; n += 32) {
    const double s = k.s[r0 + n];
    if (k.scores) k.scores[r0 + n] = s;
    bad |= s != s;
    if ((k.mask && !k.mask[r0 + n]) || !isfinite(s)) continue;
    const double r = k.risk[r0 + n];
    bad |= !(r >= 0.0);
    mx = fmax(mx, __dmul_rn(k.lam, s));
    rlo = fmin(rlo, r);
    rhi = fmax(rhi, r);
  }
  bad = __any_sync(0xffffffffu, bad);
  mx = warp_max(mx);
  rlo = -warp_max(-rlo);
  rhi = warp_max(rhi);
  const bool spread = !bad && rlo < rhi;              // else every weight is 0 (or NaN) and no sum is needed
  double z = 0.0;
  if (spread) {
    for (int n = lane; n < k.N; n += 32) {
      const double s = k.s[r0 + n];
      if ((k.mask && !k.mask[r0 + n]) || !isfinite(s)) continue;
      z += exp(__dmul_rn(k.lam, s) - mx);
    }
    z = warp_sum(z);
  }
  double R = 0.0;
  if (spread) {
    for (int n = lane; n < k.N; n += 32) {
      const double s = k.s[r0 + n];
      if ((k.mask && !k.mask[r0 + n]) || !isfinite(s)) continue;
      R += exp(__dmul_rn(k.lam, s) - mx) / z * k.risk[r0 + n];
    }
    R = warp_sum(R);
  }
  for (int n = lane; n < k.N; n += 32) {
    double w = 0.0;
    const double s = k.s[r0 + n];
    if (bad) w = (double)NAN;
    else if (spread && !(k.mask && !k.mask[r0 + n]) && isfinite(s)) w = k.lam * (exp(__dmul_rn(k.lam, s) - mx) / z) * (k.risk[r0 + n] - R);
    k.w[r0 + n] = w;
  }
  if (lane == 0) k.loss[b] = bad ? (double)NAN : spread ? R : rlo < INFINITY ? rlo : 0.0;
}

struct ScoreBwdLayout {
  ScoreMode md;
  int G, Kc, nblk;
  size_t off_coef, off_used, off_ckpt, off_scr, off_part, total;
  size_t off_logp, off_w, state;   // MWER: the state kept from forward to backward (logp | w | ckpt)
};

size_t align256s(size_t x) { return (x + 255) & ~(size_t)255; }

// false (message set) when a size overflows size_t or a grid exceeds 2^31 - 1 CTAs.  K10: one workspace, coef | used |
// ckpt | scr | part.  MWER: the checkpoints move to the state (logp | w | ckpt) and the workspace keeps the rest.
bool bwd_layout(const e2e_ctc_desc& d, int n_hyp, ScoreBwdLayout* l, bool mwer = false) {
  l->md = score_mode(d, bwd_extra(d));
  l->G = (int)(((long long)n_hyp + kScoreWarps - 1) / kScoreWarps);
  l->Kc = (2 * d.max_targets + 1 + 31) / 32;
  l->nblk = (d.max_frames + l->md.FB - 1) / l->md.FB;
  // K10's grid, B * G CTAs, is at most B * n_hyp <= 2^31 - 1 (check_score); the row kernel's is B * T / 8
  const unsigned long long groups = (unsigned long long)d.batch * l->G;
  const unsigned long long rows_bt = (unsigned long long)d.batch * d.max_frames;
  if ((rows_bt + 7) / 8 > 0x7fffffffULL) {
    set_error("score backward: batch %d x %d frames exceeds the grid (2^31 - 1 CTAs of 8 rows)", d.batch, d.max_frames);
    return false;
  }
  const size_t lane_cells = (size_t)l->Kc * 32 * sizeof(double);
  size_t ckpt, scr, part, a;
  bool ovf = __builtin_mul_overflow((size_t)d.batch * n_hyp, (size_t)l->nblk, &a) || __builtin_mul_overflow(a, lane_cells, &ckpt);
  ovf |= __builtin_mul_overflow((size_t)d.batch * n_hyp, (size_t)l->md.FB, &a) || __builtin_mul_overflow(a, lane_cells, &scr);
  ovf |= __builtin_mul_overflow((size_t)groups, (size_t)d.max_frames, &a) || __builtin_mul_overflow(a, (size_t)d.alphabet, &a) ||
         __builtin_mul_overflow(a, sizeof(double), &part);
  size_t o = 0;
  l->off_logp = l->off_w = l->state = 0;
  if (mwer) {
    const size_t row = align256s((size_t)d.batch * n_hyp * sizeof(double));
    l->off_logp = o; o += row;
    l->off_w = o; o += row;
    l->off_ckpt = o;
    ovf |= __builtin_add_overflow(o, align256s(ckpt), &o) || ckpt > ~(size_t)0 - 255;
    l->state = o;
    o = 0;
  }
  l->off_coef = o; o += align256s(groups * sizeof(double));
  l->off_used = o; o += align256s(groups * sizeof(int));
  if (!mwer) {
    l->off_ckpt = o;
    ovf |= __builtin_add_overflow(o, align256s(ckpt), &o) || ckpt > ~(size_t)0 - 255;
  }
  l->off_scr = o;
  ovf |= __builtin_add_overflow(o, align256s(scr), &o) || scr > ~(size_t)0 - 255;
  l->off_part = o;
  ovf |= __builtin_add_overflow(o, align256s(part), &o) || part > ~(size_t)0 - 255;
  if (ovf) { set_error("score backward: the workspace size overflows size_t"); return false; }
  l->total = o;
  return true;
}

// the lattice kernel's arguments, shared by K10, K12a and K12c; ws / state carved as bwd_layout says
void bwd_params(const e2e_ctc_desc& d, int n_hyp, const ScoreBwdLayout& l, const void* logits, const void* hyps,
                const void* in_len, const void* hyp_len, char* ws, char* state, ScoreBwdParams* q) {
  ScoreParams& p = q->f;
  p.x = logits; p.hyps = hyps; p.in_len = in_len; p.hyp_len = hyp_len; p.out = nullptr;
  p.sb = d.logits_stride_b; p.st = d.logits_stride_t; p.hs = d.targets_stride_b;
  p.T = d.max_frames; p.V = d.alphabet; p.Lmax = d.max_targets; p.N = n_hyp; p.G = l.G;
  p.blank = d.blank_idx; p.from_logits = d.from_logits;
  p.t_is64 = d.targets_itype == E2E_I64; p.l_is64 = d.lengths_itype == E2E_I64;
  p.dense = l.md.dense; p.FB = l.md.FB;
  q->g = nullptr; q->utt = nullptr; q->mask = nullptr; q->logp = nullptr;
  q->coef = ws ? reinterpret_cast<double*>(ws + l.off_coef) : nullptr;
  q->used = ws ? reinterpret_cast<int*>(ws + l.off_used) : nullptr;
  q->scr = ws ? reinterpret_cast<double*>(ws + l.off_scr) : nullptr;
  q->part = ws ? reinterpret_cast<double*>(ws + l.off_part) : nullptr;
  q->ckpt = reinterpret_cast<double*>((state ? state : ws) + l.off_ckpt);
  if (state) {
    q->logp = reinterpret_cast<double*>(state + l.off_logp);
    q->g = reinterpret_cast<const double*>(state + l.off_w);
  }
  q->Kc = l.Kc; q->nblk = l.nblk;
}

// one lattice launch (K10, K12a or K12c), the K variant picked by the longest lattice
template <typename T, int K, int PASS>
int launch_lattice_k(const ScoreBwdLayout& l, const ScoreBwdParams& q, unsigned grid, int kind, cudaStream_t s) {
  E2E_CUDA_TRY(cudaFuncSetAttribute(ctc_score_bwd_kernel<T, K, PASS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.md.smem));
  {
    KernelTimer timer(kind, s);
    ctc_score_bwd_kernel<T, K, PASS><<<grid, kScoreWarps * 32, l.md.smem, s>>>(q);
  }
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

template <typename T, int PASS>
int launch_lattice(const e2e_ctc_desc& d, const ScoreBwdLayout& l, const ScoreBwdParams& q, int kind, cudaStream_t s) {
  const unsigned grid = (unsigned)((long long)d.batch * l.G);
  const int cells = 2 * d.max_targets + 1;
  if (cells <= 32 * 4) return launch_lattice_k<T, 4, PASS>(l, q, grid, kind, s);
  if (cells <= 32 * 8) return launch_lattice_k<T, 8, PASS>(l, q, grid, kind, s);
  if (cells <= 32 * 16) return launch_lattice_k<T, 16, PASS>(l, q, grid, kind, s);
  return launch_lattice_k<T, 40, PASS>(l, q, grid, kind, s);
}

// the row kernel after K10 / K12c: the groups' partial rows in the input's dtype and layout
template <typename T>
int launch_rows(const e2e_ctc_desc& d, const ScoreBwdLayout& l, const ScoreBwdParams& q, void* grads, cudaStream_t s) {
  ScoreRowsParams r;
  r.x = q.f.x; r.in_len = q.f.in_len; r.part = q.part; r.coef = q.coef; r.used = q.used; r.grads = grads;
  r.sb = d.logits_stride_b; r.st = d.logits_stride_t; r.gsb = d.grads_stride_b; r.gst = d.grads_stride_t;
  r.B = d.batch; r.T = d.max_frames; r.V = d.alphabet; r.G = l.G; r.from_logits = d.from_logits; r.l_is64 = q.f.l_is64;
  const unsigned grid_rows = (unsigned)(((long long)d.batch * d.max_frames + 7) / 8);
  {
    KernelTimer timer(kKernelScoreRows, s);
    ctc_score_rows_kernel<T><<<grid_rows, 256, 0, s>>>(r);
  }
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

// the lattice pass PASS and, for K10 / K12c, the row kernel, dispatched on the input dtype
template <int PASS>
int run_passes(const e2e_ctc_desc& d, const ScoreBwdLayout& l, const ScoreBwdParams& q, void* grads, int kind,
               cudaStream_t s, const char* what) {
  int rc;
#define E2E_PASSES(TYPE)                                                      \
  rc = launch_lattice<TYPE, PASS>(d, l, q, kind, s);                         \
  if (rc == E2E_OK && PASS != kPassAlpha) rc = launch_rows<TYPE>(d, l, q, grads, s);
  switch (d.dtype) {
    case E2E_F32: E2E_PASSES(float); break;
    case E2E_BF16: E2E_PASSES(__nv_bfloat16); break;
    case E2E_F16: E2E_PASSES(__half); break;
    case E2E_F64: E2E_PASSES(double); break;
    default: set_error("%s: unsupported dtype %d", what, d.dtype); return E2E_ERR_INVALID_ARGUMENT;
  }
#undef E2E_PASSES
  return rc;
}
}  // namespace
bool score_supported(const e2e_ctc_desc& d) { return score_mode(d).FB >= 1; }

int launch_score(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                 const void* hyp_len, double* scores, cudaStream_t s) {
  const ScoreMode md = score_mode(d);
  ScoreParams p;
  p.x = logits; p.hyps = hyps; p.in_len = in_len; p.hyp_len = hyp_len; p.out = scores;
  p.sb = d.logits_stride_b; p.st = d.logits_stride_t; p.hs = d.targets_stride_b;
  p.T = d.max_frames; p.V = d.alphabet; p.Lmax = d.max_targets; p.N = n_hyp;
  p.G = (n_hyp + kScoreWarps - 1) / kScoreWarps;
  p.blank = d.blank_idx; p.from_logits = d.from_logits;
  p.t_is64 = d.targets_itype == E2E_I64; p.l_is64 = d.lengths_itype == E2E_I64;
  p.dense = md.dense; p.FB = md.FB;
  const long long grid = (long long)d.batch * p.G;
  if (grid > 0x7fffffffLL) { set_error("score: batch x hypothesis groups %lld exceeds the grid", grid); return E2E_ERR_UNSUPPORTED; }
  const int cells = 2 * d.max_targets + 1;
  KernelTimer timer(kKernelScore, s);
#define E2E_K9_(TYPE, K_)                                                                                        \
  do {                                                                                                          \
    E2E_CUDA_TRY(cudaFuncSetAttribute(ctc_score_kernel<TYPE, K_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)md.smem)); \
    ctc_score_kernel<TYPE, K_><<<(unsigned)grid, kScoreWarps * 32, md.smem, s>>>(p);                            \
  } while (0)
#define E2E_K9(TYPE)                                                                                             \
  do {                                                                                                          \
    if (cells <= 32 * 4) E2E_K9_(TYPE, 4);                                                                      \
    else if (cells <= 32 * 8) E2E_K9_(TYPE, 8);                                                                 \
    else if (cells <= 32 * 16) E2E_K9_(TYPE, 16);                                                               \
    else E2E_K9_(TYPE, 40);                                                                                     \
  } while (0)
  switch (d.dtype) {
    case E2E_F32: E2E_K9(float); break;
    case E2E_BF16: E2E_K9(__nv_bfloat16); break;
    case E2E_F16: E2E_K9(__half); break;
    case E2E_F64: E2E_K9(double); break;
    default: set_error("score: unsupported dtype %d", d.dtype); return E2E_ERR_INVALID_ARGUMENT;
  }
#undef E2E_K9
#undef E2E_K9_
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

bool score_backward_supported(const e2e_ctc_desc& d) { return score_mode(d, bwd_extra(d)).FB >= 1; }

size_t score_backward_workspace_bytes(const e2e_ctc_desc& d, int n_hyp) {
  ScoreBwdLayout l;
  return bwd_layout(d, n_hyp, &l) ? l.total : 0;
}

int launch_score_backward(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                          const void* hyp_len, const double* grad_scores, void* grads, char* ws, cudaStream_t s) {
  ScoreBwdLayout l;
  if (!bwd_layout(d, n_hyp, &l)) return E2E_ERR_UNSUPPORTED;
  ScoreBwdParams q;
  bwd_params(d, n_hyp, l, logits, hyps, in_len, hyp_len, ws, nullptr, &q);
  q.g = grad_scores;
  return run_passes<kPassBoth>(d, l, q, grads, kKernelScoreGrad, s, "score backward");
}

size_t mwer_state_bytes(const e2e_ctc_desc& d, int n_hyp) {
  ScoreBwdLayout l;
  return bwd_layout(d, n_hyp, &l, true) ? l.state : 0;
}

size_t mwer_backward_workspace_bytes(const e2e_ctc_desc& d, int n_hyp) {
  ScoreBwdLayout l;
  return bwd_layout(d, n_hyp, &l, true) ? l.total : 0;
}

int launch_mwer_forward(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                        const void* hyp_len, const double* risk, const unsigned char* mask, double score_scale,
                        double* losses, double* scores, char* state, cudaStream_t s) {
  ScoreBwdLayout l;
  if (!bwd_layout(d, n_hyp, &l, true)) return E2E_ERR_UNSUPPORTED;
  ScoreBwdParams q;
  bwd_params(d, n_hyp, l, logits, hyps, in_len, hyp_len, nullptr, state, &q);
  q.mask = mask;
  int rc = run_passes<kPassAlpha>(d, l, q, nullptr, kKernelMwerForward, s, "mwer forward");
  if (rc != E2E_OK) return rc;
  MwerWeightsParams k;
  k.s = q.logp; k.risk = risk; k.mask = mask; k.loss = losses; k.w = const_cast<double*>(q.g); k.scores = scores;
  k.lam = score_scale; k.B = d.batch; k.N = n_hyp;
  {
    KernelTimer timer(kKernelMwerWeights, s);
    ctc_mwer_weights_kernel<<<(unsigned)((d.batch + 7) / 8), 256, 0, s>>>(k);
  }
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

int launch_mwer_backward(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                         const void* hyp_len, const double* utt_scale, void* grads, char* state, char* ws, cudaStream_t s) {
  ScoreBwdLayout l;
  if (!bwd_layout(d, n_hyp, &l, true)) return E2E_ERR_UNSUPPORTED;
  ScoreBwdParams q;
  bwd_params(d, n_hyp, l, logits, hyps, in_len, hyp_len, ws, state, &q);
  q.utt = utt_scale;
  return run_passes<kPassBeta>(d, l, q, grads, kKernelMwerBackward, s, "mwer backward");
}

}  // namespace e2e

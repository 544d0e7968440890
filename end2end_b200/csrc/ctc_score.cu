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

// shared memory: labels [kScoreWarps][Lmax + 1] int | row statistics [kScoreMaxFB][2] double | staged emissions
ScoreMode score_mode(const e2e_ctc_desc& d) {
  ScoreMode m;
  const size_t head = a16((size_t)kScoreWarps * (d.max_targets + 1) * 4) + 2 * kScoreMaxFB * sizeof(double);
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

template <typename T, int K>
__global__ void __launch_bounds__(kScoreWarps * 32) ctc_score_kernel(const ScoreParams p) {
  using raw_t = typename Elem<T>::acc_t;
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
    __syncthreads();                                  // every warp is done with the previous block
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
      if (live) {                                     // gather blank + this hypothesis's labels, frame by frame
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
    if (!live) continue;
    for (int f = 0; f < nf; f++) {
      const int t = t0 + f;
      const double* e = Ew + (size_t)f * es;
      if (t == 0) {                                   // ctc_loss.cpp:39-41
#pragma unroll
        for (int c = 0; c < K; c++) {
          const int s = c * 32 + lane;
          A[c] = ((s == 0 && (Tu > 1 || S == 1)) || (s == 1 && S > 1)) ? e[idx[c]] : -INFINITY;
        }
        continue;
      }
      const int lo = max(0, S - 2 * (Tu - t)), hi = min(2 * t + 2, S);
#pragma unroll
      for (int c = K - 1; c >= 0; c--) {             // falling c: cell groups read their left neighbours' old values
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

}  // namespace e2e

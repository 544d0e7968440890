// K11: exact edit distance of N hypotheses per utterance against the utterance's reference, at token level (every token
// is a unit: CER when tokens are characters) or word level (a word is a maximal run of tokens other than the separator).
// One CTA serves one utterance and kEditWarps of its hypotheses, one warp per hypothesis, as K9 does.  The CTA stages
// the reference row in shared memory once and, at word level, builds the word table once: each word's start, length,
// a 64-bit fingerprint and its canonical index (the first reference word with the same tokens).  A hypothesis word's
// unit is the canonical index of the reference word it equals, -1 when there is none, so the DP compares integers.
// A fingerprint only filters: every equality is confirmed token by token.
//
// The DP runs along the reference: row[j] = min over alignments of hypothesis units [0, i) with reference units [0, j)
// of the key errors * kEditW - substitutions.  kEditW exceeds every substitution count (<= reference units <= 4095),
// so the minimum key is the minimum number of errors and, among those alignments, the most substitutions; insertions
// and deletions then follow from I - D = hypothesis units - reference units.  Lane l holds the contiguous cells
// [l C, l C + C) of the warp's row in shared memory.  Per hypothesis unit the lane takes the diagonal and vertical
// candidates of its cells and the horizontal min(row[j], row[j - 1] + kEditW) within its cells; a 5-step shuffle scan
// of the lanes' min-plus carries and a fix-up pass finish the horizontal recurrence across lanes.  Integer arithmetic
// and no atomics: every run gives the same counts.
#include <climits>

#include "common.cuh"

namespace e2e {

namespace {

constexpr int kEditWarps = 8;                  // hypotheses per CTA
constexpr int kEditW = 4096;                   // key weight of one error: > any substitution count
constexpr int kEditInf = 1 << 30;              // "no carry"; kEditInf + 4096 * kEditW stays below INT_MAX

struct EditParams {
  const void* hyps;       // [B * N, hyp_width] (row stride hs)
  const void* hyp_len;    // [B * N]
  const void* refs;       // [B, ref_width] (row stride rs)
  const void* ref_len;    // [B]
  long long* errors;      // [B * N] each
  long long* subs;
  long long* ins;
  long long* dels;
  long long* ref_units;   // [B]
  long long hs, rs;
  int N, G, hyp_width, ref_width, t_is64, l_is64, sep;
};

__host__ __device__ __forceinline__ size_t a16(size_t x) { return (x + 15) & ~(size_t)15; }

// most words a row of `width` tokens can hold (they are separated by at least one separator)
__host__ __device__ __forceinline__ int max_words(int width) { return (width + 1) / 2; }

// shared memory: reference tokens int64 [ref_width] | word level: fingerprints uint64 [W], canonical indices int64 [W],
// starts int32 [W], lengths int32 [W] (W = max_words) | rows int32 [kEditWarps][C * 32], C = cells per lane
struct EditLayout { size_t off_fp, off_canon, off_start, off_len, off_rows, total; int cells_per_lane; };

__host__ __device__ __forceinline__ EditLayout edit_layout(int ref_width, int words) {
  EditLayout l;
  const int W = words ? max_words(ref_width) : 0;
  size_t o = a16((size_t)ref_width * 8);
  l.off_fp = o;     o = a16(o + (size_t)W * 8);
  l.off_canon = o;  o = a16(o + (size_t)W * 8);
  l.off_start = o;  o = a16(o + (size_t)W * 4);
  l.off_len = o;    o = a16(o + (size_t)W * 4);
  l.off_rows = o;
  l.cells_per_lane = ((words ? W : ref_width) + 1 + 31) / 32;
  l.total = o + (size_t)kEditWarps * l.cells_per_lane * 32 * 4;
  return l;
}

// one token of a word, mixed with its position (splitmix64): the fingerprint of a word is the sum over its tokens, so a
// warp or a thread computes it in any order
__device__ __forceinline__ unsigned long long word_mix(long long tok, int k) {
  unsigned long long z = (unsigned long long)tok + 0x9e3779b97f4a7c15ull * (unsigned long long)(k + 1);
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

__device__ __forceinline__ long long warp_min_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, (long long)__shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// row <- the DP row after hypothesis unit i (1-based) with value hv; m reference units, C cells per lane
__device__ __forceinline__ void dp_step(int* row, const long long* units, int m, int C, int lane, int i, long long hv) {
  const int lo = lane * C, hi = min(lo + C, m + 1);
  int left = (lo >= 1 && lo <= m) ? row[lo - 1] : 0;   // cell lo - 1 of the previous row, read before any lane writes
  __syncwarp();
  int v = kEditInf;
  for (int j = lo; j < hi; ++j) {
    const int up = row[j];
    int x;
    if (j == 0) {
      x = i * kEditW;                                       // i insertions
    } else {
      x = min(left + (hv == units[j - 1] ? 0 : kEditW - 1), up + kEditW);   // match / substitution, insertion
      x = min(x, v + kEditW);                               // deletion, within the lane
    }
    row[j] = x;
    left = up;
    v = x;
  }
  // the lane maps the value of cell lo - 1 to its last cell's: c -> min(a, c + b); compose the lanes in order
  int a = hi > lo ? v : kEditInf, b = hi > lo ? (hi - lo) * kEditW : 0;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int a2 = __shfl_up_sync(0xffffffffu, a, d), b2 = __shfl_up_sync(0xffffffffu, b, d);
    if (lane >= d) { a = min(a, a2 + b); b += b2; }
  }
  int c = __shfl_up_sync(0xffffffffu, a, 1);             // final value of cell lo - 1
  if (lane == 0) c = kEditInf;
  // deletions across the lane boundary; once the carry stops improving a cell it improves none after it
  for (int j = lo; j < hi; ++j) {
    c += kEditW;
    if (c >= row[j]) break;
    row[j] = c;
  }
  __syncwarp();
}

// The words of tokens [0, n) of a row, in order, found 32 tokens at a time by the whole warp (every call is
// warp-uniform): next() gives the next word's [start, end), false past the last one.
struct WordScan {
  int n, next_base = 0, base = 0, start = -1;
  unsigned prev_tok = 0, starts = 0, ev = 0;          // prev_tok: the last token of the loaded chunk is a word token
  template <typename Tok>
  __device__ __forceinline__ bool next(long long sep, int lane, Tok tok, int* s, int* e) {
    for (;;) {
      while (ev) {                                    // a word starts at a token after a non-token and ends at the
        const int k = __ffs(ev) - 1;                  // first non-token after it: a separator or the row's end
        ev &= ev - 1;
        if ((starts >> k) & 1u) { start = base + k; continue; }
        *s = start; *e = base + k;
        return true;
      }
      if (next_base >= n) {                           // a word running to the end of a row of 32 k tokens
        if (!prev_tok) return false;
        prev_tok = 0;
        *s = start; *e = n;
        return true;
      }
      base = next_base;
      next_base += 32;
      const int pos = base + lane;
      const bool is_tok = pos < n && tok(pos) != sep;
      const unsigned tokm = __ballot_sync(0xffffffffu, is_tok);
      const unsigned prevm = (tokm << 1) | prev_tok;
      starts = tokm & ~prevm;
      ev = starts | (~tokm & prevm);
      prev_tok = tokm >> 31;
    }
  }
};

template <bool WORDS>
__global__ void __launch_bounds__(kEditWarps * 32) edit_distance_kernel(const EditParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const EditLayout L = edit_layout(p.ref_width, WORDS);
  long long* rtok = reinterpret_cast<long long*>(smem);
  unsigned long long* wfp = reinterpret_cast<unsigned long long*>(smem + L.off_fp);
  long long* canon = reinterpret_cast<long long*>(smem + L.off_canon);
  int* wstart = reinterpret_cast<int*>(smem + L.off_start);
  int* wlen = reinterpret_cast<int*>(smem + L.off_len);
  __shared__ int s_words;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x / p.G;
  const int g = blockIdx.x - b * p.G;
  const int n = g * kEditWarps + warp;
  const bool live = n < p.N;                              // the last group of an utterance may be partial
  const long long r = (long long)b * p.N + n;

  // ---- arguments: a bad length gives -1 counts (the utterance's or the pair's), never an out-of-bounds read ----
  const long long mr = load_index(p.ref_len, p.l_is64, b);
  const bool bad_ref = mr < 0 || mr > p.ref_width;
  if (bad_ref) {
    if (live && lane == 0) p.errors[r] = p.subs[r] = p.ins[r] = p.dels[r] = -1;
    if (g == 0 && threadIdx.x == 0) p.ref_units[b] = -1;
    return;                                               // uniform over the CTA
  }
  const int mt = (int)mr;
  for (int j = threadIdx.x; j < mt; j += blockDim.x) rtok[j] = load_index(p.refs, p.t_is64, (long long)b * p.rs + j);
  __syncthreads();

  const long long sep = p.sep;
  int m = mt;
  const long long* units = rtok;
  if (WORDS) {
    if (warp == 0) {
      WordScan scan{mt};
      int count = 0, ws, we;
      while (scan.next(sep, lane, [rtok](int k) { return rtok[k]; }, &ws, &we)) {
        if (lane == 0) { wstart[count] = ws; wlen[count] = we - ws; }
        ++count;
      }
      if (lane == 0) s_words = count;
    }
    __syncthreads();
    m = s_words;
    for (int w = threadIdx.x; w < m; w += blockDim.x) {
      unsigned long long f = 0;
      for (int k = 0; k < wlen[w]; ++k) f += word_mix(rtok[wstart[w] + k], k);
      wfp[w] = f;
    }
    __syncthreads();
    for (int w = threadIdx.x; w < m; w += blockDim.x) {
      int c = w;
      for (int v = 0; v < w; ++v) {
        if (wlen[v] != wlen[w] || wfp[v] != wfp[w]) continue;
        bool eq = true;
        for (int k = 0; k < wlen[w] && eq; ++k) eq = rtok[wstart[v] + k] == rtok[wstart[w] + k];
        if (eq) { c = v; break; }
      }
      canon[w] = c;
    }
    __syncthreads();
    units = canon;
  }
  if (g == 0 && threadIdx.x == 0) p.ref_units[b] = m;
  if (!live) return;                                      // no CTA-wide barrier follows

  const long long nr = load_index(p.hyp_len, p.l_is64, r);
  if (nr < 0 || nr > p.hyp_width) {
    if (lane == 0) p.errors[r] = p.subs[r] = p.ins[r] = p.dels[r] = -1;
    return;
  }
  const int nt = (int)nr;
  const long long hbase = r * p.hs;
  const void* hyps = p.hyps;
  const int t64 = p.t_is64;
  auto htok = [hyps, t64, hbase](int k) { return load_index(hyps, t64, hbase + k); };

  const int C = (m + 1 + 31) / 32;
  int* row = reinterpret_cast<int*>(smem + L.off_rows) + warp * L.cells_per_lane * 32;
  for (int j = lane; j <= m; j += 32) row[j] = j * kEditW;   // j deletions
  __syncwarp();

  int i = 0;                                              // hypothesis units so far
  if (WORDS) {
    WordScan scan{nt};
    int ws, we;
    while (scan.next(sep, lane, htok, &ws, &we)) {
      const int len = we - ws;
      unsigned long long f = 0;
      for (int k = lane; k < len; k += 32) f += word_mix(htok(ws + k), k);
      f = warp_sum(f);
      long long id = LLONG_MAX;
      for (int w = lane; w < m; w += 32) {                // canonical words only: at most one matches
        if (canon[w] != w || wlen[w] != len || wfp[w] != f) continue;
        bool eq = true;
        for (int k = 0; k < len && eq; ++k) eq = rtok[wstart[w] + k] == htok(ws + k);
        if (eq) { id = w; break; }
      }
      id = warp_min_ll(id);
      dp_step(row, units, m, C, lane, ++i, id == LLONG_MAX ? -1 : id);
    }
  } else {
    for (int base = 0; base < nt; base += 32) {
      const long long t = base + lane < nt ? htok(base + lane) : 0;
      const int cnt = min(32, nt - base);
      for (int k = 0; k < cnt; ++k) dp_step(row, units, m, C, lane, ++i, __shfl_sync(0xffffffffu, t, k));
    }
  }

  if (lane == 0) {
    const int key = row[m];
    const int e = (key + kEditW - 1) / kEditW;            // key = e * W - S with 0 <= S < W
    const int S = e * kEditW - key;
    const int ID = e - S;                                 // I + D;  I - D = i - m
    p.errors[r] = e;
    p.subs[r] = S;
    p.ins[r] = (ID + i - m) / 2;
    p.dels[r] = (ID - i + m) / 2;
  }
}

}  // namespace

size_t edit_distance_smem_bytes(int ref_width, int words) { return edit_layout(ref_width, words).total; }

int launch_edit_distance(const e2e_ctc_edit_desc& d, const void* hyps, const void* hyp_lengths, const void* refs,
                         const void* ref_lengths, int64_t* errors, int64_t* substitutions, int64_t* insertions,
                         int64_t* deletions, int64_t* reference_units, cudaStream_t s) {
  const int words = d.separator >= 0;
  EditParams p;
  p.hyps = hyps; p.hyp_len = hyp_lengths; p.refs = refs; p.ref_len = ref_lengths;
  p.errors = reinterpret_cast<long long*>(errors); p.subs = reinterpret_cast<long long*>(substitutions);
  p.ins = reinterpret_cast<long long*>(insertions); p.dels = reinterpret_cast<long long*>(deletions);
  p.ref_units = reinterpret_cast<long long*>(reference_units);
  p.hs = d.hyp_stride_b; p.rs = d.ref_stride_b;
  p.N = d.n_hyp; p.G = (d.n_hyp + kEditWarps - 1) / kEditWarps;
  p.hyp_width = d.hyp_width; p.ref_width = d.ref_width;
  p.t_is64 = d.tokens_itype == E2E_I64; p.l_is64 = d.lengths_itype == E2E_I64;
  p.sep = d.separator;
  const long long grid = (long long)d.batch * p.G;
  if (grid > 0x7fffffffLL) { set_error("edit distance: batch x hypothesis groups %lld exceeds the grid", grid); return E2E_ERR_UNSUPPORTED; }
  const size_t smem = edit_layout(d.ref_width, words).total;
  KernelTimer timer(kKernelEdit, s);
  if (words) {
    E2E_CUDA_TRY(cudaFuncSetAttribute(edit_distance_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    edit_distance_kernel<true><<<(unsigned)grid, kEditWarps * 32, smem, s>>>(p);
  } else {
    E2E_CUDA_TRY(cudaFuncSetAttribute(edit_distance_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    edit_distance_kernel<false><<<(unsigned)grid, kEditWarps * 32, smem, s>>>(p);
  }
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

}  // namespace e2e

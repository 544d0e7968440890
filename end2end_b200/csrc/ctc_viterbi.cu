// K6 -- Viterbi forced alignment over the CTC (blank-extended) or ASG (no blank) label lattice.
//
// Replaces pytorch_end2end/utils/alignment.py: _get_alignment_ctc_1d (:50-106), _get_alignment_asg_1d (:9-47) and
// the per-utterance thread fan-out of get_alignment_3d (:109-138) -- SURVEY.md 8(f2).  Same lattice as the loss
// kernels with max instead of sum and a backpointer per cell:
//   alpha[i][k] = max(alpha[i][k-1], alpha[i-1][k-1], [alpha[i-2][k-1] if the label differs from blank and from
//                 the label two cells back]) + lp[k][ext[i]]                                       (fp64, strict >)
// over the reference's window [start, end) of cells that can still reach the end / are reachable from the start;
// cells outside the window stay -inf with a backpointer of 0, as in the reference's zero-initialised path matrix.
// The best path is read back from the last frame (the final label cell wins over the final blank only when it is
// strictly better) and written as label ids [B, T] int64, -100 past the utterance's frames.
//
// Bit-exact by construction: the same fp64 additions of widened fp32 log-probabilities in the same order, the
// same strict comparisons in the same order (stay, then i-1, then i-2), the same window arithmetic.
//
// One CTA per utterance, 1 / 2 / 4 cells per thread (by lattice width): the cells' previous-frame values live in
// registers, the two neighbour cells come from a double-buffered shared-memory row (one __syncthreads per frame),
// emissions are fetched a block of frames ahead (off the dependent chain).  Backpointers are one byte per thread
// per frame (2 bits per cell): in shared memory when the utterance fits, else in the caller's workspace.
//
// Width limit: at most kVitMaxThreads threads of kVitMaxCpt cells, i.e. lattices of <= 2048 cells (CTC: 2 L + 1, so
// L <= 1023; ASG: L <= 2048).  The 4-cells-per-thread instantiations use 105-110 registers a thread, so a CTA of more
// than 576 threads could not launch at all; __launch_bounds__ holds the compiler to what 512 threads allow.
#include "common.cuh"

namespace e2e {
namespace {

struct VitParams {
  const void* lp; int dtype; long long sb, st;
  const void* targets; int tgt_is64; long long ts_b;
  const void* in_len; const void* tgt_len; int len_is64;
  long long* aligned;          // [B, T]
  unsigned char* bp_global;    // [B][T][bp_stride] backpointer bytes (used when the utterance does not fit shared memory)
  int bp_stride;               // bytes per frame = threads per CTA
  int bp_in_smem_frames;       // frames of backpointers that fit the CTA's shared memory (0: always global)
  int B, T, V, Lmax, blank, is_ctc;
  int* status;
};

constexpr long long kIgnore = -100;   // torch.full(..., fill_value=-100) in get_alignment_3d
constexpr int kVitMaxThreads = 512;
constexpr int kVitMaxCpt = 4;

// ET: the type emissions are staged in -- float for 32/16-bit inputs (exact), double for f64 inputs
// CPT: lattice cells per thread (1, 2 or 4).  Few cells per thread = more warps per scheduler to hide the latency of the
// dependent compare/select chain (with 4 cells per thread BASELINE config 2 ran one warp per scheduler at ~1200 cycles per frame).
template <typename ET, int CPT>
__global__ void __launch_bounds__(kVitMaxThreads) ctc_viterbi_kernel(const VitParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  long long* out = p.aligned + (long long)b * p.T;
  const long long Ti_ll = load_index(p.in_len, p.len_is64, b), Li_ll = load_index(p.tgt_len, p.len_is64, b);
  int bad = 0;
  if (Ti_ll < 0 || Ti_ll > p.T) bad |= kBadFrames;
  if (Li_ll < 0 || Li_ll > p.Lmax) bad |= kBadTargetLen;
  const int Ti = bad ? 0 : (int)Ti_ll, Li = bad ? 0 : (int)Li_ll;
  for (int k = Ti + tid; k < p.T; k += nthr) out[k] = kIgnore;
  if (bad) { if (tid == 0) atomicOr(p.status, bad); return; }
  if (Ti == 0) return;                                  // an empty slice: nothing is written (the row stays -100)

  // shared memory: ext labels [S], two alpha rows [S + 2] (two -inf cells in front), backpointer bytes
  const int S = p.is_ctc ? 2 * Li + 1 : Li;
  const int Smax = p.is_ctc ? 2 * p.Lmax + 1 : p.Lmax;
  int* ext = reinterpret_cast<int*>(smem_raw);
  double* row = reinterpret_cast<double*>(smem_raw + (((size_t)(Smax + 4) * 4 + 15) & ~(size_t)15));
  const int rstride = CPT * nthr + 2;
  unsigned char* bp_s = reinterpret_cast<unsigned char*>(row + 2 * rstride);
  const bool bp_smem = Ti <= p.bp_in_smem_frames;
  unsigned char* bp = bp_smem ? bp_s : p.bp_global + (size_t)b * p.T * p.bp_stride;

  __shared__ int s_bad;
  if (tid == 0) s_bad = 0;
  __syncthreads();
  for (int i = tid; i < Smax + 4; i += nthr) ext[i] = p.blank;
  __syncthreads();
  for (int i = tid; i < Li; i += nthr) {
    const long long v = load_index(p.targets, p.tgt_is64, (long long)b * p.ts_b + i);
    if (v < 0 || v >= p.V) { s_bad = kBadLabel; ext[p.is_ctc ? 2 * i + 1 : i] = p.blank; }
    else ext[p.is_ctc ? 2 * i + 1 : i] = (int)v;
  }
  for (int i = tid; i < 2 * rstride; i += nthr) row[i] = -INFINITY;
  __syncthreads();
  if (s_bad) {                                          // a label outside the alphabet: undefined behaviour in the reference
    if (tid == 0) atomicOr(p.status, s_bad);
    for (int k = tid; k < Ti; k += nthr) out[k] = kIgnore;
    return;
  }
  // the reference's early exits (alignment.py:67-73 / :20-22)
  if (S == 0) { for (int k = tid; k < Ti; k += nthr) out[k] = 0; return; }   // ASG with no targets: np.zeros
  if (p.is_ctc && S == 1) { for (int k = tid; k < Ti; k += nthr) out[k] = 0; return; }
  if (Ti == 1) { if (tid == 0) out[0] = p.is_ctc ? ext[1] : ext[0]; return; }

  const int i0 = CPT * tid;
  int lab[CPT]; bool skip_ok[CPT];
#pragma unroll
  for (int c = 0; c < CPT; c++) {
    const int i = i0 + c;
    lab[c] = i < S ? ext[i] : p.blank;
    // alignment.py:90-94: current_label != blank and i - 2 > 0 and extended_targets[i - 2] != current_label
    skip_ok[c] = p.is_ctc && i < S && lab[c] != p.blank && i - 2 > 0 && ext[i - 2] != lab[c];
  }
  const long long xbase = (long long)b * p.sb;
  auto emis = [&](int k, int c) -> ET { return i0 + c < S ? (ET)load_as_double(p.lp, p.dtype, xbase + (long long)k * p.st + lab[c]) : (ET)0; };

  // frame 0 (alignment.py:78-79 / :28)
  double a[CPT];
#pragma unroll
  for (int c = 0; c < CPT; c++) {
    const int i = i0 + c;
    a[c] = (i == 0 || (p.is_ctc && i == 1)) && i < S ? (double)emis(0, c) : -INFINITY;
  }
  double* cur = row + 2;                               // cur[i] = alpha[i][k-1]; cur[-1], cur[-2] = -inf
  double* nxt = row + rstride + 2;
#pragma unroll
  for (int c = 0; c < CPT; c++) cur[i0 + c] = a[c];
  // Emissions are fetched a BLOCK of D frames ahead: the loads of frames k0+D .. k0+2D-1 are issued before frames
  // k0 .. k0+D-1 are swept, so the L2 / HBM latency (several frames' worth of work) never sits on the per-frame chain.
  constexpr int D = sizeof(ET) == 4 ? 8 : 4;
  ET eb[D][CPT], en[D][CPT];
  auto fetch = [&](ET (&dst)[D][CPT], int k0) {
#pragma unroll
    for (int d = 0; d < D; d++)
#pragma unroll
      for (int c = 0; c < CPT; c++) dst[d][c] = k0 + d < Ti ? emis(k0 + d, c) : (ET)0;
  };
  fetch(eb, 1);
  __syncthreads();

  for (int k0 = 1; k0 < Ti; k0 += D) {
    if (k0 + D < Ti) fetch(en, k0 + D);
#pragma unroll
    for (int d = 0; d < D; d++) {
      const int k = k0 + d;
      if (k < Ti) {                                          // uniform over the CTA
        // the window of frame k (alignment.py:81-82 / :30-31)
        const int start = p.is_ctc ? max(0, S - 2 * (Ti - k)) : max(0, S - (Ti - k));
        const int end = p.is_ctc ? min(2 * k + 2, S) : min(k + 1, S);
        const double m1 = cur[i0 - 1], m2 = cur[i0 - 2];
        double pa[CPT + 2];                                 // alpha[i0-2 .. i0+CPT-1][k-1]
        pa[0] = m2; pa[1] = m1;
#pragma unroll
        for (int c = 0; c < CPT; c++) pa[c + 2] = a[c];
        unsigned code = 0;
#pragma unroll
        for (int c = 0; c < CPT; c++) {
          const int i = i0 + c;
          double best = pa[c + 2];
          unsigned cd = 0;
          if (i > 0 && pa[c + 1] > best) { best = pa[c + 1]; cd = 1; }
          if (skip_ok[c] && pa[c] > best) { best = pa[c]; cd = 2; }
          const bool in = i >= start && i < end;
          a[c] = in ? best + (double)eb[d][c] : -INFINITY;
          code |= (in ? cd : 3u) << (2 * c);                 // 3: outside the window -- the reference's path matrix holds 0 there
        }
        bp[(size_t)k * p.bp_stride + tid] = (unsigned char)code;
#pragma unroll
        for (int c = 0; c < CPT; c++) nxt[i0 + c] = a[c];
        __syncthreads();
        double* t = cur; cur = nxt; nxt = t;
      }
    }
#pragma unroll
    for (int d = 0; d < D; d++)
#pragma unroll
      for (int c = 0; c < CPT; c++) eb[d][c] = en[d][c];
  }

  // backtrace (alignment.py:99-104 / :41-45), one thread; global backpointers were written by this CTA: fence first
  __threadfence_block();
  __syncthreads();
  if (tid == 0) {
    int i = S - 1;
    if (p.is_ctc && cur[i - 1] > cur[i]) i = i - 1;
    for (int k = Ti - 1; k >= 0; k--) {
      out[k] = ext[i];
      if (k == 0) break;
      const unsigned code = (bp[(size_t)k * p.bp_stride + i / CPT] >> (2 * (i % CPT))) & 3u;
      i = code == 3 ? 0 : i - (int)code;
    }
  }
}

}  // namespace

static int viterbi_cpt(const e2e_ctc_desc& d, int is_ctc) {
  const int Smax = is_ctc ? 2 * d.max_targets + 1 : d.max_targets;
  return Smax <= 512 ? 1 : (Smax <= 1024 ? 2 : 4);          // up to 16 warps per CTA
}
static int viterbi_threads(const e2e_ctc_desc& d, int is_ctc) {
  const int Smax = is_ctc ? 2 * d.max_targets + 1 : d.max_targets;
  const int cpt = viterbi_cpt(d, is_ctc);
  int thr = (Smax + cpt - 1) / cpt;
  thr = (thr + 31) & ~31;
  return thr < 32 ? 32 : thr;
}

bool viterbi_supported(const e2e_ctc_desc& d, int is_ctc) {
  const long long cells = is_ctc ? 2LL * d.max_targets + 1 : d.max_targets;
  if (cells <= kVitMaxThreads * kVitMaxCpt) return true;
  set_error("viterbi: target length %d exceeds this build's limit %d (%s lattice of at most %d cells)", d.max_targets,
            is_ctc ? (kVitMaxThreads * kVitMaxCpt - 1) / 2 : kVitMaxThreads * kVitMaxCpt, is_ctc ? "CTC" : "ASG",
            kVitMaxThreads * kVitMaxCpt);
  return false;
}

size_t viterbi_workspace_bytes(const e2e_ctc_desc& d, int is_ctc) {
  return 256 + (size_t)d.batch * d.max_frames * viterbi_threads(d, is_ctc);
}

template <typename ET, int CPT>
static int launch_viterbi_k(const VitParams& p, unsigned B, int thr, size_t smem, cudaStream_t s) {
  static int attr_smem[64];
  int dev = 0;
  E2E_CUDA_TRY(cudaGetDevice(&dev));
  if (smem > 48 * 1024 && (dev < 0 || dev >= 64 || (int)smem > attr_smem[dev])) {
    E2E_CUDA_TRY(cudaFuncSetAttribute(ctc_viterbi_kernel<ET, CPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev >= 0 && dev < 64) attr_smem[dev] = (int)smem;
  }
  KernelTimer timer(kKernelViterbi, s);
  ctc_viterbi_kernel<ET, CPT><<<B, thr, smem, s>>>(p);
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

int launch_viterbi(const e2e_ctc_desc& d, int is_ctc, const void* lp, const void* targets, const void* in_len,
                   const void* tgt_len, int64_t* aligned, char* ws, cudaStream_t s) {
  VitParams p;
  p.lp = lp; p.dtype = d.dtype; p.sb = d.logits_stride_b; p.st = d.logits_stride_t;
  p.targets = targets; p.tgt_is64 = d.targets_itype == E2E_I64; p.ts_b = d.targets_stride_b;
  p.in_len = in_len; p.tgt_len = tgt_len; p.len_is64 = d.lengths_itype == E2E_I64;
  p.aligned = reinterpret_cast<long long*>(aligned);
  p.status = reinterpret_cast<int*>(ws);
  p.bp_global = reinterpret_cast<unsigned char*>(ws) + 256;
  p.B = d.batch; p.T = d.max_frames; p.V = d.alphabet; p.Lmax = d.max_targets; p.blank = d.blank_idx; p.is_ctc = is_ctc;
  const int cpt = viterbi_cpt(d, is_ctc), thr = viterbi_threads(d, is_ctc);
  if (!viterbi_supported(d, is_ctc)) return E2E_ERR_UNSUPPORTED;
  p.bp_stride = thr;
  const int Smax = is_ctc ? 2 * d.max_targets + 1 : d.max_targets;
  const size_t fixed = (((size_t)(Smax + 4) * 4 + 15) & ~(size_t)15) + (size_t)2 * (cpt * thr + 2) * 8;
  // backpointers in shared memory when the whole utterance fits (large batches: ~96 KB so that two CTAs share an SM;
  // a batch that cannot fill the SMs anyway may take a whole SM's shared memory), else in the workspace
  const size_t budget = d.batch <= 148 ? 200 * 1024 : 96 * 1024;
  size_t bp_bytes = (size_t)d.max_frames * thr;
  p.bp_in_smem_frames = d.max_frames;
  if (fixed + bp_bytes > budget) { bp_bytes = 0; p.bp_in_smem_frames = 0; }
  const size_t smem = fixed + bp_bytes;
  E2E_CUDA_TRY(cudaMemsetAsync(ws, 0, 256, s));
  const unsigned B = (unsigned)d.batch;
  const bool f64 = d.dtype == E2E_F64;
  if (cpt == 1) return f64 ? launch_viterbi_k<double, 1>(p, B, thr, smem, s) : launch_viterbi_k<float, 1>(p, B, thr, smem, s);
  if (cpt == 2) return f64 ? launch_viterbi_k<double, 2>(p, B, thr, smem, s) : launch_viterbi_k<float, 2>(p, B, thr, smem, s);
  return f64 ? launch_viterbi_k<double, 4>(p, B, thr, smem, s) : launch_viterbi_k<float, 4>(p, B, thr, smem, s);
}

}  // namespace e2e

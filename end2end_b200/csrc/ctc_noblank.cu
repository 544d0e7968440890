// K7 -- CTC without blank (SURVEY.md 8(f4)): loss and gradient of the blank-free lattice.
//
// Replaces pytorch_end2end/functions/ctc_without_blank.py: _ctc_without_blank_loss (:13-88) and the per-utterance
// thread fan-out _ctc_without_blank_3d_loss (:91-117).  The lattice has one cell per target label (plus, with a
// `space_idx`, one optional space cell at either end); a cell is reached from itself or from the cell before it:
//   alpha[j][t] = lse(alpha[j][t-1], alpha[j-1][t-1]) + lp[t][ext[j]]            (:49-58, the reference's window)
//   beta[j][t]  = lse(beta[j][t+1] + lp[t+1][ext[j]], beta[j+1][t+1] + lp[t+1][ext[j+1]])              (:67-79)
//   grad[t][v]  = exp(lp[t][v]) - sum_{j: ext[j]=v} exp(alpha[j][t] + beta[j][t] - logZ),  0 past the frames (:81-88,:113)
// fp64 log-space with the reference's two-argument log-sum-exp (functions/utils.py:6-24), like the reference.
//
// One CTA per utterance, one thread per lattice cell and sweep: the first half of the CTA sweeps alpha forward while
// the second half sweeps beta backward (one __syncthreads per frame for both), rows go to the workspace; then the
// warps take frames round-robin and write the gradient rows -- a symbol's cells are summed in lattice order from a
// counting-sort list built once (fixed order: bitwise reproducible, no atomics).
#include "common.cuh"

namespace e2e {
namespace {

struct NbParams {
  const void* lp; int dtype; long long sb, st;
  void* grads; long long gsb, gst;
  const void* targets; int tgt_is64; long long ts_b;
  const void* in_len; const void* tgt_len; int len_is64;
  void* losses;
  double* alpha; double* beta;    // [B][T][Smax]
  int* status;
  int B, T, V, Lmax, Smax, space, cells_thr;   // cells_thr: threads per sweep
};

__device__ __forceinline__ double nb_lse2(double a, double b) {
  if (a == -INFINITY) return b;
  if (b == -INFINITY) return a;
  if (a > b) return a + log(1.0 + exp(b - a));
  return b + log(1.0 + exp(a - b));
}

__global__ void ctc_noblank_kernel(const NbParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int b = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
  const int CT = p.cells_thr;
  // shared: ext[Smax], order[Smax] (cells grouped by symbol), ofs[V+1], two double-buffered rows per sweep
  int* ext = reinterpret_cast<int*>(smem_raw);
  int* order = ext + p.Smax + 1;
  int* ofs = order + p.Smax + 1;
  double* rows = reinterpret_cast<double*>(smem_raw + ((((size_t)(2 * p.Smax + 2 + p.V + 2)) * 4 + 15) & ~(size_t)15));
  const int rs = CT + 2;   // row stride: one -inf cell on either side
  __shared__ int s_bad;
  __shared__ double s_logz;

  const long long Ti_ll = load_index(p.in_len, p.len_is64, b), Li_ll = load_index(p.tgt_len, p.len_is64, b);
  int bad = 0;
  if (Ti_ll < 1 || Ti_ll > p.T) bad |= kBadFrames;
  if (Li_ll < 0 || Li_ll > p.Lmax) bad |= kBadTargetLen;
  const int Ti = (int)Ti_ll, Li = bad ? 0 : (int)Li_ll;
  if (tid == 0) s_bad = 0;
  __syncthreads();
  // extended targets (:26-38)
  const long long first = Li > 0 ? load_index(p.targets, p.tgt_is64, (long long)b * p.ts_b) : -1;
  const int space = p.space;
  bool uas = false;
  int S;
  if (Li == 0 || (Li == 1 && first == space)) { S = 1; }
  else if (space == -1) { S = Li; }
  else { uas = true; S = Li + 2; }
  for (int j = tid; j < S; j += nthr) {
    long long v;
    if (S == 1 && !(Li >= 1 && space == -1)) v = space;
    else if (!uas) v = load_index(p.targets, p.tgt_is64, (long long)b * p.ts_b + j);
    else v = (j == 0 || j == S - 1) ? space : load_index(p.targets, p.tgt_is64, (long long)b * p.ts_b + j - 1);
    if (v == -1) v = p.V - 1;                      // numpy's negative index of the reference: the last symbol
    if (v < 0 || v >= p.V) { s_bad = kBadLabel; v = 0; }
    ext[j] = (int)v;
  }
  __syncthreads();
  bad |= s_bad;
  const long long gbase = (long long)b * p.gsb;
  if (bad) {   // undefined behaviour in the reference: NaN loss, NaN gradient block, status bits
    if (tid == 0) { atomicOr(p.status, bad); store_from_double(p.losses, p.dtype, b, (double)NAN); }
    for (long long k = tid; k < (long long)p.T * p.V; k += nthr) store_from_double(p.grads, p.dtype, gbase + (k / p.V) * p.gst + k % p.V, (double)NAN);
    return;
  }
  // cells grouped by symbol (counting sort, one warp): symbol v owns order[ofs[v] .. ofs[v+1])
  if (tid < 32) {
    int base = 0;
    for (int v0 = 0; v0 < p.V; v0 += 32) {
      const int v = v0 + tid;
      int c = 0;
      if (v < p.V) for (int j = 0; j < S; j++) c += (ext[j] == v);
      int inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (tid >= o) inc += t; }
      int k = base + inc - c;
      if (v < p.V) { ofs[v] = k; for (int j = 0; j < S; j++) if (ext[j] == v) order[k++] = j; }
      base += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (tid == 0) ofs[p.V] = base;
  }
  for (int k = tid; k < 4 * rs; k += nthr) rows[k] = -INFINITY;
  __syncthreads();

  const long long xbase = (long long)b * p.sb;
  auto lp_at = [&](int t, int sym) -> double { return load_as_double(p.lp, p.dtype, xbase + (long long)t * p.st + sym); };
  double* A = p.alpha + (size_t)b * p.T * p.Smax;
  double* Bt = p.beta + (size_t)b * p.T * p.Smax;

  // ---- the two sweeps: threads [0, CT) alpha forward, [CT, 2 CT) beta backward (sequentially when the CTA has CT threads) ----
  const int teams = nthr / CT;
  for (int pass = 0; pass < 2 / teams; pass++) {
    const int team = teams == 2 ? tid / CT : pass;
    const int j = tid % CT;
    const bool fwd = team == 0;
    double* r0 = rows + (size_t)(2 * team) * rs + 1;      // r0[-1] and r0[CT] stay -inf
    double* r1 = r0 + rs;
    const int sym = j < S ? ext[j] : 0;
    const int sym_next = j + 1 < S ? ext[j + 1] : 0;
    double cur = -INFINITY;
    if (j < S) {
      if (fwd) {     // :42-45
        if ((Ti > 1 || S == 1) && j == 0) cur = lp_at(0, sym);
        if (S > 1 && uas && j == 1) cur = lp_at(0, sym);
      } else {       // :63-66
        if ((Ti > 1 || S == 1) && j == S - 1) cur = 0.0;
        if (S > 1 && uas && j == S - 2) cur = 0.0;
      }
      (fwd ? A : Bt)[(size_t)(fwd ? 0 : Ti - 1) * p.Smax + j] = cur;
    }
    r0[j] = cur;
    __syncthreads();
    for (int i = 1; i < Ti; i++) {
      const int t = fwd ? i : Ti - 1 - i;
      const int start = uas ? max(0, S - Ti + t - 1) : max(0, S - Ti + t);
      const int end = uas ? min(t + 2, S) : min(t + 1, S);
      double nv = -INFINITY;
      if (j >= start && j < end) {
        if (fwd) {   // :52-58
          nv = cur;
          if (j > 0) nv = nb_lse2(nv, r0[j - 1]);
          nv += lp_at(t, sym);
        } else {     // :72-79
          nv = cur + lp_at(t + 1, sym);
          if (j < S - 1) nv = nb_lse2(nv, r0[j + 1] + lp_at(t + 1, sym_next));
        }
      }
      cur = nv;
      if (j < S) (fwd ? A : Bt)[(size_t)t * p.Smax + j] = cur;
      r1[j] = cur;
      __syncthreads();
      double* tmp = r0; r0 = r1; r1 = tmp;
    }
    if (fwd && j == 0) {   // loss_forward (:59-63): r0 holds alpha[.][T-1]
      s_logz = (S > 1 && uas) ? nb_lse2(r0[S - 1], r0[S - 2]) : r0[S - 1];
    }
    __syncthreads();
  }
  const double logz = s_logz;
  if (tid == 0) store_from_double(p.losses, p.dtype, b, -logz);
  __threadfence_block();
  __syncthreads();

  // ---- gradient rows: warps over frames, lanes over symbols; frames past T_i are zero (:113, np.zeros_like) ----
  const int w = tid >> 5, lane = tid & 31, nw = nthr >> 5;
  for (int t = w; t < p.T; t += nw) {
    const long long go = gbase + (long long)t * p.gst;
    if (t >= Ti) { for (int v = lane; v < p.V; v += 32) store_from_double(p.grads, p.dtype, go + v, 0.0); continue; }
    const double* at = A + (size_t)t * p.Smax;
    const double* bt = Bt + (size_t)t * p.Smax;
    for (int v = lane; v < p.V; v += 32) {
      double post = 0.0;
      bool any = false;
      for (int k = ofs[v]; k < ofs[v + 1]; k++) {
        const int j = order[k];
        const double ab = at[j] + bt[j];
        // exp(lse_j(ab_j) - logZ) of the reference, summed in the linear domain; -inf - (-inf) = NaN as there
        post += exp(ab - logz);
        any = true;
      }
      if (!any) post = exp(-INFINITY - logz);            // no cell carries this symbol: exp(-inf - logZ) = 0 (NaN when logZ = -inf)
      // the reference exponentiates the float32 log-probabilities in float32 (np.exp of a float32 array, :87)
      const double first = p.dtype == E2E_F64 ? exp(lp_at(t, v)) : (double)expf((float)lp_at(t, v));
      store_from_double(p.grads, p.dtype, go + v, first - post);
    }
  }
}

}  // namespace

static int noblank_cells(const e2e_ctc_desc& d) { return d.max_targets + 2; }
static int noblank_cells_thr(const e2e_ctc_desc& d) { return (noblank_cells(d) + 31) & ~31; }
static size_t noblank_smem(const e2e_ctc_desc& d) {
  return ((((size_t)(2 * noblank_cells(d) + 2 + d.alphabet + 2)) * 4 + 15) & ~(size_t)15) +
         (size_t)4 * (noblank_cells_thr(d) + 2) * sizeof(double);
}

// One thread per lattice cell and sweep in one CTA: Lmax + 2 <= 1024 cells (Lmax <= 1022); the labels, the symbol
// lists and the sweep rows share one CTA's shared memory (200 KB).
bool noblank_supported(const e2e_ctc_desc& d) {
  if (d.max_targets > 1022) {
    set_error("ctc_without_blank: target length %d exceeds this build's limit 1022", d.max_targets);
    return false;
  }
  if (noblank_smem(d) > 200 * 1024) {
    set_error("ctc_without_blank: alphabet %d too large for one CTA's shared memory", d.alphabet);
    return false;
  }
  return true;
}

size_t noblank_workspace_bytes(const e2e_ctc_desc& d) {
  return 256 + (size_t)2 * d.batch * d.max_frames * noblank_cells(d) * sizeof(double);
}

int launch_noblank(const e2e_ctc_desc& d, int space_idx, const void* lp, const void* targets, const void* in_len,
                   const void* tgt_len, void* losses, void* grads, char* ws, cudaStream_t s) {
  NbParams p;
  p.lp = lp; p.dtype = d.dtype; p.sb = d.logits_stride_b; p.st = d.logits_stride_t;
  p.grads = grads; p.gsb = d.grads_stride_b; p.gst = d.grads_stride_t;
  p.targets = targets; p.tgt_is64 = d.targets_itype == E2E_I64; p.ts_b = d.targets_stride_b;
  p.in_len = in_len; p.tgt_len = tgt_len; p.len_is64 = d.lengths_itype == E2E_I64;
  p.losses = losses;
  p.B = d.batch; p.T = d.max_frames; p.V = d.alphabet; p.Lmax = d.max_targets; p.Smax = noblank_cells(d); p.space = space_idx;
  p.status = reinterpret_cast<int*>(ws);
  p.alpha = reinterpret_cast<double*>(ws + 256);
  p.beta = p.alpha + (size_t)d.batch * d.max_frames * p.Smax;
  if (!noblank_supported(d)) return E2E_ERR_UNSUPPORTED;
  const int ct = noblank_cells_thr(d);
  p.cells_thr = ct;
  const int threads = 2 * ct <= 1024 ? 2 * ct : ct;
  const size_t smem = noblank_smem(d);
  static int attr_smem[64];
  int dev = 0;
  E2E_CUDA_TRY(cudaGetDevice(&dev));
  if (smem > 48 * 1024 && (dev < 0 || dev >= 64 || (int)smem > attr_smem[dev])) {
    E2E_CUDA_TRY(cudaFuncSetAttribute(ctc_noblank_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (dev >= 0 && dev < 64) attr_smem[dev] = (int)smem;
  }
  E2E_CUDA_TRY(cudaMemsetAsync(ws, 0, 256, s));
  KernelTimer timer(kKernelNoBlank, s);
  ctc_noblank_kernel<<<(unsigned)d.batch, threads, smem, s>>>(p);
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

}  // namespace e2e

// Shared device/host helpers for the sm_100a CTC kernels.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/e2e_ctc.h"

namespace e2e {

// ------------------------------------------------------------------ lattice kernel plan -------
constexpr int kDenseMaxAlphabet = 128; // fused ("dense") mode stages whole rows by symbol
constexpr int kNegExp = -(1 << 28);    // block exponent of an all-zero block

constexpr int kNumChunks = 4;          // emission / state ring depth, in chunks of 2^chunk_log2 frames
constexpr int kMaxCombinerWarps = 4;
constexpr int kMaxProducerWarps = 4;
constexpr int kMaxCellsPerLane = 40;
constexpr int kMaxLatticeWarps = 4;    // lattice warps per sweep

// shared-memory layout of the one-warp-per-sweep lattice kernel (ctc_sweep_impl.cuh), bytes
struct SweepLayout {
  int cf, es, rawrow, vpad;
  int off_lab, off_warp, warp_bytes, w_E, w_raw, w_stat, w_rs, w_acc, w_stage;
};

// sweep kernel, narrow variants (K < 24 cells per lane): stashed rows each warp keeps in flight, and the resident CTAs
// per SM the register allocation aims at (-D overrides are for experiments)
#ifndef E2E_SWEEP_PF_SMALL
#define E2E_SWEEP_PF_SMALL 4
#endif
#ifndef E2E_SWEEP_MINBLK
#define E2E_SWEEP_MINBLK 7
#endif
#ifndef E2E_SWEEP_WIDE_MINBLK
#define E2E_SWEEP_WIDE_MINBLK 1
#endif
#ifndef E2E_SWEEP_PF_WIDE
#define E2E_SWEEP_PF_WIDE 2
#endif
constexpr int kSweepPFSmall = E2E_SWEEP_PF_SMALL;
constexpr int kSweepPFWide = E2E_SWEEP_PF_WIDE;

constexpr int kWaveCF = 8;       // wave kernel: frames per hand-off chunk
constexpr int kWaveRB = 32;      // boundary-slot ring depth (frames)
constexpr int kWavePF = 4;       // stashed rows each combiner warp keeps in flight
// combiner warps of the wave kernel: a compile-time count, so that the lattice warps' ring check is straight-line code
__host__ __device__ constexpr int wave_combiners(int NW) { return NW >= 4 ? 6 : 2; }
// shared-memory layout and role counts of the wave kernel (ctc_wave_impl.cuh)
struct WaveLayout {
  int K, NW;        // cells per lane, lattice warps per sweep
  int NP, NC;       // producer (row log-softmax) warps, combiner warps (wave_combiners(NW))
  int by_smsp;      // lay the roles out by SM sub-partition (warp id % 4): latency configurations
  int nwarps;       // warps per CTA
  int nap;          // nanoseconds a waiting producer / combiner warp sleeps between polls (0: spin)
  int R, RV;        // frames in the emission ring / in the val ring (powers of two)
  int ecs;          // the emission ring is column-major (V symbols, a zero column, the row normaliser): doubles per
                    // column, R + 1 (odd: the combiners' symbol-per-lane reads spread over the banks)
  int vpad;         // u32 posterior accumulators per combiner warp
  int off_lab, off_occ, off_E, off_valw, off_vale, off_stage, off_acc, off_bnd, off_ctl, total;
};

// shared-memory layout and role map of the general lattice kernel (ctc_fused_impl.cuh), computed once on the host
struct FzLayout {
  int NB;          // kernel class: block rows (of four cells) per lane the kernel is instantiated for: 1, 2, 4, 10
  int gather;      // 1: emissions gathered by label + compact posteriors for K3; 0: dense rows, gradient written in-kernel
  int NP, NC, PF;  // producer warps, combiner warps, stashed rows each combiner keeps in flight (2 or 4)
  int nwarps;      // warps per CTA
  int nap;         // nanoseconds a waiting producer / combiner sleeps between polls
  int R, RV, CF;   // frames in the emission ring / the val ring (powers of two), frames per ring check
  int rv_log2, neb_log2, neb_mask;   // log2(RV); emission-ring blocks R / PB: log2 and mask
  int dbg;         // debugging switches (FZ_DBG builds only)
  int PB, pb_log2; // frames per producer block
  int es;          // doubles per emission-ring frame
  int vframe;      // bytes per val-ring frame
  int srow;        // bytes per staged stash row
  int prow;        // floats per combiner posterior row
  int off_lab, off_occ, off_E, off_val, off_stage, off_post, off_ctl, total;
  signed char role[16];   // per warp: 0 lattice, 1 combiner, 2 producer, 3 idle, 4 scaler
  signed char ridx[16];   // index within the role
};

// One forward call leaves everything the backward needs in the caller's workspace.  Three lattice kernels share
// the plan: kind 0 the general kernel (ctc_fused_impl.cuh: every shape), kind 1 the wave kernel (latency shapes,
// small alphabets), kind 2 the one-warp-per-sweep kernel (throughput shapes).
enum { kPlanFused = 0, kPlanWave = 1, kPlanSweep = 2 };
struct LossPlan {
  int kind;
  FzLayout fz;
  WaveLayout wv;
  SweepLayout sw;
  int K, NW;        // wave / sweep: cells per lane, lattice warps per sweep
  int dense;        // fused mode: log-softmax + gradient write inside the lattice kernel (alphabet <= kDenseMaxAlphabet)
  int cells;        // lattice cells the kernel variant covers (>= 2*Lmax+1)
  int post_stride;  // floats per frame of the compact posterior rows (gather mode): cells/2 labels + blank total
  int roww;         // general kernel: u32 words per stash row (4 cell words + 1 exponent per block, 32*NB blocks)
  int words;        // sweep: u32 words per lane per frame in the stash rows
  int vpad;
  size_t smem;      // dynamic shared memory of the lattice kernel
  // byte offsets into the workspace
  size_t off_status, off_meet, off_flags, off_stats, off_stash, off_post, off_emis, total;
  size_t off_order; // sweep, multi-wave batches of wide lattices: utterance indices by falling frame count (0: launch in index order)
  int emis_stride;  // general kernel, gather mode: doubles per frame of the compact emission rows K1 writes (0: none)
};

// fused: the caller wants loss + gradient in one pass (dense mode is used when the alphabet allows it)
bool make_loss_plan(const e2e_ctc_desc& d, bool fused, LossPlan* p);

// status word bits (device-side argument check)
constexpr int kBadFrames = 1, kBadTargetLen = 2, kBadLabel = 4;
// per-utterance flags
constexpr int kFlagInfeasible = 1, kFlagInvalid = 2;

void set_error(const char* fmt, ...);

// Launch accounting + optional per-kernel device timing (CUDA events on the launching stream).
enum { kKernelRowStats = 0, kKernelLattice, kKernelGrad, kKernelReduce, kKernelArgmax, kKernelCollapse, kKernelScale, kKernelViterbi, kKernelNoBlank, kKernelBeam, kKernelOrder, kKernelScore, kKernelScoreGrad, kKernelScoreRows, kKernelEdit, kKernelMwerForward, kKernelMwerWeights, kKernelMwerBackward, kKernelBeamLM, kKernelNGramBuild, kKernelBeamBias, kNumKernels };
// e2e_ctc_profile_read's smallest n_kinds: the kinds up to kKernelScore (kinds added later are dropped for such callers)
constexpr int kMinProfileKinds = kKernelScore + 1;
void launch_begin(int kind, cudaStream_t s);
void launch_end(int kind, cudaStream_t s);
struct KernelTimer {   // brackets exactly one kernel launch
  int kind; cudaStream_t s;
  KernelTimer(int k, cudaStream_t st) : kind(k), s(st) { launch_begin(k, st); }
  ~KernelTimer() { launch_end(kind, s); }
};

#define E2E_CUDA_TRY(expr)                                                              \
  do {                                                                                  \
    cudaError_t e__ = (expr);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      ::e2e::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
      return E2E_ERR_CUDA;                                                              \
    }                                                                                   \
  } while (0)

// ------------------------------------------------------------------ device helpers ------------
#ifdef __CUDACC__

__device__ __forceinline__ long long load_index(const void* p, int is64, long long i) {
  return is64 ? reinterpret_cast<const long long*>(p)[i]
              : (long long)reinterpret_cast<const int*>(p)[i];
}

template <typename T> struct Elem;
template <> struct Elem<float> {
  using acc_t = float;
  static __device__ __forceinline__ float load(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ float get(float v) { return v; }
  static __device__ __forceinline__ void store(float* p, float v) { *p = v; }
};
template <> struct Elem<__nv_bfloat16> {
  using acc_t = float;
  static __device__ __forceinline__ float load(const __nv_bfloat16* p) {
    return __bfloat162float(__ldg(p));
  }
  static __device__ __forceinline__ float get(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
};
template <> struct Elem<__half> {
  using acc_t = float;
  static __device__ __forceinline__ float load(const __half* p) { return __half2float(__ldg(p)); }
  static __device__ __forceinline__ float get(__half v) { return __half2float(v); }
  static __device__ __forceinline__ void store(__half* p, float v) { *p = __float2half_rn(v); }
};
template <> struct Elem<double> {
  using acc_t = double;
  static __device__ __forceinline__ double load(const double* p) { return __ldg(p); }
  static __device__ __forceinline__ double get(double v) { return v; }
  static __device__ __forceinline__ void store(double* p, double v) { *p = v; }
};

// runtime-typed scalar load (used where the element type is not worth a template parameter)
__device__ __forceinline__ double load_as_double(const void* base, int dtype, long long idx) {
  switch (dtype) {
    case E2E_F32: return (double)__ldg(reinterpret_cast<const float*>(base) + idx);
    case E2E_BF16: return (double)__bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(base) + idx));
    case E2E_F16: return (double)__half2float(__ldg(reinterpret_cast<const __half*>(base) + idx));
    default: return __ldg(reinterpret_cast<const double*>(base) + idx);
  }
}
__device__ __forceinline__ float load_as_float(const void* base, int dtype, long long idx) {
  switch (dtype) {
    case E2E_F32: return __ldg(reinterpret_cast<const float*>(base) + idx);
    case E2E_BF16: return __bfloat162float(__ldg(reinterpret_cast<const __nv_bfloat16*>(base) + idx));
    case E2E_F16: return __half2float(__ldg(reinterpret_cast<const __half*>(base) + idx));
    default: return (float)__ldg(reinterpret_cast<const double*>(base) + idx);
  }
}
__device__ __forceinline__ void store_from_double(void* base, int dtype, long long idx, double v) {
  switch (dtype) {
    case E2E_F32: reinterpret_cast<float*>(base)[idx] = (float)v; break;
    case E2E_BF16: reinterpret_cast<__nv_bfloat16*>(base)[idx] = __float2bfloat16_rn((float)v); break;
    case E2E_F16: reinterpret_cast<__half*>(base)[idx] = __float2half_rn((float)v); break;
    default: reinterpret_cast<double*>(base)[idx] = v; break;
  }
}

// torch's row log-softmax, (x - max) - log sum exp(x - max), in the input's accumulation type; rounded to the input dtype
// for 16-bit inputs, as F.log_softmax returns it (the rule of the beam search, the scorer and the aligner)
template <typename T>
__device__ __forceinline__ double normalise(typename Elem<T>::acc_t x, typename Elem<T>::acc_t m, typename Elem<T>::acc_t ls) {
  using raw_t = typename Elem<T>::acc_t;
  raw_t v = (x - m) - ls;
  if (sizeof(T) == 2) { T r; Elem<T>::store(&r, (float)v); v = (raw_t)Elem<T>::get(r); }
  return (double)v;
}

// 2^d as a double; 0 below the normal range, clamped above.
__device__ __forceinline__ double pow2i(int d) {
  d = min(d, 1023);
  const double r = __hiloint2double((d + 1023) << 20, 0);
  return d < -1022 ? 0.0 : r;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_max_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

#endif  // __CUDACC__

// ------------------------------------------------------------------ kernel launchers ----------
int launch_row_stats(const e2e_ctc_desc& d, const void* logits, void* stats, double* emis, int emis_stride,
                     const void* targets, const void* in_len, const void* tgt_len, cudaStream_t s);
int launch_fused(const e2e_ctc_desc& d, const LossPlan& p, const void* logits, const void* targets,
                 const void* in_len, const void* tgt_len, void* losses, void* grads, double scale, char* ws,
                 cudaStream_t s);
size_t fused_ctl_bytes();
int launch_sweep(const e2e_ctc_desc& d, const LossPlan& p, const void* logits, const void* targets,
                 const void* in_len, const void* tgt_len, void* losses, void* grads, double scale, char* ws,
                 cudaStream_t s);
int launch_wave(const e2e_ctc_desc& d, const LossPlan& p, const void* logits, const void* targets,
                const void* in_len, const void* tgt_len, void* losses, void* grads, double scale, char* ws,
                cudaStream_t s);
size_t wave_ctl_bytes();
constexpr int kSweepMaxCellsPerLane = 40;   // one warp covers 32 * 40 = 1280 cells: L <= 639
int launch_grad(const e2e_ctc_desc& d, const LossPlan& p, const void* logits, const void* targets,
                const void* in_len, const void* tgt_len, const void* grad_out, int grad_out_count,
                double host_scale, void* grads, const char* ws, cudaStream_t s);
int launch_scale_rows(const e2e_ctc_desc& d, void* grads, const void* grad_out, int grad_out_count, cudaStream_t s);
int launch_reduce(const void* losses, int dtype, int B, double scale, void* out, double* out64,
                  cudaStream_t s);
int launch_greedy(const e2e_ctc_desc& d, const void* logits, const void* in_len, int64_t* decoded,
                  int64_t* decoded_len, char* ws, cudaStream_t s);
size_t beam_workspace_bytes(const e2e_ctc_desc& d, int beam_width);
bool beam_supported(const e2e_ctc_desc& d, int beam_width, bool lm = false, bool bias = false);
// decoded [B, n_best, T], decoded_len [B, n_best]; scores / log_probs [B, n_best] or null (log_probs is ignored without scores)
int launch_beam(const e2e_ctc_desc& d, int beam_width, int n_best, int space_idx, double wip, const void* logits,
                const void* in_len, int64_t* decoded, int64_t* decoded_len, double* scores, double* log_probs, int64_t* ties,
                char* ws, cudaStream_t s);
// the same search with a word n-gram LM fused (e2e_ctc_beam_lm_nbest_device): scores, lm_scores, oov_words required
// tokens: null for a character alphabet (the space is the boundary, lm.label_char every other label's character)
int launch_beam_lm(const e2e_ctc_desc& d, const e2e_ctc_ngram& lm, const e2e_ctc_ngram_tokens* tokens, int beam_width,
                   int n_best, int space_idx, double wip, double lmwt, double oov_penalty, const void* logits,
                   const void* in_len, int64_t* decoded, int64_t* decoded_len, double* scores, double* log_probs,
                   double* lm_scores, int64_t* oov_words, int64_t* ties, char* ws, cudaStream_t s);
// the same search with phrase biasing (e2e_ctc_beam_bias_nbest_device): lm null for none, tokens null for characters;
// scores and bias_scores required, lm_scores and oov_words with a model
int launch_beam_bias(const e2e_ctc_desc& d, const e2e_ctc_ngram* lm, const e2e_ctc_ngram_tokens* tokens,
                     const e2e_ctc_bias& bias, int beam_width, int n_best, int space_idx, double wip, double lmwt,
                     double oov_penalty, const void* logits, const void* in_len, int64_t* decoded, int64_t* decoded_len,
                     double* scores, double* log_probs, double* lm_scores, int64_t* oov_words, double* bias_scores,
                     int64_t* ties, char* ws, cudaStream_t s);
size_t ngram_table_bytes(long long slots);
int launch_ngram_build(void* table, long long slots, long long count, const int* ids, const int* orders, const double* probs,
                       const double* bows, cudaStream_t s);
// N hypotheses per utterance: hyps [B * n_hyp, max_targets], hyp_len [B * n_hyp], scores [B * n_hyp] = -(CTC loss)
bool score_supported(const e2e_ctc_desc& d);
int launch_score(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                 const void* hyp_len, double* scores, cudaStream_t s);
// the scorer's backward (K10 + its row kernel): grad_scores [B * n_hyp] float64, grads of desc->dtype (grads strides);
// workspace: 0 with the message set when a size overflows or a grid exceeds 2^31 - 1 CTAs
bool score_backward_supported(const e2e_ctc_desc& d);
size_t score_backward_workspace_bytes(const e2e_ctc_desc& d, int n_hyp);
int launch_score_backward(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                          const void* hyp_len, const double* grad_scores, void* grads, char* ws, cudaStream_t s);
// MWER over the N-best list (K12a/b/c, the scorer's passes split): the state kept from forward to backward and the
// backward's scratch, each 0 with the message set on overflow; the forward writes losses [B] (scores [B * n_hyp] when not
// null) and the state, the backward consumes the state (its checkpoints are overwritten: one forward, one backward)
size_t mwer_state_bytes(const e2e_ctc_desc& d, int n_hyp);
size_t mwer_backward_workspace_bytes(const e2e_ctc_desc& d, int n_hyp);
int launch_mwer_forward(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                        const void* hyp_len, const double* risk, const unsigned char* mask, double score_scale,
                        double* losses, double* scores, char* state, cudaStream_t s);
int launch_mwer_backward(const e2e_ctc_desc& d, int n_hyp, const void* logits, const void* hyps, const void* in_len,
                         const void* hyp_len, const double* utt_scale, void* grads, char* state, char* ws, cudaStream_t s);
// edit distance of n_hyp hypotheses per utterance (K11): dynamic shared memory of a launch, and the launch
size_t edit_distance_smem_bytes(int ref_width, int words);
int launch_edit_distance(const e2e_ctc_edit_desc& d, const void* hyps, const void* hyp_lengths, const void* refs,
                         const void* ref_lengths, int64_t* errors, int64_t* substitutions, int64_t* insertions,
                         int64_t* deletions, int64_t* reference_units, cudaStream_t s);
size_t noblank_workspace_bytes(const e2e_ctc_desc& d);
bool noblank_supported(const e2e_ctc_desc& d);
int launch_noblank(const e2e_ctc_desc& d, int space_idx, const void* lp, const void* targets, const void* in_len,
                   const void* tgt_len, void* losses, void* grads, char* ws, cudaStream_t s);
// n_hyp lattices per utterance: targets [B * n_hyp, max_targets], tgt_len [B * n_hyp], aligned [B * n_hyp, T];
// from_logits: raw-logit input (K1 statistics in the workspace); token spans [B * n_hyp, max_targets] and path scores
// [B * n_hyp] are optional (CTC only).  Workspace: 0 when the size overflows size_t (message set).
size_t viterbi_workspace_bytes(const e2e_ctc_desc& d, int is_ctc, int n_hyp, int from_logits);
bool viterbi_supported(const e2e_ctc_desc& d, int is_ctc);
int launch_viterbi(const e2e_ctc_desc& d, int is_ctc, int n_hyp, int from_logits, const void* lp, const void* targets,
                   const void* in_len, const void* tgt_len, int64_t* aligned, int64_t* token_starts, int64_t* token_ends,
                   double* path_scores, char* ws, cudaStream_t s);

}  // namespace e2e

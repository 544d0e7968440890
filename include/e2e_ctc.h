/*
 * e2e_ctc.h -- C ABI of the B200-native CTC engine (libe2e_ctc.so, sm_100a).
 *
 * This is the drop-in boundary for the reference's two pybind11 modules:
 *
 *   cpp_ctc_loss.CTCLossEngine(blank_idx).compute(logits, targets, logits_lengths,
 *       targets_lengths) -> (losses[B], grads[B,T,V])
 *       reference: src/losses/ctc_loss_py.cpp:5-17, src/losses/forward_backward.h:16-19,
 *                  src/losses/forward_backward.cpp:7-59, src/losses/ctc_loss.cpp:15-118
 *   cpp_ctc_decoder.CTCDecoder(...).decode_greedy(logits_, logits_lengths_)
 *       -> (decoded_targets[B,T] int64, decoded_targets_lengths[B] int64, sentences)
 *       reference: src/decoders/ctc_decoder_py.cpp:25-29, src/decoders/ctc_decoder.cpp:443-490
 *
 * Plain pointers and sizes only; no torch / pybind11 types.  Two flavours of every operation:
 *
 *   *_device entry points: all pointers are DEVICE pointers on the current CUDA device, work is
 *       enqueued on `stream` and the call returns without synchronising.  The callee never
 *       allocates or frees device memory: the caller passes a workspace of at least
 *       e2e_ctc_*_workspace_bytes() bytes (256-byte aligned).
 *   e2e_ctc_engine_* entry points: an engine handle owns a stream, device staging buffers and the
 *       workspace; pointers are HOST pointers (pinned memory makes the copies asynchronous) and
 *       the call returns when the results are in the host buffers.  This is the form the
 *       reference's `engine.compute(cpu tensors)` call maps to (see INTEGRATION.md).
 *
 * Every function returns E2E_OK (0) or an error code; e2e_last_error_string() gives the
 * thread-local message of the last failure.  inf / NaN results are values, not errors
 * (an infeasible utterance yields loss = +inf and an all-NaN gradient block, as in the reference).
 */
#ifndef E2E_CTC_H_
#define E2E_CTC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define E2E_CTC_ABI_VERSION 1

enum {
  E2E_OK = 0,
  E2E_ERR_INVALID_ARGUMENT = 1, /* bad shape / dtype / null pointer / stride                  */
  E2E_ERR_UNSUPPORTED = 2,      /* valid, but outside this build's limits (see e2e_ctc_limits) */
  E2E_ERR_WORKSPACE = 3,        /* workspace too small or misaligned                           */
  E2E_ERR_CUDA = 4,             /* a CUDA runtime call failed                                  */
  E2E_ERR_LENGTHS = 5           /* a length / label is outside its legal range (UB in the ref) */
};

/* element type of logits / losses / grads (the reference returns the caller's dtype:
 * forward_backward.cpp:55-56).  Arithmetic is fp64 lattice + fp32 transcendentals for
 * F32/BF16/F16 inputs and fp64 throughout for F64 inputs. */
enum { E2E_F32 = 0, E2E_BF16 = 1, E2E_F16 = 2, E2E_F64 = 3 };
/* integer type of targets / lengths (the reference accepts int32 or int64:
 * forward_backward.cpp:16-19) */
enum { E2E_I32 = 0, E2E_I64 = 1 };

/* Problem descriptor.  Strides are in ELEMENTS; the innermost (alphabet) stride must be 1, so a
 * time-major [T,B,V] tensor is read and written in place with stride_b = V, stride_t = B*V
 * (the reference permutes a view: modules/ctc_loss.py:42-43). */
typedef struct e2e_ctc_desc {
  int32_t batch;             /* B                                                             */
  int32_t max_frames;        /* T  (padded number of frames)                                  */
  int32_t alphabet;          /* V                                                             */
  int32_t max_targets;       /* Lmax = width of the targets matrix                            */
  int32_t blank_idx;         /* blank label, 0 <= blank_idx < V                               */
  int32_t dtype;             /* E2E_F32 / E2E_BF16 / E2E_F16 / E2E_F64                        */
  int32_t targets_itype;     /* E2E_I32 / E2E_I64                                             */
  int32_t lengths_itype;     /* E2E_I32 / E2E_I64 (both length vectors)                       */
  int32_t from_logits;       /* 1: input is raw logits, log_softmax is fused and grads are the
                                gradient w.r.t. the logits (CTCLoss(after_logsoftmax=False):
                                modules/ctc_loss.py:37-40 + autograd of log_softmax);
                                0: input is log-probabilities, grads = exp(lp) - posterior on all
                                T rows (the engine contract, ctc_loss.cpp:105-117)             */
  int32_t reserved0;
  int64_t logits_stride_b;   /* elements between utterances in logits                         */
  int64_t logits_stride_t;   /* elements between frames in logits                             */
  int64_t grads_stride_b;    /* same for the gradient output                                  */
  int64_t grads_stride_t;
  int64_t targets_stride_b;  /* elements between rows of targets                              */
} e2e_ctc_desc;

/* Build limits (so callers can test before calling). */
typedef struct e2e_ctc_limits {
  int32_t max_alphabet;      /* largest supported V                                           */
  int32_t max_targets;       /* largest supported target length per utterance                 */
  int32_t abi_version;
  int32_t sm_arch;           /* 100 (sm_100a)                                                 */
} e2e_ctc_limits;

const char* e2e_ctc_version(void);
const char* e2e_last_error_string(void);
int e2e_ctc_get_limits(e2e_ctc_limits* out);

/* ---------------------------------------------------------------- loss, device pointers ---- */

/* Bytes of workspace e2e_ctc_loss_* needs for `desc` (0 on error).  The workspace written by
 * e2e_ctc_loss_forward_device must stay untouched until e2e_ctc_loss_backward_device has run. */
size_t e2e_ctc_loss_workspace_bytes(const e2e_ctc_desc* desc);

/* Forward: row statistics (fused log-softmax), alpha/beta lattice, per-utterance losses.
 * losses: [B] of desc->dtype.  Replaces the alpha/beta/loss part of CTCLossEngine::compute_2d
 * (ctc_loss.cpp:25-100).  All pointers are required (targets may be NULL iff max_targets == 0). */
int e2e_ctc_loss_forward_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                                const void* logits_lengths, const void* targets_lengths,
                                void* losses, void* workspace, size_t workspace_bytes,
                                void* cuda_stream);

/* Backward: grads[b,t,v] = scale_b * (softmax - posterior)  (ctc_loss.cpp:102-117 fused with
 * functions/forward_backward.py:34 `grads * grad_output.view(-1,1,1)`).
 *   grad_out == NULL           : scale_b = host_scale
 *   grad_out_count == 1        : scale_b = host_scale * grad_out[0]   (reduced loss, 0-dim grad)
 *   grad_out_count == B        : scale_b = host_scale * grad_out[b]   (per-utterance loss)
 * grad_out is a device pointer of desc->dtype. */
int e2e_ctc_loss_backward_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                                 const void* logits_lengths, const void* targets_lengths,
                                 const void* grad_out, int32_t grad_out_count, double host_scale,
                                 void* grads, void* workspace, size_t workspace_bytes,
                                 void* cuda_stream);

/* Forward + backward with scale 1: exactly CTCLossEngine.compute() (ctc_loss_py.cpp:10-16).
 * Shapes with alphabet <= 128 run as ONE fused kernel (row log-softmax statistics, lattice and
 * gradient write); larger alphabets run row statistics + lattice + gradient kernels. */
int e2e_ctc_loss_fwd_bwd_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                                const void* logits_lengths, const void* targets_lengths,
                                void* losses, void* grads, void* workspace, size_t workspace_bytes,
                                void* cuda_stream);

/* One training step in one call: e2e_ctc_loss_fwd_bwd_device with the gradient scaled by
 * `grad_scale` (1/B for a mean-reduced loss: functions/forward_backward.py:34 with the constant
 * part of grad_output folded in), followed -- when `reduced` or `reduced_f64` is non-NULL -- by
 * e2e_ctc_loss_reduce_device(losses, ..., reduce_scale, reduced, reduced_f64). */
int e2e_ctc_loss_step_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                             const void* logits_lengths, const void* targets_lengths, void* losses,
                             void* grads, double grad_scale, void* reduced, double* reduced_f64,
                             double reduce_scale, void* workspace, size_t workspace_bytes,
                             void* cuda_stream);

/* grads[b,:,:] *= grad_out[b] (grad_out_count == B) or grad_out[0] (grad_out_count == 1), in
 * place; grad_out is a device pointer of desc->dtype.  Blocks whose factor is exactly 1 return
 * without touching memory, so autograd's usual all-ones grad_output costs one empty launch. */
int e2e_ctc_scale_rows_device(const e2e_ctc_desc* desc, void* grads, const void* grad_out,
                              int32_t grad_out_count, void* cuda_stream);

/* out[0] = scale * sum_b losses[b]  (modules/ctc_loss.py:52-56: sum, or mean with scale = 1/B;
 * multi-GPU callers all-reduce this scalar).  losses/out are of `dtype`; summation is fp64 in a
 * fixed order.  out_f64 (optional, may be NULL) points to TWO doubles and receives
 * {scale * sum, (double)batch}: the pair a data-parallel caller all-reduces across GPUs. */
int e2e_ctc_loss_reduce_device(const void* losses, int32_t dtype, int32_t batch, double scale,
                               void* out, double* out_f64, void* cuda_stream);

/* Device-side argument check result of the last forward on this workspace: *status_host = 0 if
 * every length / label was in range, else a bit mask (1: frames, 2: target length, 4: label).
 * Synchronises `cuda_stream`. */
int e2e_ctc_loss_check_device(const void* workspace, int32_t* status_host, void* cuda_stream);

/* ------------------------------------------------------------- multi-GPU: the one exchange ---- */

/* Utterances are independent (forward_backward.cpp:38-52), so a batch shards across GPUs with no
 * data-path collective; the only exchange is ONE NCCL all-reduce of the reduced loss scalar
 * (modules/ctc_loss.py:52-56 summed over ranks).  The communicator is owned by the library (libnccl is
 * resolved at run time) so that a host language without its own collective layer can shard a batch:
 *   rank 0: e2e_ctc_comm_unique_id(id) -> ship the 128 bytes to every rank by any means;
 *   every rank (its CUDA device current): e2e_ctc_comm_create(id, nranks, rank, &comm)  [collective];
 *   per step, after e2e_ctc_loss_step_device(..., reduced, ...):
 *       e2e_ctc_comm_allreduce_sum(comm, reduced, 1, dtype, stream)                    [in place]. */
typedef struct e2e_ctc_comm e2e_ctc_comm;
int e2e_ctc_comm_unique_id(void* out_id128);
int e2e_ctc_comm_create(const void* id128, int32_t nranks, int32_t rank, e2e_ctc_comm** out);
void e2e_ctc_comm_destroy(e2e_ctc_comm* comm);
int e2e_ctc_comm_allreduce_sum(e2e_ctc_comm* comm, void* buf, int64_t count, int32_t dtype, void* cuda_stream);

/* ------------------------------------------------------------------- CUDA-graph step -------- */

/* The training step of e2e_ctc_loss_step_device -- and, when `comm` is non-NULL, the in-place all-reduce of
 * `reduced` -- captured once into a CUDA graph bound to these buffers (SURVEY 8(f1): the reference's step is
 * modules/ctc_loss.py:37-57 + functions/forward_backward.py:6-35; here it replays with ONE driver call).
 * The buffers and the workspace must stay alive and at the same addresses for the lifetime of the graph; their
 * CONTENTS may change between launches (a training loop copies each batch into the same buffers).
 * e2e_ctc_graph_create runs the step once (results are valid afterwards) and synchronises; launch only enqueues. */
typedef struct e2e_ctc_graph e2e_ctc_graph;
int e2e_ctc_graph_create(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                         const void* logits_lengths, const void* targets_lengths, void* losses, void* grads,
                         double grad_scale, void* reduced, double* reduced_f64, double reduce_scale,
                         void* workspace, size_t workspace_bytes, e2e_ctc_comm* comm, e2e_ctc_graph** out);
int e2e_ctc_graph_launch(e2e_ctc_graph* graph, void* cuda_stream);
void e2e_ctc_graph_destroy(e2e_ctc_graph* graph);

/* ------------------------------------------------------------ Viterbi forced alignment ----- */

/* Best-path (Viterbi) alignment of every utterance's targets to its frames -- the reference's
 * pytorch_end2end/utils/alignment.py: get_alignment_3d (:109-138) over _get_alignment_ctc_1d (:50-106, is_ctc != 0:
 * blank-extended lattice) or _get_alignment_asg_1d (:9-47, is_ctc == 0: labels only).  `log_probs` are
 * log-probabilities [B,T,V] (desc strides), `aligned` is [B,T] int64: the label id of every frame, -100 past the
 * utterance's frames (the reference's fill value).  Bit-exact with the reference: fp64 max-plus recursion with its
 * comparison order and window.  desc->blank_idx is the blank (the reference hard-codes 0).  A logits length of 0
 * leaves the row at -100; out-of-range lengths / labels set status bits (e2e_ctc_loss_check_device on the
 * workspace) and leave -100.  Limit: lattices of at most 2048 cells, i.e. desc->max_targets <= 1023 for CTC
 * (2 L + 1 cells) and <= 2048 for ASG (L cells), independent of the loss's limit (e2e_ctc_get_limits); beyond it
 * the workspace query returns 0 and the alignment E2E_ERR_UNSUPPORTED, with the reason in e2e_last_error_string. */
size_t e2e_ctc_viterbi_workspace_bytes(const e2e_ctc_desc* desc, int32_t is_ctc);
int e2e_ctc_viterbi_align_device(const e2e_ctc_desc* desc, int32_t is_ctc, const void* log_probs,
                                 const void* targets, const void* logits_lengths, const void* targets_lengths,
                                 int64_t* aligned, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* ------------------------------------------- N hypotheses per utterance: alignment and timestamps ---- */

/* The best-path (Viterbi) alignment of n_hyp hypotheses per utterance over the CTC lattice, with each token's frame span
 * and the best path's log-probability: timestamps for transcripts (this library's N-best lists or any other).  Lattice
 * r = b * n_hyp + n aligns hypothesis n of utterance b against utterance b's frames, read once from `logits` (no
 * replicated input).  e2e_ctc_viterbi_align_device is the n_hyp == 1, log-prob, no-span call of the same kernel.
 *   logits: log-probabilities [B,T,V] (desc strides) when desc->from_logits == 0, raw logits when it is 1 (the row
 *       log-softmax of the scorer and the beam search: (x - max) - log sum exp in the input's precision, rounded to the
 *       input dtype for 16-bit inputs);
 *   hyps: [B * n_hyp, max_targets] of targets_itype, row stride desc->targets_stride_b (NULL allowed when max_targets
 *       == 0); hyp_lengths: [B * n_hyp]; logits_lengths: [B] or NULL for max_frames;
 *   aligned: [B * n_hyp, T] int64, row r exactly what e2e_ctc_viterbi_align_device (is_ctc = 1) writes for utterance b's
 *       frames with hypothesis r as its target: the label id of every frame, -100 past the utterance's frames;
 *   path_scores: [B * n_hyp] float64, the best path's log-probability (the final cell the backtrace starts from; the
 *       final blank wins unless the final label is strictly better): a sum of fp64-widened log-probabilities in frame
 *       order.  The empty hypothesis gives sum_t log p(blank | t); an infeasible one (T_b < L + repeats) -inf; a
 *       hypothesis length outside [0, max_targets] or a label outside [0, alphabet) NaN, and a logits length outside
 *       [1, max_frames] NaN for every hypothesis of the utterance (with -100 rows and status bits as
 *       e2e_ctc_viterbi_align_device sets them).  path_scores <= the e2e_ctc_score_device score wherever both are finite;
 *   token_starts, token_ends: [B * n_hyp, max_targets] int64 (may be NULL when max_targets == 0): token k < L covers the
 *       frames [start, end) whose path cell is label cell 2 k + 1 -- non-empty, disjoint and increasing; -1 in slots
 *       k >= L and wherever the path score is not > -inf.
 * Workspace: 256 status bytes, the row statistics of raw-logit input (8 bytes a frame, 16 for F64) and one backpointer
 * byte per thread per frame of every lattice.  Limits: those of the Viterbi alignment (max_targets <= 1023) and alphabet <=
 * e2e_ctc_limits.max_alphabet; beyond them, with n_hyp < 1, or when B * n_hyp exceeds 2^31 - 1 or the workspace size
 * overflows, the workspace query returns 0 and sets the error message. */
size_t e2e_ctc_align_nbest_workspace_bytes(const e2e_ctc_desc* desc, int32_t n_hyp);
int e2e_ctc_align_nbest_device(const e2e_ctc_desc* desc, int32_t n_hyp, const void* logits, const void* hyps,
                               const void* logits_lengths, const void* hyp_lengths, int64_t* aligned, int64_t* token_starts,
                               int64_t* token_ends, double* path_scores, void* workspace, size_t workspace_bytes,
                               void* cuda_stream);

/* ------------------------------------------------------------------- CTC without blank ----- */

/* Loss and gradient of the blank-free CTC variant -- the reference's pytorch_end2end/functions/ctc_without_blank.py:
 * _ctc_without_blank_loss (:13-88) under _ctc_without_blank_3d_loss (:91-117).  `log_probs` are log-probabilities
 * [B,T,V]; space_idx = -1: the lattice is the target sequence itself; otherwise one optional `space_idx` cell is
 * added at either end.  losses[b] = -log Z; grads[b,t,v] = exp(lp) - posterior for t < T_b and 0 past the
 * utterance's frames; an utterance with no alignment gives +inf / NaN as in the reference.  fp64 log-space.
 * Limit: desc->max_targets <= 1022, and the labels plus one int per symbol in 200 KB of shared memory (any alphabet up
 * to 40,000 symbols); beyond it the workspace query returns 0 and the loss E2E_ERR_UNSUPPORTED, with the reason in
 * e2e_last_error_string. */
size_t e2e_ctc_noblank_workspace_bytes(const e2e_ctc_desc* desc);
int e2e_ctc_noblank_fwd_bwd_device(const e2e_ctc_desc* desc, int32_t space_idx, const void* log_probs,
                                   const void* targets, const void* logits_lengths, const void* targets_lengths,
                                   void* losses, void* grads, void* workspace, size_t workspace_bytes,
                                   void* cuda_stream);

/* --------------------------------------------------------------- greedy decode, device ----- */

size_t e2e_ctc_greedy_workspace_bytes(const e2e_ctc_desc* desc);

/* decoded: [B,T] int64, zero padded; decoded_lengths: [B] int64.  logits_lengths may be NULL
 * (every utterance decoded over all T frames, decoders/ctc_decoder.py:140-141).
 * argmax = first maximum, NaN is maximal (torch.argmax, ctc_decoder.cpp:451); then emit a symbol
 * iff it is not blank and differs from the previous frame's symbol (ctc_decoder.cpp:471-482). */
int e2e_ctc_greedy_decode_device(const e2e_ctc_desc* desc, const void* logits,
                                 const void* logits_lengths, int64_t* decoded,
                                 int64_t* decoded_lengths, void* workspace, size_t workspace_bytes,
                                 void* cuda_stream);

/* ------------------------------------------------------- LM-free prefix beam search, device ----- */

/* Prefix beam search without a language model -- the reference's cpp_ctc_decoder.CTCDecoder(...).decode(logits_,
 * logits_lengths_) (src/decoders/ctc_decoder_py.cpp:30-34; src/decoders/ctc_decoder.cpp:153-198 decode, :353-441
 * decode_sentence, :241-309 get_next_prefix, :311-340 scores) with lm_path == "" (lmwt forced to 0, :76).
 *   logits: log-probabilities [B,T,V] (desc strides) when desc->from_logits == 0 -- what the reference's C++ receives --
 *       or raw logits when desc->from_logits == 1: the F.log_softmax of decoders/ctc_decoder.py:95-97 is then fused
 *       (computed in the input's precision and rounded to the input dtype, as torch does);
 *   beam_width: CTCDecoder's beam_width_ (>= 1; limits: e2e_ctc_beam_workspace_bytes returns 0 when unsupported);
 *   space_idx: index of " " in the labels or -1 (ctc_decoder.cpp:56-60) -- only the word count behind `wip` uses it;
 *   wip: word insertion penalty (score = log p(prefix) - num_words * wip, :311-315);
 *   decoded: [B,T] int64 zero padded; decoded_lengths: [B] int64.  The reference returns [B, max length]: the caller
 *       slices.  An utterance whose best prefix is EMPTY yields length 1 and the single symbol -1, as the reference does
 *       (Prefix::get_sentence pushes the root's last_char, :225-239);
 *   ties (optional, [B] int64): how many prunes of the utterance (and the final pick) had EQUAL scores on both sides of
 *       the cut.  There the reference's choice is whatever libstdc++'s std::nth_element / std::sort do; this library
 *       takes the lower position (beam order, then extensions by (member, symbol)).  0 = the result does not depend on
 *       that.  In practice ties arise only between -inf scores while fewer than beam_width prefixes are feasible (tiny
 *       alphabets with large beams) or from identical input rows.
 * The prefix trie (node = parent, symbol, reference count, child list) lives in the workspace: the reference's
 * weak_ptr lookup of a pruned-but-still-referenced child (:244-246) is reproduced exactly. */
size_t e2e_ctc_beam_workspace_bytes(const e2e_ctc_desc* desc, int32_t beam_width);
int e2e_ctc_beam_decode_device(const e2e_ctc_desc* desc, int32_t beam_width, int32_t space_idx, double wip,
                               const void* logits, const void* logits_lengths, int64_t* decoded,
                               int64_t* decoded_lengths, int64_t* ties, void* workspace, size_t workspace_bytes,
                               void* cuda_stream);

/* The N best prefixes of the same search and their scores: what a caller needs to rescore the list with a language model
 * of its own (N-best rescoring).  Nothing in the search changes: after the last frame the beam_width final prefixes are
 * ranked, and the first n_best are returned.  e2e_ctc_beam_decode_device is the n_best == 1 call.
 *   ranking: by score = log p(prefix) - num_words * wip, highest first; among EQUAL scores the lower position in the
 *       final beam goes first (the rule of the best-1 pick above).  Hypothesis 0 is what e2e_ctc_beam_decode_device
 *       returns;
 *   n_best: 1 <= n_best <= beam_width (E2E_ERR_INVALID_ARGUMENT otherwise; the workspace query then returns 0);
 *   decoded: [B,N,T] int64 zero padded; decoded_lengths: [B,N] int64.  The empty prefix is the single symbol -1 with
 *       length 1, as above;
 *   scores: [B,N] float64, the ranking score log p - num_words * wip;
 *   log_probs (optional, [B,N] float64): log p(prefix) = log(p_blank + p_not_blank), without the word penalty;
 *   slots past the number of prefixes in the final beam (short utterances, tiny alphabets): length 0, all-zero
 *       symbols, scores = log_probs = -inf;
 *   ties (optional, [B] int64): the prune ties counted as above, plus 1 when the returned list depends on equal final
 *       scores (a prefix of rank < N has the same score as another prefix of the final beam; for N = 1 that is the
 *       final-pick tie above); -1, as for e2e_ctc_beam_decode_device, when the list of pruned prefixes that still
 *       block an extension overflowed.
 * The workspace is the same as e2e_ctc_beam_workspace_bytes(desc, beam_width). */
size_t e2e_ctc_beam_nbest_workspace_bytes(const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best);
int e2e_ctc_beam_nbest_device(const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best, int32_t space_idx, double wip,
                              const void* logits, const void* logits_lengths, int64_t* decoded, int64_t* decoded_lengths,
                              double* scores, double* log_probs, int64_t* ties, void* workspace, size_t workspace_bytes,
                              void* cuda_stream);

/* ------------------------------------------------------- N hypotheses per utterance: score ---- */

/* The CTC log-likelihood log p(y | x) of n_hyp hypotheses per utterance, forward only (no gradient, nothing kept for a
 * backward): scores[b * n_hyp + n] = minus the loss of e2e_ctc_loss_forward_device for utterance b with hypothesis n as
 * its target.  For rescoring N-best lists (this library's or another system's), confidence and verification scores.
 *   hyps: [B * n_hyp, max_targets] of targets_itype, row stride desc->targets_stride_b; row b * n_hyp + n is hypothesis
 *       n of utterance b (NULL allowed when max_targets == 0);
 *   hyp_lengths: [B * n_hyp] of lengths_itype, 0 <= length <= max_targets (0: the empty hypothesis, which scores
 *       sum_t log p(blank | t));
 *   logits_lengths: [B] of lengths_itype, or NULL for max_frames;
 *   scores: [B * n_hyp] float64 whatever desc->dtype.  An infeasible hypothesis (T_b < L + repeats) scores -inf.
 *       A hypothesis length outside [0, max_targets] or a label outside [0, alphabet) gives that hypothesis NaN; a
 *       logits length outside [1, max_frames] gives every hypothesis of the utterance NaN.  Nothing out of range is read.
 *   desc->from_logits: the row log-softmax of the loss and the beam search, (x - max) - log sum exp in the input's
 *       precision, rounded to the input dtype for 16-bit inputs; the lattice is fp64.
 * Limits: max_targets <= e2e_ctc_limits.max_targets (639) and alphabet <= e2e_ctc_limits.max_alphabet; beyond them, or
 * with n_hyp < 1, the workspace query returns 0 and sets the error message.  The kernel needs no scratch memory: the
 * query returns 256 bytes within the limits, and the workspace pointer is checked like every other one. */
size_t e2e_ctc_score_workspace_bytes(const e2e_ctc_desc* desc, int32_t n_hyp);
int e2e_ctc_score_device(const e2e_ctc_desc* desc, int32_t n_hyp, const void* logits, const void* hyps,
                         const void* logits_lengths, const void* hyp_lengths, double* scores, void* workspace,
                         size_t workspace_bytes, void* cuda_stream);

/* The gradient of those scores for N-best sequence training (minimum word error rate and other objectives over the
 * list): given g[b * n_hyp + n] = d objective / d scores[b * n_hyp + n], the true derivative of the objective with respect
 * to the input, where gamma_bn(t, v) = sum_{s: ext[s] = v} alpha_t(s) beta_t(s) / p is hypothesis n's occupancy of symbol
 * v at frame t (it sums to 1 over v):
 *   log-probability input (desc->from_logits == 0): grads[b,t,v] = sum_n g[b,n] gamma_bn(t,v) for t < T_b;
 *   raw logits (desc->from_logits == 1): grads[b,t,v] = sum_n g[b,n] (gamma_bn(t,v) - softmax(x_bt)_v) for t < T_b, the
 *       softmax being exp of the row log-softmax of e2e_ctc_score_device (16-bit rounding included);
 *   padding frames t >= T_b: 0.
 * Unlike e2e_ctc_loss_backward_device on log-probability input, there is no exp(lp) term and padding rows are 0: this is
 * the derivative of the score, not the reference engine's gradient convention.  The lattice is the one the score sums
 * over; for a label equal to the blank next to a different label the reference's beta differs from it, and this gradient
 * follows the score.
 *   grad_scores: [B * n_hyp] float64 on the device.  A hypothesis with g == 0 costs no sweep and contributes nothing; an
 *       infeasible one (score -inf) contributes exactly 0 whatever its g;
 *   grads: [B,T,V] of desc->dtype with strides desc->grads_stride_b / grads_stride_t (unit alphabet stride), every element
 *       written once.  A hypothesis length or label out of range (a NaN score) makes the utterance's rows t < T_b NaN --
 *       the rows are shared by all its hypotheses -- and a logits length out of range all of its rows; other utterances
 *       are untouched.
 * fp64 lattice and accumulation in a fixed order, no floating-point atomics: bitwise reproducible.  Limits as for the
 * score.  Workspace: per hypothesis an alpha checkpoint per staged block of frames and one block of alpha, per group of
 * eight hypotheses a partial [T,V] float64 block; the query returns 0 and sets the message past the limits, with
 * n_hyp < 1, when the size overflows size_t or when a grid exceeds 2^31 - 1 CTAs.  Enqueues only; never allocates. */
size_t e2e_ctc_score_backward_workspace_bytes(const e2e_ctc_desc* desc, int32_t n_hyp);
int e2e_ctc_score_backward_device(const e2e_ctc_desc* desc, int32_t n_hyp, const void* logits, const void* hyps,
                                  const void* logits_lengths, const void* hyp_lengths, const double* grad_scores,
                                  void* grads, void* workspace, size_t workspace_bytes, void* cuda_stream);

/* -------------------------------------------------------------- engine, host pointers ------ */

typedef struct e2e_ctc_engine e2e_ctc_engine;

/* Creates an engine bound to CUDA device `device` (fails with E2E_ERR_CUDA when there is no such
 * device -- there is no CPU fallback). */
int e2e_ctc_engine_create(int32_t device, e2e_ctc_engine** out);
void e2e_ctc_engine_destroy(e2e_ctc_engine* engine);

/* Host-buffer form of CTCLossEngine.compute(): copies the inputs to the device, runs the loss
 * forward+backward there, copies losses [B] and grads back (layout given by desc strides, which
 * describe the HOST tensors; they must be dense in (t,v) blocks: either batch-major contiguous
 * or time-major contiguous).  Returns after the results have landed. */
int e2e_ctc_engine_loss_host(e2e_ctc_engine* engine, const e2e_ctc_desc* desc, const void* logits,
                             const void* targets, const void* logits_lengths,
                             const void* targets_lengths, void* losses, void* grads);

/* Host-buffer form of CTCDecoder.decode_greedy(). */
int e2e_ctc_engine_greedy_host(e2e_ctc_engine* engine, const e2e_ctc_desc* desc, const void* logits,
                               const void* logits_lengths, int64_t* decoded,
                               int64_t* decoded_lengths);

/* Host-buffer form of CTCDecoder.decode() without a language model (see e2e_ctc_beam_decode_device). */
int e2e_ctc_engine_beam_host(e2e_ctc_engine* engine, const e2e_ctc_desc* desc, int32_t beam_width, int32_t space_idx,
                             double wip, const void* logits, const void* logits_lengths, int64_t* decoded,
                             int64_t* decoded_lengths, int64_t* ties);

/* Host-buffer form of the N-best list (see e2e_ctc_beam_nbest_device); log_probs and ties may be NULL. */
int e2e_ctc_engine_beam_nbest_host(e2e_ctc_engine* engine, const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best,
                                   int32_t space_idx, double wip, const void* logits, const void* logits_lengths,
                                   int64_t* decoded, int64_t* decoded_lengths, double* scores, double* log_probs,
                                   int64_t* ties);

/* ------------------------------------------- N hypotheses per utterance: word / token errors ---- */

/* Edit distance of n_hyp hypotheses per utterance against the utterance's reference transcript: the risk of N-best
 * sequence training (minimum word error rate) and the counts behind WER / CER.  Row r = b * n_hyp + n of `hyps` is
 * compared with row b of `refs`.  A token is any integer; the units compared are
 *   separator < 0 (token level): every token row[0:length), so CER when tokens are characters;
 *   separator >= 0 (word level): the words, maximal runs of tokens other than `separator`.  Separators are never units:
 *       leading, trailing and repeated separators make no empty word.  Two words are equal iff they are the same token
 *       sequence (a fingerprint filters, every match is confirmed token by token).
 * errors is the least number of unit substitutions, insertions (a hypothesis unit with no reference counterpart) and
 * deletions (a reference unit missing from the hypothesis), each costing 1, that turn the reference into the hypothesis.
 * The split is that of the least-errors alignment with the most substitutions, so it is unique; tools with weighted
 * costs (sclite) may split the same total differently.
 *   hyps: [batch * n_hyp, hyp_width] (row stride hyp_stride_b), refs: [batch, ref_width] (row stride ref_stride_b), both
 *       of tokens_itype; hyp_lengths [batch * n_hyp] and ref_lengths [batch] of lengths_itype;
 *   errors, substitutions, insertions, deletions: [batch * n_hyp] int64; reference_units: [batch] int64, the number of
 *       reference units (the WER / CER denominator).
 * A length outside [0, width] gives -1 in every output of the pairs it belongs to (a reference length: all n_hyp pairs of
 * the utterance and its reference_units); nothing out of range is read and the other pairs are unaffected.  Integer
 * arithmetic without atomics: every run gives the same counts.  The call only enqueues work.  Limits: ref_width <= 4095
 * and hyp_width <= 65535 (the DP key errors * 4096 - substitutions stays within int32); past them the workspace query
 * returns 0 with the reason in e2e_last_error_string.  The workspace (256 bytes) is not used by the kernel. */
typedef struct e2e_ctc_edit_desc {
  int32_t batch, n_hyp, hyp_width, ref_width;
  int32_t tokens_itype;              /* E2E_I32 / E2E_I64, both token matrices  */
  int32_t lengths_itype;             /* E2E_I32 / E2E_I64, both length vectors  */
  int32_t separator;                 /* -1: token level; else word level        */
  int32_t reserved0;
  int64_t hyp_stride_b, ref_stride_b;   /* elements between rows               */
} e2e_ctc_edit_desc;
size_t e2e_ctc_edit_distance_workspace_bytes(const e2e_ctc_edit_desc* desc);
int e2e_ctc_edit_distance_device(const e2e_ctc_edit_desc* desc, const void* hyps, const void* hyp_lengths,
                                 const void* refs, const void* ref_lengths, int64_t* errors, int64_t* substitutions,
                                 int64_t* insertions, int64_t* deletions, int64_t* reference_units,
                                 void* workspace, size_t workspace_bytes, void* cuda_stream);

/* Pinned (page-locked, device-addressable) host memory for result buffers: when `losses` / `grads` of
 * e2e_ctc_engine_loss_host live in such memory the kernels store into them directly and no copy-out stage runs. */
int e2e_ctc_host_alloc(size_t bytes, void** out);
int e2e_ctc_host_free(void* p);

/* Bytes moved by the last engine call (for benchmarks): host->device and device->host.  Every byte that crosses
 * PCIe is counted, whether the copy engine moved it or -- result buffers in pinned host memory -- the kernels
 * stored it into the caller's buffer directly. */
int e2e_ctc_engine_last_traffic(const e2e_ctc_engine* engine, uint64_t* h2d_bytes,
                                uint64_t* d2h_bytes);

/* Number of kernels this library has launched from the calling process since load. */
uint64_t e2e_ctc_launch_count(void);

/* Optional per-kernel device timing for benchmarks.  While enabled, every kernel launch is
 * bracketed by CUDA events on its launching stream.  e2e_ctc_profile_read() waits for the pending
 * events, then fills ms[k] (summed device milliseconds) and launches[k] per kernel kind
 * k = 0 row_stats, 1 lattice, 2 gradient, 3 loss_reduce, 4 argmax, 5 collapse, 6 scale_rows, 7 viterbi,
 * 8 ctc_without_blank, 9 beam_search, 10 order, 11 score, 12 score_backward, 13 score_backward_rows, 14 edit_distance
 * (n_kinds >= 12;
 * the kinds past n_kinds are not reported), and clears the record.  All launches since the previous read must have been made on ONE device. */
int e2e_ctc_profile_enable(int32_t on);
int e2e_ctc_profile_read(double* ms, uint64_t* launches, int32_t n_kinds);

#ifdef __cplusplus
}
#endif
#endif /* E2E_CTC_H_ */

"""CTCDecoder -- CTC decoding on the GPU behind the reference's decoder class
(pytorch_end2end/decoders/ctc_decoder.py:25-149).

* greedy: ``decode`` with ``beam_width == 1`` and ``decode_greedy`` (decoders/ctc_decoder.py:92-93, 117-149;
  src/decoders/ctc_decoder.cpp:443-490);
* prefix beam search WITHOUT a language model: ``decode`` with ``beam_width > 1`` and no ``lm_path``
  (decoders/ctc_decoder.py:76-115; src/decoders/ctc_decoder.cpp:153-198, 353-441) -- SURVEY.md 8(f3);
* the N best prefixes of that search with their scores: ``decode_nbest``, for rescoring with any language model on the
  host (N-best rescoring);
* the exact CTC log-likelihood of given transcripts, N per utterance: ``score`` (``decode_nbest``'s list or any other);
* timestamps of given transcripts, N per utterance: ``align`` -- the best path, each token's frame span, word spans and
  the best path's log-probability;
* word and token errors of N transcripts per utterance against a reference: ``errors`` -- the risk of N-best sequence
  training and the counts behind WER / CER.

KenLM decoding (``lm_path``) stays the reference's CPU code and is out of scope; asking for it here raises
``NotImplementedError`` instead of silently decoding without the model.
"""
from collections import namedtuple

from ..engine import ALIGN_MAX_TARGETS, CTCBeamEngine
from ..utils.hypotheses import empty_marker_as_empty


class CTCDecoderError(Exception):
    pass


DecoderResults = namedtuple("DecoderResults", ["decoded_targets",
                                               "decoded_targets_lengths",
                                               "decoded_sentences"])

NBestResults = namedtuple("NBestResults", ["decoded_targets",
                                           "decoded_targets_lengths",
                                           "decoded_sentences",
                                           "scores",
                                           "log_probs"])

AlignmentResults = namedtuple("AlignmentResults", ["alignments",
                                                   "token_starts",
                                                   "token_ends",
                                                   "path_scores",
                                                   "word_spans"])

ErrorCounts = namedtuple("ErrorCounts", ["errors",
                                         "substitutions",
                                         "insertions",
                                         "deletions",
                                         "reference_units"])


def word_spans(tokens, starts, ends, labels):
    """``[(word, start_frame, end_frame)]`` of one aligned hypothesis: a word is a maximal run of tokens other than the
    label ``" "``; it spans from its first token's start to its last token's end (``-1`` where the path had no finite
    score).  ``tokens``, ``starts`` and ``ends`` are lists over the hypothesis's tokens."""
    out, word = [], None
    for tok, t0, t1 in zip(tokens, starts, ends):
        sym = labels[tok]
        if sym == " ":
            word = None
        elif word is None:
            word = [sym, t0, t1]
            out.append(word)
        else:
            word[0] += sym
            word[2] = t1
    return [tuple(w) for w in out]


class CTCDecoder:
    """
    :param beam_width: ``1``: greedy; larger: prefix beam search
    :param after_logsoftmax: the input is log-probabilities (beam search fuses the log-softmax otherwise;
        greedy decoding does not care: argmax is invariant to log-softmax)
    :param blank_idx: id of the blank label, default ``0``
    :param time_major: logits are ``(T, B, V)`` instead of ``(B, T, V)``
    :param labels: list of strings with labels (including the blank symbol), e.g. ``["_", "a", "b"]``
    :param wip: word insertion penalty of the beam search (score = log p - number of words * wip; words are
        separated by the label ``" "``)
    :param lm_path, lmwt, oov_penalty, case_sensitive: language-model options of the reference's beam search;
        accepted for signature compatibility.  A non-empty ``lm_path`` is refused by ``decode``
    """

    def __init__(self, beam_width=100, after_logsoftmax=False, blank_idx=0, time_major=False, labels=None,
                 lm_path=None, lmwt=1.0, wip=1.0, oov_penalty=-10, case_sensitive=True):
        self._beam_width = beam_width
        self._blank_idx = blank_idx
        self._after_logsoftmax = after_logsoftmax
        self._labels = list(labels or [])
        self._lm_path = lm_path or ""
        self._lmwt = lmwt
        self._wip = wip
        self._oov_penalty = oov_penalty
        self._time_major = time_major
        self._case_sensitive = case_sensitive
        self._decoder = CTCBeamEngine(self._blank_idx, max(int(self._beam_width), 1), self._labels, self._wip)

    def decode(self, logits, logits_lengths=None):
        """Prefix beam search (`<https://arxiv.org/abs/1408.2873>`_) without a language model; greedy decoding when
        ``beam_width == 1`` (decoders/ctc_decoder.py:76-115).

        :param logits: ``(T, B, V)`` if ``time_major`` else ``(B, T, V)``; CPU or CUDA tensor; log-probabilities if
            ``after_logsoftmax`` else raw network outputs
        :param logits_lengths: ``(B,)`` or ``None`` (decode all frames)
        :return: ``DecoderResults(decoded_targets [B, longest result] int64 zero padded, decoded_targets_lengths [B]
            int64, decoded_sentences list[str])`` -- CPU tensors, as in the reference.  An utterance whose best
            prefix is empty comes back as the single symbol ``-1`` with length 1 (the reference's behaviour); its
            sentence is ``""``
        """
        if self._beam_width == 1:
            return self.decode_greedy(logits, logits_lengths)
        if self._lm_path:
            raise NotImplementedError(
                "decoding with a KenLM language model stays the reference's CPU code and is outside this engine's "
                "scope; construct CTCDecoder without lm_path")
        if self._time_major:
            logits = logits.transpose(1, 0)
        decoded_targets, decoded_targets_lengths = self._decoder.decode(
            logits_=logits, logits_lengths_=logits_lengths, from_logits=not self._after_logsoftmax)
        decoded_sentences = self._sentences(decoded_targets, decoded_targets_lengths)
        return DecoderResults(decoded_targets, decoded_targets_lengths, decoded_sentences)

    def decode_nbest(self, logits, logits_lengths=None, *, n_best):
        """The ``n_best`` best prefixes of the LM-free prefix beam search and their scores, for rescoring with a
        language model of the caller's choice.  Always the prefix beam search: with ``beam_width == 1`` that is a
        beam of width 1, not the greedy path ``decode`` takes.

        :param logits: as for ``decode``
        :param logits_lengths: ``(B,)`` or ``None`` (decode all frames)
        :param n_best: ``1 <= n_best <= beam_width``
        :return: ``NBestResults(decoded_targets [B, N, longest hypothesis] int64 zero padded, decoded_targets_lengths
            [B, N] int64, decoded_sentences list[B] of list[N] str, scores [B, N] float64, log_probs [B, N] float64)``
            -- CPU tensors.  Hypotheses are ranked by ``scores = log_probs - number of words * wip``, highest first
            (equal scores in beam order), so hypothesis 0 is what ``decode`` returns for ``beam_width > 1``;
            ``log_probs`` is the prefix's acoustic log-probability without the word penalty.  The empty prefix is the
            single symbol ``-1`` with length 1, as in ``decode``; slots past the number of prefixes the final beam
            holds (short utterances, tiny alphabets) have length 0, sentence ``""`` and ``-inf`` scores
        """
        if self._lm_path:
            raise NotImplementedError(
                "decoding with a KenLM language model stays the reference's CPU code and is outside this engine's "
                "scope; construct CTCDecoder without lm_path and rescore the decode_nbest list with the model")
        if not 1 <= int(n_best) <= self._decoder.beam_width:
            raise ValueError("n_best %d outside [1, beam_width = %d]" % (int(n_best), self._decoder.beam_width))
        if self._time_major:
            logits = logits.transpose(1, 0)
        decoded_targets, decoded_targets_lengths, scores, log_probs = self._decoder.decode_nbest(
            logits, logits_lengths, n_best=int(n_best), from_logits=not self._after_logsoftmax)
        B, N = decoded_targets_lengths.shape
        flat = self._sentences(decoded_targets.reshape(B * N, -1), decoded_targets_lengths.reshape(-1))
        decoded_sentences = [flat[b * N:(b + 1) * N] for b in range(B)]
        return NBestResults(decoded_targets, decoded_targets_lengths, decoded_sentences, scores, log_probs)

    def score(self, logits, hypotheses, hypotheses_lengths, logits_lengths=None):
        """The CTC log-likelihood ``log p(hypothesis | logits)`` of N transcripts per utterance: minus the CTC loss of each
        (utterance, hypothesis) pair, summed over every alignment -- where ``decode_nbest``'s ``log_probs`` sums only the
        alignments that survived the beam.  Forward only, on the GPU; the utterance's frames are read and normalised once
        for several hypotheses, not once per hypothesis.

        :param logits: as for ``decode`` (``time_major``, ``after_logsoftmax`` and ``blank_idx`` apply)
        :param hypotheses: ``(B, N, max length)`` int32 / int64 labels, zero padded; ``decode_nbest``'s
            ``decoded_targets`` as they come
        :param hypotheses_lengths: ``(B, N)``; the single symbol ``-1`` with length 1 (``decode``'s empty result) is the
            empty hypothesis
        :param logits_lengths: ``(B,)`` or ``None`` (all frames)
        :return: ``(B, N)`` float64 CPU tensor.  An infeasible hypothesis (more labels and repeats than frames) scores
            ``-inf``; the empty hypothesis scores ``sum_t log p(blank | t)``.  Slots ``decode_nbest`` left unused
            (length 0) score as the empty transcript: mask them with ``nbest.scores == -inf``
        """
        if self._time_major:
            logits = logits.transpose(1, 0)
        hypotheses_lengths = empty_marker_as_empty(hypotheses, hypotheses_lengths)
        return self._decoder.score_device(logits, hypotheses, hypotheses_lengths, logits_lengths,
                                          from_logits=not self._after_logsoftmax).cpu()

    def align(self, logits, hypotheses, hypotheses_lengths, logits_lengths=None):
        """Timestamps of N transcripts per utterance: the best-path (Viterbi) alignment of each (utterance, hypothesis) pair,
        each token's frame span, word spans and the best path's log-probability, on the GPU.  The utterance's frames are
        read once for all of its hypotheses.  Times are frames: converting them to seconds takes the model's frame shift,
        which the decoder does not know.

        :param logits: as for ``decode`` (``time_major``, ``after_logsoftmax`` and ``blank_idx`` apply)
        :param hypotheses: ``(B, N, max length)`` int32 / int64 labels, zero padded (``decode_nbest``'s
            ``decoded_targets`` as they come), or ``(B, max length)`` for one hypothesis per utterance (``decode`` /
            ``decode_greedy``'s ``decoded_targets``)
        :param hypotheses_lengths: ``(B, N)`` or ``(B,)`` to match; the single symbol ``-1`` with length 1 (``decode``'s
            empty result) is the empty hypothesis, and so are the slots ``decode_nbest`` left unused (length 0): mask
            them with ``nbest.scores == -inf``
        :param logits_lengths: ``(B,)`` or ``None`` (all frames)
        :return: ``AlignmentResults(alignments [B, N, T] int64, token_starts [B, N, Lmax] int64, token_ends [B, N, Lmax]
            int64, path_scores [B, N] float64, word_spans)`` -- CPU tensors.  ``alignments`` holds the label id of every
            frame on the best path (``-100`` past the utterance's frames), as ``get_alignment_3d`` does; token ``k`` of a
            hypothesis covers the frames ``[token_starts, token_ends)`` (``-1`` past its length); ``path_scores`` is the
            best path's log-probability, ``<= score`` (the sum over all paths).  An infeasible hypothesis (more labels
            and repeats than frames) has ``-inf`` and spans of ``-1``.  ``word_spans[b][n]`` is a list of ``(word,
            start_frame, end_frame)``, words being runs of tokens between ``" "`` labels; ``None`` without ``labels``.
            ``Lmax`` is the width of ``hypotheses``; a width past the aligner's limit (1023) is cut to the longest
            hypothesis
        """
        if self._time_major:
            logits = logits.transpose(1, 0)
        if hypotheses.dim() == 2:                       # one hypothesis per utterance: decode's / decode_greedy's result
            hypotheses, hypotheses_lengths = hypotheses[:, None], hypotheses_lengths.reshape(-1, 1)
        hypotheses_lengths = empty_marker_as_empty(hypotheses, hypotheses_lengths)
        if hypotheses.dim() == 3 and hypotheses.size(2) > 0 and hypotheses_lengths.shape == hypotheses.shape[:2]:
            if hypotheses.size(2) > ALIGN_MAX_TARGETS and hypotheses_lengths.numel():
                hypotheses = hypotheses[:, :, :max(int(hypotheses_lengths.max()), 0)]
        aligned, starts, ends, path_scores = (t.cpu() for t in self._decoder.align_device(
            logits, hypotheses, hypotheses_lengths, logits_lengths, from_logits=not self._after_logsoftmax))
        spans = None
        if self._labels:
            B, N = path_scores.shape
            hyps, lens = hypotheses.cpu().tolist(), hypotheses_lengths.cpu().tolist()
            s0, s1 = starts.tolist(), ends.tolist()
            spans = [[word_spans(hyps[b][n][:lens[b][n]], s0[b][n], s1[b][n], self._labels) for n in range(N)]
                     for b in range(B)]
        return AlignmentResults(aligned, starts, ends, path_scores, spans)

    def errors(self, hypotheses, hypotheses_lengths, references, references_lengths, *, level="word"):
        """Word or token errors of N transcripts per utterance against the utterance's reference, on the GPU: the risk
        of minimum word error rate training and the counts behind WER and CER.  ``errors`` is the least number of unit
        substitutions, insertions (a hypothesis unit with no reference counterpart) and deletions (a reference unit the
        hypothesis misses) that turn the reference into the hypothesis, each costing 1.  The split is that of the
        least-errors alignment with the most substitutions; tools with weighted costs (sclite) can split the same total
        differently.

        :param hypotheses: ``(B, N, max length)`` int32 / int64 labels (``decode_nbest``'s ``decoded_targets`` as they
            come), or ``(B, max length)`` for one hypothesis per utterance (``decode`` / ``decode_greedy``'s
            ``decoded_targets``)
        :param hypotheses_lengths: ``(B, N)`` or ``(B,)`` to match; the single symbol ``-1`` with length 1 (``decode``'s
            empty result) is the empty hypothesis, and so are the slots ``decode_nbest`` left unused (length 0): mask
            them with ``nbest.scores == -inf``
        :param references: ``(B, max length)`` int32 / int64 labels, e.g. ``CTCLoss``'s ``targets``
        :param references_lengths: ``(B,)``, e.g. ``targets_lengths``
        :param level: ``"word"``: units are words, maximal runs of labels other than ``" "`` (which ``labels`` must
            hold), two words being equal iff they are the same labels; ``"token"``: every label is a unit (CER when the
            labels are characters)
        :return: ``ErrorCounts(errors, substitutions, insertions, deletions, reference_units)`` -- CPU int64 tensors,
            ``(B, N)`` each (``N = 1`` for the two-dimensional form) and ``reference_units`` ``(B,)``, the number of
            reference units.  WER is ``errors.sum() / reference_units.sum()`` over a corpus; ``errors / reference_units``
            per utterance.  A length outside ``[0, width]`` raises ``ValueError`` (CPU lengths) or gives ``-1`` counts
            for its pairs (CUDA lengths)
        """
        if level not in ("word", "token"):
            raise ValueError("level must be \"word\" or \"token\", got %r" % (level,))
        out = self._decoder.errors_device(hypotheses, hypotheses_lengths, references, references_lengths,
                                          words=level == "word")
        return ErrorCounts(*(t.cpu() for t in out))

    def decode_greedy(self, logits, logits_lengths=None):
        """
        :param logits: ``(T, B, V)`` if ``time_major`` else ``(B, T, V)``; CPU or CUDA tensor
        :param logits_lengths: ``(B,)`` or ``None`` (decode all frames)
        :return: ``DecoderResults(decoded_targets [B,T] int64 zero padded, decoded_targets_lengths [B]
            int64, decoded_sentences list[str])`` -- CPU tensors, as in the reference
        """
        if self._time_major:
            logits = logits.transpose(1, 0)
        decoded_targets, decoded_targets_lengths = self._decoder.decode_greedy(
            logits_=logits, logits_lengths_=logits_lengths)
        decoded_sentences = self._sentences(decoded_targets, decoded_targets_lengths)
        return DecoderResults(decoded_targets, decoded_targets_lengths, decoded_sentences)

    def _sentences(self, targets, lengths):
        # src/decoders/ctc_decoder.cpp:212-220: concatenate labels; "" for every utterance without labels
        if not self._labels:
            return [""] * targets.size(0)
        rows, lens = targets.tolist(), lengths.tolist()
        return ["".join(self._labels[i] for i in row[:n] if i >= 0) for row, n in zip(rows, lens)]

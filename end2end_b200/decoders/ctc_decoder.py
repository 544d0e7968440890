"""CTCDecoder -- CTC decoding on the GPU behind the reference's decoder class
(pytorch_end2end/decoders/ctc_decoder.py:25-149).

* greedy: ``decode`` with ``beam_width == 1`` and ``decode_greedy`` (decoders/ctc_decoder.py:92-93, 117-149;
  src/decoders/ctc_decoder.cpp:443-490);
* prefix beam search WITHOUT a language model: ``decode`` with ``beam_width > 1`` and no ``lm_path``
  (decoders/ctc_decoder.py:76-115; src/decoders/ctc_decoder.cpp:153-198, 353-441) -- SURVEY.md 8(f3);
* the N best prefixes of that search with their scores: ``decode_nbest``, for rescoring with any language model on the
  host (N-best rescoring).

KenLM decoding (``lm_path``) stays the reference's CPU code and is out of scope; asking for it here raises
``NotImplementedError`` instead of silently decoding without the model.
"""
from collections import namedtuple

import torch

from ..engine import CTCBeamEngine


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

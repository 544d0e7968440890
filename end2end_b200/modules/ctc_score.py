"""CTCScore -- the CTC log-likelihood of N hypotheses per utterance as a differentiable module, for N-best sequence
training: decode a list (``CTCDecoder.decode_nbest``), score it here, turn the scores into the objective (a softmax over
the list weighted by each hypothesis's risk, for minimum word error rate training) and ``backward`` into the logits.
The risk function and the renormalisation are the caller's; INTEGRATION.md shows them."""
import torch.nn as nn

from ..engine import CTCBeamEngine
from ..functions.ctc_score import CTCScoreFunction
from ..utils.hypotheses import empty_marker_as_empty


class CTCScore(nn.Module):
    """
    ``log p(hypothesis | logits)`` of N transcripts per utterance, with its gradient, on NVIDIA B200.

    :param blank_idx: id of the blank label, default ``0``
    :param after_logsoftmax: the input already went through log-softmax (else: raw network outputs, log-softmax fused)
    :param time_major: logits are ``(T, B, V)`` instead of ``(B, T, V)``
    """

    def __init__(self, blank_idx=0, after_logsoftmax=False, time_major=False):
        super().__init__()
        self._blank_idx = blank_idx
        self._after_logsoftmax = after_logsoftmax
        self._time_major = time_major
        self._engine = CTCBeamEngine(blank_idx, 1)

    def forward(self, logits, hypotheses, hypotheses_lengths, logits_lengths=None):
        """
        :param logits: ``(T, B, V)`` if ``time_major`` else ``(B, T, V)``, float32 / float64 / bfloat16 / float16, CPU or
            CUDA
        :param hypotheses: ``(B, N, max length)`` int32 / int64 labels, zero padded; ``decode_nbest``'s
            ``decoded_targets`` as they come
        :param hypotheses_lengths: ``(B, N)``; the single symbol ``-1`` with length 1 (``decode``'s empty result) is the
            empty hypothesis
        :param logits_lengths: ``(B,)`` or ``None`` (all frames)
        :return: ``(B, N)`` float64 on the logits' device: ``CTCDecoder.score``'s values, with a graph to the logits.  The
            gradient is the derivative of the score: ``g * gamma`` for log-probabilities, ``g * (gamma - softmax)`` for
            raw logits, 0 in padding frames (not ``CTCLoss``'s ``exp(lp) - gamma`` convention).  An infeasible
            hypothesis scores ``-inf`` and contributes nothing to the gradient; mask unused ``decode_nbest`` slots
            (``scores == -inf`` there) out of the objective, and their zero weight skips them in the backward
        """
        if self._time_major:
            logits = logits.permute(1, 0, 2)
        hypotheses_lengths = empty_marker_as_empty(hypotheses, hypotheses_lengths)
        return CTCScoreFunction.apply(self._engine, logits, hypotheses, hypotheses_lengths, logits_lengths,
                                      not self._after_logsoftmax)

"""MWERLoss -- minimum word error rate training over an N-best list (Prabhavalkar et al., 2018) as a criterion shaped
like ``CTCLoss``: decode a list from the model (``CTCDecoder.decode_nbest`` / ``CTCBeamEngine.decode_nbest_device``),
pass it here with the reference transcripts, ``backward`` into the logits.

For utterance b the list U_b is the slots in ``hypotheses_mask`` whose score ``s_bn = log p(hyp_bn | x_b)`` is finite;
``p_bn`` is the softmax of ``score_scale * s_bn`` over U_b and the loss is the expected risk ``R_b = sum_{n in U_b} p_bn
r_bn``, the risk being the word (``level="word"``) or token (``level="token"``) errors of each hypothesis against the
reference, counted on the GPU (``CTCBeamEngine.errors_device``).  ``d loss_b / d s_bn = score_scale p_bn (r_bn - R_b)``:
the baseline is built in.  The gradient reaches the logits through the CTC score's derivative (``CTCScore``'s
convention).  Everything runs on the GPU (``functions/mwer.py``); for a risk of your own call ``MWERFunction`` directly.
"""
import math

import torch.nn as nn

from ..engine import CTCBeamEngine
from ..functions.mwer import MWERFunction
from ..utils.hypotheses import empty_marker_as_empty


class MWERLoss(nn.Module):
    """
    Minimum word error rate over an N-best list, on NVIDIA B200.

    :param labels: the label strings (word level needs the ``" "`` label, which separates words)
    :param blank_idx: id of the blank label, default ``0``
    :param level: ``"word"`` (word errors, WER's numerator) or ``"token"`` (every label, CER's for characters)
    :param score_scale: ``lambda`` of the list's softmax ``exp(lambda s)``, finite and > 0
    :param size_average: average the loss over the batch (only if ``reduce`` is True)
    :param reduce: sum (or average) the per-utterance losses; ``None`` returns the ``(batch_size,)`` tensor
    :param after_logsoftmax: the input already went through log-softmax (else: raw network outputs)
    :param time_major: logits are ``(T, B, V)`` instead of ``(B, T, V)``
    """

    def __init__(self, labels=None, blank_idx=0, level="word", score_scale=1.0, size_average=None, reduce=None,
                 after_logsoftmax=False, time_major=False):
        super().__init__()
        if level not in ("word", "token"):
            raise ValueError("level must be 'word' or 'token', got %r" % (level,))
        score_scale = float(score_scale)
        if not math.isfinite(score_scale) or score_scale <= 0.0:
            raise ValueError("score_scale must be finite and > 0, got %r" % score_scale)
        self._engine = CTCBeamEngine(blank_idx, 1, labels)
        if level == "word" and self._engine.space_idx < 0:
            raise ValueError("word level needs a \" \" label to separate words; the labels have none")
        self._level = level
        self._score_scale = score_scale
        self._reduce = reduce
        self._size_average = size_average
        self._after_logsoftmax = after_logsoftmax
        self._time_major = time_major

    def forward(self, logits, hypotheses, hypotheses_lengths, logits_lengths, targets, targets_lengths,
                hypotheses_mask=None):
        """
        :param logits: ``(T, B, V)`` if ``time_major`` else ``(B, T, V)``, float32 / float64 / bfloat16 / float16, CPU or
            CUDA
        :param hypotheses: ``(B, N, max length)`` int32 / int64 labels; ``decode_nbest``'s ``decoded_targets`` as they
            come (the single symbol ``-1`` with length 1 is the empty hypothesis)
        :param hypotheses_lengths: ``(B, N)``
        :param logits_lengths: ``(B,)`` or ``None`` (all frames)
        :param targets: ``(B, max reference length)``, the reference transcripts (``CTCLoss``'s targets)
        :param targets_lengths: ``(B,)``
        :param hypotheses_mask: ``(B, N)`` bool, the slots in the list, or ``None`` (every slot); for ``decode_nbest``
            lists pass ``scores > -inf`` so that slots the final beam did not fill stay out.  Host-resident lengths and
            labels are checked for every slot, masked or not (``ValueError``); device-resident ones out of range in a
            masked-out slot change nothing
        :return: float64 losses ``(B,)`` if ``reduce`` is falsy, else a 0-dim tensor, on the logits' device
        """
        if self._time_major:
            logits = logits.permute(1, 0, 2)
        hypotheses_lengths = empty_marker_as_empty(hypotheses, hypotheses_lengths)
        risk = self._engine.errors_device(hypotheses, hypotheses_lengths, targets, targets_lengths,
                                          words=self._level == "word")[0]
        reduction = None
        if self._reduce:
            reduction = "mean" if self._size_average else "sum"
        return MWERFunction.apply(self._engine, logits, hypotheses, hypotheses_lengths, logits_lengths, risk,
                                  hypotheses_mask, self._score_scale, not self._after_logsoftmax, reduction)

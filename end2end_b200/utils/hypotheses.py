"""Hypothesis lists as the decoders return them, made ready for the scorer and the aligner."""
import torch


def empty_marker_as_empty(hypotheses, hypotheses_lengths):
    """``decode``'s empty result, the single symbol ``-1`` with length 1, as the empty hypothesis (length 0); other
    lengths unchanged.  ``hypotheses`` ``(B, N, max length)``, ``hypotheses_lengths`` ``(B, N)``; anything else is
    returned as it is.  An element-wise select: no synchronisation."""
    if hypotheses.dim() == 3 and hypotheses.size(2) > 0 and hypotheses_lengths.shape == hypotheses.shape[:2]:
        dev = hypotheses_lengths.device
        empty = (hypotheses[:, :, 0].to(dev) == -1) & (hypotheses_lengths == 1)
        hypotheses_lengths = torch.where(empty, torch.zeros_like(hypotheses_lengths), hypotheses_lengths)
    return hypotheses_lengths

"""Viterbi forced alignment on the GPU behind the reference's ``get_alignment_3d``
(pytorch_end2end/utils/alignment.py:109-138; SURVEY.md 8(f2)).

The reference runs one numba-jitted function per utterance on a Python thread
(``_get_alignment_ctc_1d`` :50-106 for CTC, ``_get_alignment_asg_1d`` :9-47 for ASG); here the whole
batch is one kernel launch (``e2e_ctc_viterbi_align_device``, csrc/ctc_viterbi.cu), bit-exact with the
reference: the same fp64 max-plus recursion, comparison order and window.  No CPU fallback.
"""
import ctypes

import torch

from .. import _lib
from ..engine import _check_logits, _dense3, _desc, _index_args, _on_device, _ptr, _require_cuda, _stream


def get_alignment_3d_device(log_probs, targets, logits_lengths, targets_lengths, is_ctc=True, blank_idx=0):
    """Device tensors in, device int64 ``[B, T]`` out (no synchronisation): the label id of every frame on the best
    path, ``-100`` past the utterance's frames."""
    _require_cuda()
    L = _lib.load()
    lp = log_probs.detach()
    B, T, _ = _check_logits(lp, blank_idx, "log_probs")
    if targets.dim() != 2 or targets.size(0) != B:
        raise ValueError("targets must be [batch, max_target_length]")
    if not lp.is_cuda:
        lp = lp.cuda()
    dev = lp.device
    if not _dense3(lp):
        lp = lp.contiguous()
    targets, ll, tl = _index_args(targets, logits_lengths, targets_lengths, dev)
    d = _desc(lp, blank_idx, targets, ll, False)
    with _on_device(dev):
        n = L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), 1 if is_ctc else 0)
        if n == 0:   # the shape is valid (checked above): the lattice or the alphabet is beyond the build's limits
            raise NotImplementedError(L.e2e_last_error_string().decode("utf-8", "replace"))
        ws = torch.empty(n, dtype=torch.uint8, device=dev)
        out = torch.empty(B, T, dtype=torch.int64, device=dev)
        _lib.check(L.e2e_ctc_viterbi_align_device(ctypes.byref(d), 1 if is_ctc else 0, _ptr(lp), _ptr(targets), _ptr(ll),
                                                  _ptr(tl), _ptr(out), _ptr(ws), ws.numel(), _stream(dev)))
    return out


def get_alignment_3d(log_probs, targets, logits_lengths, targets_lengths, is_ctc=True):
    """Same signature and result as the reference (alignment.py:109-138): a CPU ``torch.long`` tensor
    ``[batch, frames]`` filled with ``-100`` past every utterance's frames.  ``log_probs`` may live on either device."""
    return get_alignment_3d_device(log_probs, targets, logits_lengths, targets_lengths, is_ctc=is_ctc).cpu()

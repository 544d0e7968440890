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
from ..engine import _DTYPES, _ITYPES, _as_index, _dense3, _on_device, _ptr, _require_cuda, _stream


def get_alignment_3d_device(log_probs, targets, logits_lengths, targets_lengths, is_ctc=True, blank_idx=0):
    """Device tensors in, device int64 ``[B, T]`` out (no synchronisation): the label id of every frame on the best
    path, ``-100`` past the utterance's frames."""
    _require_cuda()
    L = _lib.load()
    lp = log_probs.detach()
    if lp.dim() != 3:
        raise ValueError("log_probs must be [batch, frames, alphabet]")
    if lp.dtype not in _DTYPES:
        raise TypeError("unsupported dtype %s" % lp.dtype)
    if not lp.is_cuda:
        lp = lp.cuda()
    dev = lp.device
    if not _dense3(lp):
        lp = lp.contiguous()
    B, T, V = lp.shape
    if B < 1 or T < 1 or V < 1:
        raise ValueError("empty log_probs %s" % (tuple(lp.shape),))
    if targets.dim() != 2 or targets.size(0) != B:
        raise ValueError("targets must be [batch, max_target_length]")
    if not 0 <= blank_idx < V:
        raise ValueError("blank_idx %d outside the alphabet [0,%d)" % (blank_idx, V))
    targets = _as_index(targets, dev, "targets")
    if targets.size(1) > 0 and targets.stride(1) != 1:
        targets = targets.contiguous()
    ll = _as_index(logits_lengths, dev, "logits_lengths").contiguous()
    tl = _as_index(targets_lengths, dev, "targets_lengths").contiguous()
    if ll.dtype != tl.dtype:
        ll, tl = ll.to(torch.int64), tl.to(torch.int64)
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, targets.size(1)
    d.blank_idx, d.dtype = int(blank_idx), _DTYPES[lp.dtype]
    d.targets_itype, d.lengths_itype = _ITYPES[targets.dtype], _ITYPES[ll.dtype]
    d.logits_stride_b, d.logits_stride_t = lp.stride(0), lp.stride(1)
    d.targets_stride_b = targets.stride(0) if targets.size(1) > 0 else 0
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

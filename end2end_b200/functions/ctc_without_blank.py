"""CTC without blank on the GPU behind the reference's Function
(pytorch_end2end/functions/ctc_without_blank.py:120-143; SURVEY.md 8(f4)).

The reference moves everything to numpy and runs one numba-jitted ``_ctc_without_blank_loss`` (:13-88) per
utterance on a Python thread (:91-117); here the batch is one kernel launch
(``e2e_ctc_noblank_fwd_bwd_device``, csrc/ctc_noblank.cu).  No CPU fallback.
"""
import ctypes

import torch
from torch.autograd import Function

from .. import _lib
from ..engine import _check_logits, _dense3, _desc, _index_args, _on_device, _ptr, _require_cuda, _stream


def ctc_without_blank_3d_loss(log_probs, targets, logits_lengths, targets_lengths, space_idx=-1):
    """(losses [B], grads [B,T,V]) on ``log_probs``' CUDA device, in its dtype: the device counterpart of the reference's
    ``_ctc_without_blank_3d_loss`` (:91-117).  ``grads`` is zero past every utterance's frames."""
    _require_cuda()
    L = _lib.load()
    lp = log_probs.detach()
    B, T, V = _check_logits(lp, None, "log_probs")
    if targets.dim() != 2 or targets.size(0) != B:
        raise ValueError("targets must be [batch, max_target_length]")
    if not -1 <= space_idx < V:
        raise ValueError("space_idx %d outside [-1,%d)" % (space_idx, V))
    if not lp.is_cuda:
        lp = lp.cuda()
    dev = lp.device
    if not _dense3(lp):
        lp = lp.contiguous()
    targets, ll, tl = _index_args(targets, logits_lengths, targets_lengths, dev)
    d = _desc(lp, 0, targets, ll, False)
    with _on_device(dev):
        n = L.e2e_ctc_noblank_workspace_bytes(ctypes.byref(d))
        if n == 0:   # the shape is valid (checked above): the lattice or the alphabet is beyond the build's limits
            raise NotImplementedError(L.e2e_last_error_string().decode("utf-8", "replace"))
        ws = torch.empty(n, dtype=torch.uint8, device=dev)
        losses = torch.empty(B, dtype=lp.dtype, device=dev)
        grads = torch.empty_strided(lp.size(), lp.stride(), dtype=lp.dtype, device=dev)
        d.grads_stride_b, d.grads_stride_t = grads.stride(0), grads.stride(1)
        _lib.check(L.e2e_ctc_noblank_fwd_bwd_device(ctypes.byref(d), int(space_idx), _ptr(lp), _ptr(targets), _ptr(ll), _ptr(tl),
                                                    _ptr(losses), _ptr(grads), _ptr(ws), ws.numel(), _stream(dev)))
    return losses, grads


class CTCWithoutBlankLossFunction(Function):
    """``apply(log_probs, targets, logits_lengths, targets_lengths, space_idx=-1) -> losses [B]`` (reference :120-143).
    The gradient block is produced in forward (as the reference does) and scaled by ``grad_output`` in backward."""

    @staticmethod
    def forward(ctx, log_probs, targets, logits_lengths, targets_lengths, space_idx=-1):
        losses, grads = ctc_without_blank_3d_loss(log_probs, targets, logits_lengths, targets_lengths, space_idx)
        on_host = not log_probs.is_cuda          # results live where the input lives
        ctx.grads = grads.cpu() if on_host else grads
        return losses.cpu() if on_host else losses

    @staticmethod
    def backward(ctx, grad_output):
        scale = grad_output.to(ctx.grads.device).reshape(-1, 1, 1)
        return ctx.grads * scale, None, None, None, None

"""CTCLoss -- same constructor and forward signature as the reference's module
(pytorch_end2end/modules/ctc_loss.py:15-75), computed by the sm_100a engine.

Mapping of the reference's forward (modules/ctc_loss.py:25-57) onto the fused path:

* ``after_logsoftmax=False``: the reference runs ``F.log_softmax`` as a separate autograd op; here
  the raw logits go straight to the engine (``from_logits``), which fuses the row log-softmax into
  its kernels and returns the gradient with respect to the logits.
* ``time_major=True``: the reference permutes a view; here the permuted view's strides are handed
  to the kernels, which read and write the [T,B,V] tensor in place.
* ``reduce`` / ``size_average``: ``mean()`` iff both are set, ``sum()`` iff only ``reduce`` is set,
  per-utterance losses otherwise -- the reduction runs in the engine (fp64 accumulation) and its
  scale is folded into the gradient kernel.
"""
import torch.nn as nn

from ..engine import CTCLossEngine
from ..functions.forward_backward import ForwardBackwardLossFunction


class ForwardBackwardLossBase(nn.Module):
    def __init__(self, size_average=None, reduce=None, after_logsoftmax=False, time_major=False, blank_idx=0):
        super().__init__()
        self._blank_idx = blank_idx
        self._reduce = reduce
        self._size_average = size_average
        self._after_logsoftmax = after_logsoftmax
        self._time_major = time_major
        self._engine = None

    def forward(self, logits, targets, logits_lengths, targets_lengths):
        """
        :param logits: Float/Double/BFloat16/Half tensor (network output) of shape
            ``(sequence_length, batch_size, alphabet_size)`` if ``time_major`` is True,
            else ``(batch_size, sequence_length, alphabet_size)``
        :param targets: ``(batch_size, targets_sequence_length)``
        :param logits_lengths: ``(batch_size,)``
        :param targets_lengths: ``(batch_size,)``
        :return: losses of shape ``(batch_size,)`` if ``reduce`` is falsy, else a 0-dim tensor
        """
        if self._time_major:
            logits = logits.permute(1, 0, 2)
        reduction = None
        if self._reduce:
            reduction = "mean" if self._size_average else "sum"
        return ForwardBackwardLossFunction.apply(self._engine, logits, targets, logits_lengths,
                                                 targets_lengths, not self._after_logsoftmax, reduction)

    def graphed(self, logits, targets, logits_lengths, targets_lengths, workspace=None):
        """SURVEY 8(f1): the whole step of this criterion (``forward`` + the ``backward`` of ``loss.sum()``) for
        device tensors at FIXED addresses, captured once; see :class:`GraphedCTCStep`.  A training loop whose
        batches are copied into the same buffers then pays one driver call per step instead of the Python
        autograd round trip (reference: modules/ctc_loss.py:37-57 + functions/forward_backward.py:6-35)."""
        if self._time_major:
            logits = logits.permute(1, 0, 2)
        B = logits.size(0)
        mean = bool(self._reduce and self._size_average)
        scale = 1.0 / B if mean else 1.0
        step = self._engine.graphed_step(logits, targets, logits_lengths, targets_lengths,
                                         from_logits=not self._after_logsoftmax, grad_scale=scale,
                                         reduce_scale=scale if self._reduce else None, workspace=workspace)
        return GraphedCTCStep(step, self._time_major, bool(self._reduce))


class GraphedCTCStep:
    """Forward + backward of a criterion captured into one CUDA graph (``criterion.graphed(...)``).

    ``replay()`` enqueues the step on the current stream and returns ``(loss, grad)``: the loss the module's
    ``forward`` would return (per-utterance ``[B]``, or the 0-dim sum / mean) and ``d loss.sum() / d logits`` in
    the layout of ``logits`` -- what ``loss.backward()`` leaves in ``logits.grad`` for an upstream gradient of one.
    Both are views of buffers owned by the step: they are overwritten by the next ``replay()``."""

    def __init__(self, step, time_major, reduced):
        self._step = step
        self.loss = step.reduced if reduced else step.losses
        self.grad = step.grads.permute(1, 0, 2) if time_major else step.grads

    def replay(self):
        self._step.launch()
        return self.loss, self.grad


class CTCLoss(ForwardBackwardLossBase):
    """
    Criterion to compute CTC Loss (Graves et al., 2006) on NVIDIA B200.

    :param size_average: average the loss over the batch (only if ``reduce`` is True)
    :param reduce: sum (or average) the per-utterance losses; ``None`` returns the ``(batch_size,)`` tensor
    :param after_logsoftmax: the input already went through log-softmax (else: raw network outputs)
    :param time_major: logits are ``(T, B, V)`` instead of ``(B, T, V)``
    :param blank_idx: id of the blank label, default ``0``

    With ``after_logsoftmax=True`` the gradient keeps the reference engine's convention, ``exp(lp) - posterior`` on every
    frame (``exp(lp)`` in padding rows); ``CTCScore``'s gradient is the plain derivative of the score instead.
    """

    def __init__(self, size_average=None, reduce=None, after_logsoftmax=False, time_major=False, blank_idx=0):
        super().__init__(size_average, reduce, after_logsoftmax, time_major, blank_idx)
        self._engine = CTCLossEngine(self._blank_idx)

"""Autograd bridge of the N-hypothesis CTC score: ``s[b, n] = log p(hypothesis n | x_b)`` with its gradient, for N-best
sequence training (minimum word error rate and other objectives over the list).

``forward`` is one K9 launch (``CTCBeamEngine.score_device``: the same values, bit for bit); ``backward`` is K10 and its
row kernel (``score_backward_device``) with ``grad_output`` as the per-hypothesis weight ``g``:
``sum_n g[b,n] gamma_bn(t,v)`` for log-probabilities, ``sum_n g[b,n] (gamma_bn(t,v) - softmax(x_bt)_v)`` for raw logits,
0 past each utterance's frames.  That is the derivative of the score, not ``CTCLoss``'s convention on log-probabilities
(``exp(lp) - gamma``, ``exp(lp)`` in padding rows).  Only the logits get a gradient.  CPU logits run on the current CUDA
device; the scores and the gradient come back on the logits' device.

``apply(engine, logits, hyps, hyp_lengths, logits_lengths, from_logits)``
"""
from torch.autograd import Function
from torch.autograd.function import once_differentiable


class CTCScoreFunction(Function):
    @staticmethod
    def forward(ctx, engine, logits, hyps, hyp_lengths, logits_lengths=None, from_logits=False):
        """
        :param engine: ``end2end_b200.engine.CTCBeamEngine`` (its ``blank_idx`` is the blank)
        :param logits: ``[B, T, V]`` (any batch / time strides)
        :param hyps: ``[B, N, Lmax]`` int32 / int64
        :param hyp_lengths: ``[B, N]``
        :param logits_lengths: ``[B]`` or ``None`` (all frames)
        :return: ``[B, N]`` float64 on the logits' device
        """
        ctx.engine, ctx.from_logits = engine, from_logits
        ctx.save_for_backward(logits, hyps, hyp_lengths, logits_lengths)
        scores = engine.score_device(logits, hyps, hyp_lengths, logits_lengths, from_logits)
        return scores.to(logits.device)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        logits, hyps, hyp_lengths, logits_lengths = ctx.saved_tensors
        grad = None
        if ctx.needs_input_grad[1]:
            grad = ctx.engine.score_backward_device(logits, hyps, hyp_lengths, grad_output, logits_lengths, ctx.from_logits)
            grad = grad.to(logits.device)
        return None, grad, None, None, None, None

"""Autograd bridge of minimum word error rate (MWER) training over an N-best list (Prabhavalkar et al., 2018).

For utterance b with hypotheses n: the list U_b is the slots with ``mask[b, n]`` true whose score
``s_bn = log p(hyp_bn | x_b)`` is finite; ``p_bn = exp(lambda s_bn) / sum_{m in U_b} exp(lambda s_bm)`` with ``lambda =
score_scale``; ``loss_b = R_b = sum_{n in U_b} p_bn r_bn`` for the risk ``r``.  ``d loss_b / d s_bn = lambda p_bn (r_bn -
R_b)``: the mean-risk baseline is part of the loss, so nothing needs detaching.  The gradient with respect to the input is
``CTCScore``'s with ``g_bn = w_b lambda p_bn (r_bn - R_b)``, ``w_b`` the upstream gradient of ``loss_b``.  An empty list
gives loss 0 and zero rows; equal risks over the list (a single slot included) give exactly zero rows; a NaN score (a bad
device-resident length or label) or a negative / NaN in-list risk gives that utterance a NaN loss and NaN rows.  The loss
is float64, as ``CTCScore``'s scores are.

``forward`` runs K12a (K10's alpha pass, the scores and checkpoints kept in a state buffer) and K12b (the weights);
``backward`` runs K12c (K10's beta pass from those checkpoints) and the row kernel.  The backward consumes the state's
checkpoints, so a second backward through a retained graph runs the forward kernels again first.  Under ``no_grad`` the
state goes with ``ctx``.  CPU logits run on the current CUDA device; the loss and the gradient come back on the logits'
device.

``apply(engine, logits, hyps, hyp_lengths, logits_lengths, risk, mask, score_scale, from_logits, reduction)``
    risk:      ``[B, N]``, any real dtype (word or token errors, or the caller's own risk)
    mask:      ``[B, N]`` bool or ``None`` (every slot)
    reduction: ``None`` -> losses ``[B]``; ``"sum"`` / ``"mean"`` (over utterances) -> a 0-dim tensor
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable


class MWERFunction(Function):
    @staticmethod
    def forward(ctx, engine, logits, hyps, hyp_lengths, logits_lengths, risk, mask=None, score_scale=1.0,
                from_logits=False, reduction=None):
        if reduction not in (None, "sum", "mean"):
            raise ValueError("reduction must be None, 'sum' or 'mean', got %r" % (reduction,))
        ctx.engine, ctx.from_logits, ctx.reduction, ctx.score_scale = engine, from_logits, reduction, score_scale
        # saved tensors: modifying one in place before the backward raises instead of mixing new values with old
        # checkpoints
        ctx.save_for_backward(logits, hyps, hyp_lengths, risk, mask, logits_lengths)
        losses, _, ctx.state = engine.mwer_forward_device(logits, hyps, hyp_lengths, risk, mask, logits_lengths,
                                                          from_logits, score_scale)
        ctx.fresh = True
        if reduction == "sum":
            losses = losses.sum()
        elif reduction == "mean":
            losses = losses.mean()
        return losses.to(logits.device)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        logits, hyps, hyp_lengths, risk, mask, logits_lengths = ctx.saved_tensors
        from_logits, score_scale = ctx.from_logits, ctx.score_scale
        grad = None
        if ctx.needs_input_grad[1]:
            if not ctx.fresh:   # a second backward through a retained graph: the first consumed the checkpoints
                ctx.engine.mwer_forward_device(logits, hyps, hyp_lengths, risk, mask, logits_lengths, from_logits,
                                               score_scale, state=ctx.state)
            ctx.fresh = False
            B = logits.size(0)
            dev = ctx.state.device
            w = grad_output.detach().to(dev, torch.float64)
            if ctx.reduction is not None:
                w = (w / B if ctx.reduction == "mean" else w).reshape(1).expand(B)
            grad = ctx.engine.mwer_backward_device(logits, hyps, hyp_lengths, w, ctx.state, logits_lengths, from_logits)
            grad = grad.to(logits.device)
        return None, grad, None, None, None, None, None, None, None, None

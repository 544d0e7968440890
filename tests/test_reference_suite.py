"""The test cases of the reference's own unittest files, run against the drop-in ``pytorch_end2end`` package
(SURVEY.md section 4: tests/test_ctc.py:22-191 -- five warp-ctc / TensorFlow known answers + gradcheck;
tests/test_ctc_decoder.py:44-166 -- greedy and prefix-beam known answers).

The cases' inputs and the reference's answers are stored in tests/golden/ (kat_loss.npz, f64.npz, kat_greedy.npz,
beam_kat_*.npz, written from the reference by the make_*golden.py scripts there), so the suite needs nothing outside
the repository.  The LM tests of the decoder file need KenLM + the reference's ARPA fixture and stay out
(north_star: KenLM decoding stays CPU code)."""
import os

import numpy as np
import pytest
import torch

from pytorch_end2end import CTCDecoder, CTCLoss

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gold(name):
    return np.load(os.path.join(GOLD, name + ".npz"))


def T(a):
    return torch.from_numpy(np.array(a))


def almost_equal(a, b):
    return round(abs(a - b), 5) == 0                 # unittest's assertAlmostEqual(places=5)


def test_reference_test_ctc_unmodified():
    """tests/test_ctc.py: run_grads (:22-66) on each known answer -- CTCLoss(reduce=True, size_average=False,
    after_logsoftmax=True, time_major=True) fed CPU and then CUDA log-probabilities, the cost equal to the expected
    value and on both devices -- and test_gradient (:168-191): gradcheck of CTCLoss(blank_idx=0) on the seed-678
    double fixture."""
    g = gold("kat_loss")
    for name in ("simple", "medium", "empty_label", "tf_1", "tf_2"):
        lp_tm = T(g[name + "_lp"]).permute(1, 0, 2).contiguous()
        tg, ll, tl = T(g[name + "_targets"]), T(g[name + "_ll"]), T(g[name + "_tl"])
        expected = float(g[name + "_expected"])
        crit = CTCLoss(reduce=True, size_average=False, after_logsoftmax=True, time_major=True,
                       blank_idx=int(g[name + "_blank"]))
        costs = []
        for dev in ("cpu", "cuda"):
            leaf = lp_tm.clone().to(dev).requires_grad_()
            cost = crit(leaf, tg, ll, tl)
            cost.backward()
            assert leaf.grad is not None and leaf.grad.shape == leaf.shape
            costs.append(cost.item())
            assert almost_equal(cost.item(), expected), (name, dev, cost.item(), expected)
        assert almost_equal(costs[0], costs[1]), (name, costs)
    f = gold("f64")
    x = T(f["x"]).requires_grad_()
    tg, ll, tl = T(f["targets"]), T(f["logits_lengths"]), T(f["targets_lengths"])
    crit = CTCLoss(blank_idx=0, time_major=False, after_logsoftmax=False)
    assert torch.autograd.gradcheck(crit, (x, tg, ll, tl), eps=1e-6, atol=1e-4)


def test_reference_test_ctc_decoder_unmodified():
    """tests/test_ctc_decoder.py: the greedy known answer (:44-59) and the three LM-free prefix-beam known answers
    (:86-166: greedy AND beam result of each case, beam width 20), on CPU and CUDA inputs."""
    g = gold("kat_greedy")
    cases = (("simple", "dc", None), ("sm", "", "beam_kat_sm"), ("probs_1", "ac'bdc", "beam_kat_1"),
             ("probs_2", "b'da", "beam_kat_2"))
    for name, greedy_want, beam_case in cases:
        ll = g[name + "_ll"]
        lengths = None if ll[0] < 0 else T(ll)
        labels = [str(s) for s in g[name + "_labels"]]
        dec = CTCDecoder(beam_width=1, blank_idx=int(g[name + "_blank"]), labels=labels, time_major=False)
        for dev in ("cpu", "cuda"):
            r = dec.decode(T(g[name + "_x"]).to(dev), lengths)
            assert r.decoded_sentences == [greedy_want], (name, dev, r.decoded_sentences)
            assert torch.equal(r.decoded_targets, T(g[name + "_targets"]))
            assert torch.equal(r.decoded_targets_lengths, T(g[name + "_lengths"]))
        if beam_case is None:
            continue
        z = gold(beam_case)
        beam_want = str(z["sentences"])
        assert str(z["labels"]).split("\x1f") == labels and int(z["beam"]) == 20
        dec = CTCDecoder(beam_width=20, after_logsoftmax=True, blank_idx=int(z["blank"]), labels=labels,
                         wip=float(z["wip"]))
        for dev in ("cpu", "cuda"):
            r = dec.decode(T(z["log_probs"]).to(dev), T(z["logits_lengths"]))
            assert r.decoded_sentences == [beam_want], (beam_case, dev, r.decoded_sentences)
            assert torch.equal(r.decoded_targets, T(z["targets"]))
            assert torch.equal(r.decoded_targets_lengths, T(z["targets_lengths"]))
    assert [str(gold(c)["sentences"]) for c in ("beam_kat_sm", "beam_kat_1", "beam_kat_2")] == ["a", "acdc", "b'a"]

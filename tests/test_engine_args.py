"""Argument errors of the Python entry points: each malformed input raises the same exception type, with a message that
names the argument, on the host before any device work.  Without a device the driver check is patched out
(``engine._CUDA_OK``), so a call that gets past its checks fails at its first CUDA call instead, with torch's
``RuntimeError``, which none of these cases expects."""
import pytest
import torch

B, T, V = 2, 10, 5
X = torch.randn(B, T, V)
TG, LL, TL = torch.ones(B, 4, dtype=torch.int64), torch.full((B,), T), torch.full((B,), 2)
HYPS, HL = torch.ones(B, 3, 4, dtype=torch.int64), torch.full((B, 3), 2)
REFS, RL = torch.ones(B, 5, dtype=torch.int32), torch.tensor([5, 0])
LABELS = ["_", " ", "a", "b", "c"]


def _max_alphabet():
    from end2end_b200 import _lib
    return _lib.limits().max_alphabet


def _max_targets():
    from end2end_b200 import _lib
    return _lib.limits().max_targets


@pytest.fixture
def engine(monkeypatch, lib_built):
    from end2end_b200 import engine
    monkeypatch.setattr(engine, "_CUDA_OK", True)
    return engine


# ------------------------------------------------------------------------------------------------- loss -------------
# (id, exception, key word of the message, blank_idx, arguments)
LOSS = [
    ("rank", ValueError, "logits", 0, lambda: (X[0], TG, LL, TL)),
    ("int_logits", TypeError, "dtype", 0, lambda: (X.to(torch.int32), TG, LL, TL)),
    ("empty_batch", ValueError, "empty", 0, lambda: (X[:0], TG[:0], LL[:0], TL[:0])),
    ("blank", ValueError, "blank_idx", 7, lambda: (X, TG, LL, TL)),
    ("targets_shape", ValueError, "targets", 0, lambda: (X, TG[:1], LL, TL)),
    ("logits_lengths_shape", ValueError, "length", 0, lambda: (X, TG, LL[:1], TL)),
    ("targets_lengths_shape", ValueError, "length", 0, lambda: (X, TG, LL, TL[:, None])),
    ("frames_high", ValueError, "logits_lengths", 0, lambda: (X, TG, torch.tensor([T + 1, T]), TL)),
    ("frames_low", ValueError, "logits_lengths", 0, lambda: (X, TG, torch.tensor([0, T]), TL)),
    ("targets_length_high", ValueError, "targets_lengths", 0, lambda: (X, TG, LL, torch.tensor([5, 2]))),
    ("targets_length_low", ValueError, "targets_lengths", 0, lambda: (X, TG, LL, torch.tensor([-1, 2]))),
    ("label_high", ValueError, "target labels", 0, lambda: (X, torch.full((B, 4), V), LL, TL)),
    ("label_low", ValueError, "target labels", 0, lambda: (X, torch.full((B, 4), -1), LL, TL)),
    ("width", NotImplementedError, "target length", 0,
     lambda: (X, torch.ones(B, _max_targets() + 1, dtype=torch.int64), LL, TL)),
    ("alphabet", NotImplementedError, "alphabet", 0, lambda: (torch.randn(1, 2, _max_alphabet() + 1), TG[:1], LL[:1], TL[:1])),
]


@pytest.mark.parametrize("method", ["step", "forward", "workspace_bytes"])
@pytest.mark.parametrize("case", LOSS, ids=[c[0] for c in LOSS])
def test_loss_argument_errors(engine, method, case):
    _, exc, word, blank, args = case
    with pytest.raises(exc, match=word):
        getattr(engine.CTCLossEngine(blank), method)(*args())


# --------------------------------------------------------------------------------------------- decoders -------------
# (id, exception, key word, engine arguments, logits, entry points); the greedy engine takes the blank only.
DECODERS = ("decode_greedy_device", "decode_device", "decode_nbest_device", "decode_greedy", "decode", "decode_nbest")
DECODE = [
    ("rank", ValueError, "logits", (0, 4), lambda: X[None], DECODERS),
    ("int_logits", TypeError, "dtype", (0, 4), lambda: X.to(torch.int32), DECODERS),
    ("empty_batch", ValueError, "empty", (0, 4), lambda: X[:0], DECODERS),
    ("blank", ValueError, "blank_idx", (7, 4), lambda: X, DECODERS),
    ("space", ValueError, "space", (0, 4, ["_"] * 6 + [" "]), lambda: X,
     ("decode_device", "decode_nbest_device", "decode", "decode_nbest")),
    ("beam_width", RuntimeError, "limits", (0, 257), lambda: X, ("decode_device", "decode_nbest_device")),
]


@pytest.mark.parametrize("case", DECODE, ids=[c[0] for c in DECODE])
def test_decoder_argument_errors(engine, case):
    _, exc, word, ctor, logits, methods = case
    for method in methods:
        eng = engine.CTCGreedyEngine(ctor[0]) if "greedy" in method else engine.CTCBeamEngine(*ctor)
        with pytest.raises(exc, match=word):
            getattr(eng, method)(logits(), LL)


def test_n_best_outside_the_beam(engine):
    for method in ("decode_nbest_device", "decode_nbest"):
        with pytest.raises(ValueError, match="n_best"):
            getattr(engine.CTCBeamEngine(0, 4), method)(X, LL, n_best=5)


# ------------------------------------------------------------------------------------- score, mwer, align -----------
# (id, exception, key word, blank_idx, (logits, hyps, hyp_lengths, logits_lengths))
SCORE = [
    ("rank", ValueError, "logits", 0, lambda: (X[0], HYPS, HL, None)),
    ("int_logits", TypeError, "dtype", 0, lambda: (X.to(torch.int32), HYPS, HL, None)),
    ("empty_batch", ValueError, "empty", 0, lambda: (X[:0], HYPS[:0], HL[:0], None)),
    ("blank", ValueError, "blank_idx", 7, lambda: (X, HYPS, HL, None)),
    ("hyps_shape", ValueError, "hyps", 0, lambda: (X, HYPS[:1], HL, None)),
    ("no_hypothesis", ValueError, "hyps", 0, lambda: (X, HYPS[:, :0], HL[:, :0], None)),
    ("hyp_lengths_shape", ValueError, "hyp_lengths", 0, lambda: (X, HYPS, HL[:, :2], None)),
    ("logits_lengths_shape", ValueError, "logits_lengths", 0, lambda: (X, HYPS, HL, LL[:1])),
    ("hyp_length_high", ValueError, "hyp_lengths", 0, lambda: (X, HYPS, torch.full((B, 3), 5), None)),
    ("hyp_length_low", ValueError, "hyp_lengths", 0, lambda: (X, HYPS, torch.full((B, 3), -1), None)),
    ("frames_high", ValueError, "logits_lengths", 0, lambda: (X, HYPS, HL, torch.tensor([T + 1, T]))),
    ("frames_low", ValueError, "logits_lengths", 0, lambda: (X, HYPS, HL, torch.tensor([0, T]))),
    ("label_high", ValueError, "hypothesis labels", 0, lambda: (X, torch.full((B, 3, 4), V), HL, None)),
    ("label_low", ValueError, "hypothesis labels", 0, lambda: (X, torch.full((B, 3, 4), -2), HL, None)),
    ("alphabet", NotImplementedError, "alphabet", 0,
     lambda: (torch.randn(1, 2, _max_alphabet() + 1), HYPS[:1], HL[:1], None)),
]
SCORE_WIDTH = ("width", NotImplementedError, "scorer", 0,
               lambda: (X, torch.ones(B, 3, _max_targets() + 1, dtype=torch.int64), HL, None))
ALIGN_WIDTH = ("width", NotImplementedError, "aligner", 0, lambda: (X, torch.ones(B, 3, 1024, dtype=torch.int64), HL, None))


def _score_calls(eng, logits, hyps, hl, ll):
    """Every entry point of the scorer's family on one set of arguments; the extra per-call tensors are well formed."""
    g, w = torch.ones(hl.shape, dtype=torch.float64), torch.ones(hl.shape[:1], dtype=torch.float64)
    return {"score_device": lambda: eng.score_device(logits, hyps, hl, ll),
            "score_backward_workspace_bytes": lambda: eng.score_backward_workspace_bytes(logits, hyps, hl, ll),
            "score_backward_device": lambda: eng.score_backward_device(logits, hyps, hl, g, ll),
            "mwer_workspace_bytes": lambda: eng.mwer_workspace_bytes(logits, hyps, hl, ll),
            "mwer_forward_device": lambda: eng.mwer_forward_device(logits, hyps, hl, g, None, ll),
            "mwer_backward_device": lambda: eng.mwer_backward_device(logits, hyps, hl, w, None, ll)}


@pytest.mark.parametrize("case", SCORE + [SCORE_WIDTH], ids=[c[0] for c in SCORE] + ["width"])
def test_score_argument_errors(engine, case):
    _, exc, word, blank, args = case
    for name, call in _score_calls(engine.CTCBeamEngine(blank, 1), *args()).items():
        with pytest.raises(exc, match=word):
            call()


@pytest.mark.parametrize("case", SCORE + [ALIGN_WIDTH], ids=[c[0] for c in SCORE] + ["width"])
def test_align_argument_errors(engine, case):
    _, exc, word, blank, args = case
    with pytest.raises(exc, match=word):
        engine.CTCBeamEngine(blank, 1).align_device(*args())


def test_mwer_score_scale(engine):
    for bad in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError, match="score_scale"):
            engine.CTCBeamEngine(0, 1).mwer_forward_device(X, HYPS, HL, torch.ones(B, 3), score_scale=bad)


# ------------------------------------------------------------------------------------------- edit distance ----------
# (id, exception, key word, (hyps, hyp_lengths, refs, ref_lengths))
ERRORS = [
    ("rank", ValueError, "hyps", lambda: (HYPS[0, 0], HL[0, 0], REFS, RL)),
    ("empty_batch", ValueError, "no hypothesis", lambda: (HYPS[:0], HL[:0], REFS[:0], RL[:0])),
    ("int_hyps", TypeError, "hyps", lambda: (HYPS.float(), HL, REFS, RL)),
    ("int_refs", TypeError, "refs", lambda: (HYPS, HL, REFS.float(), RL)),
    ("hyp_lengths_shape", ValueError, "hyp_lengths", lambda: (HYPS, HL[:, :2], REFS, RL)),
    ("refs_shape", ValueError, "refs", lambda: (HYPS, HL, REFS[:1], RL)),
    ("ref_lengths_shape", ValueError, "ref_lengths", lambda: (HYPS, HL, REFS, RL[:1])),
    ("hyp_length_high", ValueError, "hyp_lengths", lambda: (HYPS, torch.full((B, 3), 5), REFS, RL)),
    ("hyp_length_low", ValueError, "hyp_lengths", lambda: (HYPS, torch.full((B, 3), -1), REFS, RL)),
    ("ref_length_high", ValueError, "ref_lengths", lambda: (HYPS, HL, REFS, torch.tensor([6, 1]))),
    ("ref_length_low", ValueError, "ref_lengths", lambda: (HYPS, HL, REFS, torch.tensor([-1, 1]))),
    ("ref_width", NotImplementedError, "reference width", lambda: (HYPS, HL, torch.ones(B, 4096, dtype=torch.int64), RL)),
    ("hyp_width", NotImplementedError, "hypothesis width",
     lambda: (torch.ones(B, 1, 65536, dtype=torch.int64), HL[:, :1], REFS, RL)),
]


@pytest.mark.parametrize("case", ERRORS, ids=[c[0] for c in ERRORS])
def test_errors_argument_errors(engine, case):
    _, exc, word, args = case
    for words in (False, True):
        with pytest.raises(exc, match=word):
            engine.CTCBeamEngine(0, 1, LABELS).errors_device(*args(), words=words)


# -------------------------------------------------------------------------------- get_alignment_3d, no-blank --------
# (id, exception, key word, blank_idx or space_idx, (log_probs, targets, logits_lengths, targets_lengths)).  The
# shape checks run before CPU input is copied to the device; lengths and labels are checked on the device only.
LATTICE = [
    ("rank", ValueError, r"\[batch, frames, alphabet\]", None, lambda: (X[0], TG, LL, TL)),
    ("int_logits", TypeError, "dtype", None, lambda: (X.to(torch.int32), TG, LL, TL)),
    ("empty_batch", ValueError, "empty", None, lambda: (X[:0], TG[:0], LL[:0], TL[:0])),
    ("targets_shape", ValueError, "targets", None, lambda: (X, TG[:1], LL, TL)),
    ("targets_rank", ValueError, "targets", None, lambda: (X, TG[0], LL, TL)),
]


@pytest.mark.parametrize("case", LATTICE + [("blank", ValueError, "blank_idx", 7, lambda: (X, TG, LL, TL))],
                         ids=[c[0] for c in LATTICE] + ["blank"])
def test_get_alignment_3d_argument_errors(engine, case):
    from end2end_b200.utils.alignment import get_alignment_3d_device
    _, exc, word, blank, args = case
    with pytest.raises(exc, match=word):
        get_alignment_3d_device(*args(), blank_idx=blank or 0)


@pytest.mark.parametrize("case", LATTICE + [("space", ValueError, "space_idx", V, lambda: (X, TG, LL, TL))],
                         ids=[c[0] for c in LATTICE] + ["space"])
def test_ctc_without_blank_argument_errors(engine, case):
    from end2end_b200.functions.ctc_without_blank import ctc_without_blank_3d_loss
    _, exc, word, space, args = case
    with pytest.raises(exc, match=word):
        ctc_without_blank_3d_loss(*args(), space_idx=-1 if space is None else space)


# ------------------------------------------------------------------------------------------------- GPU --------------

@pytest.mark.gpu
def test_argument_errors_behind_a_cuda_call():
    """The checks a call reaches only after picking a device: ``compute`` on CPU tensors, and the shapes of MWER's risk,
    mask and utterance scale.  They raise before any launch."""
    from end2end_b200 import _lib
    from end2end_b200.engine import CTCBeamEngine, CTCLossEngine
    before = _lib.launch_count()
    for _, exc, word, blank, args in LOSS:
        with pytest.raises(exc, match=word):
            CTCLossEngine(blank).compute(*args())
    eng = CTCBeamEngine(0, 1)
    g = torch.ones(B, 3)
    with pytest.raises(ValueError, match="risk"):
        eng.mwer_forward_device(X, HYPS, HL, g[:, :2])
    with pytest.raises(ValueError, match="mask"):
        eng.mwer_forward_device(X, HYPS, HL, g, mask=torch.ones(B, 2, dtype=torch.bool))
    with pytest.raises(ValueError, match="utt_scale"):
        eng.mwer_backward_device(X, HYPS, HL, g, torch.empty(0, dtype=torch.uint8, device="cuda"))
    assert _lib.launch_count() == before

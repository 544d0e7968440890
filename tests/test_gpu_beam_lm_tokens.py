"""The prefix beam search with a word n-gram language model over sub-word labels (CTCDecoder.decode /
decode_nbest with lm= and the word_marker attribute set, e2e_ctc_beam_lm_tokens_nbest_device, NGramLM.lexicon(word_marker=), lm.ngram.label_kinds).

The definition (continuations, word starts and boundaries; the word count; completing a word) is include/e2e_ctc.h's, at
e2e_ctc_ngram_tokens.  The checker is tests/beam_lm_tokens_restatement.c: beam_lm_restatement.c's search with that word
rule, words spelled by characters and found by comparing spellings.  The device-free tests pin it to
beam_lm_restatement.c on character alphabets written as kinds, to beam_nbest_restatement.c without the model, and to
brute force on beams that hold every prefix.  The GPU tests compare the kernel with it: hypotheses, lengths, order, OOV
counts and tie counters bit for bit, scores, log_probs and lm_scores within 1e-12 relative.
"""
import atexit
import ctypes
import math
import os
import random
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

import oracle
from test_gpu_beam_lm import (C2_LABELS, LETTERS, _close, _log_probs, _lm_arrays, corpus_model, py_lm, random_model,
                              restate)
from test_gpu_beam_nbest import EXHAUSTIVE, beam_nbest

_HERE = os.path.dirname(os.path.abspath(__file__))
_RESTATEMENT_SRC = os.path.join(_HERE, "beam_lm_tokens_restatement.c")
_restatement_lib = None
MARK = "▁"


def _restatement():
    """gcc the C restatement into a temporary directory (once per process; the tree is left untouched)."""
    global _restatement_lib
    if _restatement_lib is None:
        d = tempfile.mkdtemp(prefix="beam_lm_tokens_restatement_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libbeam_lm_tokens_restatement.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", so,
                               _RESTATEMENT_SRC, "-lm"])
        L = ctypes.CDLL(so)
        dp, ip, i32p = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32)
        ci, cd = ctypes.c_int, ctypes.c_double
        L.ctc_beam_lm_tokens_nbest.argtypes = [dp, ci, ci, ci, ip, ci, ci, ci, cd, cd, cd, ci, ci, i32p, i32p, dp, dp, ci,
                                               i32p, i32p, i32p, i32p, i32p, i32p, ci, ci, ci, ip, ip, dp, dp, dp, ip, ip]
        L.ctc_beam_lm_tokens_nbest.restype = None
        _restatement_lib = L
    return _restatement_lib


def _kinds(labels, blank, marker, case_sensitive):
    """(kind, characters) of every label, restated here: the marker alone is 2, the marker and more is 1, else 0;
    ``marker=None`` writes a character alphabet as kinds (" " is 2, every other label 0)."""
    out = []
    for i, lab in enumerate(labels):
        if i == blank:
            out.append((0, ""))
        elif marker is None:
            out.append((2, "") if lab == " " else (0, lab))
        elif lab == marker:
            out.append((2, ""))
        elif lab.startswith(marker):
            out.append((1, lab[len(marker):]))
        else:
            out.append((0, lab))
    return [(k, t if case_sensitive else t.lower()) for k, t in out]


def restate_tokens(logits, ll, ng, labels, marker=MARK, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0,
                   case_sensitive=True, after_logsoftmax=True, time_major=False):
    """The restatement's (targets [B,N,Tw], lengths, scores, log_probs, lm_scores, oov_words, ties)."""
    with torch.no_grad():
        if not after_logsoftmax:
            logits = torch.log_softmax(logits, -1)
        if time_major:
            logits = logits.transpose(1, 0)
    logits = logits.detach().cpu()
    B, T, V = logits.shape
    if ll is None:
        ll = torch.full((B,), T, dtype=torch.int64)
    x = np.ascontiguousarray(logits.to(torch.float64).numpy())
    il = np.ascontiguousarray(ll.cpu().to(torch.int64).numpy())
    N, Tw = int(n_best), max(T, 1)
    out = np.zeros((B, N, Tw), dtype=np.int64)
    out_len = np.zeros((B, N), dtype=np.int64)
    scores, log_probs, lm_scores = (np.zeros((B, N), dtype=np.float64) for _ in range(3))
    oov = np.zeros((B, N), dtype=np.int64)
    ties = np.zeros(B, dtype=np.int64)
    ids, n, prob, bow, nv, off, chars, ok, _, bos, eos, unk = _lm_arrays(ng, labels, blank, case_sensitive)
    kt = _kinds(labels, blank, marker, case_sensitive)
    arr = lambda a: np.ascontiguousarray(np.array(a, dtype=np.int32))   # noqa: E731
    kinds = arr([k for k, _ in kt])
    loff = arr(np.cumsum([0] + [len(t) for _, t in kt]))
    lchars = arr([ord(ch) for _, t in kt for ch in t] or [0])
    P = lambda a, t: a.ctypes.data_as(ctypes.POINTER(t))   # noqa: E731
    d, i64, i32 = ctypes.c_double, ctypes.c_int64, ctypes.c_int32
    _restatement().ctc_beam_lm_tokens_nbest(
        P(x, d), B, T, V, P(il, i64), int(blank), int(beam), N, float(wip), float(lmwt), float(oov_penalty), len(ng),
        len(n), P(ids, i32), P(n, i32), P(prob, d), P(bow, d), nv, P(off, i32), P(chars, i32), P(ok, i32), P(kinds, i32),
        P(loff, i32), P(lchars, i32), bos, eos, unk, P(out, i64), P(out_len, i64), P(scores, d), P(log_probs, d),
        P(lm_scores, d), P(oov, i64), P(ties, i64))
    return tuple(torch.from_numpy(a) for a in (out, out_len, scores, log_probs, lm_scores, oov, ties))


def _render(seq, labels, marker=MARK):
    """A hypothesis as text: markers as spaces (py_lm splits words on spaces)."""
    return "".join(labels[c] for c in seq if c >= 0).replace(marker, " ")


def _words(seq, labels, marker=MARK):
    n, empty = 0, True
    for c in seq:
        lab = labels[c]
        if lab.startswith(marker):
            empty = lab == marker
            n += 0 if empty else 1
        else:
            n += 1 if empty else 0
            empty = False
    return n


# labels of every kind, 1 to 12 characters, upper case among them
TOKEN_LABELS = ["_", MARK, MARK + "the", MARK + "c", "at", "ot", MARK + "a", "t", "e", MARK + "Th", "E", MARK + "tea",
                "he", MARK + "catastrophes", "astroph", "es", MARK + "t", "o", "a", "h"]
TOKEN_WORDS = ["the", "cat", "cot", "a", "at", "to", "tea", "he", "eat", "catastrophes", "The", "tat", "hat"]


def _token_alphabet(V, seed):
    """blank, marker, then V - 2 word starts and continuations built from random letters (1-11 characters)."""
    rng = random.Random(seed)
    labels, seen = ["_", MARK], set()
    while len(labels) < V:
        piece = "".join(rng.choice(LETTERS[:8]) for _ in range(rng.choice([1, 1, 2, 2, 3, 4, 11])))
        lab = (MARK + piece) if rng.random() < 0.4 else piece
        if lab not in seen:
            seen.add(lab)
            labels.append(lab)
    return labels


def _decoder(**kw):
    """A CTCDecoder over sub-word labels (word_marker is an attribute: the constructor keeps the reference's
    signature)."""
    from end2end_b200 import CTCDecoder
    dec = CTCDecoder(**kw)
    dec.word_marker = MARK
    return dec


# ---------------------------------------------------------------------------------------------- device-free ---------

def test_label_kinds():
    from end2end_b200.lm.ngram import BOUNDARY, CONTINUATION, WORD_START, label_kinds
    kinds, texts = label_kinds(["_", MARK, MARK + "The", "e", MARK + "C", "aT"], 0, MARK, case_sensitive=False)
    assert kinds == [CONTINUATION, BOUNDARY, WORD_START, CONTINUATION, WORD_START, CONTINUATION]
    assert texts == ["", "", "the", "e", "c", "at"]
    assert label_kinds(["<b>", "##", "##ab", "a"], 0, "##")[0] == [0, 2, 1, 0]
    assert label_kinds(["", "a"], 0, MARK)[0] == [0, 0]            # the blank is never read
    for bad in (["_", ""], ["_", "a b"], ["_", " "], ["_", "a" + MARK], ["_", MARK + MARK], ["_", MARK + "a" + MARK]):
        with pytest.raises(ValueError):
            label_kinds(bad, 0, MARK)
    for marker in ("", None, 3):
        with pytest.raises(ValueError):
            label_kinds(["_", "a"], 0, marker)


def test_restatement_equals_character_restatement():
    """Character alphabets written as kinds (" " the boundary, every other label a continuation): the token restatement
    is beam_lm_restatement.c's, bit for bit, over orders 1-6 and many seeds."""
    words = ["a", "ab", "ba", "c", "cab", "dd", "Cab", "bad", "abc"]
    labels = ["_", " ", "a", "b", "C", "c", "d"]
    n = 0
    for order in range(1, 7):
        for seed in range(4):
            ng = random_model(100 * order + seed, order, words, with_unk=(seed % 2 == 0)).loaded()
            for beam, n_best, cs in ((3, 2, True), (12, 12, False), (40, 9, True)):
                x = _log_probs(3, 14, len(labels), 1000 * order + 10 * seed + beam)
                ll = torch.tensor([14, 6, 1])
                args = dict(beam=beam, n_best=n_best, wip=0.3, lmwt=0.7, oov_penalty=-2.0, case_sensitive=cs)
                got = restate_tokens(x, ll, ng, labels, marker=None, **args)
                want = restate(x, ll, ng, labels, **args)
                for a, b in zip(got, want):
                    assert torch.equal(a, b), (order, seed, beam)
                n += 1
    assert n == 6 * 4 * 3


def test_restatement_without_model_equals_lm_free():
    """lmwt = oov_penalty = wip = 0: the token search is beam_nbest_restatement.c's, bit for bit (ties included)."""
    ng = random_model(3, 3, TOKEN_WORDS).loaded()
    V = len(TOKEN_LABELS)
    for beam, n_best in ((10, 10), (3, 2), (40, 7)):
        lp = _log_probs(4, 12, V, 10 * V + beam)
        ll = torch.tensor([12, 7, 1, 3])
        t, n, sc, lpr, lm, oov, ties = restate_tokens(lp, ll, ng, TOKEN_LABELS, beam=beam, n_best=n_best, lmwt=0.0)
        ot, on, osc, olp, oties = beam_nbest(lp, ll, beam_width=beam, n_best=n_best, labels=TOKEN_LABELS,
                                             after_logsoftmax=True, wip=0.0)
        assert torch.equal(t, ot) and torch.equal(n, on) and torch.equal(ties, oties)
        assert torch.equal(sc, osc) and torch.equal(lpr, olp)


def _brute_force(lp, T, labels, ng, order, lmwt, wip, oov_penalty):
    V = len(labels)
    seqs, frontier = [[]], [[]]
    for _ in range(T):
        frontier = [s + [c] for s in frontier for c in range(1, V)]
        seqs += frontier
    k = len(seqs)
    tg = torch.zeros(k, max(1, T), dtype=torch.int64)
    for i, s in enumerate(seqs):
        if s:
            tg[i, :len(s)] = torch.tensor(s)
    tl = torch.tensor([len(s) for s in seqs])
    loss, _ = oracle.PortEngine(0).compute(lp.expand(k, -1, -1).contiguous(), tg, torch.full((k,), T, dtype=torch.int64), tl)
    out = []
    for i, s in enumerate(seqs):
        lm, oov = py_lm(ng, order, _render(s, labels))
        ll = -float(loss[i])
        out.append((((ll + lmwt * lm) - _words(s, labels) * wip) + oov * oov_penalty, ll, lm, oov, s))
    out.sort(key=lambda r: -r[0] if math.isfinite(r[0]) else math.inf)
    return out


def _check_brute(t, n, sc, lpr, lm, oov, brute, lmwt, wip, oov_penalty, labels, ng, order):
    k = int((n > 0).sum())
    fin = [r for r in brute if math.isfinite(r[0])]
    assert int(torch.isfinite(sc[:k]).sum()) == len(fin)
    for r in range(k):
        seq = t[r, :int(n[r])].tolist()
        seq = [] if seq == [-1] else seq
        want_lm, want_oov = py_lm(ng, order, _render(seq, labels))
        assert int(oov[r]) == want_oov
        assert math.isclose(float(lm[r]), want_lm, rel_tol=1e-12, abs_tol=1e-300)
        if not math.isfinite(float(sc[r])):
            continue
        want = ((float(lpr[r]) + lmwt * want_lm) - _words(seq, labels) * wip) + want_oov * oov_penalty
        assert math.isclose(float(sc[r]), want, rel_tol=1e-12)
        b = fin[r]
        assert math.isclose(float(sc[r]), b[0], rel_tol=1e-10), (r, float(sc[r]), b)
        if all(abs(b[0] - o[0]) > 1e-9 * abs(b[0]) for o in fin if o is not b):
            assert seq == b[4], (r, seq, b)


# small alphabets of every kind: "_", the marker, word starts and continuations spelling the same words two ways
_EXH_LABELS = ["_", MARK, MARK + "a", "a", MARK + "ab", "b"]


@pytest.mark.parametrize("V,T", [vt for vt in EXHAUSTIVE if vt[0] >= 3])
def test_restatement_exhaustive_matches_brute_force(V, T):
    labels = _EXH_LABELS[:V] if V <= len(_EXH_LABELS) else _EXH_LABELS + ["c%d" % i for i in range(V - len(_EXH_LABELS))]
    m = random_model(7 * V + T, 3, ["a", "aa", "ab", "ba", "b", "aab"], with_unk=(T % 2 == 0))
    ng = m.loaded()
    lmwt, wip, oovp = 0.8, 0.3, -1.5
    lp = _log_probs(2, T, V, 100 * V + T, scale=1.5)
    t, n, sc, lpr, lm, oov, _ = restate_tokens(lp, None, ng, labels, beam=256, n_best=256, wip=wip, lmwt=lmwt,
                                               oov_penalty=oovp)
    for b in range(lp.size(0)):
        brute = _brute_force(lp[b:b + 1], T, labels, ng, m.order, lmwt, wip, oovp)
        _check_brute(t[b], n[b], sc[b], lpr[b], lm[b], oov[b], brute, lmwt, wip, oovp, labels, ng, m.order)


def test_sentences_render_markers():
    from end2end_b200 import CTCDecoder
    dec = _decoder(beam_width=4, labels=["_", MARK, MARK + "the", MARK + "c", "at", " "])
    targets = torch.tensor([[2, 3, 4, 0], [1, 2, 1, 0], [-1, 0, 0, 0], [4, 1, 3, 5]])
    assert dec._sentences(targets, torch.tensor([3, 3, 1, 4])) == ["the cat", "the", "", "at  c"]
    plain = CTCDecoder(beam_width=4, labels=["_", MARK, MARK + "the", MARK + "c", "at", " "])
    assert plain._sentences(targets[:1], torch.tensor([3])) == [MARK + "the" + MARK + "cat"]
    for bad in ("", 5):
        with pytest.raises(ValueError):
            plain.word_marker = bad


# ---------------------------------------------------------------------------------------------- GPU -----------------

_MODELS = {}


def _lm(model, tmp, key=None):
    from end2end_b200 import NGramLM
    key = key or repr(model.ngrams)
    if key not in _MODELS:
        path = model.write(os.path.join(tmp, "m%d.arpa" % len(_MODELS)))
        _MODELS[key] = NGramLM.from_arpa(path)
    return _MODELS[key]


@pytest.fixture(scope="module")
def tmpdir_tok():
    d = tempfile.mkdtemp(prefix="beam_lm_tokens_models_")
    yield d
    shutil.rmtree(d, True)
    _MODELS.clear()


def _kernel(x, ll, lm, labels, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0, case_sensitive=True,
            from_logits=False, marker=MARK):
    from end2end_b200.engine import CTCBeamEngine
    eng = CTCBeamEngine(blank, beam, labels, wip)
    out = eng.decode_nbest_lm_device(x.cuda(), lm, None if ll is None else ll.cuda(), n_best, from_logits, lmwt=lmwt,
                                     oov_penalty=oov_penalty, case_sensitive=case_sensitive, word_marker=marker)
    return [t.cpu() for t in out]


def _assert_equal_restatement(x, ll, model, lm, labels, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0,
                              case_sensitive=True):
    got = _kernel(x, ll, lm, labels, blank, beam, n_best, wip, lmwt, oov_penalty, case_sensitive)
    want = restate_tokens(x, ll, model.loaded(), labels, MARK, blank, beam, n_best, wip, lmwt, oov_penalty, case_sensitive)
    ctx = (tuple(x.shape), x.dtype, beam, n_best, wip, lmwt, oov_penalty, model.order, case_sensitive)
    t, n, sc, lpr, lms, oov, ties = got
    ot, on, osc, olp, olm, ooov, oties = want
    assert torch.equal(n, on), ctx
    assert torch.equal(t, ot), ctx
    assert torch.equal(oov, ooov), ctx
    assert torch.equal(ties, oties), (ctx, ties, oties)
    _close(sc, osc, 1e-12, ctx)
    _close(lpr, olp, 1e-12, ctx)
    _close(lms, olm, 1e-12, ctx)
    return got


@pytest.mark.gpu
def test_kernel_equals_restatement_orders_beams(tmpdir_tok):
    """Orders 1-6 with and without <unk>, beams 1, 2, 7, 100 and 256, N = 1 and the full beam, both case modes."""
    V = len(TOKEN_LABELS)
    n = 0
    for order in range(1, 7):
        model = random_model(200 + order, order, TOKEN_WORDS, with_unk=order % 2 == 0)
        lm = _lm(model, tmpdir_tok)
        for beam in (1, 2, 7, 100, 256):
            T = 12 if beam >= 100 else 20
            x = _log_probs(3, T, V, 2000 * order + beam)
            ll = torch.tensor([T, T // 2, 1])
            for n_best in sorted({1, beam}):
                for cs in (True, False):
                    _assert_equal_restatement(x, ll, model, lm, TOKEN_LABELS, 0, beam, n_best, wip=0.3, lmwt=0.7,
                                              oov_penalty=-2.0, case_sensitive=cs)
                    n += 1
    assert n == 6 * 5 * 2 * 2 - 6 * 2


@pytest.mark.gpu
def test_kernel_equals_restatement_dtypes_layouts_batch(tmpdir_tok):
    """Every input dtype; raw logits (fused log-softmax) and time-major input through CTCDecoder; B = 150 > 148 SMs."""
    model = random_model(5, 3, TOKEN_WORDS)
    lm = _lm(model, tmpdir_tok)
    V = len(TOKEN_LABELS)
    x = _log_probs(4, 30, V, 6)
    ll = torch.tensor([30, 20, 3, 1])
    for dtype in (torch.float32, torch.float64, torch.bfloat16, torch.float16):
        for n_best in (1, 25):
            _assert_equal_restatement(x.to(dtype), ll, model, lm, TOKEN_LABELS, 0, 25, n_best, wip=0.5, lmwt=1.2,
                                      oov_penalty=-3.0)
    g = torch.Generator().manual_seed(8)
    raw = torch.randn(5, 40, V, generator=g) * 2.0
    rl = torch.randint(20, 41, (5,), generator=g)
    for dtype, time_major in ((torch.float32, False), (torch.float64, True)):
        xin = raw.to(dtype)
        if time_major:
            xin = xin.transpose(0, 1)
        dec = _decoder(beam_width=30, labels=TOKEN_LABELS, wip=0.5, lmwt=1.1, oov_penalty=-2.5, time_major=time_major)
        res = dec.decode_nbest(xin.cuda(), rl, n_best=10, lm=lm)
        ot, on, osc, olp, olm, ooov, oties = restate_tokens(xin, rl, model.loaded(), TOKEN_LABELS, MARK, 0, 30, 10, 0.5,
                                                            1.1, -2.5, after_logsoftmax=False, time_major=time_major)
        tol = 1e-12 if dtype == torch.float64 else 1e-6
        assert torch.equal(res.decoded_targets_lengths, on) and torch.equal(res.oov_words, ooov)
        w = res.decoded_targets.size(2)
        assert torch.equal(res.decoded_targets, ot[:, :, :w]) and not bool(ot[:, :, w:].any())
        assert torch.equal(dec._decoder.last_ties, oties)
        _close(res.scores, osc, tol)
        _close(res.log_probs, olp, tol)
        _close(res.lm_scores, olm, 1e-12)
        want = _render(ot[0, 0, :int(on[0, 0])].tolist(), TOKEN_LABELS).strip(" ")
        assert res.decoded_sentences[0][0] == want
    big = _log_probs(150, 20, V, 12)
    big_ll = torch.randint(10, 21, (150,), generator=torch.Generator().manual_seed(13))
    model = random_model(14, 4, TOKEN_WORDS)
    lm = _lm(model, tmpdir_tok)
    for n_best in (1, 40):
        _assert_equal_restatement(big, big_ll, model, lm, TOKEN_LABELS, 0, 40, n_best, wip=0.4, lmwt=0.9,
                                  oov_penalty=-2.0)


_PREFILTER_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from end2end_b200 import NGramLM
from end2end_b200.engine import CTCBeamEngine
x, labels, path, out = torch.load(sys.argv[2])
lm = NGramLM.from_arpa(path)
eng = CTCBeamEngine(0, 100, labels, 0.3)
res = eng.decode_nbest_lm_device(x.cuda(), lm, None, 100, False, lmwt=0.8, oov_penalty=-2.0, word_marker="▁")
torch.save([t.cpu() for t in res], out)
"""


@pytest.mark.gpu
def test_large_alphabet_prefilter(tmpdir_tok):
    """V = 1024 sub-word labels at beam 100: the two-class filter (102 continuations, 102 word starts, the boundary);
    the restatement's result, and identical with the filter off (E2E_CTC_BEAM_NOPREFILTER=1, read once per process: a
    child process)."""
    V = 1024
    labels = _token_alphabet(V, 15)
    rng = random.Random(16)
    pieces = [lab.lstrip(MARK) for lab in labels[2:200]]
    words = sorted({"".join(rng.choice(pieces) for _ in range(rng.randint(1, 2))) for _ in range(300)})
    model = random_model(16, 3, words, per_order=300)
    path = model.write(os.path.join(tmpdir_tok, "v1024.arpa"))
    from end2end_b200 import NGramLM
    lm = NGramLM.from_arpa(path)
    x = _log_probs(3, 16, V, 17, scale=3.0)
    x[:, :, 2:200] += 2.0                                   # words of the model are likely
    x = torch.log_softmax(x, 2)
    got = _assert_equal_restatement(x, None, model, lm, labels, 0, 100, 100, wip=0.3, lmwt=0.8, oov_penalty=-2.0)
    job = os.path.join(tmpdir_tok, "job.pt")
    out = os.path.join(tmpdir_tok, "nopre.pt")
    torch.save([x, labels, path, out], job)
    env = dict(os.environ, E2E_CTC_BEAM_NOPREFILTER="1")
    subprocess.check_call([sys.executable, "-c", _PREFILTER_SCRIPT, os.path.dirname(_HERE), job], env=env)
    other = torch.load(out)
    for a, b in zip(got, other):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_marker_mode_equals_character_mode(tmpdir_tok):
    """["_", marker, a-z, "'"] with the marker against C2_LABELS in character mode on the same c2 logits: every field
    and the tie counters identical."""
    from end2end_b200 import CTCDecoder
    model = random_model(18, 3, ["the", "cat", "cot", "a", "at", "to", "tea", "it's"])
    lm = _lm(model, tmpdir_tok)
    x, _, ll, _ = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    x, ll = x[:32].cuda(), ll[:32]
    tok_labels = ["_", MARK] + LETTERS + ["'"]
    assert len(tok_labels) == len(C2_LABELS) == 29
    for cs in (True, False):
        kw = dict(beam_width=100, wip=0.5, lmwt=1.3, oov_penalty=-4.0, case_sensitive=cs)
        char = CTCDecoder(labels=C2_LABELS, **kw)
        tok = _decoder(labels=tok_labels, **kw)
        a = char.decode_nbest(x, ll, n_best=100, lm=lm)
        b = tok.decode_nbest(x, ll, n_best=100, lm=lm)
        for f in ("decoded_targets", "decoded_targets_lengths", "scores", "log_probs", "lm_scores", "oov_words"):
            assert torch.equal(getattr(a, f), getattr(b, f)), f
        assert torch.equal(char._decoder.last_ties, tok._decoder.last_ties)
        assert [[s.strip(" ") for s in row] for row in a.decoded_sentences] == b.decoded_sentences


@pytest.mark.gpu
def test_token_fusion_changes_the_winner(tmpdir_tok):
    """Frames spelling "_a" "_c" then "at" slightly above "ot": without the model "a cat" wins, the corpus model prefers
    "a cot" and the fused search keeps and picks it."""
    lm = _lm(corpus_model(), tmpdir_tok)
    ng = corpus_model().loaded()
    assert py_lm(ng, 2, "a cot")[0] > py_lm(ng, 2, "a cat")[0] + 1.0
    labels = ["_", MARK, MARK + "a", MARK + "c", "at", "ot", "t", "o"]
    idx = {c: i for i, c in enumerate(labels)}
    T = 7
    x = torch.full((1, T, len(labels)), -12.0)
    for t, spec in enumerate([MARK + "a", "_", MARK + "c", "_", {"at": -0.6, "ot": -0.8}, "_", "_"]):
        if isinstance(spec, dict):
            for c, v in spec.items():
                x[0, t, idx[c]] = v
        else:
            x[0, t, idx[spec]] = 0.0
    x = torch.log_softmax(x, 2)
    kw = dict(beam_width=8, labels=labels, after_logsoftmax=True, wip=0.0, oov_penalty=0.0)
    free = _decoder(lmwt=0.0, **kw)
    fused = _decoder(lmwt=1.0, **kw)
    assert free.decode(x.cuda(), lm=lm).decoded_sentences == ["a cat"]
    assert free.decode(x.cuda()).decoded_sentences == ["a cat"]
    assert fused.decode(x.cuda(), lm=lm).decoded_sentences == ["a cot"]
    assert fused.decode(x, lm=lm).decoded_sentences == ["a cot"]


@pytest.mark.gpu
def test_invariants(tmpdir_tok):
    """decode(lm=) is hypothesis 0; the scores are the expression of their parts; two builds of the model agree."""
    from end2end_b200 import NGramLM
    model = random_model(19, 3, TOKEN_WORDS)
    path = model.write(os.path.join(tmpdir_tok, "inv.arpa"))
    lm, lm2 = NGramLM.from_arpa(path), NGramLM.from_arpa(path)
    x = _log_probs(16, 60, len(TOKEN_LABELS), 20, scale=2.5).to(torch.float32).cuda()
    ll = torch.randint(20, 61, (16,), generator=torch.Generator().manual_seed(21))
    dec = _decoder(beam_width=50, labels=TOKEN_LABELS, wip=0.5, lmwt=1.3, oov_penalty=-4.0, after_logsoftmax=True,
                   case_sensitive=False)
    nb = dec.decode_nbest(x, ll, n_best=50, lm=lm)
    one = dec.decode(x, ll, lm=lm)
    w = one.decoded_targets.size(1)
    assert torch.equal(nb.decoded_targets[:, 0, :w], one.decoded_targets)
    assert torch.equal(nb.decoded_targets_lengths[:, 0], one.decoded_targets_lengths)
    assert [s[0] for s in nb.decoded_sentences] == one.decoded_sentences
    words = torch.tensor([[_words(r[:k], TOKEN_LABELS) if r[:k] != [-1] else 0 for r, k in zip(rows, lens)]
                          for rows, lens in zip(nb.decoded_targets.tolist(), nb.decoded_targets_lengths.tolist())],
                         dtype=torch.float64)
    live = nb.decoded_targets_lengths > 0
    expr = ((nb.log_probs + 1.3 * nb.lm_scores) - words * 0.5) + nb.oov_words.double() * -4.0
    assert torch.equal(expr[live], nb.scores[live])
    assert bool((nb.scores[~live] == -math.inf).all()) and not bool(nb.oov_words[~live].any())
    for other in (lm, lm2):
        again = dec.decode_nbest(x, ll, n_best=50, lm=other)
        for f in ("decoded_targets", "decoded_targets_lengths", "scores", "log_probs", "lm_scores", "oov_words"):
            assert torch.equal(getattr(nb, f), getattr(again, f)), f


@pytest.mark.gpu
def test_argument_errors(tmpdir_tok):
    from end2end_b200 import CTCDecoder
    lm = _lm(random_model(22, 2, ["ab"]), tmpdir_tok)
    x = torch.log_softmax(torch.randn(2, 5, 4), 2)
    with pytest.raises(ValueError, match="marker"):
        _decoder(beam_width=4, labels=["_", MARK, "a" + MARK, "b"]).decode(x, lm=lm)
    with pytest.raises(ValueError, match="empty"):
        _decoder(beam_width=4, labels=["_", MARK, "", "b"]).decode(x, lm=lm)
    # no " " needed; a shape past the kernel's shared memory is refused
    V = 6000
    labels = ["_", MARK] + [MARK + "w%d" % i for i in range(V - 2)]
    big = torch.log_softmax(torch.randn(1, 2, V), 2).cuda()
    with pytest.raises(NotImplementedError):
        _decoder(beam_width=256, labels=labels).decode(big, lm=lm)

"""Phrase biasing inside the prefix beam search (PhraseBias, CTCDecoder.decode / decode_nbest with bias=,
CTCBeamEngine.decode_nbest_bias_device, e2e_ctc_beam_bias_nbest_device).

The definition (committed, phi, the score during the search and the final one) is include/e2e_ctc.h's, at e2e_ctc_bias.
The checker is tests/beam_bias_restatement.c: beam_lm_tokens_restatement.c's search with the bias computed by brute force
from the definition (no automaton).  The device-free tests pin the host automaton to the Python definition, the
restatement to beam_lm_tokens_restatement.c without phrases and to beam_nbest_restatement.c without a model, and both to
brute force on beams that hold every prefix.  The GPU tests compare the kernel with it: hypotheses, lengths, order, OOV
counts and tie counters bit for bit, scores, log_probs, lm_scores and bias_scores within 1e-12 relative.
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
from test_gpu_beam_lm import LETTERS, _close, _lm_arrays, _log_probs, py_lm, random_model
from test_gpu_beam_lm_tokens import (MARK, TOKEN_LABELS, TOKEN_WORDS, _kinds, _render, _token_alphabet, _words,
                                     restate_tokens)
from test_gpu_beam_nbest import EXHAUSTIVE, beam_nbest

_HERE = os.path.dirname(os.path.abspath(__file__))
_RESTATEMENT_SRC = os.path.join(_HERE, "beam_bias_restatement.c")
_restatement_lib = None


def _restatement():
    """gcc the C restatement into a temporary directory (once per process; the tree is left untouched)."""
    global _restatement_lib
    if _restatement_lib is None:
        d = tempfile.mkdtemp(prefix="beam_bias_restatement_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libbeam_bias_restatement.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", so,
                               _RESTATEMENT_SRC, "-lm"])
        L = ctypes.CDLL(so)
        dp, ip, i32p = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32)
        ci, cd = ctypes.c_int, ctypes.c_double
        L.ctc_beam_bias_nbest.argtypes = [dp, ci, ci, ci, ip, ci, ci, ci, cd, cd, cd, ci, ci, i32p, i32p, dp, dp, ci,
                                          i32p, i32p, i32p, i32p, i32p, i32p, ci, ci, ci, ci, i32p, i32p, dp, ip, ip, dp,
                                          dp, dp, ip, dp, ip]
        L.ctc_beam_bias_nbest.restype = None
        _restatement_lib = L
    return _restatement_lib


def restate_bias(logits, ll, ng, labels, phrases, weights, marker=MARK, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0,
                 oov_penalty=0.0, case_sensitive=True, after_logsoftmax=True, time_major=False):
    """The restatement's (targets [B,N,Tw], lengths, scores, log_probs, lm_scores, oov_words, bias_scores, ties);
    ``marker=None`` writes a character alphabet as kinds (with ``lmwt = oov_penalty = 0`` the LM-free search)."""
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
    scores, log_probs, lm_scores, bias_scores = (np.zeros((B, N), dtype=np.float64) for _ in range(4))
    oov = np.zeros((B, N), dtype=np.int64)
    ties = np.zeros(B, dtype=np.int64)
    ids, n, prob, bow, nv, off, chars, ok, _, bos, eos, unk = _lm_arrays(ng, labels, blank, case_sensitive)
    kt = _kinds(labels, blank, marker, case_sensitive)
    arr = lambda a: np.ascontiguousarray(np.array(a, dtype=np.int32))   # noqa: E731
    kinds = arr([k for k, _ in kt])
    loff = arr(np.cumsum([0] + [len(t) for _, t in kt]))
    lchars = arr([ord(ch) for _, t in kt for ch in t] or [0])
    poff = arr(np.cumsum([0] + [len(p) for p in phrases]))
    plab = arr([c for p in phrases for c in p] or [0])
    pw = np.ascontiguousarray(np.array(list(weights) or [0.0], dtype=np.float64))
    P = lambda a, t: a.ctypes.data_as(ctypes.POINTER(t))   # noqa: E731
    d, i64, i32 = ctypes.c_double, ctypes.c_int64, ctypes.c_int32
    _restatement().ctc_beam_bias_nbest(
        P(x, d), B, T, V, P(il, i64), int(blank), int(beam), N, float(wip), float(lmwt), float(oov_penalty), len(ng),
        len(n), P(ids, i32), P(n, i32), P(prob, d), P(bow, d), nv, P(off, i32), P(chars, i32), P(ok, i32), P(kinds, i32),
        P(loff, i32), P(lchars, i32), bos, eos, unk, len(phrases), P(poff, i32), P(plab, i32), P(pw, d), P(out, i64),
        P(out_len, i64), P(scores, d), P(log_probs, d), P(lm_scores, d), P(oov, i64), P(bias_scores, d), P(ties, i64))
    return tuple(torch.from_numpy(a) for a in (out, out_len, scores, log_probs, lm_scores, oov, bias_scores, ties))


# ---- the definition, in Python --------------------------------------------------------------------------------------

def py_committed(seq, phrases, weights):
    """Left fold over the positions of out_i: the phrases that are a suffix of seq[:i], ascending index, w * k."""
    acc = 0.0
    for i in range(1, len(seq) + 1):
        out = 0.0
        for p, w in zip(phrases, weights):
            if len(p) <= i and tuple(seq[i - len(p):i]) == tuple(p):
                out = out + w * len(p)
        acc = acc + out
    return acc


def py_phi(seq, phrases, weights):
    for d in range(len(seq), 0, -1):
        ws = [w for p, w in zip(phrases, weights) if len(p) > d and tuple(seq[len(seq) - d:]) == tuple(p[:d])]
        if ws:
            return d * max(ws)
    return 0.0


def random_phrases(rng, n, V, max_len=5, blank=0):
    """Phrases over labels 1..V-1 with shared prefixes, suffixes and infixes of each other, single labels and repeats."""
    out, seen = [], set()
    while len(out) < n:
        r = rng.random()
        if out and r < 0.25:                       # extend an existing phrase
            p = rng.choice(out) + (rng.randrange(1, V),)
        elif out and r < 0.4:                      # a suffix or an infix of one
            q = rng.choice(out)
            i = rng.randrange(len(q))
            p = q[i:rng.randint(i + 1, len(q))]
        elif r < 0.5:                              # a repeated label
            p = (rng.randrange(1, V),) * rng.randint(1, 3)
        else:
            p = tuple(rng.randrange(1, V) for _ in range(rng.randint(1, max_len)))
        p = tuple(c for c in p if c != blank)
        if p and len(p) <= max_len and p not in seen:
            seen.add(p)
            out.append(p)
    return out


def _weights(rng, n):
    return [rng.choice([0.5, 1.0, 1.5, rng.uniform(0.1, 3.0)]) for _ in range(n)]


# ---------------------------------------------------------------------------------------------- device-free ---------

def test_automaton_equals_definition():
    """The host automaton walked over random label sequences gives committed and phi equal bit for bit to the
    definition, for many phrase sets."""
    from end2end_b200.lm.bias import build_automaton
    rng = random.Random(1)
    n_sets = 0
    for trial in range(60):
        V = rng.choice([3, 4, 6, 10])
        phrases = random_phrases(rng, rng.choice([1, 2, 5, 12, 30]), V)
        weights = _weights(rng, len(phrases))
        label_col, nxt, partial, complete = build_automaton(phrases, weights)
        for _ in range(20):
            seq = [rng.randrange(1, V) for _ in range(rng.randint(0, 14))]
            node, com = 0, 0.0
            for i, c in enumerate(seq):
                j = label_col.get(c, -1)
                node = 0 if j < 0 else nxt[node][j]
                com = com if j < 0 else com + complete[node]
                assert com == py_committed(seq[:i + 1], phrases, weights), (phrases, seq[:i + 1])
                assert partial[node] == py_phi(seq[:i + 1], phrases, weights), (phrases, seq[:i + 1])
        n_sets += 1
    assert n_sets == 60
    # phrases ab and bc: phi(ab) is w_bc through the shorter suffix; a completed phrase earns no partial credit itself
    label_col, nxt, partial, complete = build_automaton([(1, 2), (2, 3)], [1.0, 2.5])
    ab = nxt[nxt[0][label_col[1]]][label_col[2]]
    assert complete[ab] == 2.0 and partial[ab] == 2.5


def test_restatement_without_phrases_equals_tokens_restatement():
    ng = random_model(3, 3, TOKEN_WORDS).loaded()
    V = len(TOKEN_LABELS)
    for beam, n_best in ((10, 10), (3, 2), (40, 7)):
        lp = _log_probs(4, 12, V, 10 * V + beam)
        ll = torch.tensor([12, 7, 1, 3])
        args = dict(beam=beam, n_best=n_best, wip=0.3, lmwt=0.7, oov_penalty=-2.0)
        got = restate_bias(lp, ll, ng, TOKEN_LABELS, [], [], **args)
        want = restate_tokens(lp, ll, ng, TOKEN_LABELS, **args)
        for a, b in zip(got[:6] + got[7:], want):
            assert torch.equal(a, b), beam
        live = got[1] > 0
        assert bool((got[6][live] == 0).all()) and bool((got[6][~live] == -math.inf).all())


def test_restatement_without_model_equals_lm_free():
    """A trivial model, lmwt = oov_penalty = 0, characters as kinds, no phrases: beam_nbest_restatement.c, bit for bit."""
    ng = random_model(4, 2, ["a", "b"]).loaded()
    labels = ["_", " "] + LETTERS[:6]
    for beam, n_best in ((10, 10), (3, 2), (40, 7), (1, 1)):
        lp = _log_probs(4, 14, len(labels), 30 + beam)
        ll = torch.tensor([14, 7, 1, 3])
        t, n, sc, lpr, _, _, bs, ties = restate_bias(lp, ll, ng, labels, [], [], marker=None, beam=beam, n_best=n_best,
                                                     wip=0.4, lmwt=0.0, oov_penalty=0.0)
        ot, on, osc, olp, oties = beam_nbest(lp, ll, beam_width=beam, n_best=n_best, labels=labels,
                                             after_logsoftmax=True, wip=0.4)
        assert torch.equal(t, ot) and torch.equal(n, on) and torch.equal(ties, oties)
        assert torch.equal(sc, osc) and torch.equal(lpr, olp)


def _brute_force(lp, T, labels, ng, order, lmwt, wip, oov_penalty, phrases, weights, marker):
    """Every prefix of up to T labels with its final score (the search's expression + committed)."""
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
        lm, oov = py_lm(ng, order, _render(s, labels, marker or " "))
        ll = -float(loss[i])
        words = _words(s, labels, marker) if marker else _space_words(s, labels)
        com = py_committed(s, phrases, weights)
        out.append(((((ll + lmwt * lm) - words * wip) + oov * oov_penalty) + com, ll, lm, oov, s, com))
    out.sort(key=lambda r: -r[0] if math.isfinite(r[0]) else math.inf)
    return out


def _space_words(seq, labels):
    n, last = 0, None
    for c in seq:
        if labels[c] != " " and (n == 0 or last == " "):
            n += 1
        last = labels[c]
    return n


_EXH_LABELS = ["_", MARK, MARK + "a", "a", MARK + "ab", "b"]
_EXH_CHARS = ["_", " ", "a", "b"]


@pytest.mark.parametrize("V,T", [vt for vt in EXHAUSTIVE if vt[0] >= 3])
@pytest.mark.parametrize("mode", ["lm_free", "tokens"])
def test_restatement_exhaustive_matches_brute_force(V, T, mode):
    """Beams that hold every prefix: the restatement's list is the brute-force ranking by the final score (oracle
    likelihood, Python ARPA scorer, Python bias definition), and bias_scores is committed."""
    if mode == "tokens":
        labels, marker = _EXH_LABELS[:V], MARK
        m = random_model(7 * V + T, 3, ["a", "aa", "ab", "ba", "b", "aab"], with_unk=(T % 2 == 0))
        lmwt, wip, oovp = 0.8, 0.3, -1.5
    else:
        labels, marker = _EXH_CHARS[:V], None
        m = random_model(7 * V + T, 2, ["a"])
        lmwt, wip, oovp = 0.0, 0.3, 0.0
    ng = m.loaded()
    rng = random.Random(V * 100 + T)
    phrases = random_phrases(rng, 4, V, max_len=3)
    weights = _weights(rng, len(phrases))
    lp = _log_probs(2, T, V, 100 * V + T, scale=1.5)
    t, n, sc, lpr, lm, oov, bs, _ = restate_bias(lp, None, ng, labels, phrases, weights, marker=marker, beam=256,
                                                 n_best=256, wip=wip, lmwt=lmwt, oov_penalty=oovp)
    for b in range(lp.size(0)):
        brute = _brute_force(lp[b:b + 1], T, labels, ng, m.order, lmwt, wip, oovp, phrases, weights, marker)
        fin = [r for r in brute if math.isfinite(r[0])]
        k = int((n[b] > 0).sum())
        assert int(torch.isfinite(sc[b, :k]).sum()) == len(fin)
        for r in range(k):
            seq = t[b, r, :int(n[b, r])].tolist()
            seq = [] if seq == [-1] else seq
            assert float(bs[b, r]) == py_committed(seq, phrases, weights)
            if not math.isfinite(float(sc[b, r])):
                continue
            assert math.isclose(float(sc[b, r]), fin[r][0], rel_tol=1e-10), (r, float(sc[b, r]), fin[r])
            if all(abs(fin[r][0] - o[0]) > 1e-9 * abs(fin[r][0]) for o in fin if o is not fin[r]):
                assert seq == fin[r][4], (r, seq, fin[r])


def test_phrase_bias_errors():
    from end2end_b200 import PhraseBias
    from end2end_b200.lm import bias as bias_mod
    dev = "cuda:0"                       # no device is touched before the first search
    labels = ["_", " ", "a", "b", "c"]
    ok = PhraseBias([[2, 3], "ab c"], 1.0, labels=labels, device=dev)
    assert ok.phrases == [(2, 3), (2, 3, 1, 4)] and ok.n_cols == 4
    assert PhraseBias([[2], [3]], [0.5, 2.0], device=dev).weights == [0.5, 2.0]
    bad = [
        (([[]], 1.0), {}),                                  # empty phrase
        (([], 1.0), {}),                                    # no phrases
        (([[0, 2]], 1.0), {}),                              # the blank
        (([[2, 5]], 1.0), dict(labels=labels)),             # out of range
        (([[-1]], 1.0), {}),
        (([[2, 3], (2, 3)], 1.0), {}),                      # duplicate
        ((["abd"], 1.0), dict(labels=labels)),              # a character with no label
        ((["ab"], 1.0), {}),                                # a string without labels
        ((["ab"], 1.0), dict(labels=["_", "ab", "b"])),     # labels of several characters
        (([[2]], 0.0), {}), (([[2]], -1.0), {}), (([[2]], math.inf), {}), (([[2]], math.nan), {}),
        (([[2], [3]], [1.0]), {}),                          # one weight for two phrases
        (([[2]], 1.0), dict(device="cpu")),
    ]
    for args, kw in bad:
        with pytest.raises(ValueError):
            PhraseBias(*args, **dict(dict(device=dev), **kw))
    old = bias_mod.MAX_TRANSITIONS
    bias_mod.MAX_TRANSITIONS = 50
    try:
        with pytest.raises(ValueError, match="transitions"):
            PhraseBias([[2, 3, 4, 2, 3, 4, 2, 3, 4, 2, 3, 4, 2, 3, 4, 2, 3]], 1.0, device=dev)
    finally:
        bias_mod.MAX_TRANSITIONS = old
    with pytest.raises(ValueError, match="labels"):
        ok.descriptor(6)                                    # built for another alphabet size
    with pytest.raises(ValueError, match="outside"):
        PhraseBias([[7]], 1.0, device=dev).descriptor(5)


# ---------------------------------------------------------------------------------------------- GPU -----------------

_MODELS = {}


def _lm(model, tmp):
    from end2end_b200 import NGramLM
    key = repr(model.ngrams)
    if key not in _MODELS:
        _MODELS[key] = NGramLM.from_arpa(model.write(os.path.join(tmp, "m%d.arpa" % len(_MODELS))))
    return _MODELS[key]


@pytest.fixture(scope="module")
def tmpdir_bias():
    d = tempfile.mkdtemp(prefix="beam_bias_models_")
    yield d
    shutil.rmtree(d, True)
    _MODELS.clear()


CHAR_LABELS = ["_", " "] + LETTERS[:10]
CHAR_WORDS = ["a", "ab", "bad", "cab", "dice", "fig", "hij", "beef"]
TRIVIAL = random_model(9, 1, ["a"])


def _mode(mode, tmp, seed=0):
    """(labels, marker, model, lm, lmwt, oov_penalty) of a search mode."""
    if mode == "lm_free":
        return CHAR_LABELS, None, TRIVIAL, None, 0.0, 0.0
    if mode == "chars":
        model = random_model(30 + seed, 3, CHAR_WORDS)
        return CHAR_LABELS, None, model, _lm(model, tmp), 0.9, -2.0
    model = random_model(40 + seed, 3, TOKEN_WORDS)
    return TOKEN_LABELS, MARK, model, _lm(model, tmp), 0.7, -2.0


def _kernel(x, ll, bias, labels, lm, marker, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0,
            from_logits=False):
    from end2end_b200.engine import CTCBeamEngine
    eng = CTCBeamEngine(blank, beam, labels, wip)
    out = eng.decode_nbest_bias_device(x.cuda(), bias, lm, None if ll is None else ll.cuda(), n_best, from_logits,
                                       lmwt=lmwt, oov_penalty=oov_penalty, word_marker=marker)
    return [t.cpu() for t in out]


def _check(got, want, ctx, with_lm, tol=1e-12):
    t, n, sc, lpr, lms, oov, bs, ties = got
    ot, on, osc, olp, olm, ooov, obs, oties = want
    assert torch.equal(n, on), ctx
    assert torch.equal(t, ot[:, :, :t.size(2)]) and not bool(ot[:, :, t.size(2):].any()), ctx
    assert torch.equal(ties, oties), (ctx, ties, oties)
    _close(sc, osc, tol, ctx)
    _close(lpr, olp, tol, ctx)
    _close(bs, obs, 1e-12, ctx)
    if with_lm:
        assert torch.equal(oov, ooov), ctx
        _close(lms, olm, 1e-12, ctx)
    else:
        live = n > 0
        assert not bool(lms.any()) and not bool(oov.any()), ctx
        assert bool((bs[~live] == -math.inf).all()), ctx


def _assert_equal_restatement(x, ll, mode, tmp, phrases, weights, beam=10, n_best=1, wip=0.0, seed=0):
    from end2end_b200 import PhraseBias
    labels, marker, model, lm, lmwt, oovp = _mode(mode, tmp, seed)
    bias = PhraseBias(phrases, weights, labels=labels)
    got = _kernel(x, ll, bias, labels, lm, marker, 0, beam, n_best, wip, lmwt, oovp)
    want = restate_bias(x, ll, model.loaded(), labels, bias.phrases, bias.weights, marker, 0, beam, n_best, wip, lmwt,
                        oovp)
    _check(got, want, (mode, tuple(x.shape), x.dtype, beam, n_best, len(phrases)), lm is not None)
    return got


def _spelling_logits(B, T, labels, phrases, seed, scale=2.0, boost=3.0):
    """Log-probabilities that sometimes spell one of the phrases (so matches happen)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, len(labels), generator=g, dtype=torch.float64) * scale
    rng = random.Random(seed)
    for b in range(B):
        t = rng.randrange(3)
        while t < T:
            p = rng.choice(phrases)
            for c in p:
                if t >= T:
                    break
                x[b, t, c] += boost
                t += 1
                if rng.random() < 0.3 and t < T:
                    x[b, t, 0] += boost        # a blank between labels (a repeated label needs one)
                    t += 1
            t += rng.randrange(1, 5)
    return torch.log_softmax(x, 2)


def _phrases_for(labels, n, seed):
    """n phrases: up to 5 multi-word ones (the space / the boundary inside), the rest from random_phrases."""
    rng = random.Random(seed)
    V = len(labels)
    sep = labels.index(" ") if " " in labels else labels.index(MARK)
    out = []
    while len(out) < min(5, n // 2):
        p = tuple(rng.randrange(2, V) for _ in range(2)) + (sep,) + tuple(rng.randrange(2, V) for _ in range(2))
        if p not in out:
            out.append(p)
    out += [p for p in random_phrases(rng, n, V, max_len=6) if p not in out]
    return out[:n]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["lm_free", "chars", "tokens"])
def test_kernel_equals_restatement_beams(mode, tmpdir_bias):
    """Beams 1, 2, 7, 100 and 256, N = 1 and the full beam, 1 and 50 phrases with matches."""
    labels = _mode(mode, tmpdir_bias)[0]
    n = 0
    for n_ph in (1, 50):
        phrases = _phrases_for(labels, n_ph, 5 + n_ph)
        weights = _weights(random.Random(n_ph), len(phrases))
        for beam in (1, 2, 7, 100, 256):
            T = 12 if beam >= 100 else 20
            x = _spelling_logits(3, T, labels, phrases, 1000 * n_ph + beam)
            ll = torch.tensor([T, T // 2, 1])
            for n_best in sorted({1, beam}):
                _assert_equal_restatement(x, ll, mode, tmpdir_bias, phrases, weights, beam, n_best, wip=0.3)
                n += 1
    assert n == 2 * (5 * 2 - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["lm_free", "chars", "tokens"])
def test_kernel_equals_restatement_dtypes_layouts_batch(mode, tmpdir_bias):
    """Every input dtype; raw logits and time-major input through CTCDecoder; B = 150 (256-thread variant); 1000
    phrases."""
    from end2end_b200 import PhraseBias
    labels, marker, model, lm, lmwt, oovp = _mode(mode, tmpdir_bias)
    phrases = _phrases_for(labels, 40, 7)
    weights = [1.2] * len(phrases)
    x = _spelling_logits(4, 30, labels, phrases, 6)
    ll = torch.tensor([30, 20, 3, 1])
    for dtype in (torch.float32, torch.float64, torch.bfloat16, torch.float16):
        for n_best in (1, 25):
            _assert_equal_restatement(x.to(dtype), ll, mode, tmpdir_bias, phrases, weights, 25, n_best, wip=0.5)
    g = torch.Generator().manual_seed(8)
    raw = torch.randn(5, 40, len(labels), generator=g) * 2.0
    raw += _spelling_logits(5, 40, labels, phrases, 9).float()
    rl = torch.randint(20, 41, (5,), generator=g)
    bias = PhraseBias(phrases, weights, labels=labels)
    for dtype, time_major in ((torch.float32, False), (torch.float64, True)):
        xin = raw.to(dtype)
        if time_major:
            xin = xin.transpose(0, 1)
        from end2end_b200 import CTCDecoder
        dec = CTCDecoder(beam_width=30, labels=labels, wip=0.5, lmwt=lmwt, oov_penalty=oovp, time_major=time_major)
        dec.word_marker = marker
        res = dec.decode_nbest(xin.cuda(), rl, n_best=10, lm=lm, bias=bias)
        want = restate_bias(xin, rl, model.loaded(), labels, bias.phrases, bias.weights, marker, 0, 30, 10, 0.5, lmwt,
                            oovp, after_logsoftmax=False, time_major=time_major)
        tol = 1e-12 if dtype == torch.float64 else 1e-6
        got = (res.decoded_targets, res.decoded_targets_lengths, res.scores, res.log_probs, res.lm_scores,
               res.oov_words, res.bias_scores, dec._decoder.last_ties)
        _check(got, want, (mode, dtype, time_major), lm is not None, tol)
    big = _spelling_logits(150, 20, labels, phrases, 12)
    big_ll = torch.randint(10, 21, (150,), generator=torch.Generator().manual_seed(13))
    for n_best in (1, 40):
        _assert_equal_restatement(big, big_ll, mode, tmpdir_bias, phrases, weights, 40, n_best, wip=0.4)
    many = _phrases_for(labels, 1000, 14)
    x = _spelling_logits(6, 24, labels, many, 15)
    _assert_equal_restatement(x, None, mode, tmpdir_bias, many, _weights(random.Random(3), len(many)), 40, 40, wip=0.4)


_PREFILTER_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from end2end_b200 import NGramLM, PhraseBias
from end2end_b200.engine import CTCBeamEngine
x, labels, path, phrases, out = torch.load(sys.argv[2])
lm = NGramLM.from_arpa(path)
eng = CTCBeamEngine(0, 100, labels, 0.3)
res = eng.decode_nbest_bias_device(x.cuda(), PhraseBias(phrases, 1.5, labels=labels), lm, None, 100, False, lmwt=0.8,
                                   oov_penalty=-2.0, word_marker="▁")
torch.save([t.cpu() for t in res], out)
"""


@pytest.mark.gpu
def test_large_alphabet_prefilter(tmpdir_bias):
    """V = 1024 sub-word labels, token LM, beam 100, 100 phrases: the filter (its selects rank labels in no phrase,
    every phrase label is extended) gives the restatement's result, and identical results with it off
    (E2E_CTC_BEAM_NOPREFILTER=1, read once per process: a child process; the uncached path)."""
    from end2end_b200 import NGramLM, PhraseBias
    V = 1024
    labels = _token_alphabet(V, 15)
    rng = random.Random(16)
    pieces = [lab.lstrip(MARK) for lab in labels[2:200]]
    words = sorted({"".join(rng.choice(pieces) for _ in range(rng.randint(1, 2))) for _ in range(300)})
    model = random_model(16, 3, words, per_order=300)
    path = model.write(os.path.join(tmpdir_bias, "v1024.arpa"))
    lm = NGramLM.from_arpa(path)
    phrases = [tuple(rng.randrange(1, V) for _ in range(rng.randint(1, 4))) for _ in range(100)]
    phrases = list(dict.fromkeys(phrases))
    x = _spelling_logits(3, 16, labels, phrases, 17, scale=3.0)
    bias = PhraseBias(phrases, 1.5, labels=labels)
    got = _kernel(x, None, bias, labels, lm, MARK, 0, 100, 100, 0.3, 0.8, -2.0)
    want = restate_bias(x, None, model.loaded(), labels, bias.phrases, bias.weights, MARK, 0, 100, 100, 0.3, 0.8, -2.0)
    _check(got, want, "v1024", True)
    assert bool((got[6][got[1] > 0] > 0).any())            # some hypotheses complete a phrase
    job = os.path.join(tmpdir_bias, "job.pt")
    out = os.path.join(tmpdir_bias, "nopre.pt")
    torch.save([x, labels, path, phrases, out], job)
    env = dict(os.environ, E2E_CTC_BEAM_NOPREFILTER="1")
    subprocess.check_call([sys.executable, "-c", _PREFILTER_SCRIPT, os.path.dirname(_HERE), job], env=env)
    other = torch.load(out)
    for a, b in zip(got, other):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["lm_free", "chars", "tokens"])
def test_unmatched_phrases_change_nothing(mode, tmpdir_bias):
    """Phrases that start with a label no kept prefix ever holds: the unbiased call's results, bit for bit."""
    from end2end_b200 import PhraseBias
    from end2end_b200.engine import CTCBeamEngine
    labels, marker, model, lm, lmwt, oovp = _mode(mode, tmpdir_bias)
    V = len(labels)
    x = _log_probs(6, 25, V, 21)
    x[:, :, V - 1] = -1e4
    x = torch.log_softmax(x, 2).cuda()
    bias = PhraseBias([(V - 1, 3), (V - 1,), (V - 1, V - 1, 2)], 2.0, labels=labels)
    eng = CTCBeamEngine(0, 16, labels, 0.4)
    got = eng.decode_nbest_bias_device(x, bias, lm, None, 16, False, lmwt=lmwt, oov_penalty=oovp, word_marker=marker)
    if lm is None:
        want = eng.decode_nbest_device(x, None, 16, False)
        idx = (0, 1, 2, 3, 7)
    else:
        want = eng.decode_nbest_lm_device(x, lm, None, 16, False, lmwt=lmwt, oov_penalty=oovp, word_marker=marker)
        idx = (0, 1, 2, 3, 4, 5, 7)
    for i, w in zip(idx, want):
        assert torch.equal(got[i].cpu(), w.cpu()), i
    live = got[1] > 0
    assert bool((got[6][live] == 0).all())


@pytest.mark.gpu
def test_bias_changes_the_winner(tmp_path):
    """Frames spelling "a c?t" with "a" slightly above "o" (LM-free: "a cat"), and with a model that knows "cat" only
    (a boosted "cet" is out of vocabulary, 3 log10 below "cat"): the boosted phrase wins when its bonus beats the model's
    and the frames' preference, and its hypothesis carries the bonus."""
    from end2end_b200 import CTCDecoder, NGramLM, PhraseBias
    labels = ["_", " "] + LETTERS
    idx = {c: i for i, c in enumerate(labels)}
    T = 8
    x = torch.full((1, T, len(labels)), -12.0)
    for t, spec in enumerate(["a", "_", " ", "c", {"a": -0.5, "o": -0.7, "e": -0.9}, "t", "_", "_"]):
        if isinstance(spec, dict):
            for c, v in spec.items():
                x[0, t, idx[c]] = v
        else:
            x[0, t, idx[spec]] = 0.0
    x = torch.log_softmax(x, 2)
    dec = CTCDecoder(beam_width=8, labels=labels, after_logsoftmax=True, wip=0.0, lmwt=1.0, oov_penalty=0.0)
    assert dec.decode(x.cuda()).decoded_sentences == ["a cat"]
    cot = PhraseBias(["cot"], 0.2, labels=labels)
    res = dec.decode_nbest(x, n_best=2, bias=cot)            # CPU logits go to the bias's device
    assert res.decoded_sentences[0] == ["a cot", "a cat"]
    assert res.bias_scores[0].tolist() == [0.2 * 3, 0.0]
    assert dec.decode(x, bias=cot).decoded_sentences == ["a cot"]
    arpa = tmp_path / "cat.arpa"
    arpa.write_text("\\data\\\nngram 1=5\n\n\\1-grams:\n-99\t<s>\n-1.0\t</s>\n-1.0\ta\n-1.0\tcat\n-4.0\t<unk>\n\n"
                    "\\end\\\n")
    lm = NGramLM.from_arpa(str(arpa))                        # cat against <unk>: 3 ln 10 = 6.9 nats, plus 0.4 acoustic
    assert dec.decode(x, lm=lm).decoded_sentences == ["a cat"]
    cet = PhraseBias(["cet"], 3.0, labels=labels)             # 9 nats once completed
    res = dec.decode_nbest(x, n_best=2, lm=lm, bias=cet)
    assert res.decoded_sentences[0] == ["a cet", "a cat"] and res.oov_words[0].tolist() == [1, 0]
    assert res.bias_scores[0].tolist() == [9.0, 0.0]
    small = PhraseBias(["cet"], 2.0, labels=labels)          # 6 nats: not enough
    assert dec.decode(x, lm=lm, bias=small).decoded_sentences == ["a cat"]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["lm_free", "tokens"])
def test_invariants(mode, tmpdir_bias):
    """decode(bias=) is hypothesis 0; scores are the unbiased expression plus bias_scores; two uploads agree."""
    from end2end_b200 import CTCDecoder, PhraseBias
    labels, marker, model, lm, lmwt, oovp = _mode(mode, tmpdir_bias)
    phrases = _phrases_for(labels, 30, 19)
    x = _spelling_logits(16, 60, labels, phrases, 20, scale=2.5).to(torch.float32).cuda()
    ll = torch.randint(20, 61, (16,), generator=torch.Generator().manual_seed(21))
    dec = CTCDecoder(beam_width=50, labels=labels, wip=0.5, lmwt=lmwt, oov_penalty=oovp, after_logsoftmax=True)
    dec.word_marker = marker
    b1, b2 = PhraseBias(phrases, 0.8, labels=labels), PhraseBias(phrases, 0.8, labels=labels)
    nb = dec.decode_nbest(x, ll, n_best=50, lm=lm, bias=b1)
    one = dec.decode(x, ll, lm=lm, bias=b1)
    w = one.decoded_targets.size(1)
    assert torch.equal(nb.decoded_targets[:, 0, :w], one.decoded_targets)
    assert torch.equal(nb.decoded_targets_lengths[:, 0], one.decoded_targets_lengths)
    assert [s[0] for s in nb.decoded_sentences] == one.decoded_sentences
    count = (lambda r: _words(r, labels, MARK)) if marker else (lambda r: _space_words(r, labels))
    words = torch.tensor([[count(r[:k]) if r[:k] != [-1] else 0 for r, k in zip(rows, lens)]
                          for rows, lens in zip(nb.decoded_targets.tolist(), nb.decoded_targets_lengths.tolist())],
                         dtype=torch.float64)
    live = nb.decoded_targets_lengths > 0
    expr = (((nb.log_probs + lmwt * nb.lm_scores) - words * 0.5) + nb.oov_words.double() * oovp) if lm is not None \
        else nb.log_probs - words * 0.5
    assert torch.equal((expr + nb.bias_scores)[live], nb.scores[live])
    assert bool((nb.bias_scores[live] > 0).any())
    for p, k, c in zip(nb.decoded_targets.tolist(), nb.decoded_targets_lengths.tolist(), nb.bias_scores.tolist()):
        for r, n, v in zip(p, k, c):
            if n > 0:
                assert v == py_committed([] if r[:n] == [-1] else r[:n], b1.phrases, b1.weights)
    again = dec.decode_nbest(x, ll, n_best=50, lm=lm, bias=b2)
    for f in nb._fields:
        a, b = getattr(nb, f), getattr(again, f)
        assert (a == b) if f == "decoded_sentences" else torch.equal(a, b), f


@pytest.mark.gpu
def test_argument_errors(tmpdir_bias):
    from end2end_b200 import CTCDecoder, PhraseBias
    labels = CHAR_LABELS
    bias = PhraseBias(["ab"], 1.0, labels=labels)
    x = torch.log_softmax(torch.randn(2, 5, len(labels)), 2)
    with pytest.raises(ValueError, match="greedy"):
        CTCDecoder(beam_width=1, labels=labels).decode(x, bias=bias)
    with pytest.raises(ValueError, match="labels"):
        CTCDecoder(beam_width=4, labels=labels + ["z"]).decode(torch.randn(2, 5, len(labels) + 1), bias=bias)
    # a shape past the kernel's shared memory is refused
    V = 6000
    big = torch.log_softmax(torch.randn(1, 2, V), 2).cuda()
    with pytest.raises(NotImplementedError):
        CTCDecoder(beam_width=256, labels=["_"] + ["w%d" % i for i in range(V - 1)]).decode(big, bias=PhraseBias([[1]], 1.0))

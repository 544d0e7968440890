"""The prefix beam search with a word n-gram language model fused in (CTCDecoder.decode / decode_nbest with lm=,
e2e_ctc_beam_lm_nbest_device, NGramLM).

The definition (words, vocabulary, when the LM scores, the backoff arithmetic, the score) is include/e2e_ctc.h's, at
e2e_ctc_ngram.  The checker is tests/beam_lm_restatement.c: beam_nbest_restatement.c's search with the LM state carried
per prefix, its n-grams found by a plain search over arrays and its words by spelling, so it shares nothing with the
device table or the lexicon trie.  The device-free tests pin it to beam_nbest_restatement.c (lmwt = 0) and, on beams that
hold every prefix, to brute force with the oracle's CTC log-likelihood and the pure-Python ARPA scorer of this module.
The GPU tests compare the kernel with it: hypotheses, lengths, order, OOV counts and tie counters bit for bit, scores,
log_probs and lm_scores within 1e-12 relative (CUDA's fp64 exp / log against the C library's).

ARPA models are generated here from a seed: random valid models of orders 1-6 and a small model estimated from a
hand-written corpus.
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
from test_gpu_beam_nbest import EXHAUSTIVE, beam_nbest

_HERE = os.path.dirname(os.path.abspath(__file__))
_RESTATEMENT_SRC = os.path.join(_HERE, "beam_lm_restatement.c")
_restatement_lib = None
LN10 = math.log(10.0)
LETTERS = [chr(ord("a") + i) for i in range(26)]
C2_LABELS = ["_", " "] + LETTERS + ["'"]


def _restatement():
    """gcc the C restatement into a temporary directory (once per process; the tree is left untouched)."""
    global _restatement_lib
    if _restatement_lib is None:
        d = tempfile.mkdtemp(prefix="beam_lm_restatement_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libbeam_lm_restatement.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-o", so,
                               _RESTATEMENT_SRC, "-lm"])
        L = ctypes.CDLL(so)
        dp, ip, i32p = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int32)
        ci, cd = ctypes.c_int, ctypes.c_double
        L.ctc_beam_lm_nbest.argtypes = [dp, ci, ci, ci, ip, ci, ci, ci, ci, cd, cd, cd, ci, ci, i32p, i32p, dp, dp, ci,
                                        i32p, i32p, i32p, i32p, ci, ci, ci, ip, ip, dp, dp, dp, ip, ip]
        L.ctc_beam_lm_nbest.restype = None
        _restatement_lib = L
    return _restatement_lib


# ---------------------------------------------------------------------------------------------- models ---------------

class Model:
    """An ARPA model as Python data: ``ngrams[k-1] = {words: (log10 prob, log10 backoff)}``, ``vocab`` in file order."""

    def __init__(self, ngrams, has_unk=True):
        self.ngrams = ngrams
        self.order = len(ngrams)
        self.has_unk = has_unk

    def write(self, path, bow_always=False):
        with open(path, "w") as f:
            f.write("\n\\data\\\n")
            for k, t in enumerate(self.ngrams, 1):
                f.write("ngram %d=%d\n" % (k, len(t)))
            for k, t in enumerate(self.ngrams, 1):
                f.write("\n\\%d-grams:\n" % k)
                for words, (p, b) in t.items():
                    if k < self.order and (b != 0.0 or bow_always):
                        f.write("%r\t%s\t%r\n" % (p, " ".join(words), b))
                    else:
                        f.write("%r\t%s\n" % (p, " ".join(words)))
            f.write("\n\\end\\\n")
        return path

    def loaded(self):
        """What the loader makes of it: <unk> added with -100 / 0 when missing."""
        ng = [dict(t) for t in self.ngrams]
        if ("<unk>",) not in ng[0]:
            ng[0][("<unk>",)] = (-100.0, 0.0)
        return ng


def random_model(seed, order, words, with_unk=True, per_order=40):
    """A valid random model: every word a unigram, higher orders over existing contexts."""
    rng = random.Random(seed)
    vocab = ["<s>", "</s>"] + list(words) + (["<unk>"] if with_unk else [])
    ng = [dict() for _ in range(order)]
    for w in vocab:
        ng[0][(w,)] = (-99.0 if w == "<s>" else round(rng.uniform(-4.0, -0.3), 6),
                       0.0 if w == "</s>" else round(rng.uniform(-1.5, 0.5), 6))
    for k in range(2, order + 1):
        ctxs = [c for c in ng[k - 2] if c[-1] != "</s>"]
        for _ in range(per_order):
            c = rng.choice(ctxs)
            w = rng.choice([x for x in vocab if x != "<s>"])
            if c + (w,) not in ng[k - 1]:
                ng[k - 1][c + (w,)] = (round(rng.uniform(-3.0, -0.05), 6),
                                       0.0 if (k == order or w == "</s>") else round(rng.uniform(-1.0, 0.3), 6))
    return Model(ng, with_unk)


CORPUS = """a cot
the cat sat on a cot
she is on a cot
a cot is a cot
the cat sat on the mat"""


def corpus_model():
    """A bigram model estimated from CORPUS by absolute discounting (D = 0.5) with backoff to the unigrams."""
    sents = [["<s>"] + s.split() + ["</s>"] for s in CORPUS.splitlines()]
    uni, bi = {}, {}
    for s in sents:
        for w in s[1:]:
            uni[w] = uni.get(w, 0) + 1
        for a, b in zip(s, s[1:]):
            bi[(a, b)] = bi.get((a, b), 0) + 1
    total = sum(uni.values())
    ctx = {}
    for (a, b), c in bi.items():
        ctx.setdefault(a, []).append(c)
    ng1, ng2 = {}, {}
    for w in ["<s>"] + sorted(uni):
        p = -99.0 if w == "<s>" else math.log10(uni[w] / total)
        if w in ctx:
            n = sum(ctx[w])
            seen = sum(uni[b] / total for (a, b) in bi if a == w)
            bow = math.log10((0.5 * len(ctx[w]) / n) / (1.0 - seen))
        else:
            bow = 0.0
        ng1[(w,)] = (p, bow)
    for (a, b), c in bi.items():
        ng2[(a, b)] = (math.log10((c - 0.5) / sum(ctx[a])), 0.0)
    return Model([ng1, ng2], has_unk=False)


def py_term(ng, order, hist, w):
    """ln10 * log10 P(w | hist) with ARPA backoff, restated independently of the C and CUDA code."""
    ctx = tuple(hist[-(order - 1):]) if order > 1 else ()
    t = 0.0
    while True:
        e = ng[len(ctx)].get(ctx + (w,)) if len(ctx) + 1 <= order else None
        if e is not None:
            t += e[0]
            break
        if not ctx:
            break
        b = ng[len(ctx) - 1].get(ctx)
        if b is not None:
            t += b[1]
        ctx = ctx[1:]
    return t * LN10


def py_lm(ng, order, text, case_sensitive=True):
    """(lm, oov) of a whole hypothesis text (words split on spaces), </s> included."""
    vocab = {w[0] for w in ng[0]} - {"<s>", "</s>", "<unk>"}
    hist, lm, oov = ["<s>"], 0.0, 0
    for word in text.split(" "):
        if not word:
            continue
        if not case_sensitive:
            word = word.lower()
        if word not in vocab:
            word, oov = "<unk>", oov + 1
        lm += py_term(ng, order, hist, word)
        hist.append(word)
    lm += py_term(ng, order, hist, "</s>")
    return lm, oov


# ---------------------------------------------------------------------------------------------- restatement ----------

def _lm_arrays(ng, labels, blank, case_sensitive):
    vocab = [w[0] for w in ng[0]]
    wid = {w: i for i, w in enumerate(vocab)}
    rows = [(k + 1, words, pb) for k, t in enumerate(ng) for words, pb in t.items()]
    ids = np.full((len(rows), 6), -1, dtype=np.int32)
    for i, (k, words, _) in enumerate(rows):
        ids[i, :k] = [wid[w] for w in words]
    n = np.array([r[0] for r in rows], dtype=np.int32)
    prob = np.array([r[2][0] for r in rows], dtype=np.float64)
    bow = np.array([r[2][1] for r in rows], dtype=np.float64)
    off, chars, ok = [0], [], []
    for w in vocab:
        spell = w not in ("<s>", "</s>", "<unk>")
        ok.append(1 if spell else 0)
        if spell:
            chars.extend(ord(ch) for ch in w)
        off.append(len(chars))
    cp = []
    for i, lab in enumerate(labels):
        if i == blank or lab == " ":
            cp.append(-1)
        else:
            f = lab if case_sensitive else lab.lower()
            cp.append(ord(f) if len(f) == 1 else -2)
    arr = lambda x: np.ascontiguousarray(np.array(x, dtype=np.int32))   # noqa: E731
    return (ids, n, prob, bow, len(vocab), arr(off), arr(chars if chars else [0]), arr(ok), arr(cp),
            wid["<s>"], wid["</s>"], wid["<unk>"])


def restate(logits, ll, ng, labels, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0,
            case_sensitive=True, after_logsoftmax=True, time_major=False):
    """The restatement's (targets [B,N,Tw], lengths, scores, log_probs, lm_scores, oov_words, ties), driven as
    test_gpu_beam_nbest.beam_nbest drives beam_nbest_restatement.c."""
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
    ids, n, prob, bow, nv, off, chars, ok, cp, bos, eos, unk = _lm_arrays(ng, labels, blank, case_sensitive)
    P = lambda a, t: a.ctypes.data_as(ctypes.POINTER(t))   # noqa: E731
    d, i64, i32 = ctypes.c_double, ctypes.c_int64, ctypes.c_int32
    _restatement().ctc_beam_lm_nbest(
        P(x, d), B, T, V, P(il, i64), int(blank), int(beam), N, labels.index(" "), float(wip), float(lmwt),
        float(oov_penalty), len(ng), len(n), P(ids, i32), P(n, i32), P(prob, d), P(bow, d), nv, P(off, i32),
        P(chars, i32), P(ok, i32), P(cp, i32), bos, eos, unk, P(out, i64), P(out_len, i64), P(scores, d),
        P(log_probs, d), P(lm_scores, d), P(oov, i64), P(ties, i64))
    return tuple(torch.from_numpy(a) for a in (out, out_len, scores, log_probs, lm_scores, oov, ties))


def _words(seq, space):
    n, last = 0, -1
    for c in seq:
        if c != space and (n == 0 or last == space):
            n += 1
        last = c
    return n


def _text(seq, labels):
    return "".join(labels[c] for c in seq if c >= 0)


def _labels(V):
    """blank, space, then V - 2 letters."""
    return ["_", " "] + LETTERS[:V - 2]


def _log_probs(B, T, V, seed, scale=2.0, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    return torch.log_softmax(torch.randn(B, T, V, generator=g, dtype=torch.float64) * scale, 2).to(dtype)


# ---------------------------------------------------------------------------------------------- device-free ---------

def _arpa_text(body):
    return "\\data\\\n" + body


@pytest.mark.parametrize("case,text", [
    ("count", "ngram 1=3\n\n\\1-grams:\n-1 <s>\n-1 </s>\n\n\\end\\\n"),
    ("no_end", "ngram 1=2\n\n\\1-grams:\n-1 <s>\n-1 </s>\n"),
    ("nan", "ngram 1=2\n\n\\1-grams:\n-1 <s>\nnan </s>\n\n\\end\\\n"),
    ("inf", "ngram 1=2\n\n\\1-grams:\n-1 <s>\n-inf </s>\n\n\\end\\\n"),
    ("order7", "".join("ngram %d=1\n" % k for k in range(1, 8)) + "\n\\1-grams:\n-1 <s>\n\n\\end\\\n"),
    ("context", "ngram 1=3\nngram 2=1\n\n\\1-grams:\n-1 <s>\n-1 </s>\n-1 a\n\n\\2-grams:\n-1 b a\n\n\\end\\\n"),
    ("duplicate", "ngram 1=3\n\n\\1-grams:\n-1 <s>\n-1 </s>\n-2 <s>\n\n\\end\\\n"),
    ("fields", "ngram 1=2\n\n\\1-grams:\n-1 <s> 0 7\n-1 </s>\n\n\\end\\\n"),
])
def test_parser_errors(tmp_path, case, text):
    from end2end_b200.lm.ngram import parse_arpa
    p = tmp_path / ("%s.arpa" % case)
    p.write_text(_arpa_text(text))
    with pytest.raises(ValueError):
        parse_arpa(str(p))


def test_parser_binary_and_unk(tmp_path):
    from end2end_b200.lm.ngram import parse_arpa
    p = tmp_path / "lm.binary"
    p.write_bytes(b"mmap lm http://kheafield.com/code format version 5\n\x00\x01\x02")
    with pytest.raises(ValueError, match="binary"):
        parse_arpa(str(p))
    m = random_model(1, 3, ["ab", "ba", "a"], with_unk=False)
    vocab, ng = parse_arpa(m.write(str(tmp_path / "nounk.arpa")))
    assert vocab[-1] == "<unk>" and ng[0][("<unk>",)] == (-100.0, 0.0)
    assert ng == m.loaded()
    m = random_model(2, 6, ["ab", "ba", "a"], with_unk=True)
    path = str(tmp_path / "unk.arpa")
    with open(path, "w") as f:   # any whitespace between fields, explicit zero backoffs
        f.write(open(m.write(path + ".tmp", bow_always=True)).read().replace("\t", "  \t "))
    vocab, ng = parse_arpa(path)
    assert ng == m.loaded() and vocab.count("<unk>") == 1 and len(ng) == 6


def test_restatement_lmwt0_equals_lm_free():
    """lmwt = 0 and oov_penalty = 0: the LM search is beam_nbest_restatement.c's, bit for bit (ties included)."""
    ng = random_model(3, 3, ["ab", "b", "ba", "abc", "c"]).loaded()
    for V, beam, n_best, wip in ((5, 10, 10, 0.4), (5, 3, 2, 0.0), (4, 40, 7, 0.7)):
        lp = _log_probs(4, 12, V, 10 * V + beam)
        ll = torch.tensor([12, 7, 1, 3])
        labels = _labels(V)
        t, n, sc, lpr, lm, oov, ties = restate(lp, ll, ng, labels, beam=beam, n_best=n_best, wip=wip, lmwt=0.0)
        ot, on, osc, olp, oties = beam_nbest(lp, ll, beam_width=beam, n_best=n_best, labels=labels, after_logsoftmax=True,
                                             wip=wip)
        assert torch.equal(t, ot) and torch.equal(n, on) and torch.equal(ties, oties)
        assert torch.equal(sc, osc) and torch.equal(lpr, olp)
        assert bool(torch.isfinite(lm[n > 0]).all())


def _brute_force(lp, V, T, labels, ng, order, lmwt, wip, oov_penalty, case_sensitive=True):
    """Every label string over the non-blank labels up to length T, scored with the oracle's CTC log-likelihood and the
    Python scorer; sorted by score, highest first."""
    seqs = [[]]
    frontier = [[]]
    for _ in range(T):
        frontier = [s + [c] for s in frontier for c in range(1, V)]
        seqs += frontier
    k = len(seqs)
    width = max(1, T)
    tg = torch.zeros(k, width, dtype=torch.int64)
    for i, s in enumerate(seqs):
        if s:
            tg[i, :len(s)] = torch.tensor(s)
    tl = torch.tensor([len(s) for s in seqs])
    loss, _ = oracle.PortEngine(0).compute(lp.expand(k, -1, -1).contiguous(), tg, torch.full((k,), T, dtype=torch.int64), tl)
    out = []
    for i, s in enumerate(seqs):
        lm, oov = py_lm(ng, order, _text(s, labels), case_sensitive)
        ll = -float(loss[i])
        sc = ((ll + lmwt * lm) - _words(s, 1) * wip) + oov * oov_penalty
        out.append((sc, ll, lm, oov, s))
    out.sort(key=lambda r: -r[0] if math.isfinite(r[0]) else math.inf)
    return out


def _check_brute(t, n, sc, lpr, lm, oov, brute, lmwt, wip, oov_penalty, labels, ng, order):
    k = int((n > 0).sum())
    fin = [r for r in brute if math.isfinite(r[0])]
    assert int(torch.isfinite(sc[:k]).sum()) == len(fin)
    for r in range(k):
        seq = t[r, :int(n[r])].tolist()
        seq = [] if seq == [-1] else seq
        want_lm, want_oov = py_lm(ng, order, _text(seq, labels))
        assert int(oov[r]) == want_oov
        assert math.isclose(float(lm[r]), want_lm, rel_tol=1e-12, abs_tol=1e-300)
        if not math.isfinite(float(sc[r])):
            continue
        want = ((float(lpr[r]) + lmwt * want_lm) - _words(seq, 1) * wip) + want_oov * oov_penalty
        assert math.isclose(float(sc[r]), want, rel_tol=1e-12)
        b = fin[r]
        assert math.isclose(float(sc[r]), b[0], rel_tol=1e-10), (r, float(sc[r]), b)
        unique = all(abs(b[0] - o[0]) > 1e-9 * abs(b[0]) for o in fin if o is not b)
        if unique:
            assert seq == b[4], (r, seq, b)


@pytest.mark.parametrize("V,T", [vt for vt in EXHAUSTIVE if vt[0] >= 3])
def test_restatement_exhaustive_matches_brute_force(V, T):
    labels = _labels(V)
    m = random_model(7 * V + T, 3, ["a", "aa", "ab", "ba", "b"], with_unk=(T % 2 == 0))
    ng = m.loaded()
    lmwt, wip, oovp = 0.8, 0.3, -1.5
    lp = _log_probs(2, T, V, 100 * V + T, scale=1.5)
    t, n, sc, lpr, lm, oov, _ = restate(lp, None, ng, labels, beam=256, n_best=256, wip=wip, lmwt=lmwt, oov_penalty=oovp)
    for b in range(lp.size(0)):
        brute = _brute_force(lp[b:b + 1], V, T, labels, ng, m.order, lmwt, wip, oovp)
        _check_brute(t[b], n[b], sc[b], lpr[b], lm[b], oov[b], brute, lmwt, wip, oovp, labels, ng, m.order)


def test_py_scorer_known_answers():
    m = corpus_model()
    ng = m.loaded()
    # seen bigrams, then a backoff: P(mat | cat) backs off to the unigram
    p_the = ng[1][("<s>", "the")][0]
    p_cat = ng[1][("the", "cat")][0]
    p_mat = ng[0][("cat",)][1] + ng[0][("mat",)][0]
    p_end = ng[1][("mat", "</s>")][0]
    lm, oov = py_lm(ng, 2, "the cat mat")
    assert oov == 0 and lm == ((((0.0 + p_the) * LN10 + p_cat * LN10) + p_mat * LN10) + p_end * LN10)
    assert math.isclose(lm, (p_the + p_cat + p_mat + p_end) * LN10, rel_tol=1e-14)
    lm, oov = py_lm(ng, 2, " dog  the ")
    assert oov == 1


# ---------------------------------------------------------------------------------------------- GPU -----------------

_MODELS = {}


def _lm(model, tmp, key=None):
    """NGramLM of a Model, loaded from an ARPA file written into ``tmp`` (cached per key)."""
    from end2end_b200 import NGramLM
    key = key or repr(model.ngrams)
    if key not in _MODELS:
        path = model.write(os.path.join(tmp, "m%d.arpa" % len(_MODELS)))
        _MODELS[key] = NGramLM.from_arpa(path)
    return _MODELS[key]


@pytest.fixture(scope="module")
def tmpdir_lm():
    d = tempfile.mkdtemp(prefix="beam_lm_models_")
    yield d
    shutil.rmtree(d, True)
    _MODELS.clear()


def _kernel(x, ll, lm, labels, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0, case_sensitive=True,
            from_logits=False):
    from end2end_b200.engine import CTCBeamEngine
    eng = CTCBeamEngine(blank, beam, labels, wip)
    out = eng.decode_nbest_lm_device(x.cuda(), lm, None if ll is None else ll.cuda(), n_best, from_logits, lmwt=lmwt,
                                     oov_penalty=oov_penalty, case_sensitive=case_sensitive)
    return [t.cpu() for t in out]


def _close(got, want, rtol, ctx=None):
    fin = torch.isfinite(want)
    assert torch.equal(fin, torch.isfinite(got)) and torch.equal(got[~fin], want[~fin]), ctx
    assert torch.allclose(got[fin], want[fin], rtol=rtol, atol=0), (ctx, (got[fin] - want[fin]).abs().max())


def _assert_equal_restatement(x, ll, model, lm, labels, blank=0, beam=10, n_best=1, wip=0.0, lmwt=1.0, oov_penalty=0.0,
                              case_sensitive=True):
    got = _kernel(x, ll, lm, labels, blank, beam, n_best, wip, lmwt, oov_penalty, case_sensitive)
    want = restate(x, ll, model.loaded(), labels, blank, beam, n_best, wip, lmwt, oov_penalty, case_sensitive)
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
def test_kernel_equals_restatement_orders_beams(tmpdir_lm):
    """Orders 1-6 with and without <unk>, beams 1, 2, 7, 100 and 256, N = 1 and the full beam, both case modes."""
    labels = ["_", " ", "a", "b", "C", "c", "d"]
    words = ["a", "ab", "ba", "c", "cab", "dd", "Cab", "bad", "abc"]
    V = len(labels)
    n = 0
    for order in range(1, 7):
        model = random_model(100 + order, order, words, with_unk=order % 2 == 0)
        lm = _lm(model, tmpdir_lm)
        for beam in (1, 2, 7, 100, 256):
            T = 14 if beam >= 100 else 20
            x = _log_probs(3, T, V, 1000 * order + beam)
            ll = torch.tensor([T, T // 2, 1])
            for n_best in sorted({1, beam}):
                for cs in (True, False):
                    _assert_equal_restatement(x, ll, model, lm, labels, 0, beam, n_best, wip=0.3, lmwt=0.7,
                                              oov_penalty=-2.0, case_sensitive=cs)
                    n += 1
    assert n == 6 * 5 * 2 * 2 - 6 * 2


@pytest.mark.gpu
def test_kernel_equals_restatement_dtypes_layouts(tmpdir_lm):
    """Every input dtype on log-probabilities; raw logits (fused log-softmax) and time-major views through CTCDecoder."""
    from end2end_b200 import CTCDecoder
    model = random_model(5, 3, ["the", "cat", "cot", "a", "at", "to", "tea"])
    lm = _lm(model, tmpdir_lm)
    x = _log_probs(4, 30, 29, 6)
    ll = torch.tensor([30, 20, 3, 1])
    for dtype in (torch.float32, torch.float64, torch.bfloat16, torch.float16):
        for n_best in (1, 25):
            _assert_equal_restatement(x.to(dtype), ll, model, lm, C2_LABELS, 0, 25, n_best, wip=0.5, lmwt=1.2,
                                      oov_penalty=-3.0)
    g = torch.Generator().manual_seed(8)
    raw = torch.randn(5, 40, 29, generator=g) * 2.0
    rl = torch.randint(20, 41, (5,), generator=g)
    for dtype, time_major, where in ((torch.float32, False, "cuda"), (torch.float64, True, "cuda"),
                                     (torch.float32, True, "cpu")):
        xin = raw.to(dtype)
        if time_major:
            xin = xin.transpose(0, 1)
        dec = CTCDecoder(beam_width=30, labels=C2_LABELS, wip=0.5, lmwt=1.1, oov_penalty=-2.5, time_major=time_major)
        res = dec.decode_nbest(xin.cuda() if where == "cuda" else xin, rl, n_best=10, lm=lm)
        ot, on, osc, olp, olm, ooov, _ = restate(xin, rl, model.loaded(), C2_LABELS, 0, 30, 10, 0.5, 1.1, -2.5,
                                                 after_logsoftmax=False, time_major=time_major)
        tol = 1e-12 if dtype == torch.float64 else 1e-6
        ctx = (dtype, time_major, where)
        assert torch.equal(res.decoded_targets_lengths, on) and torch.equal(res.oov_words, ooov), ctx
        w = res.decoded_targets.size(2)
        assert torch.equal(res.decoded_targets, ot[:, :, :w]) and not bool(ot[:, :, w:].any()), ctx
        _close(res.scores, osc, tol)
        _close(res.log_probs, olp, tol)
        _close(res.lm_scores, olm, 1e-12)
        assert res.decoded_sentences[0][0] == _text(ot[0, 0, :int(on[0, 0])].tolist(), C2_LABELS)


@pytest.mark.gpu
def test_spaces_empty_prefix_and_large_batch(tmpdir_lm):
    """Leading, trailing and doubled spaces; the empty best prefix (-1, scored </s> | <s>); B = 150 > 148 SMs (the
    256-thread CTA)."""
    model = random_model(9, 2, ["ab", "b", "ba"])
    lm = _lm(model, tmpdir_lm)
    labels = ["_", " ", "a", "b"]
    T = 12
    x = torch.full((3, T, 4), -30.0, dtype=torch.float64)
    x[0, :, 0] = 0.0                                          # all blank: the empty prefix
    spell = [1, 0, 2, 3, 1, 0, 1, 3, 1, 0, 1, 0]             # " ab  b  ": leading, doubled and trailing spaces
    for t, c in enumerate(spell):
        x[1, t, c] = 0.0
    x[2] = _log_probs(1, T, 4, 11)[0]
    x = torch.log_softmax(x, 2)
    t, n, sc, lpr, lms, oov, _ = _assert_equal_restatement(x, None, model, lm, labels, 0, 8, 8, wip=0.2, lmwt=1.0,
                                                           oov_penalty=-1.0)
    assert t[0, 0, 0] == -1 and n[0, 0] == 1
    ng = model.loaded()
    assert math.isclose(float(lms[0, 0]), py_term(ng, 2, ["<s>"], "</s>"), rel_tol=1e-12)
    assert _text(t[1, 0, :int(n[1, 0])].tolist(), labels) == " ab  b  "
    want_lm, want_oov = py_lm(ng, 2, " ab  b  ")
    assert math.isclose(float(lms[1, 0]), want_lm, rel_tol=1e-12) and int(oov[1, 0]) == want_oov
    big = _log_probs(150, 20, 29, 12)
    big_ll = torch.randint(10, 21, (150,), generator=torch.Generator().manual_seed(13))
    model = random_model(14, 4, ["the", "cat", "a", "at", "tea", "eat"])
    lm = _lm(model, tmpdir_lm)
    for n_best in (1, 40):
        _assert_equal_restatement(big, big_ll, model, lm, C2_LABELS, 0, 40, n_best, wip=0.4, lmwt=0.9, oov_penalty=-2.0)


_PREFILTER_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from end2end_b200 import NGramLM
from end2end_b200.engine import CTCBeamEngine
x, labels, path, out = torch.load(sys.argv[2])
lm = NGramLM.from_arpa(path)
eng = CTCBeamEngine(0, 100, labels, 0.3)
res = eng.decode_nbest_lm_device(x.cuda(), lm, None, 100, False, lmwt=0.8, oov_penalty=-2.0)
torch.save([t.cpu() for t in res], out)
"""


@pytest.mark.gpu
def test_large_alphabet_prefilter(tmpdir_lm):
    """V = 300 one-character labels at beam 100: only the 102 most probable symbols plus the space are extended; the
    result is the restatement's, and identical with the filter switched off (E2E_CTC_BEAM_NOPREFILTER=1, read once per
    process: a child process)."""
    V = 300
    labels = ["_", " "] + [chr(0x400 + i) for i in range(V - 2)]
    rng = random.Random(15)
    words = ["".join(rng.choice(labels[2:60]) for _ in range(rng.randint(1, 3))) for _ in range(200)]
    model = random_model(16, 3, sorted(set(words)), per_order=300)
    path = model.write(os.path.join(tmpdir_lm, "v300.arpa"))
    from end2end_b200 import NGramLM
    lm = NGramLM.from_arpa(path)
    x = _log_probs(3, 16, V, 17, scale=3.0)
    x[:, :, 2:60] += 2.0                                    # words of the model are likely
    x = torch.log_softmax(x, 2)
    got = _assert_equal_restatement(x, None, model, lm, labels, 0, 100, 100, wip=0.3, lmwt=0.8, oov_penalty=-2.0)
    job = os.path.join(tmpdir_lm, "job.pt")
    out = os.path.join(tmpdir_lm, "nopre.pt")
    torch.save([x, labels, path, out], job)
    env = dict(os.environ, E2E_CTC_BEAM_NOPREFILTER="1")
    subprocess.check_call([sys.executable, "-c", _PREFILTER_SCRIPT, os.path.dirname(_HERE), job], env=env)
    other = torch.load(out)
    for a, b in zip(got, other):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_invariants(tmpdir_lm):
    from end2end_b200 import CTCDecoder, NGramLM
    model = random_model(18, 3, ["the", "cat", "cot", "a", "at", "to", "tea"])
    path = model.write(os.path.join(tmpdir_lm, "inv.arpa"))
    lm, lm2 = NGramLM.from_arpa(path), NGramLM.from_arpa(path)
    x, _, ll, _ = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    x, ll = x[:16].cuda(), ll[:16]
    # lmwt = 0, oov_penalty = 0: the LM-free search, bit for bit, ties included
    free = CTCDecoder(beam_width=50, labels=C2_LABELS, wip=0.5)
    zero = CTCDecoder(beam_width=50, labels=C2_LABELS, wip=0.5, lmwt=0.0, oov_penalty=0.0)
    a = free.decode_nbest(x, ll, n_best=50)
    ta = free._decoder.last_ties.clone()
    b = zero.decode_nbest(x, ll, n_best=50, lm=lm)
    tb = zero._decoder.last_ties.clone()
    assert torch.equal(a.decoded_targets, b.decoded_targets) and torch.equal(a.decoded_targets_lengths,
                                                                             b.decoded_targets_lengths)
    assert torch.equal(a.scores, b.scores) and torch.equal(a.log_probs, b.log_probs) and torch.equal(ta, tb)
    # decode(lm=) is hypothesis 0; the scores are the expression of the parts; two runs and two builds agree
    dec = CTCDecoder(beam_width=50, labels=C2_LABELS, wip=0.5, lmwt=1.3, oov_penalty=-4.0)
    nb = dec.decode_nbest(x, ll, n_best=50, lm=lm)
    one = dec.decode(x, ll, lm=lm)
    w = one.decoded_targets.size(1)
    assert torch.equal(nb.decoded_targets[:, 0, :w], one.decoded_targets)
    assert torch.equal(nb.decoded_targets_lengths[:, 0], one.decoded_targets_lengths)
    assert [s[0] for s in nb.decoded_sentences] == one.decoded_sentences
    words = torch.tensor([[_words(r[:k], 1) if r[:k] != [-1] else 0 for r, k in zip(rows, lens)]
                          for rows, lens in zip(nb.decoded_targets.tolist(), nb.decoded_targets_lengths.tolist())],
                         dtype=torch.float64)
    live = nb.decoded_targets_lengths > 0
    expr = ((nb.log_probs + 1.3 * nb.lm_scores) - words * 0.5) + nb.oov_words.double() * -4.0
    assert torch.equal(expr[live], nb.scores[live])
    assert bool((nb.scores[live] > -math.inf).all()) and bool((nb.scores[~live] == -math.inf).all())
    assert bool((nb.lm_scores[~live] == -math.inf).all()) and not bool(nb.oov_words[~live].any())
    for other in (lm, lm2):
        again = dec.decode_nbest(x, ll, n_best=50, lm=other)
        for f in ("decoded_targets", "decoded_targets_lengths", "scores", "log_probs", "lm_scores", "oov_words"):
            assert torch.equal(getattr(nb, f), getattr(again, f)), f


@pytest.mark.gpu
@pytest.mark.parametrize("V,T", [vt for vt in EXHAUSTIVE if vt[0] >= 3])
def test_exhaustive_kernel_matches_brute_force(V, T, tmpdir_lm):
    labels = _labels(V)
    m = random_model(7 * V + T, 3, ["a", "aa", "ab", "ba", "b"], with_unk=(T % 2 == 1))
    lm = _lm(m, tmpdir_lm)
    lmwt, wip, oovp = 0.8, 0.3, -1.5
    lp = _log_probs(2, T, V, 100 * V + T + 1, scale=1.5)
    t, n, sc, lpr, lms, oov, _ = _kernel(lp, None, lm, labels, 0, 256, 256, wip, lmwt, oovp)
    for b in range(lp.size(0)):
        brute = _brute_force(lp[b:b + 1], V, T, labels, m.loaded(), m.order, lmwt, wip, oovp)
        _check_brute(t[b], n[b], sc[b], lpr[b], lms[b], oov[b], brute, lmwt, wip, oovp, labels, m.loaded(), m.order)


@pytest.mark.gpu
def test_lm_changes_the_winner(tmpdir_lm):
    """Frames that spell "c?t" with a slightly stronger "a" than "o": without the LM "cat" wins; the corpus model
    prefers "cot" after "a" ("a cot"), and with lmwt > 0 the search keeps and picks it."""
    from end2end_b200 import CTCDecoder
    lm = _lm(corpus_model(), tmpdir_lm)
    ng = corpus_model().loaded()
    assert py_lm(ng, 2, "a cot")[0] > py_lm(ng, 2, "a cat")[0] + 1.0
    idx = {c: i for i, c in enumerate(C2_LABELS)}
    T = 9
    x = torch.full((1, T, 29), -12.0)
    for t, spec in enumerate(["a", " ", "c", "_", {"a": -0.6, "o": -0.8}, "t", "_", "_", "_"]):
        if isinstance(spec, dict):
            for c, v in spec.items():
                x[0, t, idx[c]] = v
        else:
            x[0, t, idx[spec]] = 0.0
    x = torch.log_softmax(x, 2)
    free = CTCDecoder(beam_width=8, labels=C2_LABELS, after_logsoftmax=True, wip=0.0, lmwt=0.0, oov_penalty=0.0)
    fused = CTCDecoder(beam_width=8, labels=C2_LABELS, after_logsoftmax=True, wip=0.0, lmwt=1.0, oov_penalty=0.0)
    assert free.decode(x.cuda(), lm=lm).decoded_sentences == ["a cat"]
    assert free.decode(x.cuda()).decoded_sentences == ["a cat"]
    assert fused.decode(x.cuda(), lm=lm).decoded_sentences == ["a cot"]
    assert fused.decode(x, lm=lm).decoded_sentences == ["a cot"]         # CPU logits go to the model's device


@pytest.mark.gpu
def test_argument_errors(tmpdir_lm):
    from end2end_b200 import CTCDecoder
    lm = _lm(random_model(19, 2, ["ab"]), tmpdir_lm)
    x = torch.log_softmax(torch.randn(2, 5, 4), 2)
    with pytest.raises(ValueError, match="greedy"):
        CTCDecoder(beam_width=1, labels=["_", " ", "a", "b"]).decode(x, lm=lm)
    with pytest.raises(ValueError, match="\" \""):
        CTCDecoder(beam_width=4, labels=["_", "c", "a", "b"]).decode(x, lm=lm)
    with pytest.raises(ValueError, match="one character"):
        CTCDecoder(beam_width=4, labels=["_", " ", "aa", "b"]).decode(x, lm=lm)
    with pytest.raises(NotImplementedError):
        CTCDecoder(beam_width=4, labels=["_", " ", "a", "b"], lm_path="/no/such.arpa").decode_nbest(x, n_best=2, lm=lm)
    with pytest.raises(ValueError, match="n_best"):
        CTCDecoder(beam_width=4, labels=["_", " ", "a", "b"]).decode_nbest(x, n_best=5, lm=lm)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError, match="language model on"):
            CTCDecoder(beam_width=4, labels=["_", " ", "a", "b"]).decode(x.to("cuda:1"), lm=lm)

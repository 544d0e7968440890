"""Word and token errors of N hypotheses per utterance against the utterance's reference (CTCDecoder.errors,
CTCBeamEngine.errors_device, e2e_ctc_edit_distance_device).

The checker is tests/edit_distance_restatement.c: the textbook Levenshtein table over (errors, substitutions) pairs with
words compared token by token, compiled into a temporary directory.  It is pinned here to brute-force enumeration of
every alignment on short sequences and, at word level, to token level over a host mapping of words to ids.  The kernel
computes integers, so every output is compared for equality.
"""
import atexit
import ctypes
import itertools
import os
import random
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import oracle

MAX_REF, MAX_HYP = 4095, 65535
SPACE = 1                       # the separator of the word-level tests: labels[1] == " "
LABELS = ["_", " "] + list("abcdefghijklmnopqrstuvwxyz'")      # V = 29 (c2)

_HERE = os.path.dirname(os.path.abspath(__file__))
_RESTATEMENT_SRC = os.path.join(_HERE, "edit_distance_restatement.c")
_restatement_lib = None


def _restatement():
    """gcc the C restatement into a temporary directory (once per process; the tree is left untouched)."""
    global _restatement_lib
    if _restatement_lib is None:
        d = tempfile.mkdtemp(prefix="edit_distance_restatement_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libedit_distance_restatement.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", so, _RESTATEMENT_SRC])
        L = ctypes.CDLL(so)
        ip, i, i64 = ctypes.POINTER(ctypes.c_int64), ctypes.c_int, ctypes.c_int64
        L.edit_restatement_pair.argtypes = [ip, i, ip, i, i64, ip]
        L.edit_restatement_pair.restype = i64
        L.edit_restatement.argtypes = [i, i, ip, i, ip, ip, i, ip, i64, ip, ip, ip, ip, ip]
        L.edit_restatement.restype = None
        _restatement_lib = L
    return _restatement_lib


def _iptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))


def pair(hyp, ref, sep=-1):
    """(errors, S, I, D, reference units) of one pair of token lists."""
    h = np.ascontiguousarray(hyp, dtype=np.int64).reshape(-1)
    r = np.ascontiguousarray(ref, dtype=np.int64).reshape(-1)
    out = np.zeros(4, dtype=np.int64)
    m = _restatement().edit_restatement_pair(_iptr(h), len(h), _iptr(r), len(r), sep, _iptr(out))
    return tuple(int(v) for v in out) + (int(m),)


def restated(hyps, hl, refs, rl, sep=-1):
    """The restatement on hyps [B, N, W], hl [B, N], refs [B, Wr], rl [B] (any layout / integer type): the five outputs
    as CPU int64 tensors."""
    hyps = np.ascontiguousarray(torch.as_tensor(hyps).cpu().to(torch.int64).numpy())
    refs = np.ascontiguousarray(torch.as_tensor(refs).cpu().to(torch.int64).numpy())
    hl = np.ascontiguousarray(torch.as_tensor(hl).cpu().to(torch.int64).numpy())
    rl = np.ascontiguousarray(torch.as_tensor(rl).cpu().to(torch.int64).numpy())
    B, N, W = hyps.shape
    outs = [np.zeros((B, N), dtype=np.int64) for _ in range(4)] + [np.zeros(B, dtype=np.int64)]
    _restatement().edit_restatement(B, N, _iptr(hyps), W, _iptr(hl), _iptr(refs), refs.shape[1], _iptr(rl), sep,
                                    *(_iptr(o) for o in outs))
    return tuple(torch.from_numpy(o) for o in outs)


def brute_force(hyp, ref):
    """Least errors, then most substitutions, over every alignment enumerated explicitly: (errors, S, I, D)."""
    best = None

    def walk(i, j, e, s, ins):
        nonlocal best
        if i == len(hyp) and j == len(ref):
            key = (e, -s)
            if best is None or key < best[0]:
                best = (key, (e, s, ins, e - s - ins))
            return
        if i < len(hyp) and j < len(ref):
            walk(i + 1, j + 1, e + (hyp[i] != ref[j]), s + (hyp[i] != ref[j]), ins)
        if i < len(hyp):
            walk(i + 1, j, e + 1, s, ins + 1)
        if j < len(ref):
            walk(i, j + 1, e + 1, s, ins)

    walk(0, 0, 0, 0, 0)
    return best[1]


def words_as_ids(rows, sep, table):
    """Rows of tokens -> rows of word ids (one id per distinct token sequence, shared through `table`)."""
    out = []
    for row in rows:
        words, cur = [], []
        for t in list(row) + [sep]:
            if t == sep:
                if cur:
                    words.append(table.setdefault(tuple(cur), len(table)))
                cur = []
            else:
                cur.append(t)
        out.append(words)
    return out


def word_rows(g, n_rows, width, V=6, sep=SPACE):
    """Random rows rich in separators and in words that share a prefix, differ only in length or in one inner token."""
    base = [[2, 3, 4], [2, 3], [2, 3, 4, 5], [2, 5, 4], [3], [2, 3, 4, 2]]
    rows = []
    for _ in range(n_rows):
        row = []
        while len(row) < width:
            if g.random() < 0.3:
                row.append(sep)
            elif g.random() < 0.5:
                row += base[g.randrange(len(base))]
            else:
                row.append(g.randrange(V))
        rows.append(row[:width])
    return rows


# ---------------------------------------------------------------------- device-free: the restatement -----------------

def test_restatement_equals_brute_force():
    """Every pair over a 3-symbol alphabet up to length 3, and random pairs up to length 6: total and split."""
    seqs = [s for n in range(4) for s in itertools.product(range(3), repeat=n)]
    for h in seqs:
        for r in seqs:
            got = pair(h, r)
            assert got[:4] == brute_force(h, r), (h, r, got)
            assert got[4] == len(r)
    g = random.Random(5)
    for _ in range(300):
        h = [g.randrange(3) for _ in range(g.randrange(7))]
        r = [g.randrange(3) for _ in range(g.randrange(7))]
        assert pair(h, r)[:4] == brute_force(h, r), (h, r)


def test_restatement_textbook_pairs():
    enc = lambda s: [ord(c) for c in s]     # noqa: E731
    assert pair(enc("sitting"), enc("kitten")) == (3, 2, 1, 0, 6)      # kitten -> sitting
    assert pair(enc("kitten"), enc("sitting")) == (3, 2, 0, 1, 7)
    assert pair(enc("lawn"), enc("flaw")) == (2, 0, 1, 1, 4)             # most substitutions among 2-error alignments
    assert pair(enc("execution"), enc("intention")) == brute_force(enc("execution"), enc("intention")) + (9,)
    assert pair(enc("execution"), enc("intention"))[0] == 5
    assert pair([], enc("abc")) == (3, 0, 0, 3, 3)
    assert pair(enc("abc"), []) == (3, 0, 3, 0, 0)
    assert pair([], []) == (0, 0, 0, 0, 0)


def test_restatement_word_level_is_token_level_over_word_ids():
    g = random.Random(7)
    table = {}
    for _ in range(400):
        h, r = word_rows(g, 1, g.randrange(25))[0], word_rows(g, 1, g.randrange(25))[0]
        hw, rw = words_as_ids([h, r], SPACE, table)
        assert pair(h, r, SPACE) == pair(hw, rw), (h, r)
    # separators are never units; equal words are the same token sequence, nothing less
    assert pair([SPACE, 2, 3, SPACE, SPACE, 4, SPACE], [2, 3, 4], SPACE) == (2, 1, 1, 0, 1)
    assert pair([SPACE, 2, 3, SPACE, SPACE, 4, SPACE], [2, 3, SPACE, 4], SPACE) == (0, 0, 0, 0, 2)
    assert pair([2, 3], [2, 3, 4], SPACE) == (1, 1, 0, 0, 1)          # a prefix is another word
    assert pair([2, 5, 4], [2, 3, 4], SPACE) == (1, 1, 0, 0, 1)       # one inner token differs
    assert pair([SPACE, SPACE], [2, SPACE, 3], SPACE) == (2, 0, 0, 2, 2)


# ---------------------------------------------------------------------- device-free: the C entry points --------------

def _edesc(B=2, N=3, W=10, Wr=8, itype=1, sep=-1):
    from end2end_b200 import _lib
    d = _lib.EditDesc()
    d.batch, d.n_hyp, d.hyp_width, d.ref_width = B, N, W, Wr
    d.tokens_itype = d.lengths_itype = itype
    d.separator = sep
    d.hyp_stride_b, d.ref_stride_b = W, Wr
    return d


def test_edit_workspace_query_limits(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    q = lambda d: L.e2e_ctc_edit_distance_workspace_bytes(ctypes.byref(d))   # noqa: E731
    for sep in (-1, SPACE):
        assert q(_edesc(Wr=MAX_REF, sep=sep)) == 256
        assert q(_edesc(Wr=MAX_REF + 1, sep=sep)) == 0
        assert "reference width 4096" in L.e2e_last_error_string().decode()
        assert q(_edesc(W=MAX_HYP, sep=sep)) == 256
        assert q(_edesc(W=MAX_HYP + 1, sep=sep)) == 0
        assert "hypothesis width 65536" in L.e2e_last_error_string().decode()
    assert q(_edesc(W=0, Wr=0)) == 256
    assert q(_edesc(B=1 << 16, N=(1 << 18) + 1)) == 0 and "grid" in L.e2e_last_error_string().decode()
    for bad in (_edesc(B=0), _edesc(N=0), _edesc(W=-1), _edesc(Wr=-1), _edesc(itype=2), _edesc(sep=-2)):
        assert q(bad) == 0
    bad = _edesc()
    bad.lengths_itype = -1
    assert q(bad) == 0 and "index type" in L.e2e_last_error_string().decode()


def test_edit_device_argument_errors(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    fake = ctypes.c_void_p(256)              # never dereferenced: every case fails before a launch
    # hyps, hyp_lengths, refs, ref_lengths, errors, S, I, D, reference_units, ws, ws_bytes, stream
    ok = [fake, fake, fake, fake, fake, fake, fake, fake, fake, None, 256, None]

    def call(desc, args):
        return L.e2e_ctc_edit_distance_device(ctypes.byref(desc) if desc is not None else None, *args)

    assert call(None, ok) == 1
    for i in range(9):
        args = list(ok)
        args[i] = None
        assert call(_edesc(), args) == 1 and "null pointer" in L.e2e_last_error_string().decode(), i
    # zero-width rows may be NULL; the call passes the pointer checks and stops at the (null) workspace
    assert call(_edesc(W=0, Wr=0), [None, fake, None, fake] + ok[4:]) == 3
    assert "workspace" in L.e2e_last_error_string().decode()
    for field, value in (("tokens_itype", 2), ("lengths_itype", 7), ("separator", -5)):
        d = _edesc()
        setattr(d, field, value)
        assert call(d, ok) == 1, field
    d = _edesc()
    d.hyp_stride_b = 9
    assert call(d, ok) == 1 and "row stride" in L.e2e_last_error_string().decode()
    d = _edesc()
    d.ref_stride_b = 7
    assert call(d, ok) == 1
    assert call(_edesc(Wr=MAX_REF + 1), ok) == 2
    for ws, n in ((None, 256), (ctypes.c_void_p(512), 255), (ctypes.c_void_p(384), 256)):   # null, short, misaligned
        args = list(ok)
        args[9], args[10] = ws, n
        assert call(_edesc(), args) == 3, (ws, n)


def test_python_errors_before_device_work(monkeypatch, lib_built):
    """Every argument error is raised on the host before anything touches a device (so this runs without one)."""
    from end2end_b200 import CTCDecoder, engine
    monkeypatch.setattr(engine, "_CUDA_OK", True)
    eng = engine.CTCBeamEngine(0, 1, LABELS)
    hyps, hl = torch.ones(2, 3, 4, dtype=torch.int64), torch.full((2, 3), 2)
    refs, rl = torch.ones(2, 5, dtype=torch.int32), torch.tensor([5, 0])
    cases = [(ValueError, (hyps, torch.full((2, 3), 5), refs, rl)),            # hypothesis length > width
             (ValueError, (hyps, torch.full((2, 3), -1), refs, rl)),
             (ValueError, (hyps, hl, refs, torch.tensor([6, 1]))),                # reference length > width
             (ValueError, (hyps, hl, refs, torch.tensor([-1, 1]))),
             (ValueError, (hyps, torch.full((2, 4), 2), refs, rl)),              # shapes
             (ValueError, (hyps, hl, refs[:1], rl)),
             (ValueError, (hyps, hl, refs, rl[:1])),
             (ValueError, (hyps[:, :0], hl[:, :0], refs, rl)),
             (ValueError, (hyps[0, 0], hl[0, 0], refs, rl)),
             (TypeError, (hyps.float(), hl, refs, rl)),
             (NotImplementedError, (hyps, hl, torch.ones(2, MAX_REF + 1, dtype=torch.int64), rl)),
             (NotImplementedError, (torch.ones(2, 1, MAX_HYP + 1, dtype=torch.int64), hl[:, :1], refs, rl))]
    for exc, args in cases:
        for words in (False, True):
            with pytest.raises(exc):
                eng.errors_device(*args, words=words)
    with pytest.raises(ValueError):
        engine.CTCBeamEngine(0, 1, ["_", "a"]).errors_device(hyps, hl, refs, rl, words=True)   # no " " label
    with pytest.raises(ValueError):
        CTCDecoder(labels=LABELS).errors(hyps, hl, refs, rl, level="char")


# ------------------------------------------------------------------------------------------------- GPU ---------------

def run(hyps, hl, refs, rl, words=False, labels=LABELS):
    from end2end_b200.engine import CTCBeamEngine
    return tuple(t.cpu() for t in CTCBeamEngine(0, 1, labels).errors_device(hyps, hl, refs, rl, words=words))


def assert_exact(hyps, hl, refs, rl, words=False, ctx=None):
    got = run(hyps, hl, refs, rl, words)
    if hyps.dim() == 2:
        hyps, hl = hyps[:, None], hl.reshape(-1, 1)
    want = restated(hyps, hl, refs, rl, SPACE if words else -1)
    for name, a, b in zip(("errors", "substitutions", "insertions", "deletions", "reference_units"), got, want):
        assert a.dtype == torch.int64 and a.shape == b.shape, (ctx, name, a.shape, b.shape)
        bad = (a != b).nonzero()
        assert bad.numel() == 0, (ctx, name, bad[:5].tolist(), a[tuple(bad[0])].item(), b[tuple(bad[0])].item())
    return got


def random_rows(g, shape, width, V, sep_rate=0.15):
    """Tokens in [0, V) with the space label at `sep_rate`, and lengths in [0, width] hitting 0, 1 and width."""
    t = torch.randint(2, V, shape + (width,), generator=g)
    t = torch.where(torch.rand(t.shape, generator=g) < sep_rate, torch.full_like(t, SPACE), t)
    lens = torch.randint(0, width + 1, shape, generator=g)
    flat = lens.reshape(-1)
    for k, v in enumerate((0, 1, width)):
        if flat.numel() > k:
            flat[k] = v
    return t, lens


# (B, hypothesis width, reference width, V) shaped after BASELINE's c1-c5 (c5's batch cut to keep the checker quick)
SHAPES = {"c1": (4, 50, 29, 28), "c2": (64, 300, 200, 29), "c3": (1024, 60, 40, 96), "c4": (128, 120, 80, 1024),
          "c5": (96, 800, 600, 29)}


@pytest.mark.gpu
@pytest.mark.parametrize("words", [False, True])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_exact_config_shapes(name, words):
    B, W, Wr, V = SHAPES[name]
    g = torch.Generator().manual_seed(10 * sorted(SHAPES).index(name) + words)
    N = 3 if name != "c3" else 2
    hyps, hl = random_rows(g, (B, N), W, V)
    refs, rl = random_rows(g, (B,), Wr, V)
    hyps[:, 1, :Wr] = refs                           # near matches: the reference with a few tokens changed
    hl[:, 1] = torch.minimum(rl, torch.full_like(rl, W))
    flip = torch.rand(B, Wr, generator=g) < 0.05
    hyps[:, 1, :Wr] = torch.where(flip, torch.randint(2, V, (B, Wr), generator=g), hyps[:, 1, :Wr])
    assert_exact(hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda(), words, ctx=name)


@pytest.mark.gpu
@pytest.mark.parametrize("words", [False, True])
@pytest.mark.parametrize("N", [1, 7, 8, 9, 100])
def test_exact_n_hypotheses(N, words):
    g = torch.Generator().manual_seed(N)
    B = 5
    hyps, hl = random_rows(g, (B, N), 70, 8)
    refs, rl = random_rows(g, (B,), 60, 8)
    assert_exact(hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda(), words, ctx=N)


@pytest.mark.gpu
@pytest.mark.parametrize("words", [False, True])
@pytest.mark.parametrize("Wr", [31, 32, 33, 63, 64, 65, 1023, 1024, MAX_REF])
def test_exact_reference_widths(Wr, words):
    """Reference widths around the lanes' cell boundaries (32 cells, then 2, ... 128 per lane)."""
    g = torch.Generator().manual_seed(Wr)
    B, N = 3, 9
    W = min(Wr + 40, 400)
    hyps, hl = random_rows(g, (B, N), W, 6, sep_rate=0.3 if words else 0.15)
    refs, rl = random_rows(g, (B,), Wr, 6, sep_rate=0.3 if words else 0.15)
    rl[0] = Wr
    hyps[1, 0, :min(W, Wr)] = refs[1, :min(W, Wr)]
    assert_exact(hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda(), words, ctx=Wr)


@pytest.mark.gpu
def test_words_separators_and_exact_equality():
    """Leading, trailing and doubled separators, all-separator rows, and words that share a prefix, differ only in
    length or in one inner token; at word level the kernel equals token level over the host's word ids."""
    g = random.Random(11)
    B, N, W, Wr = 40, 6, 48, 40
    refs = word_rows(g, B, Wr)
    hyps = [word_rows(g, N, W) for _ in range(B)]
    refs[0] = [SPACE] * Wr
    hyps[1][0] = [SPACE] * W
    hyps[2][0] = [SPACE, SPACE] + refs[2] + [SPACE] * (W - Wr - 2)           # the reference between extra separators
    hyps[3][0] = refs[3][:W] + [SPACE] * (W - Wr)
    assert all(len(r) == Wr for r in refs) and all(len(h) == W for hs in hyps for h in hs)
    rt, ht = torch.tensor(refs), torch.tensor(hyps)
    rl = torch.full((B,), Wr)
    hl = torch.randint(0, W + 1, (B, N), generator=torch.Generator().manual_seed(3))
    hl[:4, 0] = W
    got = assert_exact(ht.cuda(), hl.cuda(), rt.cuda(), rl.cuda(), words=True)
    table = {}
    for b in range(B):
        rw = words_as_ids([refs[b][:Wr]], SPACE, table)[0]
        assert got[4][b] == len(rw)
        for n in range(N):
            hw = words_as_ids([hyps[b][n][:int(hl[b, n])]], SPACE, table)[0]
            assert tuple(int(t[b, n]) for t in got[:4]) == pair(hw, rw)[:4], (b, n)


@pytest.mark.gpu
@pytest.mark.parametrize("words", [False, True])
def test_index_types_and_layouts(words):
    """int32 / int64 tokens and lengths, mixed, and non-contiguous [B, N, W] views: the same counts."""
    g = torch.Generator().manual_seed(21)
    B, N, W, Wr = 6, 5, 40, 35
    hyps, hl = random_rows(g, (B, N), W, 7)
    refs, rl = random_rows(g, (B,), Wr, 7)
    want = assert_exact(hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda(), words)
    for th, tr, lh, lr in itertools.product((torch.int32, torch.int64), repeat=4):
        got = run(hyps.to(th).cuda(), hl.to(lh).cuda(), refs.to(tr).cuda(), rl.to(lr).cuda(), words)
        assert all(torch.equal(a, b) for a, b in zip(got, want)), (th, tr, lh, lr)
    big = torch.zeros(N, B, 2 * W, dtype=torch.int64)
    big[:, :, ::2] = hyps.transpose(0, 1)
    view = big.transpose(0, 1)[:, :, ::2]                        # strided in every dimension
    rbig = torch.zeros(Wr + 3, B, dtype=torch.int32)
    rbig[:Wr] = refs.t()
    got = run(view.cuda(), hl.t().contiguous().t().cuda(), rbig.t()[:, :Wr].cuda(), rl.cuda(), words)
    assert all(torch.equal(a, b) for a, b in zip(got, want))


@pytest.fixture(scope="module")
def c2_nbest():
    from end2end_b200 import CTCDecoder
    x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    dec = CTCDecoder(beam_width=100, labels=LABELS)
    nb = dec.decode_nbest(x.cuda(), ll, n_best=100)
    return dec, x, tg, ll, tl, nb


@pytest.mark.gpu
@pytest.mark.parametrize("level", ["token", "word"])
def test_decode_nbest_c2_against_targets(c2_nbest, level):
    """decode_nbest's list of c2 against the batch's targets, through CTCDecoder.errors (unused slots: length 0)."""
    dec, x, tg, ll, tl, nb = c2_nbest
    got = dec.errors(nb.decoded_targets, nb.decoded_targets_lengths, tg, tl, level=level)
    hl = torch.where((nb.decoded_targets_lengths == 1) & (nb.decoded_targets[:, :, 0] == -1),
                     torch.zeros_like(nb.decoded_targets_lengths), nb.decoded_targets_lengths)
    want = restated(nb.decoded_targets, hl, tg, tl, SPACE if level == "word" else -1)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    assert (got.errors >= 0).all() and (got.insertions - got.deletions == _units(nb, hl, level) - got.reference_units[:, None]).all()


def _units(nb, hl, level):
    rows, lens = nb.decoded_targets.tolist(), hl.tolist()
    B, N = hl.shape
    if level == "token":
        return hl
    return torch.tensor([[len(words_as_ids([rows[b][n][:lens[b][n]]], SPACE, {})[0]) for n in range(N)] for b in range(B)])


@pytest.mark.gpu
def test_decode_and_greedy_results_and_empty_marker():
    """The [B, W] form of decode / decode_greedy, and decode's [-1] empty result counted as the empty hypothesis."""
    from end2end_b200 import CTCDecoder
    from end2end_b200.utils.hypotheses import empty_marker_as_empty
    x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS["c1"][:6])
    for bw in (1, 8):
        dec = CTCDecoder(beam_width=bw, labels=LABELS[:28])
        r = dec.decode(x.cuda(), ll)
        for level in ("token", "word"):
            got = dec.errors(r.decoded_targets, r.decoded_targets_lengths, tg, tl, level=level)
            h3 = r.decoded_targets[:, None]
            want = restated(h3, empty_marker_as_empty(h3, r.decoded_targets_lengths[:, None]), tg, tl,
                            SPACE if level == "word" else -1)
            assert all(torch.equal(a, b) for a, b in zip(got, want)) and got.errors.shape == (4, 1)
    dec = CTCDecoder(beam_width=4, labels=LABELS)
    hyps = torch.tensor([[-1, 0, 0], [2, 3, 4]])                 # decode's empty result, then a real hypothesis
    lens = torch.tensor([1, 3])
    refs, rl = torch.tensor([[2, 3], [2, 3]]), torch.tensor([2, 2])
    got = dec.errors(hyps, lens, refs, rl, level="token")
    assert got.errors.tolist() == [[2], [1]] and got.deletions.tolist() == [[2], [0]]
    got3 = dec.errors(hyps[:, None], lens[:, None], refs, rl, level="word")
    assert got3.errors.tolist() == [[1], [1]] and got3.deletions.tolist() == [[1], [0]]


@pytest.mark.gpu
@pytest.mark.parametrize("words", [False, True])
def test_symmetry(words):
    """Swapping hypothesis and reference keeps errors and substitutions and exchanges insertions and deletions."""
    g = torch.Generator().manual_seed(41)
    B, W = 64, 90
    a, al = random_rows(g, (B,), W, 6)
    b, bl = random_rows(g, (B,), W, 6)
    e1 = run(a[:, None].cuda(), al[:, None].cuda(), b.cuda(), bl.cuda(), words)
    e2 = run(b[:, None].cuda(), bl[:, None].cuda(), a.cuda(), al.cuda(), words)
    assert torch.equal(e1[0], e2[0]) and torch.equal(e1[1], e2[1])
    assert torch.equal(e1[2], e2[3]) and torch.equal(e1[3], e2[2])


@pytest.mark.gpu
def test_word_units_agree_with_align_word_spans():
    """A hypothesis has as many word units as CTCDecoder.align's word_spans lists for it."""
    from end2end_b200 import CTCDecoder
    x, tg, ll, tl = oracle.make_inputs(4, 120, 29, 10, 40, 9, full_length=True)
    dec = CTCDecoder(beam_width=16, labels=LABELS)
    nb = dec.decode_nbest(x.cuda(), ll, n_best=16)
    hyps, hl = nb.decoded_targets, nb.decoded_targets_lengths
    al = dec.align(x.cuda(), hyps, hl, ll)
    B, N = hl.shape
    empty = torch.zeros(B, 0, dtype=torch.int64)
    e = dec.errors(hyps, hl, empty, torch.zeros(B, dtype=torch.int64), level="word")
    assert (e.insertions == e.errors).all()
    assert e.insertions.tolist() == [[len(al.word_spans[b][n]) for n in range(N)] for b in range(B)]
    same = dec.errors(hyps[:, :1], hl[:, :1], hyps[:, 0], torch.where(hyps[:, 0, 0] == -1, 0, hl[:, 0]), level="word")
    assert (same.errors == 0).all() and same.reference_units.tolist() == [len(al.word_spans[b][0]) for b in range(B)]


@pytest.mark.gpu
@pytest.mark.parametrize("words", [False, True])
def test_bad_lengths_isolated(words):
    """Device-resident bad lengths give -1 in their pairs only (a reference's: all N of the utterance); host-resident
    ones raise; CPU input runs on the current device."""
    g = torch.Generator().manual_seed(51)
    B, N, W, Wr = 6, 9, 30, 25
    hyps, hl = random_rows(g, (B, N), W, 6)
    refs, rl = random_rows(g, (B,), Wr, 6)
    want = restated(hyps, hl, refs, rl, SPACE if words else -1)
    bhl, brl = hl.clone(), rl.clone()
    bhl[0, 3], bhl[2, 8], brl[4] = W + 1, -1, Wr + 1
    got = run(hyps.cuda(), bhl.cuda(), refs.cuda(), brl.cuda(), words)
    bad = torch.zeros(B, N, dtype=torch.bool)
    bad[0, 3] = bad[2, 8] = True
    bad[4] = True
    for a, b in zip(got[:4], want[:4]):
        assert (a[bad] == -1).all() and torch.equal(a[~bad], b[~bad])
    assert got[4][4] == -1 and torch.equal(got[4][torch.arange(B) != 4], want[4][torch.arange(B) != 4])
    with pytest.raises(ValueError):
        run(hyps.cuda(), bhl, refs.cuda(), rl.cuda(), words)
    with pytest.raises(ValueError):
        run(hyps.cuda(), hl.cuda(), refs.cuda(), brl, words)
    cpu = run(hyps, hl, refs, rl, words)
    assert all(torch.equal(a, b) for a, b in zip(cpu, want))


@pytest.mark.gpu
def test_repeatable_and_permutation_invariant():
    g = torch.Generator().manual_seed(61)
    B, N, W, Wr = 16, 12, 200, 150
    hyps, hl = random_rows(g, (B, N), W, 5)
    refs, rl = random_rows(g, (B,), Wr, 5)
    for words in (False, True):
        first = run(hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda(), words)
        for _ in range(3):
            again = run(hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda(), words)
            assert all(torch.equal(a, b) for a, b in zip(first, again))
        pb, pn = torch.randperm(B, generator=g), torch.randperm(N, generator=g)
        perm = run(hyps[pb][:, pn].cuda(), hl[pb][:, pn].cuda(), refs[pb].cuda(), rl[pb].cuda(), words)
        assert all(torch.equal(a, b[pb][:, pn]) for a, b in zip(perm[:4], first[:4]))
        assert torch.equal(perm[4], first[4][pb])


@pytest.mark.gpu
def test_cuda_graph_capture_replays():
    """errors_device on device tensors captures into a CUDA graph (it never synchronises) and replays on new contents."""
    from end2end_b200.engine import CTCBeamEngine
    eng = CTCBeamEngine(0, 1, LABELS)
    g = torch.Generator().manual_seed(71)
    B, N, W, Wr = 8, 10, 60, 50
    hyps, hl = random_rows(g, (B, N), W, 6)
    refs, rl = random_rows(g, (B,), Wr, 6)
    dh, dhl, dr, drl = hyps.cuda(), hl.cuda(), refs.cuda(), rl.cuda()
    eng.errors_device(dh, dhl, dr, drl, words=True)              # warm up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = eng.errors_device(dh, dhl, dr, drl, words=True)
    graph.replay()
    torch.cuda.synchronize()
    want = restated(hyps, hl, refs, rl, SPACE)
    assert all(torch.equal(a.cpu(), b) for a, b in zip(out, want))
    hyps2, hl2 = random_rows(g, (B, N), W, 6)
    dh.copy_(hyps2)
    dhl.copy_(hl2)
    graph.replay()
    torch.cuda.synchronize()
    want2 = restated(hyps2, hl2, refs, rl, SPACE)
    assert all(torch.equal(a.cpu(), b) for a, b in zip(out, want2))


@pytest.mark.gpu
def test_mwer_step_with_device_word_errors():
    """INTEGRATION.md's MWER step with the risk from errors_device equals, bit for bit, the same step with the risk
    from the restatement."""
    from end2end_b200 import CTCDecoder, CTCScore
    from end2end_b200.utils.hypotheses import empty_marker_as_empty
    x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS["c1"][:6])
    x = x.double()
    N = 10
    dec = CTCDecoder(beam_width=N, labels=LABELS[:28])
    hyps, hl, scores, _, _ = dec._decoder.decode_nbest_device(x.cuda(), ll.cuda(), n_best=N, from_logits=True)
    used = scores > -float("inf")

    def step(risk):
        xa = x.cuda().requires_grad_()
        s = CTCScore()(xa, hyps, hl, ll.cuda())
        p = torch.softmax(s.masked_fill(~used, float("-inf")), dim=1)
        (p * risk).sum().backward()
        return xa.grad

    risk_dev = dec._decoder.errors_device(hyps, hl, tg.cuda(), tl.cuda(), words=True)[0].double()
    risk_host = restated(hyps, empty_marker_as_empty(hyps, hl).cpu(), tg, tl, SPACE)[0].double().cuda()
    assert torch.equal(risk_dev, risk_host) and float(risk_dev.max()) > 0
    ga, gb = step(risk_dev), step(risk_host)
    assert float(ga.abs().max()) > 0 and torch.equal(ga, gb)

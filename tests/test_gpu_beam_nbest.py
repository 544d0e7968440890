"""The N best prefixes of the LM-free prefix beam search and their scores (CTCDecoder.decode_nbest,
e2e_ctc_beam_nbest_device, e2e_ctc_engine_beam_nbest_host).

The list is the first N entries of the reference's final sorted list (src/decoders/ctc_decoder.cpp:413-419), ranked by
score = log p - words * wip with equal scores in beam order.  The checker is a C restatement of the search, which
the device-free tests pin to oracle.beam_decode (N = 1) and, on beams large enough to hold every prefix, to the CTC loss of
each hypothesis (the search is exact there).  The restatement is tests/beam_nbest_restatement.c, compiled by this module
into a temporary directory.  The GPU tests compare the kernel with the restatement on log-probability
input -- hypotheses, lengths, order and tie counters bit for bit, scores within 1e-12 relative (the kernel's fp64 exp and
log are CUDA's, within one ulp, the restatement's the C library's: the same expression can differ in its last bits) --
and check the exhaustive beams against the engine's own loss.
"""
import atexit
import ctypes
import glob
import math
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN = sorted(glob.glob(os.path.join(GOLD, "beam_*.npz")))
# (V, T): beam_width 256 holds every prefix, so nothing is ever pruned
EXHAUSTIVE = ((2, 1), (2, 7), (2, 40), (2, 100), (3, 1), (3, 4), (3, 6), (4, 2), (4, 4))


_HERE = os.path.dirname(os.path.abspath(__file__))
_RESTATEMENT_SRC = os.path.join(_HERE, "beam_nbest_restatement.c")
_restatement_lib = None


def _restatement():
    """gcc the C restatement into a temporary directory (once per process; the tree is left untouched)."""
    global _restatement_lib
    if _restatement_lib is None:
        d = tempfile.mkdtemp(prefix="beam_nbest_restatement_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libbeam_nbest_restatement.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-o", so, _RESTATEMENT_SRC, "-lm"])
        L = ctypes.CDLL(so)
        dp, ip = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)
        L.ctc_oracle_beam_nbest.argtypes = [dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ip, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_double, ip, ip, dp, dp, ip]
        L.ctc_oracle_beam_nbest.restype = None
        _restatement_lib = L
    return _restatement_lib


def beam_nbest(logits, logits_lengths=None, blank_idx=0, beam_width=100, n_best=1, time_major=False, labels=None,
               after_logsoftmax=False, wip=0.0, oov_penalty=-1000.0):
    """The n_best best prefixes of the LM-free prefix beam search through the C restatement, driven as
    oracle.beam_decode drives the search (log_softmax first unless after_logsoftmax).  Returns (targets
    [B, N, max(T, 1)] i64 zero padded, lengths [B, N] i64, scores [B, N] f64, log_probs [B, N] f64, ties [B] i64); slots
    past the final beam have length 0 and -inf scores."""
    with torch.no_grad():
        if not after_logsoftmax:
            logits = torch.log_softmax(logits, -1)
        if time_major:
            logits = logits.transpose(1, 0)
    logits = logits.detach().cpu()
    B, T, V = logits.shape
    if logits_lengths is None:
        logits_lengths = torch.full((B,), T, dtype=torch.int64)
    x = np.ascontiguousarray(logits.to(torch.float64).numpy())
    il = np.ascontiguousarray(logits_lengths.cpu().to(torch.int64).numpy())
    N, Tw = int(n_best), max(T, 1)
    out = np.zeros((B, N, Tw), dtype=np.int64)
    out_len = np.zeros((B, N), dtype=np.int64)
    scores = np.zeros((B, N), dtype=np.float64)
    log_probs = np.zeros((B, N), dtype=np.float64)
    ties = np.zeros(B, dtype=np.int64)
    dptr = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))    # noqa: E731
    iptr = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))     # noqa: E731
    _restatement().ctc_oracle_beam_nbest(dptr(x), B, T, V, iptr(il), int(blank_idx), int(beam_width), N,
                                         oracle._space_id(labels), float(wip), float(oov_penalty), iptr(out),
                                         iptr(out_len), dptr(scores), dptr(log_probs), iptr(ties))
    return (torch.from_numpy(out), torch.from_numpy(out_len), torch.from_numpy(scores), torch.from_numpy(log_probs),
            torch.from_numpy(ties))


def _labels(z):
    s = str(z["labels"])
    return s.split("\x1f") if s else []


def _golden_id(p):
    return os.path.basename(p)[:-4]


def _space_labels(V, blank):
    labels = [chr(33 + i) for i in range(V)]
    labels[1 if blank == 0 else 0] = " "
    return labels


def _words(seq, space):
    """ctc_decoder.cpp:252-257: a symbol other than the space starts a word after the root or after a space."""
    n, last = 0, -1
    for c in seq:
        if c != space and (n == 0 or last == space):
            n += 1
        last = c
    return n


def _hyp_targets(targets, lengths):
    """Hypotheses [N, T] -> CTC targets [N, max(L, 1)] and their lengths; the empty prefix (-1, length 1) is L = 0."""
    rows = []
    for r, n in zip(targets.tolist(), lengths.tolist()):
        seq = r[:n]
        rows.append([] if seq == [-1] else seq)
    width = max(1, max(len(s) for s in rows))
    tg = torch.zeros(len(rows), width, dtype=torch.int64)
    for i, s in enumerate(rows):
        tg[i, :len(s)] = torch.tensor(s, dtype=torch.int64)
    return tg, torch.tensor([len(s) for s in rows], dtype=torch.int64)


def _exhaustive_input(V, T, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.log_softmax(torch.randn(2, T, V, generator=g, dtype=torch.float64) * 1.5, 2)


# ---------------------------------------------------------------------------------------------- device-free ---------

@pytest.mark.parametrize("path", GOLDEN, ids=_golden_id)
def test_restatement_n1_equals_beam_decode(path):
    z = np.load(path, allow_pickle=False)
    lp = torch.from_numpy(z["log_probs"])
    ll = torch.from_numpy(z["logits_lengths"])
    kw = dict(blank_idx=int(z["blank"]), beam_width=int(z["beam"]), labels=_labels(z), after_logsoftmax=True,
              wip=float(z["wip"]))
    t1, n1, _, ties1 = oracle.beam_decode(lp, ll, prefer="port", return_ties=True, **kw)
    t, n, sc, lpr, ties = beam_nbest(lp, ll, n_best=1, **kw)
    assert torch.equal(n[:, 0], n1) and torch.equal(ties, ties1)
    w = t1.size(1)
    assert torch.equal(t[:, 0, :w], t1) and not bool(t[:, 0, w:].any())
    space = oracle._space_id(_labels(z))
    words = torch.tensor([_words(r[:k], space) if r[:k] != [-1] else 0 for r, k in zip(t[:, 0].tolist(), n[:, 0].tolist())],
                         dtype=torch.float64)
    assert torch.equal(sc[:, 0], lpr[:, 0] - float(z["wip"]) * words)


@pytest.mark.parametrize("V,T", EXHAUSTIVE)
def test_restatement_exhaustive_beam_is_exact(V, T):
    """Nothing is pruned when the beam holds every prefix: each hypothesis's log_probs is minus its CTC loss and the
    list carries the whole probability mass."""
    lp = _exhaustive_input(V, T, 100 * V + T)
    t, n, sc, lpr, ties = beam_nbest(lp, None, beam_width=256, n_best=256, after_logsoftmax=True)
    for b in range(lp.size(0)):
        have = n[b] > 0
        k = int(have.sum())
        assert bool(have[:k].all()) and not bool(have[k:].any())
        assert bool(torch.isinf(lpr[b, k:]).all()) and bool(torch.isinf(sc[b, k:]).all())
        tg, tl = _hyp_targets(t[b, :k], n[b, :k])
        loss, _ = oracle.PortEngine(0).compute(lp[b:b + 1].expand(k, -1, -1).contiguous(), tg,
                                               torch.full((k,), T, dtype=torch.int64), tl)
        assert torch.allclose(lpr[b, :k], -loss, rtol=1e-10, atol=0), (lpr[b, :k] + loss).abs().max()
        assert abs(float(torch.logsumexp(lpr[b, :k], 0))) <= 1e-10
        assert torch.equal(sc[b], lpr[b])                     # wip = 0
        assert bool((sc[b, :k - 1] >= sc[b, 1:k]).all())


def test_nbest_workspace_query_and_errors(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = 8, 50, 29, 0
    d.blank_idx, d.dtype = 0, _lib.E2E_F32
    d.targets_itype = d.lengths_itype = _lib.E2E_I64
    d.logits_stride_b, d.logits_stride_t = 50 * 29, 29
    for beam in (1, 10, 256):
        for n_best in (1, beam // 2 + 1, beam):
            n = L.e2e_ctc_beam_nbest_workspace_bytes(ctypes.byref(d), beam, n_best)
            assert n > 0 and n % 256 == 0
            assert n == L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), beam)
        for n_best in (0, beam + 1, 257):
            assert L.e2e_ctc_beam_nbest_workspace_bytes(ctypes.byref(d), beam, n_best) == 0
            assert "n_best %d" % n_best in L.e2e_last_error_string().decode()
            rc = L.e2e_ctc_beam_nbest_device(ctypes.byref(d), beam, n_best, -1, 0.0, None, None, None, None, None, None,
                                             None, None, 0, None)
            assert rc == 1                                          # E2E_ERR_INVALID_ARGUMENT
            assert "n_best %d outside [1, beam_width = %d]" % (n_best, beam) in L.e2e_last_error_string().decode()
            rc = L.e2e_ctc_engine_beam_nbest_host(None, ctypes.byref(d), beam, n_best, -1, 0.0, None, None, None, None,
                                                  None, None, None)
            assert rc == 1
    assert L.e2e_ctc_beam_nbest_workspace_bytes(ctypes.byref(d), 257, 1) == 0     # beam limits are unchanged
    assert "limits" in L.e2e_last_error_string().decode()


def test_decode_nbest_argument_errors(lib_built):
    from pytorch_end2end import CTCDecoder
    x = torch.zeros(1, 2, 3)
    with pytest.raises(NotImplementedError):
        CTCDecoder(beam_width=10, lm_path="/no/such/model.arpa").decode_nbest(x, n_best=2)
    for n_best in (0, 11, 257):
        with pytest.raises(ValueError, match="n_best"):
            CTCDecoder(beam_width=10).decode_nbest(x, n_best=n_best)


# ---------------------------------------------------------------------------------------------- GPU -----------------

def _kernel(lp, ll, blank, beam, n_best, labels=None, wip=0.0, from_logits=False):
    from end2end_b200.engine import CTCBeamEngine
    eng = CTCBeamEngine(blank, beam, labels, wip)
    return [t.cpu() for t in eng.decode_nbest_device(lp, ll, n_best, from_logits)]


def _assert_equal_restatement(x, ll, blank, beam, n_best, labels=None, wip=0.0):
    """Kernel == restatement on log-probability input: hypotheses, their order, lengths and tie counters exactly; scores
    and log_probs to the last few ulps (see the module docstring)."""
    t, n, sc, lpr, ties = _kernel(x.cuda(), None if ll is None else ll.cuda(), blank, beam, n_best, labels, wip)
    ot, on, osc, olp, oties = beam_nbest(x, ll, blank_idx=blank, beam_width=beam, n_best=n_best, labels=labels,
                                         after_logsoftmax=True, wip=wip)
    ctx = (tuple(x.shape), x.dtype, blank, beam, n_best, wip)
    assert torch.equal(n, on), ctx
    assert torch.equal(t, ot), ctx
    assert torch.equal(ties, oties), (ctx, ties, oties)
    _assert_scores_close(sc, osc, 1e-12, ctx)
    _assert_scores_close(lpr, olp, 1e-12, ctx)
    return t, n, sc, lpr, ties


def _assert_scores_close(got, want, rtol, ctx=None):
    fin = torch.isfinite(want)
    assert torch.equal(fin, torch.isfinite(got)) and torch.equal(got[~fin], want[~fin]), ctx
    assert torch.allclose(got[fin], want[fin], rtol=rtol, atol=0), (ctx, (got[fin] - want[fin]).abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLDEN, ids=_golden_id)
@pytest.mark.parametrize("where", ["host", "cuda"])
def test_hypothesis0_equals_decode(path, where):
    from pytorch_end2end import CTCDecoder
    z = np.load(path, allow_pickle=False)
    lp = torch.from_numpy(z["log_probs"])
    ll = torch.from_numpy(z["logits_lengths"])
    labels = _labels(z)
    beam = int(z["beam"])
    x = lp.cuda() if where == "cuda" else lp
    dec = CTCDecoder(beam_width=beam, after_logsoftmax=True, blank_idx=int(z["blank"]), labels=labels or None,
                     wip=float(z["wip"]))
    res = dec.decode(x, ll)
    ties = dec._decoder.last_ties.clone()
    for n_best in sorted({1, min(3, beam), beam}):
        nb = dec.decode_nbest(x, ll, n_best=n_best)
        assert not nb.decoded_targets.is_cuda and nb.scores.dtype == torch.float64 and nb.log_probs.dtype == torch.float64
        assert nb.decoded_targets.shape[:2] == (lp.size(0), n_best) and len(nb.decoded_sentences) == lp.size(0)
        assert torch.equal(nb.decoded_targets_lengths[:, 0], res.decoded_targets_lengths)
        w = res.decoded_targets.size(1)
        assert torch.equal(nb.decoded_targets[:, 0, :w], res.decoded_targets)
        assert not bool(nb.decoded_targets[:, 0, w:].any())
        assert [s[0] for s in nb.decoded_sentences] == res.decoded_sentences
        if n_best == 1:
            assert nb.decoded_targets.shape == res.decoded_targets.unsqueeze(1).shape
            assert torch.equal(dec._decoder.last_ties, ties)
        else:
            assert bool((dec._decoder.last_ties >= ties).all())
    free = torch.from_numpy(z["ties"]) == 0
    want_t, want_l = torch.from_numpy(z["targets"]), torch.from_numpy(z["targets_lengths"])
    nb = dec.decode_nbest(x, ll, n_best=1)
    for i in range(lp.size(0)):
        if free[i]:
            k = int(want_l[i])
            assert int(nb.decoded_targets_lengths[i, 0]) == k
            assert nb.decoded_targets[i, 0, :k].tolist() == want_t[i, :k].tolist()


@pytest.mark.gpu
def test_kernel_equals_restatement_sweep():
    """Alphabets (1024: the large-alphabet prefilter; 200 at beam 256: no key cache), beams, N in {1, 2, 5, beam}, blank
    0 and V-1, words with a word insertion penalty."""
    g = torch.Generator().manual_seed(21)
    n = 0
    for V in (2, 3, 5, 29, 200, 1024):
        for beam in (2, 5, 100, 256):
            T = 12 if V * beam > 100000 else 30
            blank = 0 if (V + beam) % 2 else V - 1
            lp = torch.log_softmax(torch.randn(3, T, V, generator=g, dtype=torch.float64) * 2.0, 2)
            ll = torch.tensor([T, max(1, T // 2), 1])
            labels, wip = (None, 0.0) if V < 5 else (_space_labels(V, blank), 0.6)
            for n_best in sorted({1, 2, 5, beam}):
                if n_best <= beam:
                    _assert_equal_restatement(lp, ll, blank, beam, n_best, labels, wip)
                    n += 1
    assert n == 78


@pytest.mark.gpu
def test_kernel_equals_restatement_ties_variants_dtypes():
    """Equal final scores (uniform rows, impossible symbols), the 256-thread variant (B > 148) and every input dtype."""
    V, T = 5, 4
    uniform = torch.full((2, T, V), -math.log(V), dtype=torch.float64)
    for n_best in (1, 2, 5, 10):
        _, _, _, _, ties = _assert_equal_restatement(uniform, None, 0, 10, n_best)
        assert bool((ties > 0).all())
    g = torch.Generator().manual_seed(22)
    holes = torch.log_softmax(torch.randn(3, 6, 4, generator=g, dtype=torch.float64), 2)
    holes[:, :, 2] = -math.inf                                 # a symbol that never occurs: -inf ties in the final beam
    for n_best in (1, 3, 50):
        _assert_equal_restatement(holes, None, 0, 50, n_best)
    big = torch.log_softmax(torch.randn(150, 20, 29, generator=g, dtype=torch.float64) * 2.0, 2)
    big_ll = torch.randint(10, 21, (150,), generator=g)
    for n_best in (1, 7, 40):
        _assert_equal_restatement(big, big_ll, 28, 40, n_best, _space_labels(29, 28), 0.4)
    x = torch.log_softmax(torch.randn(4, 25, 29, generator=g) * 2.0, 2)
    ll = torch.tensor([25, 20, 3, 1])
    for dtype in (torch.float32, torch.float64, torch.bfloat16, torch.float16):
        for n_best in (1, 5, 30):
            _assert_equal_restatement(x.to(dtype), ll, 0, 30, n_best, _space_labels(29, 0), 0.5)


def _assert_raw_logits(x, ll, blank, beam, n_best, time_major=False, where="cuda", labels=None, wip=0.0):
    """Raw logits: the log-softmax is fused, so scores agree within the input precision's tolerance; hypotheses and
    their order are those of the restatement."""
    from pytorch_end2end import CTCDecoder
    dec = CTCDecoder(beam_width=beam, blank_idx=blank, time_major=time_major, labels=labels, wip=wip)
    res = dec.decode_nbest(x.cuda() if where == "cuda" else x, ll, n_best=n_best)
    ot, on, osc, olp, _ = beam_nbest(x, ll, blank_idx=blank, beam_width=beam, n_best=n_best, time_major=time_major,
                                            labels=labels, wip=wip)
    tol = 1e-12 if x.dtype == torch.float64 else 1e-6
    assert torch.equal(res.decoded_targets_lengths, on)
    w = res.decoded_targets.size(2)
    assert torch.equal(res.decoded_targets, ot[:, :, :w]) and not bool(ot[:, :, w:].any())
    _assert_scores_close(res.scores, osc, tol)
    _assert_scores_close(res.log_probs, olp, tol)


@pytest.mark.gpu
def test_raw_logits_layouts_and_host_input():
    g = torch.Generator().manual_seed(23)
    x = torch.randn(5, 60, 29, generator=g) * 2.0
    ll = torch.randint(40, 61, (5,), generator=g)
    labels = _space_labels(29, 0)
    _assert_raw_logits(x, ll, 0, 50, 10, labels=labels, wip=0.5)
    _assert_raw_logits(x, ll.int(), 0, 50, 50)
    _assert_raw_logits(x, None, 0, 20, 5)
    _assert_raw_logits(x, ll, 0, 50, 10, where="host", labels=labels, wip=0.5)
    _assert_raw_logits(x.double(), ll, 3, 40, 40)
    _assert_raw_logits(x.double(), ll.int(), 3, 40, 8, where="host")
    xt = x.transpose(0, 1)                                      # [T, B, V] view
    _assert_raw_logits(xt, ll, 0, 50, 10, time_major=True)
    _assert_raw_logits(xt.contiguous(), ll, 0, 50, 10, time_major=True, where="host")


@pytest.mark.gpu
@pytest.mark.parametrize("V,T", EXHAUSTIVE)
def test_exhaustive_beam_matches_the_engine_loss(V, T):
    """Without pruning the search is exact: log_probs is minus the CTC loss of each hypothesis, computed by the library's
    own loss kernels, and the list carries probability 1.  Independent of the restatement."""
    from end2end_b200 import CTCLossEngine
    lp = _exhaustive_input(V, T, 100 * V + T + 1).cuda()
    blank = V - 1
    t, n, sc, lpr, _ = _kernel(lp, None, blank, 256, 256)
    for b in range(lp.size(0)):
        k = int((n[b] > 0).sum())
        assert bool((n[b, :k] > 0).all()) and not bool(n[b, k:].any()) and not bool(t[b, k:].any())
        assert bool(torch.isinf(lpr[b, k:]).all()) and bool((lpr[b, k:] < 0).all())
        tg, tl = _hyp_targets(t[b, :k], n[b, :k])
        loss, _ = CTCLossEngine(blank).compute(lp[b:b + 1].expand(k, -1, -1).contiguous(), tg.cuda(),
                                              torch.full((k,), T, dtype=torch.int64).cuda(), tl.cuda())
        loss = loss.cpu()
        assert torch.allclose(lpr[b, :k], -loss, rtol=1e-10, atol=0), (lpr[b, :k] + loss).abs().max()
        assert abs(float(torch.logsumexp(lpr[b, :k], 0))) <= 1e-10


@pytest.mark.gpu
def test_list_invariants_c2():
    """BASELINE config 2 (B=64, T=400, V=29) at beam 100, N = 100."""
    from pytorch_end2end import CTCDecoder
    x, _, ll, _ = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    labels = ["_", " "] + [chr(ord("a") + i) for i in range(26)] + ["'"]
    wip = 0.5
    dec = CTCDecoder(beam_width=100, labels=labels, wip=wip)
    res = dec.decode_nbest(x.cuda(), ll, n_best=100)
    t, n, sc, lpr = res.decoded_targets, res.decoded_targets_lengths, res.scores, res.log_probs
    assert t.shape[:2] == (64, 100)
    assert bool((sc[:, :-1] >= sc[:, 1:]).all())
    for b in range(64):
        k = int((n[b] > 0).sum())
        assert not bool(n[b, k:].any()) and not bool(t[b, k:].any())
        assert bool(torch.isinf(sc[b, k:]).all()) and bool(torch.isinf(lpr[b, k:]).all())
        hyps = [tuple(t[b, i, :int(n[b, i])].tolist()) for i in range(k)]
        assert len(set(hyps)) == k
        words = torch.tensor([_words(h, 1) for h in hyps], dtype=torch.float64)
        assert torch.equal(sc[b, :k], lpr[b, :k] - wip * words)
        assert res.decoded_sentences[b][:k] == ["".join(labels[c] for c in h) for h in hyps]
    best = dec.decode(x.cuda(), ll)
    assert torch.equal(t[:, 0, :best.decoded_targets.size(1)], best.decoded_targets)


@pytest.mark.gpu
def test_raw_c_abi_n1_writes_what_decode_writes():
    """e2e_ctc_beam_nbest_device with N = 1 writes exactly the bytes e2e_ctc_beam_decode_device writes (padding included);
    with N > the final beam, the empty slots are cleared whatever the buffers held."""
    from end2end_b200 import _lib
    from end2end_b200.engine import CTCBeamEngine
    L = _lib.load()
    g = torch.Generator().manual_seed(24)
    B, T, V, beam = 6, 30, 12, 16
    lp = torch.log_softmax(torch.randn(B, T, V, generator=g) * 2.0, 2).cuda()
    ll = torch.tensor([30, 29, 10, 2, 1, 0]).cuda()
    labels = [chr(65 + i) for i in range(V - 1)] + [" "]
    eng = CTCBeamEngine(0, beam, labels, 0.3)
    d = eng._beam_desc(lp, ll, False)
    ws = torch.empty(L.e2e_ctc_beam_nbest_workspace_bytes(ctypes.byref(d), beam, 1), dtype=torch.uint8, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())                # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def garbage(*shape, dtype=torch.int64):
        return torch.full(shape, 0x7A7A, dtype=dtype, device="cuda")

    dec, dl, ties = garbage(B, T), garbage(B), garbage(B)
    _lib.check(L.e2e_ctc_beam_decode_device(ctypes.byref(d), beam, eng.space_idx, eng.wip, p(lp), p(ll), p(dec), p(dl),
                                            p(ties), p(ws), ws.numel(), stream))
    for with_lp in (True, False):
        dec1, dl1, ties1 = garbage(B, 1, T), garbage(B, 1), garbage(B)
        sc1, lp1 = garbage(B, 1, dtype=torch.float64), garbage(B, 1, dtype=torch.float64)
        _lib.check(L.e2e_ctc_beam_nbest_device(ctypes.byref(d), beam, 1, eng.space_idx, eng.wip, p(lp), p(ll), p(dec1),
                                               p(dl1), p(sc1), p(lp1) if with_lp else None, p(ties1), p(ws), ws.numel(),
                                               stream))
        torch.cuda.synchronize()
        assert torch.equal(dec1[:, 0], dec) and torch.equal(dl1[:, 0], dl) and torch.equal(ties1, ties)
        assert bool((sc1 <= 0).all())
        assert with_lp == bool((lp1 <= 0).all())                # log_probs may be NULL: the buffer is left alone
        assert with_lp != bool((lp1 == 0x7A7A).all())
    # N = beam: utterances of 0-2 frames hold fewer prefixes than that
    N = beam
    decN, dlN, tiesN = garbage(B, N, T), garbage(B, N), garbage(B)
    scN, lpN = garbage(B, N, dtype=torch.float64), garbage(B, N, dtype=torch.float64)
    _lib.check(L.e2e_ctc_beam_nbest_device(ctypes.byref(d), beam, N, eng.space_idx, eng.wip, p(lp), p(ll), p(decN), p(dlN),
                                           p(scN), p(lpN), p(tiesN), p(ws), ws.numel(), stream))
    torch.cuda.synchronize()
    decN, dlN, scN, lpN = decN.cpu(), dlN.cpu(), scN.cpu(), lpN.cpu()
    assert int((dlN[5] > 0).sum()) == 1 and dlN[5, 0] == 1 and decN[5, 0, 0] == -1     # T = 0: the empty prefix only
    absent = dlN == 0
    assert bool(absent[3:].any())
    assert not bool(decN[absent].any())
    assert bool(torch.isinf(scN[absent]).all()) and bool(torch.isinf(lpN[absent]).all())
    assert bool((scN[absent] < 0).all()) and bool((lpN[absent] < 0).all())
    pad = torch.arange(T)[None, None, :] >= dlN[:, :, None]
    assert not bool(decN[pad].any())
    ot, on, osc, olp, oties = beam_nbest(lp.cpu(), ll.cpu(), beam_width=beam, n_best=N, labels=labels,
                                                after_logsoftmax=True, wip=0.3)
    assert torch.equal(decN, ot) and torch.equal(dlN, on) and torch.equal(tiesN.cpu(), oties)
    _assert_scores_close(scN, osc, 1e-12)
    _assert_scores_close(lpN, olp, 1e-12)


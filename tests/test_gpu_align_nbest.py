"""Viterbi alignment of N hypotheses per utterance with token timestamps and the best path's score
(CTCDecoder.align, CTCBeamEngine.align_device, e2e_ctc_align_nbest_device).

Lattice r = b * N + n aligns hypothesis n of utterance b against utterance b's frames.  The checker is
tests/align_cells_restatement.c, the oracle's Viterbi alignment restated to also return the path's cell at every
frame and the final cell's value; this module compiles it into a temporary directory and pins its labels to
oracle.get_alignment_3d on every alignment golden file.  On log-probability input the kernel adds the same fp64-widened
values in the same order as the restatement, so alignments, token spans and path scores are compared bit for bit.
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
import torch.nn.functional as F

import oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALIGN_GOLDEN = sorted(p for p in glob.glob(os.path.join(GOLD, "align_*.npz"))
                      if "asg" not in p and "loss_module" not in p)
MAX_TARGETS = 1023
# ctc_viterbi.cu: 1 / 2 / 4 cells per thread by lattice width; these Lmax sit at and next to each boundary
CPT_BOUNDARIES = (255, 256, 511, 512, 1023)

_HERE = os.path.dirname(os.path.abspath(__file__))
_RESTATEMENT_SRC = os.path.join(_HERE, "align_cells_restatement.c")
_restatement_lib = None


def _restatement():
    """gcc the C restatement into a temporary directory (once per process; the tree is left untouched)."""
    global _restatement_lib
    if _restatement_lib is None:
        d = tempfile.mkdtemp(prefix="align_cells_restatement_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libalign_cells_restatement.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-o", so, _RESTATEMENT_SRC, "-lm"])
        L = ctypes.CDLL(so)
        dp, ip, i = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.c_int
        L.ctc_restatement_align_cells.argtypes = [dp, i, i, i, i, ip, ip, i, ip, ip, i, ip, ip, dp]
        L.ctc_restatement_align_cells.restype = None
        _restatement_lib = L
    return _restatement_lib


def align_cells(lp, hyps, hl, ll, blank):
    """The restatement on lp [B, T, V] (widened to fp64), hyps [B, N, Lmax], hl [B, N], ll [B] (None: T).  Returns
    (aligned [B, N, T], cells [B, N, T] (-1 past the frames), value [B, N] f64, starts [B, N, Lmax], ends [B, N, Lmax]),
    the spans rebuilt from the cells exactly as the aligner defines them."""
    lp = np.ascontiguousarray(lp.detach().cpu().to(torch.float64).numpy())
    B, T, V = lp.shape
    N, Lmax = hyps.size(1), hyps.size(2)
    R = B * N
    tg = np.ascontiguousarray(hyps.cpu().to(torch.int64).reshape(R, Lmax).numpy()) if Lmax else np.zeros((R, 1), np.int64)
    tl = np.ascontiguousarray(hl.cpu().to(torch.int64).reshape(R).numpy())
    il = np.full(B, T, np.int64) if ll is None else np.ascontiguousarray(ll.cpu().to(torch.int64).numpy())
    utt = np.repeat(np.arange(B, dtype=np.int64), N)
    out = np.zeros((R, T), np.int64)
    cells = np.zeros((R, T), np.int64)
    value = np.zeros(R, np.float64)
    dptr = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))    # noqa: E731
    iptr = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))     # noqa: E731
    _restatement().ctc_restatement_align_cells(dptr(lp), B, T, V, R, iptr(utt), iptr(tg), max(Lmax, 1), iptr(il), iptr(tl),
                                               int(blank), iptr(out), iptr(cells), dptr(value))
    starts = np.full((R, Lmax), -1, np.int64)
    ends = np.full((R, Lmax), -1, np.int64)
    for r in range(R):
        if not value[r] > -math.inf:
            continue
        c = cells[r]
        for k in range(int(tl[r])):
            f = np.nonzero(c == 2 * k + 1)[0]
            starts[r, k], ends[r, k] = f[0], f[-1] + 1
    sh = lambda a: torch.from_numpy(a).reshape(B, N, *a.shape[1:])      # noqa: E731
    return sh(out), sh(cells), sh(value), sh(starts), sh(ends)


def random_hyps(g, B, N, Lmax, V, blank):
    """Mixed lengths inside every launch: 0, 1, Lmax and random; runs of repeated labels; blank-valued labels; lengths
    past what the frames allow (infeasible)."""
    hl = torch.randint(0, Lmax + 1, (B, N), generator=g)
    fixed = torch.tensor([0, 1, Lmax, max(Lmax - 1, 0)])
    hl[:, :min(N, 4)] = fixed[:min(N, 4)].clamp(max=Lmax)
    hyps = torch.randint(0, V, (B, N, max(Lmax, 1)), generator=g)[:, :, :Lmax].clone()
    if Lmax > 1:
        rep = torch.rand(B, N, Lmax, generator=g) < 0.3
        rep[:, :, 0] = False
        for k in range(1, Lmax):
            hyps[:, :, k] = torch.where(rep[:, :, k], hyps[:, :, k - 1], hyps[:, :, k])
    if Lmax > 0:
        hyps[torch.rand(B, N, Lmax, generator=g) < 0.05] = blank
    return hyps, hl


def align(lp, hyps, hl, ll=None, blank=0, from_logits=False):
    from end2end_b200.engine import CTCBeamEngine
    return CTCBeamEngine(blank, 1).align_device(lp, hyps, hl, ll, from_logits=from_logits)


def assert_exact(lp, hyps, hl, ll, blank, ctx=None):
    """Kernel == restatement bit for bit on log-probability input; returns the kernel's outputs (CPU)."""
    got = [t.cpu() for t in align(lp, hyps, hl, ll, blank)]
    want_al, _, want_v, want_s, want_e = align_cells(lp, hyps, hl, ll, blank)
    assert torch.equal(got[0], want_al), ctx
    assert torch.equal(got[1], want_s), ctx
    assert torch.equal(got[2], want_e), ctx
    v = got[3]
    assert torch.equal(torch.isnan(v), torch.isnan(want_v)), ctx
    ok = ~torch.isnan(v)
    assert torch.equal(v[ok], want_v[ok]), (ctx, (v[ok] - want_v[ok]).abs().max())
    return got


def assert_span_invariants(aligned, starts, ends, hyps, hl, scores, blank):
    """Spans are disjoint and increasing, every frame inside span k holds token k, every frame outside the spans is blank;
    a hypothesis without a finite path score has no spans."""
    B, N, T = aligned.shape
    for b in range(B):
        for n in range(N):
            L = int(hl[b, n])
            s, e = starts[b, n].tolist(), ends[b, n].tolist()
            assert all(x == -1 for x in s[L:]) and all(x == -1 for x in e[L:])
            if not float(scores[b, n]) > -math.inf:
                assert all(x == -1 for x in s) and all(x == -1 for x in e), (b, n)
                continue
            row = aligned[b, n].tolist()
            covered = [False] * T
            prev_end = 0
            for k in range(L):
                assert prev_end <= s[k] < e[k], (b, n, k, s[k], e[k])
                prev_end = e[k]
                for f in range(s[k], e[k]):
                    assert row[f] == int(hyps[b, n, k]), (b, n, k, f)
                    covered[f] = True
            for f in range(T):                    # (the empty hypothesis keeps the reference's row of zeros)
                if not covered[f] and row[f] != -100 and L > 0:
                    assert row[f] == blank, (b, n, f)


def _log_probs(name, dtype):
    B, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS[name]
    x, _, ll, _ = oracle.make_inputs(B, T, V, Lmin, Lmax, seed, torch.float32, full)
    return F.log_softmax(x.to(torch.float64), -1).to(dtype), ll, Lmax


# ---------------------------------------------------------------------------------------------- device-free ---------

@pytest.mark.parametrize("path", ALIGN_GOLDEN, ids=lambda p: os.path.basename(p)[:-4])
def test_restatement_labels_equal_oracle(path):
    z = np.load(path, allow_pickle=False)
    lp, tg = torch.from_numpy(z["log_probs"]), torch.from_numpy(z["targets"])
    ll, tl = torch.from_numpy(z["logits_lengths"]), torch.from_numpy(z["targets_lengths"])
    want = oracle.get_alignment_3d(lp, tg, ll, tl, is_ctc=True)
    assert torch.equal(want, torch.from_numpy(z["aligned"]))
    al, cells, value, _, _ = align_cells(lp, tg[:, None], tl[:, None], ll, 0)
    assert torch.equal(al[:, 0], want)
    for b in range(lp.size(0)):                  # the cells are the labels' cells, the value the path's sum
        T, L = int(ll[b]), int(tl[b])
        if T < 2 or L < 1 or not float(value[b, 0]) > -math.inf:
            continue
        c = cells[b, 0, :T]
        ext = torch.where(c % 2 == 1, tg[b].index_select(0, (c // 2).clamp(max=max(L - 1, 0))), torch.zeros_like(c))
        assert torch.equal(ext, want[b, :T])
        s = sum(float(lp[b, t, int(want[b, t])]) for t in range(T))
        assert abs(s - float(value[b, 0])) <= 1e-9 * abs(s)


def _desc(B, T, V, Lmax, blank=0, dtype=None, from_logits=0, itype=1):
    from end2end_b200 import _lib
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
    d.blank_idx, d.dtype = blank, _lib.E2E_F64 if dtype is None else dtype
    d.targets_itype = d.lengths_itype = itype
    d.from_logits = from_logits
    d.logits_stride_b, d.logits_stride_t = T * V, V
    d.targets_stride_b = Lmax
    return d


def _threads(Lmax):
    S = 2 * Lmax + 1
    cpt = 1 if S <= 512 else (2 if S <= 1024 else 4)
    thr = ((S + cpt - 1) // cpt + 31) & ~31
    return max(thr, 32)


def test_align_workspace_query(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    lim = _lib.limits()
    for B, T, V, Lmax in ((4, 50, 29, 0), (64, 400, 29, 200), (128, 250, 1024, 80), (3, 2100, 8, MAX_TARGETS)):
        for n_hyp in (1, 3, 100):
            for fl, dt in ((0, _lib.E2E_F32), (1, _lib.E2E_F32), (1, _lib.E2E_BF16), (1, _lib.E2E_F64)):
                d = _desc(B, T, V, Lmax, dtype=dt, from_logits=fl)
                stats = B * T * (16 if dt == _lib.E2E_F64 else 8) if fl else 0
                want = 256 + stats + B * n_hyp * T * _threads(Lmax)
                assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(d), n_hyp) == (want + 255) // 256 * 256
        # N = 1 on log-probs is the Viterbi alignment's own workspace
        d = _desc(B, T, V, Lmax)
        assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(d), 1) == L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), 1)
    assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(_desc(2, 50, 29, MAX_TARGETS + 1)), 1) == 0
    assert "target length 1024" in L.e2e_last_error_string().decode()
    assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(_desc(2, 50, lim.max_alphabet, 10, from_logits=1)), 1) > 0
    assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(_desc(2, 50, lim.max_alphabet + 1, 10, from_logits=1)), 1) == 0
    assert "alphabet %d" % (lim.max_alphabet + 1) in L.e2e_last_error_string().decode()
    for n_hyp in (0, -1):
        assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(_desc(4, 50, 29, 10)), n_hyp) == 0
        assert "n_hyp %d" % n_hyp in L.e2e_last_error_string().decode()
    assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(_desc(1 << 16, 50, 29, 10)), 1 << 15) == 0   # 2^31 CTAs
    assert "grid" in L.e2e_last_error_string().decode()
    assert L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(_desc(1, 0x7fffffff, 29, 1000)), 0x7fffffff) == 0
    assert "overflows" in L.e2e_last_error_string().decode()


def test_align_device_argument_errors(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    d = _desc(2, 10, 5, 3)
    fake = ctypes.c_void_p(256)              # never dereferenced: every case fails before a launch
    # logits, hyps, logits_lengths, hyp_lengths, aligned, token_starts, token_ends, path_scores, ws, ws_bytes, stream
    ok = [fake, fake, None, fake, fake, fake, fake, fake, None, 1 << 20, None]

    def call(desc, n_hyp, args):
        return L.e2e_ctc_align_nbest_device(ctypes.byref(desc) if desc is not None else None, n_hyp, *args)

    assert call(None, 1, ok) == 1
    assert call(d, 0, ok) == 1 and "n_hyp 0" in L.e2e_last_error_string().decode()
    for i in (0, 1, 3, 4, 5, 6, 7):
        args = list(ok)
        args[i] = None
        assert call(d, 2, args) == 1 and "null pointer" in L.e2e_last_error_string().decode(), i
    # no labels: hyps and the spans may be NULL; the call passes the pointer checks and stops at the (null) workspace
    assert call(_desc(2, 10, 5, 0), 2, [fake, None, None, fake, fake, None, None, fake, None, 1 << 20, None]) == 3
    assert "workspace" in L.e2e_last_error_string().decode()
    bad = _desc(2, 10, 5, 3)
    bad.targets_stride_b = 2
    assert call(bad, 2, ok) == 1 and "row stride" in L.e2e_last_error_string().decode()
    bad = _desc(2, 10, 5, 3)
    bad.blank_idx = 5
    assert call(bad, 2, ok) == 1
    need = L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(d), 2)
    for ws, n in ((None, need), (ctypes.c_void_p(512), need - 1), (ctypes.c_void_p(384), need)):   # null, short, misaligned
        args = list(ok)
        args[8], args[9] = ws, n
        assert call(d, 2, args) == 3, (ws, n)


def test_python_errors_before_device_work(monkeypatch, lib_built):
    """Every argument error is raised on the host before anything touches a device (so this runs without one)."""
    from end2end_b200 import engine
    monkeypatch.setattr(engine, "_CUDA_OK", True)
    x = torch.randn(2, 10, 5)
    hyps, hl = torch.ones(2, 3, 4, dtype=torch.int64), torch.full((2, 3), 2)
    eng = engine.CTCBeamEngine(0, 1)
    cases = [(ValueError, (x, hyps, torch.full((2, 3), 5))),                  # length > Lmax
             (ValueError, (x, hyps, torch.full((2, 3), -1))),
             (ValueError, (x, torch.full((2, 3, 4), 5), hl)),                  # label == V
             (ValueError, (x, torch.full((2, 3, 4), -2), hl)),
             (ValueError, (x, hyps, hl, torch.tensor([10, 11]))),              # frames > T
             (ValueError, (x, hyps, hl, torch.tensor([0, 10]))),
             (ValueError, (x, hyps, torch.full((2, 4), 2))),                   # shapes
             (ValueError, (x, hyps[:1], hl)),
             (ValueError, (x, hyps[:, :0], hl[:, :0])),
             (ValueError, (x[0], hyps, hl)),
             (ValueError, (x, hyps, hl, torch.tensor([10]))),
             (TypeError, (x.to(torch.int32), hyps, hl)),
             (NotImplementedError, (x, torch.ones(2, 3, MAX_TARGETS + 1, dtype=torch.int64), hl))]
    for exc, args in cases:
        with pytest.raises(exc):
            eng.align_device(*args)
    with pytest.raises(ValueError):
        engine.CTCBeamEngine(7, 1).align_device(x, hyps, hl)                  # blank outside the alphabet


def test_word_spans_grouping():
    from end2end_b200.decoders.ctc_decoder import word_spans
    labels = ["_", " ", "a", "b", "c"]
    sp, a, b, c = 1, 2, 3, 4
    # tokens, starts, ends -> words
    assert word_spans([a, b, sp, c], [0, 2, 5, 7], [1, 4, 6, 9], labels) == [("ab", 0, 4), ("c", 7, 9)]
    assert word_spans([sp, a, b], [0, 3, 5], [2, 4, 8], labels) == [("ab", 3, 8)]                  # leading space
    assert word_spans([a, sp], [1, 4], [3, 6], labels) == [("a", 1, 3)]                           # trailing space
    assert word_spans([a, sp, sp, b, c], [0, 2, 4, 6, 8], [1, 3, 5, 7, 9], labels) == [("a", 0, 1), ("bc", 6, 9)]
    assert word_spans([c, a, b, b], [0, 3, 5, 8], [2, 4, 7, 10], labels) == [("cabb", 0, 10)]    # no space at all
    assert word_spans([sp, sp], [0, 1], [1, 2], labels) == []
    assert word_spans([], [], [], labels) == []
    assert word_spans([a, sp, b], [-1, -1, -1], [-1, -1, -1], labels) == [("a", -1, -1), ("b", -1, -1)]   # no finite path


# ---------------------------------------------------------------------------------------------- GPU ----------------

@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16, torch.float16],
                         ids=["f32", "f64", "bf16", "f16"])
@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_oracle_exact_configs(name, dtype):
    """Log-prob input, N = 3: every (utterance, hypothesis) pair bit for bit.  c2 at N = 3 is 192 lattices, past the
    148 that get 200 KB of shared memory, so its backpointers go to the workspace."""
    lp, ll, Lmax = _log_probs(name, dtype)
    g = torch.Generator().manual_seed(11)
    B, V = lp.size(0), lp.size(2)
    hyps, hl = random_hyps(g, B, 3, Lmax, V, 0)
    got = assert_exact(lp.cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), 0, (name, dtype))
    assert_span_invariants(got[0], got[1], got[2], hyps, hl, got[3], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("name,N", [("c1", 1), ("c1", 100), ("c4", 1), ("c4", 100), ("c2", 1)])
def test_oracle_exact_n(name, N):
    lp, ll, Lmax = _log_probs(name, torch.float32)
    g = torch.Generator().manual_seed(N)
    hyps, hl = random_hyps(g, lp.size(0), N, Lmax, lp.size(2), 0)
    assert_exact(lp.cuda(), hyps, hl, ll, 0, (name, N))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [4, 5])
def test_backpointers_shared_and_global(N):
    """37 utterances of 400 frames, Lmax 200 (166 KB of backpointers): 148 lattices keep them in shared memory, 185 in
    the workspace.  Both are exact."""
    g = torch.Generator().manual_seed(5)
    lp = F.log_softmax(torch.randn(37, 400, 29, generator=g, dtype=torch.float64) * 2, -1).float()
    ll = torch.randint(300, 401, (37,), generator=g)
    hyps, hl = random_hyps(g, 37, N, 200, 29, 0)
    assert_exact(lp.cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), 0, N)


@pytest.mark.gpu
@pytest.mark.parametrize("V,blank", [(7, 0), (7, 3), (7, 6), (40, 39)])
def test_blanks_short_frames_and_inf_rows(V, blank):
    """blank 0 / 3 / V-1; utterances of 1, 2 and T frames; -inf emissions (whole rows and single symbols); hypotheses
    made of repeats only, of blank-valued labels only, and infeasible ones."""
    g = torch.Generator().manual_seed(V + blank)
    B, T, Lmax, N = 6, 30, 14, 8
    lp = F.log_softmax(torch.randn(B, T, V, generator=g, dtype=torch.float64) * 2, -1)
    lp[3, 5, :] = -math.inf                      # a frame that no path can cross
    lp[4, :, 1 if blank != 1 else 2] = -math.inf  # a symbol that never appears
    lp[5, 7:9, blank] = -math.inf
    ll = torch.tensor([1, 2, T, T, T, T - 3])
    hyps, hl = random_hyps(g, B, N, Lmax, V, blank)
    hyps[:, 4] = 2 if blank != 2 else 1          # repeats only
    hl[:, 4] = torch.tensor([1, 1, 14, 10, 5, 13])
    hyps[:, 5] = blank                           # blank-valued labels only
    hl[:, 5] = torch.tensor([1, 2, 3, 14, 2, 7])
    hl[:, 6] = 1
    for dtype in (torch.float64, torch.float32):
        got = assert_exact(lp.to(dtype).cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), blank, dtype)
        assert_span_invariants(got[0], got[1], got[2], hyps, hl, got[3], blank)
        assert bool(torch.isneginf(got[3][3]).all())   # the -inf frame blocks every path
        assert bool(torch.isneginf(got[3][0][hl[0] >= 2]).all())   # one frame holds one label at most


@pytest.mark.gpu
@pytest.mark.parametrize("Lmax", CPT_BOUNDARIES)
def test_cells_per_thread_boundaries(Lmax):
    g = torch.Generator().manual_seed(Lmax)
    B, N, V = 2, 3, 6
    T = 2 * Lmax + 12
    lp = F.log_softmax(torch.randn(B, T, V, generator=g, dtype=torch.float64) * 2, -1).float()
    hyps, hl = random_hyps(g, B, N, Lmax, V, 0)
    hl[:, 2] = Lmax
    got = assert_exact(lp.cuda(), hyps.cuda(), hl.cuda(), torch.tensor([T, T - 5]).cuda(), 0, Lmax)
    assert_span_invariants(got[0], got[1], got[2], hyps, hl, got[3], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ALIGN_GOLDEN, ids=lambda p: os.path.basename(p)[:-4])
def test_agrees_with_get_alignment_3d(path):
    """N = 1: alignments byte for byte what get_alignment_3d_device writes; N = 3: each row what it writes on the
    log-probs repeated three times."""
    from end2end_b200.utils.alignment import get_alignment_3d_device
    z = np.load(path, allow_pickle=False)
    lp, tg = torch.from_numpy(z["log_probs"]).cuda(), torch.from_numpy(z["targets"]).cuda()
    ll, tl = torch.from_numpy(z["logits_lengths"]).cuda(), torch.from_numpy(z["targets_lengths"]).cuda()
    ref = get_alignment_3d_device(lp, tg, ll, tl, is_ctc=True)
    al = align(lp, tg[:, None], tl[:, None], ll)[0]
    assert torch.equal(al[:, 0], ref)
    g = torch.Generator().manual_seed(3)
    B, Lmax = tg.shape
    hyps = torch.stack([tg.cpu(), torch.randint(1, lp.size(2), (B, Lmax), generator=g), tg.cpu().flip(1)], 1)
    hl = torch.stack([tl.cpu(), torch.randint(0, Lmax + 1, (B,), generator=g), tl.cpu()], 1)
    al = align(lp, hyps.cuda(), hl.cuda(), ll)[0]
    ref = get_alignment_3d_device(lp.repeat_interleave(3, 0), hyps.reshape(3 * B, Lmax).cuda(), ll.repeat_interleave(3, 0),
                                  hl.reshape(-1).cuda(), is_ctc=True)
    assert torch.equal(al.reshape(3 * B, -1), ref)


def _rescore(lp, aligned, hl, hyps):
    """The path the kernel returned, scored under lp (fp64, frame order)."""
    B, N, T = aligned.shape
    out = torch.full((B, N), math.nan, dtype=torch.float64)
    for b in range(B):
        for n in range(N):
            row = aligned[b, n]
            f = row != -100
            out[b, n] = lp[b, torch.arange(T)[f], row[f]].to(torch.float64).sum()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,rtol", [(torch.float32, 1e-6), (torch.float64, 1e-12), (torch.bfloat16, 2.0 ** -7),
                                        (torch.float16, 2.0 ** -10)], ids=["f32", "f64", "bf16", "f16"])
def test_raw_logits(dtype, rtol):
    """Raw logits against the restatement on F.log_softmax(logits): the path score within 1e-6 relative for fp32 and
    one ulp of the input dtype per frame for 16-bit input (at most eps * |score|, every log-prob being <= 0), and the
    kernel's path, re-scored under those log-probs, within the same tolerance of the restatement's best.  16-bit
    log-probs are rounded to the input dtype as torch's CUDA log_softmax rounds them, so they differ from torch's only
    where the fp32 value sits at a rounding boundary: nearly every path score is then bit-equal to the restatement's."""
    from end2end_b200.engine import CTCBeamEngine
    g = torch.Generator().manual_seed(9)
    B, T, V, Lmax, N = 16, 120, 29, 40, 4
    x = (torch.randn(B, T, V, generator=g) * 3).to(dtype)
    ll = torch.randint(T // 2, T + 1, (B,), generator=g)
    hyps, hl = random_hyps(g, B, N, Lmax, V, 0)
    lp = F.log_softmax(x.cuda(), -1).cpu()        # torch's CUDA kernel: fp32 (x - max) - logsum, rounded to the dtype
    _, _, want, _, _ = align_cells(lp, hyps, hl, ll, 0)
    fin = torch.isfinite(want)

    def check(got, ctx):
        al, s0, s1, sc = (t.cpu() for t in got)
        assert torch.equal(torch.isfinite(sc), fin), ctx
        assert torch.equal(sc[~fin], want[~fin]), ctx
        assert bool(((sc[fin] - want[fin]).abs() <= rtol * want[fin].abs()).all()), (ctx, (sc - want)[fin].abs().max())
        re = _rescore(lp, al, hl, hyps)
        assert bool(((re[fin] - want[fin]).abs() <= rtol * want[fin].abs()).all()), ctx
        if dtype in (torch.bfloat16, torch.float16):
            assert float((sc[fin] == want[fin]).double().mean()) >= 0.9, (ctx, float((sc[fin] == want[fin]).double().mean()))
        assert_span_invariants(al, s0, s1, hyps, hl, sc, 0)

    eng = CTCBeamEngine(0, 1)
    check(eng.align_device(x.cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), from_logits=True), "batch-major")
    xt = x.transpose(0, 1).contiguous().cuda().transpose(0, 1)   # time-major storage
    check(eng.align_device(xt, hyps.int().cuda(), hl.int().cuda(), ll.int().cuda(), from_logits=True), "time-major int32")
    check(eng.align_device(x, hyps, hl, ll, from_logits=True), "host input")
    full = torch.full((B,), T)
    _, _, want, _, _ = align_cells(lp, hyps, hl, full, 0)
    fin = torch.isfinite(want)
    check(eng.align_device(x.cuda(), hyps.cuda(), hl.cuda(), None, from_logits=True), "no lengths")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c2", "c4"])
def test_greedy_round_trip(name):
    """align of decode_greedy's result is the per-frame argmax path: on continuous random logits that path is the unique
    best path of its own transcript."""
    from end2end_b200 import CTCDecoder
    B, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS[name]
    x, _, ll, _ = oracle.make_inputs(B, T, V, Lmin, Lmax, seed, torch.float32, full)
    labels = ["_", " "] + [chr(97 + i % 26) for i in range(V - 2)]
    dec = CTCDecoder(beam_width=1, labels=labels)
    res = dec.decode_greedy(x.cuda(), ll.cuda())
    out = dec.align(x.cuda(), res.decoded_targets, res.decoded_targets_lengths, ll.cuda())
    am = x.argmax(-1)
    want = torch.where(torch.arange(T)[None] < ll[:, None], am, torch.full_like(am, -100))
    assert torch.equal(out.alignments[:, 0], want)
    assert bool(torch.isfinite(out.path_scores).all())
    assert_span_invariants(out.alignments, out.token_starts, out.token_ends, res.decoded_targets[:, None],
                           res.decoded_targets_lengths[:, None], out.path_scores, 0)
    lp = F.log_softmax(x, -1).double()
    best = lp.max(-1).values
    want_s = torch.stack([best[b, :int(ll[b])].sum() for b in range(B)])
    assert bool(((out.path_scores[:, 0] - want_s).abs() <= 1e-6 * want_s.abs()).all())
    for b in range(B):                            # the words are the sentence's
        assert " ".join(w for w, _, _ in out.word_spans[b][0]) == " ".join(res.decoded_sentences[b].split())


@pytest.mark.gpu
def test_nbest_lists_bounded_by_score():
    """On decode_nbest lists: path_scores <= score within 1e-11 relative wherever finite; spans hold their invariants;
    unused slots and decode's empty result are the empty hypothesis."""
    from end2end_b200 import CTCDecoder
    B, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS["c2"]
    x, _, ll, _ = oracle.make_inputs(B, T, V, Lmin, Lmax, seed, torch.float32, full)
    x, ll = x[:16].cuda(), ll[:16].cuda()
    dec = CTCDecoder(beam_width=100, labels=["_", " "] + [chr(97 + i) for i in range(V - 2)], wip=0.0)
    nb = dec.decode_nbest(x, ll, n_best=10)
    al = dec.align(x, nb.decoded_targets, nb.decoded_targets_lengths, ll)
    sc = dec.score(x, nb.decoded_targets, nb.decoded_targets_lengths, ll)
    ps = al.path_scores
    fin = torch.isfinite(ps) & torch.isfinite(sc)
    assert bool(fin.any())
    assert bool((ps[fin] <= sc[fin] + 1e-11 * sc[fin].abs()).all())
    lens = nb.decoded_targets_lengths.clone()
    lens[(nb.decoded_targets[:, :, 0] == -1) & (lens == 1)] = 0   # decode's empty result is the empty hypothesis
    assert bool((al.token_starts[lens == 0] == -1).all())
    assert_span_invariants(al.alignments, al.token_starts, al.token_ends, nb.decoded_targets, lens, ps, 0)
    assert len(al.word_spans) == 16 and all(len(r) == 10 for r in al.word_spans)


@pytest.mark.gpu
def test_repeat_and_permutation():
    lp, ll, Lmax = _log_probs("c4", torch.float32)
    lp, ll = lp[:24].cuda(), ll[:24].cuda()
    g = torch.Generator().manual_seed(2)
    hyps, hl = random_hyps(g, 24, 7, Lmax, lp.size(2), 0)
    hyps, hl = hyps.cuda(), hl.cuda()
    a = align(lp, hyps, hl, ll)
    b = align(lp, hyps, hl, ll)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert torch.equal(a[3].view(torch.int64), b[3].view(torch.int64))
    perm = torch.randperm(7, generator=g).cuda()
    c = align(lp, hyps[:, perm], hl[:, perm], ll)
    for u, v in zip(a, c):
        assert torch.equal(u[:, perm], v)


@pytest.mark.gpu
def test_bad_rows_are_isolated():
    """Device-resident bad hypothesis lengths / labels give NaN and -1 spans for their own rows; a bad logits length
    for every hypothesis of its utterance; every other row is exact."""
    lp, ll, Lmax = _log_probs("c1", torch.float64)
    g = torch.Generator().manual_seed(4)
    B, V, N = lp.size(0), lp.size(2), 3
    hyps, hl = random_hyps(g, B, N, Lmax, V, 0)
    hl[0, 1] = Lmax + 1
    hl[1, 2] = -1
    hyps[2, 0, 0], hl[2, 0] = V, max(int(hl[2, 0]), 1)
    ll = ll.clone()
    ll[3] = lp.size(1) + 1
    al, s0, s1, sc = (t.cpu() for t in align(lp.cuda(), hyps.cuda(), hl.cuda(), ll.cuda()))
    bad = torch.zeros(B, N, dtype=torch.bool)
    bad[0, 1] = bad[1, 2] = bad[2, 0] = True
    bad[3, :] = True
    assert bool(torch.isnan(sc[bad]).all()) and not bool(torch.isnan(sc[~bad]).any())
    assert bool((s0[bad] == -1).all()) and bool((s1[bad] == -1).all())
    assert bool((al[bad] == -100).all())
    ok_hl = torch.where(bad, torch.zeros_like(hl), hl)
    ok_hyps = torch.where(hyps >= V, torch.zeros_like(hyps), hyps)
    ll_ok = ll.clone()
    ll_ok[3] = lp.size(1)
    want_al, _, want_v, want_s, want_e = align_cells(lp, ok_hyps, ok_hl, ll_ok, 0)
    assert torch.equal(al[~bad], want_al[~bad])
    assert torch.equal(s0[~bad], want_s[~bad]) and torch.equal(s1[~bad], want_e[~bad])
    assert torch.equal(sc[~bad], want_v[~bad])

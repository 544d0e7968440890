"""The kernels next to the loss, variant by variant: K6 Viterbi alignment (csrc/ctc_viterbi.cu), K7 CTC without blank
(csrc/ctc_noblank.cu), K5 greedy decoding (csrc/ctc_greedy.cu), and a guard on the beam search's large-alphabet
prefilter (csrc/ctc_beam.cu).

Each kernel is driven onto every compiled variant and every launch path, at the shapes and values where such kernels go
wrong (variant boundaries, prefetch tails, ties, NaN / -inf, strided views, infeasible utterances), and compared with a
plain reference of the same operation:
* Viterbi and greedy against the C oracle (oracle.get_alignment_3d, oracle.greedy_decode): integers, bit-exact;
* CTC without blank against the C oracle for 32- and 16-bit inputs, and for float64 inputs against `_nb_ref` below, a
  float64 numpy restatement of the recursions (the oracle reads float32, so it cannot check float64 arithmetic);
* beam search against the C restatement of the reference's decoder, tie counters included.
"""
import ctypes
import ctypes.util

import numpy as np
import pytest
import torch

import oracle

pytestmark = pytest.mark.gpu
NINF = float("-inf")


def _gen(seed):
    return np.random.default_rng(seed)


def _log_softmax(rng, B, T, V, dtype, scale=1.0):
    x = torch.from_numpy(rng.standard_normal((B, T, V)) * scale)
    return torch.log_softmax(x, 2).to(dtype)


def _labels(rng, B, Lmax, V, excluded=None, repeat=0.25):
    """[B, Lmax] int64 labels in [0, V) without `excluded`, with adjacent repeats at the given rate."""
    if excluded is None:
        tg = rng.integers(0, V, (B, max(Lmax, 0)))
    else:
        tg = rng.integers(0, V - 1, (B, max(Lmax, 0)))
        tg = tg + (tg >= excluded)
    rep = rng.random(tg.shape) < repeat
    for i in range(1, tg.shape[1]):
        tg[:, i] = np.where(rep[:, i], tg[:, i - 1], tg[:, i])
    return tg


def _repeats(row, L):
    return int(np.count_nonzero(row[1:L] == row[:L - 1])) if L > 1 else 0


# ---------------------------------------------------------------------------------------------------------------------
# K6 Viterbi forced alignment
# ---------------------------------------------------------------------------------------------------------------------
ALIGN_KINDS = ("ragged", "T0", "T1", "tight", "infeasible", "L0", "ragged", "full")


def _align_rows(rng, B, T, V, Lmax, is_ctc, blank=0, kinds=ALIGN_KINDS, repeat=0.25):
    """Targets, frame and label lengths: L spread over 0..Lmax (Lmax itself included), row kinds cycling over `kinds`.
    A CTC path needs L + (adjacent repeats) frames, an ASG path L frames; "tight" rows get exactly that many,
    "infeasible" rows one fewer."""
    tg = _labels(rng, B, Lmax, V, excluded=blank if is_ctc else None, repeat=repeat)
    L = np.linspace(0, Lmax, B).round().astype(np.int64)
    rng.shuffle(L)
    L[0] = Lmax
    ll = np.zeros(B, dtype=np.int64)
    for b in range(B):
        kind = kinds[b % len(kinds)]
        if kind == "L0":
            L[b] = 0
        need = lambda: int(L[b]) + (_repeats(tg[b], int(L[b])) if is_ctc else 0)   # noqa: E731
        if kind in ("tight", "infeasible"):
            while need() > T:
                L[b] -= 1
        n = need()
        ll[b] = {"ragged": rng.integers(min(n, T), T + 1), "full": T, "T0": 0, "T1": 1, "tight": n,
                 "infeasible": max(n - 1, 0), "L0": rng.integers(1, T + 1)}[kind]
    return torch.from_numpy(tg), torch.from_numpy(ll), torch.from_numpy(L)


def _align_check(lp, tg, ll, tl, is_ctc, blank=0, dev_lp=None, itype=torch.int64):
    from end2end_b200.utils.alignment import get_alignment_3d_device
    x = lp.cuda() if dev_lp is None else dev_lp
    out = get_alignment_3d_device(x, tg.to(itype).cuda(), ll.to(itype).cuda(), tl.to(itype).cuda(), is_ctc=is_ctc,
                                  blank_idx=blank).cpu()
    ref = oracle.get_alignment_3d(lp, tg, ll, tl, is_ctc=is_ctc, blank_idx=blank)
    bad = (out != ref).any(1).nonzero().flatten().tolist()
    assert not bad, "rows %s differ (T_i %s, L_i %s)" % (bad[:8], ll[bad[:8]].tolist(), tl[bad[:8]].tolist())
    return out


# CTC: 2 L + 1 cells, 1 / 2 / 4 cells per thread up to 512 / 1024 / 2048 cells; ASG: L cells
VIT_WIDTHS = [(True, 255), (True, 256), (True, 511), (True, 512), (True, 639), (True, 1023),
              (False, 512), (False, 513), (False, 1024), (False, 1025), (False, 2048)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("is_ctc,Lmax", VIT_WIDTHS, ids=["%s%d" % ("ctc" if c else "asg", w) for c, w in VIT_WIDTHS])
def test_viterbi_width_matrix_vs_oracle(is_ctc, Lmax, dtype):
    """Every cells-per-thread variant in both staging types, at and next to each variant boundary and at the widest
    lattice: ragged, empty (T_i = 0), one-frame, tight, one-frame-short and label-free rows."""
    rng = _gen(Lmax * 2 + is_ctc)
    B, V = 24, 29
    T = int(1.3 * Lmax) + 12
    tg, ll, tl = _align_rows(rng, B, T, V, Lmax, is_ctc)
    _align_check(_log_softmax(rng, B, T, V, dtype), tg, ll, tl, is_ctc)


def test_viterbi_bf16_widest():
    rng = _gen(7)
    B, V, Lmax = 12, 29, 1023
    T = int(1.3 * Lmax) + 12
    tg, ll, tl = _align_rows(rng, B, T, V, Lmax, True)
    _align_check(_log_softmax(rng, B, T, V, torch.bfloat16), tg, ll, tl, True)


def test_viterbi_one_label_past_the_limit_raises():
    from end2end_b200.utils.alignment import get_alignment_3d_device
    for is_ctc, widest in ((True, 1023), (False, 2048)):
        lp = torch.log_softmax(torch.randn(1, widest + 20, 8), 2).cuda()
        tg = torch.ones(1, widest + 1, dtype=torch.int64).cuda()
        ll, tl = torch.tensor([widest + 20]).cuda(), torch.tensor([widest]).cuda()
        with pytest.raises(NotImplementedError):
            get_alignment_3d_device(lp, tg, ll, tl, is_ctc=is_ctc)
        get_alignment_3d_device(lp, tg[:, :widest], ll, tl, is_ctc=is_ctc)       # the widest lattice runs


@pytest.mark.parametrize("Lmax,T", [(200, 300), (256, 400), (512, 560)], ids=["cpt1", "cpt2", "cpt4"])
def test_viterbi_backpointers_shared_and_workspace(Lmax, T):
    """Backpointers go to shared memory while they fit the CTA's budget (200 KB up to 148 utterances, 96 KB above) and
    to the workspace otherwise: these shapes need 126-184 KB, so the same utterances take shared memory in a batch of
    148 and the workspace in a batch of 149."""
    rng = _gen(Lmax)
    V = 29
    tg, ll, tl = _align_rows(rng, 149, T, V, Lmax, True, repeat=0.05)
    lp = _log_softmax(rng, 149, T, V, torch.float32)
    a = _align_check(lp[:148], tg[:148], ll[:148], tl[:148], True)
    b = _align_check(lp, tg, ll, tl, True)
    assert torch.equal(a, b[:148])


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32_D8", "f64_D4"])
@pytest.mark.parametrize("Lmax", [6, 600], ids=["cpt1", "cpt4"])
def test_viterbi_prefetch_tails(dtype, Lmax):
    """Emissions are fetched D frames ahead (D = 8 for float staging, 4 for double): every utterance length from 1 to
    2 D + 1, so every tail of the prefetch block, with short label sequences in (padded) target columns."""
    D = 8 if dtype == torch.float32 else 4
    rng = _gen(D + Lmax)
    Ts = np.arange(1, 2 * D + 2)
    B, T, V = len(Ts) * 2, 2 * D + 1, 11
    for is_ctc in (True, False):
        tg = torch.from_numpy(_labels(rng, B, Lmax, V, excluded=0 if is_ctc else None))
        ll = torch.from_numpy(np.concatenate([Ts, Ts]))
        tl = torch.from_numpy(np.concatenate([(Ts + 1) // 3, np.minimum(Ts, 5)]))
        _align_check(_log_softmax(rng, B, T, V, dtype), tg, ll, tl, is_ctc)


@pytest.mark.parametrize("Lmax", [400, 700], ids=["cpt2", "cpt4"])
def test_viterbi_blank_index(Lmax):
    rng = _gen(Lmax + 1)
    B, V = 8, 17
    T = int(1.3 * Lmax) + 12
    for blank in (0, 3, V - 1):
        tg, ll, tl = _align_rows(rng, B, T, V, Lmax, True, blank=blank)
        _align_check(_log_softmax(rng, B, T, V, torch.float32), tg, ll, tl, True, blank=blank)


@pytest.mark.parametrize("is_ctc,Lmax", [(True, 200), (True, 400), (True, 700), (False, 400), (False, 700), (False, 1500)])
def test_viterbi_minus_inf_inputs(is_ctc, Lmax):
    """-inf log-probabilities: one symbol impossible in every frame (and used as a label), plus scattered -inf cells."""
    rng = _gen(Lmax + 3)
    B, V = 8, 13
    T = int(1.3 * Lmax) + 12
    tg, ll, tl = _align_rows(rng, B, T, V, Lmax, is_ctc)
    tg[1::2, 3] = 5                                  # the impossible symbol in every other utterance's targets
    lp = _log_softmax(rng, B, T, V, torch.float64)
    lp[:, :, 5] = NINF
    lp[torch.from_numpy(rng.random(lp.shape) < 0.03)] = NINF
    _align_check(lp, tg, ll, tl, is_ctc)
    _align_check(lp.float(), tg, ll, tl, is_ctc)


@pytest.mark.parametrize("is_ctc,Lmax", [(True, 200), (True, 400), (True, 900), (False, 400), (False, 900), (False, 1800)],
                         ids=["ctc_cpt1", "ctc_cpt2", "ctc_cpt4", "asg_cpt1", "asg_cpt2", "asg_cpt4"])
def test_viterbi_uniform_rows_and_fp64_near_ties(is_ctc, Lmax):
    """Uniform rows make every comparison an exact tie, so the comparison order decides every cell (stay, then i-1,
    then i-2; the first wins).  The same rows with jitter of ~1e-12 are ties in float32 but not in float64: only
    float64 staging of float64 inputs gets them right."""
    rng = _gen(Lmax + 5)
    B, V = 8, 7
    T = int(1.3 * Lmax) + 12
    tg, ll, tl = _align_rows(rng, B, T, V, Lmax, is_ctc)
    flat = torch.full((B, T, V), -float(np.log(V)), dtype=torch.float64)
    _align_check(flat, tg, ll, tl, is_ctc)
    _align_check(flat.float(), tg, ll, tl, is_ctc)
    jit = flat + torch.from_numpy(rng.standard_normal((B, T, V)) * 1e-12)
    assert torch.equal(jit.float(), flat.float())
    _align_check(jit, tg, ll, tl, is_ctc)


def test_viterbi_fp64_planted_near_tie():
    """Two ASG paths over labels (1, 2) whose scores differ by 1e-12: the second frame's label 1 is better than its
    label 2 by that much, so the path 1 1 2 wins.  Rounded to float32 both are -1 and the tie keeps the stay, 1 2 2."""
    from end2end_b200.utils.alignment import get_alignment_3d_device
    lp = torch.full((1, 3, 4), -5.0, dtype=torch.float64)
    lp[0, :, 1] = lp[0, :, 2] = -1.0
    lp[0, 1, 1] = -1.0 + 1e-12
    tg, ll, tl = torch.tensor([[1, 2]]), torch.tensor([3]), torch.tensor([2])
    assert oracle.get_alignment_3d(lp, tg, ll, tl, is_ctc=False)[0].tolist() == [1, 1, 2]
    out = get_alignment_3d_device(lp.cuda(), tg.cuda(), ll.cuda(), tl.cuda(), is_ctc=False).cpu()
    assert out[0].tolist() == [1, 1, 2]


@pytest.mark.parametrize("is_ctc,Lmax", [(True, 300), (True, 800), (False, 1600)])
def test_viterbi_peaky_logits(is_ctc, Lmax):
    rng = _gen(Lmax + 9)
    B, V = 12, 29
    T = int(1.3 * Lmax) + 12
    tg, ll, tl = _align_rows(rng, B, T, V, Lmax, is_ctc)
    _align_check(_log_softmax(rng, B, T, V, torch.float32, scale=8.0), tg, ll, tl, is_ctc)


@pytest.mark.parametrize("is_ctc,Lmax", [(True, 700), (False, 1500)])
def test_viterbi_time_major_view_int32_indices_cpt4(is_ctc, Lmax):
    rng = _gen(Lmax + 11)
    B, V = 8, 29
    T = int(1.3 * Lmax) + 12
    tg, ll, tl = _align_rows(rng, B, T, V, Lmax, is_ctc)
    for dtype in (torch.float32, torch.float64):
        lp = _log_softmax(rng, B, T, V, dtype)
        tm = lp.permute(1, 0, 2).contiguous().cuda().permute(1, 0, 2)        # time-major storage, read in place
        _align_check(lp, tg, ll, tl, is_ctc, dev_lp=tm, itype=torch.int32)


def test_viterbi_fuzz():
    rng = _gen(2024)
    bins = {True: [(0, 8), (30, 90), (250, 262), (505, 520), (700, 1023)],
            False: [(0, 8), (60, 200), (505, 520), (1020, 1030), (1500, 2048)]}
    for case in range(150):
        is_ctc = bool(rng.integers(0, 2))
        lo, hi = bins[is_ctc][rng.integers(0, 5)]
        Lmax = int(rng.integers(lo, hi + 1))
        B = int(rng.integers(1, 5))
        V = int(rng.integers(3, 40))
        T = int(rng.integers(1, 20) + Lmax * rng.choice([0.6, 1.0, 1.3, 1.7]))
        dtype = [torch.float32, torch.float64, torch.bfloat16][rng.integers(0, 3)]
        blank = int(rng.choice([0, rng.integers(0, V), V - 1]))
        kinds = [("ragged", "full", "L0"), ("tight", "T1"), ("infeasible", "T0")][rng.integers(0, 3)]
        tg, ll, tl = _align_rows(rng, B, T, V, Lmax, is_ctc, blank=blank, kinds=kinds)
        mode = rng.integers(0, 3)
        lp = _log_softmax(rng, B, T, V, torch.float64, scale=[1.0, 8.0, 0.0][mode])
        if mode == 2:
            lp = lp + torch.from_numpy(rng.standard_normal(lp.shape) * 1e-12)
        lp = lp.to(dtype)
        layout = rng.integers(0, 3)
        if layout == 1:
            dev = lp.permute(1, 0, 2).contiguous().cuda().permute(1, 0, 2)
        elif layout == 2:
            dev = torch.cat([lp, lp[:, :, :3]], 2).cuda()[:, :, :V]          # an alphabet slice of a wider tensor
        else:
            dev = lp.cuda()
        try:
            _align_check(lp, tg, ll, tl, is_ctc, blank=blank, dev_lp=dev,
                         itype=torch.int32 if rng.integers(0, 2) else torch.int64)
        except AssertionError as e:
            raise AssertionError("case %d (is_ctc %s Lmax %d B %d T %d V %d %s blank %d mode %d layout %d): %s"
                                 % (case, is_ctc, Lmax, B, T, V, dtype, blank, mode, layout, e)) from None


# ---------------------------------------------------------------------------------------------------------------------
# K7 CTC without blank
# ---------------------------------------------------------------------------------------------------------------------
def _lse2(a, b):
    """The reference's two-argument log-sum-exp (functions/utils.py:6-24), elementwise, as the kernel computes it."""
    with np.errstate(all="ignore"):
        hi = np.where(a > b, a, b)
        lo = np.where(a > b, b, a)
        r = hi + np.log(1.0 + np.exp(lo - hi))
    return np.where(a == NINF, b, np.where(b == NINF, a, r))


def _nb_utterance(lp, tg, Ti, Li, space):
    """One utterance in float64: -log Z and the posterior of every symbol per frame, [Ti, V].  The recursions of the
    csrc/ctc_noblank.cu header and of the reference (ctc_without_blank.py:13-88), with its window and start / end cells."""
    V = lp.shape[1]
    first = int(tg[0]) if Li > 0 else -1
    if Li == 0 or (Li == 1 and first == space):
        ext, uas = [space], False
    elif space == -1:
        ext, uas = [int(v) for v in tg[:Li]], False
    else:
        ext, uas = [space] + [int(v) for v in tg[:Li]] + [space], True
    ext = np.array([v + V if v < 0 else v for v in ext])      # numpy's negative index of the reference: -1 is V - 1
    S = len(ext)
    j = np.arange(S)
    A = np.full((Ti, S), NINF)
    Bt = np.full((Ti, S), NINF)

    def window(t):
        return (max(0, S - Ti + t - 1), min(t + 2, S)) if uas else (max(0, S - Ti + t), min(t + 1, S))

    if Ti > 1 or S == 1:
        A[0, 0] = lp[0, ext[0]]
    if S > 1 and uas:
        A[0, 1] = lp[0, ext[1]]
    for t in range(1, Ti):
        s, e = window(t)
        prev = A[t - 1]
        nv = _lse2(prev, np.concatenate(([NINF], prev[:-1]))) + lp[t, ext]
        A[t] = np.where((j >= s) & (j < e), nv, NINF)
    if Ti > 1 or S == 1:
        Bt[Ti - 1, S - 1] = 0.0
    if S > 1 and uas:
        Bt[Ti - 1, S - 2] = 0.0
    for t in range(Ti - 2, -1, -1):
        s, e = window(t)
        nxt = Bt[t + 1] + lp[t + 1, ext]
        nv = _lse2(nxt, np.concatenate((nxt[1:], [NINF])))
        Bt[t] = np.where((j >= s) & (j < e), nv, NINF)
    logz = _lse2(A[Ti - 1, S - 1], A[Ti - 1, S - 2]) if (S > 1 and uas) else A[Ti - 1, S - 1]
    with np.errstate(all="ignore"):
        post = np.zeros((Ti, V))
        post[:, np.setdiff1d(np.arange(V), ext)] = np.exp(NINF - logz)     # no cell: exp(-inf - logZ), NaN if logZ = -inf
        for jj in range(S):                                                   # lattice order, linear domain
            post[:, ext[jj]] += np.exp(A[:, jj] + Bt[:, jj] - logz)
    return -float(logz), post


def _nb_ref(lp, tg, ll, tl, space, first=np.exp):
    """Batch restatement: (losses [B], grads [B, T, V]) in float64, grads = first(lp) - posterior, 0 past T_i."""
    lp = np.asarray(lp, dtype=np.float64)
    B, T, V = lp.shape
    losses = np.zeros(B)
    grads = np.zeros((B, T, V))
    for b in range(B):
        Ti, Li = int(ll[b]), int(tl[b])
        losses[b], post = _nb_utterance(lp[b], np.asarray(tg[b]), Ti, Li, space)
        grads[b, :Ti] = first(lp[b, :Ti]) - post
    return torch.from_numpy(losses), torch.from_numpy(grads)


_libm = None


def _expf(x):
    """float32 exp through the C library's expf, as the oracle computes the reference's np.exp of float32 inputs."""
    global _libm
    if _libm is None:
        _libm = ctypes.CDLL(ctypes.util.find_library("m"))
        _libm.expf.restype, _libm.expf.argtypes = ctypes.c_float, [ctypes.c_float]
    f = np.frompyfunc(lambda v: float(_libm.expf(float(v))), 1, 1)
    return f(np.asarray(x, dtype=np.float32)).astype(np.float64)


def _close(ours, ref, rtol, atol, what):
    ours, ref = ours.detach().cpu().double(), ref.detach().cpu().double()
    assert ours.shape == ref.shape, what
    assert torch.equal(torch.isnan(ours), torch.isnan(ref)), what + ": NaN positions differ"
    assert torch.equal(torch.isinf(ours), torch.isinf(ref)), what + ": inf positions differ"
    fin = torch.isfinite(ref)
    if bool(fin.any()):
        err = (ours[fin] - ref[fin]).abs()
        assert torch.equal(ours[torch.isinf(ref)], ref[torch.isinf(ref)]), what + ": inf signs differ"
        assert bool((err <= atol + rtol * ref[fin].abs()).all()), "%s: max err %.3e" % (what, float(err.max()))


NB_KINDS = ("ragged", "tight", "infeasible", "T1", "L0", "full")


def _nb_rows(rng, B, T, V, Lmax, kinds=NB_KINDS, plant=None):
    """Targets and lengths for CTC without blank: a path needs L frames; T_i >= 1 always."""
    tg = _labels(rng, B, Lmax, V)
    if plant is not None and Lmax > 2:
        tg[::2, 1] = plant
    L = np.linspace(0, Lmax, B).round().astype(np.int64)
    rng.shuffle(L)
    L[0] = Lmax
    ll = np.zeros(B, dtype=np.int64)
    for b in range(B):
        kind = kinds[b % len(kinds)]
        if kind == "L0":
            L[b] = 0
        if kind in ("tight", "infeasible"):
            L[b] = min(max(min(L[b], T), 2), Lmax)
        n = int(L[b])
        ll[b] = {"ragged": rng.integers(max(min(n, T), 1), T + 1), "full": T, "T1": 1, "tight": max(n, 1),
                 "infeasible": max(n - 1, 1), "L0": rng.integers(1, T + 1)}[kind]
    return torch.from_numpy(tg), torch.from_numpy(ll), torch.from_numpy(L)


def _nb_run(lp, tg, ll, tl, space, dev_lp=None, itype=torch.int64, ltype=None):
    from end2end_b200.functions.ctc_without_blank import ctc_without_blank_3d_loss
    x = lp.cuda() if dev_lp is None else dev_lp
    ltype = itype if ltype is None else ltype
    losses, grads = ctc_without_blank_3d_loss(x, tg.to(itype).cuda(), ll.to(ltype).cuda(), tl.to(ltype).cuda(), space)
    assert losses.dtype == x.dtype and grads.dtype == x.dtype and grads.stride() == x.stride()
    return losses, grads


# float64 kernel vs float64 restatement: the same operations in the same order, so only the last ulp of CUDA's and the
# host's exp / log can differ.  Measured on a B200 (1000 W) over the team-mode shapes and 60 fuzz shapes: identical
# losses, gradients within 8.8e-14 absolute (posteriors from alpha + beta - logZ of magnitude up to ~3,500).
NB64_TOL = 1e-12


def _nb_check64(lp, tg, ll, tl, space, what, **kw):
    losses, grads = _nb_run(lp, tg, ll, tl, space, **kw)
    l_ref, g_ref = _nb_ref(lp.numpy(), tg.numpy(), ll, tl, space)
    _close(losses, l_ref, NB64_TOL, NB64_TOL, what + " f64 losses")
    _close(grads, g_ref, NB64_TOL, NB64_TOL, what + " f64 grads")


def _nb_check_oracle(lp, tg, ll, tl, space, what, tol=1e-5, **kw):
    losses, grads = _nb_run(lp, tg, ll, tl, space, **kw)
    l_ref, g_ref = oracle.ctc_without_blank(lp.float(), tg, ll, tl, space)
    _close(losses, l_ref, tol, tol, what + " losses")
    _close(grads, g_ref, tol, tol, what + " grads")


def test_noblank_restatement_matches_oracle():
    """The float64 restatement is the oracle's computation: on float32 inputs (what the oracle reads) they agree to 1e-10,
    with spaces, ragged / tight / infeasible / one-frame / label-free rows and -inf inputs."""
    rng = _gen(11)
    B, T, V = 12, 40, 9
    for space in (-1, 0, 4, V - 1):
        tg, ll, tl = _nb_rows(rng, B, T, V, 30, plant=space if space >= 0 else None)
        lp = _log_softmax(rng, B, T, V, torch.float32)
        lp[3, :, 2] = NINF
        l_ref, g_ref = oracle.ctc_without_blank(lp, tg, ll, tl, space)
        l_me, g_me = _nb_ref(lp.double().numpy(), tg.numpy(), ll, tl, space, first=_expf)
        _close(l_me, l_ref, 1e-10, 1e-10, "space %d losses" % space)
        _close(g_me, g_ref, 1e-10, 1e-10, "space %d grads" % space)


@pytest.mark.parametrize("Lmax", [30, 510, 511, 1022], ids=["two_teams_30", "two_teams_510", "one_team_511", "one_team_1022"])
def test_noblank_team_modes(Lmax):
    """Lmax + 2 cells on one thread each: up to 512 cells the alpha and beta sweeps run side by side in one CTA (two
    teams), above it one after the other (one team), up to the limit of 1024 cells.  The space symbol is absent, the
    first or last symbol, or a symbol that also occurs in the targets.  With space = -1 a label-free row has the
    single cell -1, which the reference indexes as numpy does (symbol V - 1); the kernel and the oracle do the same, and
    such rows are included."""
    rng = _gen(Lmax)
    B, V = 6, 23
    T = int(1.1 * Lmax) + 8
    for space in (-1, 0, V - 1, 7):
        tg, ll, tl = _nb_rows(rng, B, T, V, Lmax, plant=7 if space == 7 else None)
        lp = _log_softmax(rng, B, T, V, torch.float64)
        _nb_check64(lp, tg, ll, tl, space, "Lmax %d space %d" % (Lmax, space))
        _nb_check_oracle(lp.float(), tg, ll, tl, space, "Lmax %d space %d f32" % (Lmax, space))


def test_noblank_one_label_past_the_limit_raises():
    from end2end_b200.functions.ctc_without_blank import ctc_without_blank_3d_loss
    lp = torch.log_softmax(torch.randn(1, 1040, 8), 2).cuda()
    tg = torch.ones(1, 1023, dtype=torch.int64).cuda()
    with pytest.raises(NotImplementedError):
        ctc_without_blank_3d_loss(lp, tg, torch.tensor([1040]).cuda(), torch.tensor([1000]).cuda())


@pytest.mark.parametrize("dtype,tol", [(torch.bfloat16, 2.0 ** -8), (torch.float16, 2.0 ** -11)], ids=["bf16", "f16"])
def test_noblank_16bit_inputs(dtype, tol):
    """16-bit inputs against the oracle on the widened input, within one ulp of the stored type."""
    rng = _gen(16)
    B, T, V = 16, 120, 29
    for space, Lmax in ((-1, 60), (3, 60), (-1, 600)):
        T_ = max(T, int(1.1 * Lmax) + 8)
        tg, ll, tl = _nb_rows(rng, B, T_, V, Lmax)
        lp = _log_softmax(rng, B, T_, V, dtype)
        _nb_check_oracle(lp, tg, ll, tl, space, "%s space %d" % (dtype, space), tol=tol)


def test_noblank_layouts_and_index_types():
    """A time-major storage read through a batch-major view, and an alphabet slice of a wider tensor: the gradient is
    written with the input's strides.  int32 and int64 index tensors, mixed."""
    rng = _gen(17)
    B, T, V = 8, 70, 19
    tg, ll, tl = _nb_rows(rng, B, T, V, 40)
    for dtype in (torch.float64, torch.float32):
        lp = _log_softmax(rng, B, T, V, dtype)
        tm = lp.permute(1, 0, 2).contiguous().cuda().permute(1, 0, 2)
        wide = torch.cat([lp, lp[:, :, :5]], 2).cuda()[:, :, :V]
        for dev, itype, ltype in ((tm, torch.int32, torch.int64), (wide, torch.int64, torch.int32), (tm, torch.int32, torch.int32)):
            kw = dict(dev_lp=dev, itype=itype, ltype=ltype)
            if dtype == torch.float64:
                _nb_check64(lp, tg, ll, tl, 4, "layout", **kw)
            else:
                _nb_check_oracle(lp, tg, ll, tl, 4, "layout", **kw)


def test_noblank_fuzz():
    rng = _gen(4096)
    for case in range(100):
        B = int(rng.integers(1, 6))
        V = int(rng.integers(2, 40))
        Lmax = int(rng.choice([rng.integers(0, 8), rng.integers(8, 80), rng.integers(480, 540)]))
        T = max(1, int(rng.integers(1, 12) + Lmax * rng.choice([0.7, 1.0, 1.3])))
        space = int(rng.choice([-1, 0, rng.integers(0, V), V - 1]))
        tg, ll, tl = _nb_rows(rng, B, T, V, Lmax, kinds=[NB_KINDS, ("tight", "T1"), ("infeasible", "L0")][rng.integers(0, 3)])
        dtype = torch.float64 if rng.integers(0, 2) else torch.float32
        lp = _log_softmax(rng, B, T, V, dtype, scale=float(rng.choice([1.0, 5.0])))
        layout = rng.integers(0, 3)
        dev = (lp.permute(1, 0, 2).contiguous().cuda().permute(1, 0, 2) if layout == 1 else
               torch.cat([lp, lp[:, :, :2]], 2).cuda()[:, :, :V] if layout == 2 else lp.cuda())
        kw = dict(dev_lp=dev, itype=torch.int32 if rng.integers(0, 2) else torch.int64,
                  ltype=torch.int32 if rng.integers(0, 2) else torch.int64)
        what = "case %d (B %d T %d V %d Lmax %d space %d %s layout %d)" % (case, B, T, V, Lmax, space, dtype, layout)
        if dtype == torch.float64:
            _nb_check64(lp, tg, ll, tl, space, what, **kw)
        else:
            _nb_check_oracle(lp, tg, ll, tl, space, what, **kw)


# ---------------------------------------------------------------------------------------------------------------------
# K5 greedy decoding
# ---------------------------------------------------------------------------------------------------------------------
GREEDY_DTYPES = [torch.float32, torch.float64, torch.bfloat16, torch.float16]
VEC_N = {torch.float32: 4, torch.float64: 2, torch.bfloat16: 8, torch.float16: 8}   # elements per 16-byte load


def _greedy_check(x, ll=None, blank=0, dev_x=None, what=""):
    from end2end_b200.engine import CTCGreedyEngine
    d = x.cuda() if dev_x is None else dev_x
    dec, lens = CTCGreedyEngine(blank).decode_greedy_device(d, None if ll is None else ll.cuda())
    rt, rl = oracle.greedy_decode(x, ll, blank_idx=blank, prefer="port")[:2]
    assert torch.equal(lens.cpu(), rl), what + ": lengths differ"
    bad = (dec.cpu() != rt).any(1).nonzero().flatten().tolist()
    assert not bad, "%s: utterances %s differ" % (what, bad[:8])


def _plant(rng, x, N):
    """Per frame, equal maxima (or NaNs, or +-0 / +inf ties) at positions the kernel reads from the same vector, the same
    lane in another 32-lane chunk, adjacent lanes, or lanes far apart.  The first one must win."""
    B, T, V = x.shape
    offs = [1, N - 1, N, N + 1, 32, 32 * N, 32 * N - 1, 64 * N, 3, 7 * N + 2]
    for b in range(B):
        for t in range(T):
            p = int(rng.integers(0, V))
            q = [p + o for o in offs if p + o < V] or [max(p - 1, 0)]
            q = int(rng.choice(q))
            kind = rng.integers(0, 8)
            if kind <= 3:                              # equal finite maxima, sometimes three of them
                x[b, t, p] = x[b, t, q] = 9.0
                if kind == 3:
                    x[b, t, int(rng.integers(0, V))] = 9.0
            elif kind == 4:                            # NaNs: the first NaN wins over everything
                x[b, t, q] = x[b, t, p] = float("nan")
                x[b, t, int(rng.integers(0, V))] = float("inf")
            elif kind == 5:                            # -0 and +0 are equal: the lower index wins
                x[b, t] = -torch.rand(V, dtype=torch.float64).to(x.dtype) - 1
                x[b, t, p], x[b, t, q] = -0.0, 0.0
                if rng.integers(0, 2):
                    x[b, t, p], x[b, t, q] = 0.0, -0.0
            elif kind == 6:
                x[b, t, p] = x[b, t, q] = float("inf")
            elif t % 2:
                x[b, t] = NINF if rng.integers(0, 2) else float("nan")   # all -inf: index 0; all NaN: index 0


def _greedy_vs(dtype):
    N = VEC_N[dtype]
    vec = [32 * N * nv for nv in (1, 2, 4, 8)] + [32 * N * 3 + N]             # NV = 1, 2, 4, 8 and a partial last chunk
    return vec, N


@pytest.mark.parametrize("dtype", GREEDY_DTYPES, ids=["f32", "f64", "bf16", "f16"])
def test_greedy_vector_paths_and_planted_ties(dtype):
    """Every vector-load variant (NV = 1, 2, 4, 8 loads per lane) and the scalar path through each of its gates on its
    own: an alphabet that is not a multiple of the vector, one larger than 8 loads per lane, a base address that is not
    16-byte aligned, a row stride that is not a multiple of 16 bytes.  Every frame has planted ties / NaNs / zeros."""
    vec, N = _greedy_vs(dtype)
    rng = _gen(N)
    B, T = 3, 40
    ll = torch.tensor([T, T - 7, 1])
    cases = [("vec V=%d" % V, V, None) for V in vec]
    cases += [("V % N", 32 * N + 1, None), ("V > 32*N*8", 32 * N * 8 + N, None),
              ("unaligned base", 32 * N * 2, "base"), ("row stride", 32 * N * 2, "stride")]
    for what, V, view in cases:
        x = (torch.rand(B, T, V, dtype=torch.float64) * 8 - 4).to(dtype)
        _plant(rng, x, N)
        if view == "base":
            # row stride V + N elements (a 16-byte multiple), base one element past a 16-byte boundary
            dev = torch.cat([x[:, :, :1], x, x[:, :, :N - 1]], 2).cuda()[:, :, 1:V + 1]
        elif view == "stride":
            dev = torch.cat([x, x[:, :, :1]], 2).cuda()[:, :, :V]    # aligned base, row stride V + 1
        else:
            dev = None
        for blank in (0, V - 1):
            _greedy_check(x, ll, blank=blank, dev_x=dev, what="%s %s blank %d" % (dtype, what, blank))


@pytest.mark.parametrize("T", [1, 31, 32, 33, 255, 256, 257, 1000])
def test_greedy_collapse_boundaries(T):
    """The collapse kernel scans 256 frames per step in eight 32-frame warps: runs of one symbol across the 32- and
    256-frame boundaries (the previous frame of a step's first frame is the last frame of the step before)."""
    rng = _gen(T)
    B, V = 6, 12
    for blank in (0, V - 1):
        sym = rng.integers(0, V, (B, T))
        for b in range(B):
            for edge in range(32, T, 32):
                if rng.random() < 0.7:
                    s = int(rng.integers(0, V))
                    sym[b, max(edge - int(rng.integers(1, 4)), 0):edge + int(rng.integers(1, 4))] = s
            if b % 3 == 0:
                sym[b, :] = (blank + 1) % V                          # one run over everything
        x = torch.from_numpy(rng.standard_normal((B, T, V)) * 0.1).float()
        x.scatter_(2, torch.from_numpy(sym).unsqueeze(2), 5.0)
        for ll in (None, torch.zeros(B, dtype=torch.int64), torch.ones(B, dtype=torch.int64), torch.full((B,), T),
                   torch.from_numpy(rng.integers(0, T + 1, B))):
            _greedy_check(x, ll, blank=blank, what="T %d blank %d lengths %s" % (T, blank, None if ll is None else ll.tolist()))


def test_greedy_host_input_equals_device_input():
    from end2end_b200.engine import CTCGreedyEngine
    rng = _gen(5)
    for dtype in GREEDY_DTYPES:
        x = (torch.rand(4, 300, 29, dtype=torch.float64) * 8 - 4).to(dtype)
        _plant(rng, x, VEC_N[dtype])
        ll = torch.tensor([300, 257, 1, 0])
        eng = CTCGreedyEngine(0)
        host = eng.decode_greedy(x, ll)
        dev = eng.decode_greedy(x.cuda(), ll.cuda())
        assert torch.equal(host[0], dev[0]) and torch.equal(host[1], dev[1])
        ref = oracle.greedy_decode(x, ll, prefer="port")
        assert torch.equal(host[0], ref[0]) and torch.equal(host[1], ref[1])


def test_greedy_fuzz():
    rng = _gen(777)
    for case in range(200):
        dtype = GREEDY_DTYPES[rng.integers(0, 4)]
        N = VEC_N[dtype]
        V = int(rng.choice([rng.integers(2, 40), 32 * N * int(rng.integers(1, 9)), rng.integers(40, 2 * 32 * N * 8)]))
        B, T = int(rng.integers(1, 5)), int(rng.integers(1, 300))
        x = (torch.rand(B, T, V, dtype=torch.float64) * 8 - 4).to(dtype)
        if rng.integers(0, 2):
            _plant(rng, x, N)
        blank = int(rng.choice([0, V - 1, rng.integers(0, V)]))
        ll = None if rng.integers(0, 3) == 0 else torch.from_numpy(rng.integers(0, T + 1, B))
        layout = rng.integers(0, 4)
        dev = (x.permute(1, 0, 2).contiguous().cuda().permute(1, 0, 2) if layout == 1 else
               torch.cat([x[:, :, :1], x], 2).cuda()[:, :, 1:] if layout == 2 else
               torch.cat([x, x[:, :, :3]], 2).cuda()[:, :, :V] if layout == 3 else None)
        _greedy_check(x, ll, blank=blank, dev_x=dev,
                      what="case %d (%s B %d T %d V %d blank %d layout %d)" % (case, dtype, B, T, V, blank, layout))


# ---------------------------------------------------------------------------------------------------------------------
# Beam search: the large-alphabet prefilter at small beams
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("beam,V", [(2, 9700), (3, 6500), (4, 5000), (5, 4000)])
def test_beam_prefilter_small_beams(beam, V):
    """With beam x alphabet above the 19,200 cached extensions each frame extends only the beam + 2 most probable
    symbols and the space.  Children that are pruned, or that already exist in the beam, must not change the result:
    every utterance equals the unfiltered C restatement of the reference's decoder, tie counters included."""
    from pytorch_end2end import CTCDecoder
    assert V * beam > 19200
    rng = _gen(beam)
    B, T = 4, 50
    labels = [chr(0x4e00 + i) for i in range(V)]
    space = int(rng.integers(1, V))
    labels[space] = " "
    for scale, wip in ((6.0, 0.0), (1.0, 0.5), (0.3, -0.7)):                 # peaky, flatter, near-flat rows
        x = torch.from_numpy(rng.standard_normal((B, T, V)) * scale).float()
        x[:, ::3, space] += 4.0                                               # spaces get extended often
        lp = torch.log_softmax(x, 2)
        ll = torch.tensor([T, T - 9, 1, 17])
        for lab in (labels, None):
            dec = CTCDecoder(beam_width=beam, after_logsoftmax=True, labels=lab, wip=wip if lab else 0.0)
            res = dec.decode(lp.cuda(), ll)
            port = oracle.beam_decode(lp, ll, beam_width=beam, labels=lab, after_logsoftmax=True,
                                      wip=wip if lab else 0.0, prefer="port", return_ties=True)
            got = [res.decoded_targets[i, :int(res.decoded_targets_lengths[i])].tolist() for i in range(B)]
            want = [port[0][i, :int(port[1][i])].tolist() for i in range(B)]
            assert got == want, (scale, wip, lab is not None)
            assert torch.equal(dec._decoder.last_ties, port[3])

"""Minimum word error rate over an N-best list (MWERLoss, MWERFunction, CTCBeamEngine.mwer_forward_device /
mwer_backward_device, e2e_ctc_mwer_*).

The definition checked here: for utterance b the list U_b is the slots in the mask whose score s_bn is finite,
p_bn = softmax(lambda s_b)_n over U_b, loss_b = R_b = sum_{U_b} p_bn r_bn and d loss_b / d s_bn = lambda p_bn (r_bn - R_b).
The scores are checked bit for bit against score_device, the loss against a host fp64 evaluation of the definition, and
the gradient against score_backward_device fed the host's weights (the scorer's gradient is tested against the oracle in
test_gpu_score_grad.py), against the composed CTCScore + softmax recipe, and with gradcheck.
"""
import ctypes

import pytest
import torch

import oracle

H = 8                                      # hypotheses per CTA (ctc_score.cu: kScoreWarps)
MAX_TARGETS = 639
K_BOUNDARIES = (15, 63, 64, 127, 128, 255, 256, 638, 639)
LABELS = ["_", " "] + list("abcdefghijklmnopqrstuvwxyz'")      # V = 29 (c2); label 1 separates words
NAN = float("nan")


def _desc(B, T, V, Lmax, blank=0, dtype=None, from_logits=0, itype=1):
    from end2end_b200 import _lib
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
    d.blank_idx, d.dtype = blank, _lib.E2E_F64 if dtype is None else dtype
    d.targets_itype = d.lengths_itype = itype
    d.from_logits = from_logits
    d.logits_stride_b, d.logits_stride_t = T * V, V
    d.grads_stride_b, d.grads_stride_t = T * V, V
    d.targets_stride_b = Lmax
    return d


def _a(x, k):
    return (x + k - 1) // k * k


def frames_per_block(V, Lmax):
    """ctc_score.cu: score_mode with K10's extra shared memory (test_gpu_score_grad.py's formula)."""
    Lp = Lmax + 1
    head = _a(H * Lp * 4, 16) + 2 * 32 * 8 + _a(H * Lp * 4, 16) + H * 16
    row = V * 8
    fb = min(32, max(8, 64 * 1024 // row))
    if head + fb * row <= 160 * 1024:
        return fb
    return min(32, (160 * 1024 - head) // (H * Lp * 8))


def mwer_bytes(B, T, V, Lmax, N):
    """(state, backward scratch): K10's workspace with the checkpoints moved to the state beside the scores and weights."""
    G, Kc, FB = (N + H - 1) // H, (2 * Lmax + 1 + 31) // 32, frames_per_block(V, Lmax)
    nblk = (T + FB - 1) // FB
    state = 2 * _a(B * N * 8, 256) + _a(B * N * nblk * Kc * 256, 256)
    ws = _a(B * G * 8, 256) + _a(B * G * 4, 256) + _a(B * N * FB * Kc * 256, 256) + _a(B * G * T * V * 8, 256)
    return state, ws


def engine(blank=0, labels=None):
    from end2end_b200.engine import CTCBeamEngine
    return CTCBeamEngine(blank, 1, labels)


def hyps_for(g, B, N, Lmax, V, blank=0):
    """Mixed lengths (0, 1, Lmax, random) and runs of repeated labels; blank never a label."""
    others = torch.tensor([v for v in range(V) if v != blank])
    hl = torch.randint(0, Lmax + 1, (B, N), generator=g)
    fixed = torch.tensor([0, 1, Lmax, max(Lmax - 1, 0)])
    hl[:, :min(N, 4)] = fixed[:min(N, 4)].clamp(max=Lmax)
    hyps = others[torch.randint(0, len(others), (B, N, max(Lmax, 1)), generator=g)][:, :, :Lmax].clone()
    if Lmax > 1:
        rep = torch.rand(B, N, Lmax, generator=g) < 0.3
        rep[:, :, 0] = False
        for k in range(1, Lmax):
            hyps[:, :, k] = torch.where(rep[:, :, k], hyps[:, :, k - 1], hyps[:, :, k])
    return hyps, hl


def host_mwer(s, risk, mask, lam):
    """The definition in fp64 on the host: (loss [B], d loss / d s [B, N])."""
    s, risk = s.detach().cpu().double(), risk.detach().cpu().double()
    mask = torch.ones_like(s, dtype=torch.bool) if mask is None else mask.cpu().bool()
    B, N = s.shape
    loss, g = torch.zeros(B, dtype=torch.float64), torch.zeros(B, N, dtype=torch.float64)
    for b in range(B):
        u = mask[b] & torch.isfinite(s[b])
        if bool(torch.isnan(s[b]).any()) or bool((~(risk[b][u] >= 0)).any()):
            loss[b], g[b] = NAN, NAN
            continue
        if not bool(u.any()):
            continue
        r = risk[b][u]
        if bool((r == r[0]).all()):
            loss[b] = r[0]
            continue
        p = torch.softmax(lam * s[b][u], 0)
        R = (p * r).sum()
        loss[b] = R
        g[b][u] = lam * p * (r - R)
    return loss, g


def assert_close(got, want, rtol, atol=0.0, ctx=None, norm=False):
    """Element-wise relative, or with ``norm`` relative to the largest magnitude: a raw-logit gradient sums g gamma and
    -(sum g) softmax with sum g = 0, so its small elements are differences of large ones."""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    assert torch.equal(torch.isnan(got), torch.isnan(want)), ctx
    ok = ~torch.isnan(want)
    err = (got[ok] - want[ok]).abs()
    bound = rtol * (want[ok].abs().max() if norm and bool(ok.any()) else want[ok].abs()) + atol
    assert bool((err <= bound).all()), (ctx, float(err.max()) if err.numel() else 0.0)


def _cfg(name, B):
    Bc, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS[name]
    x, tg, ll, tl = oracle.make_inputs(min(Bc, B), T, V, Lmin, Lmax, seed, full_length=full)
    return x.double(), ll, Lmax, tg, tl


# ---------------------------------------------------------------------------------------------- device-free ---------

def test_mwer_size_queries(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    lim = _lib.limits()
    for (B, T, V, Lmax) in ((4, 50, 29, 0), (4, 50, 29, 200), (3, 70, 1024, 80), (2, 70, 4096, 30), (2, 9, 29, MAX_TARGETS),
                            (1, 5, lim.max_alphabet, MAX_TARGETS)):
        for N in (1, H, H + 1, 100):
            d = ctypes.byref(_desc(B, T, V, Lmax))
            got = (L.e2e_ctc_mwer_state_bytes(d, N), L.e2e_ctc_mwer_backward_workspace_bytes(d, N))
            assert got == mwer_bytes(B, T, V, Lmax, N), (B, T, V, Lmax, N, got)
    for q in (L.e2e_ctc_mwer_state_bytes, L.e2e_ctc_mwer_backward_workspace_bytes):
        assert q(ctypes.byref(_desc(4, 50, 29, MAX_TARGETS + 1)), 1) == 0
        assert "target length 640" in L.e2e_last_error_string().decode()
        assert q(ctypes.byref(_desc(4, 50, lim.max_alphabet + 1, 10)), 1) == 0
        assert q(ctypes.byref(_desc(4, 50, 29, 10)), 0) == 0
        assert q(ctypes.byref(_desc(1, 2 ** 31 - 1, lim.max_alphabet, 4)), 2 ** 31 - 1) == 0


def test_mwer_argument_errors(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    d = _desc(2, 10, 5, 3)
    st = L.e2e_ctc_mwer_state_bytes(ctypes.byref(d), 2)
    ws = L.e2e_ctc_mwer_backward_workspace_bytes(ctypes.byref(d), 2)
    fake = ctypes.c_void_p(256)              # never dereferenced: every case fails before a launch
    fwd = [fake, fake, None, fake, fake, None, 1.0, fake, None, fake, st, None]

    def call_fwd(args, desc=d):
        return L.e2e_ctc_mwer_forward_device(ctypes.byref(desc), 2, *args)

    for i in (0, 1, 3, 4, 7):                # logits, hyps, hyp_lengths, risk, losses
        args = list(fwd)
        args[i] = None
        assert call_fwd(args) == 1 and "null pointer" in L.e2e_last_error_string().decode(), i
    for lam in (0.0, -1.0, float("inf"), NAN):
        args = list(fwd)
        args[6] = lam
        assert call_fwd(args) == 1 and "score_scale" in L.e2e_last_error_string().decode(), lam
    args = list(fwd)
    args[10] = st - 1
    assert call_fwd(args) == 3 and "too small" in L.e2e_last_error_string().decode()
    assert call_fwd(fwd, _desc(2, 10, 5, MAX_TARGETS + 1)) == 2
    bwd = [fake, fake, None, fake, fake, fake, fake, st, fake, ws, None]

    def call_bwd(args):
        return L.e2e_ctc_mwer_backward_device(ctypes.byref(d), 2, *args)

    for i in (0, 1, 3, 4, 5):                # logits, hyps, hyp_lengths, utt_scale, grads
        args = list(bwd)
        args[i] = None
        assert call_bwd(args) == 1 and "null pointer" in L.e2e_last_error_string().decode(), i
    for i, short in ((7, st - 1), (9, ws - 1)):
        args = list(bwd)
        args[i] = short
        assert call_bwd(args) == 3 and "too small" in L.e2e_last_error_string().decode(), i


def test_module_arguments(lib_built):
    from end2end_b200 import MWERLoss
    with pytest.raises(ValueError, match="score_scale"):
        MWERLoss(LABELS, score_scale=0.0)
    with pytest.raises(ValueError, match="score_scale"):
        MWERLoss(LABELS, score_scale=float("nan"))
    with pytest.raises(ValueError, match="\" \""):
        MWERLoss(list("_abc"), level="word")
    with pytest.raises(ValueError, match="level"):
        MWERLoss(LABELS, level="char")
    MWERLoss(list("_abc"), level="token")


# ---------------------------------------------------------------------------------------------- GPU -----------------

def _forward(eng, x, hyps, hl, risk, mask=None, ll=None, from_logits=False, lam=1.0):
    return eng.mwer_forward_device(x.cuda(), hyps.cuda(), hl.cuda(), risk.cuda(), None if mask is None else mask.cuda(),
                                   None if ll is None else ll.cuda(), from_logits, lam)


def _grad(eng, x, hyps, hl, state, w, ll=None, from_logits=False):
    return eng.mwer_backward_device(x.cuda(), hyps.cuda(), hl.cuda(), w.cuda(), state, None if ll is None else ll.cuda(),
                                    from_logits)


def _same_bits(a, b):
    a, b = a.cpu(), b.cpu()
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(0.0), b.nan_to_num(0.0))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("from_logits", [False, True])
@pytest.mark.parametrize("name,N", [("c1", 9), ("c2", 8), ("c3", 7), ("c4", 100), ("c2", 1)])
def test_scores_are_score_device(dtype, from_logits, name, N):
    x, ll, Lmax, _, _ = _cfg(name, 3 if N == 100 else 6)
    B, T, V = x.shape
    x = (x if from_logits else torch.log_softmax(x, 2)).to(dtype)
    g = torch.Generator().manual_seed(N)
    hyps, hl = hyps_for(g, B, N, min(Lmax, 60), V)
    mask = torch.rand(B, N, generator=g) < 0.8
    eng = engine()
    want = eng.score_device(x.cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), from_logits)
    _, s, _ = _forward(eng, x, hyps, hl, torch.rand(B, N, generator=g), mask, ll, from_logits)
    assert _same_bits(s[mask.cuda()], want[mask.cuda()])
    assert bool((s[~mask.cuda()] == float("-inf")).all())


@pytest.mark.gpu
@pytest.mark.parametrize("Lmax", K_BOUNDARIES)
def test_scores_k_variants(Lmax):
    g = torch.Generator().manual_seed(Lmax)
    B, N, V = 2, 9, 12
    T = 2 * Lmax + 10
    x = torch.log_softmax(torch.randn(B, T, V, generator=g, dtype=torch.float64), 2)
    hyps, hl = hyps_for(g, B, N, Lmax, V)
    ll = torch.tensor([T, max(T - 5, 1)])
    eng = engine()
    want = eng.score_device(x.cuda(), hyps.cuda(), hl.cuda(), ll.cuda())
    risk = torch.rand(B, N, generator=g, dtype=torch.float64)
    loss, s, state = _forward(eng, x, hyps, hl, risk, None, ll)
    assert _same_bits(s, want)
    wl, wg = host_mwer(want, risk, None, 1.0)
    assert_close(loss, wl, 1e-14, ctx=Lmax)
    got = _grad(eng, x, hyps, hl, state, torch.ones(B, dtype=torch.float64), ll)
    ref = eng.score_backward_device(x.cuda(), hyps.cuda(), hl.cuda(), wg.cuda(), ll.cuda())
    assert_close(got, ref, 1e-12, ctx=Lmax, norm=True)


def _nbest_case(B=8, N=8, seed=1):
    """c2-shaped utterances, the model's own N-best list and the utterances' references."""
    x, ll, _, tg, tl = _cfg("c2", B)
    eng = engine(0, LABELS)
    eng.beam_width = N
    hyps, hl, scores, _, _ = eng.decode_nbest_device(x.cuda(), ll.cuda(), n_best=N, from_logits=True)
    return x, ll, tg, tl, hyps, hl, scores > float("-inf")


@pytest.mark.gpu
@pytest.mark.parametrize("words", [True, False])
@pytest.mark.parametrize("lam", [0.3, 1.0, 2.0])
def test_loss_and_gradient_match_definition(words, lam):
    x, ll, tg, tl, hyps, hl, used = _nbest_case()
    eng = engine(0, LABELS)
    risk = eng.errors_device(hyps, hl, tg.cuda(), tl.cuda(), words=words)[0]
    loss, s, state = eng.mwer_forward_device(x.cuda(), hyps, hl, risk, used, ll.cuda(), True, lam)
    want_s = eng.score_device(x.cuda(), hyps, hl, ll.cuda(), True)
    assert _same_bits(s[used], want_s[used])
    wl, wg = host_mwer(s, risk, used, lam)
    assert_close(loss, wl, 1e-14, ctx=(words, lam))
    w = torch.linspace(0.5, 2.0, x.size(0), dtype=torch.float64)
    got = eng.mwer_backward_device(x.cuda(), hyps, hl, w.cuda(), state, ll.cuda(), True)
    ref = eng.score_backward_device(x.cuda(), hyps, hl, (wg * w[:, None]).cuda(), ll.cuda(), True)
    assert float(ref.abs().max()) > 1e-6
    assert_close(got, ref, 1e-12, ctx=(words, lam), norm=True)


@pytest.mark.gpu
def test_matches_composed_recipe():
    """INTEGRATION's composed recipe (CTCScore, errors_device, masked softmax, autograd) on c2's own list."""
    from end2end_b200 import CTCScore, MWERLoss
    x, ll, tg, tl, hyps, hl, used = _nbest_case(B=64, N=16)
    eng = engine(0, LABELS)
    xa = x.cuda().requires_grad_()
    s = CTCScore()(xa, hyps, hl, ll.cuda())
    risk = eng.errors_device(hyps, hl, tg.cuda(), tl.cuda(), words=True)[0].double()
    p = torch.softmax(s.masked_fill(~used, float("-inf")), dim=1)
    want = (p * risk).sum()
    want.backward()
    xb = x.cuda().requires_grad_()
    loss = MWERLoss(LABELS, reduce=True)(xb, hyps, hl, ll.cuda(), tg.cuda(), tl.cuda(), used)
    loss.backward()
    assert loss.dtype == torch.float64 and loss.dim() == 0
    assert abs(float(loss.detach()) - float(want.detach())) <= 1e-12 * abs(float(want.detach()))
    assert float(xa.grad.abs().max()) > 1e-4
    assert_close(xb.grad, xa.grad, 1e-10, norm=True)


@pytest.mark.gpu
@pytest.mark.parametrize("from_logits", [False, True])
def test_gradcheck_float64(from_logits):
    from end2end_b200.functions.mwer import MWERFunction
    g = torch.Generator().manual_seed(5)
    B, T, V, N = 2, 7, 5, 4
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64)
    if not from_logits:
        x = torch.log_softmax(x, 2)
    hyps = torch.tensor([[[1, 2], [2, 2], [3, 0], [4, 1]], [[1, 1], [2, 0], [3, 4], [1, 3]]]).cuda()
    hl = torch.tensor([[2, 2, 1, 2], [1, 1, 2, 2]]).cuda()
    mask = torch.tensor([[True, True, False, True], [True, True, True, True]]).cuda()
    risk = torch.tensor([[1.0, 2.0, 0.0, 3.5], [0.0, 1.0, 2.5, 4.0]], dtype=torch.float64).cuda()
    ll = torch.tensor([7, 5]).cuda()
    eng = engine()
    xc = x.cuda().requires_grad_()
    assert torch.autograd.gradcheck(
        lambda t: MWERFunction.apply(eng, t, hyps, hl, ll, risk, mask, 0.7, from_logits, None), (xc,),
        eps=1e-6, atol=1e-8, rtol=1e-6)


@pytest.mark.gpu
def test_masked_slots_change_nothing():
    g = torch.Generator().manual_seed(7)
    x, ll, Lmax, _, _ = _cfg("c1", 4)
    B, T, V = x.shape
    N = 12
    hyps, hl = hyps_for(g, B, N, 10, V)
    risk = torch.randint(0, 6, (B, N), generator=g).double()
    mask = torch.rand(B, N, generator=g) < 0.6
    mask[:, 0] = True
    # garbage in the masked slots: bad lengths and labels, a negative risk
    hb, hlb, rb = hyps.clone(), hl.clone(), risk.clone()
    hb[~mask] = -7
    hlb[~mask] = 99
    rb[~mask] = -1.0
    eng = engine()
    loss, s, st = _forward(eng, x, hb, hlb, rb, mask, ll, True, 1.5)
    grad = _grad(eng, x, hb, hlb, st, torch.ones(B, dtype=torch.float64), ll, True)
    # the compacted list: each utterance's in-mask slots only, padded with masked-out copies of slot 0
    K = int(mask.sum(1).max())
    hc, hlc = torch.zeros(B, K, 10, dtype=torch.int64), torch.zeros(B, K, dtype=torch.int64)
    rc, mc = torch.zeros(B, K, dtype=torch.float64), torch.zeros(B, K, dtype=torch.bool)
    for b in range(B):
        idx = mask[b].nonzero().flatten()
        hc[b, :len(idx)], hlc[b, :len(idx)], rc[b, :len(idx)], mc[b, :len(idx)] = hyps[b, idx], hl[b, idx], risk[b, idx], True
    loss_c, _, st_c = _forward(eng, x, hc, hlc, rc, mc, ll, True, 1.5)
    grad_c = _grad(eng, x, hc, hlc, st_c, torch.ones(B, dtype=torch.float64), ll, True)
    assert_close(loss, loss_c, 1e-13)
    assert_close(grad, grad_c, 1e-13, norm=True)
    assert bool(torch.isfinite(grad).all())


@pytest.mark.gpu
def test_zero_gradient_rules():
    """N = 1, a single in-list slot, equal risks: exactly zero rows; an empty or all-infeasible list: loss 0."""
    g = torch.Generator().manual_seed(9)
    x, ll, _, _, _ = _cfg("c1", 4)
    B, T, V = x.shape
    eng = engine()
    one = torch.ones(B, dtype=torch.float64)
    hyps, hl = hyps_for(g, B, 1, 8, V)
    risk = torch.tensor([[2.0], [0.0], [5.0], [1.0]])
    loss, _, st = _forward(eng, x, hyps, hl, risk, None, ll, True)
    assert torch.equal(loss.cpu(), risk[:, 0].double())
    assert bool((_grad(eng, x, hyps, hl, st, one, ll, True) == 0).all())
    hyps, hl = hyps_for(g, B, 6, 8, V)
    mask = torch.zeros(B, 6, dtype=torch.bool)
    mask[:, 3] = True                                   # a single in-list slot
    risk = torch.arange(B * 6, dtype=torch.float64).reshape(B, 6)
    loss, _, st = _forward(eng, x, hyps, hl, risk, mask, ll, True)
    assert torch.equal(loss.cpu(), risk[:, 3])
    assert bool((_grad(eng, x, hyps, hl, st, one, ll, True) == 0).all())
    risk = torch.full((B, 6), 3.0, dtype=torch.float64)  # equal risks
    loss, _, st = _forward(eng, x, hyps, hl, risk, None, ll, True, 0.5)
    assert bool((loss.cpu() == 3.0).all())
    assert bool((_grad(eng, x, hyps, hl, st, one, ll, True) == 0).all())
    mask[:] = False                                     # empty lists
    risk = torch.rand(B, 6, generator=g, dtype=torch.float64)
    loss, s, st = _forward(eng, x, hyps, hl, risk, mask, ll, True)
    assert bool((loss == 0).all()) and bool((s == float("-inf")).all())
    assert bool((_grad(eng, x, hyps, hl, st, one, ll, True) == 0).all())
    hyps = torch.full((B, 6, 40), 3, dtype=torch.int64)  # 40 repeats in <= 50 frames: every hypothesis infeasible
    hl = torch.full((B, 6), 40, dtype=torch.int64)
    loss, s, st = _forward(eng, x, hyps, hl, risk, None, ll, True)
    assert bool((loss == 0).all()) and bool((s == float("-inf")).all())
    assert bool((_grad(eng, x, hyps, hl, st, one, ll, True) == 0).all())


@pytest.mark.gpu
def test_bad_arguments_are_isolated():
    from end2end_b200 import MWERLoss
    g = torch.Generator().manual_seed(11)
    x, ll, _, tg, tl = _cfg("c1", 4)
    B, T, V = x.shape
    N = 5
    hyps, hl = hyps_for(g, B, N, 8, V)
    hyps = hyps.clamp(min=1)
    risk = torch.rand(B, N, generator=g, dtype=torch.float64)
    eng = engine()
    one = torch.ones(B, dtype=torch.float64)
    base_loss, _, st = _forward(eng, x, hyps, hl, risk, None, ll, True)
    base = _grad(eng, x, hyps, hl, st, one, ll, True)
    cases = []
    h2 = hl.clone(); h2[1, 2] = 99
    cases.append((hyps, h2, risk, ll, 1))
    l2 = ll.clone(); l2[2] = 0
    cases.append((hyps, hl, risk, l2, 2))
    r2 = risk.clone(); r2[3, 1] = -1.0                 # K11's -1 for a bad device-resident reference length
    cases.append((hyps, hl, r2, ll, 3))
    y2 = hyps.clone(); y2[0, 0, 0] = V
    h3 = hl.clone(); h3[0, 0] = max(int(h3[0, 0]), 1)
    cases.append((y2, h3, risk, ll, 0))
    for hy, hh, rr, lll, bad in cases:
        loss, _, st = _forward(eng, x, hy, hh, rr, None, lll, True)
        grad = _grad(eng, x, hy, hh, st, one, lll, True)
        assert bool(torch.isnan(loss[bad])), bad
        rows = grad[bad, :int(lll[bad])] if int(lll[bad]) > 0 else grad[bad]
        assert bool(torch.isnan(rows).all()), bad
        keep = [b for b in range(B) if b != bad and not (bad == 0 and b == 0)]
        if bad != 0:
            assert _same_bits(loss[keep], base_loss[keep]) and _same_bits(grad[keep], base[keep]), bad
        else:                                           # hypothesis (0, 0) changed: only its own utterance differs
            assert _same_bits(loss[1:], base_loss[1:]) and _same_bits(grad[1:], base[1:])
    # device-resident reference length past the reference: the utterance's loss is NaN
    tl2 = tl.clone(); tl2[1] = tg.size(1) + 5
    hypsn, hln = hyps, hl
    loss = MWERLoss(LABELS, level="token")(x.cuda(), hypsn.cuda(), hln.cuda(), ll.cuda(), tg.cuda(), tl2.cuda())
    assert bool(torch.isnan(loss[1])) and bool(torch.isfinite(loss[[0, 2, 3]]).all())
    # host-resident bad lengths raise
    crit = MWERLoss(LABELS, level="token")
    with pytest.raises(ValueError):
        crit(x.cuda(), hyps, h2, ll, tg, tl)
    with pytest.raises(ValueError):
        crit(x.cuda(), hyps, hl, l2, tg, tl)
    with pytest.raises(ValueError):
        crit(x.cuda(), hyps, hl, ll, tg, tl2)
    with pytest.raises(ValueError):
        eng.mwer_forward_device(x.cuda(), hyps.cuda(), hl.cuda(), risk.cuda(), None, ll.cuda(), True, -1.0)
    with pytest.raises(NotImplementedError):
        eng.mwer_forward_device(x.cuda(), torch.zeros(B, N, MAX_TARGETS + 1, dtype=torch.int64).cuda(), hl.cuda(),
                                risk.cuda(), None, ll.cuda(), True)


@pytest.mark.gpu
def test_reductions_and_second_backward():
    from end2end_b200.functions.mwer import MWERFunction
    x, ll, tg, tl, hyps, hl, used = _nbest_case(B=6, N=8)
    eng = engine(0, LABELS)
    risk = eng.errors_device(hyps, hl, tg.cuda(), tl.cuda(), words=True)[0]
    B = x.size(0)

    def run(reduction, upstream):
        xa = x.cuda().requires_grad_()
        loss = MWERFunction.apply(eng, xa, hyps, hl, ll.cuda(), risk, used, 1.3, True, reduction)
        loss.backward(upstream, retain_graph=True)
        first = xa.grad.clone()
        xa.grad = None
        loss.backward(upstream)
        assert _same_bits(xa.grad, first), reduction
        return loss, first

    w = torch.linspace(-1.0, 2.5, B, dtype=torch.float64).cuda()
    per, g_per = run(None, w)
    tot, g_sum = run("sum", torch.tensor(0.75, dtype=torch.float64).cuda())
    mean, g_mean = run("mean", torch.tensor(0.75, dtype=torch.float64).cuda())
    assert abs(float(tot) - float(per.sum())) <= 1e-14 * abs(float(tot))
    assert abs(float(mean) - float(per.mean())) <= 1e-14 * abs(float(mean))
    _, wg = host_mwer(eng.score_device(x.cuda(), hyps, hl, ll.cuda(), True), risk, used, 1.3)
    for got, scale in ((g_per, w.cpu()), (g_sum, torch.full((B,), 0.75, dtype=torch.float64)),
                       (g_mean, torch.full((B,), 0.75 / B, dtype=torch.float64))):
        ref = eng.score_backward_device(x.cuda(), hyps, hl, (wg * scale[:, None]).cuda(), ll.cuda(), True)
        assert_close(got, ref, 1e-12, norm=True)
    with torch.no_grad():
        out = MWERFunction.apply(eng, x.cuda(), hyps, hl, ll.cuda(), risk, used, 1.3, True, None)
    assert _same_bits(out, per.detach())


@pytest.mark.gpu
def test_layouts_indices_and_host_input():
    from end2end_b200 import MWERLoss
    x, ll, tg, tl, hyps, hl, used = _nbest_case(B=5, N=6)
    crit = MWERLoss(LABELS)

    def grad_of(xx, hh, hll, lls, tgg, tll, mm, c=crit):
        xx = xx.detach().clone().requires_grad_()
        loss = c(xx, hh, hll, lls, tgg, tll, mm)
        loss.sum().backward()
        return loss.detach().cpu(), xx.grad.cpu()

    base = grad_of(x.cuda(), hyps, hl, ll.cuda(), tg.cuda(), tl.cuda(), used)
    assert float(base[1].abs().max()) > 0
    variants = [
        grad_of(x.cuda(), hyps.int(), hl.int(), ll.cuda().int(), tg.cuda().int(), tl.cuda().int(), used),
        grad_of(x, hyps.cpu(), hl.cpu(), ll, tg, tl, used.cpu()),
    ]
    xt = x.cuda().transpose(0, 1).contiguous()            # time-major storage
    lt, gt = grad_of(xt, hyps, hl, ll.cuda(), tg.cuda(), tl.cuda(), used, MWERLoss(LABELS, time_major=True))
    variants.append((lt, gt.transpose(0, 1)))
    wide = torch.zeros(x.size(0), x.size(1), x.size(2) + 3, dtype=x.dtype)
    wide[:, :, :x.size(2)] = x
    wide = wide.cuda().requires_grad_()                  # a strided view: row stride V + 3
    lw = crit(wide[:, :, :x.size(2)], hyps, hl, ll.cuda(), tg.cuda(), tl.cuda(), used)
    lw.sum().backward()
    assert bool((wide.grad[:, :, x.size(2):] == 0).all())
    variants.append((lw.detach().cpu(), wide.grad[:, :, :x.size(2)].cpu()))
    for i, (l, gr) in enumerate(variants):
        assert _same_bits(l, base[0]) and _same_bits(gr, base[1]), i
    # repeatability and utterance permutations
    again = grad_of(x.cuda(), hyps, hl, ll.cuda(), tg.cuda(), tl.cuda(), used)
    assert _same_bits(again[0], base[0]) and _same_bits(again[1], base[1])
    perm = torch.tensor([3, 0, 4, 2, 1])
    pl, pg = grad_of(x[perm].cuda(), hyps[perm.cuda()], hl[perm.cuda()], ll[perm].cuda(), tg[perm].cuda(), tl[perm].cuda(),
                     used[perm.cuda()])
    assert _same_bits(pl, base[0][perm]) and _same_bits(pg, base[1][perm])


@pytest.mark.gpu
def test_cuda_graph_capture():
    x, ll, tg, tl, hyps, hl, used = _nbest_case(B=6, N=8)
    eng = engine(0, LABELS)
    xc, llc = x.cuda(), ll.cuda()
    risk = eng.errors_device(hyps, hl, tg.cuda(), tl.cuda(), words=True)[0].double()
    w = torch.linspace(0.5, 1.5, x.size(0), dtype=torch.float64).cuda()

    def step():
        loss, _, st = eng.mwer_forward_device(xc, hyps, hl, risk, used, llc, True, 1.0)
        return loss, eng.mwer_backward_device(xc, hyps, hl, w, st, llc, True)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        want = step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        got = step()
    graph.replay()
    torch.cuda.synchronize()
    assert _same_bits(got[0], want[0]) and _same_bits(got[1], want[1])
    graph.replay()
    torch.cuda.synchronize()
    assert _same_bits(got[1], want[1])


@pytest.mark.gpu
def test_cuda_graph_capture_module():
    """The public path captured whole: MWERLoss's forward (errors_device, K12a, K12b) and its backward through autograd
    (K12c and the row kernel) replay to the bits of the eager step."""
    from end2end_b200 import MWERLoss
    x, ll, tg, tl, hyps, hl, used = _nbest_case(B=6, N=8)
    crit = MWERLoss(LABELS, reduce=True, size_average=True)
    llc, tgc, tlc = ll.cuda(), tg.cuda(), tl.cuda()
    eager = x.cuda().requires_grad_()
    want_loss = crit(eager, hyps, hl, llc, tgc, tlc, used)
    want_loss.backward()
    static = x.cuda().requires_grad_()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            static.grad = None
            crit(static, hyps, hl, llc, tgc, tlc, used).backward()
    torch.cuda.current_stream().wait_stream(side)
    static.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = crit(static, hyps, hl, llc, tgc, tlc, used)
        loss.backward()
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert _same_bits(loss.detach(), want_loss.detach()) and _same_bits(static.grad, eager.grad)

"""The gradient of the N-hypothesis CTC score (CTCScore, CTCScoreFunction, CTCBeamEngine.score_backward_device,
e2e_ctc_score_backward_device).

For upstream weights g[b, n] the gradient is sum_n g[b, n] gamma_bn(t, v) on log-probabilities and
sum_n g[b, n] (gamma_bn(t, v) - softmax(x_bt)_v) on raw logits, 0 past the utterance's frames.  The oracle's gamma is
exp(lp) - grad of oracle.PortEngine (the C restatement of the reference's loss) on each (utterance, hypothesis) pair.
The reference's beta decides the skip edge s -> s + 2 by the source label and its alpha by the target label; the two
differ only for a label equal to the blank next to a different label, where this gradient follows the score (the
derivative, checked with gradcheck) and the oracle comparisons keep blank-valued labels in runs of their own.
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import oracle

H = 8                                      # hypotheses per CTA (ctc_score.cu: kScoreWarps)
MAX_TARGETS = 639
K_BOUNDARIES = (15, 63, 64, 127, 128, 255, 256, 638, 639)


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
    """ctc_score.cu: score_mode with K10's extra shared memory -- the staged block, hence the checkpoint spacing."""
    Lp = Lmax + 1
    head = _a(H * Lp * 4, 16) + 2 * 32 * 8 + _a(H * Lp * 4, 16) + H * 16
    row = V * 8
    fb = min(32, max(8, 64 * 1024 // row))
    if head + fb * row <= 160 * 1024:
        return fb
    return min(32, (160 * 1024 - head) // (H * Lp * 8))


def workspace_bytes(B, T, V, Lmax, N):
    G, Kc, FB = (N + H - 1) // H, (2 * Lmax + 1 + 31) // 32, frames_per_block(V, Lmax)
    nblk = (T + FB - 1) // FB
    return (_a(B * G * 8, 256) + _a(B * G * 4, 256) + _a(B * N * nblk * Kc * 256, 256) + _a(B * N * FB * Kc * 256, 256)
            + _a(B * G * T * V * 8, 256))


def engine(blank=0):
    from end2end_b200.engine import CTCBeamEngine
    return CTCBeamEngine(blank, 1)


def hyps_for(g, B, N, Lmax, V, blank, lmin=0):
    """Mixed lengths in every CTA (0, 1, Lmax, random), runs of repeated labels, and blank-valued labels in runs that fill
    a hypothesis (where the reference's lattice is the score's)."""
    others = torch.tensor([v for v in range(V) if v != blank])
    hl = torch.randint(lmin, Lmax + 1, (B, N), generator=g)
    fixed = torch.tensor([0, 1, Lmax, max(Lmax - 1, 0)])
    hl[:, :min(N, 4)] = fixed[:min(N, 4)].clamp(min=lmin, max=Lmax)
    hyps = others[torch.randint(0, len(others), (B, N, max(Lmax, 1)), generator=g)][:, :, :Lmax].clone()
    if Lmax > 1:
        rep = torch.rand(B, N, Lmax, generator=g) < 0.3
        rep[:, :, 0] = False
        for k in range(1, Lmax):
            hyps[:, :, k] = torch.where(rep[:, :, k], hyps[:, :, k - 1], hyps[:, :, k])
    if N > 4 and Lmax > 0:
        hyps[:, 4] = blank
        hl[:, 4] = hl[:, 4].clamp(max=3)
    return hyps, hl


def oracle_gamma(lp, hyps, hl, ll, blank):
    """gamma [B, N, T, V] float64 (0 past T_b) and feasibility [B, N] from oracle.PortEngine."""
    lp = lp.detach().cpu().double()
    B, N = hl.shape
    T, V = lp.shape[1:]
    eng = oracle.PortEngine(blank)
    gam = torch.zeros(B, N, T, V, dtype=torch.float64)
    feas = torch.zeros(B, N, dtype=torch.bool)
    for b in range(B):
        tg = hyps[b].cpu().long() if hyps.size(2) > 0 else torch.zeros(N, 0, dtype=torch.int64)
        loss, grad = eng.compute(lp[b:b + 1].expand(N, -1, -1).contiguous(), tg, ll[b:b + 1].cpu().expand(N),
                                 hl[b].cpu().long())
        Tb = int(ll[b])
        feas[b] = torch.isfinite(loss)
        gam[b, :, :Tb] = torch.exp(lp[b, :Tb]).unsqueeze(0) - grad[:, :Tb].double()
    return gam, feas


def expected(gam, feas, g, sm=None, ll=None):
    w = torch.where(feas, g.cpu(), torch.zeros_like(g.cpu()))
    out = torch.einsum("bn,bntv->btv", w, torch.where(feas[:, :, None, None], gam, torch.zeros_like(gam)))
    if sm is not None:
        T = sm.size(1)
        live = (torch.arange(T)[None, :] < ll.cpu()[:, None]).double()
        out = out - w.sum(1)[:, None, None] * sm.cpu() * live[:, :, None]
    return out


def assert_close(got, want, scale=1.0, rtol=1e-10, atol=1e-12, ctx=None):
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    err = (got - want).abs()
    bound = rtol * want.abs() + atol * max(1.0, scale)
    assert bool((err <= bound).all()), (ctx, float(err.max()), float((err - bound).max()))


def weights(g, B, N):
    w = torch.randn(B, N, generator=g, dtype=torch.float64)
    w[torch.rand(B, N, generator=g) < 0.25] = 0.0
    return w


# ---------------------------------------------------------------------------------------------- device-free ---------

def test_score_backward_workspace_query(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    lim = _lib.limits()
    for (B, T, V, Lmax) in ((4, 50, 29, 0), (4, 50, 29, 200), (3, 70, 1024, 80), (2, 70, 4096, 30), (2, 9, 29, MAX_TARGETS),
                            (1, 5, lim.max_alphabet, MAX_TARGETS)):
        for N in (1, H, H + 1, 100):
            n = L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(B, T, V, Lmax)), N)
            assert n == workspace_bytes(B, T, V, Lmax, N), (B, T, V, Lmax, N, n)
    assert L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(4, 50, 29, MAX_TARGETS + 1)), 1) == 0
    assert "target length 640" in L.e2e_last_error_string().decode()
    assert L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(4, 50, lim.max_alphabet + 1, 10)), 1) == 0
    assert "alphabet %d" % (lim.max_alphabet + 1) in L.e2e_last_error_string().decode()
    for n_hyp in (0, -1):
        assert L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(4, 50, 29, 10)), n_hyp) == 0
        assert "n_hyp %d" % n_hyp in L.e2e_last_error_string().decode()
    # B x T rows of the row kernel past 2^31 - 1 CTAs of eight warps
    assert L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(2 ** 31 - 1, 16, 29, 10)), 1) == 0
    assert "exceeds the grid" in L.e2e_last_error_string().decode()
    # K10's grid, B x ceil(N / 8) CTAs, never exceeds B x N, which the scorer's check bounds by 2^31 - 1 first
    assert L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(2 ** 28, 16, 29, 10)), 64) == 0
    assert "exceed this build's limit" in L.e2e_last_error_string().decode()
    # 2^28 groups x 2^31 frames x 32768 symbols of partial rows
    assert L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(_desc(1, 2 ** 31 - 1, lim.max_alphabet, 4)), 2 ** 31 - 1) == 0
    assert "overflows" in L.e2e_last_error_string().decode()


def test_score_backward_argument_errors(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    d = _desc(2, 10, 5, 3)
    need = L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(d), 2)
    fake = ctypes.c_void_p(256)              # never dereferenced: every case fails before a launch
    ok_args = [fake, fake, None, fake, fake, fake, fake, need, None]

    def call(desc, n_hyp, args):
        return L.e2e_ctc_score_backward_device(ctypes.byref(desc) if desc is not None else None, n_hyp, *args)

    assert call(None, 2, ok_args) == 1
    assert call(d, 0, ok_args) == 1 and "n_hyp 0" in L.e2e_last_error_string().decode()
    for i in (0, 1, 3, 4, 5):                # logits, hyps, hyp_lengths, grad_scores, grads
        args = list(ok_args)
        args[i] = None
        assert call(d, 2, args) == 1 and "null pointer" in L.e2e_last_error_string().decode(), i
    args = list(ok_args)
    args[6] = None                           # null workspace
    assert call(d, 2, args) == 3 and "workspace" in L.e2e_last_error_string().decode()
    args = list(ok_args)
    args[7] = need - 1                       # short workspace
    assert call(d, 2, args) == 3 and "too small" in L.e2e_last_error_string().decode()
    args = list(ok_args)
    args[6] = ctypes.c_void_p(255 + 256)     # misaligned workspace
    assert call(d, 2, args) == 3
    bad = _desc(2, 10, 5, 3)
    bad.grads_stride_t = -1
    assert call(bad, 2, ok_args) == 1 and "gradient stride" in L.e2e_last_error_string().decode()
    assert call(_desc(2, 10, 5, MAX_TARGETS + 1), 1, ok_args) == 2


# ---------------------------------------------------------------------------------------------- GPU -----------------

def _cfg(name, B):
    Bc, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS[name]
    x, _, ll, _ = oracle.make_inputs(min(Bc, B), T, V, Lmin, Lmax, seed, full_length=full)
    return x.double(), ll, Lmax


def _check_oracle(x, hyps, hl, ll, blank, g, ctx):
    """Both input kinds against the oracle: log-probs log_softmax(x), and x itself as raw logits."""
    lp = torch.log_softmax(x, 2)
    gam, feas = oracle_gamma(lp, hyps, hl, ll, blank)
    eng = engine(blank)
    scale = float(g.abs().sum(1).max())
    got = eng.score_backward_device(lp.cuda(), hyps.cuda(), hl.cuda(), g.cuda(), ll.cuda())
    assert got.dtype == torch.float64 and got.shape == x.shape
    assert_close(got, expected(gam, feas, g), scale, ctx=ctx)
    got = eng.score_backward_device(x.cuda(), hyps.cuda(), hl.cuda(), g.cuda(), ll.cuda(), from_logits=True)
    assert_close(got, expected(gam, feas, g, torch.exp(lp), ll), scale, ctx=(ctx, "logits"))
    return feas


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
@pytest.mark.parametrize("N", [1, 3, H - 1, H, H + 1, 100])
def test_oracle_parity_configs(name, N):
    """c1-c4 shapes (a few utterances each), N in {1, 3, 7, 8, 9, 100}, blank 0 / 3 / V - 1, T_b in {T, 1, 2}, random g
    with zeros, repeats, blank-valued runs and infeasible hypotheses."""
    B = 3
    if name == "c4" and N == 100:
        N, B = 2 * H + 3, 2                  # the oracle's replicated gradient at V = 1024: 2 MB per hypothesis
    x, ll, Lmax = _cfg(name, B)
    B, T, V = x.shape
    g = torch.Generator().manual_seed(2000 + N)
    for blank in (0, 3, V - 1):
        hyps, hl = hyps_for(g, B, N, Lmax, V, blank)
        ll2 = ll.clone()
        ll2[0] = T
        if B > 2:
            ll2[1], ll2[2] = 1, 2
        feas = _check_oracle(x, hyps, hl, ll2, blank, weights(g, B, N), (name, N, blank))
        if N >= 3 and B > 2:
            assert not bool(feas[1].all())   # T_b = 1: infeasible hypotheses with nonzero weight are in the batch


@pytest.mark.gpu
@pytest.mark.parametrize("Lmax", K_BOUNDARIES)
def test_oracle_parity_k_variants(Lmax):
    """Every cells-per-lane variant at and next to its width boundary; lengths 0 / 1 / Lmax in one CTA, a full-length
    hypothesis that just fits, T_b in {T, 1, 2, Lmax + 1}."""
    g = torch.Generator().manual_seed(Lmax)
    B, V = 4, 29
    T = 2 * Lmax + 2
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64) * 2.0
    ll = torch.tensor([T, 1, 2, Lmax + 1])
    hyps, hl = hyps_for(g, B, H + 1, Lmax, V, 0)
    hl[:, 5] = Lmax
    hyps[:, 5] = torch.arange(Lmax) % (V - 1) + 1            # no repeats: feasible in Lmax + 1 frames
    feas = _check_oracle(x, hyps, hl, ll, 0, weights(g, B, H + 1), Lmax)
    assert bool(feas[3, 5]) and bool(feas[0, 5])


@pytest.mark.gpu
@pytest.mark.parametrize("V,blank", [(4096, 0), (4096, 4095), (3000, 7)])
def test_oracle_parity_gathered_columns(V, blank):
    """Alphabets whose row block does not fit shared memory: the CTA gathers each hypothesis's columns and the blank."""
    g = torch.Generator().manual_seed(V + blank)
    B, T, Lmax, N = 2, 70, 30, H + 3
    assert frames_per_block(V, Lmax) < 32 or V * 8 * 8 > 64 * 1024
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64) * 3.0
    hyps, hl = hyps_for(g, B, N, Lmax, V, blank)
    _check_oracle(x, hyps, hl, torch.tensor([T, 41]), blank, weights(g, B, N), (V, blank))


@pytest.mark.gpu
@pytest.mark.parametrize("V", [29, 1024])
def test_oracle_parity_checkpoint_boundaries(V):
    """Utterance lengths that put a staged-block (checkpoint) boundary on, before and after the last frame."""
    g = torch.Generator().manual_seed(V)
    Lmax, N = 20, H + 2
    FB = frames_per_block(V, Lmax)
    lens = [FB - 1, FB, FB + 1, 2 * FB - 1, 2 * FB, 2 * FB + 1]
    T = max(lens) + 3
    x = torch.randn(len(lens), T, V, generator=g, dtype=torch.float64) * 2.0
    hyps, hl = hyps_for(g, len(lens), N, Lmax, V, 0)
    _check_oracle(x, hyps, hl, torch.tensor(lens), 0, weights(g, len(lens), N), (V, FB))


@pytest.mark.gpu
@pytest.mark.parametrize("from_logits", [False, True])
def test_gradcheck_float64(from_logits):
    """torch.autograd.gradcheck of CTCScore in float64 -- a label equal to the blank next to other labels included, where
    the reference's beta is not the score's and this gradient follows the score."""
    from end2end_b200 import CTCScore
    g = torch.Generator().manual_seed(11 + from_logits)
    B, T, V, N, blank = 2, 7, 5, 4, 1
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64)
    if not from_logits:
        x = torch.log_softmax(x, 2)              # gradcheck perturbs log-probs freely: the score is still defined
    hyps = torch.tensor([[[2, 2, 3], [1, 4, 0], [3, 1, 1], [4, 0, 2]],
                         [[0, 1, 2], [2, 3, 4], [1, 0, 0], [4, 4, 0]]])
    hl = torch.tensor([[3, 3, 2, 2], [3, 3, 3, 0]])
    ll = torch.tensor([7, 5])
    mod = CTCScore(blank_idx=blank, after_logsoftmax=not from_logits)
    xc = x.cuda().requires_grad_()
    assert torch.autograd.gradcheck(lambda t: mod(t, hyps.cuda(), hl.cuda(), ll.cuda()), (xc,), eps=1e-6, atol=1e-7,
                                    rtol=1e-6)


def _no_blank_hyps(g, B, N, Lmax, V, lmin=1):
    hl = torch.randint(lmin, Lmax + 1, (B, N), generator=g)
    hyps = torch.randint(1, V, (B, N, Lmax), generator=g)
    return hyps, hl


@pytest.mark.gpu
def test_matches_torch_ctc_loss_replicated():
    """fp32 raw logits: torch's ctc_loss(reduction='none') on the replicated input, backpropagated through the same fp32
    log_softmax and summed with weights -g, within 1e-5 per unit of sum_n |g|.  Torch's lattice runs in fp64 on the fp32
    log-probabilities, as K10's does (in fp32 its log-space sums drift by ~1e-5 per hypothesis at these lengths)."""
    from end2end_b200 import CTCScore
    g = torch.Generator().manual_seed(5)
    B, T, V, N, Lmax = 3, 60, 30, H + 3, 12
    x = torch.randn(B, T, V, generator=g) * 2.0
    ll = torch.tensor([60, 45, 33])
    hyps, hl = _no_blank_hyps(g, B, N, Lmax, V)
    w = weights(g, B, N)
    xc = x.cuda().requires_grad_()
    s = CTCScore()(xc, hyps.cuda(), hl.cuda(), ll.cuda())
    (s * w.cuda()).sum().backward()
    xr = x.cuda().repeat_interleave(N, 0).requires_grad_()
    losses = F.ctc_loss(F.log_softmax(xr, 2).double().transpose(0, 1), hyps.reshape(B * N, Lmax).cuda(),
                        ll.repeat_interleave(N).cuda(), hl.reshape(-1).cuda(), blank=0, reduction="none")
    assert torch.allclose(-losses.double().cpu().reshape(B, N), s.detach().cpu(), rtol=1e-5, atol=1e-4)
    (losses * (-w.reshape(-1)).cuda()).sum().backward()
    want = xr.grad.reshape(B, N, T, V).sum(1)
    assert_close(xc.grad, want, float(w.abs().sum(1).max()), rtol=1e-5, atol=1e-5, ctx="ctc_loss")


@pytest.mark.gpu
def test_n1_matches_ctc_loss_module():
    """N = 1 with g = -1 is the loss's gradient: CTCLoss(after_logsoftmax=False, reduce=False) on fp64 raw logits, within
    the loss's own tolerance against the oracle (1e-5; its linear-domain kernels differ from the log domain by ~1e-7)."""
    from end2end_b200 import CTCLoss, CTCScore
    x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    x = x[:8].double()
    tg, ll, tl = tg[:8], ll[:8], tl[:8]
    xa = x.cuda().requires_grad_()
    CTCLoss(after_logsoftmax=False, reduce=False)(xa, tg.cuda(), ll.cuda(), tl.cuda()).sum().backward()
    xb = x.cuda().requires_grad_()
    s = CTCScore()(xb, tg[:, None].cuda(), tl[:, None].cuda(), ll.cuda())
    (-s).sum().backward()
    live = (torch.arange(x.size(1))[None, :] < ll[:, None]).cuda()[:, :, None]
    assert_close(xb.grad, torch.where(live, xa.grad, torch.zeros_like(xa.grad)), rtol=1e-5, atol=1e-5, ctx="CTCLoss")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_16bit_inputs(dtype):
    """16-bit raw logits: within one ulp of the stored type of the f64 result on the same rounded log-probs (the rule of
    test_gpu_score.py: torch's device log-softmax, rounded to the input dtype)."""
    g = torch.Generator().manual_seed(17)
    B, T, V, N, Lmax = 3, 50, 40, H + 2, 15
    xh = (torch.randn(B, T, V, generator=g) * 2.5).to(dtype).cuda()
    ll = torch.tensor([50, 30, 2]).cuda()
    hyps, hl = hyps_for(g, B, N, Lmax, V, 0)
    w = weights(g, B, N).cuda()
    eng = engine(0)
    got = eng.score_backward_device(xh, hyps.cuda(), hl.cuda(), w, ll, from_logits=True)
    assert got.dtype == dtype
    lph = F.log_softmax(xh, 2).double()
    gam = eng.score_backward_device(lph, hyps.cuda(), hl.cuda(), w, ll)          # sum_n g gamma on the rounded lp
    fin = torch.isfinite(eng.score_device(lph, hyps.cuda(), hl.cuda(), ll))
    c = torch.where(fin, w, torch.zeros_like(w)).sum(1)
    live = (torch.arange(T, device="cuda")[None, :] < ll[:, None])[:, :, None]
    want = torch.where(live, gam - c[:, None, None] * torch.exp(lph), torch.zeros_like(gam))
    ulp = 2.0 ** -7 if dtype == torch.bfloat16 else 2.0 ** -10
    tiny = torch.finfo(dtype).tiny
    assert bool(((got.double() - want).abs() <= ulp * want.abs() + tiny).all())
    # the forward: score_device's values bit for bit
    from end2end_b200 import CTCScore
    assert torch.equal(CTCScore()(xh, hyps.cuda(), hl.cuda(), ll), eng.score_device(xh, hyps.cuda(), hl.cuda(), ll,
                                                                                   from_logits=True))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("after_logsoftmax", [False, True])
def test_forward_is_score_device(dtype, after_logsoftmax):
    from end2end_b200 import CTCScore
    g = torch.Generator().manual_seed(3)
    B, T, V, N, Lmax = 3, 40, 29, H + 1, 14
    x = torch.randn(B, T, V, generator=g)
    if after_logsoftmax:
        x = torch.log_softmax(x, 2)
    x = x.to(dtype).cuda()
    hyps, hl = hyps_for(g, B, N, Lmax, V, 0)
    ll = torch.tensor([40, 20, 3]).cuda()
    got = CTCScore(after_logsoftmax=after_logsoftmax)(x, hyps.cuda(), hl.cuda(), ll)
    assert got.dtype == torch.float64 and got.device == x.device
    assert torch.equal(got, engine(0).score_device(x, hyps.cuda(), hl.cuda(), ll, from_logits=not after_logsoftmax))


@pytest.mark.gpu
def test_skips_nan_rows_padding_and_determinism():
    g = torch.Generator().manual_seed(23)
    B, T, V, N, Lmax = 3, 60, 29, 2 * H + 3, 20
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64).cuda()
    ll = torch.tensor([60, 41, 30]).cuda()
    hyps, hl = hyps_for(g, B, N, Lmax, V, 0, lmin=1)
    hyps, hl = hyps.cuda(), hl.cuda()
    w = weights(g, B, N).cuda()
    w[0, 3] = 1.5
    eng = engine(0)
    run = lambda hh, ln, ww, lls=ll: eng.score_backward_device(x, hh, ln, ww, lls, from_logits=True)   # noqa: E731
    g0 = run(hyps, hl, w)
    assert torch.equal(g0, run(hyps, hl, w))                                      # bitwise reproducible
    assert bool((g0[1, 41:] == 0).all()) and bool((g0[2, 30:] == 0).all())         # padding frames
    # a zero weight skips the hypothesis, whatever it holds
    z = w.clone()
    z[0, 3] = 0.0
    h2 = hyps.clone()
    h2[0, 3] = (h2[0, 3] + 1) % V
    assert torch.equal(run(hyps, hl, z), run(h2, hl, z))
    # an infeasible hypothesis with a nonzero weight changes nothing
    inf_h, inf_l = hyps.clone(), hl.clone()
    inf_l[2, 6] = Lmax
    inf_h[2, 6] = 5                                                               # 20 repeats: 39 frames > 30
    assert bool(torch.isneginf(eng.score_device(x, inf_h, inf_l, ll, from_logits=True)[2, 6]))
    zw = w.clone()
    zw[2, 6] = 0.0
    w6 = w.clone()
    w6[2, 6] = 2.0
    assert torch.equal(run(inf_h, inf_l, w6), run(inf_h, inf_l, zw))
    # a device-resident bad length or label: NaN rows for that utterance only
    bad_h, bad_l = hyps.clone(), hl.clone()
    bad_l[1, 2] = Lmax + 1
    g1 = run(bad_h, bad_l, w)
    assert bool(torch.isnan(g1[1, :41]).all()) and bool((g1[1, 41:] == 0).all())
    assert torch.equal(g1[[0, 2]], g0[[0, 2]])
    bad_h[0, 9, 0] = V
    g2 = run(bad_h, hl, w)
    assert bool(torch.isnan(g2[0]).all()) and torch.equal(g2[1:], g0[1:])
    ll_bad = ll.clone()
    ll_bad[2] = T + 1
    g3 = run(hyps, hl, w, ll_bad)
    assert bool(torch.isnan(g3[2]).all()) and torch.equal(g3[:2], g0[:2])


@pytest.mark.gpu
def test_layouts_indices_and_host_input():
    """Time-major and strided views (gradient in the input's layout), int32 / int64 indices, missing lengths, CPU logits."""
    from end2end_b200 import CTCScore
    g = torch.Generator().manual_seed(29)
    B, T, V, N, Lmax, blank = 3, 50, 31, H + 2, 16, 3
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64)
    ll = torch.tensor([50, 33, 12])
    hyps, hl = hyps_for(g, B, N, Lmax, V, blank)
    w = weights(g, B, N)
    mod = CTCScore(blank_idx=blank)

    def grad_of(xx, hh, ln, lls, m=mod):
        xx = xx.detach().requires_grad_()
        (m(xx, hh, ln, lls) * w.to(xx.device)).sum().backward()
        return xx.grad

    base = grad_of(x.cuda(), hyps.cuda(), hl.cuda(), ll.cuda())
    assert torch.equal(grad_of(x.cuda(), hyps.int().cuda(), hl.int().cuda(), ll.int().cuda()), base)
    host = grad_of(x, hyps, hl, ll)
    assert host.device.type == "cpu" and torch.equal(host, base.cpu())
    wide = torch.randn(B, T, V + 5, generator=g, dtype=torch.float64)
    wide[:, :, :V] = x
    assert torch.equal(grad_of(wide.cuda()[:, :, :V], hyps.cuda(), hl.cuda(), ll.cuda()), base)
    tm = x.transpose(0, 1).contiguous().cuda()
    gt = grad_of(tm, hyps.cuda(), hl.cuda(), ll.cuda(), CTCScore(blank_idx=blank, time_major=True))
    assert torch.equal(gt.transpose(0, 1), base)
    direct = engine(blank).score_backward_device(tm.transpose(0, 1), hyps.cuda(), hl.cuda(), w.cuda(), ll.cuda(),
                                                 from_logits=True)
    assert direct.stride() == tm.transpose(0, 1).stride() and torch.equal(direct, base)
    full = grad_of(x.cuda(), hyps.cuda(), hl.cuda(), None)
    assert torch.equal(full, grad_of(x.cuda(), hyps.cuda(), hl.cuda(), torch.full((B,), T).cuda()))


@pytest.mark.gpu
def test_python_errors_before_device_work():
    from end2end_b200 import _lib
    eng = engine(0)
    x = torch.randn(2, 10, 5).cuda()
    hyps = torch.ones(2, 3, 4, dtype=torch.int64)
    hl = torch.full((2, 3), 2)
    w = torch.ones(2, 3, dtype=torch.float64)
    eng.score_backward_device(x, hyps, hl, w)
    before = _lib.launch_count()
    for exc, args in ((ValueError, (x, hyps, hl, w[:, :2])), (ValueError, (x, hyps, torch.full((2, 3), 5), w)),
                      (NotImplementedError, (x, torch.ones(2, 3, MAX_TARGETS + 1, dtype=torch.int64), hl, w))):
        with pytest.raises(exc):
            eng.score_backward_device(*args)
    assert _lib.launch_count() == before


def mwer_objective(s, used, risk):
    """INTEGRATION.md's MWER example, line for line: the expected risk over the list, unused slots masked."""
    p = torch.softmax(s.masked_fill(~used, float("-inf")), dim=1)
    return (p * risk).sum()


@pytest.mark.gpu
def test_mwer_step_matches_replicated_ctc_loss():
    """decode_nbest -> CTCScore -> the documented MWER objective -> backward, against the same objective on torch's
    ctc_loss over the replicated logits; the step moves the logits (a nonzero gradient)."""
    from end2end_b200 import CTCDecoder, CTCScore
    x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS["c1"][:6])
    x = x.double()
    B, T, V = x.shape
    N = 10
    nb = CTCDecoder(beam_width=N).decode_nbest(x.cuda(), ll, n_best=N)
    hyps, hl = nb.decoded_targets, nb.decoded_targets_lengths
    used = (nb.scores > -float("inf")).cuda()
    g = torch.Generator().manual_seed(31)
    risk = torch.rand(B, N, generator=g, dtype=torch.float64).cuda()      # stands in for each hypothesis's word errors

    xa = x.cuda().requires_grad_()
    mwer_objective(CTCScore()(xa, hyps.cuda(), hl.cuda(), ll.cuda()), used, risk).backward()
    assert float(xa.grad.abs().max()) > 1e-3
    hl0 = torch.where((hl == 1) & (hyps[:, :, 0] == -1), torch.zeros_like(hl), hl)
    Lw = max(hyps.size(2), 1)
    tgt = torch.zeros(B, N, Lw, dtype=torch.int64)
    tgt[:, :, :hyps.size(2)] = hyps.clamp(min=0)
    xr = x.cuda().repeat_interleave(N, 0).requires_grad_()
    losses = F.ctc_loss(F.log_softmax(xr, 2).transpose(0, 1), tgt.reshape(B * N, Lw).cuda(), ll.repeat_interleave(N).cuda(),
                        hl0.reshape(-1).cuda(), blank=0, reduction="none")
    mwer_objective(-losses.reshape(B, N), used, risk).backward()
    want = xr.grad.reshape(B, N, T, V).sum(1)
    assert_close(xa.grad, want, rtol=1e-7, atol=1e-9, ctx="mwer")

"""The CTC log-likelihood of N hypotheses per utterance (CTCDecoder.score, CTCBeamEngine.score_device,
e2e_ctc_score_device).

score[b, n] is minus the CTC loss of utterance b with hypothesis n as its target.  The checker is oracle.PortEngine, the
C restatement of the reference's loss, run on each utterance's fp64 log-probabilities replicated once per hypothesis.
The kernel's fp64 exp / log are CUDA's (within one ulp), the oracle's the C library's, so scores agree to a few ulps
per frame: the tolerance is 1e-11 relative.
"""
import ctypes
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle

H = 8                                      # hypotheses per CTA (ctc_score.cu: kScoreWarps)
TOL = 1e-11
MAX_TARGETS = 639
# ctc_score.cu: K cells per lane by max_targets; these Lmax sit at and next to each variant's width boundary
K_BOUNDARIES = (15, 63, 64, 127, 128, 255, 256, 638, 639)
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_LOSS = ("c1", "c2_b4", "c2_b4_peaky", "c4_b2", "edge_blank0", "edge_blank3")


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


def oracle_scores(lp, hyps, hl, ll, blank):
    """-loss of every (utterance, hypothesis) pair through oracle.PortEngine: lp [B, T, V] (widened to fp64), hyps
    [B, N, Lmax], hl [B, N], ll [B].  Returns [B, N] float64."""
    lp = lp.detach().cpu().to(torch.float64)
    B, N = hl.shape
    Lmax = hyps.size(2)
    out = torch.empty(B, N, dtype=torch.float64)
    eng = oracle.PortEngine(blank)
    for b in range(B):
        tg = hyps[b].cpu().to(torch.int64) if Lmax > 0 else torch.zeros(N, 0, dtype=torch.int64)
        loss, _ = eng.compute(lp[b:b + 1].expand(N, -1, -1), tg, ll[b:b + 1].cpu().expand(N),
                              hl[b].cpu().to(torch.int64))
        out[b] = -loss
    return out


def assert_scores(got, want, rtol=TOL, ctx=None):
    got, want = got.cpu(), want.cpu()
    fin = torch.isfinite(want)
    assert torch.equal(fin, torch.isfinite(got)), (ctx, got[fin != torch.isfinite(got)], want[fin != torch.isfinite(got)])
    assert torch.equal(got[~fin], want[~fin]), ctx
    err = (got[fin] - want[fin]).abs()
    bound = rtol * want[fin].abs().clamp(min=1.0)
    assert bool((err <= bound).all()), (ctx, float(err.max()) if err.numel() else 0.0)


def random_hyps(g, B, N, Lmax, V, blank):
    """Mixed lengths inside every CTA: 0, 1, Lmax and random; runs of repeated labels; blank-valued labels; lengths past
    what the frames allow (infeasible)."""
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


def score(lp, hyps, hl, ll=None, blank=0, from_logits=False):
    from end2end_b200.engine import CTCBeamEngine
    return CTCBeamEngine(blank, 1).score_device(lp, hyps, hl, ll, from_logits=from_logits)


# ---------------------------------------------------------------------------------------------- device-free ---------

def test_score_workspace_query_limits(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    lim = _lib.limits()
    assert lim.max_targets == MAX_TARGETS
    for V, Lmax in ((29, 0), (29, 200), (1024, 80), (29, MAX_TARGETS), (lim.max_alphabet, MAX_TARGETS)):
        for n_hyp in (1, H, 100):
            n = L.e2e_ctc_score_workspace_bytes(ctypes.byref(_desc(4, 50, V, Lmax)), n_hyp)
            assert n == 256, (V, Lmax, n_hyp)
    assert L.e2e_ctc_score_workspace_bytes(ctypes.byref(_desc(4, 50, 29, MAX_TARGETS + 1)), 1) == 0
    assert "target length 640" in L.e2e_last_error_string().decode()
    assert L.e2e_ctc_score_workspace_bytes(ctypes.byref(_desc(4, 50, lim.max_alphabet + 1, 10)), 1) == 0
    assert "alphabet %d" % (lim.max_alphabet + 1) in L.e2e_last_error_string().decode()
    for n_hyp in (0, -1):
        assert L.e2e_ctc_score_workspace_bytes(ctypes.byref(_desc(4, 50, 29, 10)), n_hyp) == 0
        assert "n_hyp %d" % n_hyp in L.e2e_last_error_string().decode()


def test_score_device_argument_errors(lib_built):
    from end2end_b200 import _lib
    L = _lib.load()
    d = _desc(2, 10, 5, 3)
    fake = ctypes.c_void_p(256)              # never dereferenced: every case fails before a launch
    ok_args = [fake, fake, None, fake, fake, fake, 256, None]

    def call(desc, n_hyp, args):
        return L.e2e_ctc_score_device(ctypes.byref(desc) if desc is not None else None, n_hyp, *args)

    assert call(None, 1, ok_args) == 1
    assert call(d, 0, ok_args) == 1 and "n_hyp 0" in L.e2e_last_error_string().decode()
    for i in (0, 1, 3, 4):                   # logits, hyps, hyp_lengths, scores
        args = list(ok_args)
        args[i] = None
        assert call(d, 2, args) == 1 and "null pointer" in L.e2e_last_error_string().decode(), i
    # no labels at all: hyps may be NULL; this call passes the pointer checks and stops at the (null) workspace
    assert call(_desc(2, 10, 5, 0), 2, [fake, None, None, fake, fake, None, 256, None]) == 3
    assert "workspace" in L.e2e_last_error_string().decode()
    bad = _desc(2, 10, 5, 3)
    bad.targets_stride_b = 2
    assert call(bad, 2, ok_args) == 1 and "row stride" in L.e2e_last_error_string().decode()
    bad = _desc(2, 10, 5, 3)
    bad.blank_idx = 5
    assert call(bad, 2, ok_args) == 1
    bad = _desc(2, 10, 5, 3)
    bad.dtype = 9
    assert call(bad, 2, ok_args) == 1
    args = list(ok_args)
    args[6] = 255                            # workspace too small
    assert call(d, 2, args) == 3
    args = list(ok_args)
    args[5] = ctypes.c_void_p(255 + 256)     # misaligned workspace
    assert call(d, 2, args) == 3
    assert call(_desc(2, 10, 5, MAX_TARGETS + 1), 1, ok_args) == 2


# ---------------------------------------------------------------------------------------------- GPU -----------------

def _cfg_input(name, B, dtype):
    Bc, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS[name]
    x, _, ll, _ = oracle.make_inputs(min(Bc, B), T, V, Lmin, Lmax, seed, full_length=full)
    return torch.log_softmax(x.double(), 2).to(dtype), ll, Lmax


@pytest.mark.gpu
@pytest.mark.parametrize("name,dtype", [("c1", torch.float32), ("c2", torch.float32), ("c3", torch.bfloat16),
                                        ("c4", torch.float32), ("c2", torch.float64), ("c1", torch.float16)])
@pytest.mark.parametrize("N", [1, 3, H - 1, H, H + 1, 100])
def test_oracle_parity_configs(name, dtype, N):
    """Log-prob input in every dtype: the values, widened, are the oracle's input."""
    if name == "c4" and N == 100:
        N = 2 * H + 3                        # the oracle's replicated gradient at V = 1024 would be 200 MB per utterance
    lp, ll, Lmax = _cfg_input(name, 3, dtype)
    B, T, V = lp.shape
    g = torch.Generator().manual_seed(1000 + N)
    for blank in (0, 3, V - 1):
        hyps, hl = random_hyps(g, B, N, Lmax, V, blank)
        ll2 = ll.clone()
        ll2[0] = T
        if B > 2:
            ll2[1], ll2[2] = 1, 2
        got = score(lp.cuda(), hyps.cuda(), hl.cuda(), ll2.cuda(), blank)
        assert got.dtype == torch.float64 and got.shape == (B, N)
        assert_scores(got, oracle_scores(lp, hyps, hl, ll2, blank), ctx=(name, dtype, N, blank))


@pytest.mark.gpu
@pytest.mark.parametrize("Lmax", K_BOUNDARIES)
def test_oracle_parity_k_variants(Lmax):
    """Every cells-per-lane variant at and next to its width boundary, with full-length hypotheses and the length-0 / 1
    ones in the same CTA; T just enough for the longest (tight) and T_i in {1, 2, T}."""
    g = torch.Generator().manual_seed(Lmax)
    B, V = 4, 29
    T = 2 * Lmax + 2
    lp = torch.log_softmax(torch.randn(B, T, V, generator=g, dtype=torch.float64) * 2.0, 2)
    ll = torch.tensor([T, 1, 2, Lmax + 1])
    hyps, hl = random_hyps(g, B, H + 1, Lmax, V, 0)
    hl[:, 4] = Lmax
    hyps[:, 4] = torch.arange(Lmax) % (V - 1) + 1           # no repeats: feasible in Lmax + 1 frames
    got = score(lp.cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), 0)
    want = oracle_scores(lp, hyps, hl, ll, 0)
    assert_scores(got, want, ctx=Lmax)
    assert math.isfinite(float(want[3, 4])) and math.isfinite(float(want[0, 4]))


@pytest.mark.gpu
@pytest.mark.parametrize("V,blank", [(4096, 0), (4096, 4095), (3000, 7)])
def test_oracle_parity_gathered_columns(V, blank):
    """Alphabets whose row block does not fit shared memory: the CTA gathers each hypothesis's columns and the blank."""
    g = torch.Generator().manual_seed(V + blank)
    B, T, Lmax, N = 2, 70, 30, H + 3
    x = torch.randn(B, T, V, generator=g, dtype=torch.float64) * 3.0
    lp = torch.log_softmax(x, 2)
    ll = torch.tensor([T, 41])
    hyps, hl = random_hyps(g, B, N, Lmax, V, blank)
    want = oracle_scores(lp, hyps, hl, ll, blank)
    assert_scores(score(lp.cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), blank), want, ctx=(V, blank))
    got = score(x.float().cuda(), hyps.cuda(), hl.cuda(), ll.cuda(), blank, from_logits=True)
    want = oracle_scores(F.log_softmax(x.float(), 2), hyps, hl, ll, blank)
    assert_scores(got, want, rtol=1e-6, ctx=(V, blank, "logits"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_LOSS)
def test_reference_anchor_golden(name):
    """N = 1 on the reference's own loss vectors: minus its stored loss, within the loss's tolerance (1e-5)."""
    z = np.load(os.path.join(GOLD, name + ".npz"))
    lp = torch.log_softmax(torch.from_numpy(z["x"]), 2)
    tg = torch.from_numpy(z["targets"])
    ll, tl = torch.from_numpy(z["logits_lengths"]), torch.from_numpy(z["targets_lengths"])
    got = score(lp.cuda(), tg[:, None, :].cuda(), tl[:, None].cuda(), ll.cuda(), int(z["blank"]))[:, 0].cpu()
    ref = -torch.from_numpy(z["engine_losses"]).double()
    fin = torch.isfinite(ref)
    assert torch.equal(fin, torch.isfinite(got)) and torch.equal(got[~fin], ref[~fin])
    assert bool(((got[fin] - ref[fin]).abs() <= 1e-5 + 1e-5 * ref[fin].abs()).all()), (got, ref)


@pytest.mark.gpu
def test_raw_logits_layouts_and_host_input():
    """fp32 raw logits within 1e-6 of the oracle on F.log_softmax; bf16 / f16 within one ulp of the stored type;
    time-major, non-contiguous, int32 indices, missing lengths and CPU input through CTCDecoder.score."""
    from pytorch_end2end import CTCDecoder
    g = torch.Generator().manual_seed(7)
    B, T, V, Lmax, N = 3, 60, 40, 25, H + 2
    x = torch.randn(B, T, V, generator=g) * 2.5
    ll = torch.tensor([60, 33, 2])
    blank = 3
    hyps, hl = random_hyps(g, B, N, Lmax, V, blank)
    want = oracle_scores(F.log_softmax(x, 2), hyps, hl, ll, blank)
    dec = CTCDecoder(blank_idx=blank)
    for xx, hh, ln, lls in ((x.cuda(), hyps.cuda(), hl.cuda(), ll.cuda()),
                            (x, hyps, hl, ll),                                                     # CPU input
                            (x.cuda(), hyps.int().cuda(), hl.int().cuda(), ll.int().cuda()),       # int32
                            (x.cuda(), hyps.int(), hl.int(), ll)):                                 # mixed residence
        got = dec.score(xx, hh, ln, lls)
        assert got.device.type == "cpu" and got.dtype == torch.float64
        assert_scores(got, want, rtol=1e-6)
    wide = torch.randn(B, T, V + 9, generator=g)
    wide[:, :, :V] = x
    assert_scores(dec.score(wide.cuda()[:, :, :V], hyps.cuda(), hl.cuda(), ll.cuda()), want, rtol=1e-6)   # strided
    tm = CTCDecoder(blank_idx=blank, time_major=True)
    assert_scores(tm.score(x.transpose(0, 1).contiguous().cuda(), hyps.cuda(), hl.cuda(), ll.cuda()), want, rtol=1e-6)
    full = oracle_scores(F.log_softmax(x, 2), hyps, hl, torch.full((B,), T), blank)
    assert_scores(dec.score(x.cuda(), hyps.cuda(), hl.cuda()), full, rtol=1e-6)                   # logits_lengths=None
    lpd = CTCDecoder(blank_idx=blank, after_logsoftmax=True)
    assert_scores(lpd.score(F.log_softmax(x.double(), 2).cuda(), hyps.cuda(), hl.cuda(), ll.cuda()),
                  oracle_scores(F.log_softmax(x.double(), 2), hyps, hl, ll, blank))
    for dt, rtol in ((torch.bfloat16, 2.0 ** -8), (torch.float16, 2.0 ** -10)):
        xh = x.to(dt)
        # torch's own log-softmax on the device: (x - max) - log sum exp in fp32, rounded to the input dtype.  (Its CPU
        # kernel orders the float arithmetic differently, so single elements land one 16-bit ulp apart.)
        want_h = oracle_scores(F.log_softmax(xh.cuda(), 2), hyps, hl, ll, blank)
        assert_scores(dec.score(xh.cuda(), hyps.cuda(), hl.cuda(), ll.cuda()), want_h, rtol=rtol, ctx=dt)


def _exhaustive_input(V, T, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.log_softmax(torch.randn(2, T, V, generator=g, dtype=torch.float64) * 1.5, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("V,T", [(2, 1), (2, 7), (2, 40), (2, 100), (3, 1), (3, 4), (3, 6), (4, 2), (4, 4)])
def test_nbest_round_trip_exhaustive(V, T):
    """Beams that hold every prefix are exact: score(decode_nbest(...)) == log_probs, the -1 empty marker included."""
    from pytorch_end2end import CTCDecoder
    lp = _exhaustive_input(V, T, 100 * V + T).cuda()
    dec = CTCDecoder(beam_width=256, after_logsoftmax=True, blank_idx=V - 1, wip=0.0)
    nb = dec.decode_nbest(lp, n_best=256)
    sc = dec.score(lp, nb.decoded_targets, nb.decoded_targets_lengths)
    real = nb.scores > -math.inf
    assert bool(torch.allclose(sc[real], nb.log_probs[real], rtol=1e-10, atol=0)), (sc[real] - nb.log_probs[real]).abs().max()
    empty = (nb.decoded_targets_lengths == 1) & (nb.decoded_targets[:, :, 0] == -1)
    assert bool(empty.any())
    used = nb.decoded_targets_lengths > 0
    # members of the final beam with probability 0 (fewer feasible prefixes than the beam is wide) are infeasible
    assert bool(torch.isneginf(sc[used & ~real]).all())
    blank_path = lp[:, :, V - 1].sum(1).cpu()
    for b in range(lp.size(0)):                                      # unused slots score as the empty transcript
        assert bool((sc[b][~used[b]] == sc[b][empty[b]]).all()) and abs(float(sc[b][empty[b]][0] - blank_path[b])) < 1e-10


@pytest.mark.gpu
def test_nbest_round_trip_c2_bound():
    """c2 batch at beam 100, N = 100: the beam sums a subset of the alignments the forward algorithm sums."""
    from pytorch_end2end import CTCDecoder
    x, _, ll, _ = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    dec = CTCDecoder(beam_width=100)
    nb = dec.decode_nbest(x.cuda(), ll, n_best=100)
    sc = dec.score(x.cuda(), nb.decoded_targets.cuda(), nb.decoded_targets_lengths.cuda(), ll.cuda())
    real = nb.scores > -math.inf
    assert bool(real.all())
    assert bool((sc[real] >= nb.log_probs[real] - 1e-12 * sc[real].abs()).all())


@pytest.mark.gpu
def test_isolation_and_determinism():
    g = torch.Generator().manual_seed(3)
    B, T, V, Lmax, N = 3, 80, 29, 60, 2 * H + 5
    lp = torch.log_softmax(torch.randn(B, T, V, generator=g, dtype=torch.float64), 2).cuda()
    ll = torch.tensor([80, 70, 50]).cuda()
    hyps, hl = random_hyps(g, B, N, Lmax, V, 0)
    hyps, hl = hyps.cuda(), hl.cuda()
    s0 = score(lp, hyps, hl, ll)
    assert torch.equal(s0, score(lp, hyps, hl, ll))                               # bit-identical runs
    perm = torch.randperm(N, generator=g).cuda()
    assert torch.equal(score(lp, hyps[:, perm], hl[:, perm], ll), s0[:, perm])    # permutation, bit for bit
    bad_h, bad_l = hyps.clone(), hl.clone()
    bad_l[0, 5] = 5
    bad_h[0, 5, 2] = V                                                             # label out of range (device-resident)
    bad_l[1, 9] = Lmax + 1                                                         # length out of range
    bad_l[2, 0] = -1
    s1 = score(lp, bad_h, bad_l, ll)
    flagged = torch.zeros(B, N, dtype=torch.bool, device="cuda")
    flagged[0, 5] = flagged[1, 9] = flagged[2, 0] = True
    assert bool(torch.isnan(s1[flagged]).all())
    assert torch.equal(s1[~flagged], s0[~flagged])
    ll_bad = ll.clone()
    ll_bad[1] = T + 1                                                              # frames out of range: the utterance's row
    s2 = score(lp, hyps, hl, ll_bad)
    assert bool(torch.isnan(s2[1]).all()) and torch.equal(s2[[0, 2]], s0[[0, 2]])
    ll_bad[1] = 0
    assert bool(torch.isnan(score(lp, hyps, hl, ll_bad)[1]).all())


@pytest.mark.gpu
def test_python_errors_before_device_work():
    from end2end_b200 import _lib
    from pytorch_end2end import CTCDecoder
    dec = CTCDecoder(blank_idx=0)
    x = torch.randn(2, 10, 5)
    hyps = torch.ones(2, 3, 4, dtype=torch.int64)
    hl = torch.full((2, 3), 2)
    dec.score(x.cuda(), hyps.cuda(), hl.cuda())
    before = _lib.launch_count()
    cases = [(ValueError, (x, hyps, torch.full((2, 3), 5))),                  # length > Lmax
             (ValueError, (x, hyps, torch.full((2, 3), -1))),
             (ValueError, (x, torch.full((2, 3, 4), 5), hl)),                  # label == V
             (ValueError, (x, torch.full((2, 3, 4), -2), hl)),
             (ValueError, (x, hyps, hl, torch.tensor([10, 11]))),              # frames > T
             (ValueError, (x, hyps, hl, torch.tensor([0, 10]))),
             (ValueError, (x, hyps, torch.full((2, 4), 2))),                   # shapes
             (ValueError, (x, hyps[:1], hl)),
             (NotImplementedError, (x, torch.ones(2, 3, MAX_TARGETS + 1, dtype=torch.int64), hl)),
             (NotImplementedError, (torch.randn(1, 2, _lib.limits().max_alphabet + 1), hyps[:1], hl[:1]))]
    for exc, args in cases:
        with pytest.raises(exc):
            dec.score(*args)
        with pytest.raises(exc):
            dec.score(args[0].cuda(), *args[1:])
    assert _lib.launch_count() == before


@pytest.mark.gpu
def test_raw_c_abi_n1_matches_python_and_loss():
    """n_hyp = 1 on a [B, Lmax] target matrix: the Python path's bytes on fp64 log-probs, and minus the loss engine's
    forward within the loss's tolerance."""
    from end2end_b200 import CTCLossEngine, _lib
    L = _lib.load()
    x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS["c2"][:6])
    lp = torch.log_softmax(x.double(), 2).cuda()
    tg, ll, tl = tg.cuda(), ll.cuda(), tl.cuda()
    B, T, V = lp.shape
    d = _desc(B, T, V, tg.size(1))
    ws = torch.empty(L.e2e_ctc_score_workspace_bytes(ctypes.byref(d), 1), dtype=torch.uint8, device="cuda")
    out = torch.full((B,), 7.0, dtype=torch.float64, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())                # noqa: E731
    _lib.check(L.e2e_ctc_score_device(ctypes.byref(d), 1, p(lp), p(tg), p(ll), p(tl), p(out), p(ws), ws.numel(),
                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert torch.equal(out, score(lp, tg[:, None], tl[:, None], ll)[:, 0])
    loss, _ = CTCLossEngine(0).forward(lp, tg, ll, tl)
    diff = (out + loss).abs()
    print("largest |score + loss| on c2 (fp64):", float(diff.max()))
    assert bool((diff <= 1e-5 + 1e-5 * loss.abs()).all())

"""Host-side logic and the C-ABI surface -- no GPU needed (no compute calls)."""
import ctypes
import os
import re
import subprocess
import sys
import tempfile

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L(lib_built):
    from end2end_b200 import _lib
    return _lib.load()


def _desc(B=4, T=50, V=28, Lmax=29, dtype=0, blank=0):
    from end2end_b200 import _lib
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets, d.blank_idx, d.dtype = B, T, V, Lmax, blank, dtype
    d.targets_itype = d.lengths_itype = _lib.E2E_I64
    d.logits_stride_b, d.logits_stride_t = T * V, V
    d.grads_stride_b, d.grads_stride_t = T * V, V
    d.targets_stride_b = Lmax
    return d


def test_library_exports_every_declared_symbol(L):
    from end2end_b200 import _lib
    header = open(os.path.join(ROOT, "include", "e2e_ctc.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(e2e_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(L, name), name
    syms = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (e2e_\w+)", syms))
    assert declared <= exported
    assert b"sm_100a" in L.e2e_ctc_version()


def test_descriptor_layout_matches_the_header():
    from end2end_b200 import _lib
    src = r'''
#include <stdio.h>
#include <stddef.h>
#include "e2e_ctc.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu\n", sizeof(e2e_ctc_desc), offsetof(e2e_ctc_desc, from_logits),
         offsetof(e2e_ctc_desc, logits_stride_b), offsetof(e2e_ctc_desc, targets_stride_b),
         sizeof(e2e_ctc_limits), offsetof(e2e_ctc_desc, lengths_itype));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, "l.c")
        open(c, "w").write(src)
        exe = os.path.join(td, "l")
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        got = [int(v) for v in subprocess.check_output([exe]).split()]
    D = _lib.Desc
    assert got == [ctypes.sizeof(D), D.from_logits.offset, D.logits_stride_b.offset, D.targets_stride_b.offset,
                   ctypes.sizeof(_lib.Limits), D.lengths_itype.offset]


def test_limits_and_workspace_planning(L):
    from end2end_b200 import _lib
    lim = _lib.limits()
    assert lim.abi_version == 1 and lim.sm_arch == 100 and lim.max_targets >= 600 and lim.max_alphabet >= 1024
    sizes = {}
    for name, (B, T, V, Lmax) in {"c1": (4, 50, 28, 29), "c2": (64, 400, 29, 200), "c3": (1024, 128, 96, 40),
                                  "c4": (128, 250, 1024, 80), "c5": (2048, 1600, 29, 600)}.items():
        n = L.e2e_ctc_loss_workspace_bytes(ctypes.byref(_desc(B, T, V, Lmax)))
        cells = 2 * Lmax + 1
        assert n >= B * T * cells * 4 and n % 256 == 0, name      # stashed half-lattice: 4 bytes per cell
        assert n <= B * T * (cells + 256) * 9 + (1 << 20), name        # padding stays bounded
        sizes[name] = n
    assert sizes["c5"] < 60 * 2 ** 30                                    # fits a 180 GB part with room to spare
    assert L.e2e_ctc_greedy_workspace_bytes(ctypes.byref(_desc(128, 250, 1024, 0))) >= 128 * 250 * 4
    # L = 0 everywhere is legal (blank-only lattices)
    assert L.e2e_ctc_loss_workspace_bytes(ctypes.byref(_desc(2, 5, 3, 0))) > 0


@pytest.mark.parametrize("mutate,code", [
    (dict(batch=0), 1), (dict(alphabet=0), 1), (dict(dtype=9), 1), (dict(blank_idx=28), 1), (dict(blank_idx=-1), 1),
    (dict(lengths_itype=5), 1), (dict(max_targets=-1), 1), (dict(max_targets=100000), 2), (dict(alphabet=10 ** 6), 2),
])
def test_bad_descriptors_are_rejected_with_a_message(L, mutate, code):
    d = _desc()
    for k, v in mutate.items():
        setattr(d, k, v)
    assert L.e2e_ctc_loss_workspace_bytes(ctypes.byref(d)) == 0
    dummy = ctypes.c_void_p(256)
    rc = L.e2e_ctc_loss_fwd_bwd_device(ctypes.byref(d), dummy, dummy, dummy, dummy, dummy, dummy, dummy, 1 << 40, None)
    assert rc == code
    assert len(L.e2e_last_error_string()) > 0


def test_null_and_workspace_errors_without_touching_the_gpu(L):
    d = _desc()
    dummy = ctypes.c_void_p(256)
    assert L.e2e_ctc_loss_fwd_bwd_device(ctypes.byref(d), None, dummy, dummy, dummy, dummy, dummy, dummy, 1 << 40, None) == 1
    assert L.e2e_ctc_loss_fwd_bwd_device(ctypes.byref(d), dummy, dummy, dummy, dummy, dummy, dummy, dummy, 16, None) == 3
    assert L.e2e_ctc_loss_fwd_bwd_device(ctypes.byref(d), dummy, dummy, dummy, dummy, dummy, dummy, ctypes.c_void_p(8), 1 << 40, None) == 3
    assert L.e2e_ctc_loss_backward_device(ctypes.byref(d), dummy, dummy, dummy, dummy, dummy, 3, 1.0, dummy, dummy, 1 << 40, None) == 1
    assert L.e2e_ctc_greedy_decode_device(ctypes.byref(d), dummy, None, None, dummy, dummy, 1 << 40, None) == 1
    assert L.e2e_ctc_loss_reduce_device(None, 0, 4, 1.0, dummy, None, None) == 1
    assert L.e2e_ctc_engine_loss_host(None, ctypes.byref(d), dummy, dummy, dummy, dummy, dummy, dummy) == 1


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback_anywhere(L):
    import end2end_b200
    import pytorch_end2end
    assert pytorch_end2end.CTCLoss is end2end_b200.CTCLoss and pytorch_end2end.CTCDecoder is end2end_b200.CTCDecoder
    h = ctypes.c_void_p(0)
    assert L.e2e_ctc_engine_create(0, ctypes.byref(h)) == 4 and not h.value
    x = torch.randn(2, 6, 5)
    tg, ll, tl = torch.tensor([[1, 2], [3, 1]]), torch.tensor([6, 6]), torch.tensor([2, 2])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        end2end_b200.CTCLoss(reduce=True)(x.requires_grad_(), tg, ll, tl)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        end2end_b200.CTCLossEngine(0).compute(torch.log_softmax(x, 2), tg, ll, tl)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        end2end_b200.CTCDecoder(beam_width=1).decode(x)


def test_product_never_touches_the_oracle():
    pat = re.compile(r"^\s*(from|import)\s+oracle\b|oracle/|libctc_oracle|ctc_oracle", re.M)
    for pkg in ("end2end_b200", "pytorch_end2end", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cpp")):
                    text = open(os.path.join(dirpath, f), errors="replace").read()
                    assert not pat.search(text), os.path.join(dirpath, f)


def test_missing_library_fails_loudly(monkeypatch):
    from end2end_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libe2e_ctc.so")
    with pytest.raises(ImportError, match="no CPU fallback"):
        _lib.load()


def test_module_api_surface():
    import inspect
    import end2end_b200 as e
    sig = inspect.signature(e.CTCLoss.__init__)
    assert list(sig.parameters)[1:] == ["size_average", "reduce", "after_logsoftmax", "time_major", "blank_idx"]
    assert [p.default for p in list(sig.parameters.values())[1:]] == [None, None, False, False, 0]
    sig = inspect.signature(e.CTCDecoder.__init__)
    assert list(sig.parameters)[1:] == ["beam_width", "after_logsoftmax", "blank_idx", "time_major", "labels",
                                        "lm_path", "lmwt", "wip", "oov_penalty", "case_sensitive"]
    dec = e.CTCDecoder(beam_width=20, lm_path="/no/such/model.arpa")   # KenLM decoding stays the reference's CPU code
    with pytest.raises(NotImplementedError):
        dec.decode(torch.zeros(1, 2, 3))
    if not torch.cuda.is_available():                                     # beam search without a device fails loudly
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            e.CTCDecoder(beam_width=20).decode(torch.zeros(1, 2, 3))
    assert list(inspect.signature(e.CTCLossEngine.compute).parameters)[1:5] == [
        "logits", "targets", "logits_lengths", "targets_lengths"]
    assert list(inspect.signature(e.CTCGreedyEngine.decode_greedy).parameters)[1:] == ["logits_", "logits_lengths_"]


def test_ctc_encoder():
    from pytorch_end2end import CTCEncoder
    enc = CTCEncoder("ABC ", blank_id=1)
    assert enc.char2id == {"A": 0, "B": 2, "C": 3, " ": 4} and enc.num_symbols == 5
    ids = enc.encode("a cab!")
    assert ids.tolist() == [0, 4, 3, 0, 2]
    assert enc.decode([0, 0, 1, 0, 4, 4, 1, 3]) == "AA C"
    assert enc.decode_pure([0, 1, 2]) == "AB" and enc.clean("x-b") == "B"


# ------------------------------------------------------------------------------------------------
# multi-GPU host logic: the shard planner and the (gloo, world_size 2) loss all-reduce
# ------------------------------------------------------------------------------------------------
def test_plan_shards_is_a_balanced_partition():
    from end2end_b200.distributed import plan_shards, utterance_cost
    g = torch.Generator().manual_seed(0)
    for world in (1, 2, 4, 8):
        ll = torch.randint(1200, 1601, (2048,), generator=g)
        tl = torch.randint(300, 601, (2048,), generator=g)
        buckets = plan_shards(ll, tl, 29, world)
        assert len(buckets) == world
        assert sorted(i for b in buckets for i in b) == list(range(2048))
        cost = [utterance_cost(a, b, 29) for a, b in zip(ll.tolist(), tl.tolist())]
        loads = [sum(cost[i] for i in b) for b in buckets]
        assert max(loads) - min(loads) <= max(cost)                      # LPT bound
        for b in buckets:                                                # length-sorted inside a bucket
            assert [cost[i] for i in b] == sorted((cost[i] for i in b), reverse=True)
        assert plan_shards(ll, tl, 29, world) == buckets                 # deterministic
    assert plan_shards([5], [1], 4, 3) == [[0], [], []]
    with pytest.raises(ValueError):
        plan_shards([5, 6], [1], 4, 2)


def _gloo_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import oracle
    from end2end_b200.distributed import ShardedCTCLoss, plan_shards, take_shard
    dist.init_process_group("gloo", rank=rank, world_size=world)

    class OracleStandIn:                        # test-only stand-in for the CUDA engine (host-tensor contract)
        def compute(self, logits, targets, ll, tl, from_logits=False):
            if not from_logits:
                return oracle.PortEngine(0).compute(logits, targets, ll, tl)
            with torch.enable_grad():           # called from inside an autograd Function's forward
                leaf = logits.detach().clone().requires_grad_()
                losses = oracle.ctc_loss_module(oracle.PortEngine(0), leaf, targets, ll, tl)
                losses[torch.isfinite(losses)].sum().backward()
            return losses.detach(), leaf.grad

    x, tg, ll, tl = oracle.make_inputs(10, 30, 8, 2, 9, 3)
    buckets = plan_shards(ll, tl, 8, world)
    for mean in (False, True):
        for gb in (None, 10):
            xs, tgs, lls, tls = take_shard(buckets[rank], x, tg, ll, tl)
            leaf = xs.clone().requires_grad_()
            crit = ShardedCTCLoss(reduce=True, size_average=mean, global_batch=gb, engine=OracleStandIn())
            loss = crit(leaf, tgs, lls, tls)
            loss.backward()
            torch.save({"loss": loss.detach(), "grad": leaf.grad, "idx": buckets[rank]},
                       os.path.join(out_dir, "r%d_m%d_g%s.pt" % (rank, mean, gb)))
    # reduce falsy: local per-utterance losses, nothing exchanged
    xs, tgs, lls, tls = take_shard(buckets[rank], x, tg, ll, tl)
    local = ShardedCTCLoss(engine=OracleStandIn())(xs, tgs, lls, tls)
    assert local.shape == (len(buckets[rank]),)
    dist.destroy_process_group()


def test_sharded_loss_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    import oracle
    port = 29500 + os.getpid() % 2000
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    x, tg, ll, tl = oracle.make_inputs(10, 30, 8, 2, 9, 3)
    for mean in (False, True):
        leaf = x.clone().requires_grad_()
        ref = oracle.ctc_loss_module(oracle.PortEngine(0), leaf, tg, ll, tl, reduce=True, size_average=mean)
        ref.backward()
        for gb in (None, 10):
            parts = [torch.load(os.path.join(str(tmp_path), "r%d_m%d_g%s.pt" % (r, mean, gb))) for r in range(2)]
            for p in parts:                                              # same global scalar on every rank
                assert torch.allclose(p["loss"], ref.detach(), rtol=1e-6, atol=1e-6)
                assert torch.allclose(p["grad"], leaf.grad[p["idx"]], rtol=1e-6, atol=1e-7)


def test_beam_workspace_query_and_limits(lib_built):
    """Host-only entry point of the prefix beam search: the size query works without a device and states its limits."""
    import ctypes
    from end2end_b200 import _lib
    L = _lib.load()
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = 64, 400, 29, 0
    d.blank_idx, d.dtype = 0, _lib.E2E_F32
    d.targets_itype = d.lengths_itype = _lib.E2E_I64
    d.logits_stride_b, d.logits_stride_t = 400 * 29, 29
    n = L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), 100)
    nodes = 64 * (400 * 100 + 1) * 16                      # one 16-byte trie node per frame and beam slot, plus the root
    assert nodes <= n < nodes + 256
    assert L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), 257) == 0          # beam_width beyond the build's limit
    assert "limits" in L.e2e_last_error_string().decode()
    assert L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), 0) == 0
    d.alphabet, d.logits_stride_t, d.logits_stride_b = 1024, 1024, 400 * 1024                # large alphabets are pre-filtered per frame
    assert L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), 100) > 0
    d.alphabet = 32768                                     # rows of this size do not fit shared memory
    assert L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), 100) == 0


def _neighbour_desc(B, T, V, Lmax):
    from end2end_b200 import _lib
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
    d.blank_idx, d.dtype = 0, _lib.E2E_F32
    d.targets_itype = d.lengths_itype = _lib.E2E_I64
    d.logits_stride_b, d.logits_stride_t = T * V, V
    d.targets_stride_b = Lmax
    return d


def test_viterbi_workspace_query_and_limits(lib_built):
    """The alignment has its own width limit, lattices of at most 2048 cells, not the loss's 639 labels: CTC (2 L + 1
    cells) up to L = 1023, ASG (L cells) up to L = 2048.  One label more is refused by the size query, without a device."""
    import ctypes
    from end2end_b200 import _lib
    L = _lib.load()
    for is_ctc, widest in ((1, 1023), (0, 2048)):
        d = _neighbour_desc(4, 2 * widest, 29, widest)
        n = L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), is_ctc)
        assert 256 + 4 * 2 * widest * 512 <= n < 256 + 4 * 2 * widest * 512 + 256   # one backpointer byte per thread and frame
        for lmax in (640, widest // 2):                                # beyond the loss's limit, below the alignment's
            d.max_targets = lmax
            assert L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), is_ctc) > 0
        d.max_targets = widest + 1
        assert L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), is_ctc) == 0
        assert "limit" in L.e2e_last_error_string().decode()
    d = _neighbour_desc(4, 50, 29, 0)
    assert L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), 1) > 0
    d.max_targets = -1
    assert L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), 1) == 0


def test_noblank_workspace_query_and_limits(lib_built):
    """CTC without blank runs one thread per lattice cell in one CTA: Lmax + 2 <= 1024 cells.  The size query applies
    that limit (and the shared-memory bound on the alphabet) so that nothing is allocated for a shape that cannot run."""
    import ctypes
    from end2end_b200 import _lib
    L = _lib.load()
    d = _neighbour_desc(4, 1100, 29, 1022)
    n = L.e2e_ctc_noblank_workspace_bytes(ctypes.byref(d))
    assert n == 256 + 2 * 4 * 1100 * 1024 * 8                    # alpha and beta rows in fp64
    d.max_targets = 1023
    assert L.e2e_ctc_noblank_workspace_bytes(ctypes.byref(d)) == 0
    assert "1022" in L.e2e_last_error_string().decode()
    d.max_targets, d.alphabet, d.logits_stride_t = 30, 40000, 40000
    assert L.e2e_ctc_noblank_workspace_bytes(ctypes.byref(d)) > 0
    d.alphabet = d.logits_stride_t = 60000                          # the per-symbol lists no longer fit shared memory
    assert L.e2e_ctc_noblank_workspace_bytes(ctypes.byref(d)) == 0
    assert "alphabet" in L.e2e_last_error_string().decode()

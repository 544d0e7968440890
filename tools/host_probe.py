"""Where does the host-buffer call (CTCLossEngine.compute on CPU tensors -> e2e_ctc_engine_loss_host) spend its time?
Prints PCIe copy times at the batch's sizes, the call's time per chunk count, and the fixed per-call overhead.
    python tools/host_probe.py [c2]"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import oracle  # noqa: E402
from end2end_b200 import CTCLossEngine  # noqa: E402

cfg = sys.argv[1] if len(sys.argv) > 1 else "c2"
B, T, V, Lmin, Lmax, seed, dtype, full = oracle.CONFIGS[cfg]
x, tg, ll, tl = oracle.make_inputs(B, T, V, Lmin, Lmax, seed, dtype=dtype, full_length=full)


def timeit(fn, n=50, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e6


# 1. raw PCIe copies, pinned, at the batch's sizes
for nbytes in (x.numel() * x.element_size() // 3, x.numel() * x.element_size()):
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    t_in = timeit(lambda: d.copy_(h, non_blocking=True))
    t_out = timeit(lambda: h.copy_(d, non_blocking=True))
    print("pinned copy %8d B: H2D %.1f us (%.1f GB/s)  D2H %.1f us (%.1f GB/s)" % (nbytes, t_in, nbytes / t_in / 1e3, t_out, nbytes / t_out / 1e3))
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def both():
        with torch.cuda.stream(s1):
            d.copy_(h, non_blocking=True)
        with torch.cuda.stream(s2):
            h2.copy_(d2, non_blocking=True)
    h2, d2 = torch.empty_like(h).pin_memory(), torch.empty_like(d)
    print("   both directions at once: %.1f us" % timeit(both))

eng = CTCLossEngine(0)
xp = x.pin_memory()
pins = (tg.pin_memory(), ll.pin_memory(), tl.pin_memory())
# 2. the call, by chunk count; small tensors pageable vs pinned
for chunks in ("-1", "1", "2", "3", "4", "6", "8"):
    os.environ["E2E_CTC_HOST_CHUNKS"] = chunks
    a = timeit(lambda: eng.compute(xp, tg, ll, tl, from_logits=True), n=40)
    b = timeit(lambda: eng.compute(xp, *pins, from_logits=True), n=40)
    print("chunks %2s: %.1f us/call (%.0f utt/s)   all-pinned inputs: %.1f us/call (%.0f utt/s)" % (chunks, a, B / a * 1e6, b, B / b * 1e6))
os.environ.pop("E2E_CTC_HOST_CHUNKS")
# 3. fixed overhead: a one-utterance, eight-frame call
x1, tg1, ll1, tl1 = oracle.make_inputs(1, 8, V, 1, 2, 3)
x1 = x1.pin_memory()
print("B=1 T=8 call: %.1f us" % timeit(lambda: eng.compute(x1, tg1, ll1, tl1, from_logits=True), n=100))
# 4. device-resident step for comparison
xc, tgc, llc, tlc = x.cuda(), tg.cuda(), ll.cuda(), tl.cuda()
print("device step (engine.step): %.1f us" % timeit(lambda: eng.step(xc, tgc, llc, tlc, True, 1.0 / B, 1.0 / B), n=100))
g = eng.graphed_step(xc, tgc, llc, tlc, True, 1.0 / B, 1.0 / B)
print("device step (graph replay): %.1f us" % timeit(lambda: g.launch(), n=200))
# 5. where the Python wrapper's time goes (the pieces of CTCLossEngine._compute_host, timed separately)
import ctypes
from end2end_b200 import _lib
from end2end_b200.engine import _Problem, _host_engine, _ptr
cpu = torch.device("cpu")


def t_us(fn, n=200):
    fn()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    return (time.perf_counter() - t0) / n * 1e6


print("_Problem(...) host: %.1f us" % t_us(lambda: _Problem(0, xp, tg, ll, tl, True, cpu, validate=False)))
print("torch.empty(B, pinned): %.1f us" % t_us(lambda: torch.empty(B, dtype=xp.dtype, pin_memory=True)))
print("torch.empty_strided(logits, pinned): %.1f us" % t_us(lambda: torch.empty_strided(xp.size(), xp.stride(), dtype=xp.dtype, pin_memory=True)))
keep = []
print("  ... while the previous one is still alive: %.1f us" % t_us(lambda: (keep.append(torch.empty_strided(xp.size(), xp.stride(), dtype=xp.dtype, pin_memory=True)), len(keep) > 1 and keep.pop(0))))
pb = _Problem(0, xp, tg, ll, tl, True, cpu, validate=False)
losses = torch.empty(B, dtype=xp.dtype, pin_memory=True)
grads = torch.empty_strided(xp.size(), xp.stride(), dtype=xp.dtype, pin_memory=True)
h = _host_engine(eng._host)
L = _lib.load()
for chunks in ("1", "2", "3", "4", "6", "8"):
    os.environ["E2E_CTC_HOST_CHUNKS"] = chunks
    print("C call only, chunks %s: %.1f us" % (chunks, t_us(lambda: L.e2e_ctc_engine_loss_host(
        h.handle, ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths), _ptr(pb.targets_lengths), _ptr(losses), _ptr(grads)), n=60)))

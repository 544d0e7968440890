#!/usr/bin/env python
"""Benchmark of the CTC hot path (BASELINE.json metric: CTC fwd+bwd utterances/s & HBM GB/s % peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

One "step" = one forward+backward pass of CTCLoss(reduce=True, size_average=True,
after_logsoftmax=False) over one synthetic batch of the named workload (default BASELINE
configs[1]: LibriSpeech-shaped B=64, T=400, V=29, L<=200, fp32), i.e. the reference call stack
modules/ctc_loss.py:25-57 -> functions/forward_backward.py:6-35 -> src/losses/*.cpp.

Our arm (default):
  value      whole-job utterances/s with the inputs resident in HBM: K replays of the criterion's captured step
             (criterion.graphed(...): memset + lattice kernel(s) + loss reduction [+ all-reduce], SURVEY 8(f1)),
             timed with CUDA events on the launching stream between barriers, max over ranks;
             `autograd` repeats the measurement through loss = crit(...); loss.backward();
  e2e        the same metric through the reference-facing engine call on HOST (pinned) buffers:
             CTCLossEngine.compute() -> e2e_ctc_engine_loss_host() copies the inputs in, runs the
             kernels, copies losses + gradient back -- all inside the timed region;
  roofline   the dominant kernel timed live with CUDA events by the library's profile hooks:
             algorithmic bytes (logits read + gradient write, SURVEY 8d) per launch / mean launch time,
             against MEASURED_PEAKS.json hbm_gbs; `step_frac` is the same for the whole step;
  parity_check  BEFORE the timed region every rank compares its bucket's losses and gradients (autograd path
             and graph replay) with the CPU oracle, and the all-reduced loss with the oracle's global mean;
  per_workload / greedy / strong   (N=1: the other BASELINE shapes; c4 greedy decode; every N: c3 at a FIXED
             global batch sharded over the ranks);
  cpu_baseline  the reference CPU engine (oracle/_ref, else the C port) on this box's host cores, the
             better of OMP_NUM_THREADS=1 and =cores (the engine already runs one thread per utterance).
N ranks (under torchrun): ONE global batch of N x B utterances is drawn identically on every rank, cut into
cost-balanced buckets by end2end_b200.distributed.plan_shards (LPT), and each rank runs the pipeline on its
bucket; the only exchange is the all-reduce of the scalar loss, enqueued on a side stream so that it overlaps
the next step's lattice kernel (the gradient never depends on it: the global batch size is folded in).

--impl reference times the reference's own CPU implementation on the same workload and prints the
same JSON line with "impl": "reference".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (B, T, V, Lmin, Lmax, seed, dtype, full_length, description)
    "c1": (4, 50, 28, 10, 29, 0, "f32", True, "README CTCLoss example B=4 T=50 V=28 L 10-29 fp32"),
    "c2": (64, 400, 29, 100, 200, 1, "f32", False, "LibriSpeech-shaped char CTC B=64 T=400 V=29 L 100-200 fp32"),
    "c3": (1024, 128, 96, 20, 40, 2, "bf16", False, "OCR lines B=1024 T=128 V=96 L 20-40 bf16"),
    "c4": (128, 250, 1024, 40, 80, 3, "f32", False, "subword CTC B=128 T=250 V=1024 L 40-80 fp32"),
    "c5": (2048, 1600, 29, 300, 600, 4, "f32", False, "long-form ASR B=2048 T=1600 V=29 L 300-600 fp32"),
}
L2_BYTES = 126 * 2 ** 20
LOSS = "CTCLoss(reduce=True, size_average=True, after_logsoftmax=False)"


def config_for(wl, world):
    """The `config` object: the same keys and values from both arms (the driver compares them)."""
    B, T, V, Lmin, Lmax, seed, dt, full, desc = WORKLOADS[wl]
    return {"workload": "%s: %s" % (wl, desc), "batch_per_gpu": B, "io_dtype": dt, "loss": LOSS,
            "l2": "distinct resident batches rotated so that > 2 x 126 MB streams between reuses of one; workloads "
                  "too small for that flush L2 (256 MB write) between steps and time every step with its own events",
            "parallelism": ("one global batch of %d utterances, LPT length-balanced buckets over %d GPUs, one scalar "
                            "loss all-reduce per step" % (B * world, world)) if world > 1 else "single GPU"}


def make_inputs(B, T, V, Lmin, Lmax, seed, dtype, full_length):
    """SURVEY.md 8(d) draw order: logits, target lengths, targets (blank 0 never a target), frames."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, V, generator=g).to(dtype)
    tl = torch.randint(Lmin, Lmax + 1, (B,), generator=g)
    tg = torch.randint(1, V, (B, Lmax), generator=g)
    ll = torch.full((B,), T, dtype=torch.int64) if full_length else torch.randint(3 * T // 4, T + 1, (B,), generator=g)
    return x, tg, ll, tl


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=3.0):
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def summary(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        inside = [r for (t, r) in self.rows if t0 <= t <= t1]
        rows = inside or [r for (t, r) in self.rows if t0 - 0.1 <= t <= t1 + 0.1] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [c.strip() for c in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_inside_timed_region": len(inside), "reasons": sorted(reasons)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(workload, kernel=None):
    """dram bytes/launch of the workload's dominant kernel from the committed ncu --set full capture, if any."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(workload, {}).get("lattice_dram_bytes_per_launch")
    return None


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ----------------------------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation, timed in a child process per OMP_NUM_THREADS setting
# ----------------------------------------------------------------------------------------------------------
def reference_child(args):
    """One timing of the reference CPU path under the OMP_NUM_THREADS of this process's environment."""
    import torch
    import oracle
    wl = args.workload
    B, T, V, Lmin, Lmax, seed, dt, full, desc = WORKLOADS[wl]
    sample_B = min(B, args.ref_batch)       # the reference keeps ~46 MB of fp64 lattices live per long utterance
    x, tg, ll, tl = make_inputs(sample_B, T, V, Lmin, Lmax, seed, torch.float32, full)
    if dt == "bf16":
        x = x.to(torch.bfloat16).float()      # SURVEY 7.3: the oracle for bf16 logits is the reference on logits.float()
    eng = oracle.engine(0, prefer="reference")

    def step():
        # the reference's Python drives its engine like this (oracle.ctc_loss_module restates modules/ctc_loss.py:25-57)
        leaf = x.detach().clone().requires_grad_()
        loss = oracle.ctc_loss_module(eng, leaf, tg, ll, tl, reduce=True, size_average=True, after_logsoftmax=False)
        loss.backward()
        return float(loss)

    for _ in range(max(1, min(args.warmup, 2))):
        step()
    n, t0 = 0, time.perf_counter()
    if args.cpu_seconds > 0:
        while n < 1 or time.perf_counter() - t0 < args.cpu_seconds:
            step(); n += 1
    else:
        for _ in range(args.steps):
            step(); n += 1
    dt_s = time.perf_counter() - t0
    out = {"value": sample_B * n / dt_s, "ms_per_step": 1e3 * dt_s / n, "steps": n, "sample_B": sample_B, "kind": eng.kind,
           "omp": os.environ.get("OMP_NUM_THREADS"), "greedy": None}
    if args.greedy:
        xg = x if sample_B == B else make_inputs(B, T, V, Lmin, Lmax, seed, torch.float32, full)[0]
        oracle.greedy_decode(xg[:8], None)
        m, t0 = 0, time.perf_counter()
        while m < 1 or time.perf_counter() - t0 < max(1.0, args.cpu_seconds / 3):
            oracle.greedy_decode(xg, None); m += 1
        out["greedy"] = {"value": xg.size(0) * m / (time.perf_counter() - t0), "kind": "reference" if oracle.have_ref() else "port"}
    print("REFCHILD " + json.dumps(out), flush=True)


def measure_reference(wl, steps, warmup, ref_batch, cpu_seconds=0.0, greedy=False):
    """The reference CPU arm under OMP_NUM_THREADS=1 and =cores (child processes: the OpenMP runtime reads the
    variable once); returns (best, all).  The engine runs one host thread per utterance (forward_backward.cpp:37),
    so extra OpenMP threads inside every torch op mostly oversubscribe the cores."""
    cores = os.cpu_count() or 1
    runs = []
    for omp in sorted({1, cores}):
        env = dict(os.environ, OMP_NUM_THREADS=str(omp), MKL_NUM_THREADS=str(omp))
        for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
            env.pop(k, None)
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--_child", "--workload", wl, "--steps", str(steps),
               "--warmup", str(warmup), "--ref-batch", str(ref_batch), "--cpu-seconds", str(cpu_seconds)] + (["--greedy"] if greedy else [])
        try:
            r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
            line = [l for l in r.stdout.splitlines() if l.startswith("REFCHILD ")]
            if line:
                runs.append(json.loads(line[-1][9:]))
        except (subprocess.TimeoutExpired, OSError):
            pass
    if not runs:
        return None, []
    return max(runs, key=lambda d: d["value"]), runs


def run_reference(args, wl):
    rank, _, world = dist_env()
    if rank != 0:
        return
    best, runs = measure_reference(wl, args.steps, args.warmup, args.ref_batch)
    if best is None:
        print(json.dumps({"impl": "reference", "unavailable": "the reference child process produced no timing"}))
        return
    cores = os.cpu_count()
    sample = ("%d utterances of %s per step, %d steps; one host thread per utterance (the reference's pool) on %d cores; "
              "OMP_NUM_THREADS=%s (the better of %s)" % (best["sample_B"], wl, best["steps"], cores, best["omp"],
                                                         ", ".join("%s: %.0f utt/s" % (r["omp"], r["value"]) for r in runs)))
    print(json.dumps({
        "impl": "reference", "metric": "ctc_fwd_bwd_utterances_per_s", "value": best["value"], "unit": "utterances/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": best["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_for(wl, max(1, args.gpus)),
        "cpu_baseline": {"value": best["value"], "unit": "utterances/s", "cores": cores, "kind": best["kind"], "sample": sample},
        "e2e": {"value": best["value"], "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ----------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------
class Bucket:
    """This rank's share of one global batch of a workload, resident on the device in `n_rot` rotating slots
    (slot 0: the seeded SURVEY 8(d) draw; the others: fresh N(0,1) logits for the same labels and lengths)."""

    def __init__(self, wl, dev, rank, world, per_rank_batch=None, max_rotate=128, global_batch=None):
        import torch
        from end2end_b200.distributed import plan_shards
        B, T, V, Lmin, Lmax, seed, dt, full, desc = WORKLOADS[wl]
        if per_rank_batch:
            B = per_rank_batch
        self.wl, self.T, self.V, self.dt = wl, T, V, dt
        self.dtype = {"f32": torch.float32, "bf16": torch.bfloat16}[dt]
        self.esize = 2 if dt == "bf16" else 4
        if global_batch is None:                       # weak scaling: every rank contributes one workload batch
            parts = [make_inputs(B, T, V, Lmin, Lmax, seed + 7919 * r, self.dtype, full) for r in range(world)]
            gx, gtg, gll, gtl = (torch.cat([p[i] for p in parts]) for i in range(4))
        else:                                          # strong scaling: one workload batch over all the ranks
            gx, gtg, gll, gtl = make_inputs(global_batch, T, V, Lmin, Lmax, seed, self.dtype, full)
        self.global_B = gx.size(0)
        self.buckets = plan_shards(gll, gtl, V, world)
        idx = torch.tensor(self.buckets[rank], dtype=torch.int64)
        self.cpu = (gx[idx], gtg[idx], gll[idx], gtl[idx])
        self.B = idx.numel()
        self.tg, self.ll, self.tl = (t.to(dev) for t in self.cpu[1:])
        batch_bytes = self.B * T * V * self.esize
        self.alg_bytes = 2 * batch_bytes               # logits read + gradient write (SURVEY 8d)
        n_rot = max(2, min(max_rotate, -(-2 * L2_BYTES // (2 * batch_bytes))))
        self.flush = 2 * batch_bytes * n_rot < 2 * L2_BYTES      # too small to out-stream L2 by rotation
        if self.flush:
            n_rot = 2
        if 2 * batch_bytes * n_rot > 24 * 2 ** 30:
            n_rot = max(1, (24 * 2 ** 30) // (2 * batch_bytes))
        self.n_rot = n_rot
        gen = torch.Generator(device=dev).manual_seed(seed + 1000003 * rank + 17)
        self.x = [self.cpu[0].to(dev)]
        for _ in range(1, n_rot):
            self.x.append(torch.randn(self.B, T, V, generator=gen, device=dev, dtype=torch.float32).to(self.dtype))
        self.l2_note = ("L2 flushed between steps (256 MB write), every step timed with its own CUDA events" if self.flush else
                        "rotating %d distinct resident batches (%.0f MB of logits + gradients streamed between reuses > 126 MB L2)"
                        % (n_rot, n_rot * 2 * batch_bytes / 2 ** 20))


def oracle_reference(x, tg, ll, tl, dtype_is_bf16, sub=64):
    """(losses, d loss_b / d logits) of the reference for raw logits, the oracle sub-batched."""
    import torch
    import oracle
    losses, grads = [], []
    eng = oracle.engine(0)
    for i in range(0, x.size(0), sub):
        sl = slice(i, i + sub)
        lp = torch.log_softmax(x[sl].float(), 2)
        l_, g_ = eng.compute(lp, tg[sl], ll[sl], tl[sl])
        for r_, n_ in enumerate(ll[sl].tolist()):      # log_softmax backward: ~0 on the padding rows (SURVEY 8a notes)
            g_[r_, n_:] = 0
            if not torch.isfinite(l_[r_]):
                g_[r_] = float("nan")
        losses.append(l_); grads.append(g_)
    return torch.cat(losses), torch.cat(grads), eng.kind


def parity_check(bk, crit, dev, world, n_chk):
    """Before anything is timed: this rank's bucket through the autograd path and through the captured step, against
    the CPU oracle (first n_chk utterances: losses and gradients; the whole bucket's loss sum when it is small enough),
    and the all-reduced loss against the oracle's global mean.  Raises on a mismatch."""
    import torch
    x, tg, ll, tl = bk.cpu
    n = min(n_chk, bk.B)
    bf16 = bk.dt == "bf16"
    rtol, atol = (2.0 ** -8, 1e-5) if bf16 else (1e-5, 1e-5)
    l_ref, g_ref, kind = oracle_reference(x[:n], tg[:n], ll[:n], tl[:n], bf16)
    scale = 1.0 / bk.global_B
    leaf = bk.x[0].detach().clone().requires_grad_()
    loss = crit(leaf, bk.tg, bk.ll, bk.tl)
    loss.backward()
    step = crit.graphed(bk.x[0], bk.tg, bk.ll, bk.tl)
    g_loss, g_grad = step.replay()
    if hasattr(step, "wait"):
        step.wait()
    torch.cuda.synchronize()
    out = {"world": world, "oracle": kind, "utterances_checked_per_rank": n, "rtol": rtol, "atol": atol}
    worst = 0.0
    for name, grad in (("autograd", leaf.grad), ("graph", g_grad)):
        err = (grad[:n].detach().float().cpu().double() - (g_ref * scale).double()).abs()
        tol = atol * scale + rtol * (g_ref * scale).double().abs()
        bad = int((err > tol).sum())
        out["max_grad_err_" + name] = float(err.max()) / scale          # in units of d loss_b / d logits
        worst = max(worst, bad)
        if bad:
            raise AssertionError("parity check failed (%s path): %d gradient elements outside tolerance, max err %.3e"
                                 % (name, bad, float(err.max()) / scale))
    # the reduced loss: local sum of oracle losses over the whole bucket (when affordable), all-reduced on the host side
    if bk.B * bk.T <= 256 * 400 + 1 and n < bk.B:
        l_all = oracle_reference(x, tg, ll, tl, bf16)[0]
    else:
        l_all = l_ref if n == bk.B else None
    if l_all is not None:
        tot = torch.tensor([float(l_all.double().sum())], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(tot)
        ref_mean = float(tot.item()) / bk.global_B
        for name, v in (("autograd", float(loss.detach())), ("graph", float(g_loss))):
            lim = (2.0 ** -8 if bf16 else 1e-5) * abs(ref_mean) + 1e-5
            out["loss_" + name] = v
            if not abs(v - ref_mean) <= lim:
                raise AssertionError("parity check failed: %s loss %.6f vs oracle global mean %.6f" % (name, v, ref_mean))
        out["loss_oracle_global_mean"] = ref_mean
    out["ok"] = True
    del step
    return out


def timed_replays(steps_fn, n_steps, bk, dev, barrier, flush_buf, after=None):
    """Time n_steps calls of steps_fn(i) on the current stream with CUDA events.  Rotation workloads: ONE event pair
    around the whole region; flush workloads: an event pair per step with an L2 flush in between (not timed)."""
    import torch
    if not bk.flush:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(n_steps):
            steps_fn(i)
        if after:
            after()
        e1.record()
        barrier()
        return e0.elapsed_time(e1)
    pairs = []
    barrier()
    for i in range(n_steps):
        flush_buf.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        steps_fn(i)
        if after:
            after()
        b.record()
        pairs.append((a, b))
    barrier()
    return sum(a.elapsed_time(b) for a, b in pairs)


def measure_bucket(bk, dev, world, steps, warmup, barrier, flush_buf, with_autograd=True, profile_steps=20,
                   keep_outputs=False):
    """value / per-kernel times of one workload on this rank's bucket (max over ranks is taken by the caller).
    keep_outputs: also return, copied to the host, the (loss, grad) the last timed replay produced."""
    import torch
    from end2end_b200 import CTCLoss, _lib
    from end2end_b200.distributed import ShardedCTCLoss
    if world > 1:
        crit = ShardedCTCLoss(reduce=True, size_average=True, after_logsoftmax=False, global_batch=bk.global_B)
    else:
        crit = CTCLoss(reduce=True, size_average=True, after_logsoftmax=False)
    eng = crit._engine
    ws = torch.empty(eng.workspace_bytes(bk.x[0], bk.tg, bk.ll, bk.tl, True), dtype=torch.uint8, device=dev)
    graphs = [crit.graphed(x, bk.tg, bk.ll, bk.tl, workspace=ws) for x in bk.x]     # replayed one after another: one scratch
    n = len(graphs)

    def replay(i):
        return graphs[i % n].replay()

    def join():                                       # the side-stream all-reduces belong to the timed region
        if world > 1:
            for g in graphs[-2:] if n >= 2 else graphs:
                g.wait()

    for i in range(max(3, warmup, n)):
        replay(i)
    join()
    torch.cuda.synchronize()
    res = {}
    l0 = _lib.launch_count()
    ms = timed_replays(replay, steps, bk, dev, barrier, flush_buf, after=join)
    res["launches"] = _lib.launch_count() - l0
    res["ms"] = ms
    res["loss"] = float(graphs[(steps - 1) % n].loss if hasattr(graphs[0], "loss") else graphs[(steps - 1) % n].total)
    if keep_outputs:
        last = graphs[(steps - 1) % n]
        res["outputs"] = ((last.loss if hasattr(last, "loss") else last.total).cpu(), last.grad.cpu())
    if with_autograd:
        leaves = [x.detach().requires_grad_() for x in bk.x]

        def auto(i):
            x = leaves[i % n]
            x.grad = None
            loss = crit(x, bk.tg, bk.ll, bk.tl)
            loss.backward()
            return loss
        for i in range(max(3, n)):
            auto(i)
        res["autograd_ms"] = timed_replays(auto, steps, bk, dev, barrier, flush_buf)
    # per-kernel device times, live, with the library's event hooks (the plain launch sequence, no graph)
    _lib.profile_enable(True)
    _lib.profile_read()
    scale = 1.0 / bk.global_B
    for i in range(min(steps, profile_steps)):
        if bk.flush:
            flush_buf.add_(1)
        eng.step(bk.x[i % n], bk.tg, bk.ll, bk.tl, True, scale, scale)
    torch.cuda.synchronize()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    res["kernel_ms"] = {k: v[0] / v[1] for k, v in prof.items() if v[1]}
    res["crit"] = crit
    del graphs
    return res


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(dirname, loss, grad, rank, world):
    """Write what the last timed step returned to its caller -- the reduced loss and d loss / d logits -- as
    <dirname>/loss.npy and grad.npy (float32; float64 for float64 logits), so that two builds can be compared on the
    same seeded inputs.  A gradient larger than the budget (64 MB over all ranks) is cut to a seeded sample of whole
    utterances, whose batch indices go to grad_utterances.npy.  Under torchrun every rank writes its bucket's
    outputs with a _rank<r> suffix."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    out_dtype = torch.float64 if grad.dtype == torch.float64 else torch.float32
    row_bytes = grad[0].numel() * (8 if out_dtype == torch.float64 else 4)
    keep = max(1, (DUMP_BYTES // world - 4096) // (row_bytes + 8))     # 4 kB: .npy headers and the loss
    arrays = {"loss": loss.to(out_dtype)}
    if grad.size(0) > keep:
        idx = torch.randperm(grad.size(0), generator=torch.Generator().manual_seed(0))[:keep].sort().values
        grad = grad[idx]
        arrays["grad_utterances"] = idx.to(torch.float64)
    arrays["grad"] = grad.to(out_dtype)
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + suffix + ".npy"), t.numpy())


def roofline_block(bk, res, steps, peak, peak_src, wl):
    kern = res["kernel_ms"]
    dominant = max(kern, key=kern.get)
    step_ms = res["ms"] / steps
    stream_ms = sum(v for k, v in kern.items() if k in ("row_stats", "lattice", "gradient"))
    # one launch of the dominant kernel processes the whole bucket; for a multi-kernel pipeline (large alphabets:
    # row statistics + lattice + gradient) the bytes are charged to the pipeline's kernels together
    t_ms = stream_ms if len([k for k in kern if k in ("row_stats", "gradient")]) else kern[dominant]
    achieved = bk.alg_bytes / (t_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": recorded_traffic(wl), "peak_source": peak_src, "algorithmic_bytes_per_launch": bk.alg_bytes,
            "kernel_ms": kern, "timed_over": "row_stats + lattice + gradient" if t_ms == stream_ms and t_ms != kern[dominant] else dominant,
            "step_frac": bk.alg_bytes / (step_ms * 1e-3) / 1e9 / peak}


def run_ours(args, wl):
    import torch
    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the CTC engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        # The only collective of this path is a scalar all-reduce: NVLink SHARP multicast buys nothing, and its
        # set-up makes a TWO-rank communicator on a larger NVSwitch box 2-3x slower per step (measured:
        # profiles/r01/scale_r01e.md).  NCCL caches the setting at the first communicator, so it is set here.
        if world == 2:      # with 4 or 8 ranks the in-switch reduction helps (8 ranks: 0.167 vs 0.219 ms/step)
            os.environ.setdefault("NCCL_NVLS_ENABLE", "0")
        dist.init_process_group("nccl", device_id=dev)
    from end2end_b200 import CTCGreedyEngine, CTCLossEngine, _lib

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    peak, peak_src = measured_peak()
    flush_buf = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)
    B0, T, V = WORKLOADS[wl][:3]
    bk = Bucket(wl, dev, rank, world, per_rank_batch=args.batch or None, max_rotate=args.max_rotate)

    # ---- parity first: this rank's bucket against the oracle, the all-reduced loss against the global mean ----
    from end2end_b200 import CTCLoss
    from end2end_b200.distributed import ShardedCTCLoss
    crit0 = (ShardedCTCLoss(reduce=True, size_average=True, after_logsoftmax=False, global_batch=bk.global_B) if world > 1
             else CTCLoss(reduce=True, size_average=True, after_logsoftmax=False))
    n_chk = args.check if args.check >= 0 else (8 if bk.T > 1000 else 64)
    parity = parity_check(bk, crit0, dev, world, n_chk) if n_chk else {"ok": None, "skipped": True}
    ok = torch.tensor([1 if parity.get("ok", True) is not False else 0], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
    assert int(ok.item()) == 1, "parity check failed on some rank"

    # ---- the timed region: K replays of the captured step; clocks sampled from before the barrier ----
    try:
        gpu_id = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        gpu_id = str(local_rank)
    sampler = ClockSampler(gpu_id) if rank == 0 else None
    if sampler:
        sampler.wait_first()
    w0 = time.perf_counter()
    res = measure_bucket(bk, dev, world, args.steps, args.warmup, barrier, flush_buf, with_autograd=False, profile_steps=0,
                         keep_outputs=bool(args.dump_outputs))
    w1 = time.perf_counter()
    clocks = sampler.summary(w0, w1) if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res.pop("outputs"), rank, world)
    ms = max_over_ranks(res["ms"])
    assert res["loss"] == res["loss"] and abs(res["loss"]) != float("inf"), "non-finite loss in the timed region"
    launches = res["launches"]
    # autograd path + per-kernel times (separate passes, not part of `value`)
    res2 = measure_bucket(bk, dev, world, args.steps, args.warmup, barrier, flush_buf, with_autograd=True)
    auto_ms = max_over_ranks(res2["autograd_ms"])
    res["kernel_ms"] = res2["kernel_ms"]
    roofline = roofline_block(bk, res, args.steps, peak, peak_src, wl)

    # ---- end to end through the engine call on HOST buffers (pinned), copies inside the timing ----
    eng = CTCLossEngine(0)
    hx, htg, hll, htl = (t.pin_memory() for t in bk.cpu)
    for _ in range(max(3, min(args.warmup, 20)) + 20):     # the pinned result blocks reach their steady state (recycled, not re-pinned)
        hl, hg = eng.compute(hx, htg, hll, htl, from_logits=True)
    barrier()
    esteps = max(1, min(args.steps, 50))
    t0 = time.perf_counter()
    for _ in range(esteps):
        hl, hg = eng.compute(hx, htg, hll, htl, from_logits=True)
        float(hl[0])                                   # the result is on the host when compute() returns
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    h2d, d2h = eng.last_host_traffic()
    e2e_value = bk.global_B * esteps / e2e_s
    del hx, hg

    extras = {}
    # ---- strong scaling: c3 at its FIXED global batch, sharded over the ranks by plan_shards ----
    if not args.no_extras:
        sB = WORKLOADS["c3"][0]
        sbk = Bucket("c3", dev, rank, world, max_rotate=64, global_batch=sB)     # enough slots to stay in rotation mode at 8 ranks
        sres = measure_bucket(sbk, dev, world, 20, 3, barrier, flush_buf, with_autograd=False, profile_steps=0)
        s_ms = max_over_ranks(sres["ms"]) / 20
        extras["strong"] = {"workload": "c3: " + WORKLOADS["c3"][8], "global_batch": sB, "bucket_sizes": [len(b) for b in sbk.buckets],
                            "value": sB / (s_ms * 1e-3), "unit": "utterances/s", "ms_per_step": s_ms, "scaling": "strong",
                            "step_frac": 2 * sB * WORKLOADS["c3"][1] * WORKLOADS["c3"][2] * 2 / (s_ms * 1e-3) / 1e9 / peak / world}
        del sbk, sres
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1:
        # ---- the other BASELINE shapes, one compact block each ----
        if not args.no_extras:
            per = {}
            for w in ("c1", "c2", "c3", "c4", "c5"):
                if w == wl:
                    continue
                try:
                    wb = Bucket(w, dev, 0, 1, max_rotate=32)
                    k = 5 if w == "c5" else 30
                    r = measure_bucket(wb, dev, 1, k, 3, barrier, flush_buf, with_autograd=False, profile_steps=min(k, 10))
                    rf = roofline_block(wb, r, k, peak, peak_src, w)
                    per[w] = {"value": wb.B * k / (r["ms"] * 1e-3), "ms_per_step": r["ms"] / k, "batch": wb.B, "step_frac": rf["step_frac"],
                              "frac": rf["frac"], "kernel_ms": {a: round(b, 5) for a, b in rf["kernel_ms"].items()}, "l2": wb.l2_note}
                    del wb, r
                except RuntimeError as err:            # e.g. out of memory on a smaller part
                    per[w] = {"error": str(err)[:200]}
                torch.cuda.empty_cache()
            extras["per_workload"] = per
            # ---- greedy decode of the c4 logits (BASELINE configs[3]) ----
            Bg, Tg, Vg, Lmin, Lmax, seed = WORKLOADS["c4"][:6]
            xs = [make_inputs(Bg, Tg, Vg, Lmin, Lmax, seed, torch.float32, False)]
            gx = [xs[0][0].to(dev), torch.randn(Bg, Tg, Vg, device=dev)]
            gll = xs[0][2].to(dev)
            dec = CTCGreedyEngine(0)
            for i in range(4):
                dec.decode_greedy_device(gx[i % 2], gll)
            _lib.profile_enable(True); _lib.profile_read()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(20):
                dec.decode_greedy_device(gx[i % 2], gll)
            e1.record()
            torch.cuda.synchronize()
            gprof = _lib.profile_read(); _lib.profile_enable(False)
            g_ms = e0.elapsed_time(e1) / 20
            g_bytes = Bg * Tg * Vg * 4 + Bg * Tg * 8 + Bg * 8          # SURVEY 8d: 131,329,024 B
            hxg = xs[0][0].pin_memory()
            hlg = xs[0][2]
            for _ in range(2):
                dec.decode_greedy(hxg, hlg)
            t0 = time.perf_counter()
            for _ in range(10):
                dec.decode_greedy(hxg, hlg)
            g_e2e = Bg * 10 / (time.perf_counter() - t0)
            extras["greedy"] = {"workload": "c4 greedy decode (argmax + collapse repeats / drop blank), B=%d T=%d V=%d fp32" % (Bg, Tg, Vg),
                                "value": Bg / (g_ms * 1e-3), "unit": "utterances/s", "ms_per_step": g_ms,
                                "algorithmic_bytes": g_bytes, "achieved_gbs": g_bytes / (g_ms * 1e-3) / 1e9,
                                "frac": g_bytes / (g_ms * 1e-3) / 1e9 / peak,
                                "kernel_ms": {k: v[0] / v[1] for k, v in gprof.items() if v[1]},
                                "e2e_value": g_e2e, "l2": "two distinct 131 MB logit blocks alternate (> 126 MB L2)"}
            del gx, hxg
            torch.cuda.empty_cache()
            # ---- Viterbi forced alignment (SURVEY 8(f2)) of the c2 batch's log-probabilities ----
            from end2end_b200.utils.alignment import get_alignment_3d_device
            import oracle
            Ba, Ta, Va, Lmin, Lmax, seed = WORKLOADS["c2"][:6]
            ax, atg, all_, atl = make_inputs(Ba, Ta, Va, Lmin, Lmax, seed, torch.float32, False)
            alp = torch.log_softmax(ax, 2)
            dlp, dtg, dll, dtl = alp.to(dev), atg.to(dev), all_.to(dev), atl.to(dev)
            got = get_alignment_3d_device(dlp, dtg, dll, dtl)
            want = oracle.get_alignment_3d(alp, atg, all_, atl)
            assert torch.equal(got.cpu(), want), "alignment differs from the oracle"
            _lib.profile_enable(True); _lib.profile_read()
            for i in range(20):
                flush_buf.add_(1)
                get_alignment_3d_device(dlp, dtg, dll, dtl)
            torch.cuda.synchronize()
            aprof = _lib.profile_read(); _lib.profile_enable(False)
            a_ms = aprof["viterbi"][0] / max(1, aprof["viterbi"][1])
            t0 = time.perf_counter()
            for _ in range(3):
                oracle.get_alignment_3d(alp, atg, all_, atl)
            a_cpu = Ba * 3 / (time.perf_counter() - t0)
            # ---- CTC without blank (SURVEY 8(f4)) on the same log-probabilities ----
            from end2end_b200.functions.ctc_without_blank import ctc_without_blank_3d_loss
            nl, ng = ctc_without_blank_3d_loss(dlp, dtg, dll, dtl, -1)
            rl, rg = oracle.ctc_without_blank(alp, atg, all_, atl, -1)
            n_err = float((ng.cpu().double() - rg).abs().max())
            assert n_err <= 1e-5 and float((nl.cpu().double() - rl).abs().max()) <= 1e-5 * float(rl.abs().max()) + 1e-5, "ctc_without_blank differs from the oracle"
            _lib.profile_enable(True); _lib.profile_read()
            for i in range(10):
                flush_buf.add_(1)
                ctc_without_blank_3d_loss(dlp, dtg, dll, dtl, -1)
            torch.cuda.synchronize()
            nprof = _lib.profile_read(); _lib.profile_enable(False)
            n_ms = nprof["ctc_without_blank"][0] / max(1, nprof["ctc_without_blank"][1])
            t0 = time.perf_counter()
            for _ in range(2):
                oracle.ctc_without_blank(alp, atg, all_, atl, -1)
            n_cpu = Ba * 2 / (time.perf_counter() - t0)
            extras["ctc_without_blank"] = {"workload": "CTC-without-blank loss + gradient of the c2 batch, B=%d T=%d V=%d fp32 log-probs, space_idx=-1" % (Ba, Ta, Va),
                                           "value": Ba / (n_ms * 1e-3), "unit": "utterances/s", "kernel_ms": n_ms, "max_grad_err_vs_oracle": n_err,
                                           "algorithmic_bytes": 2 * Ba * Ta * Va * 4, "frac": 2 * Ba * Ta * Va * 4 / (n_ms * 1e-3) / 1e9 / peak,
                                           "cpu_baseline": {"value": n_cpu, "unit": "utterances/s", "kind": "port", "cores": os.cpu_count(),
                                                            "sample": "2 passes of the same batch, C restatement of the reference's numba code, OpenMP over utterances"}}
            a_bytes = Ba * Ta * Va * 4 + Ba * Ta * 8
            extras["alignment"] = {"workload": "Viterbi forced alignment (CTC lattice) of the c2 batch, B=%d T=%d V=%d fp32 log-probs" % (Ba, Ta, Va),
                                   "value": Ba / (a_ms * 1e-3), "unit": "utterances/s", "kernel_ms": a_ms, "bit_exact_vs_oracle": True,
                                   "algorithmic_bytes": a_bytes, "frac": a_bytes / (a_ms * 1e-3) / 1e9 / peak,
                                   "l2": "L2 flushed between launches (256 MB write), kernel timed by the library's event hooks",
                                   "cpu_baseline": {"value": a_cpu, "unit": "utterances/s", "kind": "port", "cores": os.cpu_count(),
                                                    "sample": "3 passes of the same batch, C restatement of the reference's numba code, "
                                                              "OpenMP over utterances (the reference: one Python thread per utterance)"}}
            # ---- LM-free prefix beam search (SURVEY 8(f3)) of the c2 logits, the reference's default beam of 100 ----
            from end2end_b200.engine import CTCBeamEngine
            beng = CTCBeamEngine(0, 100)
            dx = ax.to(dev)
            bdec, blen, bties = beng.decode_device(dx, dll, from_logits=True)
            nb_chk = 4                                   # parity against the oracle on a few utterances (the CPU search is slow)
            want = oracle.beam_decode(ax[:nb_chk], all_[:nb_chk], beam_width=100, after_logsoftmax=False, return_ties=True,
                                      prefer="reference" if oracle.have_ref() else "port")
            for i in range(nb_chk):
                n_i = int(want[1][i])
                assert int(blen[i]) == n_i and bdec[i, :n_i].cpu().tolist() == want[0][i, :n_i].tolist(), "beam search differs from the oracle"
            _lib.profile_enable(True); _lib.profile_read()
            for i in range(5):
                flush_buf.add_(1)
                beng.decode_device(dx, dll, from_logits=True)
            torch.cuda.synchronize()
            bprof = _lib.profile_read(); _lib.profile_enable(False)
            b_ms = bprof["beam_search"][0] / max(1, bprof["beam_search"][1])
            hx = ax.pin_memory()
            beng.decode(hx, all_, from_logits=True)
            t0 = time.perf_counter()
            for _ in range(3):
                beng.decode(hx, all_, from_logits=True)
            b_e2e = Ba * 3 / (time.perf_counter() - t0)
            t0 = time.perf_counter()
            nb_cpu = min(Ba, 2 * (os.cpu_count() or 1))
            oracle.beam_decode(ax[:nb_cpu], all_[:nb_cpu], beam_width=100, after_logsoftmax=False)
            b_cpu = nb_cpu / (time.perf_counter() - t0)
            extras["beam_search"] = {"workload": "LM-free prefix beam search (beam_width 100) of the c2 logits, B=%d T=%d V=%d fp32, log-softmax fused" % (Ba, Ta, Va),
                                     "value": Ba / (b_ms * 1e-3), "unit": "utterances/s", "kernel_ms": b_ms, "e2e_value": b_e2e,
                                     "bit_exact_vs_oracle": True, "checked_utterances": nb_chk, "ties": int(bties.sum()),
                                     "l2": "L2 flushed between launches (256 MB write), kernel timed by the library's event hooks",
                                     "cpu_baseline": {"value": b_cpu, "unit": "utterances/s", "cores": os.cpu_count(),
                                                      "kind": "reference" if oracle.have_ref() else "port",
                                                      "sample": "%d utterances of the same batch, one host thread per utterance (the reference's pool)" % nb_cpu}}
            del dx, hx
        if not args.no_cpu_baseline:
            best, runs = measure_reference(wl, 0, 1, args.ref_batch, cpu_seconds=args.cpu_seconds / 2, greedy=False)
            if best:
                cpu_baseline = {"value": best["value"], "unit": "utterances/s", "cores": os.cpu_count(), "kind": best["kind"],
                                "sample": "%d utterances of %s x %d passes (%.1f s), one host thread per utterance (the reference's pool) "
                                          "on %d cores, OMP_NUM_THREADS=%s (the better of %s)"
                                          % (best["sample_B"], wl, best["steps"], best["steps"] * best["ms_per_step"] / 1e3, os.cpu_count(), best["omp"],
                                             ", ".join("%s: %.0f utt/s" % (r["omp"], r["value"]) for r in runs))}
            if "greedy" in extras:
                gb, _ = measure_reference("c4", 0, 0, 16, cpu_seconds=2.0, greedy=True)
                if gb and gb.get("greedy"):
                    extras["greedy"]["cpu_baseline"] = {"value": gb["greedy"]["value"], "unit": "utterances/s", "kind": gb["greedy"]["kind"],
                                                        "omp": gb["omp"], "cores": os.cpu_count()}

    if rank == 0:
        cfg = config_for(wl, world)
        line = {
            "metric": "ctc_fwd_bwd_utterances_per_s", "value": bk.global_B * args.steps / (ms * 1e-3),
            "unit": "utterances/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg,
            "step": "criterion.graphed(...).replay(): CUDA graph of {status memset, lattice kernel(s), loss reduction}"
                    + (" + scalar all-reduce on a side stream" if world > 1 else ""),
            "l2": bk.l2_note, "bucket_sizes": [len(b) for b in bk.buckets],
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "utterances/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "CTCLossEngine.compute(host pinned tensors, from_logits=True) -> e2e_ctc_engine_loss_host"},
            "gpu_launches": launches,
            "autograd": {"value": bk.global_B * args.steps / (auto_ms * 1e-3), "ms_per_step": auto_ms / args.steps,
                         "api": "loss = CTCLoss(...)(logits, ...); loss.backward()"},
            "roofline": roofline,
            "parity_check": parity,
            "cpu_baseline": cpu_baseline,
        }
        line.update(extras)
        out_line = json.dumps(line)
    else:
        out_line = None
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return out_line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override the workload's per-GPU batch size (experiments)")
    ap.add_argument("--max-rotate", type=int, default=128)
    ap.add_argument("--ref-batch", type=int, default=64, help="utterances per reference-CPU step (bounded sample)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--check", type=int, default=-1, help="utterances per rank compared with the oracle before timing (0: skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per_workload / greedy / strong blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the loss and gradient of the last timed step to DIR/<name>.npy (at most 64 MB)")
    ap.add_argument("--greedy", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--_child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    _, _, world = dist_env()
    if args.gpus != world and world > 1:
        args.gpus = world
    if args.impl == "reference":
        if args._child:
            reference_child(args)
        else:
            run_reference(args, args.workload)
    else:
        os.environ.setdefault("OMP_NUM_THREADS", "1")     # our arm's host side is single-threaded issue work
        # ONE JSON line on stdout, whatever the libraries underneath print (NCCL writes its version banner to stdout):
        # everything else this process writes to fd 1 goes to stderr, the line itself to the real stdout
        sys.stdout.flush()
        real_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            line = run_ours(args, args.workload)
        finally:
            sys.stdout.flush()
            os.dup2(real_stdout, 1)
            os.close(real_stdout)
        if line is not None:
            print(line, flush=True)


if __name__ == "__main__":
    main()

"""Time the edit-distance kernel (K11) and the MWER step it serves.

    python tools/edit_distance_time.py [--launches 50] [--steps 5] [--out results/edit_distance_time.json]

Inputs: the seeded c2 (B=64, T=400, V=29) and c4 (B=128, T=250, V=1024) batches of oracle.CONFIGS, decoded with
CTCDecoder.decode_nbest (beam 100) and compared with their own targets; c2 at N in {1, 10, 100}, c4 at N in {1, 10};
token level, and word level with label 1 standing in for the space.  Per case:
  kernel_ms: K11's device time per launch from the library's CUDA-event hooks, averaged over --launches launches after
             two warm-up launches;
  host_ms:   the C restatement (tests/edit_distance_restatement.c, gcc -O2 into a temporary directory) on the host, per
             call, the N-best list already on the host;
and the kernel's counts are checked against the restatement's.  Then a whole MWER step on c2 with word errors at
N in {10, 100}: decode_nbest_device -> risk -> CTCScore forward and backward of the expected risk, the risk computed on
the host (copy the list out, restatement, copy the risk in) or on the device (errors_device); host clock around each
step, which ends in a device synchronise, median of --steps steps after one warm-up.  The card's name, power limit and
max SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = (("c2", 1), ("c2", 10), ("c2", 100), ("c4", 1), ("c4", 10))
BEAM = 100
SPACE = 1


def restatement():
    d = tempfile.mkdtemp(prefix="edit_distance_time_")
    so = os.path.join(d, "librestatement.so")
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", so, os.path.join(ROOT, "tests", "edit_distance_restatement.c")])
    L = ctypes.CDLL(so)
    shutil.rmtree(d, True)                       # the library stays mapped
    ip, i, i64 = ctypes.POINTER(ctypes.c_int64), ctypes.c_int, ctypes.c_int64
    L.edit_restatement.argtypes = [i, i, ip, i, ip, ip, i, ip, i64, ip, ip, ip, ip, ip]
    L.edit_restatement.restype = None
    return L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import oracle
    from end2end_b200 import CTCScore, _lib
    from end2end_b200.engine import CTCBeamEngine
    from end2end_b200.utils.hypotheses import empty_marker_as_empty
    if not torch.cuda.is_available():
        raise SystemExit("edit_distance_time.py measures on the GPU; no CUDA device here")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    R = restatement()
    iptr = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))      # noqa: E731

    def host_counts(hyps, hl, refs, rl, sep):
        h = np.ascontiguousarray(hyps.numpy().astype(np.int64))
        r = np.ascontiguousarray(refs.numpy().astype(np.int64))
        hl_, rl_ = np.ascontiguousarray(hl.numpy().astype(np.int64)), np.ascontiguousarray(rl.numpy().astype(np.int64))
        B, N, W = h.shape
        outs = [np.zeros((B, N), dtype=np.int64) for _ in range(4)] + [np.zeros(B, dtype=np.int64)]
        R.edit_restatement(B, N, iptr(h), W, iptr(hl_), iptr(r), r.shape[1], iptr(rl_), sep, *(iptr(o) for o in outs))
        return [torch.from_numpy(o) for o in outs]

    rows, batches = [], {}
    for cfg, N in CASES:
        if cfg not in batches:
            x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS[cfg][:6])
            eng = CTCBeamEngine(0, BEAM, ["_", " "] + ["x"] * (x.size(2) - 2))
            dec, dl, _, _, _ = eng.decode_nbest_device(x.cuda(), ll.cuda(), n_best=BEAM, from_logits=True)
            batches[cfg] = (eng, x, tg, ll, tl, dec, dl)
        eng, x, tg, ll, tl, dec, dl = batches[cfg]
        hyps, hl = dec[:, :N].contiguous(), dl[:, :N].contiguous()
        hl = empty_marker_as_empty(hyps, hl)
        width = int(hl.max())
        hyps = hyps[:, :, :max(width, 1)].contiguous()
        refs, rls = tg.cuda(), tl.cuda()
        hh, hlh = hyps.cpu(), hl.cpu()
        for level, words in (("token", False), ("word", True)):
            for _ in range(2):
                out = eng.errors_device(hyps, hl, refs, rls, words=words)
            torch.cuda.synchronize()
            _lib.profile_enable(True)
            _lib.profile_read()
            for _ in range(a.launches):
                eng.errors_device(hyps, hl, refs, rls, words=words)
            prof = _lib.profile_read()
            _lib.profile_enable(False)
            ms, cnt = prof["edit_distance"]
            t0 = time.perf_counter()
            reps = 0
            while True:
                want = host_counts(hh, hlh, tg, tl, SPACE if words else -1)
                reps += 1
                if time.perf_counter() - t0 > 0.5 or reps >= 20:
                    break
            host_ms = (time.perf_counter() - t0) * 1e3 / reps
            same = all(torch.equal(o.cpu(), w) for o, w in zip(out, want))
            rows.append({"config": cfg, "N": N, "level": level, "hyp_width": hyps.size(2), "ref_width": tg.size(1),
                         "kernel_ms": ms / max(cnt, 1), "launches": cnt, "host_ms": host_ms, "counts_equal": same,
                         "mean_errors": float(out[0].double().mean()), "reference_units": int(out[4].sum())})
            print(json.dumps(rows[-1]), flush=True)

    # the whole MWER step on c2, word errors
    eng, x, tg, ll, tl, _, _ = batches["c2"]
    xs, lls, tgs, tls = x.cuda(), ll.cuda(), tg.cuda(), tl.cuda()
    mwer = []
    for N in (10, 100):
        def step(on_device):
            dec, dl, scores, _, _ = eng.decode_nbest_device(xs, lls, n_best=N, from_logits=True)
            dl = empty_marker_as_empty(dec, dl)
            if on_device:
                risk = eng.errors_device(dec, dl, tgs, tls, words=True)[0].double()
            else:
                risk = host_counts(dec.cpu(), dl.cpu(), tg, tl, SPACE)[0].double().cuda()
            xa = xs.detach().requires_grad_()
            s = CTCScore()(xa, dec, dl, lls)
            p = torch.softmax(s.masked_fill(scores == -float("inf"), float("-inf")), dim=1)
            (p * risk).sum().backward()
            torch.cuda.synchronize()
            return xa.grad

        times = {"host": [], "device": []}
        grads = {}
        for arm in ("host", "device"):
            grads[arm] = step(arm == "device")
        for _ in range(a.steps):
            for arm in ("host", "device"):                 # alternating
                t0 = time.perf_counter()
                step(arm == "device")
                times[arm].append((time.perf_counter() - t0) * 1e3)
        mwer.append({"config": "c2", "N": N, "host_risk_ms": statistics.median(times["host"]),
                     "device_risk_ms": statistics.median(times["device"]), "host_runs": times["host"],
                     "device_runs": times["device"], "grads_equal": bool(torch.equal(grads["host"], grads["device"]))})
        print(json.dumps(mwer[-1]), flush=True)

    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi (name, power.limit, clocks.max.sm)": smi[:1],
              "kernel": rows, "mwer_step": mwer}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report["nvidia_smi (name, power.limit, clocks.max.sm)"]))


if __name__ == "__main__":
    main()

"""Time an MWER training step two ways: INTEGRATION's composed recipe against the packaged MWERLoss.

    python tools/mwer_time.py [--steps 10] [--out results/mwer_time.json]

Inputs: the seeded c2 (B=64, T=400, V=29, fp32) and c4 (B=128, T=250, V=1024, fp32) batches of oracle.CONFIGS, each with
its own decode_nbest_device list (beam 100, raw logits) cut to N in {1, 4, 8, 16, 100}, unfilled slots masked out, word
errors against the batch's targets with label 1 as the space.  The list is decoded once per case, outside the step: both
arms share it.  The arms, per step (forward and backward into the logits, risk included):
  composed: errors_device -> CTCScore -> masked softmax -> (p * risk).sum() -> autograd (K11, K9, K10 + rows, torch glue);
  packaged: MWERLoss(reduce=True) -> backward (K11, K12a, K12b, K12c + rows).
Per case:
  step_ms:    host clock around a step that ends in a device synchronise; arms alternating, two warm-up steps each,
              median and [min, max] of --steps steps;
  kernels_ms: the library's CUDA-event times per kernel kind over one further step of each arm;
  peak_mb:    torch's peak allocated device memory during one step, above what was allocated before it;
  state_mb:   MWERLoss's state (scores, weights, checkpoints), held from forward to backward;
and the two arms' gradients must agree within 1e-10 relative to the gradient's largest magnitude, plus 1e-14 absolute:
where every list's risks are equal the packaged gradient is exactly 0 and the composed one the softmax's rounding residue
(asserted).  The card's
name, power limit and max SM clock are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONFIGS = ("c2", "c4")
NS = (1, 4, 8, 16, 100)
BEAM = 100


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    sys.path.insert(0, ROOT)
    import oracle
    from end2end_b200 import CTCScore, MWERLoss, _lib
    from end2end_b200.engine import CTCBeamEngine
    if not torch.cuda.is_available():
        raise SystemExit("mwer_time.py measures on the GPU; no CUDA device here")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rows = []
    for cfg in CONFIGS:
        x, tg, ll, tl = oracle.make_inputs(*oracle.CONFIGS[cfg][:6])
        labels = ["_", " "] + ["x%d" % v for v in range(x.size(2) - 2)]
        eng = CTCBeamEngine(0, BEAM, labels)
        xs, lls, tgs, tls = x.cuda(), ll.cuda(), tg.cuda(), tl.cuda()
        dec_all, dl_all, sc_all, _, _ = eng.decode_nbest_device(xs, lls, n_best=BEAM, from_logits=True)
        score, crit = CTCScore(), MWERLoss(labels, reduce=True)
        for N in NS:
            dec, dl = dec_all[:, :N].contiguous(), dl_all[:, :N].contiguous()
            used = sc_all[:, :N] > float("-inf")

            def composed():
                xa = xs.detach().requires_grad_()
                risk = eng.errors_device(dec, dl, tgs, tls, words=True)[0].double()
                s = score(xa, dec, dl, lls)
                p = torch.softmax(s.masked_fill(~used, float("-inf")), dim=1)
                (p * risk).sum().backward()
                torch.cuda.synchronize()
                return xa.grad

            def packaged():
                xa = xs.detach().requires_grad_()
                crit(xa, dec, dl, lls, tgs, tls, used).backward()
                torch.cuda.synchronize()
                return xa.grad

            arms = {"composed": composed, "packaged": packaged}
            grads = {}
            for name, f in arms.items():
                for _ in range(2):
                    grads[name] = f()
            scale = float(grads["composed"].abs().max())
            diff = float((grads["packaged"] - grads["composed"]).abs().max())
            assert diff <= 1e-10 * scale + 1e-14, (cfg, N, diff, scale)
            del grads
            times = {k: [] for k in arms}
            for _ in range(a.steps):
                for name, f in arms.items():                 # alternating
                    t0 = time.perf_counter()
                    f()
                    times[name].append((time.perf_counter() - t0) * 1e3)
            kernels, peak = {}, {}
            for name, f in arms.items():
                _lib.profile_enable(True)
                _lib.profile_read()
                f()
                prof = _lib.profile_read()
                _lib.profile_enable(False)
                kernels[name] = {k: round(ms, 4) for k, (ms, cnt) in prof.items() if cnt}
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                f()
                peak[name] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)
            st, ws = eng.mwer_workspace_bytes(xs, dec, dl, lls, True)
            row = {"config": cfg, "N": N, "max_grad_diff": diff, "max_grad": scale,
                   "state_mb": round(st / 2 ** 20, 2), "backward_scratch_mb": round(ws / 2 ** 20, 2)}
            for name in arms:
                row[name] = {"step_ms": round(statistics.median(times[name]), 3),
                             "step_ms_range": [round(min(times[name]), 3), round(max(times[name]), 3)],
                             "kernels_ms": kernels[name], "peak_mb": peak[name]}
            rows.append(row)
            print(json.dumps(row), flush=True)
    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi (name, power.limit, clocks.max.sm)": smi[:1],
              "steps": a.steps, "rows": rows}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report["nvidia_smi (name, power.limit, clocks.max.sm)"]))


if __name__ == "__main__":
    main()

"""Time the N-hypothesis CTC scorer against the loss forward on replicated logits.

    python tools/score_time.py [--reps 3] [--launches 10] [--out results/score_time.json]

Shapes: c2 (B=64, T=400, V=29) and c4 (B=128, T=250, V=1024) of oracle.CONFIGS, fp32 raw logits (log-softmax fused).
The hypotheses are the N-best lists of the same batch (CTCDecoder.decode_nbest, beam 100), N in {1, 10, 100}, so their
lengths are what a rescoring caller has.  Two arms per (shape, N):
  score: CTCBeamEngine.score_device (one K9 launch);
  loss:  CTCLossEngine.forward on logits.repeat_interleave(N, 0) with the flattened hypotheses -- the only way to get
         these numbers without the scorer -- every kernel it launches, and its workspace bytes.
Kernel times come from the library's CUDA-event hooks, with L2 flushed (256 MB write) before every launch, averaged over
--launches launches after two warm-up launches; each arm is repeated --reps times and the report gives every repetition
and the range.  The card's name, power limit and max SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = ("c2", "c4")
BEAM = 100
N_HYP = (1, 10, 100)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    sys.path.insert(0, ROOT)
    import oracle
    from end2end_b200 import CTCDecoder, CTCLossEngine, _lib
    from end2end_b200.engine import CTCBeamEngine
    if not torch.cuda.is_available():
        raise SystemExit("score_time.py measures on the GPU; no CUDA device here")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)

    def timed(launch):
        """{kernel kind: mean ms per launch} over a.launches launches, L2 flushed before each."""
        for _ in range(2):
            launch()
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        _lib.profile_read()
        for _ in range(a.launches):
            flush.add_(1)
            launch()
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile_enable(False)
        return {k: ms / a.launches for k, (ms, n) in prof.items() if n}

    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi (name, power.limit, clocks.max.sm)": smi[:1],
              "beam_width": BEAM, "launches": a.launches, "reps": a.reps,
              "l2": "flushed (256 MB write) before every launch", "shapes": {}}
    for name in SHAPES:
        B, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS[name]
        x, _, ll, _ = oracle.make_inputs(B, T, V, Lmin, Lmax, seed, full_length=full)
        x, ll = x.to(dev), ll.to(dev)
        nb = CTCDecoder(beam_width=BEAM).decode_nbest(x, ll, n_best=max(N_HYP))
        shape = {}
        for N in N_HYP:
            hyps = nb.decoded_targets[:, :N].to(dev)
            hl = nb.decoded_targets_lengths[:, :N].to(dev)
            hl = torch.where((hl == 1) & (hyps[:, :, 0] == -1), torch.zeros_like(hl), hl)   # decode's empty result
            hyps = hyps.clamp(min=0).contiguous()
            eng = CTCBeamEngine(0, 1)
            xr = x.repeat_interleave(N, 0)
            tg, tl, llr = hyps.reshape(B * N, -1), hl.reshape(B * N), ll.repeat_interleave(N)
            loss_eng = CTCLossEngine(0)
            sc = eng.score_device(x, hyps, hl, ll, from_logits=True)
            losses, _ = loss_eng.forward(xr, tg, llr, tl, from_logits=True)
            diff = float(((sc.reshape(-1) + losses.double()).abs() / losses.double().abs().clamp(min=1)).max())
            runs = {"score": [], "loss": []}
            for r in range(a.reps):
                arms = [("score", lambda: eng.score_device(x, hyps, hl, ll, from_logits=True)),
                        ("loss", lambda: loss_eng.forward(xr, tg, llr, tl, from_logits=True))]
                for tag, fn in (arms if r % 2 == 0 else arms[::-1]):
                    runs[tag].append(timed(fn))
            res = {"mean_hyp_length": float(hl.double().mean()), "max_hyp_length": int(hl.max()),
                   "max_rel_diff_score_vs_fp32_loss": diff,
                   "score_workspace_bytes": 256,
                   "loss_workspace_bytes": loss_eng.workspace_bytes(xr, tg, llr, tl, from_logits=True),
                   "loss_replicated_logits_bytes": xr.numel() * xr.element_size()}
            for tag in runs:
                tot = [sum(k.values()) for k in runs[tag]]
                res[tag] = {"kernels_ms": runs[tag], "total_ms": tot, "min": min(tot), "max": max(tot)}
            res["speedup_min_over_min"] = res["loss"]["min"] / res["score"]["min"]
            shape["N=%d" % N] = res
            del xr
        report["shapes"][name] = shape
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

"""Time the gradient of the N-hypothesis CTC score against the loss's forward + backward on replicated logits.

    python tools/score_grad_time.py [--reps 3] [--launches 5] [--out results/score_grad_time.json]

Shapes: c2 (B=64, T=400, V=29) and c4 (B=128, T=250, V=1024) of oracle.CONFIGS, fp32 raw logits (log-softmax fused).
The hypotheses are the N-best lists of the same batch (CTCDecoder.decode_nbest, beam 100), N in {1, 10, 100}; the
upstream gradient g[b, n] is random.  Two arms per (shape, N):
  score: CTCBeamEngine.score_device + score_backward_device (K9, then K10 and its row kernel);
  loss:  CTCLossEngine.forward + backward on logits.repeat_interleave(N, 0) with the flattened hypotheses and per-row
         weights -g, then the [B, N, T, V] sum of the gradient blocks -- the way to get this gradient without K10.
Kernel times come from the library's CUDA-event hooks with L2 flushed (256 MB write) before every library call, averaged
over --launches steps after two warm-up steps.  score_backward_device is one call that enqueues K10 and its row kernel back
to back, so the row kernel runs without a flush in between (it reads the partial rows K10 has just written, which are far
larger than L2 at N >= 10).  The loss arm's two torch kernels -- the repeat_interleave copy of the logits and the block
sum -- are timed with CUDA events, each after a flush, and reported as torch_repeat and torch_block_sum.  Each arm is
repeated --reps times, alternating, and the report gives every repetition and the range, the workspace bytes, the peak
torch.cuda.max_memory_allocated of a step (inputs excluded), and the two arms' largest gradient difference.  The card's
name, power limit and max SM clock are read in the same run.
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
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    sys.path.insert(0, ROOT)
    import oracle
    from end2end_b200 import CTCDecoder, CTCLossEngine, _lib
    from end2end_b200.engine import CTCBeamEngine
    if not torch.cuda.is_available():
        raise SystemExit("score_grad_time.py measures on the GPU; no CUDA device here")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)

    def timed(step):
        """{kernel kind: mean ms per step} over a.launches steps, L2 flushed before each library call; step(flush_fn)
        returns {name: ms} of the torch kernels it timed itself."""
        def fl():
            flush.add_(1)
        for _ in range(2):
            step(fl)
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        _lib.profile_read()
        extra = {}
        for _ in range(a.launches):
            for k, ms in step(fl).items():
                extra[k] = extra.get(k, 0.0) + ms
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile_enable(False)
        out = {k: ms / a.launches for k, (ms, n) in prof.items() if n}
        for k, ms in extra.items():
            out[k] = ms / a.launches
        return out

    def peak(step):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        step(lambda: None)
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated(dev) - base

    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi (name, power.limit, clocks.max.sm)": smi[:1],
              "beam_width": BEAM, "launches": a.launches, "reps": a.reps,
              "l2": "flushed (256 MB write) before every library launch", "shapes": {}}
    for name in a.shapes.split(","):
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
            g = torch.randn(B, N, dtype=torch.float64, device=dev, generator=torch.Generator(dev).manual_seed(N))
            eng = CTCBeamEngine(0, 1)
            loss_eng = CTCLossEngine(0)
            tg, tl, llr = hyps.reshape(B * N, -1), hl.reshape(B * N), ll.repeat_interleave(N)
            w = (-g).reshape(B * N).float()

            def score_step(fl):
                fl()
                eng.score_device(x, hyps, hl, ll, from_logits=True)
                fl()
                return eng.score_backward_device(x, hyps, hl, g, ll, from_logits=True), {}

            def loss_step(fl):
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                fl()
                ev[0].record()
                xr = x.repeat_interleave(N, 0)
                ev[1].record()
                fl()
                _, state = loss_eng.forward(xr, tg, llr, tl, from_logits=True)
                fl()
                gr = loss_eng.backward(state, w)
                fl()
                ev[2].record()
                out = gr.view(B, N, T, V).sum(1)
                ev[3].record()
                ev[3].synchronize()
                return out, {"torch_repeat": ev[0].elapsed_time(ev[1]), "torch_block_sum": ev[2].elapsed_time(ev[3])}

            g_score = score_step(lambda: None)[0]
            g_loss = loss_step(lambda: None)[0]
            live = (torch.arange(T, device=dev)[None, :] < ll[:, None])[:, :, None]
            diff = float(((g_score - torch.where(live, g_loss, torch.zeros_like(g_loss))).abs()).max())
            runs = {"score": [], "loss": []}
            for r in range(a.reps):
                arms = [("score", lambda fl: score_step(fl)[1]), ("loss", lambda fl: loss_step(fl)[1])]
                for tag, fn in (arms if r % 2 == 0 else arms[::-1]):
                    runs[tag].append(timed(fn))
            res = {"mean_hyp_length": float(hl.double().mean()), "max_hyp_length": int(hl.max()),
                   "max_abs_grad_diff_score_vs_replicated_loss": diff,
                   "score_backward_workspace_bytes": eng.score_backward_workspace_bytes(x, hyps, hl, ll, from_logits=True),
                   "loss_workspace_bytes": loss_eng.workspace_bytes(x.repeat_interleave(N, 0), tg, llr, tl, from_logits=True),
                   "score_peak_bytes": peak(score_step), "loss_peak_bytes": peak(loss_step)}
            for tag in runs:
                tot = [sum(k.values()) for k in runs[tag]]
                res[tag] = {"kernels_ms": runs[tag], "total_ms": tot, "min": min(tot), "max": max(tot)}
            res["speedup_min_over_min"] = res["loss"]["min"] / res["score"]["min"]
            shape["N=%d" % N] = res
            del g_score, g_loss
            torch.cuda.empty_cache()
        report["shapes"][name] = shape
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

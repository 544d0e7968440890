"""Time phrase biasing inside the prefix beam search, against the same search without it and the parent commit's build.

    python tools/beam_bias_time.py --base-root <checkout of the parent commit, library built> [--reps 3]
                                   [--launches 10] [--out results/beam_bias_time.json]

Data, generated from seeds at run time by tools/beam_lm_tokens_time.py's generators: a vocabulary of 3000 words over
a-z, a corpus of sentences drawn from it (Zipf-like), a 3-gram ARPA model over them, and fp32 raw logits that spell
corpus sentences (every label peaks on one or two frames, then a blank frame, plus N(0, 1) noise).  Phrases are corpus
words drawn at random (seeded), so the logits spell some of them now and then:
  * c2 (B=64, T=400, V=29, labels blank, space, a-z, '): the LM-free search and the character-mode LM, each without a
    bias and with 100 and with 1000 phrases (the words' letters);
  * c4 (B=128, T=250, V=1024 sub-word units): the token-mode LM without a bias and with 100 phrases (the words'
    tokenisation), and the labels the symbol filter extends per frame (ties aside) with and without the phrases.
beam_width 100, N = 100, lmwt 0.8, wip 0.5, oov_penalty -2, weight 1.0 per token.  Every time is the kernel's device time
from the library's CUDA-event hooks (beam_search, beam_search_lm or beam_search_bias), with L2 flushed (256 MB write)
before every launch, averaged over --launches launches after two warm-up launches.  Each repetition runs the parent
build's unbiased c2 calls and this build's calls in fresh processes, alternating their order; the unbiased results of
both builds are compared by hash.  Also reported: PhraseBias's host build time for 1000 and 100,000 phrases, and the
card's name, power limit and max SM clock, read in the same run.
"""
import argparse
import hashlib
import json
import os
import random
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from beam_lm_tokens_time import (BEAM, C2_LABELS, LMWT, MARK, N_BEST, OOVP, SHAPES, WIP, corpus, logits_for,  # noqa: E402
                                 token_labels, tokenize, write_model)

WEIGHT = 1.0


def phrases_for(words, labels, n, seed, marker):
    rng = random.Random(seed)
    picked = rng.sample(words, n)
    if marker is None:
        return [[labels.index(ch) for ch in w] for w in picked]
    return [list(p) for p in dict.fromkeys(tuple(tokenize([w], labels)) for w in picked)]


def child(args):
    import ctypes
    import torch
    sys.path.insert(0, args.root)
    from end2end_b200 import NGramLM, _lib
    from end2end_b200.engine import CTCBeamEngine
    L = _lib.load()
    kinds = {k: i for i, k in enumerate(_lib.KERNEL_KINDS)}
    nk = len(_lib.KERNEL_KINDS)
    dev = torch.device("cuda:0")
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)

    def timed(launch, kind):
        for _ in range(2):
            launch()
        torch.cuda.synchronize()
        ms, cnt = (ctypes.c_double * nk)(), (ctypes.c_uint64 * nk)()
        _lib.check(L.e2e_ctc_profile_enable(1))
        _lib.check(L.e2e_ctc_profile_read(ms, cnt, nk))
        for _ in range(args.launches):
            flush.add_(1)
            launch()
        torch.cuda.synchronize()
        _lib.check(L.e2e_ctc_profile_read(ms, cnt, nk))
        _lib.check(L.e2e_ctc_profile_enable(0))
        assert cnt[kinds[kind]] == args.launches, cnt[kinds[kind]]
        return ms[kinds[kind]] / args.launches

    def digest(out):
        return hashlib.sha1(b"".join(t.detach().cpu().contiguous().view(torch.uint8).numpy().tobytes()
                                     for t in out)).hexdigest()

    data = torch.load(os.path.join(args.data, "%s.pt" % args.shape))
    x, labels = data["x"].to(dev), data["labels"]
    lm = NGramLM.from_arpa(os.path.join(args.data, "model.arpa"))
    eng = CTCBeamEngine(0, BEAM, labels, WIP)
    marker = MARK if args.shape == "c4" else None
    kw = dict(lmwt=LMWT, oov_penalty=OOVP, word_marker=marker)
    arms = [("LM-free", None, 0), ("LM", lm, 0)] if args.shape == "c2" else [("LM", lm, 0)]
    if not args.base:
        from end2end_b200 import PhraseBias
        counts = (100, 1000) if args.shape == "c2" else (100,)
        arms += [(name, m, n) for name, m, _ in list(arms) for n in counts]
    if args.rep % 2:
        arms = arms[::-1]
    res = {}
    for name, m, n in arms:
        key = "%s %d phrases" % (name, n)
        if n == 0 and m is None:
            run, kind = (lambda: eng.decode_nbest_device(x, None, N_BEST, True)), "beam_search"
        elif n == 0:
            run, kind = (lambda: eng.decode_nbest_lm_device(x, m, None, N_BEST, True, **kw)), "beam_search_lm"
        else:
            bias = PhraseBias(data["phrases"][n], WEIGHT, labels=labels)
            run = lambda: eng.decode_nbest_bias_device(x, bias, m, None, N_BEST, True, **kw)   # noqa: E731
            kind = "beam_search_bias"
        res[key + " ms"] = timed(run, kind)
        out = run()
        res[key + " sha1"] = digest(out)
        if n:
            res[key + " top hypotheses with a phrase"] = int((out[6][:, 0] > 0).sum())
            unbiased = eng.decode_nbest_device(x, None, N_BEST, True) if m is None else \
                eng.decode_nbest_lm_device(x, m, None, N_BEST, True, **kw)
            res[key + " top hypotheses changed"] = int(sum(
                a[:k].tolist() != b[:j].tolist() for a, k, b, j in zip(out[0][:, 0], out[1][:, 0].tolist(),
                                                                         unbiased[0][:, 0], unbiased[1][:, 0].tolist())))
    print("RESULT " + json.dumps(res), flush=True)


def filter_labels(labels, phrase_labels):
    """Labels per frame the symbol filter extends every member with in token mode, ties aside: the beam_width + 2 most probable
    continuations and word starts (of no phrase) plus every boundary and phrase label."""
    import torch
    kinds = torch.tensor([0 if i == 0 else (2 if lab == MARK else (1 if lab.startswith(MARK) else 0))
                          for i, lab in enumerate(labels)])
    kinds[0] = -1
    free = torch.ones(len(labels), dtype=torch.bool)
    free[sorted(phrase_labels)] = False
    n = 0
    for k in (0, 1):
        n += min(BEAM + 2, int(((kinds == k) & free).sum()))
    n += int((kinds == 2).sum()) + len(phrase_labels)
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-root", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--base", action="store_true")
    ap.add_argument("--rep", type=int, default=0)
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--shape")
    ap.add_argument("--data")
    a = ap.parse_args()
    if a.child:
        return child(a)
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[:1], "beam_width": BEAM, "n_best": N_BEST,
              "weight": WEIGHT, "launches": a.launches, "l2": "flushed (256 MB write) before every launch", "runs": {}}
    sys.path.insert(0, ROOT)
    from end2end_b200 import PhraseBias
    rng = random.Random(5)
    for n in (1000, 100000):
        ph = list({"".join(rng.choice("abcdefghijklmnopqrstuvwxyz") for _ in range(rng.randint(3, 12))): 0
                   for _ in range(n)})
        t0 = time.perf_counter()
        b = PhraseBias(ph, WEIGHT, labels=C2_LABELS, device="cuda:0")
        report["host build %d phrases" % len(ph)] = {"s": time.perf_counter() - t0, "nodes": b.nodes,
                                                     "n_cols": b.n_cols}
    with tempfile.TemporaryDirectory(prefix="beam_bias_") as md:
        words, sents = corpus()
        report["model_ngrams"] = write_model(os.path.join(md, "model.arpa"), words, sents)
        c4_labels = token_labels(sents, SHAPES["c4"][2])
        B, T, V = SHAPES["c4"]
        c4_phrases = {100: phrases_for(words, c4_labels, 100, 7, MARK)}
        x4 = logits_for(sents, c4_labels, B, T, 3, False)
        torch.save({"x": x4, "labels": c4_labels, "phrases": c4_phrases}, os.path.join(md, "c4.pt"))
        report["c4 labels extended per frame, ties aside"] = {
            "without phrases": filter_labels(c4_labels, set()),
            "100 phrases": filter_labels(c4_labels, {c for p in c4_phrases[100] for c in p})}
        B, T, V = SHAPES["c2"]
        torch.save({"x": logits_for(sents, C2_LABELS, B, T, 1, True), "labels": C2_LABELS,
                    "phrases": {n: phrases_for(words, C2_LABELS, n, 8, None) for n in (100, 1000)}},
                   os.path.join(md, "c2.pt"))
        procs = [("c2 parent", "c2", True, os.path.abspath(a.base_root)), ("c2 this", "c2", False, ROOT),
                 ("c4 this", "c4", False, ROOT)]
        for r in range(a.reps):
            for name, shape, base, root in (procs if r % 2 == 0 else procs[::-1]):
                cmd = [sys.executable, os.path.abspath(__file__), "--base-root", a.base_root, "--child", "--root", root,
                       "--shape", shape, "--data", md, "--launches", str(a.launches), "--rep", str(r)] + \
                      (["--base"] if base else [])
                proc = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
                line = [x for x in proc.stdout.splitlines() if x.startswith("RESULT ")]
                if proc.returncode != 0 or not line:
                    raise SystemExit("%s failed:\n%s\n%s" % (name, proc.stdout, proc.stderr))
                report["runs"].setdefault(name, []).append(json.loads(line[0][7:]))
    summary = {}
    for name, runs in report["runs"].items():
        for key in runs[0]:
            if key.endswith(" ms"):
                v = [run[key] for run in runs]
                summary["%s: %s" % (name, key)] = {"ms": v, "min": min(v), "spread": (max(v) - min(v)) / min(v)}
    for arm in ("LM-free 0 phrases", "LM 0 phrases"):
        shas = {run[arm + " sha1"] for name in ("c2 parent", "c2 this") for run in report["runs"][name]}
        summary["c2 %s identical to the parent build" % arm] = len(shas) == 1
    report["summary"] = summary
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

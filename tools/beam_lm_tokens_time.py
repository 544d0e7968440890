"""Time the prefix beam search with a word n-gram LM over sub-word labels (c4) and over characters (c2, against the
parent commit's build).

    python tools/beam_lm_tokens_time.py --base-root <checkout of the parent commit, library built> [--reps 3]
                                        [--launches 10] [--out results/beam_lm_tokens_time.json]

Data, all generated from seeds at run time: a vocabulary of 3000 words over a-z, a corpus of sentences drawn from it, and a
3-gram ARPA model whose unigrams are the vocabulary and whose bigrams and trigrams are the corpus's (random valid
weights).  Logits spell corpus sentences: every label of the sentence's label sequence peaks (+8) on one or two frames,
followed by a blank frame, plus N(0, 1) noise everywhere, so the decoded words are mostly the model's own.
  * c4 (B=128, T=250, V=1024, fp32 raw logits): blank, the marker U+2581, and 1022 sub-word units (every letter as a
    continuation and as a word start, then the corpus's most frequent word-start and continuation pieces of 2-4
    letters); sentences are tokenised greedily, longest piece first.  Arms: the LM-free N-best list, the token-mode
    LM, and the token-mode LM with the symbol filter off (E2E_CTC_BEAM_NOPREFILTER=1, a process of its own).
  * c2 (B=64, T=400, V=29, fp32 raw logits, labels blank, space, a-z, '): the character-mode LM with this build and
    with the parent's, in alternating processes.
beam_width 100, N = 100, lmwt 0.8, wip 0.5, oov_penalty -2.  Every time is the kernel's device time from the library's
CUDA-event hooks (beam_search or beam_search_lm), with L2 flushed (256 MB write) before every launch, averaged over
--launches launches after two warm-up launches.  The results of arms that must agree are compared by hash, and the share
of decoded words that are out of vocabulary is reported.  The card's name, power limit and max SM clock are read in the
same run.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MARK = "▁"
BEAM, N_BEST, LMWT, WIP, OOVP = 100, 100, 0.8, 0.5, -2.0
SHAPES = {"c4": (128, 250, 1024), "c2": (64, 400, 29)}
C2_LABELS = ["_", " "] + [chr(ord("a") + i) for i in range(26)] + ["'"]


def corpus(seed=1, n_words=3000, n_sents=20000):
    import numpy as np
    rng = np.random.default_rng(seed)
    letters = np.array(list("abcdefghijklmnopqrstuvwxyz"))
    words = set()
    while len(words) < n_words:
        words.add("".join(rng.choice(letters, size=int(rng.integers(1, 9)))))
    words = sorted(words)
    freq = 1.0 / np.arange(1, n_words + 1)                    # Zipf-like word frequencies
    freq /= freq.sum()
    sents = [[words[i] for i in rng.choice(n_words, size=int(rng.integers(3, 14)), p=freq)] for _ in range(n_sents)]
    return words, sents


def write_model(path, words, sents, seed=2):
    import numpy as np
    rng = np.random.default_rng(seed)
    bi, tri = set(), set()
    for s in sents:
        w = ["<s>"] + s + ["</s>"]
        bi.update(zip(w, w[1:]))
        tri.update(zip(w, w[1:], w[2:]))
    uni = ["<s>", "</s>", "<unk>"] + words
    ctx2 = {b for b in bi}
    tri = sorted(t for t in tri if t[:2] in ctx2)
    bi = sorted(bi)
    with open(path, "w") as f:
        f.write("\\data\\\nngram 1=%d\nngram 2=%d\nngram 3=%d\n\n\\1-grams:\n" % (len(uni), len(bi), len(tri)))
        for w in uni:
            f.write("%.4f\t%s\t%.4f\n" % (-99.0 if w == "<s>" else rng.uniform(-6, -1), w, rng.uniform(-1, 0.3)))
        f.write("\n\\2-grams:\n")
        for a, b in bi:
            f.write("%.4f\t%s %s\t%.4f\n" % (rng.uniform(-3, -0.1), a, b, 0.0 if b == "</s>" else rng.uniform(-1, 0.3)))
        f.write("\n\\3-grams:\n")
        for a, b, c in tri:
            f.write("%.4f\t%s %s %s\n" % (rng.uniform(-2, -0.05), a, b, c))
        f.write("\n\\end\\\n")
    return len(uni) + len(bi) + len(tri)


def token_labels(sents, V):
    """blank, the marker, every letter as continuation and word start, then the most frequent pieces."""
    from collections import Counter
    letters = [chr(ord("a") + i) for i in range(26)]
    labels = ["_", MARK] + letters + [MARK + c for c in letters]
    cnt = Counter()
    for s in sents[:5000]:
        for w in s:
            for n in (2, 3, 4):
                if len(w) >= n:
                    cnt[MARK + w[:n]] += 1
                    for i in range(1, len(w) - n + 1):
                        cnt[w[i:i + n]] += 1
    labels += [p for p, _ in cnt.most_common(V - len(labels))]
    assert len(labels) == V
    return labels


def tokenize(words, labels):
    idx = {lab: i for i, lab in enumerate(labels)}
    out = []
    for w in words:
        i, first = 0, True
        while i < len(w):
            for n in (4, 3, 2, 1):
                piece = (MARK if first else "") + w[i:i + n]
                if i + n <= len(w) and piece in idx:
                    out.append(idx[piece])
                    i, first = i + n, False
                    break
    return out


def logits_for(sents, labels, B, T, seed, char_mode):
    """[B, T, V] fp32 raw logits spelling corpus sentences (one after another until the frames run out)."""
    import numpy as np
    import torch
    rng = np.random.default_rng(seed)
    V = len(labels)
    x = rng.standard_normal((B, T, V)).astype(np.float32)
    space = labels.index(" ") if char_mode else None
    k = 0
    for b in range(B):
        t = 0
        while t < T - 3:
            s = sents[(seed * 7919 + k) % len(sents)]
            k += 1
            seq = [c for w in s for c in ([labels.index(ch) for ch in w] + [space])] if char_mode else tokenize(s, labels)
            for c in seq:
                for _ in range(int(rng.integers(1, 3))):
                    if t < T:
                        x[b, t, c] += 8.0
                        t += 1
                if t < T:
                    x[b, t, 0] += 8.0
                    t += 1
    return torch.from_numpy(x)


def child(args):
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
        import ctypes
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
    res = {}
    marker = MARK if args.shape == "c4" else None
    kw = dict(lmwt=LMWT, oov_penalty=OOVP)
    if marker is not None:
        kw["word_marker"] = marker
    if args.arm == "free":
        run = lambda: eng.decode_nbest_device(x, None, N_BEST, True)   # noqa: E731
        res["ms"] = timed(run, "beam_search")
    else:
        run = lambda: eng.decode_nbest_lm_device(x, lm, None, N_BEST, True, **kw)   # noqa: E731
        res["ms"] = timed(run, "beam_search_lm")
        out = run()
        res["oov_words_top"] = int(out[5][:, 0].sum())
        n, sp = 0, labels.index(" ") if marker is None else None
        for row, k in zip(out[0][:, 0].tolist(), out[1][:, 0].tolist()):
            text = "".join(labels[c] for c in row[:k] if c >= 0)
            n += len((text.replace(MARK, " ") if marker else text).split())
        res["words_top"] = n
    res["sha1"] = digest(run())
    print("RESULT " + json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-root", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--root", default=ROOT)
    ap.add_argument("--shape")
    ap.add_argument("--arm")
    ap.add_argument("--data")
    a = ap.parse_args()
    if a.child:
        return child(a)
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[:1], "beam_width": BEAM, "n_best": N_BEST,
              "launches": a.launches, "l2": "flushed (256 MB write) before every launch", "runs": {}}
    with tempfile.TemporaryDirectory(prefix="beam_lm_tokens_") as md:
        words, sents = corpus()
        report["model_ngrams"] = write_model(os.path.join(md, "model.arpa"), words, sents)
        labels = token_labels(sents, SHAPES["c4"][2])
        B, T, V = SHAPES["c4"]
        torch.save({"x": logits_for(sents, labels, B, T, 3, False), "labels": labels}, os.path.join(md, "c4.pt"))
        B, T, V = SHAPES["c2"]
        torch.save({"x": logits_for(sents, C2_LABELS, B, T, 1, True), "labels": C2_LABELS}, os.path.join(md, "c2.pt"))
        arms = [("c4 LM-free", "c4", "free", ROOT, {}), ("c4 token LM", "c4", "lm", ROOT, {}),
                ("c4 token LM, filter off", "c4", "lm", ROOT, {"E2E_CTC_BEAM_NOPREFILTER": "1"}),
                ("c2 character LM, this build", "c2", "lm", ROOT, {}),
                ("c2 character LM, parent build", "c2", "lm", os.path.abspath(a.base_root), {})]
        for r in range(a.reps):
            for name, shape, arm, root, env in (arms if r % 2 == 0 else arms[::-1]):
                cmd = [sys.executable, os.path.abspath(__file__), "--base-root", a.base_root, "--child", "--root", root,
                       "--shape", shape, "--arm", arm, "--data", md, "--launches", str(a.launches)]
                proc = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, env=dict(os.environ, **env))
                line = [x for x in proc.stdout.splitlines() if x.startswith("RESULT ")]
                if proc.returncode != 0 or not line:
                    raise SystemExit("%s failed:\n%s\n%s" % (name, proc.stdout, proc.stderr))
                report["runs"].setdefault(name, []).append(json.loads(line[0][7:]))
    summary = {}
    for name, runs in report["runs"].items():
        v = [run["ms"] for run in runs]
        summary[name] = {"ms": v, "min": min(v), "spread": (max(v) - min(v)) / min(v)}
        if "words_top" in runs[0]:
            summary[name]["oov_share_top"] = runs[0]["oov_words_top"] / max(1, runs[0]["words_top"])
    shas = lambda name: {run["sha1"] for run in report["runs"][name]}   # noqa: E731
    summary["c4 token LM identical with the filter off"] = shas("c4 token LM") == shas("c4 token LM, filter off") and \
        len(shas("c4 token LM")) == 1
    summary["c2 character LM identical to the parent build"] = \
        shas("c2 character LM, this build") == shas("c2 character LM, parent build") and \
        len(shas("c2 character LM, this build")) == 1
    report["summary"] = summary
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

"""Time the prefix beam search with a word n-gram LM fused in, against the LM-free search and a second build.

    python tools/beam_lm_time.py --base-lib end2end_b200/lib/libe2e_ctc_base.so [--reps 3] [--launches 10]
                                 [--out results/beam_lm_time.json]

Workload: c2 (B=64, T=400, V=29; labels blank, space, a-z, '), fp32 raw logits (log-softmax fused), beam_width 100,
N in {1, 100}.  Models: seeded synthetic 3-gram ARPA files written to a temporary directory at run time, "small"
(about 10^4 n-grams: its table stays in L2) and "large" (about 5 * 10^6 n-grams: a table of 16.8 M slots, 805 MB).
Every time is the beam-search kernel's device time from the library's own CUDA-event hooks (beam_search or
beam_search_lm), with L2 flushed (256 MB write) before every launch, averaged over --launches launches after two
warm-up launches.  Each repetition runs both builds in fresh processes, alternating them: the base build runs the
LM-free N-best list only; this build runs it and the LM variant with both models.  The LM-free results of both builds
are compared.  Also reported: NGramLM.from_arpa's time per model, the C restatement's CPU time on the first utterances
with the small model, and the card's name, power limit and max SM clock.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, T, V, SEED = 64, 400, 29, 1                                 # c2 (oracle.CONFIGS)
LABELS = ["_", " "] + [chr(ord("a") + i) for i in range(26)] + ["'"]
BEAM = 100
N_BEST = (1, 100)
MODELS = {"small": (300, 3000, 6700), "large": (100000, 1900000, 3000000)}   # unigrams (plus specials), bigrams, trigrams


def write_model(path, n_uni, n_bi, n_tri, seed):
    """A random valid 3-gram ARPA model over words spelled with a-z and '."""
    import numpy as np
    rng = np.random.default_rng(seed)
    letters = np.array(list("abcdefghijklmnopqrstuvwxyz'"))
    words = set()
    while len(words) < n_uni:
        for n in rng.integers(1, 8, size=n_uni):
            words.add("".join(rng.choice(letters[:26], size=n)))
    words = ["<s>", "</s>", "<unk>"] + sorted(words)[:n_uni]
    nw = len(words)
    bi = np.unique(rng.integers(2, nw, size=(n_bi, 2)), axis=0)
    bi[:, 0] = np.where(rng.random(len(bi)) < 0.05, 0, bi[:, 0])   # some bigrams after <s>
    bi = np.unique(bi, axis=0)
    pick = rng.integers(0, len(bi), size=n_tri)
    tri = np.unique(np.concatenate([bi[pick], rng.integers(1, nw, size=(n_tri, 1))], axis=1), axis=0)
    W = np.array(words, dtype=object)
    with open(path, "w") as f:
        f.write("\\data\\\nngram 1=%d\nngram 2=%d\nngram 3=%d\n\n\\1-grams:\n" % (nw, len(bi), len(tri)))
        up, ub = rng.uniform(-6, -1, nw), rng.uniform(-1, 0.3, nw)
        f.write("".join("%.4f\t%s\t%.4f\n" % (-99.0 if i == 0 else up[i], w, ub[i]) for i, w in enumerate(words)))
        f.write("\n\\2-grams:\n")
        bp, bb = rng.uniform(-4, -0.1, len(bi)), rng.uniform(-1, 0.3, len(bi))
        f.write("".join("%.4f\t%s %s\t%.4f\n" % (bp[i], a, b, bb[i]) for i, (a, b) in enumerate(W[bi])))
        f.write("\n\\3-grams:\n")
        tp = rng.uniform(-3, -0.05, len(tri))
        f.write("".join("%.4f\t%s %s %s\n" % (tp[i], a, b, c) for i, (a, b, c) in enumerate(W[tri])))
        f.write("\n\\end\\\n")
    return nw + len(bi) + len(tri)


def child(lib_path, launches, with_lm, model_dir):
    import torch
    sys.path.insert(0, ROOT)
    os.environ["E2E_CTC_LIB"] = lib_path
    import oracle
    from end2end_b200 import _lib
    L = ctypes.CDLL(lib_path)
    vp, i32, sz, dbl = ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t, ctypes.c_double
    dp = ctypes.POINTER(_lib.Desc)
    L.e2e_ctc_beam_nbest_workspace_bytes.argtypes = [dp, i32, i32]
    L.e2e_ctc_beam_nbest_workspace_bytes.restype = sz
    L.e2e_ctc_beam_nbest_device.argtypes = [dp, i32, i32, i32, dbl, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_profile_enable.argtypes = [i32]
    L.e2e_ctc_profile_read.argtypes = [ctypes.POINTER(dbl), ctypes.POINTER(ctypes.c_uint64), i32]
    L.e2e_last_error_string.restype = ctypes.c_char_p
    dev = torch.device("cuda:0")
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())                # noqa: E731
    n_kinds = 18 if not with_lm else len(_lib.KERNEL_KINDS)   # the base build may predate the LM kinds
    kind = {k: i for i, k in enumerate(_lib.KERNEL_KINDS)}

    def ok(rc):
        if rc != 0:
            raise RuntimeError(L.e2e_last_error_string().decode())

    def timed(launch, k):
        for _ in range(2):
            launch()
        torch.cuda.synchronize()
        ms = (ctypes.c_double * n_kinds)()
        cnt = (ctypes.c_uint64 * n_kinds)()
        ok(L.e2e_ctc_profile_enable(1))
        ok(L.e2e_ctc_profile_read(ms, cnt, n_kinds))
        for _ in range(launches):
            flush.add_(1)
            launch()
        torch.cuda.synchronize()
        ok(L.e2e_ctc_profile_read(ms, cnt, n_kinds))
        ok(L.e2e_ctc_profile_enable(0))
        assert cnt[kind[k]] == launches, cnt[kind[k]]
        return ms[kind[k]] / launches

    x, _, ll, _ = oracle.make_inputs(B, T, V, 1, 1, SEED)
    x, ll = x.to(dev), ll.to(dev)
    d = _lib.Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, 0
    d.blank_idx, d.dtype, d.from_logits = 0, _lib.E2E_F32, 1
    d.targets_itype = d.lengths_itype = _lib.E2E_I64
    d.logits_stride_b, d.logits_stride_t = T * V, V
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    res = {}
    for n in N_BEST:
        ws = torch.empty(L.e2e_ctc_beam_nbest_workspace_bytes(ctypes.byref(d), BEAM, n), dtype=torch.uint8, device=dev)
        dec = torch.empty(B, n, T, dtype=torch.int64, device=dev)
        dl = torch.empty(B, n, dtype=torch.int64, device=dev)
        sc, lp = (torch.empty(B, n, dtype=torch.float64, device=dev) for _ in range(2))
        ties = torch.empty(B, dtype=torch.int64, device=dev)
        res["nolm_n%d_ms" % n] = timed(lambda: ok(L.e2e_ctc_beam_nbest_device(
            ctypes.byref(d), BEAM, n, 1, 0.5, p(x), p(ll), p(dec), p(dl), p(sc), p(lp), p(ties), p(ws), ws.numel(),
            stream)), "beam_search")
        res["nolm_n%d_sha1" % n] = hashlib.sha1(torch.cat([dec.flatten(), dl.flatten(), ties, sc.flatten().view(
            torch.int64), lp.flatten().view(torch.int64)]).cpu().numpy().tobytes()).hexdigest()
    if with_lm:
        from end2end_b200 import NGramLM
        from end2end_b200.engine import CTCBeamEngine
        eng = CTCBeamEngine(0, BEAM, LABELS, 0.5)
        for name in MODELS:
            t0 = time.perf_counter()
            lm = NGramLM.from_arpa(os.path.join(model_dir, name + ".arpa"))
            torch.cuda.synchronize()
            res["%s_load_s" % name] = time.perf_counter() - t0
            res["%s_ngrams" % name] = lm.n_ngrams
            res["%s_table_MB" % name] = lm.table.numel() / 2 ** 20
            for n in N_BEST:
                res["%s_n%d_ms" % (name, n)] = timed(
                    lambda: eng.decode_nbest_lm_device(x, lm, ll, n, True, lmwt=0.8, oov_penalty=-2.0), "beam_search_lm")
                out = eng.decode_nbest_lm_device(x, lm, ll, n, True, lmwt=0.8, oov_penalty=-2.0)
                res["%s_n%d_oov_share" % (name, n)] = float(out[5][:, 0].sum()) / max(1.0, float(
                    sum(len([w for w in s.split(" ") if w]) for s in _sentences(out[0][:, 0].cpu(), out[1][:, 0].cpu()))))
            del lm
            torch.cuda.empty_cache()
    print("RESULT " + json.dumps(res), flush=True)


def _sentences(t, n):
    return ["".join(LABELS[c] for c in r[:k] if c >= 0) for r, k in zip(t.tolist(), n.tolist())]


def restatement_time(model_dir, n_utt):
    """CPU time of tests/beam_lm_restatement.c on the first n_utt utterances of c2 with the small model."""
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle
    from end2end_b200.lm.ngram import parse_arpa
    from test_gpu_beam_lm import restate
    _, ng = parse_arpa(os.path.join(model_dir, "small.arpa"))
    x, _, ll, _ = oracle.make_inputs(B, T, V, 1, 1, SEED)
    t0 = time.perf_counter()
    restate(x[:n_utt], ll[:n_utt], ng, LABELS, 0, BEAM, 100, 0.5, 0.8, -2.0, after_logsoftmax=False)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--restatement-utts", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None)
    ap.add_argument("--lm", action="store_true")
    ap.add_argument("--model-dir", default=None)
    a = ap.parse_args()
    if a.child:
        return child(a.child, a.launches, a.lm, a.model_dir)
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[:1], "shape": "c2 B=%d T=%d V=%d fp32 logits" % (B, T, V),
              "beam_width": BEAM, "launches": a.launches, "l2": "flushed (256 MB write) before every launch",
              "runs": {"base": [], "this": []}}
    with tempfile.TemporaryDirectory(prefix="beam_lm_models_") as md:
        for i, (name, sizes) in enumerate(MODELS.items()):
            t0 = time.perf_counter()
            report["%s_model_ngrams_written" % name] = write_model(os.path.join(md, name + ".arpa"), *sizes, seed=100 + i)
            report["%s_model_write_s" % name] = time.perf_counter() - t0
        this_lib = os.path.join(ROOT, "end2end_b200", "lib", "libe2e_ctc.so")
        for r in range(a.reps):
            order = [("base", a.base_lib, False), ("this", this_lib, True)]
            for tag, lib, lm in (order if r % 2 == 0 else order[::-1]):
                cmd = [sys.executable, os.path.abspath(__file__), "--base-lib", a.base_lib, "--child", lib,
                       "--launches", str(a.launches), "--model-dir", md] + (["--lm"] if lm else [])
                proc = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
                line = [x for x in proc.stdout.splitlines() if x.startswith("RESULT ")]
                if proc.returncode != 0 or not line:
                    raise SystemExit("%s failed:\n%s\n%s" % (tag, proc.stdout, proc.stderr))
                report["runs"][tag].append(json.loads(line[0][7:]))
        if a.restatement_utts > 0:
            report["restatement_cpu_s"] = {"utterances": a.restatement_utts,
                                           "seconds": restatement_time(md, a.restatement_utts)}
    summary = {}
    for tag in ("base", "this"):
        for key in report["runs"][tag][0]:
            if key.endswith("_ms") or key.endswith("_load_s"):
                v = [run[key] for run in report["runs"][tag]]
                summary["%s %s" % (tag, key)] = {"v": v, "min": min(v), "spread": (max(v) - min(v)) / min(v)}
    for n in N_BEST:
        shas = {run["nolm_n%d_sha1" % n] for tag in ("base", "this") for run in report["runs"][tag]}
        summary["LM-free N=%d results identical across builds" % n] = len(shas) == 1
    report["summary"] = summary
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

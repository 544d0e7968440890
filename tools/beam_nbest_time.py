"""Time the prefix beam search's decode and its N-best list, against a second build of the library.

    python tools/beam_nbest_time.py --base-lib end2end_b200/lib/libe2e_ctc_base.so [--reps 3] [--launches 10]
                                    [--out results/beam_nbest_time.json]

Shapes: c2 (B=64, T=400, V=29) and c4 (B=128, T=250, V=1024), fp32 raw logits (log-softmax fused), beam_width 100.
Every measurement is the beam_search kernel's device time from the library's own CUDA-event hooks, with L2 flushed
(256 MB write) before every launch, averaged over --launches launches after two warm-up launches.  Each repetition runs
both builds in fresh processes, alternating them; the base build runs `decode` only (it may predate the N-best entry
points), this tree's build runs `decode` and the N-best list for N in {1, 10, 100}.  The decode results of both builds
are compared.  The report gives, per measurement, every repetition and the spread (max - min) / min.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = {"c2": (64, 400, 29, 1), "c4": (128, 250, 1024, 3)}   # B, T, V, seed (oracle.CONFIGS)
BEAM = 100
N_BEST = (1, 10, 100)
KIND_BEAM = 9                                                  # e2e_ctc_profile_read's kind index of beam_search


def child(lib_path, launches, with_nbest):
    import torch
    sys.path.insert(0, ROOT)
    import oracle
    from end2end_b200 import _lib
    L = ctypes.CDLL(lib_path)
    vp, i32, sz, dbl = ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t, ctypes.c_double
    dp = ctypes.POINTER(_lib.Desc)
    L.e2e_ctc_beam_workspace_bytes.argtypes = [dp, i32]
    L.e2e_ctc_beam_workspace_bytes.restype = sz
    L.e2e_ctc_beam_decode_device.argtypes = [dp, i32, i32, dbl, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_profile_enable.argtypes = [i32]
    L.e2e_ctc_profile_read.argtypes = [ctypes.POINTER(dbl), ctypes.POINTER(ctypes.c_uint64), i32]
    L.e2e_last_error_string.restype = ctypes.c_char_p
    if with_nbest:
        L.e2e_ctc_beam_nbest_device.argtypes = [dp, i32, i32, i32, dbl, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    dev = torch.device("cuda:0")
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())                # noqa: E731

    def ok(rc):
        if rc != 0:
            raise RuntimeError(L.e2e_last_error_string().decode())

    def timed(launch):
        for _ in range(2):
            launch()
        torch.cuda.synchronize()
        n_kinds = len(_lib.KERNEL_KINDS)
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
        assert cnt[KIND_BEAM] == launches, cnt[KIND_BEAM]
        return ms[KIND_BEAM] / launches

    out = {}
    for name, (B, T, V, seed) in SHAPES.items():
        x, _, ll, _ = oracle.make_inputs(B, T, V, 1, 1, seed)
        x, ll = x.to(dev), ll.to(dev)
        d = _lib.Desc()
        d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, 0
        d.blank_idx, d.dtype, d.from_logits = 0, _lib.E2E_F32, 1
        d.targets_itype = d.lengths_itype = _lib.E2E_I64
        d.logits_stride_b, d.logits_stride_t = T * V, V
        ws = torch.empty(L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), BEAM), dtype=torch.uint8, device=dev)
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        dec = torch.empty(B, T, dtype=torch.int64, device=dev)
        dl = torch.empty(B, dtype=torch.int64, device=dev)
        ties = torch.empty(B, dtype=torch.int64, device=dev)
        res = {"decode_ms": timed(lambda: ok(L.e2e_ctc_beam_decode_device(
            ctypes.byref(d), BEAM, -1, 0.0, p(x), p(ll), p(dec), p(dl), p(ties), p(ws), ws.numel(), stream)))}
        res["decode_sha1"] = hashlib.sha1(torch.cat([dec.flatten(), dl, ties]).cpu().numpy().tobytes()).hexdigest()
        if with_nbest:
            for n in N_BEST:
                decn = torch.empty(B, n, T, dtype=torch.int64, device=dev)
                dln = torch.empty(B, n, dtype=torch.int64, device=dev)
                scn = torch.empty(B, n, dtype=torch.float64, device=dev)
                lpn = torch.empty(B, n, dtype=torch.float64, device=dev)
                res["nbest%d_ms" % n] = timed(lambda: ok(L.e2e_ctc_beam_nbest_device(
                    ctypes.byref(d), BEAM, n, -1, 0.0, p(x), p(ll), p(decn), p(dln), p(scn), p(lpn), p(ties), p(ws),
                    ws.numel(), stream)))
                assert torch.equal(decn[:, 0], dec) and torch.equal(dln[:, 0], dl)
        out[name] = res
    print("RESULT " + json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None)
    ap.add_argument("--nbest", action="store_true")
    a = ap.parse_args()
    if a.child:
        return child(a.child, a.launches, a.nbest)
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi[:1], "beam_width": BEAM, "launches": a.launches,
              "l2": "flushed (256 MB write) before every launch", "runs": {"base": [], "this": []}}
    this_lib = os.path.join(ROOT, "end2end_b200", "lib", "libe2e_ctc.so")
    for r in range(a.reps):
        order = [("base", a.base_lib, False), ("this", this_lib, True)]
        for tag, lib, nb in (order if r % 2 == 0 else order[::-1]):
            cmd = [sys.executable, os.path.abspath(__file__), "--base-lib", a.base_lib, "--child", lib,
                   "--launches", str(a.launches)] + (["--nbest"] if nb else [])
            proc = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
            line = [x for x in proc.stdout.splitlines() if x.startswith("RESULT ")]
            if proc.returncode != 0 or not line:
                raise SystemExit("%s failed:\n%s\n%s" % (tag, proc.stdout, proc.stderr))
            report["runs"][tag].append(json.loads(line[0][7:]))
    summary = {}
    for shape in SHAPES:
        for tag in ("base", "this"):
            for key in report["runs"][tag][0][shape]:
                if key.endswith("_ms"):
                    v = [run[shape][key] for run in report["runs"][tag]]
                    summary["%s %s %s" % (shape, tag, key)] = {"ms": v, "min": min(v), "spread": (max(v) - min(v)) / min(v)}
        shas = {run[shape]["decode_sha1"] for tag in ("base", "this") for run in report["runs"][tag]}
        summary["%s decode results identical" % shape] = len(shas) == 1
    report["summary"] = summary
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

"""Time the N-hypothesis aligner against get_alignment_3d on replicated log-probabilities.

    python tools/align_nbest_time.py [--reps 3] [--launches 10] [--parent-lib PATH] [--out results/align_nbest_time.json]

Shapes: c2 (B=64, T=400, V=29) and c4 (B=128, T=250, V=1024) of oracle.CONFIGS, fp32 raw logits.  The hypotheses are
the N-best lists of the same batch (CTCDecoder.decode_nbest, beam 100), N in {1, 10, 100}.  Two arms per (shape, N):
  align:      CTCBeamEngine.align_device(from_logits=True): K1 row statistics + one K6 launch;
  replicated: F.log_softmax + repeat_interleave(N) + get_alignment_3d_device -- what a caller without the aligner runs.
Kernel times come from the library's CUDA-event hooks (the replicated arm's log-softmax and copy are torch kernels, timed
with CUDA events around them), with L2 flushed (256 MB write) before every launch, averaged over --launches launches
after two warm-up launches; the arms alternate over --reps repetitions and the report gives every repetition and the
range.  With --parent-lib (a build of the previous commit), get_alignment_3d at c2 is also timed on both libraries in
alternating child processes, so a regression shows against the same run's spread.  The card's name, power limit and max
SM clock are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = ("c2", "c4")
BEAM = 100
N_HYP = (1, 10, 100)


def viterbi_child(lib_path, launches):
    """Mean viterbi kernel ms of get_alignment_3d at c2 through LIB directly (the parent's library lacks the newer entry
    points the package binds, so this uses only the Viterbi ABI and the timing hooks, which both builds share)."""
    import torch
    import torch.nn.functional as F
    sys.path.insert(0, ROOT)
    import oracle
    L = ctypes.CDLL(lib_path)
    vp, i32, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t
    from end2end_b200._lib import Desc
    L.e2e_ctc_viterbi_workspace_bytes.argtypes = [ctypes.POINTER(Desc), i32]
    L.e2e_ctc_viterbi_workspace_bytes.restype = sz
    L.e2e_ctc_viterbi_align_device.argtypes = [ctypes.POINTER(Desc), i32, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_profile_enable.argtypes = [i32]
    L.e2e_ctc_profile_read.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64), i32]
    B, T, V, Lmin, Lmax, seed, _, full = oracle.CONFIGS["c2"]
    x, tg, ll, tl = oracle.make_inputs(B, T, V, Lmin, Lmax, seed, full_length=full)
    dev = torch.device("cuda:0")
    lp = F.log_softmax(x, -1).to(dev)
    tg, ll, tl = tg.to(dev), ll.to(dev), tl.to(dev)
    d = Desc()
    d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
    d.blank_idx, d.dtype, d.targets_itype, d.lengths_itype = 0, 0, 1, 1
    d.logits_stride_b, d.logits_stride_t, d.targets_stride_b = T * V, V, Lmax
    ws = torch.empty(L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), 1), dtype=torch.uint8, device=dev)
    out = torch.empty(B, T, dtype=torch.int64, device=dev)
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())    # noqa: E731
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        rc = L.e2e_ctc_viterbi_align_device(ctypes.byref(d), 1, p(lp), p(tg), p(ll), p(tl), p(out), p(ws), ws.numel(), stream)
        assert rc == 0, rc
    for _ in range(2):
        launch()
    torch.cuda.synchronize()
    n = 16
    ms, cnt = (ctypes.c_double * n)(), (ctypes.c_uint64 * n)()
    L.e2e_ctc_profile_enable(1)
    L.e2e_ctc_profile_read(ms, cnt, n)
    for _ in range(launches):
        flush.add_(1)
        launch()
    torch.cuda.synchronize()
    L.e2e_ctc_profile_read(ms, cnt, n)
    L.e2e_ctc_profile_enable(0)
    print(json.dumps({"viterbi_ms": ms[7] / max(cnt[7], 1), "launches": int(cnt[7]),
                      "aligned_sha": int(out.cpu().sum())}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    ap.add_argument("--viterbi-child", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.viterbi_child:
        return viterbi_child(a.viterbi_child, a.launches)
    import torch
    import torch.nn.functional as F
    sys.path.insert(0, ROOT)
    import oracle
    from end2end_b200 import CTCDecoder, _lib
    from end2end_b200.engine import CTCBeamEngine
    from end2end_b200.utils.alignment import get_alignment_3d_device
    if not torch.cuda.is_available():
        raise SystemExit("align_nbest_time.py measures on the GPU; no CUDA device here")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.device("cuda:0")
    flush = torch.zeros(256 * 2 ** 20 // 4, dtype=torch.int32, device=dev)

    def timed(launch, torch_ops=None):
        """{kernel kind: mean ms per launch} over a.launches launches, L2 flushed before each; torch_ops (optional) runs
        first, bracketed by CUDA events, and is reported as 'torch'."""
        for _ in range(2):
            launch(torch_ops() if torch_ops else None)
        torch.cuda.synchronize()
        _lib.profile_enable(True)
        _lib.profile_read()
        t_ms = 0.0
        for _ in range(a.launches):
            flush.add_(1)
            arg = None
            if torch_ops:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                arg = torch_ops()
                e1.record()
            launch(arg)
            if torch_ops:
                e1.synchronize()
                t_ms += e0.elapsed_time(e1)
            del arg
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile_enable(False)
        res = {k: ms / a.launches for k, (ms, n) in prof.items() if n}
        if torch_ops:
            res["torch_log_softmax_repeat"] = t_ms / a.launches
        return res

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
            tg, tl, llr = hyps.reshape(B * N, -1), hl.reshape(B * N), ll.repeat_interleave(N)
            ours = eng.align_device(x, hyps, hl, ll, from_logits=True)
            rep = get_alignment_3d_device(F.log_softmax(x, -1).repeat_interleave(N, 0), tg, llr, tl)
            same = float((ours[0].reshape(B * N, -1) == rep).double().mean())
            runs = {"align": [], "replicated": []}
            for r in range(a.reps):
                arms = [("align", lambda: timed(lambda _: eng.align_device(x, hyps, hl, ll, from_logits=True))),
                        ("replicated", lambda: timed(lambda lpr: get_alignment_3d_device(lpr, tg, llr, tl),
                                                     lambda: F.log_softmax(x, -1).repeat_interleave(N, 0)))]
                for tag, fn in (arms if r % 2 == 0 else arms[::-1]):
                    runs[tag].append(fn())
            d = _lib.Desc()
            d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, tg.size(1)
            d.blank_idx, d.dtype, d.targets_itype, d.lengths_itype, d.from_logits = 0, _lib.E2E_F32, 1, 1, 1
            d.logits_stride_b, d.logits_stride_t, d.targets_stride_b = T * V, V, tg.size(1)
            L = _lib.load()
            ws_align = L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(d), N)
            d.batch, d.from_logits = B * N, 0
            ws_rep = L.e2e_ctc_viterbi_workspace_bytes(ctypes.byref(d), 1)
            res = {"mean_hyp_length": float(hl.double().mean()), "max_hyp_length": int(hl.max()),
                   "frames_equal_to_replicated_fp32_logsoftmax": same,
                   "align_workspace_bytes": ws_align, "replicated_workspace_bytes": ws_rep,
                   "replicated_input_bytes": B * N * T * V * 4}
            for tag in runs:
                tot = [sum(k.values()) for k in runs[tag]]
                res[tag] = {"kernels_ms": runs[tag], "total_ms": tot, "min": min(tot), "max": max(tot)}
            res["speedup_min_over_min"] = res["replicated"]["min"] / res["align"]["min"]
            shape["N=%d" % N] = res
        report["shapes"][name] = shape
    if a.parent_lib:
        libs = {"this": _lib.LIB_PATH, "parent": a.parent_lib}
        vit = {k: [] for k in libs}
        for r in range(a.reps):
            for tag in (("this", "parent") if r % 2 == 0 else ("parent", "this")):
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--viterbi-child", libs[tag],
                                      "--launches", str(max(a.launches, 20))], capture_output=True, text=True, check=True)
                vit[tag].append(json.loads(out.stdout.strip().splitlines()[-1]))
        report["get_alignment_3d_c2"] = {
            k: {"viterbi_ms": [v["viterbi_ms"] for v in vit[k]], "min": min(v["viterbi_ms"] for v in vit[k]),
                "max": max(v["viterbi_ms"] for v in vit[k]), "aligned_sum": vit[k][0]["aligned_sha"]} for k in vit}
    text = json.dumps(report, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

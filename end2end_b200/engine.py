"""Host-side engines over the C ABI (include/e2e_ctc.h).

``CTCLossEngine`` is the drop-in for the reference's pybind11 class
``cpp_ctc_loss.CTCLossEngine(blank_idx)`` (src/losses/ctc_loss_py.cpp:5-17): same constructor
argument, same ``compute(logits, targets, logits_lengths, targets_lengths) -> (losses, grads)``
contract (src/losses/forward_backward.cpp:7-59) -- inputs are never mutated, results come back on
the caller's device in the caller's dtype, padding rows of ``grads`` hold ``exp(lp)``, an
infeasible utterance gives ``+inf`` / an all-NaN block.  Differences, all deliberate:

* the work runs on the GPU (sm_100a kernels); with CPU tensors the engine copies in and out
  through the host-buffer entry points and there is NO CPU fallback: without a CUDA device the
  call raises;
* out-of-range lengths / labels (undefined behaviour in the reference) raise ``ValueError`` when
  the length tensors live on the host, and are flagged on the device otherwise;
* ``forward`` / ``backward`` expose the two halves separately so the autograd Function can apply
  ``grad_output`` inside the gradient kernel instead of in an extra dense pass.

PyTorch is used for device memory and streams only; every byte of arithmetic happens in
``libe2e_ctc.so``.
"""
import ctypes
import os

import torch

from . import _lib
from .utils.hypotheses import empty_marker_as_empty

_DTYPES = {torch.float32: _lib.E2E_F32, torch.bfloat16: _lib.E2E_BF16,
           torch.float16: _lib.E2E_F16, torch.float64: _lib.E2E_F64}
_ITYPES = {torch.int32: _lib.E2E_I32, torch.int64: _lib.E2E_I64}


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None and t.numel() > 0 else ctypes.c_void_p(0)


try:
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:  # pragma: no cover - older torch
    def _raw_stream(index):
        return torch.cuda.current_stream(index).cuda_stream


def _stream(device):
    return ctypes.c_void_p(_raw_stream(device.index if device.index is not None else torch.cuda.current_device()))


class _on_device:
    """``torch.cuda.device(dev)`` without its cost when ``dev`` is already current (the usual case)."""
    __slots__ = ("ctx",)

    def __init__(self, device):
        self.ctx = None if device.index is None or device.index == torch.cuda.current_device() else torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)


def _as_index(t, device, name):
    if t.dtype not in _ITYPES:
        if t.is_floating_point() or t.dtype == torch.bool:
            raise TypeError("%s must be an integer tensor, got %s" % (name, t.dtype))
        t = t.to(torch.int64)
    if t.device != device:
        t = t.to(device, non_blocking=True)
    return t


_LIMITS = None
#: longest hypothesis the Viterbi aligner takes (csrc/ctc_viterbi.cu: lattices of at most 2048 cells, 2 L + 1 for CTC)
ALIGN_MAX_TARGETS = 1023
#: widest reference and hypothesis rows the edit distance takes (csrc/edit_distance.cu: its key errors * 4096 -
#: substitutions stays within int32)
EDIT_MAX_REF_WIDTH, EDIT_MAX_HYP_WIDTH = 4095, 65535


def _limits():
    global _LIMITS
    if _LIMITS is None:
        _LIMITS = _lib.limits()
    return _LIMITS


def _dense3(x):
    """True if x[B,T,V] can be addressed as base + b*sb + t*st + v (unit alphabet stride)."""
    if x.size(2) > 1 and x.stride(2) != 1:
        return False
    # expanded (stride-0) views would alias rows of the gradient
    return all(x.stride(i) > 0 or x.size(i) == 1 for i in (0, 1))


class _Problem:
    """Validated, device-resident view of one batch plus the C descriptor."""

    def __init__(self, blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, device, validate=True):
        if logits.dim() != 3:
            raise ValueError("logits must be [batch, frames, alphabet], got %s" % (tuple(logits.shape),))
        if logits.dtype not in _DTYPES:
            raise TypeError("unsupported logits dtype %s" % logits.dtype)
        B, T, V = logits.shape
        if B < 1 or T < 1 or V < 1:
            raise ValueError("empty logits %s" % (tuple(logits.shape),))
        if not 0 <= blank_idx < V:
            raise ValueError("blank_idx %d outside the alphabet [0,%d)" % (blank_idx, V))
        if targets.dim() != 2 or targets.size(0) != B:
            raise ValueError("targets must be [batch, max_target_length], got %s" % (tuple(targets.shape),))
        if logits_lengths.dim() != 1 or logits_lengths.numel() != B or \
                targets_lengths.dim() != 1 or targets_lengths.numel() != B:
            raise ValueError("length tensors must have shape [batch]")
        Lmax = targets.size(1)
        lim = _limits()
        if Lmax > lim.max_targets or V > lim.max_alphabet:
            raise NotImplementedError("this build supports target length <= %d and alphabet <= %d"
                                      % (lim.max_targets, lim.max_alphabet))
        # the reference has undefined behaviour on these; reject when it costs no device sync
        if validate and not logits_lengths.is_cuda and not targets_lengths.is_cuda:
            ll, tl = logits_lengths.to(torch.int64), targets_lengths.to(torch.int64)
            if bool((ll < 1).any()) or bool((ll > T).any()):
                raise ValueError("logits_lengths must be in [1, %d]" % T)
            if bool((tl < 0).any()) or bool((tl > Lmax).any()):
                raise ValueError("targets_lengths must be in [0, %d]" % Lmax)
            if not targets.is_cuda and Lmax > 0:
                tg = targets.to(torch.int64)
                valid = torch.arange(Lmax).unsqueeze(0) < tl.unsqueeze(1)
                if bool(((tg < 0) | (tg >= V))[valid].any()):
                    raise ValueError("target labels must be in [0, %d)" % V)
        if not _dense3(logits):
            logits = logits.contiguous()
        targets = _as_index(targets, device, "targets")
        if Lmax > 0 and targets.stride(1) != 1:
            targets = targets.contiguous()
        logits_lengths = _as_index(logits_lengths, device, "logits_lengths")
        targets_lengths = _as_index(targets_lengths, device, "targets_lengths")
        if logits_lengths.dtype != targets_lengths.dtype:
            logits_lengths, targets_lengths = logits_lengths.to(torch.int64), targets_lengths.to(torch.int64)
        self.logits, self.targets = logits, targets
        self.logits_lengths = logits_lengths.contiguous()
        self.targets_lengths = targets_lengths.contiguous()
        self.B, self.T, self.V, self.Lmax = B, T, V, Lmax
        d = _lib.Desc()
        d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
        d.blank_idx, d.dtype = blank_idx, _DTYPES[logits.dtype]
        d.targets_itype = _ITYPES[targets.dtype]
        d.lengths_itype = _ITYPES[self.logits_lengths.dtype]
        d.from_logits = 1 if from_logits else 0
        d.logits_stride_b, d.logits_stride_t = logits.stride(0), logits.stride(1)
        d.grads_stride_b, d.grads_stride_t = logits.stride(0), logits.stride(1)
        d.targets_stride_b = targets.stride(0) if Lmax > 0 else 0
        self.desc = d
        self.workspace = None

    _FAST = {}

    @classmethod
    def make(cls, blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, device):
        """``_Problem(...)`` with a cache: when every tensor already lives on ``device`` the checks depend only
        on shapes / strides / dtypes, so a training loop (same layout every step) validates once and reuses
        the C descriptor."""
        if not (targets.is_cuda and logits_lengths.is_cuda and targets_lengths.is_cuda):
            return cls(blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, device)
        key = (logits.shape, logits.stride(), logits.dtype, targets.shape, targets.stride(), targets.dtype,
               logits_lengths.dtype, logits_lengths.stride(), targets_lengths.dtype, targets_lengths.stride(),
               targets.device, logits_lengths.device, targets_lengths.device, device, bool(from_logits), blank_idx)
        hit = cls._FAST.get(key)
        if hit is None:
            pb = cls(blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, device)
            same = (pb.logits is logits and pb.targets is targets and pb.logits_lengths is logits_lengths and
                    pb.targets_lengths is targets_lengths)
            if same:                      # nothing had to be converted or copied: the layout is reusable as is
                if len(cls._FAST) > 256:
                    cls._FAST.clear()
                cls._FAST[key] = (pb.desc, pb.B, pb.T, pb.V, pb.Lmax)
            return pb
        pb = cls.__new__(cls)
        pb.logits, pb.targets, pb.logits_lengths, pb.targets_lengths = logits, targets, logits_lengths, targets_lengths
        pb.desc, pb.B, pb.T, pb.V, pb.Lmax = hit
        pb.workspace = None
        return pb

    def new_grads(self, pin=False):
        x = self.logits
        return torch.empty_strided(x.size(), x.stride(), dtype=x.dtype, device=x.device, pin_memory=pin)


_CUDA_OK = False


def _require_cuda():
    global _CUDA_OK
    if not _CUDA_OK:
        if not torch.cuda.is_available():
            raise RuntimeError("end2end_b200 needs a CUDA device (sm_100a): the CTC engine has no CPU fallback")
        _CUDA_OK = True


class CTCLossEngine:
    """Drop-in for ``cpp_ctc_loss.CTCLossEngine`` (src/losses/ctc_loss_py.cpp:5-17)."""

    def __init__(self, blank_idx=0):
        self.blank_idx = int(blank_idx)
        self._L = _lib.load()
        self._host = {}
        self._ws_bytes = {}
        self._scratch_bufs = {}
        self._scale_desc = {}

    # ------------------------------------------------------------------ reference contract ----
    def compute(self, logits, targets, logits_lengths, targets_lengths, from_logits=False):
        """(losses[B], grads[B,T,V]) exactly as the reference engine returns them; ``logits`` are
        log-probabilities unless ``from_logits`` (then log_softmax is fused and ``grads`` is the
        gradient with respect to the raw logits)."""
        _require_cuda()
        logits = logits.detach()
        if not logits.is_cuda:
            return self._compute_host(logits, targets, logits_lengths, targets_lengths, from_logits)
        with _on_device(logits.device):
            pb = _Problem(self.blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, logits.device)
            losses = torch.empty(pb.B, dtype=logits.dtype, device=logits.device)
            grads = pb.new_grads()
            ws = self._scratch(pb)
            _lib.check(self._L.e2e_ctc_loss_fwd_bwd_device(
                ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths),
                _ptr(pb.targets_lengths), _ptr(losses), _ptr(grads), _ptr(ws), ws.numel(), _stream(logits.device)))
        return losses, grads

    # ------------------------------------------------------------------ one training step -------
    def step(self, logits, targets, logits_lengths, targets_lengths, from_logits=False, grad_scale=1.0,
             reduce_scale=None, want_pair=False):
        """Loss and gradient of one batch in ONE library call (device tensors).

        Returns ``(losses[B], grads, reduced, pair)``: ``grads = grad_scale * d loss_b / d logits``;
        ``reduced`` is the 0-dim ``reduce_scale * sum(losses)`` (``None`` if ``reduce_scale`` is None);
        ``pair`` the fp64 ``[sum(losses), B]`` a data-parallel caller all-reduces (``want_pair``).
        Alphabets <= 128 run as a single fused kernel (+ the reduction)."""
        _require_cuda()
        logits = logits.detach()
        dev = logits.device
        with _on_device(dev):
            pb = _Problem.make(self.blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, dev)
            losses = torch.empty(pb.B, dtype=logits.dtype, device=dev)
            grads = pb.new_grads()
            reduced = torch.empty((), dtype=logits.dtype, device=dev) if reduce_scale is not None else None
            pair = torch.empty(2, dtype=torch.float64, device=dev) if want_pair else None
            ws = self._scratch(pb)
            _lib.check(self._L.e2e_ctc_loss_step_device(
                ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths),
                _ptr(pb.targets_lengths), _ptr(losses), _ptr(grads), float(grad_scale), _ptr(reduced), _ptr(pair),
                float(reduce_scale if reduce_scale is not None else 1.0), _ptr(ws), ws.numel(), _stream(dev)))
        return losses, grads, reduced, pair

    def graphed_step(self, logits, targets, logits_lengths, targets_lengths, from_logits=False, grad_scale=1.0,
                     reduce_scale=None, want_pair=False, comm=None, share=None, workspace=None):
        """The same step as :meth:`step`, captured ONCE into a CUDA graph bound to these tensors
        (SURVEY 8(f1)): ``g = engine.graphed_step(...)`` runs the step and returns a :class:`GraphedStep`;
        every ``g.launch()`` replays it with one driver call.  The tensors (and the outputs ``g.losses``,
        ``g.grads``, ``g.reduced``, ``g.pair``) keep their addresses; a training loop copies each batch into
        them.  ``comm``: a library communicator handle (``distributed.LossComm``) whose scalar all-reduce of
        ``reduced`` becomes part of the graph.  ``share``: another GraphedStep over the SAME input tensors whose
        ``losses`` / ``grads`` / workspace this one reuses (only ``reduced`` / ``pair`` are its own): two such
        steps replayed alternately let a side-stream all-reduce of step k's scalar overlap step k+1.
        ``workspace``: a uint8 CUDA tensor of at least :meth:`workspace_bytes` bytes to use as scratch -- graphs
        that are only ever replayed one after another on ONE stream may share one (each otherwise owns its own)."""
        _require_cuda()
        logits = logits.detach()
        dev = logits.device
        if not (targets.is_cuda and logits_lengths.is_cuda and targets_lengths.is_cuda):
            raise ValueError("graphed_step needs device-resident targets and lengths (the graph is bound to their addresses)")
        with _on_device(dev):
            pb = _Problem(self.blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, dev)
            if pb.logits is not logits:
                raise ValueError("graphed_step needs logits with a unit alphabet stride (no hidden copy: the graph reads this tensor)")
            return GraphedStep(self, pb, float(grad_scale), reduce_scale, want_pair, comm, share, workspace)

    def workspace_bytes(self, logits, targets, logits_lengths, targets_lengths, from_logits=False):
        """Scratch bytes one step over tensors of these shapes needs (``e2e_ctc_loss_workspace_bytes``)."""
        pb = _Problem.make(self.blank_idx, logits.detach(), targets, logits_lengths, targets_lengths, from_logits, logits.device)
        return self._ws_need(pb)

    def scale_rows_(self, grads, grad_output):
        """``grads[b] *= grad_output[b or 0]`` in place (functions/forward_backward.py:34); utterances whose
        factor is exactly 1 are skipped on the device."""
        dev = grads.device
        g = grad_output.detach()
        if g.device != dev or g.dtype != grads.dtype or not g.is_contiguous():
            g = g.to(device=dev, dtype=grads.dtype).contiguous()
        if g.numel() not in (1, grads.size(0)):
            raise ValueError("grad_output must have 1 or batch elements")
        key = (grads.shape, grads.stride(), grads.dtype)
        d = self._scale_desc.get(key)
        if d is None:
            d = _lib.Desc()
            d.batch, d.max_frames, d.alphabet, d.max_targets = grads.size(0), grads.size(1), grads.size(2), 0
            d.blank_idx, d.dtype = 0, _DTYPES[grads.dtype]
            d.targets_itype = d.lengths_itype = _lib.E2E_I64
            d.grads_stride_b, d.grads_stride_t = grads.stride(0), grads.stride(1)
            d.logits_stride_b, d.logits_stride_t = grads.stride(0), grads.stride(1)
            if len(self._scale_desc) > 256:
                self._scale_desc.clear()
            self._scale_desc[key] = d
        with _on_device(dev):
            _lib.check(self._L.e2e_ctc_scale_rows_device(ctypes.byref(d), _ptr(grads), _ptr(g), g.numel(), _stream(dev)))
        return grads

    # ------------------------------------------------------------------ split halves (device) --
    def forward(self, logits, targets, logits_lengths, targets_lengths, from_logits=False):
        """Per-utterance losses [B] and an opaque state for :meth:`backward` (device tensors only)."""
        _require_cuda()
        logits = logits.detach()
        with _on_device(logits.device):
            pb = _Problem(self.blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, logits.device)
            losses = torch.empty(pb.B, dtype=logits.dtype, device=logits.device)
            pb.workspace = self._workspace(pb)
            _lib.check(self._L.e2e_ctc_loss_forward_device(
                ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths),
                _ptr(pb.targets_lengths), _ptr(losses), _ptr(pb.workspace), pb.workspace.numel(),
                _stream(logits.device)))
        return losses, pb

    def backward(self, state, grad_output=None, scale=1.0):
        """grads[b] = scale * grad_output[b or 0] * d loss_b / d logits, written in one pass."""
        pb = state
        dev = pb.logits.device
        with _on_device(dev):
            grads = pb.new_grads()
            count = 0
            if grad_output is not None:
                grad_output = grad_output.detach().to(device=dev, dtype=pb.logits.dtype).contiguous()
                count = grad_output.numel()
                if count not in (1, pb.B):
                    raise ValueError("grad_output must have 1 or batch elements")
            _lib.check(self._L.e2e_ctc_loss_backward_device(
                ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths),
                _ptr(pb.targets_lengths), _ptr(grad_output), count, float(scale), _ptr(grads),
                _ptr(pb.workspace), pb.workspace.numel(), _stream(dev)))
        return grads

    def reduce(self, losses, scale=1.0):
        """0-dim ``scale * sum(losses)`` (modules/ctc_loss.py:52-56), fp64 accumulation on the device."""
        out = torch.empty((), dtype=losses.dtype, device=losses.device)
        with _on_device(losses.device):
            _lib.check(self._L.e2e_ctc_loss_reduce_device(
                _ptr(losses), _DTYPES[losses.dtype], losses.numel(), float(scale), _ptr(out),
                ctypes.c_void_p(0), _stream(losses.device)))
        return out

    def partial_sum(self, losses):
        """fp64 device tensor ``[sum(losses), len(losses)]`` -- the pair a data-parallel caller
        all-reduces (one 16-byte collective)."""
        pair = torch.empty(2, dtype=torch.float64, device=losses.device)
        with _on_device(losses.device):
            _lib.check(self._L.e2e_ctc_loss_reduce_device(
                _ptr(losses), _DTYPES[losses.dtype], losses.numel(), 1.0, ctypes.c_void_p(0),
                _ptr(pair), _stream(losses.device)))
        return pair

    def check(self, state):
        """Device-side argument check of the forward that produced ``state`` (synchronises)."""
        st = ctypes.c_int32(0)
        with _on_device(state.logits.device):
            _lib.check(self._L.e2e_ctc_loss_check_device(_ptr(state.workspace), ctypes.byref(st),
                                                         _stream(state.logits.device)))
        return st.value

    # ------------------------------------------------------------------ internals --------------
    def _workspace(self, pb):
        key = (pb.B, pb.T, pb.V, pb.Lmax, pb.desc.dtype, _lib.forced_kernel())
        n = self._ws_bytes.get(key)
        if n is None:
            n = self._L.e2e_ctc_loss_workspace_bytes(ctypes.byref(pb.desc))
            if n == 0:
                raise _lib.E2EError(2, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            self._ws_bytes[key] = n
        return torch.empty(n, dtype=torch.uint8, device=pb.logits.device)

    def _scratch(self, pb):
        """Workspace of a call that is finished with it when the call's kernels are (the fused forward+backward
        entry points): one buffer per (device, stream), grown on demand and reused, so a training loop does not
        push a workspace-sized block through the caching allocator every step (interleaved with the live
        gradient blocks that fragments it into cudaMalloc/cudaFree cycles).  Kernels of successive calls on one
        stream are ordered, so the reuse is safe; other streams get their own buffer."""
        if os.environ.get("E2E_CTC_NO_SCRATCH_CACHE"):
            return self._workspace(pb)
        dev = pb.logits.device
        key = (dev.index, _raw_stream(dev.index if dev.index is not None else torch.cuda.current_device()))
        need = self._ws_need(pb)
        buf = self._scratch_bufs.get(key)
        if buf is None or buf.numel() < need:
            buf = torch.empty(need, dtype=torch.uint8, device=dev)
            self._scratch_bufs[key] = buf
        return buf

    def _ws_need(self, pb):
        key = (pb.B, pb.T, pb.V, pb.Lmax, pb.desc.dtype, _lib.forced_kernel())
        n = self._ws_bytes.get(key)
        if n is None:
            n = self._L.e2e_ctc_loss_workspace_bytes(ctypes.byref(pb.desc))
            if n == 0:
                raise _lib.E2EError(2, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            self._ws_bytes[key] = n
        return n

    def _host_engine(self, device):
        h = self._host.get(device)
        if h is None:
            h = _HostEngine(device)
            self._host[device] = h
        return h

    def _compute_host(self, logits, targets, logits_lengths, targets_lengths, from_logits):
        dev = torch.cuda.current_device()
        cpu = torch.device("cpu")
        if not (logits.is_contiguous() or logits.permute(1, 0, 2).is_contiguous()):
            logits = logits.contiguous()
        # lengths and labels are range-checked by the library's host entry point (plain loops over the host
        # buffers) instead of a handful of small torch ops here
        pb = _Problem(self.blank_idx, logits, targets, logits_lengths, targets_lengths, from_logits, cpu, validate=False)
        if pb.Lmax > 0 and not pb.targets.is_contiguous():
            pb.targets = pb.targets.contiguous()
            pb.desc.targets_stride_b = pb.Lmax
        # pinned results: the kernels store into them directly (no copy-out stage).  torch's caching host allocator
        # recycles the blocks; an own pool (frombuffer over cudaHostAlloc blocks) measured 20 us SLOWER per call.
        losses = torch.empty(pb.B, dtype=logits.dtype, pin_memory=True)
        grads = pb.new_grads(pin=True)
        h = self._host_engine(dev)
        try:
            _lib.check(self._L.e2e_ctc_engine_loss_host(
                h.handle, ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths),
                _ptr(pb.targets_lengths), _ptr(losses), _ptr(grads)))
        except _lib.E2EError as err:
            if err.code == _lib.E2E_ERR_LENGTHS:
                raise ValueError(str(err)) from None
            raise
        return losses, grads

    def last_host_traffic(self):
        """(h2d_bytes, d2h_bytes) of the last host-tensor call."""
        h = self._host.get(torch.cuda.current_device())
        return h.traffic() if h else (0, 0)


class GraphedStep:
    """One captured training step of the loss (``e2e_ctc_graph_*`` in include/e2e_ctc.h)."""

    def __init__(self, engine, pb, grad_scale, reduce_scale, want_pair, comm, share=None, workspace=None):
        self._L = engine._L
        self._pb = pb                       # keeps the input tensors alive
        dev = pb.logits.device
        self.device = dev
        self.losses = share.losses if share is not None else torch.empty(pb.B, dtype=pb.logits.dtype, device=dev)
        self.grads = share.grads if share is not None else pb.new_grads()
        self.reduced = torch.empty((), dtype=pb.logits.dtype, device=dev) if reduce_scale is not None else None
        self.pair = torch.empty(2, dtype=torch.float64, device=dev) if want_pair else None
        # its own workspace (graphs of several batches coexist), unless it alternates with `share` on one stream
        need = engine._ws_need(pb)
        if share is not None:
            workspace = share._ws
        if workspace is not None and (workspace.device != dev or workspace.dtype != torch.uint8 or workspace.numel() < need):
            raise ValueError("graphed_step: workspace must be a uint8 tensor of >= %d bytes on %s" % (need, dev))
        self._ws = workspace if workspace is not None else torch.empty(need, dtype=torch.uint8, device=dev)
        self._comm = comm
        self.handle = ctypes.c_void_p(0)
        _lib.check(self._L.e2e_ctc_graph_create(
            ctypes.byref(pb.desc), _ptr(pb.logits), _ptr(pb.targets), _ptr(pb.logits_lengths), _ptr(pb.targets_lengths),
            _ptr(self.losses), _ptr(self.grads), grad_scale, _ptr(self.reduced), _ptr(self.pair),
            float(reduce_scale if reduce_scale is not None else 1.0), _ptr(self._ws), self._ws.numel(),
            comm if comm is not None else ctypes.c_void_p(0), ctypes.byref(self.handle)))
        self._launch = self._L.e2e_ctc_graph_launch
        self._dev_index = dev.index if dev.index is not None else torch.cuda.current_device()

    def launch(self):
        """Enqueue one replay on the current stream; results land in ``losses`` / ``grads`` / ``reduced``."""
        rc = self._launch(self.handle, _raw_stream(self._dev_index))
        if rc:
            _lib.check(rc)
        return self

    def __del__(self):
        try:
            if self.handle:
                self._L.e2e_ctc_graph_destroy(self.handle)
                self.handle = ctypes.c_void_p(0)
        except Exception:
            pass


class _HostEngine:
    """Owns one ``e2e_ctc_engine`` handle (stream + device staging buffers) per CUDA device."""

    def __init__(self, device):
        self._L = _lib.load()
        self.handle = ctypes.c_void_p(0)
        _lib.check(self._L.e2e_ctc_engine_create(int(device), ctypes.byref(self.handle)))

    def traffic(self):
        a, b = ctypes.c_uint64(0), ctypes.c_uint64(0)
        _lib.check(self._L.e2e_ctc_engine_last_traffic(self.handle, ctypes.byref(a), ctypes.byref(b)))
        return int(a.value), int(b.value)

    def __del__(self):
        try:
            if self.handle:
                self._L.e2e_ctc_engine_destroy(self.handle)
                self.handle = ctypes.c_void_p(0)
        except Exception:
            pass


class CTCGreedyEngine:
    """Greedy half of ``cpp_ctc_decoder.CTCDecoder`` (src/decoders/ctc_decoder_py.cpp:25-29,
    src/decoders/ctc_decoder.cpp:443-490): ``decode_greedy(logits_, logits_lengths_)`` returns
    ``(decoded_targets[B,T] int64 zero padded, decoded_targets_lengths[B] int64)`` as CPU tensors
    (the sentences are assembled by the Python wrapper)."""

    def __init__(self, blank_idx=0):
        self.blank_idx = int(blank_idx)
        self._L = _lib.load()
        self._host = {}

    def _desc(self, logits, lengths):
        if logits.dim() != 3:
            raise ValueError("logits must be [batch, frames, alphabet]")
        if logits.dtype not in _DTYPES:
            raise TypeError("unsupported logits dtype %s" % logits.dtype)
        B, T, V = logits.shape
        if B < 1 or T < 1 or V < 1:
            raise ValueError("empty logits")
        if not 0 <= self.blank_idx < V:
            raise ValueError("blank_idx %d outside the alphabet [0,%d)" % (self.blank_idx, V))
        d = _lib.Desc()
        d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, 0
        d.blank_idx, d.dtype = self.blank_idx, _DTYPES[logits.dtype]
        d.targets_itype = _lib.E2E_I64
        d.lengths_itype = _ITYPES[lengths.dtype] if lengths is not None else _lib.E2E_I64
        d.logits_stride_b, d.logits_stride_t = logits.stride(0), logits.stride(1)
        return d

    def decode_greedy_device(self, logits, logits_lengths=None):
        """Device tensors in, device tensors out (no synchronisation)."""
        _require_cuda()
        logits = logits.detach()
        dev = logits.device
        if not _dense3(logits):
            logits = logits.contiguous()
        if logits_lengths is not None:
            logits_lengths = _as_index(logits_lengths, dev, "logits_lengths").contiguous()
        d = self._desc(logits, logits_lengths)
        B, T = logits.size(0), logits.size(1)
        with _on_device(dev):
            decoded = torch.empty(B, T, dtype=torch.int64, device=dev)
            lengths = torch.empty(B, dtype=torch.int64, device=dev)
            ws = torch.empty(self._L.e2e_ctc_greedy_workspace_bytes(ctypes.byref(d)), dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_greedy_decode_device(
                ctypes.byref(d), _ptr(logits), _ptr(logits_lengths), _ptr(decoded), _ptr(lengths),
                _ptr(ws), ws.numel(), _stream(dev)))
        return decoded, lengths

    def decode_greedy(self, logits_, logits_lengths_=None):
        _require_cuda()
        logits = logits_.detach()
        if logits.is_cuda:
            decoded, lengths = self.decode_greedy_device(logits, logits_lengths_)
            return decoded.cpu(), lengths.cpu()
        if not (logits.is_contiguous() or logits.permute(1, 0, 2).is_contiguous()):
            logits = logits.contiguous()
        lengths_in = None
        if logits_lengths_ is not None:
            lengths_in = _as_index(logits_lengths_, torch.device("cpu"), "logits_lengths").contiguous()
        d = self._desc(logits, lengths_in)
        B, T = logits.size(0), logits.size(1)
        decoded = torch.empty(B, T, dtype=torch.int64, pin_memory=True)
        lengths = torch.empty(B, dtype=torch.int64, pin_memory=True)
        dev = torch.cuda.current_device()
        h = self._host.get(dev)
        if h is None:
            h = self._host[dev] = _HostEngine(dev)
        _lib.check(self._L.e2e_ctc_engine_greedy_host(h.handle, ctypes.byref(d), _ptr(logits), _ptr(lengths_in),
                                                      _ptr(decoded), _ptr(lengths)))
        return decoded, lengths


class CTCBeamEngine(CTCGreedyEngine):
    """``cpp_ctc_decoder.CTCDecoder(blank_idx, beam_width_, labels, lm_path="", lmwt_, wip_, oov_penalty_,
    case_sensitive)`` without a language model (src/decoders/ctc_decoder_py.cpp:5-39): ``decode(logits_,
    logits_lengths_)`` is the prefix beam search of src/decoders/ctc_decoder.cpp:153-198,353-441 on the GPU and
    ``decode_greedy`` the inherited greedy path.  Returns CPU int64 tensors like the reference:
    ``(decoded_targets [B, max length] zero padded, decoded_targets_lengths [B])``; the sentences are assembled by
    the Python wrapper.  ``last_ties`` holds, per utterance of the last call, how many prunes had equal scores on
    both sides of the cut (where the reference's pick is libstdc++'s; see include/e2e_ctc.h)."""

    def __init__(self, blank_idx=0, beam_width=100, labels=None, wip=0.0):
        super().__init__(blank_idx)
        self.beam_width = int(beam_width)
        if self.beam_width < 1:
            raise ValueError("beam_width must be >= 1")
        labels = list(labels or [])
        # ctc_decoder.cpp:56-60: space_id = index of " " in labels, -1 when there is none
        self.space_idx = labels.index(" ") if " " in labels else -1
        self.wip = float(wip)
        self.last_ties = None

    def _beam_desc(self, logits, lengths, from_logits):
        d = self._desc(logits, lengths)
        d.from_logits = 1 if from_logits else 0
        if not -1 <= self.space_idx < logits.size(2):
            raise ValueError("the space label %d is outside the alphabet [0,%d)" % (self.space_idx, logits.size(2)))
        return d

    def decode_device(self, logits, logits_lengths=None, from_logits=False):
        """Device tensors in, device tensors out (no synchronisation): ``(decoded [B,T] int64 zero padded, lengths [B],
        ties [B])``."""
        _require_cuda()
        logits = logits.detach()
        dev = logits.device
        if not _dense3(logits):
            logits = logits.contiguous()
        if logits_lengths is not None:
            logits_lengths = _as_index(logits_lengths, dev, "logits_lengths").contiguous()
        d = self._beam_desc(logits, logits_lengths, from_logits)
        B, T = logits.size(0), logits.size(1)
        with _on_device(dev):
            need = self._L.e2e_ctc_beam_workspace_bytes(ctypes.byref(d), self.beam_width)
            if need == 0:
                raise _lib.E2EError(_lib.E2E_ERR_UNSUPPORTED, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            decoded = torch.empty(B, T, dtype=torch.int64, device=dev)
            lengths = torch.empty(B, dtype=torch.int64, device=dev)
            ties = torch.empty(B, dtype=torch.int64, device=dev)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_beam_decode_device(
                ctypes.byref(d), self.beam_width, self.space_idx, self.wip, _ptr(logits), _ptr(logits_lengths),
                _ptr(decoded), _ptr(lengths), _ptr(ties), _ptr(ws), ws.numel(), _stream(dev)))
        return decoded, lengths, ties

    def decode(self, logits_, logits_lengths_=None, from_logits=False):
        _require_cuda()
        logits = logits_.detach()
        if logits.is_cuda:
            decoded, lengths, ties = self.decode_device(logits, logits_lengths_, from_logits)
            decoded, lengths, ties = decoded.cpu(), lengths.cpu(), ties.cpu()
        else:
            if not (logits.is_contiguous() or logits.permute(1, 0, 2).is_contiguous()):
                logits = logits.contiguous()
            lengths_in = None
            if logits_lengths_ is not None:
                lengths_in = _as_index(logits_lengths_, torch.device("cpu"), "logits_lengths").contiguous()
            d = self._beam_desc(logits, lengths_in, from_logits)
            B, T = logits.size(0), logits.size(1)
            decoded = torch.empty(B, T, dtype=torch.int64, pin_memory=True)
            lengths = torch.empty(B, dtype=torch.int64, pin_memory=True)
            ties = torch.empty(B, dtype=torch.int64, pin_memory=True)
            dev = torch.cuda.current_device()
            h = self._host.get(dev)
            if h is None:
                h = self._host[dev] = _HostEngine(dev)
            _lib.check(self._L.e2e_ctc_engine_beam_host(h.handle, ctypes.byref(d), self.beam_width, self.space_idx,
                                                        self.wip, _ptr(logits), _ptr(lengths_in), _ptr(decoded),
                                                        _ptr(lengths), _ptr(ties)))
        self.last_ties = ties
        # ctc_decoder.cpp:186-196: the result matrix is as wide as the longest decoded sequence
        width = int(lengths.max()) if lengths.numel() else 0
        return decoded[:, :width].contiguous(), lengths

    def _n_best(self, n_best):
        n_best = self.beam_width if n_best is None else int(n_best)
        if not 1 <= n_best <= self.beam_width:
            raise ValueError("n_best %d outside [1, beam_width = %d]" % (n_best, self.beam_width))
        return n_best

    def decode_nbest_device(self, logits, logits_lengths=None, n_best=None, from_logits=False):
        """The ``n_best`` best prefixes of the same search (default: the whole final beam), device tensors in, device
        tensors out (no synchronisation): ``(decoded [B,N,T] int64 zero padded, lengths [B,N], scores [B,N] float64,
        log_probs [B,N] float64, ties [B])``.  Ranked by ``scores = log_probs - words * wip``, highest first, equal
        scores in beam order; hypothesis 0 is what ``decode_device`` returns.  Slots past the number of prefixes in
        the final beam have length 0 and ``-inf`` scores (see include/e2e_ctc.h)."""
        _require_cuda()
        n_best = self._n_best(n_best)
        logits = logits.detach()
        dev = logits.device
        if not _dense3(logits):
            logits = logits.contiguous()
        if logits_lengths is not None:
            logits_lengths = _as_index(logits_lengths, dev, "logits_lengths").contiguous()
        d = self._beam_desc(logits, logits_lengths, from_logits)
        B, T = logits.size(0), logits.size(1)
        with _on_device(dev):
            need = self._L.e2e_ctc_beam_nbest_workspace_bytes(ctypes.byref(d), self.beam_width, n_best)
            if need == 0:
                raise _lib.E2EError(_lib.E2E_ERR_UNSUPPORTED, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            decoded = torch.empty(B, n_best, T, dtype=torch.int64, device=dev)
            lengths = torch.empty(B, n_best, dtype=torch.int64, device=dev)
            scores = torch.empty(B, n_best, dtype=torch.float64, device=dev)
            log_probs = torch.empty(B, n_best, dtype=torch.float64, device=dev)
            ties = torch.empty(B, dtype=torch.int64, device=dev)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_beam_nbest_device(
                ctypes.byref(d), self.beam_width, n_best, self.space_idx, self.wip, _ptr(logits), _ptr(logits_lengths),
                _ptr(decoded), _ptr(lengths), _ptr(scores), _ptr(log_probs), _ptr(ties), _ptr(ws), ws.numel(),
                _stream(dev)))
        return decoded, lengths, scores, log_probs, ties

    def decode_nbest(self, logits_, logits_lengths_=None, n_best=None, from_logits=False):
        """``decode_nbest_device`` for CPU or CUDA input, CPU results (CPU input goes through the host engine, as in
        ``decode``): ``(decoded [B,N,longest hypothesis], lengths [B,N], scores [B,N], log_probs [B,N])``;
        ``last_ties`` holds the tie counters."""
        _require_cuda()
        n_best = self._n_best(n_best)
        logits = logits_.detach()
        if logits.is_cuda:
            out = self.decode_nbest_device(logits, logits_lengths_, n_best, from_logits)
            decoded, lengths, scores, log_probs, ties = (t.cpu() for t in out)
        else:
            if not (logits.is_contiguous() or logits.permute(1, 0, 2).is_contiguous()):
                logits = logits.contiguous()
            lengths_in = None
            if logits_lengths_ is not None:
                lengths_in = _as_index(logits_lengths_, torch.device("cpu"), "logits_lengths").contiguous()
            d = self._beam_desc(logits, lengths_in, from_logits)
            B, T = logits.size(0), logits.size(1)
            decoded = torch.empty(B, n_best, T, dtype=torch.int64, pin_memory=True)
            lengths = torch.empty(B, n_best, dtype=torch.int64, pin_memory=True)
            scores = torch.empty(B, n_best, dtype=torch.float64, pin_memory=True)
            log_probs = torch.empty(B, n_best, dtype=torch.float64, pin_memory=True)
            ties = torch.empty(B, dtype=torch.int64, pin_memory=True)
            dev = torch.cuda.current_device()
            h = self._host.get(dev)
            if h is None:
                h = self._host[dev] = _HostEngine(dev)
            _lib.check(self._L.e2e_ctc_engine_beam_nbest_host(
                h.handle, ctypes.byref(d), self.beam_width, n_best, self.space_idx, self.wip, _ptr(logits),
                _ptr(lengths_in), _ptr(decoded), _ptr(lengths), _ptr(scores), _ptr(log_probs), _ptr(ties)))
        self.last_ties = ties
        width = int(lengths.max()) if lengths.numel() else 0
        return decoded[:, :, :width].contiguous(), lengths, scores, log_probs

    def _score_args(self, logits, hyps, hyp_lengths, logits_lengths, from_logits):
        """The checks and the C descriptor shared by ``score_device`` and ``score_backward_device``: returns ``(logits,
        hyps [B*N, Lmax], hyp_lengths [B*N], logits_lengths, desc, device, N)`` with every tensor on the device.  It
        enters ``_on_device(device)`` itself for the copies and returns outside it: callers enter it again for their
        allocations and the launch.  Host-resident lengths / labels are checked here, device-resident ones on the device
        (the loss's rule, ``_Problem``)."""
        logits = logits.detach()
        if logits.dim() != 3:
            raise ValueError("logits must be [batch, frames, alphabet], got %s" % (tuple(logits.shape),))
        if logits.dtype not in _DTYPES:
            raise TypeError("unsupported logits dtype %s" % logits.dtype)
        B, T, V = logits.shape
        if B < 1 or T < 1 or V < 1:
            raise ValueError("empty logits %s" % (tuple(logits.shape),))
        if not 0 <= self.blank_idx < V:
            raise ValueError("blank_idx %d outside the alphabet [0,%d)" % (self.blank_idx, V))
        if hyps.dim() != 3 or hyps.size(0) != B:
            raise ValueError("hyps must be [batch, n_hyp, max_length], got %s" % (tuple(hyps.shape),))
        N, Lmax = hyps.size(1), hyps.size(2)
        if N < 1:
            raise ValueError("hyps holds no hypothesis")
        if tuple(hyp_lengths.shape) != (B, N):
            raise ValueError("hyp_lengths must have shape [batch, n_hyp] = %s, got %s" % ((B, N), tuple(hyp_lengths.shape)))
        if logits_lengths is not None and (logits_lengths.dim() != 1 or logits_lengths.numel() != B):
            raise ValueError("logits_lengths must have shape [batch]")
        lim = _limits()
        if Lmax > lim.max_targets or V > lim.max_alphabet:
            raise NotImplementedError("the scorer supports hypothesis length <= %d and alphabet <= %d"
                                      % (lim.max_targets, lim.max_alphabet))
        if logits_lengths is not None and not logits_lengths.is_cuda:
            ll = logits_lengths.to(torch.int64)
            if bool((ll < 1).any()) or bool((ll > T).any()):
                raise ValueError("logits_lengths must be in [1, %d]" % T)
        if not hyp_lengths.is_cuda:
            hl = hyp_lengths.to(torch.int64)
            if bool((hl < 0).any()) or bool((hl > Lmax).any()):
                raise ValueError("hyp_lengths must be in [0, %d]" % Lmax)
            if not hyps.is_cuda and Lmax > 0:
                valid = torch.arange(Lmax) < hl.unsqueeze(-1)
                hg = hyps.to(torch.int64)
                if bool(((hg < 0) | (hg >= V))[valid].any()):
                    raise ValueError("hypothesis labels must be in [0, %d)" % V)
        dev = logits.device if logits.is_cuda else torch.device("cuda", torch.cuda.current_device())
        with _on_device(dev):
            if not logits.is_cuda:
                logits = logits.to(dev)
            if not _dense3(logits):
                logits = logits.contiguous()
            hyps = _as_index(hyps, dev, "hyps").reshape(B * N, Lmax)
            if Lmax > 0 and hyps.stride(1) != 1:
                hyps = hyps.contiguous()
            hyp_lengths = _as_index(hyp_lengths, dev, "hyp_lengths").reshape(B * N).contiguous()
            if logits_lengths is not None:
                logits_lengths = _as_index(logits_lengths, dev, "logits_lengths").contiguous()
                if logits_lengths.dtype != hyp_lengths.dtype:
                    logits_lengths, hyp_lengths = logits_lengths.to(torch.int64), hyp_lengths.to(torch.int64)
        d = _lib.Desc()
        d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
        d.blank_idx, d.dtype = self.blank_idx, _DTYPES[logits.dtype]
        d.targets_itype, d.lengths_itype = _ITYPES[hyps.dtype], _ITYPES[hyp_lengths.dtype]
        d.from_logits = 1 if from_logits else 0
        d.logits_stride_b, d.logits_stride_t = logits.stride(0), logits.stride(1)
        d.targets_stride_b = hyps.stride(0) if Lmax > 0 else 0
        return logits, hyps, hyp_lengths, logits_lengths, d, dev, N

    def score_device(self, logits, hyps, hyp_lengths, logits_lengths=None, from_logits=False):
        """CTC log-likelihood log p(hypothesis | x) of N hypotheses per utterance: ``[B, N]`` float64 on the logits' device,
        minus the CTC loss of each (utterance, hypothesis) pair, without synchronising.  ``hyps`` ``[B, N, Lmax]`` and
        ``hyp_lengths`` ``[B, N]``, int32 or int64, any device; ``logits_lengths`` ``[B]`` or ``None`` (all frames).
        Forward only: no gradient and nothing kept for one (``score_backward_device`` computes it).  An infeasible
        hypothesis scores ``-inf``; out-of-range lengths / labels raise ``ValueError`` when they live on the host and give
        NaN scores when they live on the device.  Input on the CPU is copied to the current CUDA device."""
        _require_cuda()
        logits, hyps, hyp_lengths, logits_lengths, d, dev, N = self._score_args(logits, hyps, hyp_lengths, logits_lengths,
                                                                               from_logits)
        with _on_device(dev):
            need = self._L.e2e_ctc_score_workspace_bytes(ctypes.byref(d), N)
            if need == 0:
                raise _lib.E2EError(_lib.E2E_ERR_UNSUPPORTED, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            scores = torch.empty(d.batch, N, dtype=torch.float64, device=dev)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_score_device(
                ctypes.byref(d), N, _ptr(logits), _ptr(hyps), _ptr(logits_lengths), _ptr(hyp_lengths), _ptr(scores),
                _ptr(ws), ws.numel(), _stream(dev)))
        return scores

    def score_backward_workspace_bytes(self, logits, hyps, hyp_lengths, logits_lengths=None, from_logits=False):
        """Workspace bytes ``score_backward_device`` allocates for these arguments."""
        _require_cuda()
        _, _, _, _, d, dev, N = self._score_args(logits, hyps, hyp_lengths, logits_lengths, from_logits)
        with _on_device(dev):
            return int(self._L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(d), N))

    def score_backward_device(self, logits, hyps, hyp_lengths, grad_scores, logits_lengths=None, from_logits=False):
        """The gradient of ``sum(grad_scores * score_device(...))`` with respect to ``logits``, on the logits' device (CPU
        input: the current CUDA device) without synchronising: a tensor of the logits' shape and dtype, in their layout
        when it is dense.  With ``gamma_bn(t, v)`` the occupancy of symbol ``v`` at frame ``t`` under hypothesis ``n``:
        ``sum_n g[b,n] gamma_bn(t,v)`` for log-probabilities, ``sum_n g[b,n] (gamma_bn(t,v) - softmax(x_bt)_v)`` for raw
        logits, 0 past the utterance's frames.  This is the derivative of the score; it is not ``CTCLoss``'s convention
        (``exp(lp) - gamma`` on log-probabilities, ``exp(lp)`` in padding rows).  ``grad_scores`` ``[B, N]`` (float64
        on the device): a hypothesis with ``g == 0`` costs no sweep; an infeasible one contributes 0; a device-resident
        bad length or label gives NaN rows for its utterance only."""
        _require_cuda()
        logits, hyps, hyp_lengths, logits_lengths, d, dev, N = self._score_args(logits, hyps, hyp_lengths, logits_lengths,
                                                                               from_logits)
        B = d.batch
        if tuple(grad_scores.shape) != (B, N):
            raise ValueError("grad_scores must have shape [batch, n_hyp] = %s, got %s" % ((B, N), tuple(grad_scores.shape)))
        with _on_device(dev):
            need = self._L.e2e_ctc_score_backward_workspace_bytes(ctypes.byref(d), N)
            if need == 0:
                raise _lib.E2EError(_lib.E2E_ERR_UNSUPPORTED, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            g = grad_scores.detach().to(dev, torch.float64).contiguous()
            grads = torch.empty_like(logits)
            d.grads_stride_b, d.grads_stride_t = grads.stride(0), grads.stride(1)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_score_backward_device(
                ctypes.byref(d), N, _ptr(logits), _ptr(hyps), _ptr(logits_lengths), _ptr(hyp_lengths), _ptr(g),
                _ptr(grads), _ptr(ws), ws.numel(), _stream(dev)))
        return grads

    def align_device(self, logits, hyps, hyp_lengths, logits_lengths=None, from_logits=False):
        """Best-path (Viterbi) alignment of N hypotheses per utterance over the CTC lattice, on the logits' device and without
        synchronising: ``(alignments [B, N, T] int64, token_starts [B, N, Lmax] int64, token_ends [B, N, Lmax] int64,
        path_scores [B, N] float64)``.  ``hyps`` ``[B, N, Lmax]`` and ``hyp_lengths`` ``[B, N]``, int32 or int64, any device;
        ``logits_lengths`` ``[B]`` or ``None`` (all frames).  ``alignments[b, n]`` is the label id of every frame on the best
        path (``get_alignment_3d``'s row for that hypothesis, ``-100`` past the utterance's frames); token ``k`` covers the
        frames ``[token_starts, token_ends)``; ``path_scores`` is the best path's log-probability (``<= score_device``).  An
        infeasible hypothesis gives ``-inf`` and spans of ``-1``; out-of-range lengths / labels raise ``ValueError`` when
        they live on the host and give NaN scores and ``-1`` spans when they live on the device.  Input on the CPU is
        copied to the current CUDA device."""
        _require_cuda()
        logits = logits.detach()
        if logits.dim() != 3:
            raise ValueError("logits must be [batch, frames, alphabet], got %s" % (tuple(logits.shape),))
        if logits.dtype not in _DTYPES:
            raise TypeError("unsupported logits dtype %s" % logits.dtype)
        B, T, V = logits.shape
        if B < 1 or T < 1 or V < 1:
            raise ValueError("empty logits %s" % (tuple(logits.shape),))
        if not 0 <= self.blank_idx < V:
            raise ValueError("blank_idx %d outside the alphabet [0,%d)" % (self.blank_idx, V))
        if hyps.dim() != 3 or hyps.size(0) != B:
            raise ValueError("hyps must be [batch, n_hyp, max_length], got %s" % (tuple(hyps.shape),))
        N, Lmax = hyps.size(1), hyps.size(2)
        if N < 1:
            raise ValueError("hyps holds no hypothesis")
        if tuple(hyp_lengths.shape) != (B, N):
            raise ValueError("hyp_lengths must have shape [batch, n_hyp] = %s, got %s" % ((B, N), tuple(hyp_lengths.shape)))
        if logits_lengths is not None and (logits_lengths.dim() != 1 or logits_lengths.numel() != B):
            raise ValueError("logits_lengths must have shape [batch]")
        lim = _limits()
        if Lmax > ALIGN_MAX_TARGETS or V > lim.max_alphabet:
            raise NotImplementedError("the aligner supports hypothesis length <= %d and alphabet <= %d"
                                      % (ALIGN_MAX_TARGETS, lim.max_alphabet))
        # the loss's rule (_Problem): host-resident lengths / labels are checked here, device-resident ones on the device
        if logits_lengths is not None and not logits_lengths.is_cuda:
            ll = logits_lengths.to(torch.int64)
            if bool((ll < 1).any()) or bool((ll > T).any()):
                raise ValueError("logits_lengths must be in [1, %d]" % T)
        if not hyp_lengths.is_cuda:
            hl = hyp_lengths.to(torch.int64)
            if bool((hl < 0).any()) or bool((hl > Lmax).any()):
                raise ValueError("hyp_lengths must be in [0, %d]" % Lmax)
            if not hyps.is_cuda and Lmax > 0:
                valid = torch.arange(Lmax) < hl.unsqueeze(-1)
                hg = hyps.to(torch.int64)
                if bool(((hg < 0) | (hg >= V))[valid].any()):
                    raise ValueError("hypothesis labels must be in [0, %d)" % V)
        dev = logits.device if logits.is_cuda else torch.device("cuda", torch.cuda.current_device())
        with _on_device(dev):
            if not logits.is_cuda:
                logits = logits.to(dev)
            if not _dense3(logits):
                logits = logits.contiguous()
            hyps = _as_index(hyps, dev, "hyps").reshape(B * N, Lmax)
            if Lmax > 0 and hyps.stride(1) != 1:
                hyps = hyps.contiguous()
            hyp_lengths = _as_index(hyp_lengths, dev, "hyp_lengths").reshape(B * N).contiguous()
            if logits_lengths is not None:
                logits_lengths = _as_index(logits_lengths, dev, "logits_lengths").contiguous()
                if logits_lengths.dtype != hyp_lengths.dtype:
                    logits_lengths, hyp_lengths = logits_lengths.to(torch.int64), hyp_lengths.to(torch.int64)
            d = _lib.Desc()
            d.batch, d.max_frames, d.alphabet, d.max_targets = B, T, V, Lmax
            d.blank_idx, d.dtype = self.blank_idx, _DTYPES[logits.dtype]
            d.targets_itype, d.lengths_itype = _ITYPES[hyps.dtype], _ITYPES[hyp_lengths.dtype]
            d.from_logits = 1 if from_logits else 0
            d.logits_stride_b, d.logits_stride_t = logits.stride(0), logits.stride(1)
            d.targets_stride_b = hyps.stride(0) if Lmax > 0 else 0
            need = self._L.e2e_ctc_align_nbest_workspace_bytes(ctypes.byref(d), N)
            if need == 0:
                raise _lib.E2EError(_lib.E2E_ERR_UNSUPPORTED, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            aligned = torch.empty(B, N, T, dtype=torch.int64, device=dev)
            starts = torch.empty(B, N, Lmax, dtype=torch.int64, device=dev)
            ends = torch.empty(B, N, Lmax, dtype=torch.int64, device=dev)
            path_scores = torch.empty(B, N, dtype=torch.float64, device=dev)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_align_nbest_device(
                ctypes.byref(d), N, _ptr(logits), _ptr(hyps), _ptr(logits_lengths), _ptr(hyp_lengths), _ptr(aligned),
                _ptr(starts), _ptr(ends), _ptr(path_scores), _ptr(ws), ws.numel(), _stream(dev)))
        return aligned, starts, ends, path_scores

    def errors_device(self, hyps, hyp_lengths, refs, ref_lengths, words=False):
        """Edit distance of N hypotheses per utterance against the utterance's reference, on the GPU without
        synchronising: ``(errors, substitutions, insertions, deletions)`` ``[B, N]`` int64 and ``reference_units`` ``[B]``
        int64 (the WER / CER denominator).  ``hyps`` ``[B, N, W]`` with ``hyp_lengths`` ``[B, N]``, or ``[B, W]`` with
        ``[B]`` (one hypothesis per utterance, counted as N = 1); ``refs`` ``[B, Wr]`` with ``ref_lengths`` ``[B]`` (the
        loss's ``targets`` / ``targets_lengths``).  int32 and int64 may be mixed.  ``decode``'s empty result (the single
        symbol ``-1`` with length 1) is the empty hypothesis.  ``words=False`` counts tokens (CER for character labels);
        ``words=True`` counts words, maximal runs of tokens other than the label ``" "`` (WER).  Errors are the least
        number of unit substitutions, insertions and deletions turning the reference into the hypothesis, split as the
        least-errors alignment with the most substitutions.  Out-of-range lengths raise ``ValueError`` when they live on
        the host and give ``-1`` counts for their pairs (a reference length: all N of its utterance and its
        ``reference_units``) when they live on the device.  Input on the CPU is copied to the current CUDA device."""
        _require_cuda()
        if hyps.dim() == 2:                             # one hypothesis per utterance: decode's / decode_greedy's result
            hyps, hyp_lengths = hyps[:, None], hyp_lengths.reshape(-1, 1)
        if hyps.dim() != 3:
            raise ValueError("hyps must be [batch, n_hyp, width] or [batch, width], got %s" % (tuple(hyps.shape),))
        B, N, W = hyps.shape
        if B < 1 or N < 1:
            raise ValueError("hyps holds no hypothesis: %s" % (tuple(hyps.shape),))
        if tuple(hyp_lengths.shape) != (B, N):
            raise ValueError("hyp_lengths must have shape %s, got %s" % ((B, N), tuple(hyp_lengths.shape)))
        if refs.dim() != 2 or refs.size(0) != B:
            raise ValueError("refs must be [batch = %d, width], got %s" % (B, tuple(refs.shape)))
        if tuple(ref_lengths.shape) != (B,):
            raise ValueError("ref_lengths must have shape [batch = %d], got %s" % (B, tuple(ref_lengths.shape)))
        Wr = refs.size(1)
        if Wr > EDIT_MAX_REF_WIDTH or W > EDIT_MAX_HYP_WIDTH:
            raise NotImplementedError("the edit distance supports reference width <= %d and hypothesis width <= %d, got %d and %d"
                                      % (EDIT_MAX_REF_WIDTH, EDIT_MAX_HYP_WIDTH, Wr, W))
        sep = -1
        if words:
            if self.space_idx < 0:
                raise ValueError("word level needs a \" \" label to separate words; the labels have none")
            sep = self.space_idx
        hyp_lengths = empty_marker_as_empty(hyps, hyp_lengths)
        # the loss's rule (_Problem): host-resident lengths are checked here, device-resident ones on the device
        for name, lens, width in (("hyp_lengths", hyp_lengths, W), ("ref_lengths", ref_lengths, Wr)):
            if not lens.is_cuda:
                ll = lens.to(torch.int64)
                if bool((ll < 0).any()) or bool((ll > width).any()):
                    raise ValueError("%s must be in [0, %d]" % (name, width))
        for name, t in (("hyps", hyps), ("refs", refs)):
            if t.is_floating_point() or t.dtype == torch.bool:
                raise TypeError("%s must be an integer tensor, got %s" % (name, t.dtype))
        dev = next((t.device for t in (hyps, refs, hyp_lengths, ref_lengths) if t.is_cuda),
                   torch.device("cuda", torch.cuda.current_device()))
        with _on_device(dev):
            hyps = _as_index(hyps, dev, "hyps").reshape(B * N, W)
            refs = _as_index(refs, dev, "refs")
            if hyps.dtype != refs.dtype:
                hyps, refs = hyps.to(torch.int64), refs.to(torch.int64)
            if W > 0 and (hyps.stride(1) != 1 or hyps.stride(0) < W):
                hyps = hyps.contiguous()
            if Wr > 0 and (refs.stride(1) != 1 or refs.stride(0) < Wr):
                refs = refs.contiguous()
            hyp_lengths = _as_index(hyp_lengths, dev, "hyp_lengths").reshape(B * N).contiguous()
            ref_lengths = _as_index(ref_lengths, dev, "ref_lengths").contiguous()
            if hyp_lengths.dtype != ref_lengths.dtype:
                hyp_lengths, ref_lengths = hyp_lengths.to(torch.int64), ref_lengths.to(torch.int64)
            d = _lib.EditDesc()
            d.batch, d.n_hyp, d.hyp_width, d.ref_width = B, N, W, Wr
            d.tokens_itype, d.lengths_itype = _ITYPES[hyps.dtype], _ITYPES[hyp_lengths.dtype]
            d.separator = sep
            d.hyp_stride_b = hyps.stride(0) if W > 0 else 0
            d.ref_stride_b = refs.stride(0) if Wr > 0 else 0
            need = self._L.e2e_ctc_edit_distance_workspace_bytes(ctypes.byref(d))
            if need == 0:
                raise _lib.E2EError(_lib.E2E_ERR_UNSUPPORTED, self._L.e2e_last_error_string().decode("utf-8", "replace"))
            counts = torch.empty(4, B, N, dtype=torch.int64, device=dev)
            ref_units = torch.empty(B, dtype=torch.int64, device=dev)
            ws = torch.empty(need, dtype=torch.uint8, device=dev)
            _lib.check(self._L.e2e_ctc_edit_distance_device(
                ctypes.byref(d), _ptr(hyps), _ptr(hyp_lengths), _ptr(refs), _ptr(ref_lengths), _ptr(counts[0]),
                _ptr(counts[1]), _ptr(counts[2]), _ptr(counts[3]), _ptr(ref_units), _ptr(ws), ws.numel(), _stream(dev)))
        return counts[0], counts[1], counts[2], counts[3], ref_units

"""ctypes binding of libe2e_ctc.so -- the C ABI declared in include/e2e_ctc.h.

The library is the product: if it is missing or cannot be loaded this module raises (there is no
Python / CPU fallback anywhere on the hot path).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# E2E_CTC_LIB: developer hook -- load an experiment build of the SAME library (python -m end2end_b200.build --tag X)
LIB_PATH = os.environ.get("E2E_CTC_LIB") or os.path.join(_HERE, "lib", "libe2e_ctc.so")

E2E_OK = 0
E2E_ERR_UNSUPPORTED = 2
E2E_ERR_LENGTHS = 5
E2E_F32, E2E_BF16, E2E_F16, E2E_F64 = 0, 1, 2, 3
E2E_I32, E2E_I64 = 0, 1

#: every symbol include/e2e_ctc.h declares (tests check the .so exports all of them)
EXPORTS = (
    "e2e_ctc_version", "e2e_last_error_string", "e2e_ctc_get_limits",
    "e2e_ctc_loss_workspace_bytes", "e2e_ctc_loss_forward_device", "e2e_ctc_loss_backward_device",
    "e2e_ctc_loss_fwd_bwd_device", "e2e_ctc_loss_step_device", "e2e_ctc_scale_rows_device", "e2e_ctc_loss_reduce_device", "e2e_ctc_loss_check_device",
    "e2e_ctc_greedy_workspace_bytes", "e2e_ctc_greedy_decode_device",
    "e2e_ctc_engine_create", "e2e_ctc_engine_destroy", "e2e_ctc_engine_loss_host",
    "e2e_ctc_engine_greedy_host", "e2e_ctc_engine_last_traffic", "e2e_ctc_launch_count",
    "e2e_ctc_profile_enable", "e2e_ctc_profile_read",
    "e2e_ctc_comm_unique_id", "e2e_ctc_comm_create", "e2e_ctc_comm_destroy", "e2e_ctc_comm_allreduce_sum",
    "e2e_ctc_graph_create", "e2e_ctc_graph_launch", "e2e_ctc_graph_destroy",
    "e2e_ctc_viterbi_workspace_bytes", "e2e_ctc_viterbi_align_device",
    "e2e_ctc_noblank_workspace_bytes", "e2e_ctc_noblank_fwd_bwd_device",
    "e2e_ctc_host_alloc", "e2e_ctc_host_free",
    "e2e_ctc_beam_workspace_bytes", "e2e_ctc_beam_decode_device", "e2e_ctc_engine_beam_host",
    "e2e_ctc_beam_nbest_workspace_bytes", "e2e_ctc_beam_nbest_device", "e2e_ctc_engine_beam_nbest_host",
    "e2e_ctc_score_workspace_bytes", "e2e_ctc_score_device",
    "e2e_ctc_score_backward_workspace_bytes", "e2e_ctc_score_backward_device",
    "e2e_ctc_align_nbest_workspace_bytes", "e2e_ctc_align_nbest_device",
    "e2e_ctc_edit_distance_workspace_bytes", "e2e_ctc_edit_distance_device",
)
KERNEL_KINDS = ("row_stats", "lattice", "gradient", "loss_reduce", "argmax", "collapse", "scale_rows", "viterbi", "ctc_without_blank", "beam_search", "order", "score",
                "score_backward", "score_backward_rows", "edit_distance")


class Desc(ctypes.Structure):
    """struct e2e_ctc_desc"""
    _fields_ = [
        ("batch", ctypes.c_int32), ("max_frames", ctypes.c_int32), ("alphabet", ctypes.c_int32),
        ("max_targets", ctypes.c_int32), ("blank_idx", ctypes.c_int32), ("dtype", ctypes.c_int32),
        ("targets_itype", ctypes.c_int32), ("lengths_itype", ctypes.c_int32),
        ("from_logits", ctypes.c_int32), ("reserved0", ctypes.c_int32),
        ("logits_stride_b", ctypes.c_int64), ("logits_stride_t", ctypes.c_int64),
        ("grads_stride_b", ctypes.c_int64), ("grads_stride_t", ctypes.c_int64),
        ("targets_stride_b", ctypes.c_int64),
    ]


class EditDesc(ctypes.Structure):
    """struct e2e_ctc_edit_desc"""
    _fields_ = [
        ("batch", ctypes.c_int32), ("n_hyp", ctypes.c_int32), ("hyp_width", ctypes.c_int32),
        ("ref_width", ctypes.c_int32), ("tokens_itype", ctypes.c_int32), ("lengths_itype", ctypes.c_int32),
        ("separator", ctypes.c_int32), ("reserved0", ctypes.c_int32),
        ("hyp_stride_b", ctypes.c_int64), ("ref_stride_b", ctypes.c_int64),
    ]


class Limits(ctypes.Structure):
    """struct e2e_ctc_limits"""
    _fields_ = [("max_alphabet", ctypes.c_int32), ("max_targets", ctypes.c_int32),
                ("abi_version", ctypes.c_int32), ("sm_arch", ctypes.c_int32)]


class E2EError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libe2e_ctc error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load():
    """dlopen the library (once).  Raises if it has not been built: run ``python -m end2end_b200.build``."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "end2end_b200: %s is missing -- build it with `python -m end2end_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, sz, dbl = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t, ctypes.c_double
    dp = ctypes.POINTER(Desc)
    L.e2e_ctc_version.restype = ctypes.c_char_p
    L.e2e_last_error_string.restype = ctypes.c_char_p
    L.e2e_ctc_get_limits.argtypes = [ctypes.POINTER(Limits)]
    L.e2e_ctc_loss_workspace_bytes.argtypes = [dp]
    L.e2e_ctc_loss_workspace_bytes.restype = sz
    L.e2e_ctc_loss_forward_device.argtypes = [dp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_loss_backward_device.argtypes = [dp, vp, vp, vp, vp, vp, i32, dbl, vp, vp, sz, vp]
    L.e2e_ctc_loss_fwd_bwd_device.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_loss_step_device.argtypes = [dp, vp, vp, vp, vp, vp, vp, dbl, vp, vp, dbl, vp, sz, vp]
    L.e2e_ctc_scale_rows_device.argtypes = [dp, vp, vp, i32, vp]
    L.e2e_ctc_loss_reduce_device.argtypes = [vp, i32, i32, dbl, vp, vp, vp]
    L.e2e_ctc_loss_check_device.argtypes = [vp, ctypes.POINTER(i32), vp]
    L.e2e_ctc_greedy_workspace_bytes.argtypes = [dp]
    L.e2e_ctc_greedy_workspace_bytes.restype = sz
    L.e2e_ctc_greedy_decode_device.argtypes = [dp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_engine_create.argtypes = [i32, ctypes.POINTER(vp)]
    L.e2e_ctc_engine_destroy.argtypes = [vp]
    L.e2e_ctc_engine_destroy.restype = None
    L.e2e_ctc_engine_loss_host.argtypes = [vp, dp, vp, vp, vp, vp, vp, vp]
    L.e2e_ctc_engine_greedy_host.argtypes = [vp, dp, vp, vp, vp, vp]
    L.e2e_ctc_engine_last_traffic.argtypes = [vp, ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]
    L.e2e_ctc_launch_count.restype = ctypes.c_uint64
    L.e2e_ctc_profile_enable.argtypes = [i32]
    L.e2e_ctc_profile_read.argtypes = [ctypes.POINTER(dbl), ctypes.POINTER(ctypes.c_uint64), i32]
    L.e2e_ctc_comm_unique_id.argtypes = [vp]
    L.e2e_ctc_comm_create.argtypes = [vp, i32, i32, ctypes.POINTER(vp)]
    L.e2e_ctc_comm_destroy.argtypes = [vp]
    L.e2e_ctc_comm_destroy.restype = None
    L.e2e_ctc_comm_allreduce_sum.argtypes = [vp, vp, ctypes.c_int64, i32, vp]
    L.e2e_ctc_graph_create.argtypes = [dp, vp, vp, vp, vp, vp, vp, dbl, vp, vp, dbl, vp, sz, vp, ctypes.POINTER(vp)]
    L.e2e_ctc_viterbi_workspace_bytes.argtypes = [dp, i32]
    L.e2e_ctc_viterbi_workspace_bytes.restype = sz
    L.e2e_ctc_viterbi_align_device.argtypes = [dp, i32, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_viterbi_align_device.restype = ctypes.c_int
    L.e2e_ctc_noblank_workspace_bytes.argtypes = [dp]
    L.e2e_ctc_noblank_workspace_bytes.restype = sz
    L.e2e_ctc_noblank_fwd_bwd_device.argtypes = [dp, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_noblank_fwd_bwd_device.restype = ctypes.c_int
    L.e2e_ctc_beam_workspace_bytes.argtypes = [dp, i32]
    L.e2e_ctc_beam_workspace_bytes.restype = sz
    L.e2e_ctc_beam_decode_device.argtypes = [dp, i32, i32, dbl, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_beam_decode_device.restype = ctypes.c_int
    L.e2e_ctc_engine_beam_host.argtypes = [vp, dp, i32, i32, dbl, vp, vp, vp, vp, vp]
    L.e2e_ctc_engine_beam_host.restype = ctypes.c_int
    L.e2e_ctc_beam_nbest_workspace_bytes.argtypes = [dp, i32, i32]
    L.e2e_ctc_beam_nbest_workspace_bytes.restype = sz
    L.e2e_ctc_beam_nbest_device.argtypes = [dp, i32, i32, i32, dbl, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_beam_nbest_device.restype = ctypes.c_int
    L.e2e_ctc_engine_beam_nbest_host.argtypes = [vp, dp, i32, i32, i32, dbl, vp, vp, vp, vp, vp, vp, vp]
    L.e2e_ctc_engine_beam_nbest_host.restype = ctypes.c_int
    L.e2e_ctc_score_workspace_bytes.argtypes = [dp, i32]
    L.e2e_ctc_score_workspace_bytes.restype = sz
    L.e2e_ctc_score_device.argtypes = [dp, i32, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_score_device.restype = ctypes.c_int
    L.e2e_ctc_score_backward_workspace_bytes.argtypes = [dp, i32]
    L.e2e_ctc_score_backward_workspace_bytes.restype = sz
    L.e2e_ctc_score_backward_device.argtypes = [dp, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_score_backward_device.restype = ctypes.c_int
    L.e2e_ctc_align_nbest_workspace_bytes.argtypes = [dp, i32]
    L.e2e_ctc_align_nbest_workspace_bytes.restype = sz
    L.e2e_ctc_align_nbest_device.argtypes = [dp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_align_nbest_device.restype = ctypes.c_int
    ep = ctypes.POINTER(EditDesc)
    L.e2e_ctc_edit_distance_workspace_bytes.argtypes = [ep]
    L.e2e_ctc_edit_distance_workspace_bytes.restype = sz
    L.e2e_ctc_edit_distance_device.argtypes = [ep, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]
    L.e2e_ctc_edit_distance_device.restype = ctypes.c_int
    L.e2e_ctc_host_alloc.argtypes = [sz, ctypes.POINTER(vp)]
    L.e2e_ctc_host_alloc.restype = ctypes.c_int
    L.e2e_ctc_host_free.argtypes = [vp]
    L.e2e_ctc_host_free.restype = ctypes.c_int
    L.e2e_ctc_graph_launch.argtypes = [vp, vp]
    L.e2e_ctc_graph_destroy.argtypes = [vp]
    L.e2e_ctc_graph_destroy.restype = None
    for name in ("e2e_ctc_graph_create", "e2e_ctc_graph_launch"):
        getattr(L, name).restype = ctypes.c_int
    for name in ("e2e_ctc_comm_unique_id", "e2e_ctc_comm_create", "e2e_ctc_comm_allreduce_sum"):
        getattr(L, name).restype = ctypes.c_int
    for name in ("e2e_ctc_get_limits", "e2e_ctc_loss_forward_device", "e2e_ctc_loss_backward_device",
                 "e2e_ctc_loss_fwd_bwd_device", "e2e_ctc_loss_step_device", "e2e_ctc_scale_rows_device", "e2e_ctc_loss_reduce_device", "e2e_ctc_loss_check_device",
                 "e2e_ctc_greedy_decode_device", "e2e_ctc_engine_create", "e2e_ctc_engine_loss_host",
                 "e2e_ctc_engine_greedy_host", "e2e_ctc_engine_last_traffic", "e2e_ctc_profile_enable",
                 "e2e_ctc_profile_read"):
        getattr(L, name).restype = ctypes.c_int
    _lib = L
    return L


def check(rc):
    if rc != E2E_OK:
        raise E2EError(rc, load().e2e_last_error_string().decode("utf-8", "replace"))


def limits():
    lim = Limits()
    check(load().e2e_ctc_get_limits(ctypes.byref(lim)))
    return lim


def profile_enable(on=True):
    check(load().e2e_ctc_profile_enable(1 if on else 0))


def profile_read():
    """{kernel kind: (device ms summed, launches)} since the last read (synchronises)."""
    n = len(KERNEL_KINDS)
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_uint64 * n)()
    check(load().e2e_ctc_profile_read(ms, cnt, n))
    return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(KERNEL_KINDS)}


_forced_kernel = -1


def force_kernel(kind=-1):
    """Testing hook: force a lattice kernel where the shape allows it (-1 automatic, 0 general, 1 wave,
    2 one-warp-per-sweep).  Process-wide; the parity tests use it to run every kernel on every shape."""
    global _forced_kernel
    L = load()
    L.e2e_ctc_debug_force_kernel.argtypes = [ctypes.c_int32]
    L.e2e_ctc_debug_force_kernel.restype = ctypes.c_int
    check(L.e2e_ctc_debug_force_kernel(int(kind)))
    _forced_kernel = int(kind)


def forced_kernel():
    return _forced_kernel


def launch_count():
    return int(load().e2e_ctc_launch_count())

"""ctypes binding of ``libmmf_b200.so`` (the C ABI in ``include/mmf_b200.h``).

No torch types cross this boundary: tensors are passed as raw device pointers plus sizes, the
stream as a ``cudaStream_t`` integer.  There is NO fallback: if the shared library is missing or
the device is not sm_100, every entry point raises.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmmf_b200.so")

MAX_SD, MAX_CD, MAX_HEADS, UNITS = 4, 16, 4, 64
ABI_VERSION = 2

RESAMPLE_NONE = 0
RESAMPLE_MULTINOMIAL_STRICT = 1
RESAMPLE_MULTINOMIAL_FAST = 2
RESAMPLE_SYSTEMATIC_STRICT = 3
RESAMPLE_SYSTEMATIC_FAST = 4
ESTIMATE_WEIGHTED_AVERAGE = 0
ESTIMATE_ARGMAX = 1
PREC_FP32, PREC_BF16X3, PREC_BF16 = 0, 1, 2


class Chain(C.Structure):
    _fields_ = [
        ("in_dim", C.c_int32),
        ("n_pre_res", C.c_int32),
        ("mid_relu", C.c_int32),
        ("n_post_res", C.c_int32),
        ("out_dim", C.c_int32),
        ("reserved", C.c_int32),
        ("w", C.c_void_p),
        ("w_mma", C.c_void_p),
        ("w_bwd", C.c_void_p),
    ]


class TrajRows(C.Structure):
    _fields_ = [("in_dim", C.c_int32), ("has_encoder", C.c_int32), ("w", C.c_void_p)]


class PFModel(C.Structure):
    _fields_ = [
        ("state_dim", C.c_int32),
        ("control_dim", C.c_int32),
        ("num_heads", C.c_int32),
        ("reserved", C.c_int32),
        ("dynamics", Chain),
        ("dynamics_rows", TrajRows),
        ("heads", Chain * MAX_HEADS),
        ("head_rows", TrajRows * MAX_HEADS),
        ("q_tril", C.c_float * (MAX_SD * MAX_SD)),
    ]


class EKFModel(C.Structure):
    _fields_ = [
        ("state_dim", C.c_int32),
        ("control_dim", C.c_int32),
        ("dynamics", Chain),
        ("dynamics_rows", TrajRows),
        ("q_tril", C.c_float * (MAX_SD * MAX_SD)),
    ]


class MlpOp(C.Structure):
    _fields_ = [
        ("in_dim", C.c_int32), ("out_dim", C.c_int32), ("act", C.c_int32),
        ("src", C.c_int32), ("dst", C.c_int32), ("res", C.c_int32),
        ("w_off", C.c_int64),
    ]


MLP_MAX_OPS, MLP_MAX_IO = 24, 4
MLP_NONE, MLP_RELU, MLP_SIGMOID = 0, 1, 2


class MMFError(RuntimeError):
    pass


_lock = threading.Lock()
_lib = None

_i32, _f32, _u32, _vp, _sz = C.c_int32, C.c_float, C.c_uint32, C.c_void_p, C.c_size_t

# name -> (restype, argtypes); also the list of symbols tests check against the header
PROTOTYPES = {
    "mmf_last_error": (C.c_char_p, []),
    "mmf_abi_version": (C.c_int, []),
    "mmf_device_check": (C.c_int, []),
    "mmf_pf_init": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_pf_traj_rows": (C.c_int, [C.POINTER(PFModel), _i32, _vp, C.POINTER(_vp), _vp, _vp]),
    "mmf_pf_predict_measure": (
        C.c_int,
        [C.POINTER(PFModel), _i32, _i32, _vp, _vp, _vp, _vp, _vp, _u32, _i32, _vp, _vp, _vp, _vp],
    ),
    "mmf_pf_forward_loop": (
        C.c_int,
        [C.POINTER(PFModel), _i32, _i32, _i32, _vp, _vp, _vp, C.POINTER(_vp), _vp, _u32, _i32, _vp, _i32, _i32, _vp, _vp,
         _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_pf_resample_workspace_bytes": (_sz, [_i32, _i32]),
    "mmf_pf_normalize_resample": (
        C.c_int,
        [_i32, _i32, _i32, _vp, _vp, _i32, _i32, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_fuse_loglik": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "mmf_resample": (C.c_int, [_i32, _i32, _i32, _vp, _i32, _vp, _vp, _vp, _vp]),
    "mmf_ekf_loop_fwd": (C.c_int, [C.POINTER(EKFModel), _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_ekf_loop_train_fwd": (
        C.c_int, [C.POINTER(EKFModel), _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_ekf_loop_bwd": (
        C.c_int,
        [C.POINTER(EKFModel), _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_dynamics_jacobian": (C.c_int, [C.POINTER(EKFModel), _i32, _vp, _vp, _vp, _vp, _vp]),
    "mmf_kf_fuse_crossmodal": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_pf_forward_loop_persistent": (C.c_int, [_i32, _i32]),
    "mmf_kf_fuse_measurements": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_kf_fuse_unimodal": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "mmf_chain_bwd_bytes": (_sz, [C.POINTER(Chain)]),
    "mmf_pack_chain_bwd": (C.c_int, [C.POINTER(Chain), _vp, _vp]),
    "mmf_pf_heads_forward_train": (
        C.c_int, [C.POINTER(PFModel), _i32, _i32, _vp, _vp, _vp, _vp, _u32, _i32, _vp, _vp, _vp, _vp]),
    "mmf_pf_heads_backward": (C.c_int, [C.POINTER(PFModel), _i32, _i32, _vp, _vp, _u32, _vp, _vp]),
    "mmf_pf_heads_weight_grads_workspace_bytes": (_sz, [_i32, _i32, C.c_int64]),
    "mmf_pf_heads_weight_grads": (C.c_int, [_i32, _i32, C.c_int64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_enc_map_bytes": (_sz, [_i32]),
    "mmf_enc_trunk_scratch_bytes": (_sz, []),
    "mmf_enc_trunk_weight_bytes": (_sz, []),
    "mmf_enc_trunk": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "mmf_enc_stem": (C.c_int, [_i32, _vp, _vp, _vp, _vp]),
    "mmf_enc_conv3x3": (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "mmf_pf_reweight_train_fwd": (C.c_int, [_i32, _i32, _i32, _i32, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_pf_reweight_train_bwd": (C.c_int, [_i32, _i32, _i32, _i32, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mmf_row_mlp": (
        C.c_int,
        [C.c_int64, C.POINTER(MlpOp), _i32, _vp, C.POINTER(_vp), C.POINTER(_i32), C.POINTER(_i32), _i32, C.POINTER(_vp),
         C.POINTER(_i32), C.POINTER(_i32), _i32, _i32, _vp],
    ),
    "mmf_chain_mma_bytes": (_sz, [C.POINTER(Chain)]),
    "mmf_pack_chain_mma": (C.c_int, [C.POINTER(Chain), _vp, _vp]),
}


def load():
    """Load the shared library (once).  Raises MMFError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise MMFError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C multimodalfilter_b200/csrc`).  There is no CPU or eager fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.mmf_abi_version() != ABI_VERSION:
            raise MMFError(f"ABI mismatch: library reports version {lib.mmf_abi_version()}, binding expects {ABI_VERSION}")
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().mmf_last_error()
        raise MMFError(f"libmmf_b200 error {rc}: {msg.decode() if msg else '?'}")


_tls = threading.local()


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL).  The tensor's device is noted so that ``call`` can
    check that every buffer of one launch lives on the device the kernels are launched on."""
    if t is None:
        return None
    if not t.is_cuda:
        raise MMFError("libmmf_b200 only takes CUDA tensors: there is no CPU path")
    if not t.is_contiguous():
        raise MMFError("libmmf_b200 needs C-contiguous tensors")
    seen = getattr(_tls, "devices", None)
    if seen is None:
        seen = _tls.devices = []
    seen.append(t.device)
    return C.c_void_p(t.data_ptr())


class Stream(C.c_void_p):
    """``cudaStream_t`` argument that remembers which device it belongs to."""

    device = None


def stream_of(t):
    import torch

    s = Stream(torch.cuda.current_stream(t.device).cuda_stream)
    s.device = t.device
    return s


def call(fn, *args):
    """Run one C entry point with the CUDA device of its stream argument current.  The launchers configure and launch
    on the process-current device (cudaGetDevice), so a filter living on cuda:1 while cuda:0 is current must switch
    devices around the call; buffers on any other device than the stream's are refused."""
    import torch

    seen, _tls.devices = getattr(_tls, "devices", None) or [], []
    stream = next((a for a in reversed(args) if isinstance(a, Stream)), None)
    if stream is None or stream.device is None:
        return fn(*args)
    for d in seen:
        if d != stream.device:
            raise MMFError(f"all buffers of one libmmf_b200 call must live on one device: got {d} and {stream.device}")
    if torch.cuda.current_device() == stream.device.index:
        return fn(*args)
    with torch.cuda.device(stream.device):
        return fn(*args)

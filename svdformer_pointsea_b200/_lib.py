"""ctypes binding of the C ABI in include/pointsea_b200.h (libpointsea_b200.so).

This is the whole Python<->native boundary: raw device pointers, sizes, the device ordinal
and the current CUDA stream.  There is NO CPU fallback: if the shared library is missing or a
tensor is not on a CUDA device the call raises.
"""
import ctypes
import os
import os.path as osp

import torch

_HERE = osp.dirname(osp.abspath(__file__))
# POINTSEA_B200_LIB points at an alternative build of the same C ABI (A/B measurements)
LIB_PATH = os.environ.get("POINTSEA_B200_LIB", osp.join(_HERE, "lib", "libpointsea_b200.so"))

_c_int = ctypes.c_int
_c_void_p = ctypes.c_void_p
_c_float = ctypes.c_float

# name -> argtypes (restype is int unless stated) — mirrors include/pointsea_b200.h 1:1
_P = _c_void_p
_SIGNATURES = {
    "ps_chamfer_fwd": [_P, _P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_host": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_host_full": [_P] * 12 + [_c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_host_submit": [_P] * 12 + [_c_int, _c_int, _c_int, _c_int, _c_int, _P, ctypes.POINTER(ctypes.c_longlong)],
    "ps_chamfer_host_wait": [ctypes.c_longlong, _c_int, _P, _c_int, _c_int],
    "ps_chamfer_host_step": [_P, _P, _P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_fwd_sums": [_P, _P, _P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_loss_fwd": [_P] * 8 + [_c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_loss_bwd": [_P] * 9 + [_c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_step": [_P] * 13 + [_c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_step_prepare": [_P] * 13 + [_c_int, _c_int, _c_int, _c_int],
    "ps_chamfer_step_stats": [_c_int, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong)],
    "ps_chamfer_host_stats": [_c_int, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong)],
    "ps_chamfer_host_step_dist": [_P, _P, _P, _P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_comm_create": [_c_int, _c_int, _c_int, ctypes.POINTER(_c_void_p)],
    "ps_comm_export": [_P, _P],
    "ps_comm_connect": [_P, _P],
    "ps_comm_connect_local": [ctypes.POINTER(_c_void_p), _c_int],
    "ps_comm_allreduce": [_P, _P, _P, _c_int, _P],
    "ps_comm_status": [_P, ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(ctypes.c_longlong), ctypes.POINTER(_c_int)],
    "ps_comm_destroy": [_P],
    "ps_chamfer_sums": [_P, _P, _P, ctypes.c_longlong, ctypes.c_longlong, _c_int, _P],
    "ps_fps": [_P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_fps_sample": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_fps_sample_ex": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_fps_sample_ragged": [_P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_crop_split": [_P] * 5 + [_c_int] * 6 + [_P],
    "ps_gather_fwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_gather_bwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_group_fwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_group_bwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_ball_query": [_P, _P, _P, _c_int, _c_int, _c_int, _c_float, _c_int, _c_int, _P],
    "ps_knn": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_knn_point": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_knn_group_xyz": [_P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_knn_feat": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_edge_features_fwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_edge_features_bwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_index_points_fwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_index_points_bwd": [_P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_chamfer_metrics": [_P, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_float, _c_float, _c_float, _c_float,
                           _c_float, _c_int, _P],
    "ps_chamfer_metrics_bwd": [_P, _P, _P, _P, _P, ctypes.c_uint, _P, _P, _P, _P, _c_int, _c_int, _c_int, _c_float,
                               _c_float, _c_float, _c_float, _c_int, _P],
    "ps_scatter_max": [_P, _P, _P, _P, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong,
                       _c_int, _c_int, _P],
    "ps_three_nn": [_P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_three_interpolate_fwd": [_P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_three_interpolate_bwd": [_P, _P, _P, _P, _c_int, _c_int, _c_int, _c_int, _c_int, _P],
    "ps_device_info": [_c_int, ctypes.POINTER(_c_int), ctypes.POINTER(_c_int), ctypes.POINTER(_c_int)],
    "ps_measure_fp32_peak": [_c_int, _c_int, ctypes.POINTER(ctypes.c_double)],
}
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + ["ps_version", "ps_last_error", "ps_launch_count", "ps_comm_handle_bytes"])

_lib = None


class PointSeaError(RuntimeError):
    """Raised for every non-zero return code of the native library (`code`: the PS_ERR_* value, None for errors
    raised by the Python layer itself)."""
    code = None


PS_ERR_UNSUPPORTED = -3


def load():
    """Load libpointsea_b200.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not osp.exists(LIB_PATH):
        raise PointSeaError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
            "(svdformer_pointsea_b200/csrc/build.sh). There is no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _c_int
    lib.ps_version.argtypes = []
    lib.ps_version.restype = _c_int
    lib.ps_last_error.argtypes = []
    lib.ps_last_error.restype = ctypes.c_char_p
    lib.ps_comm_handle_bytes.argtypes = []
    lib.ps_comm_handle_bytes.restype = _c_int
    lib.ps_launch_count.argtypes = [_c_int]
    lib.ps_launch_count.restype = ctypes.c_longlong
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().ps_last_error().decode("utf-8", "replace")
        err = PointSeaError(f"{what} failed (code {rc}): {msg}")
        err.code = rc
        raise err


_checked_devices = set()


def _check_device(index):
    """Fail loudly off sm_100: the kernels are built for sm_100a only."""
    if index in _checked_devices:
        return
    sm, major, minor = _c_int(), _c_int(), _c_int()
    check(load().ps_device_info(index, ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)), "ps_device_info")
    if major.value != 10:
        raise PointSeaError(
            f"cuda:{index} has compute capability {major.value}.{minor.value}; this library is sm_100a (B200) only")
    _checked_devices.add(index)


def require(t, name, dtype, ndim):
    """The reference's CHECK_CONTIGUOUS / CHECK_IS_FLOAT / CHECK_IS_INT / CHECK_CUDA
    (pointnet2_ops/_ext-src/include/utils.h:5-25) as RuntimeErrors."""
    if not isinstance(t, torch.Tensor):
        raise PointSeaError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise PointSeaError(f"{name} must be a CUDA tensor (CPU not supported)")
    if t.dtype != dtype:
        raise PointSeaError(f"{name} must be a {'float' if dtype == torch.float32 else 'int'} tensor, got {t.dtype}")
    if t.dim() != ndim:
        raise PointSeaError(f"{name} must have {ndim} dimensions, got {tuple(t.shape)}")
    if not t.is_contiguous():
        raise PointSeaError(f"{name} must be a contiguous tensor")
    return t


def same_device(*ts):
    dev = ts[0].device
    for t in ts[1:]:
        if t.device != dev:
            raise PointSeaError(f"tensors are on different devices: {dev} vs {t.device}")
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    _check_device(index)
    return index


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(index):
    """cudaStream_t of torch's current stream on `index` as an int (ctypes converts it to void*).
    The raw getter avoids building a torch.cuda.Stream object per call (host overhead matters for
    the small shapes inside the models: a 256x256 Chamfer is ~5 us of GPU time)."""
    if _raw_stream is not None:
        return _raw_stream(index)
    return torch.cuda.current_stream(index).cuda_stream


def ptr(t):
    # 0 (empty tensor) must become NULL, not c_void_p(0) quirks: ctypes maps int 0 -> NULL for c_void_p
    return t.data_ptr() or None


def launch_count(reset=False):
    return int(load().ps_launch_count(1 if reset else 0))


def graph_stats(index=0, which="step"):
    """(exact replays, in-place retargets, instantiations) of the one-launch entry points' graph cache."""
    h, u, i = ctypes.c_longlong(), ctypes.c_longlong(), ctypes.c_longlong()
    fn = load().ps_chamfer_step_stats if which == "step" else load().ps_chamfer_host_stats
    check(fn(index, ctypes.byref(h), ctypes.byref(u), ctypes.byref(i)), "graph stats")
    return {"hits": h.value, "updates": u.value, "instantiations": i.value}


def measure_fp32_peak(index=0, reps=5):
    out = ctypes.c_double()
    check(load().ps_measure_fp32_peak(index, reps, ctypes.byref(out)), "ps_measure_fp32_peak")
    return out.value

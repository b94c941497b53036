"""ctypes binding of ``include/simple_pose_b200.h`` (the only door into the CUDA kernels).

The library is built in-tree by ``simple_pose_b200/build.py`` (``__graft_entry__.build()``).
There is no CPU or PyTorch fallback: if the shared library is missing, or a tensor is not on
a CUDA device, the call raises.
"""
import ctypes
import os
import threading

import torch

from . import build as _build

c_f32p = ctypes.c_void_p
c_void = ctypes.c_void_p
c_int = ctypes.c_int
c_dbl = ctypes.c_double
c_flt = ctypes.c_float
c_size = ctypes.c_size_t
c_ll = ctypes.c_longlong

ABI_VERSION = 2
SP_DECODE_GAUSS_TAYLOR, SP_DECODE_ARGMAX, SP_DECODE_BASIC, SP_DECODE_DARK_ORIGINAL = 0, 1, 2, 3
SP_MSE_SKIP_MASKED = 1
SP_DTYPE_F32, SP_DTYPE_F16, SP_DTYPE_BF16 = 0, 1, 2
SP_BOX_XYXY, SP_BOX_XYWH = 0, 1

# name -> (restype, argtypes); mirrors include/simple_pose_b200.h one to one
SIGNATURES = {
    "sp_abi_version": (c_int, []),
    "sp_error_string": (ctypes.c_char_p, [c_int]),
    "sp_device_info": (c_int, [ctypes.POINTER(c_int)] * 3),
    "sp_reload_tuning": (c_int, []),
    "sp_encode_f32": (c_int, [c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_dbl, c_void]),
    "sp_encode_basic_f32": (c_int, [c_void, c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_dbl, c_int, c_int, c_void]),
    "sp_mse_workspace_bytes": (c_size, []),
    "sp_mse_fwd_bwd_f32": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_size,
                                   c_int, c_int, c_int, c_flt, c_int, c_void]),
    "sp_mse_fwd_bwd": (c_int, [c_void, c_int, c_void, c_void, c_void, c_void, c_void, c_size,
                               c_int, c_int, c_int, c_flt, c_void, c_int, c_void]),
    "sp_mse_acc_workspace_bytes": (c_size, [c_int, c_int]),
    "sp_mse_acc_fwd_bwd": (c_int, [c_void, c_int] + [c_void] * 7 + [c_void, c_size, c_int, c_int, c_int, c_int, c_flt, c_void,
                                                                     c_flt, c_flt, c_int, c_void]),
    "sp_encode_mse_fwd_bwd_f32": (c_int, [c_void] * 9 + [c_size, c_int, c_int, c_int, c_int, c_dbl, c_flt, c_void]),
    "sp_encode_mse_fwd_bwd": (c_int, [c_void, c_void, c_int] + [c_void] * 7 + [c_size, c_int, c_int, c_int, c_int, c_dbl, c_flt, c_void, c_void]),
    "sp_step_f32": (c_int, [c_void] * 13 + [c_size, c_int, c_int, c_int, c_int, c_dbl, c_int, c_flt, c_void]),
    "sp_val_step_workspace_bytes": (c_size, [c_int, c_int]),
    "sp_val_step_f32": (c_int, [c_void] * 4 + [c_int] + [c_void] * 9 + [c_size, c_int, c_int, c_int, c_int, c_dbl, c_int,
                                                                   c_flt, c_flt, c_void]),
    "sp_heatmap_acc_f32": (c_int, [c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_flt, c_flt, c_void]),
    "sp_scale_inplace_f32": (c_int, [c_void, c_ll, c_void, c_void]),
    "sp_decode_f32": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_void, c_void,
                              c_int, c_int, c_int, c_int, c_int, c_int, c_void]),
    "sp_decode_workspace_bytes": (c_size, []),
    "sp_decode_ws_f32": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_void, c_void,
                                 c_int, c_int, c_int, c_int, c_int, c_int, c_void, c_size, c_void]),
    "sp_decode_rows_f32": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_int, c_void, c_void,
                                   c_int, c_int, c_int, c_int, c_int, c_int, c_void, c_size, c_void]),
    "sp_eval_rows_nms_f32": (c_int, [c_void, c_int, c_void, c_void, c_void, c_void, c_void, c_void,
                                     c_int, c_int, c_int, c_int, c_dbl, c_dbl, c_void]),
    "sp_eval_rows_nms_fanout_f32": (c_int, [c_void, c_int, c_void, c_void, c_void, c_void, c_void, c_void,
                                            c_int, c_int, c_int, c_int, c_dbl, c_dbl, c_void, c_void, c_int, c_int, c_ll, c_void]),
    "sp_person_rows_f32": (c_int, [c_void, c_void, c_void, c_int, c_int, c_void]),
    "sp_oks_iou_f64": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_int, c_int, c_int, c_dbl, c_void]),
    "sp_oks_nms_f64": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_void,
                               c_int, c_int, c_int, c_int, c_dbl, c_int, c_dbl, c_void]),
    "sp_rescore_f64": (c_int, [c_void, c_void, c_void, c_int, c_int, c_dbl, c_void]),
    "sp_pack_kps_f64": (c_int, [c_void, c_void, c_void, c_int, c_int, c_void]),
    "sp_pack_rows_f32": (c_int, [c_void, c_void, c_void, c_void, c_void, c_int, c_int, c_void]),
    "sp_coco_eval_workspace_bytes": (c_size, [c_int, c_int, c_int]),
    "sp_coco_eval_kps_f32": (c_int, [c_void, c_int, c_void, c_void, c_void, c_int,
                                     c_void, c_void, c_void, c_void, c_void, c_int, c_int,
                                     c_void, c_void, c_void, c_int, c_int, c_int, c_int, c_int,
                                     c_void, c_void, c_void, c_void, c_void, c_void, c_void, c_size, c_void]),
    "sp_box_affine_f64": (c_int, [c_void, c_int, c_void, c_void, c_void, c_void, c_void, c_void, c_int, c_dbl, c_int, c_int, c_flt, c_void]),
    "sp_center_scale_affine_f64": (c_int, [c_void, c_void, c_void, c_void, c_void, c_int, c_int, c_int, c_void]),
    "sp_center_scale_rot_affine_f64": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_int, c_int, c_int, c_void]),
    "sp_train_geometry_f32": (c_int, [c_void] * 14 + [c_int, c_int, c_int, c_int, c_int, c_int, c_flt, c_void]),
    "sp_transform_joints_f32": (c_int, [c_void, c_void, c_void, c_void, c_void, c_void, c_int, c_int, c_void]),
}

_lock = threading.Lock()
_lib = None


class ExtensionMissing(RuntimeError):
    pass


def lib():
    """The loaded shared library (loads it on first use)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = os.environ.get("SIMPLE_POSE_B200_LIB", _build.lib_path())
        if not os.path.isfile(path):
            raise ExtensionMissing(
                "simple_pose_b200: CUDA extension not built (%s missing). Run "
                "`python -m simple_pose_b200.build` (needs nvcc). There is no CPU fallback." % path)
        handle = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if handle.sp_abi_version() != ABI_VERSION:
            raise ExtensionMissing("simple_pose_b200: ABI version mismatch, rebuild the library")
        _lib = handle
        return _lib


def reload_tuning():
    """Re-read the SP_* tuning variables from ``os.environ`` (the library reads them once per process)."""
    check(lib().sp_reload_tuning())


def check(code):
    if code != 0:
        msg = lib().sp_error_string(int(code))
        raise RuntimeError("%s (code %d)" % (msg.decode() if msg else "simple_pose_b200 error", code))


def stream_ptr(device):
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors):
    """All tensors must live on one CUDA device; returns it."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError("simple_pose_b200: expected CUDA tensors (there is no CPU path); got %s"
                               % (t.device if isinstance(t, torch.Tensor) else type(t)))
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("simple_pose_b200: tensors on different devices: %s vs %s" % (dev, t.device))
    return dev


def dense(t, dtype):
    """Contiguous tensor of ``dtype`` (no copy when it already is)."""
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


def ptr(t):
    return None if t is None else t.data_ptr()


def refuse_loader_worker(what):
    """The per-sample drop-ins (``RefineSimpleTransform.get_heat_map`` ...) keep the reference's NumPy signature
    but run on the GPU. The reference calls them from ``MSCOCO.__getitem__`` inside forked DataLoader workers
    (``datasets/coco.py:58-60``), where CUDA cannot be initialised; say so instead of dying in a CUDA re-init."""
    in_worker = False
    try:
        from torch.utils.data import get_worker_info
        in_worker = get_worker_info() is not None
    except Exception:
        pass
    if in_worker or torch.cuda._is_in_bad_fork():
        raise RuntimeError(
            "simple_pose_b200: %s was called inside a DataLoader worker / forked process. The kernels need a CUDA "
            "context, which a forked worker cannot create. Ship the joints from the loader (204 B per person) and "
            "encode the whole batch on the training device with commons.transforms.encode_heat_maps(joints) or "
            "processors.loss.EncodeJointsMSELoss -- see INTEGRATION.md section 3." % what)


def default_device():
    if not torch.cuda.is_available():
        raise RuntimeError("simple_pose_b200: no CUDA device available (there is no CPU path)")
    return torch.device("cuda", torch.cuda.current_device())


def to_device(x, dtype, device=None):
    """Host array / CPU tensor / CUDA tensor -> dense CUDA tensor of ``dtype``."""
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(x)
    if not x.is_cuda:
        device = device or default_device()
        x = x.to(device=device, dtype=dtype, non_blocking=True)
    return dense(x, dtype)


_scratch = {}


def scratch(device, stream_id, nbytes, tag):
    """Zero-initialised device scratch per (tag, device, stream) for the kernels that keep a work
    counter / reduction workspace there; the kernels restore the zero state, calls on one stream
    are ordered, so one buffer per stream is enough. Callers that may run concurrently on ONE stream id
    (two host threads sharing a stream) must serialise themselves -- the C ABI documents the same rule."""
    key = (tag, device.index, stream_id)
    buf = _scratch.get(key)
    if buf is None or buf.numel() * 8 < nbytes:
        buf = torch.zeros((int(nbytes) + 7) // 8, dtype=torch.int64, device=device)
        _scratch[key] = buf
    return buf


def drop_scratch(device, stream_id=None):
    """Forget the cached workspaces of a device (one stream or all). Called when a launch that uses one
    fails: the "kernel restores the zero state" invariant assumes the kernel ran, so the next call must
    start from a freshly zeroed buffer instead of stale tickets / work counters."""
    for key in [k for k in _scratch if k[1] == device.index and (stream_id is None or k[2] == stream_id)]:
        del _scratch[key]


def check_ws(code, device, stream_id, owner=None):
    """``check`` for calls that were handed a workspace: on failure the cached per-stream scratch is dropped and an
    ``owner`` that keeps its own (``HeatmapHotPath.ws`` / ``.dws`` / ``.vws``) gets it re-zeroed."""
    if code != 0:
        drop_scratch(device, stream_id)
        if owner is not None:
            try:
                owner.ws.zero_()
                owner.dws.zero_()
                if getattr(owner, "vws", None) is not None:
                    owner.vws.zero_()
            except Exception:
                pass
    check(code)


def device_info(device=None):
    device = device or default_device()
    sm, major, minor = c_int(0), c_int(0), c_int(0)
    with torch.cuda.device(device):
        check(lib().sp_device_info(ctypes.byref(sm), ctypes.byref(major), ctypes.byref(minor)))
    return {"sm_count": sm.value, "cc": (major.value, minor.value)}

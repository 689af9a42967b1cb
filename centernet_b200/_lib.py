"""Loads the in-tree pybind11 binding of the C ABI.  No fallback: a missing or stale
extension is an ImportError that says how to build it."""
import torch

import threading

try:
    from . import _C
except ImportError as e:  # pragma: no cover - exercised only on a broken install
    raise ImportError(
        "centernet_b200: the CUDA extension is not built (%s). Run `python centernet_b200/build.py` "
        "(needs nvcc, targets sm_100a). There is no CPU fallback." % (e,)) from e


_tls = threading.local()


class _DeviceGuarded(object):
    """The C ABI launches on the CURRENT device (include/centernet_b200.h).  The reference's ATen ops follow
    their tensors instead, so every binding call is wrapped: `stream_ptr(t)` -- evaluated while the arguments
    are built -- notes t's device, and the call runs under `torch.cuda.device(that device)` when it is not
    the current one (a tensor on cuda:1 while cuda:0 is current would otherwise launch with a foreign
    stream)."""

    def __init__(self, mod):
        self._mod = mod

    def __getattr__(self, name):
        fn = getattr(self._mod, name)
        if not callable(fn):
            return fn

        def call(*args):
            dev = getattr(_tls, "dev", None)
            _tls.dev = None
            if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
                with torch.cuda.device(dev):
                    return fn(*args)
            return fn(*args)

        call.__name__ = name
        setattr(self, name, call)
        return call


C = _DeviceGuarded(_C)


def same_device(*tensors):
    """All CUDA tensors of one call must live on one device (ATen raises the same way)."""
    dev = None
    for t in tensors:
        if t is None or not t.is_cuda:
            continue
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("centernet_b200: tensors of one call are on different devices (%s vs %s)"
                               % (dev, t.device))
    return dev


def version():
    v = C.version()
    return "%d.%d.%d" % (v // 10000, (v // 100) % 100, v % 100)


def stream_ptr(t):
    """Raw cudaStream_t of the current stream on t's device (decode must be stream-ordered
    because callers immediately do dets.detach().cpu(), detectors/ctdet.py:48)."""
    _tls.dev = t.device
    return torch.cuda.current_stream(t.device).cuda_stream


def require_cuda(*tensors, what="centernet_b200"):
    same_device(*tensors)
    for t in tensors:
        if t is not None and not t.is_cuda:
            # same contract as DCNv2Function.forward (dcn_v2_func.py:23-24)
            raise NotImplementedError("%s: only implemented for CUDA tensors (no CPU fallback)" % what)


def f32c(t):
    """fp32 + contiguous view of t (no copy when it already is)."""
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def ptr(t):
    return 0 if t is None else t.data_ptr()


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)

"""ctypes binding of libssv_b200.so (the C ABI declared in include/ssv_b200.h).

No CPU fallback and no alternative backend: if the shared library is missing, or a call
returns non-zero, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os
import re
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# SSVB_LIB selects an A/B tuning build (e.g. libssv_b200_x.so) for experiments; default is the product build
LIB_PATH = os.path.join(_HERE, os.environ.get("SSVB_LIB", "libssv_b200.so"))
# the header the prototypes are bound from: the repository's include/ when the package runs in-tree (always current),
# else the copy `make` places next to the library (installed / relocated package)
_REPO_HEADER = os.path.normpath(os.path.join(_HERE, "..", "..", "include", "ssv_b200.h"))
HEADER_PATH = _REPO_HEADER if os.path.exists(_REPO_HEADER) else os.path.join(_HERE, "ssv_b200.h")

_CTYPE = {
    "int": c_int, "float": c_float, "int64_t": c_int64, "size_t": c_size_t,
    "const char*": c_char_p, "void": None, "long long": ctypes.c_longlong, "double": ctypes.c_double,
}


def _ctype_of(decl: str):
    decl = decl.strip()
    if decl.endswith("*") and decl != "const char*":
        return c_void_p
    return _CTYPE[decl]


def parse_header(path: str = HEADER_PATH):
    """Return {name: (restype, [argtypes])} for every `ssvb_*` prototype in the public header, so the
    binding can never drift from include/ssv_b200.h."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"([A-Za-z_][A-Za-z0-9_ ]*?\*?)\s*(ssvb_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        argtypes = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                # drop the parameter name
                mm = re.match(r"(.*?[\*\s])([A-Za-z_][A-Za-z0-9_]*)$", a)
                typ = mm.group(1).strip() if mm else a
                typ = typ.replace("const ", "") if not typ.startswith("const char") else typ
                typ = typ.replace(" *", "*").strip()
                argtypes.append(_ctype_of(typ))
        protos[name] = (_ctype_of(ret.replace("const char *", "const char*")), argtypes)
    return protos


c_void_p = ctypes.c_void_p  # re-exported for callers that pass raw device addresses

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"ssv_b200: {LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C self-supervised-vision_b200`). There is no CPU / PyTorch fallback.")
        l = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in parse_header().items():
            fn = getattr(l, name)  # AttributeError here == header/library mismatch: fail loudly
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = l
    return _lib


def strerror(rc: int) -> str:
    return lib().ssvb_strerror(rc).decode()


_LIMITS = ("supported envelope (INTEGRATION.md §4): fp32 rows, row stride and feature dim multiples of 4, 16-byte aligned "
           "base pointers; d <= 256 for the similarity losses (SimclrLoss / MocoLoss / RelicLoss / PirlLoss; d <= 128 is the "
           "tuned path and the only one of the peer-memory transport); "
           "K <= 65536 for DinoLoss")


def check(rc: int, what: str):
    if rc != 0:
        msg = f"{what} failed (rc={rc}): {strerror(rc)}"
        if rc < 0:   # argument / shape / alignment / unsupported: name the envelope instead of a bare code
            msg += f" -- {_LIMITS}"
        raise RuntimeError(msg)


def ptr(t):
    if t is None:
        return None
    return c_void_p(t.data_ptr())


try:   # raw current-stream handle without building a torch.cuda.Stream object (~0.3 us instead of ~2.4 us per call)
    _raw_stream = torch._C._cuda_getCurrentRawStream
except AttributeError:  # pragma: no cover  (older / newer torch without the private accessor)
    _raw_stream = None


def raw_stream(device=None) -> int:
    """Integer handle (cudaStream_t) of the current stream of `device` (a torch.device or None = current device)."""
    if _raw_stream is not None:
        idx = device.index if (device is not None and device.index is not None) else torch.cuda.current_device()
        return _raw_stream(idx)
    return torch.cuda.current_stream(device).cuda_stream


def stream_ptr(device=None):
    return c_void_p(raw_stream(device))


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("ssv_b200 runs on a B200 (sm_100a) only: got a CPU tensor; there is no CPU fallback")


def as_f32_rows(t):
    """fp32, last-dim contiguous, 16-byte aligned rows (what the C ABI requires)."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.stride(-1) != 1 or (t.stride(0) % 4) or (t.data_ptr() % 16):
        t = t.contiguous()
    return t


def byte_buffer(nbytes: int, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


# ---- host-overhead helpers: the small losses are launch-bound, every microsecond of Python per call shows -------
_WS = {}


def workspace(tag: str, nbytes: int, device):
    """Scratch buffer reused across calls of one op on one (device, stream): work is stream-ordered, so the next call
    on the same stream may overwrite it.  (`saved` blobs that must survive until backward are NOT taken from here.)"""
    key = (tag, device.index, raw_stream(device))
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


_SIZES = {}


def cached_size(fn_name: str, *args) -> int:
    """Memoised `*_saved_bytes` / `*_workspace_bytes` queries (pure functions of the shape)."""
    # (sizes follow the chunk plan, i.e. the SM count: one process drives identical GPUs of one box, and the library
    # itself caches num_sms() per process, so the device is deliberately not part of the key - a lookup per call costs
    # more than the whole ctypes call on the launch-bound small shapes)
    key = (fn_name,) + args
    v = _SIZES.get(key)
    if v is None:
        v = int(getattr(lib(), fn_name)(*args))
        _SIZES[key] = v
    return v


class _NullCtx:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NULL = _NullCtx()


def on_device(device):
    """`torch.cuda.device(device)` only when it is not already current (the context manager costs ~10 us)."""
    if torch.cuda.current_device() == device.index:
        return _NULL
    return torch.cuda.device(device)


def f32_scalar(t):
    """grad_output as a contiguous fp32 device scalar without redundant ops."""
    if t.dtype == torch.float32 and t.is_contiguous():
        return t
    return t.to(torch.float32).contiguous()

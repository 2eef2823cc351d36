"""Host-side plumbing over the C ABI for tests and bench.py: torch owns device memory and
streams, libb200va.so does the work.  Every function here ends in a C-ABI call on raw
pointers; nothing computes ``a + b`` in Python/torch (no fallback path).

Names follow the reference's process (SURVEY.md section 8(a)):
  a2 ``fill_rand_host`` / ``fill_ctr``     a4/a5 ``add``      a1 ``add_loop``
  a3+a4+a6 ``Stager`` / ``add_host``      a6 ``verify`` / ``verify_host``
whose only reference anchor is the call site ``cuda-test-deployment.yaml:18-19``.
"""
from __future__ import annotations

import ctypes as C
import subprocess

import numpy as np

from . import capi
from .capi import K_AUTO, VARIANTS, Tune, check, lib


def _torch():
    import torch
    return torch


def _variant(v) -> int:
    return VARIANTS[v] if isinstance(v, str) else int(v)


def _dev_ptr(t, name: str) -> int:
    torch = _torch()
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name} must be a CUDA tensor")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t.data_ptr()


def _stream_ptr(stream) -> int:
    torch = _torch()
    if stream is None:
        stream = torch.cuda.current_stream()
    return stream.cuda_stream


def add(a, b, out=None, *, variant=K_AUTO, tune: Tune | None = None, stream=None, inputs_stable: bool = False,
        cold: bool = False, full_matrix: bool = False):
    """C = A + B on the current CUDA stream (asynchronous). ``out`` may be ``a`` or ``b``.
    ``inputs_stable``: b200va_add_f32_ex with B200VA_F_INPUTS_STABLE (the previous launch on the
    stream does not write a or b); ``cold``: B200VA_F_COLD (operands not in L2).  ``full_matrix``: send an explicit ``tune`` to
    libb200va_tune.so, which carries every geometry (the production library refuses the
    ones AUTO never picks with ERR_VARIANT)."""
    torch = _torch()
    if a.numel() != b.numel():
        raise ValueError("a and b differ in length")
    if out is None:
        out = torch.empty_like(a)
    if out.numel() != a.numel():
        raise ValueError("out differs in length")
    pa, pb, pc = _dev_ptr(a, "a"), _dev_ptr(b, "b"), _dev_ptr(out, "out")
    with torch.cuda.device(a.device):
        if tune is not None:
            h = capi.tune_lib() if full_matrix else lib
            check(h.b200va_add_f32_tuned(pa, pb, pc, a.numel(), C.byref(tune), _stream_ptr(stream)), "b200va_add_f32_tuned")
        elif inputs_stable or cold:
            flags = (capi.F_INPUTS_STABLE if inputs_stable else 0) | (capi.F_COLD if cold else 0)
            check(lib.b200va_add_f32_ex(pa, pb, pc, a.numel(), _variant(variant), flags, _stream_ptr(stream)), "b200va_add_f32_ex")
        else:
            check(lib.b200va_add_f32(pa, pb, pc, a.numel(), _variant(variant), _stream_ptr(stream)), "b200va_add_f32")
    return out


def add_loop(a, b, out, iters: int, *, graph_batch: int = 0, variant=K_AUTO, stream=None):
    """The launch loop in-process: ``iters`` launches (CUDA-graph batched if graph_batch>1)."""
    torch = _torch()
    pa, pb, pc = _dev_ptr(a, "a"), _dev_ptr(b, "b"), _dev_ptr(out, "out")
    with torch.cuda.device(a.device):
        check(lib.b200va_add_f32_loop(pa, pb, pc, a.numel(), _variant(variant), iters, graph_batch,
                                      _stream_ptr(stream)), "b200va_add_f32_loop")
    return out


class Loop:
    """The persistent launch loop (a1): ``graph_batch`` launches captured once into a CUDA graph,
    ``run(iters)`` replays it asynchronously on the current stream (b200va_loop_*)."""

    def __init__(self, a, b, out, *, graph_batch: int = 50, variant=K_AUTO):
        torch = _torch()
        self._h = C.c_void_p()
        self._keep = (a, b, out)
        self._device = a.device
        with torch.cuda.device(a.device):
            check(lib.b200va_loop_create(C.byref(self._h), _dev_ptr(a, "a"), _dev_ptr(b, "b"), _dev_ptr(out, "out"), a.numel(),
                                         _variant(variant), graph_batch), "b200va_loop_create")

    def run(self, iters: int, *, stream=None) -> None:
        torch = _torch()
        with torch.cuda.device(self._device):
            check(lib.b200va_loop_run(self._h, iters, _stream_ptr(stream)), "b200va_loop_run")

    def close(self) -> None:
        """Destroy the graph; the stream must have drained."""
        if self._h:
            lib.b200va_loop_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        _torch().cuda.synchronize(self._device)
        self.close()


_TORCH_DT = {"f32": "float32", "f64": "float64", "f16": "float16", "bf16": "bfloat16"}


def stream(op: str, a, b=None, out=None, *, scalar: float = 0.0, stream=None):
    """STREAM-style op (copy | scale | add | triad) on CUDA tensors of f32/f64/f16/bf16
    through b200va_stream.  Asynchronous on the current stream."""
    torch = _torch()
    names = {getattr(torch, v): k for k, v in _TORCH_DT.items()}
    if not a.is_cuda or a.dtype not in names or not a.is_contiguous():
        raise TypeError("a must be a contiguous CUDA tensor of float32/float64/float16/bfloat16")
    if out is None:
        out = torch.empty_like(a)
    for t in (b, out):
        if t is not None and (t.dtype != a.dtype or t.numel() != a.numel() or not t.is_cuda or not t.is_contiguous()):
            raise TypeError("operands must match a in dtype, length and device")
    with torch.cuda.device(a.device):
        check(lib.b200va_stream(capi.OPS[op], capi.DTYPES[names[a.dtype]], a.data_ptr(), b.data_ptr() if b is not None else None,
                                out.data_ptr(), a.numel(), float(scalar), _stream_ptr(stream)), "b200va_stream")
    return out


def stream_grouped(op: str, a_list, b_list=None, out_list=None, *, scalar: float = 0.0, stream=None) -> list:
    """``stream`` over many independent vectors in one b200va_stream_grouped call: item i is
    op(a_list[i], b_list[i]) into out_list[i], bit-identical to ``stream`` on it.  Outputs are
    allocated like ``stream`` does when ``out_list`` is None.  All tensors share one dtype and
    one device; no output may overlap another item's tensors.  Asynchronous on the current stream."""
    torch = _torch()
    names = {getattr(torch, v): k for k, v in _TORCH_DT.items()}
    a_list = list(a_list)
    if out_list is None:
        out_list = [torch.empty_like(a) for a in a_list]
    out_list = list(out_list)
    b_list = [None] * len(a_list) if b_list is None else list(b_list)
    if not (len(a_list) == len(b_list) == len(out_list)):
        raise TypeError("a_list, b_list and out_list differ in length")
    if not a_list:
        return out_list
    dtype, device = a_list[0].dtype, a_list[0].device
    if dtype not in names or device.type != "cuda":
        raise TypeError("operands must be CUDA tensors of float32/float64/float16/bfloat16")
    items = (capi.Item * len(a_list))()
    for i, (a, b, c) in enumerate(zip(a_list, b_list, out_list)):
        for t in (a, b, c):
            if t is not None and (t.dtype != dtype or t.device != device or not t.is_contiguous()):
                raise TypeError(f"item {i}: operands must be contiguous tensors of one dtype on one device")
        if (b is not None and b.numel() != a.numel()) or c.numel() != a.numel():
            raise TypeError(f"item {i}: operands differ in length")
        items[i] = capi.Item(a.data_ptr(), b.data_ptr() if b is not None else None, c.data_ptr(), a.numel())
    with torch.cuda.device(device):
        check(lib.b200va_stream_grouped(capi.OPS[op], capi.DTYPES[names[dtype]], items, len(a_list), float(scalar),
                                        _stream_ptr(stream)), "b200va_stream_grouped")
    return out_list


def probe(kind: str, a, b, c, *, stream=None):
    """Ceiling probe (b200va_probe_f32): 'read2' loads a and b, 'fill' stores c, 'copy' c = a.  c is clobbered."""
    torch = _torch()
    with torch.cuda.device(c.device):
        check(lib.b200va_probe_f32(capi.PROBES[kind], a.data_ptr() if a is not None else None, b.data_ptr() if b is not None else None,
                                   _dev_ptr(c, "c"), c.numel(), _stream_ptr(stream)), "b200va_probe_f32")


def fill_ctr(out, seed: int, first: int = 0, *, stream=None):
    """Counter generator on the device: out[i] = ctr(seed, first + i)."""
    torch = _torch()
    with torch.cuda.device(out.device):
        check(lib.b200va_fill_ctr_f32(_dev_ptr(out, "out"), out.numel(), seed, first, _stream_ptr(stream)),
              "b200va_fill_ctr_f32")
    return out


def fill_ctr_host(n: int, seed: int, first: int = 0) -> np.ndarray:
    x = np.empty(n, dtype=np.float32)
    check(lib.b200va_host_fill_ctr_f32(x.ctypes.data, n, seed, first), "b200va_host_fill_ctr_f32")
    return x


def fill_rand_host(n: int) -> tuple[np.ndarray, np.ndarray]:
    """The sample's input recipe (interleaved, never-seeded rand())."""
    a, b = np.empty(n, dtype=np.float32), np.empty(n, dtype=np.float32)
    check(lib.b200va_host_fill_rand_f32(a.ctypes.data, b.ctypes.data, n), "b200va_host_fill_rand_f32")
    return a, b


def verify(a, b, c, *, stream=None) -> tuple[int, int]:
    """Device-side bitwise check; returns (mismatch count, first bad index or -1). Synchronises."""
    torch = _torch()
    res = torch.empty(2, dtype=torch.int64, device=a.device)
    with torch.cuda.device(a.device):
        check(lib.b200va_verify_f32(_dev_ptr(a, "a"), _dev_ptr(b, "b"), _dev_ptr(c, "c"), a.numel(),
                                    res.data_ptr(), _stream_ptr(stream)), "b200va_verify_f32")
    bad, first = (int(v) & 0xFFFFFFFFFFFFFFFF for v in res.tolist())
    return bad, (-1 if bad == 0 else first)


def digest(x, *, stream=None) -> tuple[int, int]:
    """(sum of uint32 bit patterns mod 2^64, xor of them) computed in HBM. Synchronises."""
    torch = _torch()
    res = torch.empty(2, dtype=torch.int64, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.b200va_digest_f32(_dev_ptr(x, "x"), x.numel(), res.data_ptr(), _stream_ptr(stream)),
              "b200va_digest_f32")
    s, xo = (int(v) & 0xFFFFFFFFFFFFFFFF for v in res.tolist())
    return s, xo


def verify_host(a: np.ndarray, b: np.ndarray, c: np.ndarray) -> int:
    """The sample's self-check made strict (bitwise). Returns -1 or the first bad index."""
    bad = C.c_size_t(0)
    rc = lib.b200va_host_verify_f32(a.ctypes.data, b.ctypes.data, c.ctypes.data, a.size, C.byref(bad))
    if rc == capi.OK:
        return -1
    if rc == capi.ERR_VERIFY:
        return bad.value
    check(rc, "b200va_host_verify_f32")
    return -1


def _host_ptr(x, name: str) -> int:
    torch = _torch()
    if isinstance(x, np.ndarray):
        if x.dtype != np.float32 or not x.flags.c_contiguous:
            raise TypeError(f"{name} must be a C-contiguous float32 array")
        return x.ctypes.data
    if isinstance(x, torch.Tensor) and not x.is_cuda and x.dtype == torch.float32 and x.is_contiguous():
        return x.data_ptr()
    raise TypeError(f"{name} must be a float32 numpy array or CPU tensor")


class PinnedBuffer:
    """Pinned, GPU-local-NUMA host memory from b200va_host_alloc, viewed as a float32 numpy
    array (``.array``).  The memory lives until ``free()`` / garbage collection."""

    def __init__(self, n: int, write_combined: bool = False):
        self._p = C.c_void_p()
        self.n = n
        check(lib.b200va_host_alloc_ex(C.byref(self._p), max(1, n) * 4, 1 if write_combined else 0), "b200va_host_alloc_ex")
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_float)), shape=(n,))

    @property
    def numa_node(self) -> int:
        """NUMA node of the first page (-1 if unknown)."""
        return int(lib.b200va_host_node_of(self._p)) if self._p else -1

    def free(self):
        if self._p:
            self.array = None
            lib.b200va_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Stager:
    """Host-buffer path (a3 + a4 + a6-copy): H2D, add and D2H pipelined in chunks."""

    def __init__(self, device: int = 0, chunk_elems: int = 0, depth: int = 0):
        self._h = C.c_void_p()
        check(lib.b200va_stager_create(C.byref(self._h), device, chunk_elems, depth), "b200va_stager_create")

    def add(self, a, b, out, *, variant=K_AUTO, zero_copy: bool = False, mode: int | None = None) -> float:
        """Synchronous; returns the device-timed milliseconds of the whole pipeline.
        mode: -1 auto (default), 0 slot streams, 1 zero-copy kernel, 2 lanes (one stream per
        direction), 3 pageable arrays through a pinned bounce ring, 4 register-once."""
        n = a.size if isinstance(a, np.ndarray) else a.numel()
        if mode is None:
            mode = capi.STAGE_ZEROCOPY if zero_copy else capi.STAGE_AUTO
        check(lib.b200va_stager_add_f32(self._h, _host_ptr(a, "a"), _host_ptr(b, "b"), _host_ptr(out, "out"), n,
                                        _variant(variant), mode), "b200va_stager_add_f32")
        ms = C.c_float()
        check(lib.b200va_stager_last_ms(self._h, C.byref(ms)), "b200va_stager_last_ms")
        return ms.value

    @property
    def last_mode(self) -> int:
        """The pipeline the last ``add`` actually ran (after AUTO / fallbacks)."""
        m = C.c_int(-2)
        check(lib.b200va_stager_last_mode(self._h, C.byref(m)), "b200va_stager_last_mode")
        return m.value

    def release_host(self) -> None:
        """Unregister the host arrays the register-once path page-locked."""
        check(lib.b200va_stager_release_host(self._h), "b200va_stager_release_host")

    def close(self):
        if self._h:
            lib.b200va_stager_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def add_host(a: np.ndarray, b: np.ndarray, out: np.ndarray | None = None, *, device: int = 0, variant=K_AUTO):
    """One ``./vectorAdd`` worth of work on host arrays: alloc, H2D, add, D2H, free."""
    if out is None:
        out = np.empty_like(a)
    check(lib.b200va_add_f32_host(_host_ptr(a, "a"), _host_ptr(b, "b"), _host_ptr(out, "out"), a.size, device,
                                  _variant(variant)), "b200va_add_f32_host")
    return out


def run_cli(*args: str, timeout: float = 600.0) -> subprocess.CompletedProcess:
    """Run the drop-in ``vectorAdd`` executable (the outer boundary)."""
    return subprocess.run([capi.CLI_PATH, *args], capture_output=True, text=True, timeout=timeout)

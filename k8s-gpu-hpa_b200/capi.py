"""ctypes binding of libb200va.so -- one Python function per symbol of include/b200va.h.

This is the same stub a maintainer would write for any other host language (see
INTEGRATION.md): plain pointers and sizes across the boundary.  The library is built
in-tree by ``make -C k8s-gpu-hpa_b200`` (``__graft_entry__.build()``); if it is missing
the import fails loudly -- there is no Python/CPU fallback for the hot path.

Reference interface replaced: the ``./vectorAdd`` process of
``cuda-test-deployment.yaml:18-19`` (SURVEY.md section 8(a)/(b)).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200va.so")
TUNE_LIB_PATH = os.path.join(_HERE, "libb200va_tune.so")   # same ABI, every b200va_tune_t combination (development)
CLI_PATH = os.path.join(_HERE, "vectorAdd")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "b200va.h")

OK = 0
ERR_INVALID, ERR_ALIGN, ERR_OVERLAP, ERR_VARIANT, ERR_NO_DEVICE, ERR_VERIFY, ERR_NOMEM = -1, -2, -3, -4, -5, -6, -7
ERR_CUDA_BASE = -1000
K_AUTO, K0_SCALAR, K1_VEC128, K2_TMA, K3_VEC256, K4_SCALAR_MLP = 0, 1, 2, 3, 4, 5
F_INPUTS_STABLE, F_COLD = 1, 2
STAGE_AUTO, STAGE_SLOTS, STAGE_ZEROCOPY, STAGE_LANES, STAGE_BOUNCE, STAGE_REGISTER = -1, 0, 1, 2, 3, 4
PROBES = {"read2": 0, "fill": 1, "copy": 2}
OPS = {"copy": 0, "scale": 1, "add": 2, "triad": 3}
DTYPES = {"f32": 0, "f64": 1, "f16": 2, "bf16": 3}
VARIANTS = {"auto": K_AUTO, "k0": K0_SCALAR, "k1": K1_VEC128, "k2": K2_TMA, "k3": K3_VEC256}


class B200VAError(RuntimeError):
    def __init__(self, code: int, what: str = ""):
        self.code = code
        super().__init__(f"{what + ': ' if what else ''}{strerror(code)} ({code})")


class Tune(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("kind", "threads", "unroll", "ctas_per_sm", "ld_hint", "st_hint",
                                       "stages", "tile_bytes", "store_mode", "early_loads", "scheduler")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}

    def kernel_name(self) -> str:
        """The kernel this tune launches, as ncu prints it minus the (int)/(bool) casts: the key
        of the per-kernel table in profiles/ncu_summary.json."""
        if self.kind == K0_SCALAR:
            return "vadd_scalar"
        if self.kind == K2_TMA:
            hint = int(self.ld_hint == 3)
            if self.store_mode == 2:
                return f"vadd_tma_clc<{hint},{self.st_hint}>"
            return f"vadd_tma<{self.store_mode},{hint},{self.st_hint if self.store_mode == 0 else 0}>"
        if self.kind == K4_SCALAR_MLP:
            return f"vadd_scalar_unrolled<{self.unroll}>"
        name = "vadd_vec_clc" if self.scheduler == 1 else "vadd_vec"
        return f"{name}<{8 if self.kind == K3_VEC256 else 4},{self.unroll},{self.ld_hint},{self.st_hint},{self.early_loads}>"


class DevInfo(C.Structure):
    _fields_ = [("device", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int), ("sm_count", C.c_int),
                ("max_smem_optin", C.c_int), ("l2_bytes", C.c_int), ("global_mem_bytes", C.c_size_t),
                ("name", C.c_char * 64)]


class Item(C.Structure):
    """b200va_item_t: one (A, B, C, n) item of b200va_stream_grouped."""
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("c", C.c_void_p), ("n", C.c_size_t)]


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `make -C {_HERE}` (or __graft_entry__.build()). "
        "The vectorAdd hot path has no fallback implementation.")

lib = C.CDLL(LIB_PATH)

_P, _SZ, _I, _U64 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64
_SIGS = {
    "b200va_abi_version": (_I, []),
    "b200va_strerror": (C.c_char_p, [_I]),
    "b200va_query": (_I, [_I, C.POINTER(DevInfo)]),
    "b200va_resolve": (_I, [_I, _SZ, C.POINTER(Tune)]),
    "b200va_resolve_ex": (_I, [_I, _SZ, C.c_uint, C.POINTER(Tune)]),
    "b200va_geometry": (_I, [C.POINTER(Tune), _SZ, _I, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(C.c_uint)]),
    "b200va_add_f32": (_I, [_P, _P, _P, _SZ, _I, _P]),
    "b200va_add_f32_tuned": (_I, [_P, _P, _P, _SZ, C.POINTER(Tune), _P]),
    "b200va_add_f32_ex": (_I, [_P, _P, _P, _SZ, _I, C.c_uint, _P]),
    "b200va_add_f32_loop": (_I, [_P, _P, _P, _SZ, _I, _I, _I, _P]),
    "b200va_loop_create": (_I, [C.POINTER(_P), _P, _P, _P, _SZ, _I, _I]),
    "b200va_loop_run": (_I, [_P, _I, _P]),
    "b200va_loop_destroy": (_I, [_P]),
    "b200va_host_fill_rand_f32": (_I, [_P, _P, _SZ]),
    "b200va_host_fill_ctr_f32": (_I, [_P, _SZ, _U64, _U64]),
    "b200va_fill_ctr_f32": (_I, [_P, _SZ, _U64, _U64, _P]),
    "b200va_host_verify_f32": (_I, [_P, _P, _P, _SZ, C.POINTER(_SZ)]),
    "b200va_verify_f32": (_I, [_P, _P, _P, _SZ, _P, _P]),
    "b200va_digest_f32": (_I, [_P, _SZ, _P, _P]),
    "b200va_stager_create": (_I, [C.POINTER(_P), _I, _SZ, _I]),
    "b200va_stager_add_f32": (_I, [_P, _P, _P, _P, _SZ, _I, _I]),
    "b200va_stager_last_ms": (_I, [_P, C.POINTER(C.c_float)]),
    "b200va_stager_last_mode": (_I, [_P, C.POINTER(_I)]),
    "b200va_stager_release_host": (_I, [_P]),
    "b200va_stager_destroy": (_I, [_P]),
    "b200va_add_f32_host": (_I, [_P, _P, _P, _SZ, _I, _I]),
    "b200va_host_alloc": (_I, [C.POINTER(_P), _SZ]),
    "b200va_host_alloc_ex": (_I, [C.POINTER(_P), _SZ, _I]),
    "b200va_host_free": (_I, [_P]),
    "b200va_host_node_of": (_I, [_P]),
    "b200va_device_numa_node": (_I, []),
    "b200va_device_numa_node_of": (_I, [_I]),
    "b200va_stream": (_I, [_I, _I, _P, _P, _P, _SZ, C.c_double, _P]),
    "b200va_stream_grouped": (_I, [_I, _I, C.POINTER(Item), _SZ, C.c_double, _P]),
    "b200va_probe_f32": (_I, [_I, _P, _P, _P, _SZ, _P]),
    "b200va_shard_range": (_I, [_SZ, _I, _I, C.POINTER(_SZ), C.POINTER(_SZ)]),
}
def _bind(handle) -> None:
    for _name, (_res, _args) in _SIGS.items():
        _f = getattr(handle, _name)          # AttributeError here = header/library mismatch
        _f.restype, _f.argtypes = _res, _args


_bind(lib)
EXPORTED = tuple(_SIGS)
_tune_lib = None


def tune_lib():
    """libb200va_tune.so: the same C ABI with the full A/B matrix of b200va_tune_t compiled in
    (the production library carries only what AUTO and the named variants resolve to)."""
    global _tune_lib
    if _tune_lib is None:
        if not os.path.exists(TUNE_LIB_PATH):
            raise ImportError(f"{TUNE_LIB_PATH} is missing: build it with `make -C {_HERE}`")
        _tune_lib = C.CDLL(TUNE_LIB_PATH)
        _bind(_tune_lib)
    return _tune_lib


def strerror(code: int) -> str:
    return lib.b200va_strerror(code).decode()


def check(code: int, what: str = "") -> None:
    if code != OK:
        raise B200VAError(code, what)


def abi_version() -> int:
    return lib.b200va_abi_version()


def query(device: int = 0) -> DevInfo:
    info = DevInfo()
    check(lib.b200va_query(device, C.byref(info)), "b200va_query")
    return info


def resolve(variant: int, n: int, flags: int = 0) -> Tune:
    t = Tune()
    check(lib.b200va_resolve_ex(variant, n, flags, C.byref(t)), "b200va_resolve_ex")
    return t


def shard_range(n: int, world: int, rank: int) -> tuple[int, int]:
    b, e = _SZ(), _SZ()
    check(lib.b200va_shard_range(n, world, rank, C.byref(b), C.byref(e)), "b200va_shard_range")
    return b.value, e.value

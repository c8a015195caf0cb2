"""ctypes binding of the C ABI (include/qdc_primitives.h, include/qdc_circuit.h).

This is the Python counterpart of the reference's Rust FFI block
(/root/reference/src/primitives_bind.rs:15-119): plain pointers and sizes, no
torch types.  There is NO fallback: if the CUDA library is missing the import
of a precision raises, loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBDIR = os.path.join(_HERE, "lib")

c_cplx_p = C.c_void_p  # device or host pointer to interleaved (re, im)
_sz = C.c_size_t
_err = C.c_void_p      # const char* (heap message, never freed -- reference convention)

# name -> (restype, argtypes); the 18 legacy symbols first
_SIGNATURES = {
    "set2standard": (None, [c_cplx_p, _sz]),
    "get_state": (_err, [C.POINTER(C.c_void_p), _sz]),
    "drop_state": (_err, [c_cplx_p]),
    "copy_to_host": (_err, [c_cplx_p, c_cplx_p, _sz]),
    "set_from_host": (_err, [c_cplx_p, c_cplx_p, _sz]),
    "q1gate": (_err, [c_cplx_p, c_cplx_p, _sz, _sz]),
    "q1gate_inv": (_err, [c_cplx_p, c_cplx_p, _sz, _sz]),
    "q2gate": (_err, [c_cplx_p, c_cplx_p, _sz, _sz, _sz]),
    "q2gate_inv": (_err, [c_cplx_p, c_cplx_p, _sz, _sz, _sz]),
    "q2gate_diag": (_err, [c_cplx_p, c_cplx_p, _sz, _sz, _sz]),
    "get_q1density": (_err, [c_cplx_p, c_cplx_p, _sz, _sz]),
    "get_q2density": (_err, [c_cplx_p, c_cplx_p, _sz, _sz, _sz]),
    "q1grad": (_err, [c_cplx_p, c_cplx_p, c_cplx_p, _sz, _sz]),
    "q2grad": (_err, [c_cplx_p, c_cplx_p, c_cplx_p, _sz, _sz, _sz]),
    "q2grad_diag": (_err, [c_cplx_p, c_cplx_p, c_cplx_p, _sz, _sz, _sz]),
    "conj_and_double": (None, [c_cplx_p, c_cplx_p, _sz]),
    "add": (None, [c_cplx_p, c_cplx_p, _sz]),
    "copy": (None, [c_cplx_p, c_cplx_p, _sz]),
}
LEGACY_SYMBOLS = tuple(_SIGNATURES)

_u32p = C.c_void_p
_CIRCUIT_SIGNATURES = {
    "qdc_precision": (C.c_char_p, []),
    "qdc_abi_version": (C.c_int, []),
    "qdc_circuit_new": (_err, [C.POINTER(C.c_void_p), _sz]),
    "qdc_circuit_new_sharded": (_err, [C.POINTER(C.c_void_p), _sz, C.c_int, C.c_int, C.c_void_p]),
    "qdc_nccl_unique_id": (_err, [C.c_void_p]),
    "qdc_circuit_peer_exchange": (C.c_int, [C.c_void_p]),
    "qdc_circuit_free": (_err, [C.c_void_p]),
    "qdc_circuit_set_state_from_host": (_err, [C.c_void_p, c_cplx_p, _sz]),
    "qdc_circuit_add": (_err, [C.c_void_p, C.c_int, _sz, _sz]),
    "qdc_circuit_add_dens": (_err, [C.c_void_p, C.c_void_p, _sz, C.c_int]),
    "qdc_circuit_add_gate": (_err, [C.c_void_p, C.c_void_p, _sz, C.c_int, C.c_int]),
    "qdc_circuit_add_gate_diag": (_err, [C.c_void_p, C.c_void_p, _sz, C.c_int, C.c_int]),
    "qdc_circuit_count": (_sz, [C.c_void_p, C.c_int]),
    "qdc_circuit_run": (_err, [C.c_void_p, c_cplx_p, _u32p, _sz, c_cplx_p, _u32p, _sz, c_cplx_p, _sz,
                               C.POINTER(_sz)]),
    "qdc_circuit_forward": (_err, [C.c_void_p, c_cplx_p, _u32p, _sz, c_cplx_p, _u32p, _sz, c_cplx_p, _sz,
                                   C.POINTER(_sz)]),
    "qdc_circuit_backward": (_err, [C.c_void_p, c_cplx_p, _u32p, _sz, c_cplx_p, _u32p, _sz, c_cplx_p, _u32p,
                                    _sz, c_cplx_p, _sz, C.POINTER(_sz)]),
    "qdc_circuit_copy_state_to_host": (_err, [C.c_void_p, c_cplx_p]),
    "qdc_circuit_state_device_ptr": (_err, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "qdc_schedule_set_strategy": (_err, [C.c_int]),
    "qdc_schedule_set_swap_min_pos": (_err, [C.c_int]),
    "qdc_circuit_save_state": (_err, [C.c_void_p, C.c_char_p]),
    "qdc_circuit_load_state": (_err, [C.c_void_p, C.c_char_p]),
    "qdc_circuit_state_layout": (_err, [C.c_void_p, C.POINTER(C.c_int)]),
    "qdc_circuit_set_stream": (_err, [C.c_void_p, C.c_void_p]),
    "qdc_circuit_set_option": (_err, [C.c_void_p, C.c_char_p, C.c_long]),
    "qdc_circuit_last_stats": (_err, [C.c_void_p, C.c_void_p]),
    "qdc_profile_categories": (C.c_int, []),
    "qdc_profile_category_name": (C.c_char_p, [C.c_int]),
    "qdc_circuit_last_profile": (_err, [C.c_void_p, C.c_int, C.c_void_p]),
    "qdc_schedule": (_err, [_sz, _sz, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, _sz, C.c_int,
                            C.c_void_p, _sz, C.POINTER(_sz)]),
    "qdc_reverse_step": (_err, [c_cplx_p, c_cplx_p, c_cplx_p, c_cplx_p, C.c_int, C.c_int, _sz, _sz, _sz]),
    "qdc_density_seed": (_err, [c_cplx_p, c_cplx_p, c_cplx_p, C.c_int, C.c_int, _sz, _sz, _sz]),
}
_SIGNATURES.update(_CIRCUIT_SIGNATURES)
ALL_SYMBOLS = tuple(_SIGNATURES)


class QdcError(RuntimeError):
    """Raised where the reference's Rust layer would panic (PyO3 PanicException)."""


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("hbm_passes", C.c_uint64),
                ("algorithmic_bytes", C.c_uint64)]


class ProfileEntry(C.Structure):
    _fields_ = [("launches", C.c_uint64), ("ms", C.c_double), ("algorithmic_bytes", C.c_uint64)]


def lib_path(precision: str) -> str:
    # QDC_LIB_VARIANT: development knob -- load lib/libqdc_b200_<precision>_<variant>.so, an experimental
    # build of the same sources with other -D flags (profiles/scripts/build_variants.py)
    variant = os.environ.get("QDC_LIB_VARIANT", "")
    if variant:
        p = os.path.join(_LIBDIR, f"libqdc_b200_{precision}_{variant}.so")
        if os.path.exists(p):
            return p
    return os.path.join(_LIBDIR, f"libqdc_b200_{precision}.so")


class Lib:
    """One loaded precision build of the library."""

    def __init__(self, precision: str, path: str | None = None):
        if precision not in ("f32", "f64"):
            raise ValueError("precision must be 'f32' or 'f64'")
        self.precision = precision
        self.cdtype = np.dtype(np.complex64 if precision == "f32" else np.complex128)
        self.path = path or lib_path(precision)
        if not os.path.exists(self.path):
            raise ImportError(
                f"{self.path} is missing: the CUDA extension was not built "
                f"(run `python -c 'import __graft_entry__ as g; g.build()'`). "
                f"There is no CPU fallback."
            )
        self.cdll = C.CDLL(self.path, mode=os.RTLD_LOCAL | os.RTLD_NOW)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(self.cdll, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        got = self.cdll.qdc_precision().decode()
        if got != precision:
            raise ImportError(f"{self.path} reports precision {got}, expected {precision}")

    # ------------------------------------------------------------------
    @staticmethod
    def check(err):
        """NULL-or-message convention (src/primitives.cu:32-49, quantized_tensor.rs:37-42)."""
        if err:
            raise QdcError(C.string_at(err).decode(errors="replace"))

    def call(self, name: str, *args):
        fn = getattr(self.cdll, name)
        out = fn(*args)
        if fn.restype is _err:
            self.check(out)
            return None
        return out

    def host(self, arr, length: int | None = None) -> np.ndarray:
        """A contiguous host array of the build's complex dtype (strict, like
        PyO3's PyReadonlyArray<Complex> extraction)."""
        a = np.asarray(arr)
        if a.dtype != self.cdtype:
            raise TypeError(f"array has dtype {a.dtype}, this build expects {self.cdtype}")
        a = np.ascontiguousarray(a)
        if length is not None and a.size != length:
            raise QdcError("Incorrect len of the gate's buffer.")
        return a


_LIBS: Dict[str, Lib] = {}


def get_lib(precision: str) -> Lib:
    if precision not in _LIBS:
        _LIBS[precision] = Lib(precision)
    return _LIBS[precision]


def schedule(instructions, n, n_loc=None, tile_bits=0, low_bits=0, max_tile_gates=0, all_densities=False,
             precision="f32", tile_strategy=-1, swap_min_pos=-1):
    """Run the C++ pass scheduler (pure host code) on `instructions`, a list of
    (kind, pos2[, pos1]) tuples; returns the int64 plan encoding of qdc_schedule."""
    lib = get_lib(precision)
    kinds = np.array([i[0] for i in instructions], dtype=np.int32)
    p2 = np.array([i[1] for i in instructions], dtype=np.uint64)
    p1 = np.array([i[2] if len(i) > 2 else 0 for i in instructions], dtype=np.uint64)
    cap = 64 + 16 * len(instructions) + 64 * len(instructions)
    out = np.zeros(cap, dtype=np.int64)
    n_out = C.c_size_t(0)
    lib.call("qdc_schedule_set_strategy", int(tile_strategy))
    lib.call("qdc_schedule_set_swap_min_pos", int(swap_min_pos))   # -1 default, -2 cost model (sharded circuits)
    lib.call("qdc_schedule", n, n if n_loc is None else n_loc, tile_bits, low_bits, max_tile_gates,
             kinds.ctypes.data, p2.ctypes.data, p1.ctypes.data, len(instructions), int(all_densities),
             out.ctypes.data, cap, C.byref(n_out))
    return out[:n_out.value].copy()


def precision_of(dtype) -> str:
    dt = np.dtype(dtype)
    if dt == np.complex64:
        return "f32"
    if dt == np.complex128:
        return "f64"
    raise TypeError(f"unsupported dtype {dt}")


def default_precision() -> str:
    """The reference builds f32 unless `--features f64` (Cargo.toml:25-27)."""
    return os.environ.get("QDC_PRECISION", "f32")

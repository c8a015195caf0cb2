"""Drop-in for the reference's native module `quantum_differentiable_circuit`
(/root/reference/src/circuit.rs:432-436): class `Circuit` with the same
builder methods, `run`, `forward`, `backward` -- same names, argument orders
(`const_gates` before `var_gates`), output ordering and failure conditions.

Where the reference walks its instruction list issuing one FFI call per
instruction (src/circuit.rs:175, 226, 278), this class hands the whole program
to the C ABI (include/qdc_circuit.h) once per call.

Precision: the reference is compiled for exactly one precision (cargo feature
`f64`).  Here both builds ship; `Circuit(n)` uses `QDC_PRECISION` (default
"f32", the reference's default feature set) and `Circuit(n, precision="f64")`
or the aliases `quantum_differentiable_circuit.f64.Circuit` pick the other.
Arrays must be contiguous and of the build's complex dtype, as with PyO3's
`PyReadonlyArray1<Complex>`.
"""
from __future__ import annotations

import ctypes as C
import types
from typing import List, Sequence

import numpy as np

from .._ffi import Lib, ProfileEntry, QdcError, Stats, default_precision, get_lib

# enum Instruction, src/circuit.rs:53-68, then the densities and the gates on 3..6 qubits and the diagonal gates on
# 1..6 qubits (include/qdc_circuit.h)
(CONST_Q2, VAR_Q2, CONST_Q2_NONU, VAR_Q2_NONU, CONST_Q2_DIAG, VAR_Q2_DIAG, CONST_Q1, CONST_Q1_NONU, VAR_Q1,
 VAR_Q1_NONU, Q2_DENS, Q1_DENS, DIFF_Q2_DENS, DIFF_Q1_DENS, DENS_K, DIFF_DENS_K, CONST_GATE_K, VAR_GATE_K,
 CONST_GATE_K_NONU, VAR_GATE_K_NONU, CONST_GATE_K_DIAG, VAR_GATE_K_DIAG, CONST_GATE_K_DIAG_NONU,
 VAR_GATE_K_DIAG_NONU) = range(24)

(N_INSTRUCTIONS, N_CONST_GATES, N_VAR_GATES, N_DENSITIES, N_DIFF_DENSITIES, RUN_OUT_LEN, FORWARD_OUT_LEN,
 BACKWARD_OUT_LEN) = range(8)


class Circuit:
    def __init__(self, qubits_number: int, precision: str | None = None):
        self._lib: Lib = get_lib(precision or default_precision())
        self.qubits_number = int(qubits_number)
        h = C.c_void_p()
        self._lib.call("qdc_circuit_new", C.byref(h), self.qubits_number)
        self._h = h
        self._kinds: List[int] = []
        self._dims: List[int] = []   # side of every instruction's density output or k-qubit gate matrix, length of a
                                     # diagonal k-qubit gate (else 0)

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                self._lib.call("qdc_circuit_free", self._h)
                self._h = None
        except Exception:
            pass

    @property
    def dtype(self):
        return self._lib.cdtype

    # ---- src/circuit.rs:104-106 ----
    def set_state_from_vector(self, vector):
        v = self._lib.host(vector)
        if v.ndim != 1:
            raise TypeError("vector must be one-dimensional")
        self._lib.call("qdc_circuit_set_state_from_host", self._h, v.ctypes.data, v.size)

    # ---- builders, src/circuit.rs:108-162 ----
    def _add(self, kind, pos2, pos1=0):
        if pos2 < 0 or pos1 < 0:
            raise OverflowError("can't convert negative int to unsigned")
        self._lib.call("qdc_circuit_add", self._h, kind, pos2, pos1)
        self._kinds.append(kind)
        self._dims.append(2 if kind in (Q1_DENS, DIFF_Q1_DENS) else 4 if kind in (Q2_DENS, DIFF_Q2_DENS) else 0)

    def _add_dens_k(self, positions: List[int], with_grad: bool):
        if any(p < 0 for p in positions):
            raise OverflowError("can't convert negative int to unsigned")
        pos = np.array(positions, dtype=np.uintp)
        self._lib.call("qdc_circuit_add_dens", self._h, pos.ctypes.data, pos.size, int(with_grad))
        self._kinds.append(DIFF_DENS_K if with_grad else DENS_K)
        self._dims.append(1 << pos.size)

    def _add_gate_k(self, positions: List[int], variable: bool, non_unitary: bool):
        if any(p < 0 for p in positions):
            raise OverflowError("can't convert negative int to unsigned")
        pos = np.array(positions, dtype=np.uintp)
        self._lib.call("qdc_circuit_add_gate", self._h, pos.ctypes.data, pos.size, int(variable), int(non_unitary))
        self._kinds.append((VAR_GATE_K if variable else CONST_GATE_K) if not non_unitary
                           else (VAR_GATE_K_NONU if variable else CONST_GATE_K_NONU))
        self._dims.append(1 << pos.size)

    def _add_gate_diag_k(self, positions: List[int], variable: bool, non_unitary: bool):
        if any(p < 0 for p in positions):
            raise OverflowError("can't convert negative int to unsigned")
        pos = np.array(positions, dtype=np.uintp)
        self._lib.call("qdc_circuit_add_gate_diag", self._h, pos.ctypes.data, pos.size, int(variable),
                       int(non_unitary))
        self._kinds.append((VAR_GATE_K_DIAG if variable else CONST_GATE_K_DIAG) if not non_unitary
                           else (VAR_GATE_K_DIAG_NONU if variable else CONST_GATE_K_DIAG_NONU))
        self._dims.append(1 << pos.size)

    def add_q2_const_gate(self, pos2: int, pos1: int): self._add(CONST_Q2, pos2, pos1)
    def add_q2_const_gate_diag(self, pos2: int, pos1: int): self._add(CONST_Q2_DIAG, pos2, pos1)
    def add_q2_const_gate_nonu(self, pos2: int, pos1: int): self._add(CONST_Q2_NONU, pos2, pos1)
    def add_q2_var_gate(self, pos2: int, pos1: int): self._add(VAR_Q2, pos2, pos1)
    def add_q2_var_gate_diag(self, pos2: int, pos1: int): self._add(VAR_Q2_DIAG, pos2, pos1)
    def add_q2_var_gate_nonu(self, pos2: int, pos1: int): self._add(VAR_Q2_NONU, pos2, pos1)
    def add_q1_const_gate(self, pos: int): self._add(CONST_Q1, pos)
    def add_q1_const_gate_nonu(self, pos: int): self._add(CONST_Q1_NONU, pos)
    def add_q1_var_gate(self, pos: int): self._add(VAR_Q1, pos)
    def add_q1_var_gate_nonu(self, pos: int): self._add(VAR_Q1_NONU, pos)
    def get_q2_dens_op(self, pos2: int, pos1: int): self._add(Q2_DENS, pos2, pos1)
    def get_q1_dens_op(self, pos: int): self._add(Q1_DENS, pos)
    def get_q2_dens_op_with_grad(self, pos2: int, pos1: int): self._add(DIFF_Q2_DENS, pos2, pos1)
    def get_q1_dens_op_with_grad(self, pos: int): self._add(DIFF_Q1_DENS, pos)

    def get_dens_op(self, positions: Sequence[int]):
        """Reduced density matrix on the qubits `positions` = [p_{k-1}, ..., p_0] (1 <= k <= 6, distinct, any order):
        rho[r, c] = sum_rest psi[r, rest] conj psi[c, rest], shape (2^k, 2^k), positions[0] the most significant bit
        of r and c.  k = 1 and 2 are get_q1_dens_op(p) and get_q2_dens_op(p2, p1)."""
        self._add_dens(positions, False)

    def get_dens_op_with_grad(self, positions: Sequence[int]):
        """`get_dens_op` with gradient: forward returns it, backward takes its (2^k, 2^k) cotangent."""
        self._add_dens(positions, True)

    def add_const_gate(self, positions: Sequence[int]):
        """Gate on the qubits `positions` = [p_{k-1}, ..., p_0] (1 <= k <= 6, distinct, any order), positions[0] the
        most significant bit of its row and column index: psi'[r, rest] = sum_c U[r, c] psi[c, rest].  U is taken
        flat (4^k entries, row-major) from the constant gate list.  k = 1 and 2 are add_q1_const_gate(p) and
        add_q2_const_gate(p2, p1)."""
        self._add_gate(positions, False, False)

    def add_var_gate(self, positions: Sequence[int]):
        """`add_const_gate` from the variable gate list: backward returns its (4^k-entry) gradient."""
        self._add_gate(positions, True, False)

    def add_const_gate_nonu(self, positions: Sequence[int]):
        """`add_const_gate` for a non-unitary U (the reverse pass un-computes with its inverse)."""
        self._add_gate(positions, False, True)

    def add_var_gate_nonu(self, positions: Sequence[int]):
        """`add_var_gate` for a non-unitary U."""
        self._add_gate(positions, True, True)

    def _add_gate(self, positions, variable: bool, non_unitary: bool):
        pos = [int(p) for p in positions]
        if len(pos) == 1:
            getattr(self, "add_q1_%s_gate%s" % ("var" if variable else "const", "_nonu" if non_unitary else ""))(pos[0])
        elif len(pos) == 2:
            getattr(self, "add_q2_%s_gate%s" % ("var" if variable else "const", "_nonu" if non_unitary else ""))(
                pos[0], pos[1])
        else:
            self._add_gate_k(pos, variable, non_unitary)

    def add_const_gate_diag(self, positions: Sequence[int]):
        """Diagonal gate on the qubits `positions` = [p_{k-1}, ..., p_0] (1 <= k <= 6, distinct, any order),
        positions[0] the most significant bit of its index j: psi'[j, rest] = d[j] psi[j, rest].  d is taken flat
        (2^k entries) from the constant gate list.  k = 2 is add_q2_const_gate_diag(p2, p1)."""
        self._add_gate_diag(positions, False, False)

    def add_var_gate_diag(self, positions: Sequence[int]):
        """`add_const_gate_diag` from the variable gate list: backward returns its (2^k-entry) gradient
        G[j] = sum_rest bwd[j, rest] fwd[j, rest]."""
        self._add_gate_diag(positions, True, False)

    def add_const_gate_diag_nonu(self, positions: Sequence[int]):
        """`add_const_gate_diag` for a non-unitary d (the reverse pass un-computes with 1 / d)."""
        self._add_gate_diag(positions, False, True)

    def add_var_gate_diag_nonu(self, positions: Sequence[int]):
        """`add_var_gate_diag` for a non-unitary d."""
        self._add_gate_diag(positions, True, True)

    def _add_gate_diag(self, positions, variable: bool, non_unitary: bool):
        pos = [int(p) for p in positions]
        if len(pos) == 2 and not non_unitary:
            (self.add_q2_var_gate_diag if variable else self.add_q2_const_gate_diag)(pos[0], pos[1])
        else:
            self._add_gate_diag_k(pos, variable, non_unitary)

    def _add_dens(self, positions, with_grad: bool):
        pos = [int(p) for p in positions]
        if len(pos) == 1:
            (self.get_q1_dens_op_with_grad if with_grad else self.get_q1_dens_op)(pos[0])
        elif len(pos) == 2:
            (self.get_q2_dens_op_with_grad if with_grad else self.get_q2_dens_op)(pos[0], pos[1])
        else:
            self._add_dens_k(pos, with_grad)

    # ---- marshalling ----
    def _flatten(self, arrays: Sequence, ndim: int):
        """list of small arrays -> (flat complex array, uint32 lens).  Strict dtype."""
        arrs = []
        for a in arrays:
            a = np.asarray(a)
            if a.dtype != self._lib.cdtype:
                raise TypeError(f"array has dtype {a.dtype}, this build expects {self._lib.cdtype}")
            if a.ndim != ndim:
                raise TypeError(f"expected a {ndim}-D array, got {a.ndim}-D")
            arrs.append(np.ascontiguousarray(a).reshape(-1))
        lens = np.array([a.size for a in arrs], dtype=np.uint32)
        flat = np.concatenate(arrs) if arrs else np.zeros(0, dtype=self._lib.cdtype)
        return np.ascontiguousarray(flat, dtype=self._lib.cdtype), lens

    def _count(self, what: int) -> int:
        return int(self._lib.cdll.qdc_circuit_count(self._h, what))

    def _sweep(self, name, const_gates, var_gates, out_len_sel, dens_kinds):
        cf, cl = self._flatten(const_gates, 1)
        vf, vl = self._flatten(var_gates, 1)
        cap = self._count(out_len_sel)
        out = np.empty(max(cap, 1), dtype=self._lib.cdtype)
        n_out = C.c_size_t(0)
        self._lib.call(name, self._h, cf.ctypes.data, cl.ctypes.data, cl.size, vf.ctypes.data, vl.ctypes.data,
                       vl.size, out.ctypes.data, cap, C.byref(n_out))
        res, o = [], 0
        for k, m in zip(self._kinds, self._dims):
            if k in dens_kinds:
                res.append(out[o:o + m * m].reshape(m, m).copy())
                o += m * m
        assert o == n_out.value
        return res

    # ---- src/circuit.rs:164-212 ----
    def run(self, const_gates, var_gates) -> List[np.ndarray]:
        return self._sweep("qdc_circuit_run", const_gates, var_gates, RUN_OUT_LEN,
                           (Q1_DENS, Q2_DENS, DIFF_Q1_DENS, DIFF_Q2_DENS, DENS_K, DIFF_DENS_K))

    # ---- src/circuit.rs:214-264 ----
    def forward(self, const_gates, var_gates) -> List[np.ndarray]:
        return self._sweep("qdc_circuit_forward", const_gates, var_gates, FORWARD_OUT_LEN,
                           (DIFF_Q1_DENS, DIFF_Q2_DENS, DIFF_DENS_K))

    # ---- src/circuit.rs:266-429 ----
    def backward(self, grads_wrt_density, const_gates, var_gates) -> List[np.ndarray]:
        df, dl = self._flatten(grads_wrt_density, 2)
        cf, cl = self._flatten(const_gates, 1)
        vf, vl = self._flatten(var_gates, 1)
        cap = self._count(BACKWARD_OUT_LEN)
        out = np.empty(max(cap, 1), dtype=self._lib.cdtype)
        n_out = C.c_size_t(0)
        self._lib.call("qdc_circuit_backward", self._h, df.ctypes.data, dl.ctypes.data, dl.size,
                       cf.ctypes.data, cl.ctypes.data, cl.size, vf.ctypes.data, vl.ctypes.data, vl.size,
                       out.ctypes.data, cap, C.byref(n_out))
        res, o = [], 0
        for k, m in zip(self._kinds, self._dims):
            if k in (VAR_Q2, VAR_Q2_NONU):
                res.append(out[o:o + 16].copy()); o += 16
            elif k in (VAR_Q2_DIAG, VAR_Q1, VAR_Q1_NONU):
                res.append(out[o:o + 4].copy()); o += 4
            elif k in (VAR_GATE_K, VAR_GATE_K_NONU):
                res.append(out[o:o + m * m].copy()); o += m * m
            elif k in (VAR_GATE_K_DIAG, VAR_GATE_K_DIAG_NONU):
                res.append(out[o:o + m].copy()); o += m
        assert o == n_out.value
        return res

    # ---- extras (not in the reference's Python surface) ----
    def get_cpu_state_copy(self) -> np.ndarray:
        """QuantizedTensor::get_cpu_state_copy of the working state (src/quantized_tensor.rs:91-99)."""
        out = np.empty(1 << self.qubits_number, dtype=self._lib.cdtype)
        self._lib.call("qdc_circuit_copy_state_to_host", self._h, out.ctypes.data)
        return out

    def save_state(self, path: str):
        """Stream this rank's working state to `path` (format: include/qdc_circuit.h, `state_io.read_state`)."""
        self._lib.call("qdc_circuit_save_state", self._h, str(path).encode())

    def load_state(self, path: str):
        """Install the state file `path` (identity layout) as the initial state, like set_state_from_vector."""
        self._lib.call("qdc_circuit_load_state", self._h, str(path).encode())

    def state_layout(self) -> List[int]:
        """Physical position of every logical qubit in the working state (identity unless sharded mid-sweep)."""
        out = (C.c_int * self.qubits_number)()
        self._lib.call("qdc_circuit_state_layout", self._h, out)
        return list(out)

    def set_option(self, key: str, value: int):
        self._lib.call("qdc_circuit_set_option", self._h, key.encode(), int(value))

    def set_stream(self, cuda_stream: int):
        self._lib.call("qdc_circuit_set_stream", self._h, C.c_void_p(cuda_stream))

    def last_stats(self) -> dict:
        s = Stats()
        self._lib.call("qdc_circuit_last_stats", self._h, C.byref(s))
        return {"kernel_launches": s.kernel_launches, "hbm_passes": s.hbm_passes,
                "algorithmic_bytes": s.algorithmic_bytes}


    def last_profile(self) -> dict:
        """Per-category device time of the last call (needs set_option("profile", 1))."""
        out = {}
        for cat in range(self._lib.cdll.qdc_profile_categories()):
            e = ProfileEntry()
            self._lib.call("qdc_circuit_last_profile", self._h, cat, C.byref(e))
            if e.launches:
                out[self._lib.cdll.qdc_profile_category_name(cat).decode()] = {
                    "launches": e.launches, "ms": e.ms, "algorithmic_bytes": e.algorithmic_bytes}
        return out


def _variant(precision: str):
    mod = types.ModuleType(f"{__name__}.{precision}")

    class _Circuit(Circuit):
        def __init__(self, qubits_number: int):
            super().__init__(qubits_number, precision=precision)

    _Circuit.__name__ = "Circuit"
    mod.Circuit = _Circuit
    return mod


f32 = _variant("f32")
f64 = _variant("f64")

__all__ = ["Circuit", "QdcError", "f32", "f64"]

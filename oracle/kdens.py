"""Oracle of the reduced density matrices on k = 1..6 qubits (`get_dens_op` / `get_dens_op_with_grad`).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

`kdensity` / `kgate` generalise `statevector.q{1,2}density` / `q{1,2}gate` to k qubits with reshape / einsum, and
`KOracleCircuit` is the VM of `oracle.circuit.OracleCircuit` with the two extra builders.  Index convention of the
product (include/qdc_circuit.h, qdc_circuit_add_dens): positions = [p_{k-1}, ..., p_0], positions[0] the most
significant bit of the row and column index, so `kdensity(s, [p2, p1])` is `q2density(s, p2, p1)`.  k <= 2 adds the
existing instruction kinds; k >= 3 adds (DENS_K | DIFF_DENS_K, positions tuple).  The backward seed is the k-qubit
form of the reference's: bwd (+)= (G^T on positions)(2 conj fwd).
"""
from __future__ import annotations

from collections import deque

import numpy as np

from . import statevector as sv
from .circuit import (_DIAG_GATES, _NONU, _Q1_GATES, _Q2_GATES, _VAR, DIFF_Q1_DENS, DIFF_Q2_DENS, Q1_DENS, Q2_DENS,
                      OracleCircuit)

DENS_K, DIFF_DENS_K = 14, 15


def _front(state: np.ndarray, positions) -> np.ndarray:
    """The state as a (2^k, 2^(n-k)) matrix: row index over `positions` (positions[0] most significant), column
    index over the other qubits in their original order."""
    n = sv.qubits_of(state)
    axes = [n - 1 - p for p in positions]            # qubit p is tensor axis n-1-p of the C-order (2,)*n view
    rest = [a for a in range(n) if a not in axes]
    return np.transpose(state.reshape((2,) * n), axes + rest).reshape(1 << len(positions), -1)


def kdensity(state: np.ndarray, positions) -> np.ndarray:
    """rho[r, c] = sum_rest psi[r, rest] conj psi[c, rest] over the qubits `positions`; shape (2^k, 2^k)."""
    assert len(set(positions)) == len(positions)
    a = _front(state, positions)
    return np.einsum("rj,cj->rc", a, a.conj())


def kgate(state: np.ndarray, matrix, positions) -> np.ndarray:
    """psi'[r, rest] = sum_c M[r, c] psi[c, rest] on the qubits `positions` (index convention of kdensity)."""
    assert len(set(positions)) == len(positions)
    n, k = sv.qubits_of(state), len(positions)
    m = np.asarray(matrix, dtype=state.dtype).reshape(1 << k, 1 << k)
    out = np.einsum("rc,cj->rj", m, _front(state, positions))
    axes = [n - 1 - p for p in positions]
    rest = [a for a in range(n) if a not in axes]
    return np.transpose(out.reshape((2,) * n), np.argsort(axes + rest)).reshape(-1)


class KOracleCircuit(OracleCircuit):
    """OracleCircuit with densities on 1..6 qubits."""

    def get_dens_op(self, positions): self._add_dens(positions, False)
    def get_dens_op_with_grad(self, positions): self._add_dens(positions, True)

    def _add_dens(self, positions, with_grad):
        pos = [int(p) for p in positions]
        if not 1 <= len(pos) <= 6:
            raise ValueError("the number of density qubits must be in 1..6.")
        if any(p < 0 or p >= self.n for p in pos):
            raise ValueError("pos is out of the bound.")
        if len(set(pos)) != len(pos):
            raise ValueError("positions must be different.")
        if len(pos) == 1:
            self.instructions.append((DIFF_Q1_DENS if with_grad else Q1_DENS, pos[0]))
        elif len(pos) == 2:
            self.instructions.append((DIFF_Q2_DENS if with_grad else Q2_DENS, pos[0], pos[1]))
        else:
            self.instructions.append((DIFF_DENS_K if with_grad else DENS_K, tuple(pos)))

    # ---- forward interpreter: OracleCircuit._sweep plus the k-qubit densities ----
    def _sweep(self, const_gates, var_gates, all_densities: bool):
        assert self.instructions, "The circuit is empty."
        out = []
        cq = deque(np.asarray(g, dtype=self.dtype).reshape(-1) for g in const_gates)
        vq = deque(np.asarray(g, dtype=self.dtype).reshape(-1) for g in var_gates)
        self.state = self.initial_state.copy()
        for inst in self.instructions:
            kind = inst[0]
            if kind in _Q1_GATES or kind in _Q2_GATES or kind in _DIAG_GATES:
                q = vq if kind in _VAR else cq
                if not q:
                    raise ValueError("The number of %s gates is less than required."
                                     % ("variable" if kind in _VAR else "constant"))
                gate = q.popleft()
                if kind in _Q1_GATES:
                    self.state = sv.q1gate(self.state, gate, inst[1])
                elif kind in _Q2_GATES:
                    self.state = sv.q2gate(self.state, gate, inst[1], inst[2])
                else:
                    self.state = sv.q2gate_diag(self.state, gate, inst[1], inst[2])
            elif kind in (DENS_K, DIFF_DENS_K):
                if all_densities or kind == DIFF_DENS_K:
                    out.append(kdensity(self.state, inst[1]))
            elif kind in (Q1_DENS, DIFF_Q1_DENS):
                if all_densities or kind == DIFF_Q1_DENS:
                    out.append(sv.q1density(self.state, inst[1]).reshape(2, 2))
            elif all_densities or kind == DIFF_Q2_DENS:
                out.append(sv.q2density(self.state, inst[1], inst[2]).reshape(4, 4))
        if cq:
            raise ValueError("Number of constant gates is more than required.")
        if vq:
            raise ValueError("Number of variable gates is more than required.")
        return out

    # ---- reverse interpreter: OracleCircuit.backward plus the k-qubit seeds ----
    def backward(self, grads_wrt_density, const_gates, var_gates):
        assert self.instructions, "The circuit is empty."
        gd = [np.asarray(g, dtype=self.dtype).reshape(-1) for g in grads_wrt_density]
        cg = [np.asarray(g, dtype=self.dtype).reshape(-1) for g in const_gates]
        vg = [np.asarray(g, dtype=self.dtype).reshape(-1) for g in var_gates]
        fwd, bwd = self.state, None
        grads = deque()
        for inst in reversed(self.instructions):
            kind = inst[0]
            if kind in (Q1_DENS, Q2_DENS, DENS_K):
                continue
            if kind in (DIFF_Q1_DENS, DIFF_Q2_DENS, DIFF_DENS_K):
                if not gd:
                    raise ValueError("The number of gradients wrt density matrices is less than required.")
                g = gd.pop()
                add = sv.conj_and_double(fwd)
                if kind == DIFF_Q1_DENS:
                    add = sv.q1gate(add, sv.q1_tr(g), inst[1])
                elif kind == DIFF_Q2_DENS:
                    add = sv.q2gate(add, sv.q2_tr(g), inst[1], inst[2])
                else:
                    d = 1 << len(inst[1])
                    add = kgate(add, g.reshape(d, d).T, inst[1])
                bwd = add if bwd is None else sv.add(add, bwd)
                continue
            is_var = kind in _VAR
            lst = vg if is_var else cg
            if not lst:
                raise ValueError("The number of gates is less than required.")
            gate = lst.pop()
            if kind in _Q1_GATES:
                pos = inst[1]
                fwd = sv.q1gate_inv(fwd, gate, pos) if kind in _NONU else sv.q1gate(fwd, sv.q1_conj_tr(gate), pos)
                if bwd is not None:
                    if is_var:
                        grads.appendleft(sv.q1grad(fwd, bwd, pos))
                    bwd = sv.q1gate(bwd, sv.q1_tr(gate), pos)
                elif is_var:
                    grads.appendleft(np.zeros(4, dtype=self.dtype))
            elif kind in _Q2_GATES:
                p2, p1 = inst[1], inst[2]
                fwd = (sv.q2gate_inv(fwd, gate, p2, p1) if kind in _NONU
                       else sv.q2gate(fwd, sv.q2_conj_tr(gate), p2, p1))
                if bwd is not None:
                    if is_var:
                        grads.appendleft(sv.q2grad(fwd, bwd, p2, p1))
                    bwd = sv.q2gate(bwd, sv.q2_tr(gate), p2, p1)
                elif is_var:
                    grads.appendleft(np.zeros(16, dtype=self.dtype))
            else:  # diagonal
                p2, p1 = inst[1], inst[2]
                fwd = sv.q2gate_diag(fwd, gate.conj(), p2, p1)
                if bwd is not None:
                    if is_var:
                        grads.appendleft(sv.q2grad_diag(fwd, bwd, p2, p1))
                    bwd = sv.q2gate_diag(bwd, gate, p2, p1)
                elif is_var:
                    grads.appendleft(np.zeros(4, dtype=self.dtype))
        self.state = fwd
        if cg or vg:
            raise ValueError("Number of constant gates is more than required.")
        if gd:
            raise ValueError("Number of gradients wrt density matrices is more than required.")
        return [np.asarray(g, dtype=self.dtype) for g in grads]

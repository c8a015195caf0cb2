"""Oracle of the diagonal gates on k = 1..6 qubits (`add_const_gate_diag` / `add_var_gate_diag` / `*_nonu`).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

`KDiagOracleCircuit` is the VM of `oracle.kgates.KGateOracleCircuit` with the four diagonal builders.  Index convention
(include/qdc_circuit.h, qdc_circuit_add_gate_diag): positions = [p_{k-1}, ..., p_0], positions[0] the most significant
bit of j, so the forward pass `kdiag(state, d, positions)` equals `kgate(state, diag(d), positions)` and a diagonal on
[p2, p1] is `q2gate_diag(s, d, p2, p1)`.  A unitary diagonal on k = 2 adds the existing Q2_DIAG kinds; every other
case adds (kind, positions tuple).  The reverse step is the two-qubit diagonal's at width k: un-compute with conj(d)
(1 / d for NonU), the gradient `kdiag_grad` (no conjugation) from the un-computed state and the adjoint, then pull the
adjoint back with d.
"""
from __future__ import annotations

from collections import deque

import numpy as np

from . import statevector as sv
from .circuit import _DIAG_GATES, _NONU, _Q1_GATES, _Q2_GATES, _VAR, DIFF_Q1_DENS, DIFF_Q2_DENS, Q1_DENS, Q2_DENS
from .kdens import DENS_K, DIFF_DENS_K, _front, kdensity, kgate
from .kgates import _K_GATES, _K_NONU, _K_VAR, KGateOracleCircuit, kgrad

CONST_GATE_K_DIAG, VAR_GATE_K_DIAG, CONST_GATE_K_DIAG_NONU, VAR_GATE_K_DIAG_NONU = 20, 21, 22, 23
_K_DIAG = (CONST_GATE_K_DIAG, VAR_GATE_K_DIAG, CONST_GATE_K_DIAG_NONU, VAR_GATE_K_DIAG_NONU)
_KD_VAR = (VAR_GATE_K_DIAG, VAR_GATE_K_DIAG_NONU)
_KD_NONU = (CONST_GATE_K_DIAG_NONU, VAR_GATE_K_DIAG_NONU)


def _index(n: int, positions) -> np.ndarray:
    """j of every amplitude index: the bits at `positions`, positions[0] the most significant."""
    idx = np.arange(1 << n)
    j = np.zeros(1 << n, dtype=np.int64)
    for p in positions:
        j = (j << 1) | ((idx >> p) & 1)
    return j


def kdiag(state: np.ndarray, d, positions) -> np.ndarray:
    """psi'[j, rest] = d[j] psi[j, rest]; `kgate(state, np.diag(d), positions)` without the dense product."""
    assert len(set(positions)) == len(positions)
    d = np.asarray(d, dtype=state.dtype).reshape(-1)
    assert d.size == 1 << len(positions)
    return state * d[_index(sv.qubits_of(state), positions)]


def kdiag_grad(fwd: np.ndarray, bwd: np.ndarray, positions) -> np.ndarray:
    """G[j] = sum_rest bwd[j, rest] fwd[j, rest] (no conjugation), flat (2^k): the diagonal of `kgrad`."""
    assert len(set(positions)) == len(positions)
    return np.sum(_front(bwd, positions) * _front(fwd, positions), axis=1)


def _inverse(d: np.ndarray) -> np.ndarray:
    zero = np.flatnonzero(d == 0)
    if zero.size:
        raise ValueError("U(%d, %d) is zero." % (zero[0] + 1, zero[0] + 1))
    return 1 / d


class KDiagOracleCircuit(KGateOracleCircuit):
    """KGateOracleCircuit with diagonal gates on 1..6 qubits."""

    def add_const_gate_diag(self, positions): self._add_gate_diag(positions, False, False)
    def add_var_gate_diag(self, positions): self._add_gate_diag(positions, True, False)
    def add_const_gate_diag_nonu(self, positions): self._add_gate_diag(positions, False, True)
    def add_var_gate_diag_nonu(self, positions): self._add_gate_diag(positions, True, True)

    def _add_gate_diag(self, positions, variable, non_unitary):
        pos = [int(p) for p in positions]
        if not 1 <= len(pos) <= 6:
            raise ValueError("the number of gate qubits must be in 1..6.")
        if any(p < 0 or p >= self.n for p in pos):
            raise ValueError("pos is out of the bound.")
        if len(set(pos)) != len(pos):
            raise ValueError("positions must be different.")
        if len(pos) == 2 and not non_unitary:
            (self.add_q2_var_gate_diag if variable else self.add_q2_const_gate_diag)(pos[0], pos[1])
            return
        kind = {(False, False): CONST_GATE_K_DIAG, (True, False): VAR_GATE_K_DIAG,
                (False, True): CONST_GATE_K_DIAG_NONU, (True, True): VAR_GATE_K_DIAG_NONU}[(variable, non_unitary)]
        self.instructions.append((kind, tuple(pos)))

    # ---- forward interpreter: KGateOracleCircuit._sweep plus the diagonal k-qubit gates ----
    def _sweep(self, const_gates, var_gates, all_densities: bool):
        assert self.instructions, "The circuit is empty."
        out = []
        cq = deque(np.asarray(g, dtype=self.dtype).reshape(-1) for g in const_gates)
        vq = deque(np.asarray(g, dtype=self.dtype).reshape(-1) for g in var_gates)
        self.state = self.initial_state.copy()
        for inst in self.instructions:
            kind = inst[0]
            if kind in _Q1_GATES or kind in _Q2_GATES or kind in _DIAG_GATES or kind in _K_GATES or kind in _K_DIAG:
                var = kind in _VAR or kind in _K_VAR or kind in _KD_VAR
                q = vq if var else cq
                if not q:
                    raise ValueError("The number of %s gates is less than required." % ("variable" if var else "constant"))
                gate = q.popleft()
                if kind in _Q1_GATES:
                    self.state = sv.q1gate(self.state, gate, inst[1])
                elif kind in _Q2_GATES:
                    self.state = sv.q2gate(self.state, gate, inst[1], inst[2])
                elif kind in _DIAG_GATES:
                    self.state = sv.q2gate_diag(self.state, gate, inst[1], inst[2])
                elif kind in _K_DIAG:
                    if gate.size != 2 ** len(inst[1]):
                        raise ValueError("Incorrect len of the gate's buffer.")
                    self.state = kdiag(self.state, gate, inst[1])
                else:
                    if gate.size != 4 ** len(inst[1]):
                        raise ValueError("Incorrect len of the gate's buffer.")
                    self.state = kgate(self.state, gate, inst[1])
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

    # ---- reverse interpreter: KGateOracleCircuit.backward plus the diagonal k-qubit gates ----
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
            is_var = kind in _VAR or kind in _K_VAR or kind in _KD_VAR
            lst = vg if is_var else cg
            if not lst:
                raise ValueError("The number of gates is less than required.")
            gate = lst.pop()
            if kind in _K_DIAG:
                pos = inst[1]
                fwd = kdiag(fwd, _inverse(gate) if kind in _KD_NONU else gate.conj(), pos)
                if bwd is not None:
                    if is_var:
                        grads.appendleft(kdiag_grad(fwd, bwd, pos))
                    bwd = kdiag(bwd, gate, pos)
                elif is_var:
                    grads.appendleft(np.zeros(gate.size, dtype=self.dtype))
            elif kind in _K_GATES:
                pos = inst[1]
                d = 1 << len(pos)
                u = gate.reshape(d, d)
                fwd = kgate(fwd, sv.inverse(gate, d).reshape(d, d) if kind in _K_NONU else u.conj().T, pos)
                if bwd is not None:
                    if is_var:
                        grads.appendleft(kgrad(fwd, bwd, pos))
                    bwd = kgate(bwd, u.T, pos)
                elif is_var:
                    grads.appendleft(np.zeros(d * d, dtype=self.dtype))
            elif kind in _Q1_GATES:
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
            else:  # two-qubit diagonal
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

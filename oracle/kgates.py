"""Oracle of the gates on k = 1..6 qubits (`add_const_gate` / `add_var_gate` / `*_nonu`).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

`KGateOracleCircuit` is the VM of `oracle.kdens.KOracleCircuit` with the four gate builders.  Index convention of the
product (include/qdc_circuit.h, qdc_circuit_add_gate): positions = [p_{k-1}, ..., p_0], positions[0] the most
significant bit of the row and column index, so the forward pass is `kdens.kgate` and a gate on [p2, p1] is
`q2gate(s, U, p2, p1)`.  k <= 2 adds the existing instruction kinds; k >= 3 adds (kind, positions tuple).  The reverse
step is the reference's at width k: un-compute with U^dagger (U^-1 for NonU, `sv.inverse`), the gradient `kgrad`
(q2grad at width k: no conjugation) from the un-computed state and the adjoint, then pull the adjoint back with U^T.
"""
from __future__ import annotations

from collections import deque

import numpy as np

from . import statevector as sv
from .circuit import _DIAG_GATES, _NONU, _Q1_GATES, _Q2_GATES, _VAR, DIFF_Q1_DENS, DIFF_Q2_DENS, Q1_DENS, Q2_DENS
from .kdens import DENS_K, DIFF_DENS_K, KOracleCircuit, _front, kdensity, kgate

CONST_GATE_K, VAR_GATE_K, CONST_GATE_K_NONU, VAR_GATE_K_NONU = 16, 17, 18, 19
_K_GATES = (CONST_GATE_K, VAR_GATE_K, CONST_GATE_K_NONU, VAR_GATE_K_NONU)
_K_VAR = (VAR_GATE_K, VAR_GATE_K_NONU)
_K_NONU = (CONST_GATE_K_NONU, VAR_GATE_K_NONU)


def kgrad(fwd: np.ndarray, bwd: np.ndarray, positions) -> np.ndarray:
    """G[r, c] = sum_rest bwd[r, rest] fwd[c, rest] (no conjugation), flat (4^k); `q1grad` / `q2grad` for k <= 2."""
    assert len(set(positions)) == len(positions)
    return np.einsum("rj,cj->rc", _front(bwd, positions), _front(fwd, positions)).reshape(-1)


class KGateOracleCircuit(KOracleCircuit):
    """KOracleCircuit with gates on 1..6 qubits."""

    def add_const_gate(self, positions): self._add_gate(positions, False, False)
    def add_var_gate(self, positions): self._add_gate(positions, True, False)
    def add_const_gate_nonu(self, positions): self._add_gate(positions, False, True)
    def add_var_gate_nonu(self, positions): self._add_gate(positions, True, True)

    def _add_gate(self, positions, variable, non_unitary):
        pos = [int(p) for p in positions]
        if not 1 <= len(pos) <= 6:
            raise ValueError("the number of gate qubits must be in 1..6.")
        if any(p < 0 or p >= self.n for p in pos):
            raise ValueError("pos is out of the bound.")
        if len(set(pos)) != len(pos):
            raise ValueError("positions must be different.")
        name = "%s_gate%s" % ("var" if variable else "const", "_nonu" if non_unitary else "")
        if len(pos) == 1:
            getattr(self, "add_q1_" + name)(pos[0])
        elif len(pos) == 2:
            getattr(self, "add_q2_" + name)(pos[0], pos[1])
        else:
            kind = {(False, False): CONST_GATE_K, (True, False): VAR_GATE_K, (False, True): CONST_GATE_K_NONU,
                    (True, True): VAR_GATE_K_NONU}[(variable, non_unitary)]
            self.instructions.append((kind, tuple(pos)))

    # ---- forward interpreter: KOracleCircuit._sweep plus the k-qubit gates ----
    def _sweep(self, const_gates, var_gates, all_densities: bool):
        assert self.instructions, "The circuit is empty."
        out = []
        cq = deque(np.asarray(g, dtype=self.dtype).reshape(-1) for g in const_gates)
        vq = deque(np.asarray(g, dtype=self.dtype).reshape(-1) for g in var_gates)
        self.state = self.initial_state.copy()
        for inst in self.instructions:
            kind = inst[0]
            if kind in _Q1_GATES or kind in _Q2_GATES or kind in _DIAG_GATES or kind in _K_GATES:
                var = kind in _VAR or kind in _K_VAR
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

    # ---- reverse interpreter: KOracleCircuit.backward plus the k-qubit gates ----
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
            is_var = kind in _VAR or kind in _K_VAR
            lst = vg if is_var else cg
            if not lst:
                raise ValueError("The number of gates is less than required.")
            gate = lst.pop()
            if kind in _K_GATES:
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

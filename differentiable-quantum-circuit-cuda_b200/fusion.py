"""`FusedCircuit`: gate fusion in front of the executor.

Same surface as `quantum_differentiable_circuit.Circuit` (the drop-in for the reference's Rust
`Circuit`, /root/reference/src/circuit.rs:93-430).  Consecutive gates that act inside the same one or
two qubits are multiplied into ONE gate before the program reaches the GPU, and the gradient of the
fused gate is chained back to its members on the host:

    U = M_k ... M_1                      (members embedded into the fused gate's 4x4 / 2x2 space)
    dL/dM_j = A_j^T  (dL/dU)  B_j^T,     A_j = M_k ... M_{j+1},   B_j = M_{j-1} ... M_1

(the reference's gradient convention is holomorphic, dL = Re sum g * dU with no conjugation on the gate
path, SURVEY.md App. A, so the chain rule is the plain matrix one), followed by the projection onto the
member's own shape (a one-qubit gate g embedded as g (x) 1 gets dL/dg[p,q] = sum_r dL/dM[(p,r),(q,r)];
a diagonal gate gets the diagonal).

Why: on the GPU a cheap gate costs almost as much as a dense one (shared-memory round trip of the tile,
gradient reduction, barrier: 0.11 / 0.14 / 0.19 ms per reverse step of a one-qubit / diagonal / dense
two-qubit gate at 26 qubits, profiles/r1_gate_kind_bench_after_diag_fix.txt).  The VQSE ansatz of
example_vqse_ising.py (ZZ ring + X rotations) halves its gate count: n dense gates per layer instead
of n diagonal + n one-qubit gates.

Fusion rules (program order is preserved wherever two gates share a qubit):
  * a one-qubit gate joins the last gate that touched its qubit, if that gate is still "open";
  * a two-qubit gate joins the last gate on BOTH its qubits if that is one and the same two-qubit gate;
    otherwise it starts a new fused gate and absorbs the still-open ONE-qubit gates of its two qubits;
  * every density instruction closes all gates (it must see the state of its program point);
  * a gate on 3..6 qubits (`add_const_gate(positions)` and friends) is a barrier like a density: it closes all
    gates and runs unfused, its matrix and gradient pass through unchanged;
  * diagonal gates are taken as unitary (the reference's un-compute multiplies by conj(d),
    src/quantized_tensor.rs:153-156): a fused gate is NonU iff one of its members is.

The host algebra is batched with NumPy over all fused gates of the same member pattern, so its cost is
milliseconds per call.  Opt-in: `FusedCircuit(n)` instead of `Circuit(n)`.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Sequence

import numpy as np

from .quantum_differentiable_circuit import (CONST_GATE_K, CONST_GATE_K_DIAG, CONST_GATE_K_DIAG_NONU,
                                             CONST_GATE_K_NONU, CONST_Q1, CONST_Q1_NONU, CONST_Q2, CONST_Q2_DIAG,
                                             CONST_Q2_NONU, DENS_K, DIFF_DENS_K, DIFF_Q1_DENS, DIFF_Q2_DENS, Q1_DENS,
                                             Q2_DENS, VAR_GATE_K, VAR_GATE_K_DIAG, VAR_GATE_K_DIAG_NONU,
                                             VAR_GATE_K_NONU, VAR_Q1, VAR_Q1_NONU, VAR_Q2, VAR_Q2_DIAG, VAR_Q2_NONU,
                                             Circuit)

_Q1 = (CONST_Q1, CONST_Q1_NONU, VAR_Q1, VAR_Q1_NONU)
_Q2D = (CONST_Q2, VAR_Q2, CONST_Q2_NONU, VAR_Q2_NONU)
_DIAG = (CONST_Q2_DIAG, VAR_Q2_DIAG)
_KDIAG = (CONST_GATE_K_DIAG, VAR_GATE_K_DIAG, CONST_GATE_K_DIAG_NONU, VAR_GATE_K_DIAG_NONU)
_KGATE = (CONST_GATE_K, VAR_GATE_K, CONST_GATE_K_NONU, VAR_GATE_K_NONU) + _KDIAG   # unfused barriers
_VAR = (VAR_Q2, VAR_Q2_NONU, VAR_Q2_DIAG, VAR_Q1, VAR_Q1_NONU, VAR_GATE_K, VAR_GATE_K_NONU, VAR_GATE_K_DIAG,
        VAR_GATE_K_DIAG_NONU)
_NONU = (CONST_Q2_NONU, VAR_Q2_NONU, CONST_Q1_NONU, VAR_Q1_NONU)
_DENS = (Q2_DENS, Q1_DENS, DIFF_Q2_DENS, DIFF_Q1_DENS, DENS_K, DIFF_DENS_K)
_SWAP = np.array([0, 2, 1, 3])  # index 2 b_hi + b_lo with the two bits exchanged

# how a member sits inside its fused gate
E_SAME, E_SWAPPED, E_DIAG, E_DIAG_SWAPPED, E_Q1_ON_2, E_Q1_ON_1, E_Q1 = range(7)


class _XGate:
    __slots__ = ("pos2", "pos1", "members", "alive")

    def __init__(self, pos2, pos1):
        self.pos2, self.pos1 = pos2, pos1  # pos1 < 0: one-qubit fused gate
        self.members = []                  # (instruction index, embedding)
        self.alive = True

    @property
    def support(self):
        return (self.pos2,) if self.pos1 < 0 else (self.pos2, self.pos1)


def plan_fusion(program: Sequence[tuple]):
    """program: [(kind, pos2[, pos1])] -> execution list of ('gate', _XGate) / ('dens' | 'kgate', instruction index)."""
    out: List[tuple] = []
    open_gate: Dict[int, _XGate] = {}
    for idx, inst in enumerate(program):
        kind, p2 = inst[0], inst[1]
        if kind in _DENS or kind in _KGATE:
            out.append(("dens" if kind in _DENS else "kgate", idx))
            open_gate.clear()
            continue
        if kind in _Q1:
            g = open_gate.get(p2)
            if g is None:
                g = _XGate(p2, -1)
                out.append(("gate", g))
                open_gate[p2] = g
                g.members.append((idx, E_Q1))
            elif g.pos1 < 0:
                g.members.append((idx, E_Q1))
            else:
                g.members.append((idx, E_Q1_ON_2 if g.pos2 == p2 else E_Q1_ON_1))
            continue
        p1 = inst[2]
        ga, gb = open_gate.get(p2), open_gate.get(p1)
        diag = kind in _DIAG
        if ga is not None and ga is gb and set(ga.support) == {p2, p1}:
            same = ga.pos2 == p2
            ga.members.append((idx, (E_DIAG if same else E_DIAG_SWAPPED) if diag else (E_SAME if same else E_SWAPPED)))
            continue
        g = _XGate(p2, p1)
        for q, emb in ((p2, E_Q1_ON_2), (p1, E_Q1_ON_1)):  # absorb still-open one-qubit gates
            h = open_gate.get(q)
            if h is not None and h.pos1 < 0:
                g.members += [(i, emb) for i, _ in h.members]
                h.alive = False
        g.members.append((idx, E_DIAG if diag else E_SAME))
        out.append(("gate", g))
        open_gate[p2] = open_gate[p1] = g
    return [(t, x) for t, x in out if t != "gate" or x.alive]


def _fused_kind(g: _XGate, program) -> int:
    kinds = [program[i][0] for i, _ in g.members]
    var = any(k in _VAR for k in kinds)
    nonu = any(k in _NONU for k in kinds)
    if g.pos1 < 0:
        return (VAR_Q1_NONU if nonu else VAR_Q1) if var else (CONST_Q1_NONU if nonu else CONST_Q1)
    if all(k in _DIAG for k in kinds):
        return VAR_Q2_DIAG if var else CONST_Q2_DIAG
    return (VAR_Q2_NONU if nonu else VAR_Q2) if var else (CONST_Q2_NONU if nonu else CONST_Q2)


def _embed(mats: np.ndarray, emb: int) -> np.ndarray:
    """Batch of member matrices (flat, as the API takes them) -> batch of matrices in the fused gate's space
    (4x4 with index 2 bit(pos2) + bit(pos1), 2x2 for a one-qubit fused gate, or a 4-vector for all-diagonal)."""
    b = mats.shape[0]
    if emb == E_Q1:
        return mats.reshape(b, 2, 2)
    if emb == E_SAME:
        return mats.reshape(b, 4, 4)
    if emb == E_SWAPPED:
        return mats.reshape(b, 4, 4)[:, _SWAP][:, :, _SWAP]
    eye = np.eye(2, dtype=mats.dtype)
    if emb == E_Q1_ON_2:
        return np.einsum("bpq,rs->bprqs", mats.reshape(b, 2, 2), eye).reshape(b, 4, 4)
    if emb == E_Q1_ON_1:
        return np.einsum("rs,bpq->brpsq", eye, mats.reshape(b, 2, 2)).reshape(b, 4, 4)
    d = mats.reshape(b, 4) if emb == E_DIAG else mats.reshape(b, 4)[:, _SWAP]
    out = np.zeros((b, 4, 4), dtype=mats.dtype)
    out[:, np.arange(4), np.arange(4)] = d
    return out


def _project(gm: np.ndarray, emb: int) -> np.ndarray:
    """Batch of dL/dM in the fused space -> flat gradients in the member's own shape."""
    b = gm.shape[0]
    if emb == E_Q1:
        return gm.reshape(b, 4)
    if emb == E_SAME:
        return gm.reshape(b, 16)
    if emb == E_SWAPPED:
        return gm[:, _SWAP][:, :, _SWAP].reshape(b, 16)
    if emb == E_Q1_ON_2:
        return np.einsum("bprqr->bpq", gm.reshape(b, 2, 2, 2, 2)).reshape(b, 4)
    if emb == E_Q1_ON_1:
        return np.einsum("brprq->bpq", gm.reshape(b, 2, 2, 2, 2)).reshape(b, 4)
    d = gm[:, np.arange(4), np.arange(4)]
    return d if emb == E_DIAG else d[:, _SWAP]


class FusedCircuit(Circuit):
    """Drop-in `Circuit` with gate fusion (see the module docstring).  `backend` is a factory of the circuit that
    executes the fused program (default: the CUDA `Circuit` of this package); the CPU suite passes the oracle."""

    def __init__(self, qubits_number: int, precision: str | None = None, backend: Callable | None = None):
        self.qubits_number = int(qubits_number)
        self._precision = precision
        self._backend = backend or (lambda n: Circuit(n, precision=precision))
        self._program: List[tuple] = []
        self._kinds: List[int] = []
        self._inner = None
        self._options: List[tuple] = []
        self._initial = None

    # the builders of Circuit funnel through _add
    def _add(self, kind, pos2, pos1=0):
        n = self.qubits_number
        if pos2 < 0 or pos1 < 0:
            raise OverflowError("can't convert negative int to unsigned")
        one = kind in _Q1 or kind in (Q1_DENS, DIFF_Q1_DENS)
        if pos2 >= n or (not one and pos1 >= n):
            raise ValueError("position out of the bound")
        if not one and pos1 == pos2:
            raise ValueError("pos1 and pos2 must be different.")
        self._program.append((kind, pos2) if one else (kind, pos2, pos1))
        self._kinds.append(kind)
        self._inner = None

    def _add_dens_k(self, positions, with_grad):
        if any(p < 0 for p in positions):
            raise OverflowError("can't convert negative int to unsigned")
        if not 1 <= len(positions) <= 6:
            raise ValueError("the number of density qubits must be in 1..6.")
        if any(p >= self.qubits_number for p in positions):
            raise ValueError("pos is out of the bound.")
        if len(set(positions)) != len(positions):
            raise ValueError("positions must be different.")
        kind = DIFF_DENS_K if with_grad else DENS_K
        self._program.append((kind, tuple(positions)))   # a barrier like every density (plan_fusion)
        self._kinds.append(kind)
        self._inner = None

    def _add_gate_k(self, positions, variable, non_unitary):
        if any(p < 0 for p in positions):
            raise OverflowError("can't convert negative int to unsigned")
        if not 1 <= len(positions) <= 6:
            raise ValueError("the number of gate qubits must be in 1..6.")
        if any(p >= self.qubits_number for p in positions):
            raise ValueError("pos is out of the bound.")
        if len(set(positions)) != len(positions):
            raise ValueError("positions must be different.")
        kind = (VAR_GATE_K if variable else CONST_GATE_K) if not non_unitary else \
            (VAR_GATE_K_NONU if variable else CONST_GATE_K_NONU)
        self._program.append((kind, tuple(positions)))   # a barrier, executed unfused (plan_fusion)
        self._kinds.append(kind)
        self._inner = None

    def _add_gate_diag_k(self, positions, variable, non_unitary):
        if any(p < 0 for p in positions):
            raise OverflowError("can't convert negative int to unsigned")
        if not 1 <= len(positions) <= 6:
            raise ValueError("the number of gate qubits must be in 1..6.")
        if any(p >= self.qubits_number for p in positions):
            raise ValueError("pos is out of the bound.")
        if len(set(positions)) != len(positions):
            raise ValueError("positions must be different.")
        kind = (VAR_GATE_K_DIAG if variable else CONST_GATE_K_DIAG) if not non_unitary else \
            (VAR_GATE_K_DIAG_NONU if variable else CONST_GATE_K_DIAG_NONU)
        self._program.append((kind, tuple(positions)))   # a barrier, executed unfused like the k-qubit gates
        self._kinds.append(kind)
        self._inner = None

    def __del__(self):
        pass

    @property
    def dtype(self):
        return self._build().dtype if hasattr(self._build(), "dtype") else np.dtype(np.complex128)

    def set_state_from_vector(self, vector):
        self._initial = np.asarray(vector)
        if self._inner is not None:
            self._inner.set_state_from_vector(self._initial)

    def set_option(self, key: str, value: int):
        self._options.append((key, int(value)))
        if self._inner is not None and hasattr(self._inner, "set_option"):
            self._inner.set_option(key, int(value))

    # statistics / state access / I/O act on the circuit that executes the fused program (built on demand)
    def last_stats(self):
        return self._build().last_stats()

    def last_profile(self):
        return self._build().last_profile()

    def get_cpu_state_copy(self):
        return self._build().get_cpu_state_copy()

    def save_state(self, path: str):
        return self._build().save_state(path)

    def load_state(self, path: str):
        return self._build().load_state(path)

    def state_layout(self):
        return self._build().state_layout()

    def set_stream(self, cuda_stream):
        return self._build().set_stream(cuda_stream)

    def _count(self, what):
        """Counts of the USER's program (not of the fused one), like Circuit._count."""
        def dens_len(inst):
            k = inst[0]
            return 4 ** len(inst[1]) if k in (DENS_K, DIFF_DENS_K) else 4 if k in (Q1_DENS, DIFF_Q1_DENS) else 16
        def gate_len(inst):
            k = inst[0]
            if k in _KDIAG:
                return 2 ** len(inst[1])
            return 4 ** len(inst[1]) if k in _KGATE else 16 if k in (CONST_Q2, VAR_Q2, CONST_Q2_NONU, VAR_Q2_NONU) else 4
        ks, prog = self._kinds, self._program
        diff = (DIFF_Q1_DENS, DIFF_Q2_DENS, DIFF_DENS_K)
        return [len(ks), sum(k not in _DENS and k not in _VAR for k in ks), sum(k in _VAR for k in ks),
                sum(k in _DENS for k in ks), sum(k in diff for k in ks), sum(dens_len(i) for i in prog if i[0] in _DENS),
                sum(dens_len(i) for i in prog if i[0] in diff), sum(gate_len(i) for i in prog if i[0] in _VAR)][what]

    @property
    def fused_gate_count(self) -> int:
        self._build()
        return len(self._xgates)

    # ---- the fused program ----
    def _build(self):
        if self._inner is not None:
            return self._inner
        prog = self._program
        self._exec = plan_fusion(prog)
        self._xgates = [x for t, x in self._exec if t == "gate"]
        inner = self._backend(self.qubits_number)
        if hasattr(inner, "set_option"):
            for k, v in self._options:
                inner.set_option(k, v)
        if self._initial is not None:
            inner.set_state_from_vector(self._initial)
        adders = {CONST_Q2: "add_q2_const_gate", VAR_Q2: "add_q2_var_gate", CONST_Q2_NONU: "add_q2_const_gate_nonu",
                  VAR_Q2_NONU: "add_q2_var_gate_nonu", CONST_Q2_DIAG: "add_q2_const_gate_diag",
                  VAR_Q2_DIAG: "add_q2_var_gate_diag", CONST_Q1: "add_q1_const_gate",
                  CONST_Q1_NONU: "add_q1_const_gate_nonu", VAR_Q1: "add_q1_var_gate", VAR_Q1_NONU: "add_q1_var_gate_nonu",
                  Q2_DENS: "get_q2_dens_op", Q1_DENS: "get_q1_dens_op", DIFF_Q2_DENS: "get_q2_dens_op_with_grad",
                  DIFF_Q1_DENS: "get_q1_dens_op_with_grad", DENS_K: "get_dens_op", DIFF_DENS_K: "get_dens_op_with_grad",
                  CONST_GATE_K: "add_const_gate", VAR_GATE_K: "add_var_gate", CONST_GATE_K_NONU: "add_const_gate_nonu",
                  VAR_GATE_K_NONU: "add_var_gate_nonu", CONST_GATE_K_DIAG: "add_const_gate_diag",
                  VAR_GATE_K_DIAG: "add_var_gate_diag", CONST_GATE_K_DIAG_NONU: "add_const_gate_diag_nonu",
                  VAR_GATE_K_DIAG_NONU: "add_var_gate_diag_nonu"}
        self._xkinds = []
        for t, x in self._exec:
            if t == "kgate":
                getattr(inner, adders[prog[x][0]])(list(prog[x][1]))
            elif t == "dens":
                inst = prog[x]
                if inst[0] in (DENS_K, DIFF_DENS_K):
                    getattr(inner, adders[inst[0]])(list(inst[1]))
                else:
                    getattr(inner, adders[inst[0]])(*inst[1:])
            else:
                k = _fused_kind(x, prog)
                self._xkinds.append(k)
                getattr(inner, adders[k])(*((x.pos2,) if x.pos1 < 0 else (x.pos2, x.pos1)))
        # where each program gate finds its matrix in the (const, var) lists of a call
        self._src = {}
        ci = vi = 0
        for idx, inst in enumerate(prog):
            if inst[0] in _DENS:
                continue
            if inst[0] in _VAR:
                self._src[idx] = (1, vi); vi += 1
            else:
                self._src[idx] = (0, ci); ci += 1
        self._n_const, self._n_var = ci, vi
        # batches: fused gates with the same member pattern are multiplied / differentiated together
        self._batches = {}
        for gi, x in enumerate(self._xgates):
            sig = (x.pos1 < 0, self._xkinds[gi] in _DIAG, tuple(e for _, e in x.members),
                   tuple(prog[i][0] in _VAR for i, _ in x.members))
            self._batches.setdefault(sig, []).append(gi)
        self._inner = inner
        return inner

    def _gather(self, const_gates, var_gates, dt):
        if len(const_gates) != self._n_const:
            raise ValueError("The number of constant gates does not match the circuit.")
        if len(var_gates) != self._n_var:
            raise ValueError("The number of variable gates does not match the circuit.")
        def strict(g):   # same strictness as Circuit (PyO3's PyReadonlyArray1<Complex>): no silent dtype casts
            g = np.asarray(g)
            if g.dtype != dt:
                raise TypeError(f"gate arrays must have dtype {dt}, got {g.dtype}")
            return g.reshape(-1)
        return [strict(g) for g in const_gates], [strict(g) for g in var_gates]

    def _fuse(self, const_gates, var_gates):
        """-> (inner const list, inner var list, per-batch member stacks for the chain rule)"""
        inner = self._build()
        dt = np.dtype(getattr(inner, "dtype", np.complex128))
        lists = self._gather(const_gates, var_gates, dt)
        fused = [None] * len(self._xgates)
        keep = {}
        for sig, gis in self._batches.items():
            one, all_diag, embs, _ = sig
            stacks = []
            for m, emb in enumerate(embs):
                flat = np.stack([lists[self._src[self._xgates[gi].members[m][0]][0]]
                                 [self._src[self._xgates[gi].members[m][0]][1]] for gi in gis])
                stacks.append(_embed(flat.astype(np.complex128), emb))
            u = stacks[0]
            for s in stacks[1:]:
                u = s @ u
            keep[sig] = stacks
            for b, gi in enumerate(gis):
                if one:
                    fused[gi] = u[b].reshape(4).astype(dt)
                elif all_diag:
                    fused[gi] = u[b].diagonal().astype(dt)
                else:
                    fused[gi] = u[b].reshape(16).astype(dt)
        # the inner program's gate lists: fused gates and the (unfused) k-qubit gates, in execution order
        cg, vg, gi = [], [], 0
        for t, x in self._exec:
            if t == "gate":
                g, k = fused[gi], self._xkinds[gi]
                gi += 1
            elif t == "kgate":
                g, k = lists[self._src[x][0]][self._src[x][1]], self._program[x][0]
            else:
                continue
            (vg if k in _VAR else cg).append(g)
        return cg, vg, keep

    def run(self, const_gates, var_gates):
        cg, vg, _ = self._fuse(const_gates, var_gates)
        return self._inner.run(cg, vg)

    def forward(self, const_gates, var_gates):
        cg, vg, _ = self._fuse(const_gates, var_gates)
        return self._inner.forward(cg, vg)

    def backward(self, grads_wrt_density, const_gates, var_gates):
        cg, vg, keep = self._fuse(const_gates, var_gates)
        inner = self._inner
        dt = np.dtype(getattr(inner, "dtype", np.complex128))
        gfused = inner.backward([np.asarray(g, dtype=dt) for g in grads_wrt_density], cg, vg)
        slot = {}
        out = [None] * self._n_var
        v = gi = 0
        for t, x in self._exec:
            if t == "gate":
                if self._xkinds[gi] in _VAR:
                    slot[gi] = v; v += 1
                gi += 1
            elif t == "kgate" and self._program[x][0] in _VAR:
                out[self._src[x][1]] = np.asarray(gfused[v], dtype=dt)   # gradient of an unfused gate: as it is
                v += 1
        for sig, gis in self._batches.items():
            one, all_diag, embs, is_var = sig
            if not any(is_var):
                continue
            stacks = keep[sig]
            dim = 2 if one else 4
            g = np.stack([np.asarray(gfused[slot[gi]], dtype=np.complex128).reshape(-1) for gi in gis])
            if all_diag:
                gu = np.zeros((len(gis), 4, 4), dtype=np.complex128)
                gu[:, np.arange(4), np.arange(4)] = g
            else:
                gu = g.reshape(len(gis), dim, dim)
            k = len(stacks)
            # prefix products B_j = M_{j-1} ... M_1 and suffix products A_j = M_k ... M_{j+1}
            eye = np.broadcast_to(np.eye(dim, dtype=np.complex128), (len(gis), dim, dim))
            pre = [eye]
            for s in stacks[:-1]:
                pre.append(s @ pre[-1])
            suf = [eye]
            for s in stacks[:0:-1]:
                suf.append(suf[-1] @ s)
            suf = suf[::-1]
            for m in range(k):
                if not is_var[m]:
                    continue
                gm = np.swapaxes(suf[m], 1, 2) @ gu @ np.swapaxes(pre[m], 1, 2)
                flat = _project(gm, embs[m])
                for b, gi in enumerate(gis):
                    idx = self._xgates[gi].members[m][0]
                    out[self._src[idx][1]] = flat[b].astype(dt)
        return out

"""CPU: the oracle of the gates on k = 1..6 qubits (add_const_gate / add_var_gate / *_nonu): kgrad against the one- and
two-qubit gradients, equality with KOracleCircuit on programs without k-qubit gates, the 8th-order finite-difference
identity of the reverse pass with unitary and NonU k-qubit gates, the k <= 2 builders, rejected inputs, and
FusedCircuit, which runs k-qubit gates unfused as barriers."""
from importlib import import_module

import numpy as np
import pytest

from conftest import haar_unitary
from oracle import statevector as sv
from oracle.circuit import vjp
from oracle.kdens import KOracleCircuit, kgate
from oracle.kgates import KGateOracleCircuit, kgrad
from test_dens_k import _kdens_gates, _kdens_program, purity_loss_and_cotangents
from test_oracle import autodiff_gates, build_autodiff_circuit, tsallis_loss_and_cotangents

# (variable, non_unitary) of the four k-qubit gate kinds
COMBOS = [(False, False), (True, False), (False, True), (True, True)]


def kgate_ops(n, kpos, layers=4):
    """A program as a list of operations: layers of one- and two-qubit gates (unitary and NonU, constant and
    variable), each layer with the four k-qubit gates on kpos[0..3] in a rotating kind, so that over four layers every
    k meets every (const / var) x (unitary / NonU) combination; k-qubit and one- and two-qubit densities in between,
    and a variable k-qubit gate after the last differentiable density (zero gradient)."""
    ops = []
    for layer in range(layers):
        odd = layer % 2 == 1
        ops += [("q1", (i,), True, odd) for i in range(n)]
        ops += [("q2", (i + 1, i), not odd, odd) for i in range(layer % 2, n - 1, 2)]
        for j in range(4):
            var, nonu = COMBOS[(j + layer) % 4]
            ops.append(("k", tuple(kpos[j]), var, nonu))
            if j == 1:
                ops.append(("dens", tuple(kpos[(j + layer) % 4]), not odd))
        ops.append(("dens", (n - 1, 0), True))
        ops.append(("dens", (layer % n,), True))
    ops.append(("k", tuple(kpos[0]), True, False))
    return ops


def apply_ops(c, ops):
    for op in ops:
        if op[0] == "dens":
            (c.get_dens_op_with_grad if op[2] else c.get_dens_op)(list(op[1]))
            continue
        kind, pos, var, nonu = op
        name = "%s_gate%s" % ("var" if var else "const", "_nonu" if nonu else "")
        if kind == "k":
            getattr(c, "add_" + name)(list(pos))
        else:
            getattr(c, "add_%s_%s" % (kind, name))(*pos)


def ops_gates(rng, ops, dtype=np.complex128):
    """(const, var) gate lists of the program, in program order: Haar unitaries, NonU ones perturbed off unitarity."""
    const, var = [], []
    for op in ops:
        if op[0] == "dens":
            continue
        d = 1 << len(op[1])
        g = haar_unitary(rng, d)
        if op[3]:
            g = g + 0.01 * (rng.normal(size=d * d) + 1j * rng.normal(size=d * d))
        (var if op[2] else const).append(np.asarray(g, dtype=dtype))
    return const, var


def _state(rng, n):
    return rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)


@pytest.mark.parametrize("pos", [0, 3, 6])
def test_kgrad_k1_is_q1grad(pos):
    rng = np.random.default_rng(pos)
    f, b = _state(rng, 7), _state(rng, 7)
    np.testing.assert_allclose(kgrad(f, b, [pos]), sv.q1grad(f, b, pos), rtol=0, atol=1e-12)


@pytest.mark.parametrize("p2,p1", [(1, 0), (0, 1), (5, 2), (2, 6)])
def test_kgrad_k2_is_q2grad(p2, p1):
    rng = np.random.default_rng(10 * p2 + p1)
    f, b = _state(rng, 7), _state(rng, 7)
    np.testing.assert_allclose(kgrad(f, b, [p2, p1]), sv.q2grad(f, b, p2, p1), rtol=0, atol=1e-12)


def test_kgrad_is_the_derivative_of_the_overlap():
    """<conj bwd, U fwd> = sum_r,c,rest bwd[r, rest] U[r, c] fwd[c, rest] is linear in U with gradient kgrad."""
    rng = np.random.default_rng(3)
    pos = [4, 0, 2]
    f, b = _state(rng, 6), _state(rng, 6)
    u = rng.normal(size=64) + 1j * rng.normal(size=64)
    np.testing.assert_allclose(np.sum(b * kgate(f, u, pos)), np.sum(kgrad(f, b, pos) * u), rtol=1e-12)


def test_k_gate_oracle_equals_the_k_oracle_without_k_gates():
    """KGateOracleCircuit restates KOracleCircuit's interpreters: on programs without k-qubit gates (every gate and
    density kind, k-qubit densities, NonU un-compute, gates after the last seed) run, forward and backward agree
    exactly."""
    n, layers = 6, 2
    const, var = autodiff_gates(np.random.default_rng(8), n, layers)
    var = var + [haar_unitary(np.random.default_rng(1), 2)]
    const7, var7 = _kdens_gates(np.random.default_rng(2), 7)
    out = []
    for cls in (KOracleCircuit, KGateOracleCircuit):
        c = cls(n)
        build_autodiff_circuit(c, n, layers)
        c.add_q1_var_gate(0)
        dens = c.forward(const, var)
        _, cts = tsallis_loss_and_cotangents(dens)
        c7 = cls(7)
        _kdens_program(c7, 7)
        dens7 = c7.forward(const7, var7)
        _, cts7 = purity_loss_and_cotangents(dens7)
        out.append((c.run(const, var), dens, vjp(c, var, const, cts), [c.state],
                    c7.run(const7, var7), dens7, vjp(c7, var7, const7, cts7), [c7.state]))
    for a, b in zip(out[0], out[1]):
        assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("nonu", [False, True])
def test_backward_with_k_gates_matches_8th_order_finite_difference(nonu):
    n, eta = 7, 1e-6
    kpos = [[2, 0, 5], [6, 1, 3, 0], [0, 4, 2, 6, 1], [5, 3, 1, 0, 2, 6]]
    ops = [op if op[0] != "k" else (op[0], op[1], op[2], nonu) for op in kgate_ops(n, kpos, layers=2)]
    rng = np.random.default_rng(42)
    c = KGateOracleCircuit(n)
    apply_ops(c, ops)
    const, var = ops_gates(rng, ops)
    assert sum(v.size for v in var) > 4 ** 6    # the k-qubit gates are among the variable ones
    pert = [rng.normal(size=v.size) + 1j * rng.normal(size=v.size) for v in var]

    def loss_at(s):
        return purity_loss_and_cotangents(c.forward(const, [v + s * eta * p for v, p in zip(var, pert)]))[0]

    fd = (loss_at(-4) / 280 - loss_at(4) / 280 - 4 * loss_at(-3) / 105 + 4 * loss_at(3) / 105
          + loss_at(-2) / 5 - loss_at(2) / 5 - 4 * loss_at(-1) / 5 + 4 * loss_at(1) / 5) / eta
    dens = c.forward(const, var)
    _, cts = purity_loss_and_cotangents(dens)
    grads = vjp(c, var, const, cts)
    assert [g.size for g in grads] == [v.size for v in var]
    assert np.array_equal(grads[-1], np.zeros(4 ** 3))   # the k-qubit gate after the last differentiable density
    ds = sum((g @ p).real for g, p in zip(grads, pert))
    assert abs(ds - fd) / min(abs(ds), abs(fd)) < 1e-9
    np.testing.assert_allclose(c.state, c.initial_state, atol=1e-9)


def test_k1_and_k2_builders_add_the_existing_kinds():
    c = KGateOracleCircuit(5)
    c.add_const_gate([3]); c.add_var_gate([1]); c.add_const_gate_nonu([0]); c.add_var_gate_nonu([4])
    c.add_const_gate([3, 0]); c.add_var_gate([1, 4]); c.add_const_gate_nonu([0, 2]); c.add_var_gate_nonu([4, 3])
    c.add_var_gate_nonu([4, 1, 0])
    assert c.instructions == [(6, 3), (8, 1), (7, 0), (9, 4), (0, 3, 0), (1, 1, 4), (2, 0, 2), (3, 4, 3),
                              (19, (4, 1, 0))]


@pytest.mark.parametrize("positions", [[1, 1, 2], [0, 3, 0, 2], [], [0, 1, 2, 3, 4, 5, 6], [0, 1, 8], [9]])
def test_bad_positions_raise(pkg, positions):
    fusion = import_module("differentiable-quantum-circuit-cuda_b200.fusion")
    for c in (KGateOracleCircuit(8), fusion.FusedCircuit(8, backend=KGateOracleCircuit)):
        for name in ("add_const_gate", "add_var_gate", "add_const_gate_nonu", "add_var_gate_nonu"):
            with pytest.raises(ValueError):
                getattr(c, name)(positions)
        assert (c.instructions if hasattr(c, "instructions") else c._program) == []


def test_fused_circuit_treats_k_gates_as_barriers(pkg):
    """FusedCircuit on the oracle backend: the same outputs and gradients as the plain VM; a k-qubit gate closes the
    fused gates around it and reaches the backend unfused; counts describe the user's program."""
    fusion = import_module("differentiable-quantum-circuit-cuda_b200.fusion")
    n = 7
    kpos = [[2, 0, 5], [6, 1, 3, 0], [0, 4, 2, 6, 1], [5, 3, 1, 0, 2, 6]]
    ops = kgate_ops(n, kpos, layers=2)
    const, var = ops_gates(np.random.default_rng(5), ops)
    o = KGateOracleCircuit(n)
    apply_ops(o, ops)
    f = fusion.FusedCircuit(n, backend=KGateOracleCircuit)
    apply_ops(f, ops)
    d_o, d_f = o.forward(const, var), f.forward(const, var)
    assert len(d_o) == len(d_f)
    for a, b in zip(d_o, d_f):
        np.testing.assert_allclose(a, b, atol=1e-10)
    _, cts = purity_loss_and_cotangents(d_o)
    g_o = vjp(o, var, const, cts)
    g_f = f.backward([ct.conj() for ct in cts], const, var)
    assert [g.size for g in g_f] == [g.size for g in g_o]
    for a, b in zip(g_o, g_f):
        np.testing.assert_allclose(a, b, atol=1e-9)
    inner = f._build().instructions
    assert [i for i in inner if i[0] >= 16] == [i for i in o.instructions if i[0] >= 16]
    assert f._count(1) == len(const) and f._count(2) == len(var)
    assert f._count(7) == sum(v.size for v in var)
    # one-qubit gates on the same qubit on both sides of a k-qubit gate on that qubit stay two gates
    g = fusion.FusedCircuit(4, backend=KGateOracleCircuit)
    g.add_q1_var_gate(0); g.add_const_gate([2, 0, 1]); g.add_q1_var_gate(0); g.add_q1_var_gate(0)
    assert g.fused_gate_count == 2
    assert [i[0] for i in g._build().instructions] == [8, 16, 8]

"""CPU: the oracle of the diagonal gates on k = 1..6 qubits (add_const_gate_diag / add_var_gate_diag / *_nonu):
kdiag / kdiag_grad against the dense k-qubit gate and the two-qubit diagonal, equality with KGateOracleCircuit on
programs without the new kinds, the 8th-order finite-difference identity with unitary and NonU diagonals, the builders,
FusedCircuit (diagonals are unfused barriers), and the host-side sharding and scheduling rules
(tests/cpp/diag_k_host_check.cpp)."""
import os
import subprocess
from importlib import import_module

import numpy as np
import pytest

from oracle import statevector as sv
from oracle.circuit import vjp
from oracle.kdens import kgate
from oracle.kdiag import KDiagOracleCircuit, kdiag, kdiag_grad
from oracle.kgates import KGateOracleCircuit, kgrad
from test_dens_k import purity_loss_and_cotangents
from test_gate_k import COMBOS, apply_ops, kgate_ops, ops_gates

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# scattered positions of the diagonals on k = 1..6 qubits (any order)
SCATTERED = [[4], [0, 6], [2, 0, 5], [6, 1, 3, 0], [0, 4, 2, 6, 1], [5, 3, 1, 0, 2, 6]]


def kdiag_ops(n, dpos, layers=2, nonu=None):
    """kgate_ops with diagonal k-qubit gates on dpos (k = 1..6) in a rotating (const / var) x (unitary / NonU) kind
    after every layer's k-qubit gates, and a variable diagonal after the last differentiable density (zero gradient).
    Operations: ("kd", positions, var, nonu)."""
    ops = []
    layer = 0
    for op in kgate_ops(n, [[2, 0, 5], [6, 1, 3, 0], [0, 4, 2, 6, 1], [5, 3, 1, 0, 2, 6]], layers)[:-1]:
        ops.append(op)
        if op[0] == "dens" and len(op[1]) == 1:   # the end of a layer
            for j, pos in enumerate(dpos):
                var, nu = COMBOS[(j + layer) % 4]
                ops.append(("kd", tuple(pos), var, nu if nonu is None else nonu))
            layer += 1
    ops.append(("kd", tuple(dpos[2]), True, False))
    return ops


def apply_dops(c, ops):
    for op in ops:
        if op[0] == "kd":
            getattr(c, "add_%s_gate_diag%s" % ("var" if op[2] else "const", "_nonu" if op[3] else ""))(list(op[1]))
        else:
            apply_ops(c, [op])


def dops_gates(rng, ops, dtype=np.complex128):
    """ops_gates, with unit-modulus diagonals for the unitary diagonal gates and perturbed ones for NonU."""
    const, var = [], []
    for op in ops:
        if op[0] != "kd":
            c, v = ops_gates(rng, [op], dtype)
            const += c
            var += v
            continue
        d = np.exp(1j * rng.uniform(0, 2 * np.pi, size=1 << len(op[1])))
        if op[3]:
            d = d * (1 + 0.05 * rng.uniform(-1, 1, size=d.size))
        (var if op[2] else const).append(np.asarray(d, dtype=dtype))
    return const, var


def _state(rng, n):
    return rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)


@pytest.mark.parametrize("k", range(1, 7))
def test_kdiag_is_the_dense_gate_on_diag_d(k):
    rng = np.random.default_rng(k)
    pos = SCATTERED[k - 1]
    s, b = _state(rng, 7), _state(rng, 7)
    d = rng.normal(size=1 << k) + 1j * rng.normal(size=1 << k)
    np.testing.assert_allclose(kdiag(s, d, pos), kgate(s, np.diag(d).reshape(-1), pos), rtol=0, atol=1e-12)
    g = kgrad(s, b, pos).reshape(1 << k, 1 << k)
    np.testing.assert_allclose(kdiag_grad(s, b, pos), np.diag(g), rtol=0, atol=1e-11)


@pytest.mark.parametrize("p2,p1", [(1, 0), (0, 1), (5, 2), (2, 6)])
def test_kdiag_k2_is_q2gate_diag(p2, p1):
    rng = np.random.default_rng(10 * p2 + p1)
    s, b = _state(rng, 7), _state(rng, 7)
    d = rng.normal(size=4) + 1j * rng.normal(size=4)
    np.testing.assert_allclose(kdiag(s, d, [p2, p1]), sv.q2gate_diag(s, d, p2, p1), rtol=0, atol=1e-12)
    np.testing.assert_allclose(kdiag_grad(s, b, [p2, p1]), sv.q2grad_diag(s, b, p2, p1), rtol=0, atol=1e-12)


def test_k_diag_oracle_equals_the_k_gate_oracle_without_diagonals():
    """KDiagOracleCircuit restates KGateOracleCircuit's interpreters: on programs without the new kinds (every gate and
    density kind, k-qubit gates and densities) run, forward and backward agree exactly."""
    n = 7
    ops = kgate_ops(n, [[2, 0, 5], [6, 1, 3, 0], [0, 4, 2, 6, 1], [5, 3, 1, 0, 2, 6]], layers=2)
    const, var = ops_gates(np.random.default_rng(8), ops)
    out = []
    for cls in (KGateOracleCircuit, KDiagOracleCircuit):
        c = cls(n)
        apply_ops(c, ops)
        dens = c.forward(const, var)
        _, cts = purity_loss_and_cotangents(dens)
        out.append((c.run(const, var), dens, vjp(c, var, const, cts), [c.state]))
    for a, b in zip(out[0], out[1]):
        assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("nonu", [False, True])
def test_backward_with_diagonals_matches_8th_order_finite_difference(nonu):
    n, eta = 7, 1e-5
    ops = kdiag_ops(n, SCATTERED, nonu=nonu)
    rng = np.random.default_rng(42)
    c = KDiagOracleCircuit(n)
    apply_dops(c, ops)
    const, var = dops_gates(rng, ops)
    pert = [rng.normal(size=v.size) + 1j * rng.normal(size=v.size) for v in var]

    def loss_at(s):
        return purity_loss_and_cotangents(c.forward(const, [v + s * eta * p for v, p in zip(var, pert)]))[0]

    fd = (loss_at(-4) / 280 - loss_at(4) / 280 - 4 * loss_at(-3) / 105 + 4 * loss_at(3) / 105
          + loss_at(-2) / 5 - loss_at(2) / 5 - 4 * loss_at(-1) / 5 + 4 * loss_at(1) / 5) / eta
    dens = c.forward(const, var)
    _, cts = purity_loss_and_cotangents(dens)
    grads = vjp(c, var, const, cts)
    assert [g.size for g in grads] == [v.size for v in var]
    assert np.array_equal(grads[-1], np.zeros(8))   # the diagonal after the last differentiable density
    terms = [(g @ p).real for g, p in zip(grads, pert)]
    ds = sum(terms)
    # relative to the terms' magnitude (with every diagonal NonU their sum nearly cancels: |ds| = 0.07)
    assert abs(ds - fd) / sum(abs(t) for t in terms) < 1e-9
    np.testing.assert_allclose(c.state, c.initial_state, atol=1e-9)


def test_builders_map_k2_unitary_to_the_q2_diag_kinds():
    c = KDiagOracleCircuit(5)
    c.add_const_gate_diag([3, 0]); c.add_var_gate_diag([1, 4])
    c.add_const_gate_diag_nonu([0, 2]); c.add_var_gate_diag_nonu([4, 3])
    c.add_const_gate_diag([3]); c.add_var_gate_diag_nonu([4, 1, 0])
    assert c.instructions == [(4, 3, 0), (5, 1, 4), (22, (0, 2)), (23, (4, 3)), (20, (3,)), (23, (4, 1, 0))]


@pytest.mark.parametrize("positions", [[1, 1, 2], [0, 3, 0, 2], [], [0, 1, 2, 3, 4, 5, 6], [0, 1, 8], [9]])
def test_bad_positions_raise(pkg, positions):
    fusion = import_module("differentiable-quantum-circuit-cuda_b200.fusion")
    for c in (KDiagOracleCircuit(8), fusion.FusedCircuit(8, backend=KDiagOracleCircuit)):
        for name in ("add_const_gate_diag", "add_var_gate_diag", "add_const_gate_diag_nonu", "add_var_gate_diag_nonu"):
            with pytest.raises(ValueError):
                getattr(c, name)(positions)
        assert (c.instructions if hasattr(c, "instructions") else c._program) == []


def test_fused_circuit_treats_diagonals_as_barriers(pkg):
    """FusedCircuit on the oracle backend: the same outputs and gradients as the plain VM; a diagonal k-qubit gate
    closes the fused gates around it and reaches the backend unfused; counts describe the user's program."""
    fusion = import_module("differentiable-quantum-circuit-cuda_b200.fusion")
    n = 7
    ops = kdiag_ops(n, SCATTERED)
    const, var = dops_gates(np.random.default_rng(5), ops)
    o = KDiagOracleCircuit(n)
    apply_dops(o, ops)
    f = fusion.FusedCircuit(n, backend=KDiagOracleCircuit)
    apply_dops(f, ops)
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
    assert [i for i in inner if i[0] >= 20] == [i for i in o.instructions if i[0] >= 20]
    assert f._count(1) == len(const) and f._count(2) == len(var)
    assert f._count(7) == sum(v.size for v in var)
    # one-qubit gates on the same qubit on both sides of a diagonal on that qubit stay two gates
    g = fusion.FusedCircuit(4, backend=KDiagOracleCircuit)
    g.add_q1_var_gate(0); g.add_const_gate_diag([2, 0, 1]); g.add_q1_var_gate(0); g.add_q1_var_gate(0)
    assert g.fused_gate_count == 2
    assert [i[0] for i in g._build().instructions] == [8, 20, 8]


def test_sharding_fold_scatter_and_plans(tmp_path):
    """csrc/diag_k_host.hpp and csrc/scheduler.hpp: no exchange for a diagonal on global qubits, the diagonal is a wall,
    and the fold / scatter against a brute-force enumeration (tests/cpp/diag_k_host_check.cpp)."""
    exe = str(tmp_path / "diag_k_host_check")
    csrc = os.path.join(ROOT, "differentiable-quantum-circuit-cuda_b200", "csrc")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", csrc, os.path.join(ROOT, "tests", "cpp", "diag_k_host_check.cpp"),
                    "-o", exe], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and "OK" in out.stdout, out.stdout + out.stderr

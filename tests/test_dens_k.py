"""CPU: the oracle of the k-qubit reduced density matrices (get_dens_op / get_dens_op_with_grad, 1 <= k <= 6):
kdensity / kgate against the one- and two-qubit primitives, partial traces, the 8th-order finite-difference identity
of the reverse pass with k = 3 and 4 differentiable densities, and the rejected inputs."""
import numpy as np
import pytest

from conftest import haar_unitary
from oracle import statevector as sv
from oracle.circuit import OracleCircuit, vjp
from test_oracle import autodiff_gates, build_autodiff_circuit, tsallis_loss_and_cotangents
from oracle.kdens import KOracleCircuit, kdensity, kgate


def _state(rng, n):
    return rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)


def _ptrace_first(rho, k):
    """Trace out the most significant qubit (positions[0]) of a k-qubit density."""
    d = 1 << (k - 1)
    return np.einsum("aiaj->ij", rho.reshape(2, d, 2, d))


@pytest.mark.parametrize("pos", [0, 3, 6])
def test_kdensity_k1_is_q1density(pos):
    s = _state(np.random.default_rng(pos), 7)
    np.testing.assert_allclose(kdensity(s, [pos]).reshape(-1), sv.q1density(s, pos), rtol=0, atol=1e-12)


@pytest.mark.parametrize("p2,p1", [(1, 0), (0, 1), (5, 2), (2, 6)])
def test_kdensity_k2_is_q2density(p2, p1):
    s = _state(np.random.default_rng(10 * p2 + p1), 7)
    np.testing.assert_allclose(kdensity(s, [p2, p1]).reshape(-1), sv.q2density(s, p2, p1), rtol=0, atol=1e-12)


@pytest.mark.parametrize("pos", [0, 4])
def test_kgate_k1_is_q1gate(pos):
    rng = np.random.default_rng(pos)
    s, g = _state(rng, 6), rng.normal(size=4) + 1j * rng.normal(size=4)
    np.testing.assert_allclose(kgate(s, g, [pos]), sv.q1gate(s, g, pos), rtol=0, atol=1e-12)


@pytest.mark.parametrize("p2,p1", [(1, 0), (0, 1), (5, 2), (2, 5)])
def test_kgate_k2_is_q2gate(p2, p1):
    rng = np.random.default_rng(p2 + 7 * p1)
    s, g = _state(rng, 6), rng.normal(size=16) + 1j * rng.normal(size=16)
    np.testing.assert_allclose(kgate(s, g, [p2, p1]), sv.q2gate(s, g, p2, p1), rtol=0, atol=1e-12)


@pytest.mark.parametrize("positions", [[2, 0, 5], [6, 1, 3, 0], [0, 1, 2, 3, 4], [7, 5, 3, 1, 0, 2]])
def test_partial_traces_give_smaller_densities(positions):
    rng = np.random.default_rng(len(positions))
    s = _state(rng, 8)
    rho = kdensity(s, positions)
    k = len(positions)
    np.testing.assert_allclose(rho, rho.conj().T, atol=1e-12)
    np.testing.assert_allclose(np.trace(rho), np.vdot(s, s), rtol=1e-12)
    # the (k-1)-qubit density on positions[1:]
    np.testing.assert_allclose(_ptrace_first(rho, k), kdensity(s, positions[1:]), atol=1e-10)
    # the 2-qubit density on the last two positions, by tracing out every other qubit
    r = rho.reshape((2,) * (2 * k))
    keep = [k - 2, k - 1]
    letters = "abcdefghijkl"
    row = [letters[i] for i in range(k)]
    col = [letters[6 + i] if i in keep else letters[i] for i in range(k)]
    out = "".join(letters[i] for i in keep) + "".join(letters[6 + i] for i in keep)
    two = np.einsum("".join(row) + "".join(col) + "->" + out, r).reshape(4, 4)
    np.testing.assert_allclose(two.reshape(-1), sv.q2density(s, positions[-2], positions[-1]), atol=1e-10)


def _kdens_program(c, n):
    """A VM program with NonU gates and k = 3 and 4 differentiable densities between layers (plus q1 / q2 ones)."""
    for layer in range(2):
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(0, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        c.get_dens_op_with_grad([2, 0, 5] if layer == 0 else [6, 1, 3, 0])
        c.get_q2_dens_op_with_grad(1, 0)
        for i in range(1, n - 1, 2):
            c.add_q2_var_gate_nonu(i + 1, i)
        for i in range(n):
            c.add_q1_var_gate_nonu(i)
        c.get_dens_op([3, 4, 5])
        c.get_dens_op_with_grad([0, 4, 2, 6] if layer == 0 else [5, 3, 1])
        c.get_q1_dens_op_with_grad(layer)


def _kdens_gates(rng, n, dtype=np.complex128):
    rc = lambda k: rng.normal(size=k * k) + 1j * rng.normal(size=k * k)  # noqa: E731
    var = []
    for _ in range(2):
        var += [haar_unitary(rng, 2) for _ in range(n)]
        var += [haar_unitary(rng, 4) for _ in range(0, n - 1, 2)]
        var += [0.01 * rc(4) + haar_unitary(rng, 4) for _ in range(1, n - 1, 2)]
        var += [0.01 * rc(2) + haar_unitary(rng, 2) for _ in range(n)]
    return [], [np.asarray(v, dtype=dtype) for v in var]


def purity_loss_and_cotangents(dens):
    """sum tr rho^2 and its JAX cotangents (2 rho^T)."""
    return sum(np.einsum("ij,ji->", d, d).real for d in dens), [2.0 * d.T for d in dens]


def test_backward_with_k_densities_matches_8th_order_finite_difference():
    n, eta = 7, 1e-6
    rng = np.random.default_rng(42)
    c = KOracleCircuit(n)
    _kdens_program(c, n)
    const, var = _kdens_gates(rng, n)
    pert = [rng.normal(size=v.size) + 1j * rng.normal(size=v.size) for v in var]

    def loss_at(s):
        return purity_loss_and_cotangents(c.forward(const, [v + s * eta * p for v, p in zip(var, pert)]))[0]

    fd = (loss_at(-4) / 280 - loss_at(4) / 280 - 4 * loss_at(-3) / 105 + 4 * loss_at(3) / 105
          + loss_at(-2) / 5 - loss_at(2) / 5 - 4 * loss_at(-1) / 5 + 4 * loss_at(1) / 5) / eta
    dens = c.forward(const, var)
    assert [d.shape for d in dens] == [(8, 8), (4, 4), (16, 16), (2, 2), (16, 16), (4, 4), (8, 8), (2, 2)]
    _, cts = purity_loss_and_cotangents(dens)
    grads = vjp(c, var, const, cts)
    ds = sum((g @ p).real for g, p in zip(grads, pert))
    assert abs(ds - fd) / min(abs(ds), abs(fd)) < 1e-9
    np.testing.assert_allclose(c.state, c.initial_state, atol=1e-9)
    # run() returns every density in program order, the non-differentiable ones included
    assert [d.shape for d in c.run(const, var)] == [(8, 8), (4, 4), (8, 8), (16, 16), (2, 2), (16, 16), (4, 4),
                                                     (8, 8), (8, 8), (2, 2)]


def test_k1_and_k2_builders_add_the_existing_kinds():
    c = KOracleCircuit(5)
    c.get_dens_op([3])
    c.get_dens_op_with_grad([2, 4])
    c.get_dens_op_with_grad([4, 1, 0])
    assert c.instructions == [(11, 3), (12, 2, 4), (15, (4, 1, 0))]


@pytest.mark.parametrize("positions", [[1, 1, 2], [0, 3, 0, 2], [], [0, 1, 2, 3, 4, 5, 6], [0, 1, 8], [9]])
def test_bad_positions_raise(positions):
    c = KOracleCircuit(8)
    with pytest.raises(ValueError):
        c.get_dens_op(positions)
    with pytest.raises(ValueError):
        c.get_dens_op_with_grad(positions)
    assert c.instructions == []


def test_fused_circuit_treats_k_densities_as_barriers(pkg):
    """FusedCircuit on the oracle backend: same outputs and gradients as the plain VM, output lengths in count."""
    from importlib import import_module
    fusion = import_module("differentiable-quantum-circuit-cuda_b200.fusion")
    n = 7
    rng = np.random.default_rng(5)
    const, var = _kdens_gates(rng, n)
    o = KOracleCircuit(n)
    _kdens_program(o, n)
    f = fusion.FusedCircuit(n, backend=lambda m: KOracleCircuit(m))
    _kdens_program(f, n)
    d_o, d_f = o.forward(const, var), f.forward(const, var)
    assert len(d_o) == len(d_f)
    for a, b in zip(d_o, d_f):
        np.testing.assert_allclose(a, b, atol=1e-10)
    _, cts = purity_loss_and_cotangents(d_o)
    g_o = vjp(o, var, const, cts)
    g_f = f.backward([ct.conj() for ct in cts], const, var)
    for a, b in zip(g_o, g_f):
        np.testing.assert_allclose(a, b, atol=1e-9)
    assert f._count(3) == 10 and f._count(4) == 8
    assert f._count(5) == sum(d.size for d in o.run(const, var))
    assert f._count(6) == sum(d.size for d in d_o)


def test_k_oracle_equals_the_vm_without_k_densities():
    """KOracleCircuit restates OracleCircuit's interpreters: on a program without k-qubit densities (every gate and
    density kind, NonU un-compute, gates after the last seed) run, forward and backward agree exactly."""
    n, layers = 6, 2
    const, var = autodiff_gates(np.random.default_rng(8), n, layers)
    out = []
    for cls in (OracleCircuit, KOracleCircuit):
        c = cls(n)
        build_autodiff_circuit(c, n, layers)
        c.add_q1_var_gate(0)
        var_c = var + [haar_unitary(np.random.default_rng(1), 2)]
        dens = c.forward(const, var_c)
        _, cts = tsallis_loss_and_cotangents(dens)
        out.append((c.run(const, var_c), dens, vjp(c, var_c, const, cts), c.state))
    for a, b in zip(out[0][:3], out[1][:3]):
        assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))
    assert np.array_equal(out[0][3], out[1][3])

"""Gate fusion in front of the executor (differentiable-quantum-circuit-cuda_b200/fusion.py): the fused
program + the host-side chain rule must reproduce the densities and the per-gate gradients of the original
program.  CPU: the fused program runs on the oracle VM (checker backend injected by the test); GPU: on the
CUDA `Circuit`."""
import importlib

import numpy as np
import pytest

from oracle.circuit import OracleCircuit, vjp
from conftest import haar_unitary
from test_oracle import autodiff_gates, build_autodiff_circuit, tsallis_loss_and_cotangents
from test_scheduler import brickwork, vqse

pkg = importlib.import_module("differentiable-quantum-circuit-cuda_b200")
fusion = importlib.import_module("differentiable-quantum-circuit-cuda_b200.fusion")


def _gates_for(o, rng, dtype=np.complex128):
    const, var = [], []
    for inst in o.instructions:
        k = inst[0]
        if k in (10, 11, 12, 13):
            continue
        if k in (0, 1):
            g = haar_unitary(rng, 4, dtype)
        elif k in (2, 3):
            g = (haar_unitary(rng, 4) + 0.05 * (rng.normal(size=16) + 1j * rng.normal(size=16))).astype(dtype)
        elif k in (4, 5):
            g = np.exp(1j * rng.normal(size=4)).astype(dtype)
        elif k in (6, 8):
            g = haar_unitary(rng, 2, dtype)
        else:
            g = (haar_unitary(rng, 2) + 0.05 * (rng.normal(size=4) + 1j * rng.normal(size=4))).astype(dtype)
        (var if k in (1, 3, 5, 8, 9) else const).append(g)
    return const, var


def _mixed(c, n):
    """every fusion rule: one-qubit chains, one-qubit gates absorbed by / joining two-qubit gates, repeated
    pairs in both qubit orders, diagonal-only pairs, NonU members, densities in between."""
    c.add_q1_var_gate(0); c.add_q1_const_gate(0); c.add_q1_var_gate_nonu(1)
    c.add_q2_var_gate(1, 0); c.add_q2_var_gate(0, 1); c.add_q1_var_gate(1)
    c.add_q2_var_gate_diag(2, 3); c.add_q2_var_gate_diag(3, 2); c.add_q2_const_gate_diag(2, 3)
    c.add_q2_var_gate_diag(1, 2); c.add_q1_var_gate(2); c.add_q1_var_gate(3)
    c.get_q2_dens_op_with_grad(1, 2); c.get_q1_dens_op(0)
    c.add_q1_var_gate(2); c.add_q2_const_gate(2, 4); c.add_q2_var_gate_nonu(4, 2); c.add_q1_const_gate_nonu(4)
    c.add_q2_var_gate(3, n - 1); c.add_q1_var_gate(3)
    for i in range(n):
        c.get_q1_dens_op_with_grad(i)
    c.get_q2_dens_op_with_grad(0, n - 1)
    c.add_q1_var_gate(0)   # after the last differentiable density: zero gradient


def _build(case, c, n):
    if case == "brickwork":
        brickwork(c, n, 5)
    elif case == "vqse":
        vqse(c, n, 3)
    elif case == "autodiff":
        build_autodiff_circuit(c, n, 2)
    else:
        _mixed(c, n)


@pytest.mark.parametrize("case", ["mixed", "vqse", "autodiff", "brickwork"])
def test_fused_program_on_the_oracle_equals_the_original(case):
    n = 7
    rng = np.random.default_rng(8)
    o = OracleCircuit(n)
    _build(case, o, n)
    const, var = _gates_for(o, rng)
    f = fusion.FusedCircuit(n, backend=lambda q: OracleCircuit(q))
    _build(case, f, n)
    dens_o, dens_f = o.forward(const, var), f.forward(const, var)
    assert len(dens_o) == len(dens_f)
    for a, b in zip(dens_f, dens_o):
        np.testing.assert_allclose(a, b, atol=1e-12)
    for a, b in zip(f.run(const, var), o.run(const, var)):
        np.testing.assert_allclose(a, b, atol=1e-12)
    cts = []
    for d in dens_o:
        a = rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)
        cts.append((a + a.conj().T) / 2)
    grads_o = vjp(o, var, const, cts)
    f.forward(const, var)
    grads_f = f.backward([ct.conj() for ct in cts], const, var)
    assert len(grads_f) == len(grads_o) == len(var)
    scale = max(np.abs(g).max() for g in grads_o)
    for a, b in zip(grads_f, grads_o):
        assert a.shape == b.shape
        np.testing.assert_allclose(a, b, atol=1e-11 * scale)
    n_gates = sum(1 for i in o.instructions if i[0] < 10)
    if case == "vqse":
        assert f.fused_gate_count <= n_gates // 2 + n   # n dense gates per layer instead of 2 n cheap ones
    elif case == "brickwork":
        assert f.fused_gate_count == n_gates            # nothing to fuse: distinct pairs alternate
    else:
        assert f.fused_gate_count < n_gates


def test_fusion_plan_structure():
    prog = [(8, 0), (8, 1), (1, 1, 0), (5, 0, 1), (8, 1), (1, 1, 2), (12, 1, 0), (8, 0)]
    ex = fusion.plan_fusion(prog)
    kinds = [t for t, _ in ex]
    assert kinds == ["gate", "gate", "dens", "gate"]
    first = ex[0][1]
    assert (first.pos2, first.pos1) == (1, 0)
    assert [i for i, _ in first.members] == [1, 0, 2, 3, 4]   # both one-qubit gates absorbed, then the pair's gates
    assert [i for i, _ in ex[1][1].members] == [5] and [i for i, _ in ex[3][1].members] == [7]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_fused_circuit_on_the_gpu_matches_the_oracle(precision):
    n = 13
    dtype = np.complex64 if precision == "f32" else np.complex128
    rng = np.random.default_rng(9)
    for case in ("vqse", "mixed"):
        o = OracleCircuit(n)
        _build(case, o, n)
        const, var = _gates_for(o, rng, dtype)
        f = fusion.FusedCircuit(n, precision=precision)
        f.set_option("tile_bits", 11)
        _build(case, f, n)
        dens_o = o.forward(const, var)
        dens_f = f.forward(const, var)
        tol = 1e-5 if precision == "f32" else 1e-12
        for a, b in zip(dens_f, dens_o):
            assert np.abs(a - b).max() < tol
        _, cts = tsallis_loss_and_cotangents(dens_o)
        grads_o = vjp(o, var, const, cts)
        grads_f = f.backward([np.asarray(ct, dtype=dtype).conj() for ct in cts], const, var)
        scale = max(np.abs(g).max() for g in grads_o)
        assert max(np.abs(a - b).max() for a, b in zip(grads_f, grads_o)) / scale < tol


@pytest.mark.gpu
def test_autograd_circuit_with_fusion_matches_the_plain_one():
    """qdc.AutoGradCircuit(fused=True): same densities and vjp as the unfused wrapper (f64, VQSE ansatz)."""
    from qdc import AutoGradCircuit
    n, layers = 12, 2
    rng = np.random.default_rng(12)
    res = {}
    o = OracleCircuit(n)
    vqse(o, n, layers)
    _, var = _gates_for(o, rng)
    for fused in (False, True):
        c = AutoGradCircuit(n, precision="f64", fused=fused)
        vqse(c, n, layers)
        simple_run, autodiff_run = c.build()
        dens = autodiff_run.forward(var, [])
        _, cts = tsallis_loss_and_cotangents(dens)
        res[fused] = (dens, autodiff_run.vjp(var, [], cts), simple_run(var, []))
    for a, b in zip(res[True][0] + res[True][2], res[False][0] + res[False][2]):
        np.testing.assert_allclose(a, b, atol=1e-12)
    scale = max(np.abs(g).max() for g in res[False][1])
    for a, b in zip(res[True][1], res[False][1]):
        np.testing.assert_allclose(a, b, atol=1e-11 * scale)


@pytest.mark.parametrize("seed", range(8))
def test_random_programs_fuse_exactly(seed):
    """Random programs over every instruction kind: fused program + chain rule == original (oracle VM)."""
    from random_programs import _random_program
    rng = np.random.default_rng(200 + seed)
    n = 6
    o, const, var = _random_program(rng, n, 50)
    f = fusion.FusedCircuit(n, backend=lambda q: OracleCircuit(q))
    adders = {0: "add_q2_const_gate", 1: "add_q2_var_gate", 2: "add_q2_const_gate_nonu", 3: "add_q2_var_gate_nonu",
              4: "add_q2_const_gate_diag", 5: "add_q2_var_gate_diag", 6: "add_q1_const_gate",
              7: "add_q1_const_gate_nonu", 8: "add_q1_var_gate", 9: "add_q1_var_gate_nonu", 10: "get_q2_dens_op",
              11: "get_q1_dens_op", 12: "get_q2_dens_op_with_grad", 13: "get_q1_dens_op_with_grad"}
    for inst in o.instructions:
        getattr(f, adders[inst[0]])(*inst[1:])
    dens_o, dens_f = o.forward(const, var), f.forward(const, var)
    for a, b in zip(dens_f, dens_o):
        np.testing.assert_allclose(a, b, atol=1e-11)
    cts = []
    for d in dens_o:
        a = rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)
        cts.append((a + a.conj().T) / 2)
    grads_o = vjp(o, var, const, cts)
    grads_f = f.backward([ct.conj() for ct in cts], const, var)
    scale = max([np.abs(g).max() for g in grads_o] + [1e-30])
    for a, b in zip(grads_f, grads_o):
        np.testing.assert_allclose(a, b, atol=1e-10 * scale)
    assert f.fused_gate_count <= sum(1 for i in o.instructions if i[0] < 10)

"""GPU: the tensor-core fused 6-qubit blocks (option "tc", csrc/tc_exec.cuh + tc_block.cuh) against the per-gate
streaming executor, the oracle VM, the f64 per-gate executor's stored results at 30 q and, where oracle/_ref is built,
the reference's own CUDA library, at north_star's 1e-5 (f32)."""
import gc
import importlib
import os

import numpy as np
import pytest

from oracle import ref_replay as rr
from oracle.circuit import OracleCircuit, vjp
from test_oracle import autodiff_gates, build_autodiff_circuit, tsallis_loss_and_cotangents

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _max_rel(got, ref):
    scale = max(float(np.abs(r).max()) for r in ref)
    return max(float(np.abs(np.asarray(g).reshape(-1) - np.asarray(r).reshape(-1)).max()) for g, r in zip(got, ref)) / scale


def _brickwork(n, depth, options):
    bench = importlib.import_module("bench")
    from quantum_differentiable_circuit import Circuit
    var, cts = bench.brickwork_inputs(n, depth, np.complex64)
    c = Circuit(n, precision="f32")
    for k, v in options:
        c.set_option(k, v)
    c.set_option("profile", 1)
    bench.build_brickwork(c, n, depth)
    dens = [np.array(d) for d in c.forward([], var)]
    prof_f = c.last_profile()
    grads = [np.array(g) for g in c.backward([x.conj() for x in cts], [], var)]
    prof_b = c.last_profile()
    init = np.zeros(1 << n, dtype=np.complex64); init[0] = 1
    back = float(np.abs(c.get_cpu_state_copy() - init).max())
    del c
    gc.collect()
    return dens, grads, prof_f, prof_b, back


@pytest.mark.parametrize("n,depth,extra", [(16, 10, ()), (22, 12, ()), (16, 10, (("tc_rev", 0),)), (20, 12, (("tc_products", 6),))])
def test_tc_brickwork_equals_per_gate_executor(pkg, n, depth, extra):
    """Default: the fused one-sweep reverse step (tc_rev.cuh); tc_rev = 0: the three-sweep form; tc_products = 6."""
    dens0, grads0, _, _, _ = _brickwork(n, depth, (("fuse", 0),))
    dens, grads, pf, pb, back = _brickwork(n, depth, (("tc", 1),) + tuple(extra))
    assert pf.get("tc_fwd", {}).get("launches", 0) > 0 and pb.get("tc_bwd", {}).get("launches", 0) > 0, \
        "the tensor-core blocks must be the ones that ran"
    assert _max_rel(dens, dens0) < TOL and _max_rel(grads, grads0) < TOL, (_max_rel(dens, dens0), _max_rel(grads, grads0))
    assert back < TOL      # every block un-computed: the working state is |0..0> again


def test_tc_every_instruction_kind_matches_oracle(pkg):
    """Circuit of src/test_autodiff.py:51-81: NonU windows fall back to the FP32 tile kernels, one-qubit, diagonal and
    constant gates ride inside the blocks, densities interleave with the gates."""
    from quantum_differentiable_circuit import Circuit
    n, layers = 15, 2
    rng = np.random.default_rng(42)
    c = Circuit(n, precision="f32")
    c.set_option("tc", 1)
    c.set_option("profile", 1)
    o = OracleCircuit(n)
    build_autodiff_circuit(c, n, layers)
    build_autodiff_circuit(o, n, layers)
    const, var = autodiff_gates(rng, n, layers, np.complex64)
    dens, dens_o = c.forward(const, var), o.forward(const, var)
    assert _max_rel(dens, dens_o) < TOL
    _, cts = tsallis_loss_and_cotangents(dens_o)
    grads_o = vjp(o, var, const, cts)
    grads = c.backward([np.asarray(ct, dtype=np.complex64).conj() for ct in cts], const, var)
    assert [g.size for g in grads] == [g.size for g in grads_o]
    assert _max_rel(grads, grads_o) < TOL, _max_rel(grads, grads_o)


def test_tc_mixed_gate_kinds_in_blocks_match_oracle(pkg):
    """Unitary one-qubit, dense, diagonal, constant and variable gates riding INSIDE tensor-core blocks (also on
    qubits 0..2), densities between the layers: every gradient layout of the chain rule against the oracle VM."""
    from quantum_differentiable_circuit import Circuit
    from conftest import haar_unitary
    n = 15
    rng = np.random.default_rng(3)
    c = Circuit(n, precision="f32")
    c.set_option("tc", 1)
    c.set_option("profile", 1)
    o = OracleCircuit(n)
    const, var = [], []
    for layer in range(6):
        for q in range(n):
            kind = (q + layer) % 4
            for x in (c, o):
                (x.add_q1_var_gate if kind < 2 else x.add_q1_const_gate)(q)
            (var if kind < 2 else const).append(haar_unitary(rng, 2, np.complex64))
        for q in range(layer % 2, n - 1, 2):
            kind = (q // 2 + layer) % 4
            a, b = (q + 1, q) if (q // 2) % 2 else (q, q + 1)
            if kind == 0:
                for x in (c, o):
                    x.add_q2_var_gate(a, b)
                var.append(haar_unitary(rng, 4, np.complex64))
            elif kind == 1:
                for x in (c, o):
                    x.add_q2_var_gate_diag(a, b)
                var.append(np.exp(1j * rng.normal(size=4)).astype(np.complex64))
            elif kind == 2:
                for x in (c, o):
                    x.add_q2_const_gate(a, b)
                const.append(haar_unitary(rng, 4, np.complex64))
            else:
                for x in (c, o):
                    x.add_q2_const_gate_diag(a, b)
                const.append(np.exp(1j * rng.normal(size=4)).astype(np.complex64))
        if layer in (2, 5):
            for q in range(0, n - 1, 3):
                for x in (c, o):
                    x.get_q2_dens_op_with_grad(q + 1, q)
            for x in (c, o):
                x.get_q1_dens_op_with_grad(n - 1)
    dens, dens_o = c.forward(const, var), o.forward(const, var)
    assert c.last_profile().get("tc_fwd", {}).get("launches", 0) > 0, "tensor-core blocks must have run"
    assert _max_rel(dens, dens_o) < TOL
    _, cts = tsallis_loss_and_cotangents(dens_o)
    grads_o = vjp(o, var, const, cts)
    grads = c.backward([np.asarray(ct, dtype=np.complex64).conj() for ct in cts], const, var)
    assert c.last_profile().get("tc_bwd", {}).get("launches", 0) > 0
    assert [g.size for g in grads] == [g.size for g in grads_o]
    assert _max_rel(grads, grads_o) < TOL, _max_rel(grads, grads_o)


def test_tc_vqse_equals_per_gate_executor(pkg):
    """Diagonal ZZ ring + X rotations (example_vqse_ising.py) at 21 qubits: diagonal and one-qubit gates inside blocks."""
    from quantum_differentiable_circuit import Circuit
    from test_circuit_gpu import build_vqse, tfim_h, vqse_gates
    n, layers = 21, 3
    rng = np.random.default_rng(7)
    gates = vqse_gates(rng.normal(size=2 * layers), n, np.complex64)
    h = tfim_h(np.complex64)
    init = (np.ones(1 << n) / np.sqrt(1 << n)).astype(np.complex64)
    out = {}
    for key, opts in ((0, (("fuse", 0),)), (1, (("tc", 1),))):
        c = Circuit(n, precision="f32")
        for k, v in opts:
            c.set_option(k, v)
        c.set_state_from_vector(init)
        build_vqse(c, n, layers)
        dens = c.forward([], gates)
        grads = c.backward([h.T.copy().conj() for _ in dens], [], gates)
        out[key] = (dens, grads)
    assert _max_rel(out[1][0], out[0][0]) < TOL and _max_rel(out[1][1], out[0][1]) < TOL


def test_tc_matches_the_unmodified_reference_at_30q(pkg):
    """30 q brickwork depth 8 through the tensor-core blocks against the f64 per-gate streaming executor's results for
    the same complex64 inputs, stored in tests/golden/brickwork_30q_f64.npz (tests/golden/make_brickwork_golden.py),
    and against the reference's own library (4 x 8 GiB) where oracle/_ref is built."""
    import torch
    live = rr.ref_available("f32")
    need = 52 if live else 20
    if torch.cuda.mem_get_info()[0] / 2.0 ** 30 < need:
        pytest.skip(f"needs {need} GiB of free device memory")
    n, depth = 30, 8
    dens, grads, pf, pb, _ = _brickwork(n, depth, (("tc", 1),))
    assert pf.get("tc_fwd", {}).get("launches", 0) > 0
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "brickwork_30q_f64.npz"))
    dens_s, grads_s = list(z["depth8/f32/densities"]), list(z["depth8/f32/gradients"])
    assert _max_rel(dens, dens_s) < TOL and _max_rel(grads, grads_s) < TOL, (_max_rel(dens, dens_s), _max_rel(grads, grads_s))
    if live:
        bench = importlib.import_module("bench")
        var, cts = bench.brickwork_inputs(n, depth, np.complex64)
        r = rr.RefCircuit(n, "f32")
        bench.build_brickwork(r, n, depth)
        dens_r = r.forward([], var)
        grads_r = r.backward([x.conj() for x in cts], [], var)
        r.state_t.drop(); r.initial_t.drop()
        assert _max_rel(dens, dens_r) < TOL and _max_rel(grads, grads_r) < TOL, (_max_rel(dens, dens_r), _max_rel(grads, grads_r))

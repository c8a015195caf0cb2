"""GPU: diagonal gates on k = 1..6 qubits (add_const_gate_diag / add_var_gate_diag / *_nonu, kinds 20..23) against the
oracle VM in both precisions and every executor, the un-computed state, the k = 2 unitary builders against the
two-qubit diagonal, run-to-run identical gradients, rejected inputs, finite differences, the torch glue with gate
tensors on the GPU, a 30-qubit register checked against the dense k-qubit gate on diag(d), and a 2-GPU sharded
register with diagonals on the global qubit."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import TOL, haar_unitary
from oracle.circuit import vjp
from oracle.kdiag import KDiagOracleCircuit
from test_diag_k import apply_dops, dops_gates, kdiag_ops

pytestmark = pytest.mark.gpu

# positions of the k = 1..6 diagonals of a case (n qubits): inside the low tile lanes (0..3 included), at the top of
# the register, mixed and unsorted; "small" is a register that fits one tile
CASES = {
    "low": (14, [[0], [1, 0], [2, 0, 1], [3, 1, 0, 2], [0, 2, 4, 1, 3], [5, 4, 3, 2, 1, 0]]),
    "high": (15, [[14], [13, 14], [14, 12, 13], [14, 13, 11, 10], [10, 14, 12, 11, 13], [9, 14, 10, 13, 11, 12]]),
    "mixed": (16, [[15], [0, 15], [15, 0, 7], [1, 14, 5, 0], [15, 2, 0, 13, 6], [0, 15, 3, 14, 1, 8]]),
    "small": (9, [[8], [8, 0], [8, 0, 5], [2, 8, 4, 7], [0, 1, 2, 3, 4], [8, 7, 0, 1, 6, 3]]),
}


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max()


def _check_circuit(c, n, dpos, precision, seed=7):
    """run / forward / backward of the diagonal program against KDiagOracleCircuit, relative to the largest entry, and
    the un-computed working state."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    tol = TOL[np.dtype(dtype)]
    ops = kdiag_ops(n, dpos)
    rng = np.random.default_rng(seed)
    const, var = dops_gates(rng, ops)
    o = KDiagOracleCircuit(n)
    apply_dops(o, ops)
    dens_all_o, dens_o = o.run(const, var), o.forward(const, var)
    cts = [rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape) for d in dens_o]
    grads_o = vjp(o, var, const, cts)
    apply_dops(c, ops)
    cg, vg = [g.astype(dtype) for g in const], [g.astype(dtype) for g in var]
    for a, b in zip(c.run(cg, vg), dens_all_o):
        assert a.shape == b.shape and _rel(a, b) < tol
    dens = c.forward(cg, vg)
    assert [d.shape for d in dens] == [d.shape for d in dens_o]
    for a, b in zip(dens, dens_o):
        assert _rel(a, b) < tol
    grads = c.backward([ct.conj().astype(dtype) for ct in cts], cg, vg)
    assert [g.shape for g in grads] == [g.shape for g in grads_o]
    scale = max(np.abs(g).max() for g in grads_o)
    err = max(np.abs(a - b).max() for a, b in zip(grads, grads_o)) / scale
    assert err < tol, err
    assert grads[-1].shape == (8,) and not grads[-1].any()   # the diagonal after the last differentiable density
    # backward un-computed every gate: the working state is |0..0> again
    state = c.get_cpu_state_copy()
    init = np.zeros_like(state)
    init[0] = 1
    assert np.abs(state - init).max() < 10 * tol
    return c


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("fuse", [0, 1, 2])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_diagonals_match_oracle(pkg, case, fuse, precision):
    n, dpos = CASES[case]
    c = pkg.Circuit(n, precision=precision)
    c.set_option("fuse", fuse)
    c.set_option("tc", 0)
    c.set_option("profile", 1)
    _check_circuit(c, n, dpos, precision)
    prof = c.last_profile()
    assert prof["diag_k_rev"]["launches"] > 0


@pytest.mark.parametrize("case", ["low", "high", "mixed"])
def test_diagonals_border_tensor_core_blocks(pkg, case):
    """f32 with the tensor-core 6-qubit blocks forced on: the blocks end and start at the diagonals."""
    n, dpos = CASES[case]
    c = pkg.Circuit(n, precision="f32")
    c.set_option("tc", 1)
    c.set_option("profile", 1)
    _check_circuit(c, n, dpos, "f32")
    prof = c.last_profile()
    assert prof.get("tc_bwd", {}).get("launches", 0) + prof.get("tc_fwd", {}).get("launches", 0) > 0
    assert prof.get("diag_k_rev", {}).get("launches", 0) > 0


def _program(c, n, new):
    for i in range(n):
        c.add_q1_var_gate(i)
    if new:
        c.add_var_gate_diag([3, 9]); c.add_const_gate_diag([12, 0]); c.add_var_gate_diag([1, 2])
    else:
        c.add_q2_var_gate_diag(3, 9); c.add_q2_const_gate_diag(12, 0); c.add_q2_var_gate_diag(1, 2)
    c.add_var_gate_diag_nonu([5, 0, 11])
    c.get_q1_dens_op_with_grad(5)
    c.get_dens_op_with_grad([12, 3, 9])


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_k2_unitary_builders_are_the_q2_diag_kinds(pkg, precision):
    """add_*_gate_diag([p2, p1]) adds the two-qubit diagonal kinds: bit-identical outputs and gradients."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    n = 13
    rng = np.random.default_rng(11)
    ph = lambda m: np.exp(1j * rng.uniform(0, 6.3, size=m)).astype(dtype)  # noqa: E731
    var = [haar_unitary(rng, 2, dtype) for _ in range(n)] + [ph(4), ph(4), (ph(8) * 1.02).astype(dtype)]
    const = [ph(4)]
    cts = [(rng.normal(size=(s, s)) + 1j * rng.normal(size=(s, s))).astype(dtype) for s in (2, 8)]
    out = []
    for new in (False, True):
        c = pkg.Circuit(n, precision=precision)
        _program(c, n, new)
        assert c._kinds[n:n + 4] == [5, 4, 5, 23]
        out.append((c.run(const, var), c.forward(const, var), c.backward(cts, const, var)))
    for a, b in zip(out[0], out[1]):
        assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_gradients_are_identical_run_to_run(pkg, precision):
    n, dpos = CASES["mixed"]
    dtype = np.complex64 if precision == "f32" else np.complex128
    ops = kdiag_ops(n, dpos)
    const, var = dops_gates(np.random.default_rng(3), ops, dtype)
    c = pkg.Circuit(n, precision=precision)
    apply_dops(c, ops)
    out = []
    for _ in range(2):
        dens = c.forward(const, var)
        out.append(c.backward([np.ones_like(d) for d in dens], const, var))
    assert all(np.array_equal(x, y) for x, y in zip(out[0], out[1]))


def test_bad_inputs_are_errors(pkg):
    from quantum_differentiable_circuit import QdcError
    c = pkg.Circuit(8, precision="f64")
    for pos, msg in (([1, 1, 2], "must be different"), ([0, 3, 4, 0], "must be different"),
                     ([0, 1, 8], "out of the bound"), ([], "1..6"), (list(range(7)), "1..6")):
        for name in ("add_const_gate_diag", "add_var_gate_diag", "add_const_gate_diag_nonu", "add_var_gate_diag_nonu"):
            with pytest.raises(QdcError, match=msg):
                getattr(c, name)(pos)
    for kind in (20, 21, 22, 23):
        with pytest.raises(QdcError, match="qdc_circuit_add_gate_diag"):
            c._add(kind, 0, 1)
    assert c._count(0) == 0
    # a diagonal takes 2^k entries; a zero entry of a NonU diagonal fails the un-compute with the inverse's text
    c.add_var_gate_diag_nonu([5, 0, 2])
    c.get_dens_op_with_grad([5, 0, 2])
    d = np.exp(1j * np.arange(8.0))
    with pytest.raises(QdcError, match="Incorrect len"):
        c.forward([], [d[:4]])
    with pytest.raises(QdcError, match="Incorrect len"):
        c.forward([], [np.diag(d).reshape(-1)])
    assert c._count(7) == 8
    d[3] = 0
    c.forward([], [d])
    with pytest.raises(QdcError, match=r"U\(4, 4\) is zero"):
        c.backward([np.eye(8, dtype=np.complex128)], [], [d])


def test_finite_difference_f64(pkg):
    """The test_autodiff_finite_difference_f64 recipe (n = 15, 8th-order central difference, rel 1e-9 of the terms)
    with unitary and NonU variable diagonals (k = 1..6) and the purity loss sum tr rho^2."""
    from qdc import AutoGradCircuit
    n, eta = 15, 1e-5
    dpos = [[14], [3, 12], [14, 3, 0], [2, 13, 7, 0], [1, 6, 12, 4, 0], [5, 0, 14, 9, 10, 3]]
    ops = [op if op[0] != "kd" else (op[0], op[1], True, op[3]) for op in kdiag_ops(n, dpos)]
    rng = np.random.default_rng(42)
    c = AutoGradCircuit(n, precision="f64")
    apply_dops(c.circuit, ops)
    const, var = dops_gates(rng, ops)
    pert = [rng.normal(size=v.size) + 1j * rng.normal(size=v.size) for v in var]
    _, run = c.build()

    def loss_and_cts(dens):
        return sum(np.einsum("ij,ji->", d, d).real for d in dens), [2.0 * d.T for d in dens]

    def loss_at(s):
        return loss_and_cts(run([v + s * eta * p for v, p in zip(var, pert)], const))[0]

    fd = (loss_at(-4) / 280 - loss_at(4) / 280 - 4 * loss_at(-3) / 105 + 4 * loss_at(3) / 105
          + loss_at(-2) / 5 - loss_at(2) / 5 - 4 * loss_at(-1) / 5 + 4 * loss_at(1) / 5) / eta
    _, cts = loss_and_cts(run(var, const))
    grads = run.vjp(var, const, cts)
    assert {2, 8, 16, 32, 64} <= {g.size for g in grads}
    terms = [(g @ p).real for g, p in zip(grads, pert)]
    assert abs(sum(terms) - fd) / sum(abs(t) for t in terms) < 1e-9


def test_torch_autograd_glue(pkg):
    """autodiff_run with gate tensors on the GPU: torch.autograd equals the raw vjp, gradients land on the device."""
    import torch
    from qdc import AutoGradCircuit
    n = 13
    rng = np.random.default_rng(3)
    c = AutoGradCircuit(n, precision="f64")
    for i in range(n):
        c.add_q1_var_gate(i)
    c.add_var_gate_diag([12, 0, 6, 3])
    c.add_const_gate_diag([1, 2, 11])
    c.add_var_gate_diag_nonu([4, 9])
    c.add_var_gate_diag([7])
    c.get_dens_op_with_grad([12, 0, 6])
    c.get_q2_dens_op_with_grad(5, 9)
    var = ([haar_unitary(rng, 2) for _ in range(n)] + [np.exp(1j * rng.normal(size=16)),
                                                      1.05 * np.exp(1j * rng.normal(size=4)),
                                                      np.exp(1j * rng.normal(size=2))])
    const = [np.exp(1j * rng.normal(size=8))]
    _, run = c.build()
    tv = [torch.tensor(v, requires_grad=True, device="cuda") for v in var]
    dens = run(tv, [torch.tensor(g, device="cuda") for g in const])
    assert [tuple(d.shape) for d in dens] == [(8, 8), (4, 4)] and dens[0].is_cuda
    loss = sum(torch.einsum("ij,ji->", d, d).real for d in dens)
    loss.backward()
    dens_np = run.forward(var, const)
    grads = run.vjp(var, const, [2.0 * d.T for d in dens_np])
    assert [g.size for g in grads[n:]] == [16, 4, 2]
    for t, g in zip(tv, grads):
        assert t.grad.is_cuda
        np.testing.assert_allclose(t.grad.cpu().numpy(), g.conj(), rtol=1e-10, atol=1e-12)


def test_30_qubits_diagonal_equals_the_dense_gate(pkg):
    """n = 30, f32 with default options: every diagonal (k = 1..6, low, high and mixed positions) against the dense
    k-qubit gate on diag(d): densities within 1e-5 and the gradient equal to the diagonal of the dense gradient within
    1e-5 (relative to the largest entry)."""
    dtype = np.complex64
    n = 30
    rng = np.random.default_rng(30)
    dpos = [[29], [0, 17], [29, 2, 0], [3, 1, 2, 0], [28, 27, 26, 25, 24], [0, 29, 14, 3, 27, 8]]
    var = [haar_unitary(rng, 2, dtype) for _ in range(n)] + [haar_unitary(rng, 4, dtype) for _ in range(0, n - 1, 2)]
    ds = [np.exp(1j * rng.uniform(0, 6.3, size=1 << len(p))).astype(dtype) for p in dpos]
    cts = None

    def run(diag):
        nonlocal cts
        c = pkg.Circuit(n, precision="f32")
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(0, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        for p in dpos:
            (c.add_var_gate_diag if diag else c.add_var_gate)(p)
        c.get_dens_op_with_grad([29, 0, 5])
        c.get_q2_dens_op_with_grad(17, 22)
        vv = var + (ds if diag else [np.diag(d).reshape(-1) for d in ds])
        dens = c.forward([], vv)
        if cts is None:
            cts = [(rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)).astype(dtype) for d in dens]
        grads = c.backward(cts, [], vv)
        del c
        return dens, grads

    dens_d, g_d = run(True)
    dens_u, g_u = run(False)
    for x, y in zip(dens_d, dens_u):
        assert _rel(x, y) < 1e-5
    m = len(var)
    sc = max(np.abs(g).max() for g in g_u)
    assert max(np.abs(x - y).max() for x, y in zip(g_d[:m], g_u[:m])) / sc < 1e-5
    for gd, gu, p in zip(g_d[m:], g_u[m:], dpos):
        dim = 1 << len(p)
        assert _rel(gd, np.diag(gu.reshape(dim, dim))) < 1e-5


# ------------------------------------------------------------------------------------------------ sharded, world 2
def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, precision, q):
    try:
        _worker_body(rank, world, port, precision, q)
    except BaseException as e:  # noqa: BLE001
        import traceback
        q.put((rank, "error", f"{type(e).__name__}: {e}\n{traceback.format_exc()}"))
        raise


def _worker_body(rank, world, port, precision, q):
    import importlib
    import torch
    import torch.distributed as dist
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    pkg = importlib.import_module("differentiable-quantum-circuit-cuda_b200")
    sharded = importlib.import_module("differentiable-quantum-circuit-cuda_b200.sharded")
    from conftest import haar_unitary as hu
    dtype = np.complex64 if precision == "f32" else np.complex128
    n = 15
    rng = np.random.default_rng(9)
    # every gate and density on the local qubits 0..13; the diagonals hold the global qubit 14 (k = 1..6)
    dpos = [[14], [14, 3], [2, 14, 0], [14, 3, 9, 0], [0, 5, 14, 1, 8], [6, 14, 2, 12, 10, 0]]
    var = [hu(rng, 2, dtype) for _ in range(14)] + [hu(rng, 4, dtype) for _ in range(0, 13, 2)]
    ds = [(np.exp(1j * rng.uniform(0, 6.3, size=1 << len(p))) * (1.03 if j % 2 else 1)).astype(dtype)
          for j, p in enumerate(dpos)]
    out = []
    for c in (sharded.ShardedCircuit(n, precision=precision), pkg.Circuit(n, precision=precision)):
        c.set_option("profile", 1)
        for layer in range(2):
            for i in range(14):
                c.add_q1_var_gate(i)
            for i in range(layer % 2, 13, 2):
                c.add_q2_var_gate(i + 1, i)
            for j, p in enumerate(dpos):
                (c.add_var_gate_diag_nonu if j % 2 else c.add_var_gate_diag)(p)
            c.get_dens_op_with_grad([3, 0, 9])
            c.get_q1_dens_op_with_grad(layer)
        vv = []
        for layer in range(2):
            vv += var[:14] + [var[14 + (i - layer % 2) // 2] for i in range(layer % 2, 13, 2)] + ds
        run = c.run([], vv)
        fwd = c.forward([], vv)
        r2 = np.random.default_rng(4)
        cts = [(r2.normal(size=d.shape) + 1j * r2.normal(size=d.shape)).astype(dtype) for d in fwd]
        out.append((run, fwd, c.backward(cts, [], vv)))
        if len(out) == 1:
            assert "exchange" not in c.last_profile(), c.last_profile()
    errs = []
    for a, b in zip(out[0], out[1]):
        sc = max(np.abs(x).max() for x in b)
        errs.append(max(np.abs(x - y).max() for x, y in zip(a, b)) / sc)
    q.put((rank, "ok", errs))
    dist.destroy_process_group()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_sharded_diagonals_on_the_global_qubit(precision):
    import torch.multiprocessing as mp
    world = 2
    if _ngpus() < world:
        pytest.skip(f"needs >= {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, precision, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=300) for _ in range(world)]
    assert not any(r[1] == "error" for r in results), [r[2] for r in results if r[1] == "error"]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    tol = 1e-5 if precision == "f32" else 1e-12
    for rank, _, errs in results:
        assert max(errs) < tol, (rank, errs)

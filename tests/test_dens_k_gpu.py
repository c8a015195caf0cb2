"""GPU: reduced density matrices on k = 3..6 qubits (get_dens_op / get_dens_op_with_grad, kinds DENS_K / DIFF_DENS_K)
against the oracle VM in both precisions, the k <= 2 builders against the existing kinds, finite differences, the torch
glue, a 30-qubit register, and a 2-GPU sharded register."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import TOL, haar_unitary
from oracle.circuit import vjp
from oracle.kdens import KOracleCircuit

pytestmark = pytest.mark.gpu

# positions of the k = 3, 4, 5, 6 densities of a case (n qubits): inside the low tile lanes, at the top of the
# register, mixed and unsorted; "small" is a register that fits one tile (loaded as it is)
CASES = {
    "low": (14, [[2, 0, 1], [3, 1, 0, 2], [0, 2, 4, 1, 3], [5, 4, 3, 2, 1, 0]]),
    "high": (15, [[14, 12, 13], [14, 13, 11, 10], [10, 14, 12, 11, 13], [9, 14, 10, 13, 11, 12]]),
    "mixed": (16, [[15, 0, 7], [1, 14, 5, 0], [15, 2, 0, 13, 6], [0, 15, 3, 14, 1, 8]]),
    "small": (9, [[8, 0, 5], [2, 8, 4, 7], [0, 1, 2, 3, 4], [8, 7, 0, 1, 6, 3]]),
}


def _program(c, n, kpos):
    """Two layers of one-qubit, dense two-qubit and NonU gates, with k-qubit densities interleaved with one- and
    two-qubit ones, differentiable and not."""
    for layer in range(2):
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(layer, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        c.get_dens_op_with_grad(kpos[2 * layer])
        c.get_q2_dens_op_with_grad(n - 1, 0)
        c.get_dens_op(kpos[3 - layer])
        for i in range(1 - layer, n - 1, 2):
            c.add_q2_const_gate_nonu(i + 1, i)
        for i in range(n):
            c.add_q1_var_gate_nonu(i)
        c.get_q1_dens_op(layer)
        c.get_dens_op_with_grad(kpos[2 * layer + 1])
        c.get_q1_dens_op_with_grad(n - 1 - layer)


def _gates(rng, n):
    rc = lambda k: rng.normal(size=k * k) + 1j * rng.normal(size=k * k)  # noqa: E731
    const, var = [], []
    for layer in range(2):
        var += [haar_unitary(rng, 2) for _ in range(n)]
        var += [haar_unitary(rng, 4) for _ in range(layer, n - 1, 2)]
        const += [0.01 * rc(4) + haar_unitary(rng, 4) for _ in range(1 - layer, n - 1, 2)]
        var += [0.01 * rc(2) + haar_unitary(rng, 2) for _ in range(n)]
    return const, var


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max()


def _oracle(n, kpos, rng):
    const, var = _gates(rng, n)
    o = KOracleCircuit(n)
    _program(o, n, kpos)
    dens_all = o.run(const, var)
    dens = o.forward(const, var)
    cts = [rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape) for d in dens]
    grads = vjp(o, var, const, cts)
    return const, var, dens_all, dens, cts, grads


def _check_circuit(pkg, c, n, kpos, precision, rng_seed=7):
    dtype = np.complex64 if precision == "f32" else np.complex128
    tol = TOL[np.dtype(dtype)]
    const, var, dens_all_o, dens_o, cts, grads_o = _oracle(n, kpos, np.random.default_rng(rng_seed))
    _program(c, n, kpos)
    cg, vg = [g.astype(dtype) for g in const], [g.astype(dtype) for g in var]
    dens_all = c.run(cg, vg)
    assert [d.shape for d in dens_all] == [d.shape for d in dens_all_o]
    for a, b in zip(dens_all, dens_all_o):
        assert _rel(a, b) < tol
    dens = c.forward(cg, vg)
    assert [d.shape for d in dens] == [d.shape for d in dens_o]
    for a, b in zip(dens, dens_o):
        assert _rel(a, b) < tol
    grads = c.backward([ct.conj().astype(dtype) for ct in cts], cg, vg)
    scale = max(np.abs(g).max() for g in grads_o)
    err = max(np.abs(a - b).max() for a, b in zip(grads, grads_o)) / scale
    assert err < tol, err
    # backward un-computed every gate: the working state is |0..0> again
    state = c.get_cpu_state_copy()
    init = np.zeros_like(state)
    init[0] = 1
    assert np.abs(state - init).max() < 10 * tol
    return c


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("fuse", [0, 1, 2])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_k_densities_match_oracle(pkg, case, fuse, precision):
    n, kpos = CASES[case]
    c = pkg.Circuit(n, precision=precision)
    c.set_option("fuse", fuse)
    c.set_option("tc", 0)
    _check_circuit(pkg, c, n, kpos, precision)


@pytest.mark.parametrize("case", ["low", "high", "mixed"])
def test_k_densities_border_tensor_core_blocks(pkg, case):
    """f32 with the tensor-core 6-qubit blocks forced on: the blocks end and start at the k-density barriers."""
    n, kpos = CASES[case]
    c = pkg.Circuit(n, precision="f32")
    c.set_option("tc", 1)
    c.set_option("profile", 1)
    _check_circuit(pkg, c, n, kpos, "f32")
    assert c.last_profile().get("tc_bwd", {}).get("launches", 0) + c.last_profile().get("tc_fwd", {}).get(
        "launches", 0) > 0


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_k1_and_k2_builders_are_the_existing_kinds(pkg, precision):
    """get_dens_op([p]) / get_dens_op([p2, p1]) add Q1_DENS / Q2_DENS: bit-identical outputs and gradients."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    n = 13
    rng = np.random.default_rng(11)
    var = [haar_unitary(rng, 2, dtype) for _ in range(n)] + [haar_unitary(rng, 4, dtype) for _ in range(0, n - 1, 2)]
    cts = [(rng.normal(size=(s, s)) + 1j * rng.normal(size=(s, s))).astype(dtype) for s in (2, 4, 4, 2)]
    out = []
    for new in (False, True):
        c = pkg.Circuit(n, precision=precision)
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(0, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        if new:
            c.get_dens_op_with_grad([5]); c.get_dens_op_with_grad([12, 3]); c.get_dens_op_with_grad([0, 7])
            c.get_dens_op([2]); c.get_dens_op_with_grad([11])
        else:
            c.get_q1_dens_op_with_grad(5); c.get_q2_dens_op_with_grad(12, 3); c.get_q2_dens_op_with_grad(0, 7)
            c.get_q1_dens_op(2); c.get_q1_dens_op_with_grad(11)
        assert c._kinds[-5:] == [13, 12, 12, 11, 13]
        out.append((c.run([], var), c.forward([], var), c.backward(cts, [], var)))
    for a, b in zip(out[0], out[1]):
        assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_bad_inputs_are_errors(pkg):
    from quantum_differentiable_circuit import QdcError
    c = pkg.Circuit(8, precision="f64")
    for pos, msg in (([1, 1, 2], "must be different"), ([0, 3, 4, 0], "must be different"), ([0, 1, 8], "out of the bound"),
                     ([], "1..6"), (list(range(7)), "1..6")):
        with pytest.raises(QdcError, match=msg):
            c.get_dens_op(pos)
        with pytest.raises(QdcError, match=msg):
            c.get_dens_op_with_grad(pos)
    with pytest.raises(QdcError, match="qdc_circuit_add_dens"):
        c._add(14, 0, 1)
    with pytest.raises(QdcError, match="qdc_circuit_add_dens"):
        c._add(15, 0, 1)
    assert c._count(0) == 0


def test_finite_difference_f64(pkg):
    """The test_autodiff_finite_difference_f64 recipe (n = 15, 8th-order central difference, eta = 1e-6, rel 1e-9)
    with k = 3 and 5 differentiable densities and the purity loss sum tr rho^2."""
    from qdc import AutoGradCircuit
    n, eta = 15, 1e-6
    rng = np.random.default_rng(42)
    c = AutoGradCircuit(n, precision="f64")
    for layer in range(3):
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(layer % 2, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        for i in range(n):
            c.add_q1_var_gate_nonu(i)
        c.get_dens_op_with_grad([14, 3, 0] if layer != 1 else [2, 13, 7, 0, 9])
        c.get_dens_op_with_grad([1, 6, 12, 4, 0] if layer != 1 else [5, 0, 14])
    const = []
    rc = lambda k: rng.normal(size=k * k) + 1j * rng.normal(size=k * k)  # noqa: E731
    var = []
    for layer in range(3):
        var += [haar_unitary(rng, 2) for _ in range(n)]
        var += [haar_unitary(rng, 4) for _ in range(layer % 2, n - 1, 2)]
        var += [0.01 * rc(2) + haar_unitary(rng, 2) for _ in range(n)]
    pert = [rng.normal(size=v.size) + 1j * rng.normal(size=v.size) for v in var]
    _, run = c.build()

    def loss_and_cts(dens):
        return sum(np.einsum("ij,ji->", d, d).real for d in dens), [2.0 * d.T for d in dens]

    def loss_at(s):
        return loss_and_cts(run([v + s * eta * p for v, p in zip(var, pert)], const))[0]

    fd = (loss_at(-4) / 280 - loss_at(4) / 280 - 4 * loss_at(-3) / 105 + 4 * loss_at(3) / 105
          + loss_at(-2) / 5 - loss_at(2) / 5 - 4 * loss_at(-1) / 5 + 4 * loss_at(1) / 5) / eta
    dens = run(var, const)
    assert sorted({d.shape for d in dens}) == [(8, 8), (32, 32)]
    _, cts = loss_and_cts(dens)
    grads = run.vjp(var, const, cts)
    ds = sum((g @ p).real for g, p in zip(grads, pert))
    assert abs(ds - fd) / min(abs(ds), abs(fd)) < 1e-9


def test_torch_autograd_glue(pkg):
    """autodiff_run with a k-density loss: torch.autograd equals the raw vjp."""
    import torch
    from qdc import AutoGradCircuit
    n = 13
    rng = np.random.default_rng(3)
    c = AutoGradCircuit(n, precision="f64")
    for i in range(n):
        c.add_q1_var_gate(i)
    for i in range(0, n - 1, 2):
        c.add_q2_var_gate(i + 1, i)
    c.get_dens_op_with_grad([12, 0, 6, 3])
    c.get_q1_dens_op_with_grad(5)
    c.get_dens_op_with_grad([1, 2, 11])
    var = [haar_unitary(rng, 2) for _ in range(n)] + [haar_unitary(rng, 4) for _ in range(n // 2)]
    _, run = c.build()
    tv = [torch.tensor(v, requires_grad=True) for v in var]
    dens = run(tv, [])
    assert [tuple(d.shape) for d in dens] == [(16, 16), (2, 2), (8, 8)]
    loss = sum(torch.einsum("ij,ji->", d, d).real for d in dens)
    loss.backward()
    dens_np = run.forward(var, [])
    grads = run.vjp(var, [], [2.0 * d.T for d in dens_np])
    for t, g in zip(tv, grads):
        np.testing.assert_allclose(t.grad.numpy(), g.conj(), rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_30_qubits_four_qubit_density(pkg, precision):
    """n = 30 (f32 with default options, f64): a 4-qubit density over low and high positions.  Tracing out two of its
    qubits gives get_q2_dens_op, its trace is |psi|^2, it is Hermitian and positive semidefinite; with the cotangent
    C2 (x) I on the traced-out pair its gate gradients equal those of a q2 density on the kept pair with cotangent C2."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    tol = TOL[np.dtype(dtype)]
    n, pos = 30, [29, 1, 17, 0]          # kept pair (29, 1), traced out (17, 0)
    rng = np.random.default_rng(30)
    var = [haar_unitary(rng, 2, dtype) for _ in range(n)] + [haar_unitary(rng, 4, dtype) for _ in range(0, n - 1, 2)]
    c2 = (rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4))).astype(dtype)

    def build(c, with_k):
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(0, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        if with_k:
            c.get_dens_op_with_grad(pos)
            c.get_q2_dens_op(29, 1)
        else:
            c.get_q2_dens_op_with_grad(29, 1)

    c = pkg.Circuit(n, precision=precision)
    build(c, True)
    rho4, rho2 = c.run([], var)
    scale = np.abs(rho4).max()
    assert rho4.shape == (16, 16)
    traced = np.einsum("aibi->ab", rho4.reshape(4, 4, 4, 4).astype(np.complex128))
    assert np.abs(traced - rho2).max() / np.abs(rho2).max() < tol
    assert abs(np.trace(rho4) - 1.0) < 10 * tol     # unitary gates from |0..0>: |psi|^2 = 1
    assert np.abs(rho4 - rho4.conj().T).max() / scale < tol
    assert np.linalg.eigvalsh((rho4 + rho4.conj().T).astype(np.complex128) / 2).min() >= -tol * scale
    c.forward([], var)
    g_k = c.backward([np.kron(c2, np.eye(4, dtype=dtype))], [], var)
    del c
    c = pkg.Circuit(n, precision=precision)
    build(c, False)
    c.forward([], var)
    g_2 = c.backward([c2], [], var)
    del c
    sc = max(np.abs(g).max() for g in g_2)
    assert max(np.abs(a - b).max() for a, b in zip(g_k, g_2)) / sc < tol


# ------------------------------------------------------------------------------------------------ sharded, world 2
def _ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _worker(rank, world, port, precision, peer, q):
    try:
        _worker_body(rank, world, port, precision, peer, q)
    except BaseException as e:  # noqa: BLE001
        import traceback
        q.put((rank, "error", f"{type(e).__name__}: {e}\n{traceback.format_exc()}"))
        raise


def _worker_body(rank, world, port, precision, peer, q):
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
    dtype = np.complex64 if precision == "f32" else np.complex128
    n = 15
    # the k = 4 density holds the global qubit 14 (top physical position of the 2-rank register)
    kpos = [[2, 0, 14], [14, 3, 9, 0], [0, 5, 13, 1, 8], [6, 4, 2, 12, 10, 0]]
    const, var = _gates(np.random.default_rng(9), n)
    cg, vg = [g.astype(dtype) for g in const], [g.astype(dtype) for g in var]
    out = []
    for c in (sharded.ShardedCircuit(n, precision=precision), pkg.Circuit(n, precision=precision)):
        if isinstance(c, sharded.ShardedCircuit):
            c.set_option("peer", peer)
        _program(c, n, kpos)
        run = c.run(cg, vg)
        fwd = c.forward(cg, vg)
        rng = np.random.default_rng(4)
        cts = [(rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)).astype(dtype) for d in fwd]
        out.append((run, fwd, c.backward(cts, cg, vg)))
    errs = []
    for a, b in zip(out[0], out[1]):
        sc = max(np.abs(x).max() for x in b)
        errs.append(max(np.abs(x - y).max() for x, y in zip(a, b)) / sc)
    q.put((rank, "ok", errs))
    dist.destroy_process_group()


@pytest.mark.parametrize("peer", [1, 0])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_sharded_k_density_on_the_global_qubit(precision, peer):
    import torch.multiprocessing as mp
    world = 2
    if _ngpus() < world:
        pytest.skip(f"needs >= {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, precision, peer, q)) for r in range(world)]
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

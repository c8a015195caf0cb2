"""GPU: gates on k = 3..6 qubits (add_const_gate / add_var_gate / *_nonu, kinds 16..19) against the oracle VM in both
precisions and every executor, the k <= 2 builders against the existing kinds, rejected inputs, finite differences,
the torch glue with gate tensors on the GPU, a 30-qubit register checked against two-qubit gates, and a 2-GPU sharded
register."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import TOL, haar_unitary
from oracle.circuit import vjp
from oracle.kgates import KGateOracleCircuit
from test_gate_k import apply_ops, kgate_ops, ops_gates

pytestmark = pytest.mark.gpu

# positions of the k = 3, 4, 5, 6 gates of a case (n qubits): inside the low tile lanes, at the top of the register,
# mixed and unsorted; "small" is a register that fits one tile (loaded as it is)
CASES = {
    "low": (14, [[2, 0, 1], [3, 1, 0, 2], [0, 2, 4, 1, 3], [5, 4, 3, 2, 1, 0]]),
    "high": (15, [[14, 12, 13], [14, 13, 11, 10], [10, 14, 12, 11, 13], [9, 14, 10, 13, 11, 12]]),
    "mixed": (16, [[15, 0, 7], [1, 14, 5, 0], [15, 2, 0, 13, 6], [0, 15, 3, 14, 1, 8]]),
    "small": (9, [[8, 0, 5], [2, 8, 4, 7], [0, 1, 2, 3, 4], [8, 7, 0, 1, 6, 3]]),
}


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max()


def _check_circuit(c, n, kpos, precision, seed=7):
    """run / forward / backward of the k-gate program against KGateOracleCircuit, relative to the largest entry, and
    the un-computed working state."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    tol = TOL[np.dtype(dtype)]
    ops = kgate_ops(n, kpos)
    rng = np.random.default_rng(seed)
    const, var = ops_gates(rng, ops)
    o = KGateOracleCircuit(n)
    apply_ops(o, ops)
    dens_all_o, dens_o = o.run(const, var), o.forward(const, var)
    cts = [rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape) for d in dens_o]
    grads_o = vjp(o, var, const, cts)
    apply_ops(c, ops)
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
    assert [g.shape for g in grads] == [g.shape for g in grads_o]
    scale = max(np.abs(g).max() for g in grads_o)
    err = max(np.abs(a - b).max() for a, b in zip(grads, grads_o)) / scale
    assert err < tol, err
    assert not grads[-1].any()     # the k-qubit gate after the last differentiable density
    # backward un-computed every gate: the working state is |0..0> again
    state = c.get_cpu_state_copy()
    init = np.zeros_like(state)
    init[0] = 1
    assert np.abs(state - init).max() < 10 * tol
    return c


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("fuse", [0, 1, 2])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_k_gates_match_oracle(pkg, case, fuse, precision):
    n, kpos = CASES[case]
    c = pkg.Circuit(n, precision=precision)
    c.set_option("fuse", fuse)
    c.set_option("tc", 0)
    c.set_option("profile", 1)
    _check_circuit(c, n, kpos, precision)
    prof = c.last_profile()
    assert prof["gate_k_rev"]["launches"] > 0


@pytest.mark.parametrize("case", ["low", "high", "mixed"])
def test_k_gates_border_tensor_core_blocks(pkg, case):
    """f32 with the tensor-core 6-qubit blocks forced on: the blocks end and start at the k-qubit gates."""
    n, kpos = CASES[case]
    c = pkg.Circuit(n, precision="f32")
    c.set_option("tc", 1)
    c.set_option("profile", 1)
    _check_circuit(c, n, kpos, "f32")
    prof = c.last_profile()
    assert prof.get("tc_bwd", {}).get("launches", 0) + prof.get("tc_fwd", {}).get("launches", 0) > 0
    assert prof.get("gate_k_rev", {}).get("launches", 0) > 0


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_k1_and_k2_builders_are_the_existing_kinds(pkg, precision):
    """add_*_gate([p]) / add_*_gate([p2, p1]) add the Q1 / Q2 kinds: bit-identical outputs and gradients."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    n = 13
    rng = np.random.default_rng(11)
    pert = lambda d: (0.01 * (rng.normal(size=d * d) + 1j * rng.normal(size=d * d))).astype(dtype)  # noqa: E731
    const = [haar_unitary(rng, 2, dtype), haar_unitary(rng, 4, dtype) + pert(4), haar_unitary(rng, 4, dtype)]
    var = ([haar_unitary(rng, 2, dtype) for _ in range(n)] + [haar_unitary(rng, 2, dtype) + pert(2)]
           + [haar_unitary(rng, 4, dtype) for _ in range(0, n - 1, 2)] + [haar_unitary(rng, 4, dtype) + pert(4)])
    cts = [(rng.normal(size=(s, s)) + 1j * rng.normal(size=(s, s))).astype(dtype) for s in (2, 4)]
    out = []
    for new in (False, True):
        c = pkg.Circuit(n, precision=precision)
        if new:
            for i in range(n):
                c.add_var_gate([i])
            c.add_const_gate([3]); c.add_var_gate_nonu([7])
            for i in range(0, n - 1, 2):
                c.add_var_gate([i + 1, i])
            c.add_const_gate_nonu([2, 9]); c.add_var_gate_nonu([12, 0]); c.add_const_gate([5, 11])
        else:
            for i in range(n):
                c.add_q1_var_gate(i)
            c.add_q1_const_gate(3); c.add_q1_var_gate_nonu(7)
            for i in range(0, n - 1, 2):
                c.add_q2_var_gate(i + 1, i)
            c.add_q2_const_gate_nonu(2, 9); c.add_q2_var_gate_nonu(12, 0); c.add_q2_const_gate(5, 11)
        c.get_q1_dens_op_with_grad(5)
        c.get_q2_dens_op_with_grad(12, 3)
        assert c._kinds[n:n + 2] == [6, 9] and c._kinds[-5:-2] == [2, 3, 0]
        out.append((c.run(const, var), c.forward(const, var), c.backward(cts, const, var)))
    for a, b in zip(out[0], out[1]):
        assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_bad_inputs_are_errors(pkg):
    from quantum_differentiable_circuit import QdcError
    c = pkg.Circuit(8, precision="f64")
    for pos, msg in (([1, 1, 2], "must be different"), ([0, 3, 4, 0], "must be different"),
                     ([0, 1, 8], "out of the bound"), ([], "1..6"), (list(range(7)), "1..6")):
        for name in ("add_const_gate", "add_var_gate", "add_const_gate_nonu", "add_var_gate_nonu"):
            with pytest.raises(QdcError, match=msg):
                getattr(c, name)(pos)
    for kind in (16, 17, 18, 19):
        with pytest.raises(QdcError, match="qdc_circuit_add_gate"):
            c._add(kind, 0, 1)
    assert c._count(0) == 0
    # a k-qubit gate takes 4^k entries; a singular NonU gate fails the un-compute with the reference's text
    c.add_var_gate_nonu([5, 0, 2])
    c.get_dens_op_with_grad([5, 0, 2])
    u = haar_unitary(np.random.default_rng(0), 8)
    with pytest.raises(QdcError, match="Incorrect len"):
        c.forward([], [u[:16]])
    assert c._count(7) == 64
    singular = u.reshape(8, 8).copy()
    singular[:, 3] = 0
    c.forward([], [singular.reshape(-1)])
    with pytest.raises(QdcError, match=r"U\(\d+, \d+\) is zero"):
        c.backward([np.eye(8, dtype=np.complex128)], [], [singular.reshape(-1)])


def test_finite_difference_f64(pkg):
    """The test_autodiff_finite_difference_f64 recipe (n = 15, 8th-order central difference, eta = 1e-6, rel 1e-9)
    with unitary and NonU variable k-qubit gates (k = 3..6) and the purity loss sum tr rho^2."""
    from qdc import AutoGradCircuit
    n, eta = 15, 1e-6
    kpos = [[14, 3, 0], [2, 13, 7, 0], [1, 6, 12, 4, 0], [5, 0, 14, 9, 10, 3]]
    ops = [op if op[0] != "k" else (op[0], op[1], True, op[3]) for op in kgate_ops(n, kpos, layers=2)]
    rng = np.random.default_rng(42)
    c = AutoGradCircuit(n, precision="f64")
    apply_ops(c.circuit, ops)
    const, var = ops_gates(rng, ops)
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
    assert sorted({g.size for g in grads}) == [4, 16, 64, 256, 1024, 4096]
    ds = sum((g @ p).real for g, p in zip(grads, pert))
    assert abs(ds - fd) / min(abs(ds), abs(fd)) < 1e-9


def test_torch_autograd_glue(pkg):
    """autodiff_run with gate tensors on the GPU: torch.autograd equals the raw vjp, gradients land on the device."""
    import torch
    from qdc import AutoGradCircuit
    n = 13
    rng = np.random.default_rng(3)
    c = AutoGradCircuit(n, precision="f64")
    for i in range(n):
        c.add_q1_var_gate(i)
    c.add_var_gate([12, 0, 6, 3])
    c.add_const_gate([1, 2, 11])
    c.add_var_gate_nonu([4, 9, 5])
    c.get_dens_op_with_grad([12, 0, 6])
    c.get_q2_dens_op_with_grad(5, 9)
    var = ([haar_unitary(rng, 2) for _ in range(n)] + [haar_unitary(rng, 16)]
           + [haar_unitary(rng, 8) + 0.01 * rng.normal(size=64)])
    const = [haar_unitary(rng, 8)]
    _, run = c.build()
    tv = [torch.tensor(v, requires_grad=True, device="cuda") for v in var]
    dens = run(tv, [torch.tensor(g, device="cuda") for g in const])
    assert [tuple(d.shape) for d in dens] == [(8, 8), (4, 4)] and dens[0].is_cuda
    loss = sum(torch.einsum("ij,ji->", d, d).real for d in dens)
    loss.backward()
    dens_np = run.forward(var, const)
    grads = run.vjp(var, const, [2.0 * d.T for d in dens_np])
    for t, g in zip(tv, grads):
        assert t.grad.is_cuda
        np.testing.assert_allclose(t.grad.cpu().numpy(), g.conj(), rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("k,pos", [(3, [17, 2, 0]), (6, [29, 28, 27, 26, 25, 24])])
@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_30_qubits_gate_equals_two_two_qubit_gates(pkg, precision, k, pos):
    """n = 30 (f32 with default options, f64): the k-qubit gate W = (A (x) I)(I (x) B), A on the first two of its
    positions and B on the last two, multiplied on the host, gives the densities of the program with the two-qubit
    gates B and A; its gradient satisfies Re sum G_W dW = Re sum G_A dA for dW = (dA (x) I)(I (x) B), and the other
    gradients are those of the two-gate program."""
    dtype = np.complex64 if precision == "f32" else np.complex128
    tol = TOL[np.dtype(dtype)]
    n = 30
    rng = np.random.default_rng(30 + k)
    var = [haar_unitary(rng, 2, dtype) for _ in range(n)] + [haar_unitary(rng, 4, dtype) for _ in range(0, n - 1, 2)]
    a, b = haar_unitary(rng, 4).reshape(4, 4), haar_unitary(rng, 4).reshape(4, 4)
    da = rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4))
    eye = np.eye(1 << (k - 2))
    w = np.kron(a, eye) @ np.kron(eye, b)
    dw = np.kron(da, eye) @ np.kron(eye, b)
    cts = None

    def run(with_k):
        nonlocal cts
        c = pkg.Circuit(n, precision=precision)
        for i in range(n):
            c.add_q1_var_gate(i)
        for i in range(0, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
        if with_k:
            c.add_var_gate(pos)
            vv = var + [w.reshape(-1).astype(dtype)]
            const = []
        else:
            c.add_q2_const_gate(pos[-2], pos[-1])
            c.add_var_gate([pos[0], pos[1]])
            vv = var + [a.reshape(-1).astype(dtype)]
            const = [b.reshape(-1).astype(dtype)]
        c.get_dens_op_with_grad([pos[0], pos[-1], 5])
        c.get_q2_dens_op_with_grad(pos[1], 22)
        dens = c.forward(const, vv)
        if cts is None:
            cts = [(rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)).astype(dtype) for d in dens]
        grads = c.backward(cts, const, vv)
        del c
        return dens, grads

    dens_k, g_k = run(True)
    dens_2, g_2 = run(False)
    for x, y in zip(dens_k, dens_2):
        assert _rel(x, y) < tol
    sc = max(np.abs(g).max() for g in g_2[:-1])
    assert max(np.abs(x - y).max() for x, y in zip(g_k[:-1], g_2[:-1])) / sc < tol
    lhs = np.sum(g_k[-1].astype(np.complex128) * dw.reshape(-1)).real
    rhs = np.sum(g_2[-1].astype(np.complex128) * da.reshape(-1)).real
    assert abs(lhs - rhs) / np.sum(np.abs(g_2[-1]) * np.abs(da).reshape(-1)) < 10 * tol


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
    tg = importlib.import_module("test_gate_k")
    dtype = np.complex64 if precision == "f32" else np.complex128
    n = 15
    # the k = 3 and 4 gates hold the global qubit 14 (top physical position of the 2-rank register)
    kpos = [[2, 0, 14], [14, 3, 9, 0], [0, 5, 13, 1, 8], [6, 4, 2, 12, 10, 0]]
    ops = tg.kgate_ops(n, kpos)
    const, var = tg.ops_gates(np.random.default_rng(9), ops, dtype)
    out = []
    for c in (sharded.ShardedCircuit(n, precision=precision), pkg.Circuit(n, precision=precision)):
        tg.apply_ops(c, ops)
        run = c.run(const, var)
        fwd = c.forward(const, var)
        rng = np.random.default_rng(4)
        cts = [(rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)).astype(dtype) for d in fwd]
        out.append((run, fwd, c.backward(cts, const, var)))
    errs = []
    for a, b in zip(out[0], out[1]):
        sc = max(np.abs(x).max() for x in b)
        errs.append(max(np.abs(x - y).max() for x, y in zip(a, b)) / sc)
    q.put((rank, "ok", errs))
    dist.destroy_process_group()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_sharded_k_gate_on_the_global_qubit(precision):
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

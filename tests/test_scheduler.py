"""CPU tests of the host-side scheduling logic (csrc/scheduler.hpp through the
C ABI entry `qdc_schedule`; pure host code, no GPU): every plan -- re-ordered,
tiled, sharded -- executed by the oracle's plan interpreter must reproduce the
program-order oracle VM (densities AND reverse-mode gradients), and must obey
the structural rules the CUDA executor relies on."""
import os
import sys

import numpy as np
import pytest

from oracle import plan as op
from oracle.circuit import OracleCircuit
from conftest import haar_unitary
from random_programs import _random_program, all_kinds_program, unitary_program
from test_oracle import autodiff_gates, build_autodiff_circuit, tsallis_loss_and_cotangents

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def brickwork(c, n, depth):
    for layer in range(depth):
        for i in range(layer % 2, n - 1, 2):
            c.add_q2_var_gate(i + 1, i)
    for i in range(0, n - 1, 2):
        c.get_q2_dens_op_with_grad(i + 1, i)


def vqse(c, n, layers):
    for _ in range(layers):
        for i in range(n - 1):
            c.add_q2_var_gate_diag(i, i + 1)
        c.add_q2_var_gate_diag(0, n - 1)
        for i in range(n):
            c.add_q1_var_gate(i)
    for i in range(n - 1):
        c.get_q2_dens_op_with_grad(i, i + 1)
    c.get_q2_dens_op_with_grad(0, n - 1)


def make_case(name, n, rng):
    o = OracleCircuit(n)
    if name == "brickwork":
        brickwork(o, n, 6)
        const, var = [], [haar_unitary(rng, 4) for i in o.instructions if i[0] == 1]
    elif name == "vqse":
        vqse(o, n, 2)
        var = []
        for i in o.instructions:
            if i[0] == 5:
                var.append(np.exp(1j * rng.normal(size=4)))
            elif i[0] == 8:
                var.append(haar_unitary(rng, 2))
        const = []
    else:
        build_autodiff_circuit(o, n, 2)
        const, var = autodiff_gates(rng, n, 2)
    return o, const, var


def reference_results(o, const, var):
    dens = o.forward(const, var)
    _, cts = tsallis_loss_and_cotangents(dens)
    cts_conj = [c.conj() for c in cts]
    grads = o.backward(cts_conj, const, var)
    return dens, cts_conj, grads


def check_plan(pkg, o, const, var, n, n_loc, tile_bits, low_bits, max_tile_gates=0, tile_strategy=-1, swap_min_pos=-1):
    dens_ref, cts_conj, grads_ref = reference_results(o, const, var)
    enc = pkg._ffi.schedule(o.instructions, n, n_loc, tile_bits, low_bits, max_tile_gates,
                            tile_strategy=tile_strategy, swap_min_pos=swap_min_pos)
    steps, final_map = op.decode_plan(enc)
    # structure
    seen = []
    for st in steps:
        if st["type"] == op.ST_TILE:
            assert len(st["bits"]) <= tile_bits and st["bits"][:low_bits] == list(range(low_bits))
            assert 2 <= len(st["gates"]) <= (max_tile_gates or 24)
            assert all(b < n_loc for b in st["bits"])
        if st["type"] == op.ST_SWAP:
            assert 0 <= st["gbit"] < n - n_loc and 0 <= st["lpos"] < n_loc
    for st in op.flat_steps(steps):
        if st["type"] in (op.ST_GATE, op.ST_DENS):
            seen.append(st["inst"])
    expect = [i for i, inst in enumerate(o.instructions) if inst[0] not in (10, 11)]  # forward skips non-diff densities
    assert sorted(seen) == expect, "every instruction exactly once"
    assert sorted(final_map) == list(range(n))
    dens, grads, final = op.run_plan_global(steps, o.instructions, n, n_loc, const, var, cts_conj)
    assert len(dens) == len(dens_ref) and len(grads) == len(grads_ref)
    for a, b in zip(dens, dens_ref):
        np.testing.assert_allclose(a, b, atol=1e-12)
    scale = max(np.abs(g).max() for g in grads_ref)
    for a, b in zip(grads, grads_ref):
        assert np.abs(a - b).max() / scale < 1e-12
    # after backward every swap has been undone: identity layout, initial state
    init = np.zeros(1 << n, dtype=np.complex128); init[0] = 1
    np.testing.assert_allclose(final, init, atol=1e-10)
    return steps


@pytest.mark.parametrize("case", ["brickwork", "vqse", "autodiff"])
def test_untiled_single_gpu_plan_is_program_order(pkg, case):
    n = 8
    o, const, var = make_case(case, n, np.random.default_rng(0))
    steps = check_plan(pkg, o, const, var, n, n, 0, 0)
    order = [st["inst"] for st in steps]
    assert order == sorted(order)
    assert all(st["type"] in (op.ST_GATE, op.ST_DENS) for st in steps)


@pytest.mark.parametrize("case", ["brickwork", "vqse", "autodiff"])
@pytest.mark.parametrize("tile_bits,low_bits", [(5, 2), (6, 3), (4, 1)])
def test_tiled_plans_are_exact(pkg, case, tile_bits, low_bits):
    n = 9
    o, const, var = make_case(case, n, np.random.default_rng(1))
    steps = check_plan(pkg, o, const, var, n, n, tile_bits, low_bits, max_tile_gates=7)
    if case == "brickwork":
        tiles = [st for st in steps if st["type"] == op.ST_TILE]
        assert tiles


@pytest.mark.parametrize("case", ["brickwork", "vqse", "autodiff"])
@pytest.mark.parametrize("g", [1, 2, 3])
@pytest.mark.parametrize("tile_bits", [0, 5])
def test_sharded_plans_are_exact(pkg, case, g, tile_bits):
    n = 9
    o, const, var = make_case(case, n, np.random.default_rng(2))
    check_plan(pkg, o, const, var, n, n - g, tile_bits, 2 if tile_bits else 0)


@pytest.mark.parametrize("case", ["brickwork", "vqse", "autodiff"])
@pytest.mark.parametrize("g", [1, 2, 3])
@pytest.mark.parametrize("swap_min_pos", [0, 1, 2, 3, -2])
def test_sharded_plans_are_exact_wherever_the_remap_victims_sit(pkg, case, g, swap_min_pos):
    """A sharded circuit lets a cost model choose the lowest position of its remap victims (scheduler.hpp:
    schedule_best; -2 here): every candidate plan, and the chosen one, must be exact -- also with 6-position windows."""
    n = 10
    o, const, var = make_case(case, n, np.random.default_rng(3))
    check_plan(pkg, o, const, var, n, n - g, 6, 0, max_tile_gates=32, swap_min_pos=swap_min_pos)


def test_cost_model_keeps_the_windows_of_the_benchmark_plans_whole(pkg):
    """33 / 35 qubits on 2 / 8 ranks, depth 100, 6-position windows: victims from position 4 upwards cut an island off
    the low end of the chain (187 / 205 block passes); the cost model moves them down (175 / 192) with the same number of
    exchanges.  34 qubits on 4 ranks keep position 4."""
    for n, g, default_tiles, best_tiles, low in ((33, 1, 187, 175, 2), (34, 2, 190, 190, 4), (35, 3, 205, 192, 3)):
        o = OracleCircuit.__new__(OracleCircuit)
        o.instructions = []
        brickwork(o, n, 100)
        got = {}
        for mp in (-1, -2):
            steps, _ = op.decode_plan(pkg._ffi.schedule(o.instructions, n, n - g, 6, 0, 32, swap_min_pos=mp))
            got[mp] = (sum(st["type"] == op.ST_TILE for st in steps), [st["lpos"] for st in steps if st["type"] == op.ST_SWAP])
        assert got[-1][0] == default_tiles and got[-2][0] == best_tiles, (n, got[-1][0], got[-2][0])
        assert len(got[-2][1]) == len(got[-1][1]) and min(got[-2][1]) == low, (n, got)


def test_brickwork_swap_count_follows_the_light_cone(pkg):
    """35 qubits on 8 ranks, depth 100: a naive executor needs a remap for every
    layer touching a global qubit (~2 per layer); the scheduler's light-cone
    order needs an order of magnitude fewer half-shard exchanges."""
    n, g, depth = 35, 3, 100
    o = OracleCircuit.__new__(OracleCircuit)
    o.instructions = []
    brickwork(o, n, depth)
    enc = pkg._ffi.schedule(o.instructions, n, n - g, 0, 0)
    steps, _ = op.decode_plan(enc)
    swaps = sum(1 for st in steps if st["type"] == op.ST_SWAP)
    gates = sum(1 for st in steps if st["type"] == op.ST_GATE)
    assert gates == 1700
    assert swaps <= 40, swaps


@pytest.mark.parametrize("case", ["brickwork", "vqse", "autodiff"])
@pytest.mark.parametrize("strategy", [0, 1, 2])
@pytest.mark.parametrize("g", [0, 2])
def test_every_tiling_strategy_is_exact(pkg, case, strategy, g):
    """First-fit, window growth and window growth with look-ahead (scheduler.hpp: tile_strategy) all
    reproduce the program-order densities and gradients, single GPU and sharded over 4 ranks."""
    n = 9
    o, const, var = make_case(case, n, np.random.default_rng(6))
    check_plan(pkg, o, const, var, n, n - g, 5, 2, tile_strategy=strategy)


def test_window_tiling_halves_the_passes_of_a_brickwork_circuit(pkg):
    """32 qubits, depth 100, 2^12 tiles with 4 forced low positions: first-fit in program order scatters a
    tile's positions over unrelated pairs (207 passes); windows hold light-cone strips of 8 qubits."""
    o = OracleCircuit.__new__(OracleCircuit)
    o.instructions = []
    brickwork(o, 32, 100)
    passes = {}
    for strategy in (0, 1, 2):
        enc = pkg._ffi.schedule(o.instructions, 32, 32, 12, 4, 32, tile_strategy=strategy)
        steps, _ = op.decode_plan(enc)
        tiles = [st for st in steps if st["type"] == op.ST_TILE]
        assert sum(len(t["gates"]) for t in tiles) + sum(1 for st in steps if st["type"] == op.ST_GATE) == 1550
        passes[strategy] = len(tiles)
    assert passes[1] <= 0.55 * passes[0] and passes[2] <= passes[1], passes


def test_remap_victims_avoid_short_run_positions(pkg):
    """Remap swaps pick their local victim among physical positions >= 4 (128-byte runs in the exchanged
    halves: 695 vs 320-510 GB/s per direction measured over NVLink, profiles/r1_exchange_bench_2gpu.txt)
    whenever a less urgent qubit lives there, without needing more exchanges than the pure
    farthest-next-use choice did (4 / 10 / 14 for 33 / 34 / 35 qubits at depth 100)."""
    for n, g, expect in ((33, 1, 4), (34, 2, 10), (35, 3, 14)):
        o = OracleCircuit.__new__(OracleCircuit)
        o.instructions = []
        brickwork(o, n, 100)
        enc = pkg._ffi.schedule(o.instructions, n, n - g, 12, 4)
        steps, _ = op.decode_plan(enc)
        swaps = [st for st in steps if st["type"] == op.ST_SWAP]
        assert len(swaps) <= expect, (n, len(swaps))
        assert all(st["lpos"] >= 4 for st in swaps), [(st["gbit"], st["lpos"]) for st in swaps]
    # a register whose only less-urgent local qubits sit at low positions must still make progress
    n, g = 7, 2
    o, const, var = make_case("brickwork", n, np.random.default_rng(4))
    check_plan(pkg, o, const, var, n, n - g, 0, 0)


def _gloo_worker(rank, world, port, case, n, tile_bits, q):
    import torch
    import torch.distributed as dist
    import importlib
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    pkg = importlib.import_module("differentiable-quantum-circuit-cuda_b200")
    o, const, var = make_case(case, n, np.random.default_rng(3))
    dens_ref, cts_conj, grads_ref = reference_results(o, const, var)
    g = world.bit_length() - 1
    enc = pkg._ffi.schedule(o.instructions, n, n - g, tile_bits, 2 if tile_bits else 0)
    steps, _ = op.decode_plan(enc)

    def exchange(buf, partner):
        send = torch.from_numpy(np.ascontiguousarray(buf).view(np.float64).copy())
        recv = torch.empty_like(send)
        reqs = dist.batch_isend_irecv([dist.P2POp(dist.isend, send, partner), dist.P2POp(dist.irecv, recv, partner)])
        for r in reqs:
            r.wait()
        return recv.numpy().view(np.complex128)

    def allreduce(arr):
        t = torch.from_numpy(np.ascontiguousarray(arr).view(np.float64).copy())
        dist.all_reduce(t)
        return t.numpy().view(np.complex128)

    runner = op.ShardedPlanRunner(n, rank, world, exchange, allreduce)
    dens, grads, shard = runner.run(steps, o.instructions, const, var, cts_conj)
    err_d = max(np.abs(a - b).max() for a, b in zip(dens, dens_ref))
    scale = max(np.abs(x).max() for x in grads_ref)
    err_g = max(np.abs(a - b).max() for a, b in zip(grads, grads_ref)) / scale
    init = np.zeros(1 << (n - g), dtype=np.complex128)
    if rank == 0:
        init[0] = 1
    err_s = np.abs(shard - init).max()
    nswap = sum(1 for st in steps if st["type"] == op.ST_SWAP)
    q.put((rank, err_d, err_g, err_s, nswap))
    dist.destroy_process_group()


@pytest.mark.parametrize("case,world,tile_bits", [("brickwork", 2, 0), ("autodiff", 2, 5), ("vqse", 4, 0)])
def test_sharded_execution_over_gloo(case, world, tile_bits):
    """world_size-2/4 gloo run of the multi-rank path: per-rank NumPy shards, the
    C++ scheduler's plan, half-shard exchanges over torch.distributed, partial
    densities / gradients all-reduced; every rank must reproduce the oracle."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    n = 8
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, case, n, tile_bits, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, err_d, err_g, err_s, nswap in results:
        assert err_d < 1e-12 and err_g < 1e-12 and err_s < 1e-10, (rank, err_d, err_g, err_s)
    assert results[0][4] >= 1, "the sharded plan must contain at least one exchange"


@pytest.mark.parametrize("seed", range(8))
def test_random_programs_are_scheduled_exactly(pkg, seed):
    """Random programs over every instruction kind, and programs of the two families of the GPU differential tests
    (tests/random_programs.py), every tiling strategy, single GPU and sharded: the plan executed by the oracle's
    interpreter reproduces the program-order densities and gradients."""
    rng = np.random.default_rng(100 + seed)
    n = 7
    programs = (_random_program(rng, n, 40), unitary_program(n, 300 + seed, 60),
                all_kinds_program(n, 400 + seed, 60, k_rate=0))
    for o, const, var in programs:
        for strategy in (0, 1, 2):
            for g, tile_bits in ((0, 5), (2, 4), (1, 0)):
                check_plan(pkg, o, const, var, n, n - g, tile_bits, 2 if tile_bits else 0, tile_strategy=strategy)

"""CPU: the random programs of the GPU differential tests (tests/random_programs.py, fixed seeds) reach, through the pass
scheduler's plans at the executor's own tile parameters, every kernel branch the circuit-level tests with 1-D
nearest-neighbour circuits never select.  A generator change that loses one of them fails here, without a GPU."""
import numpy as np
import pytest

from oracle import circuit as oc
from oracle import plan as op
from random_programs import MULTI_TILE, N_QUBITS, UNITARY_SEEDS, unitary_program

# (precision, tile bits, low bits, max gates per pass) of the FP32 / FP64 tile passes: circuit.cuh base_options
TILE_PARAMS = (("f32", 12, 4, 32), ("f32", 11, 4, 32), ("f64", 11, 3, 24))
_DENSE_Q2 = (oc.CONST_Q2, oc.VAR_Q2, oc.CONST_Q2_NONU, oc.VAR_Q2_NONU)


def _tiles(pkg, o, n, precision, tile_bits, low_bits, max_gates):
    enc = pkg._ffi.schedule(o.instructions, n, n, tile_bits, low_bits, max_gates, precision=precision, tile_strategy=2)
    steps, _ = op.decode_plan(enc)
    return [st for st in steps if st["type"] == op.ST_TILE]


def tile_features(tiles, instructions):
    """Counts of the two-qubit dense-gate geometries of tile passes (bits: the pass's physical positions, ascending, so
    the tile position of a gate operand is its index there)."""
    f = {"pos2_below_pos1": 0, "tile_distance_ge_4": 0, "pos2_on_tile_bit_0": 0}
    for t in tiles:
        for g in t["gates"]:
            if instructions[g["inst"]][0] not in _DENSE_Q2:
                continue
            t2, t1 = t["bits"].index(g["p2"]), t["bits"].index(g["p1"])
            f["pos2_below_pos1"] += t2 < t1
            f["tile_distance_ge_4"] += abs(t2 - t1) >= 4
            f["pos2_on_tile_bit_0"] += t2 == 0 and t1 > 0
    return f


def window_features(tiles, instructions, n):
    """Counts of the tensor-core window geometries (6 / 0 windows: tc_exec.cuh tc_prepare, tc_block.cuh make_params)."""
    f = {"fewer_than_6": 0, "has_0": 0, "has_1_or_2_not_0": 0, "all_ge_5": 0, "has_top": 0, "q1_or_diag_only": 0}
    for t in tiles:
        bits = t["bits"]
        f["fewer_than_6"] += len(bits) < 6
        f["has_0"] += 0 in bits
        f["has_1_or_2_not_0"] += (1 in bits or 2 in bits) and 0 not in bits
        f["all_ge_5"] += min(bits) >= 5
        f["has_top"] += n - 1 in bits
        f["q1_or_diag_only"] += all(instructions[g["inst"]][0] not in _DENSE_Q2 for g in t["gates"])
    return f


def _sum(dicts):
    out = {}
    for d in dicts:
        for k, v in d.items():
            out[k] = out.get(k, 0) + v
    return out


@pytest.mark.parametrize("precision,tile_bits,low_bits,max_gates", TILE_PARAMS)
def test_random_programs_reach_every_tile_pass_geometry(pkg, precision, tile_bits, low_bits, max_gates):
    feats = []
    for seed in UNITARY_SEEDS:
        o, _, _ = unitary_program(N_QUBITS, seed)
        feats.append(tile_features(_tiles(pkg, o, N_QUBITS, precision, tile_bits, low_bits, max_gates), o.instructions))
    total = _sum(feats)
    assert all(v > 0 for v in total.values()), total


def test_random_programs_reach_every_tensor_core_window_geometry(pkg):
    feats = []
    for seed in UNITARY_SEEDS:
        o, _, _ = unitary_program(N_QUBITS, seed)
        feats.append(window_features(_tiles(pkg, o, N_QUBITS, "f32", 6, 0, 32), o.instructions, N_QUBITS))
    total = _sum(feats)
    assert all(v > 0 for v in total.values()), total


def test_multi_tile_program_holds_tensor_core_windows_everywhere(pkg):
    """The 22-qubit program run with several tiles per CTA: its windows cover low, high and the top position."""
    n, seed, length = MULTI_TILE
    o, _, _ = unitary_program(n, seed, length)
    f = window_features(_tiles(pkg, o, n, "f32", 6, 0, 32), o.instructions, n)
    for k in ("has_0", "has_1_or_2_not_0", "all_ge_5", "has_top", "fewer_than_6"):
        assert f[k] > 0, f


def test_generator_is_a_function_of_its_seed():
    a, b = unitary_program(N_QUBITS, UNITARY_SEEDS[0]), unitary_program(N_QUBITS, UNITARY_SEEDS[0])
    assert a[0].instructions == b[0].instructions
    assert all(np.array_equal(x, y) for x, y in zip(a[1] + a[2], b[1] + b[2]))

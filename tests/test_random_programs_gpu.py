"""GPU: the fused executors on random programs (tests/random_programs.py) -- gates on arbitrary qubit pairs in both
operand orders, densities on far pairs and on qubit 0, k-qubit instructions between them -- against the complex128
oracle VM at 15 qubits, against the f64 per-gate executor at 22 qubits (several tiles per tensor-core CTA), and run to
run.  Tolerances relative to the largest entry: 1e-5 (f32), 1e-12 (f64)."""
import gc

import numpy as np
import pytest

from conftest import random_state_unnormalized
from random_programs import ALL_KINDS_SEEDS, MULTI_TILE, N_QUBITS, UNITARY_SEEDS, all_kinds_program, replay
from random_programs import unitary_program

pytestmark = pytest.mark.gpu
TOL = {"f32": 1e-5, "f64": 1e-12}
DTYPE = {"f32": np.complex64, "f64": np.complex128}

PROGRAMS = [("unitary", s) for s in UNITARY_SEEDS] + [("all_kinds", s) for s in ALL_KINDS_SEEDS]
# executor options of each variant and the profile categories whose kernels it must have launched (forward, backward)
F32_VARIANTS = {
    "fuse0": ((("fuse", 0), ("tc", 0)), ("fwd_q2", "rev_q2")),
    "fuse1": ((("fuse", 1), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "fuse2": ((("fuse", 2), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "soa0": ((("soa", 0), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "rb_policy0": ((("rb_policy", 0), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "rb_policy1": ((("rb_policy", 1), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "tile_strategy0": ((("tile_strategy", 0), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "tile_bits11": ((("tile_bits", 11), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "max_tile_gates2": ((("max_tile_gates", 2), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "batch_dens0": ((("batch_dens", 0), ("tc", 0)), ("tile_fwd", "tile_bwd")),
    "tc_rev1": ((("tc", 1), ("tc_rev", 1)), ("tc_fwd", "tc_bwd")),
    "tc_rev0": ((("tc", 1), ("tc_rev", 0)), ("tc_fwd", "tc_bwd")),
    "tc_products8": ((("tc", 1), ("tc_products", 8)), ("tc_fwd", "tc_bwd")),
}
F64_VARIANTS = {
    "fuse0": ((("fuse", 0),), ("fwd_q2", "rev_q2")),
    "fuse1": ((("fuse", 1),), ("tile_fwd", "tile_bwd")),
    "fuse2": ((("fuse", 2),), ("tile_fwd", "tile_bwd")),
    "rb_policy1": ((("rb_policy", 1),), ("tile_fwd", "tile_bwd")),
    "tile_strategy0": ((("tile_strategy", 0),), ("tile_fwd", "tile_bwd")),
}


def _program(family, seed, n=N_QUBITS, length=200):
    return unitary_program(n, seed, length) if family == "unitary" else all_kinds_program(n, seed, length)


def _initial(init, n, dtype):
    if init == "zero":
        v = np.zeros(1 << n, dtype=dtype)
        v[0] = 1
        return v
    return random_state_unnormalized(np.random.default_rng(5 + n), n, dtype)


def _cotangents(dens, seed):
    rng = np.random.default_rng(seed)
    out = []
    for d in dens:
        a = rng.normal(size=d.shape) + 1j * rng.normal(size=d.shape)
        out.append((a + a.conj().T) / 2)
    return out


def _max_rel(got, ref):
    assert len(got) == len(ref)
    scale = max(float(np.abs(r).max()) for r in ref)
    return max(float(np.abs(np.asarray(g).reshape(-1) - np.asarray(r).reshape(-1)).max()) for g, r in zip(got, ref)) / scale


_ORACLE = {}


def oracle_results(family, seed, init, precision):
    """run / forward / backward / state after backward of the complex128 oracle, on the inputs rounded to the precision
    under test (so both sides see the same numbers), computed once per program."""
    key = (family, seed, init, precision)
    if key not in _ORACLE:
        o, const, var = _program(family, seed)
        dt = DTYPE[precision]
        const = [np.asarray(g, dtype=dt) for g in const]
        var = [np.asarray(g, dtype=dt) for g in var]
        o.set_state_from_vector(_initial(init, N_QUBITS, dt))
        runs = o.run(const, var)
        dens = o.forward(const, var)
        cts = _cotangents(dens, seed)
        grads = o.backward(cts, const, var)
        _ORACLE[key] = (o.instructions, const, var, cts, runs, dens, grads, o.state.copy())
    return _ORACLE[key]


def _execute(precision, options, instructions, n, initial, const, var, cts):
    from quantum_differentiable_circuit import Circuit
    c = Circuit(n, precision=precision)
    for k, v in options:
        c.set_option(k, v)
    c.set_option("profile", 1)
    c.set_state_from_vector(initial)
    replay(c, instructions)
    dt = DTYPE[precision]
    runs = c.run(const, var)
    dens = c.forward(const, var)
    prof_f = c.last_profile()
    grads = c.backward([np.asarray(x, dtype=dt) for x in cts], const, var)
    prof_b = c.last_profile()
    state = c.get_cpu_state_copy()
    del c
    gc.collect()
    return runs, dens, grads, state, prof_f, prof_b


def _check_against_oracle(precision, variant, family, seed, init):
    options, (cat_f, cat_b) = (F32_VARIANTS if precision == "f32" else F64_VARIANTS)[variant]
    instructions, const, var, cts, runs_o, dens_o, grads_o, state_o = oracle_results(family, seed, init, precision)
    initial = _initial(init, N_QUBITS, DTYPE[precision])
    runs, dens, grads, state, pf, pb = _execute(precision, options, instructions, N_QUBITS, initial, const, var, cts)
    assert pf.get(cat_f, {}).get("launches", 0) > 0 and pb.get(cat_b, {}).get("launches", 0) > 0, (pf, pb)
    if variant == "fuse0":
        assert "tile_fwd" not in pf and "tc_fwd" not in pf
    tol = TOL[precision]
    errs = {"run": _max_rel(runs, runs_o), "forward": _max_rel(dens, dens_o), "backward": _max_rel(grads, grads_o),
            "state": _max_rel([state], [state_o])}
    assert max(errs.values()) < tol, errs
    # the working state after backward is the initial state again (the oracle's, too, up to the rounding of the gates)
    assert _max_rel([state], [initial]) < tol


@pytest.mark.parametrize("init", ["zero", "random"])
@pytest.mark.parametrize("family,seed", PROGRAMS)
@pytest.mark.parametrize("variant", list(F32_VARIANTS))
def test_f32_executors_match_oracle_on_random_programs(pkg, variant, family, seed, init):
    _check_against_oracle("f32", variant, family, seed, init)


@pytest.mark.parametrize("init", ["zero", "random"])
@pytest.mark.parametrize("family,seed", PROGRAMS)
@pytest.mark.parametrize("variant", list(F64_VARIANTS))
def test_f64_executors_match_oracle_on_random_programs(pkg, variant, family, seed, init):
    _check_against_oracle("f64", variant, family, seed, init)


@pytest.fixture(scope="module")
def multi_tile(pkg):
    """The 22-qubit unitary program (>= 6 tiles per tensor-core CTA, so the 4-stage ring wraps) on an unnormalised
    random state, and the results of the f64 per-gate executor for the same complex64 inputs, which the 15-qubit tests
    tie to the oracle."""
    n, seed, length = MULTI_TILE
    o, const, var = unitary_program(n, seed, length)
    const = [np.asarray(g, dtype=np.complex64) for g in const]
    var = [np.asarray(g, dtype=np.complex64) for g in var]
    initial = _initial("random", n, np.complex64)
    wide = [[g.astype(np.complex128) for g in gs] for gs in (const, var)]
    from quantum_differentiable_circuit import Circuit
    c = Circuit(n, precision="f64")
    c.set_option("fuse", 0)
    c.set_state_from_vector(initial.astype(np.complex128))
    replay(c, o.instructions)
    dens = c.forward(*wide)
    cts = _cotangents(dens, seed)
    grads = c.backward(cts, *wide)
    del c
    gc.collect()
    return n, o.instructions, const, var, initial, cts, dens, grads


@pytest.mark.parametrize("tc_rev", [1, 0])
def test_tc_blocks_with_several_tiles_per_cta_match_f64_executor(pkg, multi_tile, tc_rev):
    n, instructions, const, var, initial, cts, dens_r, grads_r = multi_tile
    _, dens, grads, state, pf, pb = _execute("f32", (("tc", 1), ("tc_rev", tc_rev)), instructions, n, initial, const, var,
                                             cts)
    assert pf.get("tc_fwd", {}).get("launches", 0) > 0 and pb.get("tc_bwd", {}).get("launches", 0) > 0, (pf, pb)
    errs = {"forward": _max_rel(dens, dens_r), "backward": _max_rel(grads, grads_r), "state": _max_rel([state], [initial])}
    assert max(errs.values()) < TOL["f32"], errs


@pytest.mark.parametrize("options", [(("tc", 1),), (("tc", 1), ("tc_rev", 0)), (("tc", 0),)], ids=["tc", "tc_rev0", "tile"])
def test_fused_executors_are_bit_identical_run_to_run(pkg, multi_tile, options):
    """The barrier-free slicing grid and the fixed-order gradient sums keep the results a pure function of the inputs:
    two identical runs give the same bits in densities, gradients and the working state."""
    n, instructions, const, var, initial, cts, _, _ = multi_tile
    a = _execute("f32", options, instructions, n, initial, const, var, cts)
    b = _execute("f32", options, instructions, n, initial, const, var, cts)
    assert a[4].get("tc_fwd" if options[0][1] else "tile_fwd", {}).get("launches", 0) > 0
    for x, y in zip(a[:3], b[:3]):
        assert len(x) == len(y) and all(np.array_equal(p, q) for p, q in zip(x, y))
    assert np.array_equal(a[3], b[3])

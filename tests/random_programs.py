"""Random circuit programs for the differential tests of the executors (not a test module).

Two families, each a pure function of the qubit count and a seed, return `(oracle, const, var)`: a
`oracle.kdiag.KDiagOracleCircuit` holding the instructions, and the constant and variable gate lists in program order.
`replay(circuit, instructions)` adds the same instructions to a `Circuit` (or any object with the same builders).

- `unitary_program`: unitary one- and two-qubit gates, dense and diagonal, const and var, on pairs that are half near
  (|a - b| <= 3) and half anywhere, in both operand orders, and one- / two-qubit densities with and without grad on
  random qubits.  Some program points carry a burst of densities, so the batched density sweeps see far pairs and pairs
  on qubit 0.  Its windows become tensor-core blocks.
- `all_kinds_program`: the 14 one- and two-qubit instruction kinds, NonU included, plus (at `k_rate`) k-qubit gates,
  diagonal gates and densities with 3 <= k <= 6 on random qubits.  The pass scheduler's C entry point takes only the
  14 kinds, so the plan tests use `k_rate=0`.
"""
import numpy as np

from conftest import haar_unitary
from oracle import circuit as oc
from oracle.kdens import DENS_K, DIFF_DENS_K
from oracle.kdiag import CONST_GATE_K_DIAG, CONST_GATE_K_DIAG_NONU, VAR_GATE_K_DIAG, VAR_GATE_K_DIAG_NONU
from oracle.kdiag import KDiagOracleCircuit
from oracle.kgates import CONST_GATE_K, CONST_GATE_K_NONU, VAR_GATE_K, VAR_GATE_K_NONU

# builder of every instruction kind: (name, takes a positions list)
BUILDERS = {
    oc.CONST_Q2: ("add_q2_const_gate", False), oc.VAR_Q2: ("add_q2_var_gate", False),
    oc.CONST_Q2_NONU: ("add_q2_const_gate_nonu", False), oc.VAR_Q2_NONU: ("add_q2_var_gate_nonu", False),
    oc.CONST_Q2_DIAG: ("add_q2_const_gate_diag", False), oc.VAR_Q2_DIAG: ("add_q2_var_gate_diag", False),
    oc.CONST_Q1: ("add_q1_const_gate", False), oc.CONST_Q1_NONU: ("add_q1_const_gate_nonu", False),
    oc.VAR_Q1: ("add_q1_var_gate", False), oc.VAR_Q1_NONU: ("add_q1_var_gate_nonu", False),
    oc.Q2_DENS: ("get_q2_dens_op", False), oc.Q1_DENS: ("get_q1_dens_op", False),
    oc.DIFF_Q2_DENS: ("get_q2_dens_op_with_grad", False), oc.DIFF_Q1_DENS: ("get_q1_dens_op_with_grad", False),
    DENS_K: ("get_dens_op", True), DIFF_DENS_K: ("get_dens_op_with_grad", True),
    CONST_GATE_K: ("add_const_gate", True), VAR_GATE_K: ("add_var_gate", True),
    CONST_GATE_K_NONU: ("add_const_gate_nonu", True), VAR_GATE_K_NONU: ("add_var_gate_nonu", True),
    CONST_GATE_K_DIAG: ("add_const_gate_diag", True), VAR_GATE_K_DIAG: ("add_var_gate_diag", True),
    CONST_GATE_K_DIAG_NONU: ("add_const_gate_diag_nonu", True), VAR_GATE_K_DIAG_NONU: ("add_var_gate_diag_nonu", True),
}


def replay(circuit, instructions):
    for inst in instructions:
        name, listed = BUILDERS[inst[0]]
        if listed:
            getattr(circuit, name)(list(inst[1]))
        else:
            getattr(circuit, name)(*inst[1:])


def _pair(rng, n):
    """Half the pairs within distance 3, half uniform; either operand first."""
    if rng.random() < 0.5:
        a = int(rng.integers(n))
        b = a + int(rng.choice([-3, -2, -1, 1, 2, 3]))
        if not 0 <= b < n:
            b = a - (b - a)
    else:
        a, b = (int(x) for x in rng.choice(n, size=2, replace=False))
    return (a, b) if rng.random() < 0.5 else (b, a)


def _density(o, rng, n):
    grad = rng.random() < 0.75
    if rng.random() < 0.3:
        (o.get_q1_dens_op_with_grad if grad else o.get_q1_dens_op)(int(rng.integers(n)))
    else:
        a, b = _pair(rng, n) if rng.random() < 0.5 else (int(x) for x in rng.choice(n, size=2, replace=False))
        if rng.random() < 0.25:                      # a pair on qubit 0
            a, b = (0, int(rng.integers(1, n))) if rng.random() < 0.5 else (int(rng.integers(1, n)), 0)
        (o.get_q2_dens_op_with_grad if grad else o.get_q2_dens_op)(a, b)


def unitary_program(n, seed, length=200):
    rng = np.random.default_rng(seed)
    o = KDiagOracleCircuit(n)
    const, var = [], []
    for _ in range(length):
        r = rng.random()
        if r < 0.55:
            a, b = _pair(rng, n)
            variable, diag = rng.random() < 0.5, rng.random() < 0.35
            if diag:
                (o.add_q2_var_gate_diag if variable else o.add_q2_const_gate_diag)(a, b)
                g = np.exp(1j * rng.normal(size=4))
            else:
                (o.add_q2_var_gate if variable else o.add_q2_const_gate)(a, b)
                g = haar_unitary(rng, 4)
            (var if variable else const).append(g)
        elif r < 0.88:
            variable = rng.random() < 0.5
            (o.add_q1_var_gate if variable else o.add_q1_const_gate)(int(rng.integers(n)))
            (var if variable else const).append(haar_unitary(rng, 2))
        elif r < 0.95:
            _density(o, rng, n)
        else:                                        # a program point with several densities
            for _ in range(int(rng.integers(2, 6))):
                _density(o, rng, n)
    o.get_q2_dens_op_with_grad(n - 1, 0)
    return o, const, var


def _nonu(rng, g):
    return g + 0.05 * (rng.normal(size=g.size) + 1j * rng.normal(size=g.size))


def _k_instruction(o, rng, n, const, var):
    k = int(rng.integers(3, 7))
    pos = [int(p) for p in rng.choice(n, size=k, replace=False)]
    r = rng.random()
    if r < 0.3:
        (o.get_dens_op_with_grad if rng.random() < 0.7 else o.get_dens_op)(pos)
        return
    variable, nonu = rng.random() < 0.5, rng.random() < 0.3
    suffix = "_nonu" if nonu else ""
    if r < 0.65:
        getattr(o, "add_%s_gate%s" % ("var" if variable else "const", suffix))(pos)
        g = haar_unitary(rng, 1 << k)
    else:
        getattr(o, "add_%s_gate_diag%s" % ("var" if variable else "const", suffix))(pos)
        g = np.exp(1j * rng.normal(size=1 << k))
    (var if variable else const).append(_nonu(rng, g) if nonu else g)


def _random_program(rng, n, length, k_rate=0.0):
    """A random program over all 14 one- and two-qubit instruction kinds (gates on random qubits, densities sprinkled
    in), with k-qubit instructions at `k_rate`.  For k_rate = 0 the draws, and so the programs, do not depend on it."""
    o = KDiagOracleCircuit(n)
    const, var = [], []
    adders2 = ("add_q2_const_gate", "add_q2_var_gate", "add_q2_const_gate_nonu", "add_q2_var_gate_nonu",
               "add_q2_const_gate_diag", "add_q2_var_gate_diag")
    adders1 = ("add_q1_const_gate", "add_q1_const_gate_nonu", "add_q1_var_gate", "add_q1_var_gate_nonu")
    for _ in range(length):
        if k_rate and rng.random() < k_rate:
            _k_instruction(o, rng, n, const, var)
            continue
        r = rng.random()
        if r < 0.55:
            name = adders2[rng.integers(len(adders2))]
            a, b = rng.choice(n, size=2, replace=False)
            getattr(o, name)(int(a), int(b))
            if name.endswith("diag"):
                g = np.exp(1j * rng.normal(size=4))
            else:
                g = haar_unitary(rng, 4)
                if name.endswith("nonu"):
                    g = _nonu(rng, g)
            (var if "_var_" in name else const).append(g)
        elif r < 0.85:
            name = adders1[rng.integers(len(adders1))]
            getattr(o, name)(int(rng.integers(n)))
            g = haar_unitary(rng, 2)
            if name.endswith("nonu"):
                g = _nonu(rng, g)
            (var if "_var_" in name else const).append(g)
        elif r < 0.93:
            a, b = rng.choice(n, size=2, replace=False)
            (o.get_q2_dens_op_with_grad if rng.random() < 0.7 else o.get_q2_dens_op)(int(a), int(b))
        else:
            (o.get_q1_dens_op_with_grad if rng.random() < 0.7 else o.get_q1_dens_op)(int(rng.integers(n)))
    o.get_q2_dens_op_with_grad(1, 0)
    return o, const, var


def all_kinds_program(n, seed, length=200, k_rate=0.04):
    return _random_program(np.random.default_rng(seed), n, length, k_rate)


# the programs of the GPU differential tests (tests/test_random_programs_gpu.py); tests/test_random_programs.py checks
# on the CPU that their plans reach every kernel branch those tests are meant to cover
N_QUBITS = 15
UNITARY_SEEDS = (11, 12, 13)
ALL_KINDS_SEEDS = (21, 22)
MULTI_TILE = (22, 31, 300)   # qubits, seed, length of the unitary program run with several tiles per tensor-core CTA

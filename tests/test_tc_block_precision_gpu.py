"""GPU: the error of ONE tensor-core block (tc_block.cuh forward, tc_rev.cuh / the three-sweep reverse step) against
NumPy complex128, per block rather than over a whole circuit, at the bounds DESIGN.md section 4 derives for the bf16
slice products (about 4x its figures): forward state 1e-6 of the largest amplitude with 6 products and 2.5e-7 with 8,
gradients 5e-6 of the largest gradient entry, un-computed state 1e-6.

Each case is one window of 9 unitary gates, dense and diagonal, one- and two-qubit, const and var, on at most 6 qubits,
followed by a differentiable density on two of them, through the public `Circuit` (tc = 1).  The initial states probe
the per-warp slicing grid (seeded from the CTA's first tile, then only raised by its warp) and the exponent clamp of
`magic_of`: a normalised Gaussian state, the same state scaled by 2^40 and 2^-40, a state whose first tiles are small
while later tiles spread 18 binades over the block index (22 qubits), and a sparse state whose first tiles are zero."""
import gc

import numpy as np
import pytest

from conftest import haar_unitary
from oracle.circuit import OracleCircuit

pytestmark = pytest.mark.gpu
FWD_TOL = {6: 1e-6, 8: 2.5e-7}
GRAD_TOL = 5e-6
BACK_TOL = 1e-6

POSITIONS = {
    "low": lambda n: [0, 1, 2, 3, 4, 5],
    "1_2_not_0": lambda n: [2, 1, 4, 6, 7, 9],
    "top": lambda n: list(range(n - 6, n)),
    "scattered": lambda n: [0, 3, 7, 11, min(16, n - 2), n - 1],
    "four": lambda n: [1, 4, 8, 12],   # a 4-qubit window: tc_prepare pads it with idle positions
}
STATES = ("gauss", "gauss_x2^40", "gauss_x2^-40", "sparse")


def block_program(n, pos, seed):
    """9 unitary gates touching every qubit of `pos`, then a differentiable two-qubit density on two of them."""
    rng = np.random.default_rng(seed)
    o = OracleCircuit(n)
    const, var = [], []
    pairs = [(pos[i], pos[i + 1]) for i in range(0, len(pos) - 1, 2)]
    while len(pairs) < 9:
        a, b = rng.choice(len(pos), size=2, replace=False)
        pairs.append((pos[a], pos[b]) if rng.random() < 0.7 else (pos[a], -1))
    for k, (a, b) in enumerate(pairs):
        if rng.random() < 0.5:
            a, b = (b, a) if b >= 0 else (a, b)
        variable = k % 2 == 0
        if b < 0:
            (o.add_q1_var_gate if variable else o.add_q1_const_gate)(a)
            g = haar_unitary(rng, 2)
        elif rng.random() < 0.3:
            (o.add_q2_var_gate_diag if variable else o.add_q2_const_gate_diag)(a, b)
            g = np.exp(1j * rng.normal(size=4))
        else:
            (o.add_q2_var_gate if variable else o.add_q2_const_gate)(a, b)
            g = haar_unitary(rng, 4)
        (var if variable else const).append(g.astype(np.complex64))
    o.get_q2_dens_op_with_grad(pos[-1], pos[0])
    return o, const, var


def initial_state(kind, n, pos, seed):
    rng = np.random.default_rng(seed)
    gauss = rng.normal(size=1 << n) + 1j * rng.normal(size=1 << n)
    gauss /= np.linalg.norm(gauss)
    idx = np.arange(1 << n)
    if kind == "gauss":
        v = gauss
    elif kind == "gauss_x2^40":
        v = gauss * 2.0 ** 40
    elif kind == "gauss_x2^-40":
        v = gauss * 2.0 ** -40
    elif kind == "unbalanced":
        # top qubit 0 (every CTA's first tile: tile index < 148 < 2^(n - 12) / 2): magnitude 2^-12; top qubit 1:
        # 2^(-3 popcount(j)), j the block-qubit index, so one tile's fill warps see values up to 18 binades apart
        assert n - 1 not in pos
        pop = sum((idx >> p) & 1 for p in pos)
        mag = np.where((idx >> (n - 1)) & 1, 2.0 ** (-3.0 * pop), 2.0 ** -12)
        v = mag * np.exp(2j * np.pi * rng.random(1 << n))
    else:
        # sparse: non-zero only where the two highest non-block qubits are both 1, so the first tiles of the CTAs are
        # all zero (seed exponent 0, clamped by magic_of)
        hi = [q for q in range(n - 1, -1, -1) if q not in pos][:2]
        v = gauss * (((idx >> hi[0]) & 1) & ((idx >> hi[1]) & 1))
    return v.astype(np.complex64)


def _rel(got, ref):
    got = [np.asarray(g).reshape(-1) for g in got]
    ref = [np.asarray(r).reshape(-1) for r in ref]
    return max(float(np.abs(g - r).max()) for g, r in zip(got, ref)) / max(float(np.abs(r).max()) for r in ref)


def measure(n, pos_name, state):
    """Per-block errors of every (products, tc_rev) setting of one case: {(products, tc_rev): {fwd, grad, back}}."""
    from quantum_differentiable_circuit import Circuit
    pos = POSITIONS[pos_name](n)
    seed = 1000 * n + len(pos) + sorted(POSITIONS).index(pos_name)
    o, const, var = block_program(n, pos, seed)
    init = initial_state(state, n, pos, seed + 1)
    o.set_state_from_vector(init)
    dens_o = o.forward(const, var)
    fwd_o = o.state.copy()
    rng = np.random.default_rng(seed + 2)
    a = rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4))
    ct = ((a + a.conj().T) / 2 * (np.abs(dens_o[0]).max() or 1.0) ** -1)   # an O(1) loss gradient for every scale
    grads_o = o.backward([ct], const, var)
    back_o = o.state
    out = {}
    for products in (6, 8):
        for tc_rev in (1, 0):
            c = Circuit(n, precision="f32")
            for k, v in (("tc", 1), ("tc_products", products), ("tc_rev", tc_rev), ("profile", 1)):
                c.set_option(k, v)
            c.set_state_from_vector(init)
            for inst in o.instructions:
                name = {0: "add_q2_const_gate", 1: "add_q2_var_gate", 4: "add_q2_const_gate_diag",
                        5: "add_q2_var_gate_diag", 6: "add_q1_const_gate", 8: "add_q1_var_gate",
                        12: "get_q2_dens_op_with_grad"}[inst[0]]
                getattr(c, name)(*inst[1:])
            c.forward(const, var)
            prof = c.last_profile()
            assert prof.get("tc_fwd", {}).get("launches", 0) == 1, prof
            fwd = c.get_cpu_state_copy()
            grads = c.backward([ct.astype(np.complex64)], const, var)
            assert c.last_profile().get("tc_bwd", {}).get("launches", 0) > 0
            back = c.get_cpu_state_copy()
            del c
            gc.collect()
            out[(products, tc_rev)] = {"fwd": _rel([fwd], [fwd_o]), "grad": _rel(grads, grads_o),
                                       "back": _rel([back], [back_o])}
    return out


def _check(n, pos_name, state):
    for (products, tc_rev), e in measure(n, pos_name, state).items():
        assert e["fwd"] < FWD_TOL[products] and e["grad"] < GRAD_TOL and e["back"] < BACK_TOL, (products, tc_rev, e)


@pytest.mark.parametrize("state", STATES)
@pytest.mark.parametrize("pos_name", list(POSITIONS))
@pytest.mark.parametrize("n", [15, 22])
def test_one_tc_block_meets_its_error_bound(pkg, n, pos_name, state):
    _check(n, pos_name, state)


@pytest.mark.parametrize("pos_name", ["low", "1_2_not_0", "four"])
def test_one_tc_block_meets_its_error_bound_on_an_unbalanced_state(pkg, pos_name):
    _check(22, pos_name, "unbalanced")

"""GPU parity at the sizes that are MEASURED (bench.py: 32 local qubits, default tile geometry, fuse = 2):

* 30 q, the largest size of the unmodified reference CUDA library (`int` shifts, SURVEY.md App. B): brickwork
  depth 4 + ring densities, f32 and f64, default tiles (2^12 / 2^11) -- against the f64 per-gate streaming executor's
  results stored in tests/golden/brickwork_30q_f64.npz (tests/golden/make_brickwork_golden.py), and against the
  reference's own library where oracle/_ref is built;
* 32 q f32, the benchmark's size (64-bit tile addressing, `TileGeo::tile` / `BitDeposit`): against the shift-patched
  build of the reference library and against the per-gate streaming executor.

Style of src/test_autodiff.py:133-165: every density and every gradient entry, relative to the largest entry, at
north_star's 1e-5 (f32) / 1e-12 (f64).  The reference needs four resident state buffers (src/circuit.rs:96-102,
396-398), so at 32 q (4 x 32 GiB) the two libraries run one after the other.
"""
import gc
import importlib
import json
import os

import numpy as np
import pytest

from oracle import ref_replay as rr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_30Q = os.path.join(ROOT, "tests", "golden", "brickwork_30q_f64.npz")


def _free_gib():
    import torch
    return torch.cuda.mem_get_info()[0] / 2.0 ** 30


def _record(name, payload):
    """Keep the measured deviations (gpurun_out/ travels back from the GPU box)."""
    try:
        d = os.path.join(ROOT, "gpurun_out")
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "parity_large.jsonl"), "a") as f:
            f.write(json.dumps({"test": name, **payload}) + "\n")
    except OSError:
        pass


def _run(circ, var, cts_conj):
    dens = circ.forward([], var)
    grads = circ.backward(cts_conj, [], var)
    return [np.array(d) for d in dens], [np.array(g) for g in grads]


def _max_rel(got, ref):
    scale = max(float(np.abs(r).max()) for r in ref)
    return max(float(np.abs(np.asarray(g).reshape(-1) - np.asarray(r).reshape(-1)).max()) for g, r in zip(got, ref)) / scale


def _ours(n, depth, precision, options=()):
    bench = importlib.import_module("bench")
    from quantum_differentiable_circuit import Circuit
    dtype = np.complex64 if precision == "f32" else np.complex128
    var, cts = bench.brickwork_inputs(n, depth, dtype)
    c = Circuit(n, precision=precision)
    for k, v in options:
        c.set_option(k, v)
    bench.build_brickwork(c, n, depth)
    out = _run(c, var, [x.conj() for x in cts])
    passes = c.last_stats()["hbm_passes"]
    del c
    gc.collect()
    return out, passes


def _reference(n, depth, precision):
    bench = importlib.import_module("bench")
    dtype = np.complex64 if precision == "f32" else np.complex128
    var, cts = bench.brickwork_inputs(n, depth, dtype)
    r = rr.RefCircuit(n, precision)
    bench.build_brickwork(r, n, depth)
    out = _run(r, var, [x.conj() for x in cts])
    r.state_t.drop(); r.initial_t.drop()
    del r
    gc.collect()
    return out


def _stored(depth, precision):
    """Densities and gradients of the 30 q brickwork from the f64 per-gate streaming executor, for inputs of the given
    precision (tests/golden/make_brickwork_golden.py)."""
    z = np.load(GOLDEN_30Q)
    return list(z[f"depth{depth}/{precision}/densities"]), list(z[f"depth{depth}/{precision}/gradients"])


@pytest.mark.parametrize("precision,options", [("f32", ()), ("f32", (("tc", 0),)), ("f64", ())],
                         ids=["f32-default(tensor-core blocks)", "f32-fp32-tile-kernels", "f64"])
def test_default_tiles_match_the_unmodified_reference_at_30q(pkg, precision, options):
    n, depth = 30, 4
    live = rr.ref_available(precision)
    need = (2 + 4 * live) * (8 if precision == "f32" else 16) + 2
    if _free_gib() < need:
        pytest.skip(f"needs {need} GiB of free device memory")
    tol = 1e-5 if precision == "f32" else 1e-12
    # library defaults: fuse = 2; f32: tensor-core 6-qubit blocks (tc = 0: 2^12 FP32 tiles); f64: 2^11 tiles
    (dens, grads), passes = _ours(n, depth, precision, options)
    assert passes < 2 * 58 / 3, "a fused executor must be the one that ran"
    dens_s, grads_s = _stored(depth, precision)
    rec = {"precision": precision, "options": dict(options), "depth": depth, "hbm_passes": passes,
           "err_density_vs_stored": _max_rel(dens, dens_s), "err_gradient_vs_stored": _max_rel(grads, grads_s)}
    if live:
        dens_r, grads_r = _reference(n, depth, precision)
        rec["err_density"], rec["err_gradient"] = _max_rel(dens, dens_r), _max_rel(grads, grads_r)
    _record("30q_vs_reference", rec)
    assert rec["err_density_vs_stored"] < tol and rec["err_gradient_vs_stored"] < tol, rec
    if live:
        assert rec["err_density"] < tol and rec["err_gradient"] < tol, rec


def test_default_tiles_match_reference_and_per_gate_executor_at_32q(pkg):
    """The benchmark's register: 2^32 amplitudes, tile bases beyond 32 bits.

    At this size the REFERENCE's own f32 gradient reduction is the least accurate party: every thread of its
    <<<128,128>>> launch adds 2^31 / 16384 = 131072 products sequentially in f32 (src/primitives.cu:222-247).
    Measured on B200: tiled vs per-gate executor 1.7e-7, either of them vs the reference 4.2e-5.  The f64
    build (which matched the reference's f64 build to 1e-15 at 30 q, profiles/r2_parity_30q_32q_final.jsonl) is
    therefore the arbiter:
    this library must be within 1e-5 of it, and its distance to the reference must be explained by the
    reference's own distance to the arbiter."""
    n, depth = 32, 2
    if _free_gib() < 4 * 32 + 4:
        pytest.skip("needs 132 GiB of free device memory")
    (dens, grads), passes = _ours(n, depth, "f32")
    (dens0, grads0), passes0 = _ours(n, depth, "f32", (("fuse", 0),))
    assert passes < passes0 / 3
    e0d, e0g = _max_rel(dens, dens0), _max_rel(grads, grads0)
    rec = {"precision": "f32", "depth": depth, "err_density_vs_per_gate": e0d, "err_gradient_vs_per_gate": e0g}
    assert abs(float(np.trace(dens[0]).real) - 1.0) < 1e-5
    (dens64, grads64), _ = _ours(n, depth, "f64")                    # arbiter (2 x 64 GiB)
    rec["err_density_vs_f64"] = _max_rel(dens, dens64)
    rec["err_gradient_vs_f64"] = _max_rel(grads, grads64)
    if rr.ref_available("f32", big=True):
        dens_r, grads_r = _reference(n, depth, "f32")
        rec["err_density_vs_reference"] = _max_rel(dens, dens_r)
        rec["err_gradient_vs_reference"] = _max_rel(grads, grads_r)
        rec["reference_err_density_vs_f64"] = _max_rel(dens_r, dens64)
        rec["reference_err_gradient_vs_f64"] = _max_rel(grads_r, grads64)
    _record("32q", rec)
    assert e0d < 1e-5 and e0g < 1e-5, rec
    assert rec["err_density_vs_f64"] < 1e-5 and rec["err_gradient_vs_f64"] < 1e-5, rec
    if "err_density_vs_reference" in rec:
        # |ours - ref| <= |ours - exact| + |ref - exact|: nothing beyond the reference's own rounding error
        assert rec["err_density_vs_reference"] < 1e-5 + rec["reference_err_density_vs_f64"], rec
        assert rec["err_gradient_vs_reference"] < 1e-5 + rec["reference_err_gradient_vs_f64"], rec


def test_tensor_core_blocks_at_depth_40_against_the_f64_build_at_30q(pkg):
    """Accumulated rounding of the tensor-core blocks at a realistic depth: 30 q brickwork depth 40 (620 gates, ~70
    blocks forward, as many fused reverse steps) against the f64 build as arbiter (which matched the reference's f64
    build to 1e-15 at 30 q, profiles/r2_parity_30q_32q_final.jsonl), with 8 (default) and 6 slice products per block, and the FP32 tile kernels beside them."""
    n, depth = 30, 40
    if _free_gib() < 2 * 16 + 2 * 8 + 4:
        pytest.skip("needs 52 GiB of free device memory")
    (dens64, grads64), _ = _ours(n, depth, "f64")
    rec = {"precision": "f32", "depth": depth}
    for name, options in (("tc8", (("tc", 1), ("tc_products", 8))), ("tc6", (("tc", 1), ("tc_products", 6))), ("fp32_tiles", (("tc", 0),))):
        (dens, grads), _ = _ours(n, depth, "f32", options)
        rec["err_density_" + name] = _max_rel(dens, dens64)
        rec["err_gradient_" + name] = _max_rel(grads, grads64)
    _record("30q_depth40_vs_f64", rec)
    for name in ("tc8", "tc6", "fp32_tiles"):
        assert rec["err_density_" + name] < 1e-5 and rec["err_gradient_" + name] < 1e-5, rec

"""Densities and gradients of the 30-qubit brickwork circuits that tests/test_large_gpu.py and tests/test_tc_gpu.py
compare with, stored in brickwork_30q_f64.npz so that those tests need nothing outside the repository.

The values are computed by this library's f64 build with the per-gate streaming executor (fuse = 0): one kernel
pass per gate, and a reverse pass that un-computes, pulls back and reduces gate by gate as the reference's
src/circuit.rs does.  The tests run the default executors (tiled passes, tensor-core blocks), so they compare two
different code paths.  They are not the reference's own outputs, which need the reference's library (oracle/_ref,
built by oracle/Makefile from the reference's sources); where that library is built the tests also compare with it.

Inputs are bench.brickwork_inputs (seeded).  Under "f32" the gates and cotangents are first rounded to complex64,
the inputs an f32 run receives, and then computed in f64; under "f64" they are used as generated.  Rounded gates
are unitary only to about 6e-8, so the "f32" values are not those of a light-cone window of the register: the
norm changes made by gates outside the window show up at about 1e-7.

    python tests/golden/make_brickwork_golden.py [out.npz]      # one B200, about 50 GB of device memory
"""
import gc
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

N = 30
CASES = [(4, "f32"), (4, "f64"), (8, "f32")]     # (depth, precision of the inputs)


def _run(n, depth, inputs):
    bench = importlib.import_module("bench")
    from quantum_differentiable_circuit import Circuit
    var, cts = bench.brickwork_inputs(n, depth, np.complex64 if inputs == "f32" else np.complex128)
    var = [v.astype(np.complex128) for v in var]
    cts = [c.astype(np.complex128) for c in cts]
    c = Circuit(n, precision="f64")
    c.set_option("fuse", 0)
    bench.build_brickwork(c, n, depth)
    dens = np.stack([np.array(d).reshape(4, 4) for d in c.forward([], var)])
    grads = np.stack([np.array(g).reshape(16) for g in c.backward([x.conj() for x in cts], [], var)])
    del c
    gc.collect()
    return dens, grads


def main(out_path):
    importlib.import_module("differentiable-quantum-circuit-cuda_b200")
    data = {}
    for depth, inputs in CASES:
        dens, grads = _run(N, depth, inputs)
        data[f"depth{depth}/{inputs}/densities"] = dens
        data[f"depth{depth}/{inputs}/gradients"] = grads
    np.savez_compressed(out_path, **data)
    print("wrote", out_path, len(data), "arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(__file__), "brickwork_30q_f64.npz"))

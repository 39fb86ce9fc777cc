"""Digests of the reference's compiled CPU backend's outputs over the randomised sweeps of tests/test_oracle_golden.py,
produced by RUNNING THE REFERENCE'S OWN KERNELS (oracle/_ref, compiled from the reference's sources by oracle/build_ref.py):

    python oracle/build_ref.py && python tests/golden/make_golden_compiled_reference.py

Writes tests/golden/compiled_reference_digests.npz: one SHA-256 per output of each sweep, in sweep order.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))

if __name__ == "__main__":
    sys.path[:0] = [REPO, os.path.join(REPO, "tests")]
    from oracle import oracle as O
    from oracle.build_ref import load_ref
    from test_oracle_golden import _digest, sweep_block_residual, sweep_ops

    ref = load_ref()
    assert ref is not None, "oracle/_ref is missing (python oracle/build_ref.py)"
    O.build()
    out = {key: np.array([_digest(ref_out().numpy()) for _, ref_out in sweep(O, ref)])
           for key, sweep in (("ops", sweep_ops), ("block_residual", sweep_block_residual))}
    np.savez_compressed(os.path.join(HERE, "compiled_reference_digests.npz"), **out)
    print({k: len(v) for k, v in out.items()})

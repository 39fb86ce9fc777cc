"""Golden output of the reference's own CUDA path, produced by RUNNING THE REFERENCE ITSELF on a GPU:

    python baseline/build_ref.py && python tests/golden/make_golden_reference_cuda.py [OUT.npz]

baseline/run_reference.py runs the unmodified reference (its python package, its sige.cuda kernels rebuilt for sm_100a,
cuDNN, fp32 with TF32 off) on the DDPM-256 workload at a 1.2 % edit, with this repository's numpy-seeded weights and
inputs.  Written to tests/golden/ddpm256_reference_cuda_golden.npz (or OUT.npz):

    sparse_delta_q,      the sparse step on the edited image at full resolution, stored as its difference from the
    sparse_delta_scale   reference's CPU-path output in ddpm256_golden.npz (same weights, inputs and edit; the two paths
                         differ by a few 1e-6): sparse_out = golden sparse_out + sparse_delta_q * sparse_delta_scale,
                         int8 steps of scale = max |difference| / 127, so the rebuilt output is within scale / 2 of the
                         CUDA path's (3e-8 for the stored run) and the file stays small
    full0_sub            the dense pass on the original image, every 4th row and column: (1, 3, 64, 64) float32
    ratio, gpu           the edit ratio and the device the reference ran on
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
RATIO = 0.012


def store(out, sparse_out, full0_out, gpu):
    cpu = np.load(os.path.join(HERE, "ddpm256_golden.npz"))
    assert float(cpu["ratio"][0]) == RATIO
    delta = sparse_out.astype(np.float64) - cpu["sparse_out"]
    scale = max(float(np.abs(delta).max()), 1e-30) / 127
    np.savez_compressed(out, sparse_delta_q=np.round(delta / scale).astype(np.int8), sparse_delta_scale=np.array([scale]),
                        full0_sub=full0_out[:, :, ::4, ::4].astype(np.float32), ratio=np.array([RATIO]), gpu=np.array([gpu]))


if __name__ == "__main__":
    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import loader

    assert loader.available(cuda=True), "baseline/_ref/sige/cuda.so is missing (python baseline/build_ref.py)"
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ddpm256_reference_cuda_golden.npz")
    dump = os.path.join(tempfile.mkdtemp(prefix="sige_refcuda_"), "ref.npz")
    r = subprocess.run([sys.executable, os.path.join(REPO, "baseline", "run_reference.py"), "--backend", "cuda", "--no-tf32", "--steps", "2",
                        "--warmup", "1", "--ratio", str(RATIO), "--dump", dump], env=loader.reference_env(), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    info = json.loads(r.stdout.strip().splitlines()[-1])
    assert info["sige_file"].startswith(os.path.realpath(os.path.join(REPO, "baseline", "_ref"))), info
    ref = np.load(dump)
    store(out, ref["sparse_out"], ref["full0_out"], info["gpu"])
    print("%s: %d bytes (reference on %s)" % (out, os.path.getsize(out), info["gpu"]))

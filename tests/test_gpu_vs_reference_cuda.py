"""Ours vs the REFERENCE'S OWN CUDA PATH on a B200 (north star: "outputs match the reference's own CUDA path on
identical inputs").  tests/golden/ddpm256_reference_cuda_golden.npz holds what the unmodified reference — its python
package, its sige.cuda kernels rebuilt for sm_100a, cuDNN, fp32 without TF32 — computed for the DDPM-256 workload
(tests/golden/make_golden_reference_cuda.py: the sparse output at full resolution, the dense one at every 4th pixel); this
process runs the same architecture on this repository's sige.  Same weights, same inputs (numpy-seeded)."""
import numpy as np
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def reference_cuda_run():
    G = golden("ddpm256_reference_cuda_golden.npz")
    cpu = golden("ddpm256_golden.npz")
    assert float(cpu["ratio"][0]) == float(G["ratio"][0])
    sparse = (cpu["sparse_out"] + G["sparse_delta_q"].astype(np.float64) * G["sparse_delta_scale"][0]).astype(np.float32)
    return {"full0_sub": G["full0_sub"], "sparse_out": sparse}, {"gpu": str(G["gpu"][0]), "ratio": float(G["ratio"][0])}


def test_against_the_references_own_cuda_path(reference_cuda_run):
    import warnings

    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, SIGEDDPMUNet, init_deterministic, synthetic_inputs

    ref, info = reference_cuda_run
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        cfg = DDPMConfig()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model = init_deterministic(SIGEDDPMUNet(cfg), seed=0).eval().to(DEV)
        x0, x1, mask, t = synthetic_inputs(cfg, info["ratio"], seed=0)
        with torch.no_grad():
            model.set_mode("full")
            full0 = model(x0.to(DEV), t.to(DEV))
            model.set_masks(downsample_mask(mask.to(DEV), min_res=8))
            model.set_mode("sparse")
            model.set_fused(False)
            ours_fp32 = model(x1.to(DEV), t.to(DEV))                  # eager operator modules, exact fp32 kernels
            model.set_fused(True, dtype=torch.float16)
            ours_fused = model(x1.to(DEV), t.to(DEV))                 # fused step, fp16 tensor-core arithmetic
            assert model.fused_step is not None and model.fused_step.eager_nodes == []
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    want = ref["sparse_out"]
    scale = np.abs(want).max()
    e_full = np.abs(full0.cpu().numpy()[:, :, ::4, ::4] - ref["full0_sub"]).max() / np.abs(ref["full0_sub"]).max()
    e32 = np.abs(ours_fp32.cpu().numpy() - want).max() / scale
    e16 = np.abs(ours_fused.cpu().numpy() - want).max() / scale
    big = np.abs(want) >= 0.05 * scale
    r16 = (np.abs(ours_fused.cpu().numpy() - want)[big] / np.abs(want[big])).max()
    print("vs the reference's CUDA path on %s: dense pass %.3g; sparse fp32 modules %.3g; sparse fp16 fused max %.3g rel(|ref|>5%%) %.3g" % (info["gpu"], e_full, e32, e16, r16))
    assert e_full <= 1e-5, "same dense pass (same cuDNN) expected"
    assert e32 <= 1e-5, "fp32 operator modules vs the reference's CUDA kernels + cuDNN (north star: 1e-5 rel fp32)"
    assert e16 <= 5e-3, "fp16 fused step vs the reference's fp32 CUDA path"

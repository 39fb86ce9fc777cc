"""Tracing + lowering of an unmodified forward (sige_b200.lazy / sige_b200.fused), checked on the CPU.

The launch records the lowering produces are interpreted by tests/sim_executor.py (plain fp32 torch ops following
the contract of include/sige_b200.h) and the result is compared with the golden output the REFERENCE produced for the
same weights and inputs (tests/golden/*.npz, made by tests/golden/make_golden.py).  This pins WHICH launches are
emitted, with which buffers, folds and index lists; the kernels themselves are checked on the GPU.
"""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

from conftest import REPO, golden

sys.path.insert(0, os.path.join(REPO, "tests"))
sys.path.insert(0, os.path.join(REPO, "baseline"))


def _prepared(kind, cfg, ratio):
    import loader
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import SIGEDDPMUNet, init_deterministic, synthetic_inputs

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if kind == "reference":
            if not loader.available():
                pytest.skip("baseline/_ref absent (python baseline/build_ref.py)")
            model = loader.reference_ddpm_on_this_repo(cfg)
        else:
            model = SIGEDDPMUNet(cfg)
        model = init_deterministic(model, seed=0).eval()
    x0, x1, mask, t = synthetic_inputs(cfg, ratio, seed=0)
    with torch.no_grad():
        model.set_mode("full")
        model(x0, t)
        model.set_masks(downsample_mask(mask, min_res=8))
        model.set_mode("sparse")
    return model, x1, t


@pytest.mark.parametrize("kind", ["reference", "intree"])
@pytest.mark.parametrize("opts", [{}, {"producer_preop": False}, {"fuse_shortcut": False, "sparse_stem": False}, {"tc5": False}])
def test_traced_ddpm_small_matches_reference_golden(kind, opts):
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig
    from sim_executor import SimExecutor

    G = golden("ddpm_small_golden.npz")
    model, x1, t = _prepared(kind, DDPMConfig.small(), float(G["ratio"][0]))
    with torch.no_grad():
        step = FusedStep(model, x1, t, executor=SimExecutor(), **opts)
    assert step.eager_nodes == [], "every op of the DDPM forward must be lowered to a fused launch"
    kinds = [k for k, _ in step.steps]
    assert kinds.count("conv_in") == 1 and kinds.count("tail") == 1 and kinds.count("attention") == 4
    n_sc = sum(1 for f in step.fused if f.spec.shortcut is not None)
    assert (n_sc > 0) == (opts.get("fuse_shortcut", True) and opts.get("tc5", True) and opts.get("producer_preop", True))
    ref = G["sparse_out"]
    out = step.output.numpy()
    assert np.abs(out - ref).max() / np.abs(ref).max() < 1e-5
    # a replay rewrites the same tiles with the same values
    again = step.replay().numpy().copy()
    assert np.array_equal(out, again)


def test_traced_reference_ddpm256_launch_list():
    """The north-star model file, unmodified: 86 fused launches + stem + 6 attention cores + tail, nothing eager."""
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig
    from sim_executor import SimExecutor

    G = golden("ddpm256_golden.npz")
    model, x1, t = _prepared("reference", DDPMConfig(), float(G["ratio"][0]))
    with torch.no_grad():
        step = FusedStep(model, x1, t, executor=SimExecutor())
    assert step.eager_nodes == []
    assert len(step.fused) == 86 and [k for k, _ in step.steps].count("attention") == 6
    names = [f.name for f in step.fused]
    assert "down.0.block.0.scatter_gather" in names and "up.0.block.2.scatter" in names
    # tile counts of the reference (golden): 64 tiles at 256^2
    assert step.fused[0].spec.N == 64
    ref = G["sparse_out"]
    assert np.abs(step.output.numpy() - ref).max() / np.abs(ref).max() < 1e-5


def test_eager_islands_keep_the_result_exact():
    """An op the lowering does not know (here: the attention core with its kernel disabled) runs as recorded torch calls
    between the fused launches; everything around it stays fused."""
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig
    from sim_executor import SimExecutor

    G = golden("ddpm_small_golden.npz")
    model, x1, t = _prepared("intree", DDPMConfig.small(), float(G["ratio"][0]))
    with torch.no_grad():
        step = FusedStep(model, x1, t, executor=SimExecutor(), fused_attention=False)
    assert "softmax" in step.eager_nodes and len(step.fused) == 34
    ref = G["sparse_out"]
    assert np.abs(step.output.numpy() - ref).max() / np.abs(ref).max() < 1e-5


def test_attention_outside_the_cluster_kernels_range_takes_the_flash_kernel():
    """The miniature's 128-channel attention cores are below the cluster attention kernel's range (256 / 512 channels): they go out
    as `sige_sparse_attention` launches on the channel slices of the NHWC qkv buffer — nothing eager (what `smoke()` asserts on
    the GPU box)."""
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig
    from sim_executor import SimExecutor

    class NoClusterAttention(SimExecutor):
        def attention_supported(self, n_tokens, channels):
            return False

    G = golden("ddpm_small_golden.npz")
    model, x1, t = _prepared("intree", DDPMConfig.small(), float(G["ratio"][0]))
    with torch.no_grad():
        step = FusedStep(model, x1, t, executor=NoClusterAttention())
    kinds = [k for k, _ in step.steps]
    assert step.eager_nodes == [] and kinds.count("sparse_attention") == 4 and kinds.count("attention") == 0 and len(step.fused) == 34
    ref = G["sparse_out"]
    assert np.abs(step.output.numpy() - ref).max() / np.abs(ref).max() < 1e-5


def test_foreign_math_on_the_tile_stack_falls_back_per_op():
    """GauGAN-style: plain torch math on the gathered stack between Gather and the conv
    (reference gaugan/models/sige_normalization.py:84-86).  The gather is materialised, the torch ops run as recorded,
    and the conv + scatter still go out as ONE fused launch that reads the stack."""
    from torch import nn

    from sige.nn import Gather, Scatter, SIGEConv2d, SIGEModel, SIGEModule
    from sige_b200.fused import FusedStep
    from sige_b200.masks import reduce_mask  # noqa: F401
    from sim_executor import SimExecutor

    class Block(SIGEModule):
        def __init__(self):
            super().__init__()
            self.conv = SIGEConv2d(64, 64, 3, padding=1)
            self.gather = Gather(self.conv, 6)
            self.scatter = Scatter(self.gather)

        def forward(self, x, gamma):
            h = self.gather(x)
            if self.mode == "sparse":
                h = nn.functional.leaky_relu(h * (1 + gamma), 0.2)
            else:
                h = nn.functional.leaky_relu(x * (1 + gamma), 0.2)
            return self.scatter(self.conv(h))

    class Net(SIGEModel):
        def __init__(self):
            super().__init__()
            self.block = Block()

        def forward(self, x):
            return self.block(x, 0.25)

    torch.manual_seed(0)
    net = Net().eval()
    x0 = torch.randn(1, 64, 24, 32)
    mask = torch.zeros(24, 32, dtype=torch.bool)
    mask[5:9, 20:27] = True
    x1 = x0 + torch.randn_like(x0) * mask
    with torch.no_grad():
        net.set_mode("full")
        net(x0)
        dense = net(x1)
        net(x0)
        net.set_masks({(24, 32): mask})
        net.set_mode("sparse")
        step = FusedStep(net, x1, executor=SimExecutor())
    assert len(step.fused) == 1 and step.fused[0].spec.src_is_stack and step.fused[0].spec.dst is not None
    assert any(n.startswith("gather") for n in step.eager_nodes) and "leaky_relu" in step.eager_nodes
    assert torch.allclose(step.output, dense, atol=1e-5)


def test_value_dependent_forward_is_rejected():
    from sige.nn import SIGEModel
    from sige_b200.fused import FusedStep
    from sige_b200.lazy import TraceUnsupported
    from sim_executor import SimExecutor

    class Net(SIGEModel):
        def forward(self, x):
            return x * 2 if float(x.sum()) > 0 else x

    net = Net().eval()
    net.set_mode("sparse")
    with pytest.raises(TraceUnsupported):
        FusedStep(net, torch.ones(1, 8, 4, 4), executor=SimExecutor())


def test_batch_of_independent_edits_equals_one_edit_at_a_time():
    """E edits of ONE original image, each with its own mask, in one fused step (per-tile image index; weights read once):
    row e of the batched output == the single-edit fused output of edit e (BASELINE.json configs[4])."""
    from sige.utils import downsample_mask
    from sige_b200.fused import FusedStep
    from sige_b200.masks import stack_mask_pyramids
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs
    from sim_executor import SimExecutor

    cfg = DDPMConfig.small()
    model, _, t = _prepared("intree", cfg, 0.05)
    edits = []
    for e, (ratio, shift) in enumerate([(0.05, (0, 0)), (0.02, (-14, 9)), (0.09, (11, -13))]):
        x0, x1, mask, _ = synthetic_inputs(cfg, ratio, seed=0, edit_seed=e)
        mask = torch.roll(mask, shift, (0, 1))                      # edits at different places
        x1 = x0 + torch.roll(x1 - x0, shift, (2, 3))
        edits.append((x1, mask))
    singles = []
    with torch.no_grad():
        for x1, mask in edits:
            model.set_masks(downsample_mask(mask, min_res=8))
            singles.append(FusedStep(model, x1, t, executor=SimExecutor()).output.clone())
        model.set_masks(stack_mask_pyramids([downsample_mask(m, min_res=8) for _, m in edits]))
        xb = torch.cat([x for x, _ in edits], 0)
        step = FusedStep(model, xb, t, executor=SimExecutor())
    assert step.eager_nodes == [] and step.output.shape[0] == 3
    sparse = [f for f in step.fused if f.spec.tile_img is not None]
    assert len(sparse) > 10 and sparse[0].spec.N == sum(int((f.spec.tile_img == e).sum()) for f in sparse[:1] for e in range(3))
    for e in range(3):
        assert torch.allclose(step.output[e], singles[e][0], atol=2e-5), "edit %d differs from its single-edit step" % e
    # the eager operator modules share one tile list across the batch: they must refuse, not mis-compute
    model.set_fused(False)
    with pytest.raises((NotImplementedError, RuntimeError)):
        with torch.no_grad():
            model(xb, t)


def test_new_masks_are_installed_without_recompiling():
    """A later edit with its own mask re-uses the compiled step: `set_masks` + the next call rewrite the fixed-capacity index
    buffers (padded with SIGE_TILE_NONE), the shortcut flags and restore the cached buffers — same result as a fresh build."""
    from sige.utils import downsample_mask
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs
    from sim_executor import SimExecutor

    cfg = DDPMConfig.small()
    model, x_a, t = _prepared("intree", cfg, 0.05)
    x0, _, _, _ = synthetic_inputs(cfg, 0.05, seed=0)
    with torch.no_grad():
        step = FusedStep(model, x_a, t, executor=SimExecutor())
        out_a = step.output.clone()
        n_before = {k: sl.n for k, sl in step.low.slots.items()}
        # edit B: a smaller mask elsewhere in the image (every tile list fits the capacities of edit A)
        _, x_b, mask_b, _ = synthetic_inputs(cfg, 0.03, seed=0, edit_seed=5)
        mask_b = torch.roll(mask_b, (9, -11), (0, 1))
        x_b = x0 + torch.roll(x_b - x0, (9, -11), (2, 3))
        model.set_masks(downsample_mask(mask_b, min_res=8))
        assert step.rebind(), "the new tile lists fit: no recompilation"
        assert {k: sl.n for k, sl in step.low.slots.items()} != n_before
        out_b = step(x_b, t).clone()
        fresh = FusedStep(model, x_b, t, executor=SimExecutor()).output
        assert torch.allclose(out_b, fresh, atol=2e-5), float((out_b - fresh).abs().max())
        assert float((out_b - out_a).abs().max()) > 1e-2
        # back to edit A: identical to the first result (buffers fully restored)
        _, _, mask_a, _ = synthetic_inputs(cfg, 0.05, seed=0)
        model.set_masks(downsample_mask(mask_a, min_res=8))
        assert step.rebind()
        assert torch.allclose(step(x_a, t), out_a, atol=1e-6)
        # a larger mask does not fit: the caller recompiles
        _, _, mask_c, _ = synthetic_inputs(cfg, 0.20, seed=0)
        model.set_masks(downsample_mask(mask_c, min_res=8))
        assert not step.rebind()


def test_device_side_install_of_a_tile_list_pads_truncates_and_flags_overflow():
    """`IdxSlot.install_device` (the sync-free `set_masks_async` path) is plain tensor arithmetic: the first min(count, capacity)
    origins of the reduction, SIGE_TILE_NONE behind them, bit 0 of the status word when the list did not fit — checked here
    on CPU tensors against the host-side `reload`."""
    from types import SimpleNamespace

    from sige_b200._cabi import TILE_NONE
    from sige_b200.fused import IdxSlot

    first = torch.tensor([[0, 0], [0, 4], [4, 8], [8, 8], [12, 0]], dtype=torch.int32)
    g = SimpleNamespace(active_indices=first, tile_images=None)
    sl = IdxSlot(g, torch.device("cpu"), headroom=0.6)
    assert sl.cap == 8 and sl.n == 5 and bool((sl.buf[5:] == TILE_NONE).all())
    cand = torch.arange(40, dtype=torch.int32).view(20, 2)             # what sige_reduce_mask leaves: `count` real rows, garbage behind
    status = torch.zeros(1, dtype=torch.int32)
    sl.install_device(cand, torch.tensor([3], dtype=torch.int32), status)
    assert torch.equal(sl.buf[:3], cand[:3]) and bool((sl.buf[3:] == TILE_NONE).all()) and int(status) == 0
    sl.install_device(cand, torch.tensor([8], dtype=torch.int32), status)       # exactly full
    assert torch.equal(sl.buf, cand[:8]) and int(status) == 0
    sl.install_device(cand, torch.tensor([0], dtype=torch.int32), status)       # no active tile: every entry is padding
    assert bool((sl.buf == TILE_NONE).all()) and int(status) == 0
    sl.install_device(cand, torch.tensor([13], dtype=torch.int32), status)      # does not fit: truncated AND reported
    assert torch.equal(sl.buf, cand[:8]) and int(status) & 1
    short = cand[:5]                                                             # fewer candidate rows than the capacity
    status.zero_()
    sl.install_device(short, torch.tensor([5], dtype=torch.int32), status)
    assert torch.equal(sl.buf[:5], short) and bool((sl.buf[5:] == TILE_NONE).all()) and int(status) == 0
    g.active_indices = first[:2]
    sl.reload()                                                                  # the synchronous path resets the host-side count
    assert sl.n == 2 and torch.equal(sl.buf[:2], first[:2]) and bool((sl.buf[2:] == TILE_NONE).all())

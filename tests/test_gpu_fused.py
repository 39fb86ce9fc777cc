"""The fused step (sige_b200.fused) on the GPU: the DDPM U-Net of the in-tree workload (the reference's architecture, its
parameter names and weights), through the public call ``model(x, t)``, against the reference's golden outputs
(tests/golden/*.npz)."""
import warnings

import numpy as np
import pytest
import torch

from conftest import golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def _exact_fp32_dense_pass():
    """The dense pass of an fp32 model goes through cuDNN; TF32 (torch's default for convolutions) would put 1e-3-level
    noise into the caches and hide what the sparse path itself contributes."""
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


def _model(cfg):
    from sige_b200.workloads.ddpm import SIGEDDPMUNet, init_deterministic

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return init_deterministic(SIGEDDPMUNet(cfg), seed=0).eval()


def _prepared(cfg, ratio, dtype, channels_last=True):
    """dtype fp32: the reference's own flow — fp32 model, fp32 dense pass — with the sparse steps opted into fp16 tensor-core
    arithmetic (set_fused(dtype=...)); dtype fp16: a half model end to end."""
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import synthetic_inputs

    model = _model(cfg).to(DEV).to(dtype)
    if channels_last:
        model = model.to(memory_format=torch.channels_last)
    x0, x1, mask, t = synthetic_inputs(cfg, ratio, seed=0)
    with torch.no_grad():
        model.set_mode("full")
        model(x0.to(DEV).to(dtype), t.to(DEV))
        model.set_masks(downsample_mask(mask.to(DEV), min_res=8))
        model.set_mode("sparse")
    if dtype == torch.float32:
        model.set_fused(True, dtype=torch.float16)
    return model, x1.to(DEV).to(dtype), t.to(DEV)


def _errs(out, ref):
    """(max-normalised max error, max-normalised rms, worst per-element relative error over |ref| >= 5 % of max)."""
    out, ref = np.asarray(out, np.float64), np.asarray(ref, np.float64)
    scale = np.abs(ref).max()
    d = np.abs(out - ref)
    big = np.abs(ref) >= 0.05 * scale
    return d.max() / scale, np.sqrt((d ** 2).mean()) / scale, (d[big] / np.abs(ref[big])).max()


# fp16 tolerances.  Measured on B200 (see DESIGN.md section 5b): DDPM-256 @1.2 % fused-vs-golden max-normalised 2.2e-3;
# the asserted bounds are <= 2x the measured values.
TOL_MAX, TOL_RMS, TOL_REL = 5e-3, 6e-4, 5e-2


@pytest.mark.parametrize("channels_last", [False, True])
def test_ddpm256_model_runs_fused(channels_last):
    """north star: the DDPM-256 U-Net on this repo's sige.nn, full -> set_masks -> sparse through model(x, t); the sparse
    call is ONE fused launch per wrapped layer."""
    from sige_b200.parallel import cache_tensors
    from sige_b200.workloads.ddpm import DDPMConfig

    G = golden("ddpm256_golden.npz")
    model, x1, t = _prepared(DDPMConfig(), float(G["ratio"][0]), torch.float32, channels_last)
    pristine = [(n, v.clone()) for n, v in cache_tensors(model)]
    with torch.no_grad():
        out1 = model(x1, t)
        out2 = model(x1, t)
    step = model.fused_step
    assert step is not None, "the sparse call must have run as a fused step"
    assert step.eager_nodes == [], step.eager_nodes
    assert len(step.fused) == 86 and step.graph is not None
    from sige_b200 import _cabi

    plans = [(_cabi.TileConvPlan(), f) for f in step.fused]
    n_tc5 = 0
    for pl, f in plans:
        assert _cabi.lib().sige_tile_conv_plan(ctypes_ref(f.desc), ctypes_ref(pl)) == 0
        n_tc5 += pl.path
    assert n_tc5 >= 81, "the tcgen05 kernel must carry the step (%d of %d launches)" % (n_tc5, len(step.fused))
    assert out1.dtype == torch.float32 and out1.data_ptr() != out2.data_ptr() and torch.equal(out1, out2), "results are fresh tensors, replay is idempotent"
    for (n, a), (_, b) in zip(pristine, cache_tensors(model)):
        assert torch.equal(a, b), "the fused step must not touch the module caches (%s)" % n
    e_max, e_rms, e_rel = _errs(out1.float().cpu().numpy(), G["sparse_out"])
    print("DDPM-256 model fused (channels_last=%s): max %.3g rms %.3g rel %.3g, %d launches/step" % (channels_last, e_max, e_rms, e_rel, step.launches_per_step))
    assert e_max <= TOL_MAX and e_rms <= TOL_RMS and e_rel <= TOL_REL
    # the eager fp32 operator modules reproduce the reference to fp32 accuracy; the fp16 fused step stays within the fp16 tolerance of them
    model.set_fused(False)
    with torch.no_grad():
        via_modules = model(x1, t).float()
    m_max, _, _ = _errs(via_modules.cpu().numpy(), G["sparse_out"])
    e_mod = float((out1.float() - via_modules).abs().max() / via_modules.abs().max())
    print("eager fp32 modules vs reference golden: %.3g; fused fp16 vs modules: %.3g" % (m_max, e_mod))
    assert model.fused_step is step and m_max <= 2e-5 and e_mod <= TOL_MAX


def ctypes_ref(obj):
    import ctypes

    return ctypes.byref(obj)


@pytest.mark.parametrize("opts", [
    {"tc5": False, "producer_preop": False, "pdl": False, "fused_attention": False, "sparse_stem": False},
    {"tc5": False, "producer_preop": True, "pdl": False},
    {"tc5": True, "producer_preop": True, "pdl": False, "fuse_shortcut": False},
    {"tc5": True, "producer_preop": True, "pdl": True},
    {"tc5": True, "producer_preop": False, "pdl": True},
])
@pytest.mark.parametrize("tag", ["ddpm_small", "ddpm256"])
def test_fused_step_options_vs_modules_and_reference(tag, opts):
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig

    G = golden(tag + "_golden.npz")
    cfg = DDPMConfig.small() if tag == "ddpm_small" else DDPMConfig()
    model, x1, t = _prepared(cfg, float(G["ratio"][0]), torch.float16)
    model.set_fused(False)
    with torch.no_grad():
        via_modules = model(x1, t).float()
        step = FusedStep(model, x1, t, **opts)
    out1 = step.replay().clone()
    out2 = step.replay().clone()
    torch.cuda.synchronize()
    assert torch.equal(out1, out2), "replaying the step must be idempotent (in-place scatter rewrites the same tiles)"
    eager = step.run_eager().clone()
    assert torch.equal(eager, out1), "graph replay == eager launch sequence"
    ref = G["sparse_out"]
    e_mod = float((out1.float() - via_modules).abs().max() / via_modules.abs().max())
    e_max, e_rms, e_rel = _errs(out1.float().cpu().numpy(), ref)
    print("%s %s: fused-vs-modules %.3g, fused-vs-reference max %.3g rms %.3g rel %.3g, %d fused launches, eager: %s" %
          (tag, opts, e_mod, e_max, e_rms, e_rel, len(step.fused), step.eager_nodes))
    assert e_mod <= TOL_MAX and e_max <= TOL_MAX and e_rms <= TOL_RMS
    assert step.launches_per_step >= len(step.fused) > 0


@pytest.mark.parametrize("tag,tol_max,tol_rms", [("ddpm256_r05", 1e-2, 1e-3), ("ddpm256_r15", 2e-2, 2e-3), ("ddpm256_r30", 6e-2, 3e-3)])
def test_fused_step_edit_sweep_vs_reference_golden(tag, tol_max, tol_rms):
    """BASELINE.json configs[4]: 5 / 15 / 30 % edits (256 / 676 / 1296 tiles at 256x256: wide grids, BN = 128, no split-K).
    With random-init weights a large random edit makes the network strongly error-amplifying (the reference's own
    sparse-vs-dense difference is 0.9 at 30 %): two fp16 evaluation orders differ by a few 1e-2 max-normalised while the
    rms stays at the fp16 level; the fp32 module path pins the graph exactly (test_gpu_model.py)."""
    from sige_b200.workloads.ddpm import DDPMConfig

    G = golden(tag + "_golden.npz")
    model, x1, t = _prepared(DDPMConfig(), float(G["ratio"][0]), torch.float32)
    with torch.no_grad():
        out = model(x1, t).float().cpu().numpy()
    assert model.fused_step is not None and model.fused_step.eager_nodes == []
    if "sparse_out" in G.files:
        ref, got = G["sparse_out"], out
    else:
        ref, got = G["sparse_out_sub"], out[:, :, ::2, ::2]
    e_max, e_rms, e_rel = _errs(got, ref)
    print("%s: fused-vs-reference max %.3g rms %.3g rel(|ref|>5%%) %.3g" % (tag, e_max, e_rms, e_rel))
    assert e_max <= tol_max and e_rms <= tol_rms


def test_recompiles_when_masks_or_caches_change():
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model, x1, t = _prepared(cfg, 0.05, torch.float16)
    with torch.no_grad():
        a = model(x1, t)
        s1 = model.fused_step
        model(x1, t)
        assert model.fused_step is s1
        _, x2, mask2, _ = synthetic_inputs(cfg, 0.10, seed=0)
        model.set_masks(downsample_mask(mask2.to(DEV), min_res=8))
        b = model(x2.to(DEV).half(), t)
        s2 = model.fused_step
        assert s2 is not s1 and s2.fused[0].spec.N != s1.fused[0].spec.N
        model.set_fused(False)
        b_mod = model(x2.to(DEV).half(), t)
    assert float((b - b_mod).abs().max() / b_mod.abs().max()) <= TOL_MAX and a.shape == b.shape


def test_batch_of_independent_edits_on_gpu():
    """E edits of one original image, each with its own mask, in ONE fused step (per-tile image index in the tcgen05,
    mma.sync and stem kernels): edit e of the batched output == the single-edit fused step of edit e."""
    from sige.utils import downsample_mask
    from sige_b200.masks import stack_mask_pyramids
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig()
    model, _, t = _prepared(cfg, 0.012, torch.float32)
    edits = []
    for e, (ratio, shift) in enumerate([(0.012, (0, 0)), (0.012, (-70, 45)), (0.03, (60, -80)), (0.006, (-100, -100))]):
        x0, x1, mask, _ = synthetic_inputs(cfg, ratio, seed=0, edit_seed=e)
        mask = torch.roll(mask, shift, (0, 1))
        x1 = x0 + torch.roll(x1 - x0, shift, (2, 3))
        edits.append((x1.to(DEV), mask.to(DEV)))
    singles = []
    with torch.no_grad():
        for x1, mask in edits:
            model.set_masks(downsample_mask(mask, min_res=8))
            singles.append(model(x1, t))
        model.set_masks(stack_mask_pyramids([downsample_mask(m, min_res=8) for _, m in edits]))
        out = model(torch.cat([x for x, _ in edits], 0), t)
    step = model.fused_step
    assert step.eager_nodes == [] and out.shape[0] == len(edits)
    assert sum(1 for f in step.fused if f.spec.tile_img is not None) >= 30
    for e in range(len(edits)):
        d = float((out[e] - singles[e][0]).abs().max() / singles[e][0].abs().max())
        print("edit %d: batched vs single %.3g" % (e, d))
        # same arithmetic per tile; split-K / tile-width choices differ with the total tile count -> fp16 reassociation only
        assert d <= 3e-3


def test_set_masks_again_with_the_same_masks_is_free():
    """Stable Diffusion's sampler calls set_masks(conv_masks) before every step with the same dict
    (stable-diffusion/ldm/models/diffusion/ddim.py:203-204): no kernel, no host sync, the compiled step stays valid."""
    from sige.utils import downsample_mask
    from sige_b200 import ops
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model, x1, t = _prepared(cfg, 0.05, torch.float16)
    _, _, mask, _ = synthetic_inputs(cfg, 0.05, seed=0)
    masks = downsample_mask(mask.to(DEV), min_res=8)
    with torch.no_grad():
        model.set_masks(masks)
        a = model(x1, t)
        step, stamp, launches = model.fused_step, model.timestamp, ops.launch_count
        model.set_masks(masks)
        assert model.timestamp == stamp and ops.launch_count == launches
        b = model(x1, t)
        assert model.fused_step is step and torch.equal(a, b)
        masks2 = {k: v.clone() for k, v in masks.items()}           # new tensors: a real set_masks (one sync for all geometries)
        model.set_masks(masks2)
        assert model.timestamp == stamp + 1
        c = model(x1, t)
    assert torch.equal(a, c)


def test_multi_step_cached_flow_on_the_fused_path():
    """The all-steps cache protocol (reference diffusion_demo/samplers/ddim_ddpm_sampler.py:60-66): dense passes fill
    original_outputs[step] for every step id once; an edit then runs sparse for all steps with no dense pass.  On the fused
    path every step id gets its own compiled step (own buffers, initialised from that id's caches) which later edits with
    the same masks reuse."""
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model = _model(cfg).to(DEV)
    x0, x1, mask, t = synthetic_inputs(cfg, 0.05, seed=0)
    x0, x1, t = x0.to(DEV), x1.to(DEV), t.to(DEV)
    ids = [0, 1, 2]
    with torch.no_grad():
        model.set_mode("full")
        for s in ids:
            model.set_cache_id(s)
            model(x0 * (1 + 0.1 * s), t + 10 * s)
        model.set_masks(downsample_mask(mask.to(DEV), min_res=8))
        model.set_mode("sparse")
        eager, fused, steps = [], [], []
        model.set_fused(False)
        for s in ids:
            model.set_cache_id(s)
            eager.append(model(x1 * (1 + 0.1 * s), t + 10 * s))
        model.set_fused(True, dtype=torch.float16)
        for rnd in range(2):
            for s in ids:
                model.set_cache_id(s)
                out = model(x1 * (1 + 0.1 * s), t + 10 * s)
                if rnd == 0:
                    fused.append(out)
                    steps.append(model.fused_step)
                else:
                    assert model.fused_step is steps[s], "the step compiled for cache id %d is reused" % s
                    assert torch.equal(out, fused[s])
    assert len({id(s) for s in steps}) == 3
    for s in ids:
        e = float((fused[s] - eager[s]).abs().max() / eager[s].abs().max())
        assert e <= TOL_MAX, "cache id %d: fused vs eager %g" % (s, e)
    assert float((eager[0] - eager[1]).abs().max()) > 1e-3, "the step ids really hold different caches"


def test_resblock_entry_point_equals_its_two_launches():
    """sige_resblock (C-ABI): conv1 -> conv2 of one residual block as one call == the two sige_tile_conv launches."""
    import ctypes

    from sige_b200 import _cabi
    from sige_b200.fused import FusedStep
    from sige_b200.workloads.ddpm import DDPMConfig

    model, x1, t = _prepared(DDPMConfig.small(), 0.05, torch.float16)
    with torch.no_grad():
        step = FusedStep(model, x1, t, use_graph=False)
    by_name = {f.name: f for f in step.fused}
    c1, c2 = by_name["down.0.block.0.scatter_gather"], by_name["down.0.block.0.scatter"]
    dst = c2.spec.dst.raw
    step.run_eager()
    torch.cuda.synchronize()
    want = dst.clone()
    dst.zero_()
    stream = torch.cuda.current_stream().cuda_stream
    rc = _cabi.lib().sige_resblock(ctypes.byref(c1.desc), ctypes.byref(c2.desc), stream)
    assert rc == 0, _cabi.last_error()
    torch.cuda.synchronize()
    idx = c2.spec.idx.long()
    # the call rewrites exactly the active output tiles
    for (iy, ix) in idx.tolist()[:8]:
        oy, ox = iy + c2.spec.off, ix + c2.spec.off
        assert torch.equal(dst[:, :, oy:oy + 4, ox:ox + 4], want[:, :, oy:oy + 4, ox:ox + 4])
    # a conv2 that does not read conv1's output is refused
    other = by_name["down.1.block.0.scatter"]
    assert _cabi.lib().sige_resblock(ctypes.byref(c1.desc), ctypes.byref(other.desc), stream) != 0


def test_next_edit_reuses_the_compiled_step():
    """Interactive editing: a NEW mask whose tile lists fit the capacities of the compiled step is installed in place
    (index buffers padded with SIGE_TILE_NONE, shortcut flags, cached buffers restored) — no re-trace, no re-capture."""
    import time

    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig()
    model, x_a, t = _prepared(cfg, 0.012, torch.float32)
    x0, _, _, _ = synthetic_inputs(cfg, 0.012, seed=0)
    with torch.no_grad():
        out_a = model(x_a, t)
        step = model.fused_step
        _, x_b, mask_b, _ = synthetic_inputs(cfg, 0.005, seed=0, edit_seed=3)      # a smaller edit elsewhere: every tile list fits
        mask_b = torch.roll(mask_b, (-60, 44), (0, 1))
        x_b = (x0 + torch.roll(x_b - x0, (-60, 44), (2, 3))).to(DEV)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.set_masks(downsample_mask(mask_b.to(DEV), min_res=8))
        out_b = model(x_b, t)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert model.fused_step is step, "the second edit must re-use the compiled step"
        model.set_fused(False)
        want_b = model(x_b, t)
        model.set_fused(True, dtype=torch.float16)
    e = float((out_b - want_b).abs().max() / want_b.abs().max())
    print("second edit: set_masks + first step %.1f ms (no recompilation), fused-vs-eager %.3g" % (1e3 * dt, e))
    assert e <= TOL_MAX and float((out_b - out_a).abs().max()) > 1e-2


def test_capacity_headroom_lets_a_larger_mask_in():
    """set_fused(headroom=0.5): tile-list buffers 50 % larger than needed — a later, LARGER edit still re-uses the compiled step;
    CTAs made only of SIGE_TILE_NONE padding exit at once (SIGE_CONV_PADDED)."""
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model, x_a, t = _prepared(cfg, 0.04, torch.float16)
    model.set_fused(True, headroom=0.6)
    x0, _, _, _ = synthetic_inputs(cfg, 0.04, seed=0)
    with torch.no_grad():
        model(x_a, t)
        step = model.fused_step
        assert any(sl.cap - sl.n >= 8 for sl in step.low.slots.values())
        _, x_b, mask_b, _ = synthetic_inputs(cfg, 0.055, seed=0, edit_seed=2)       # more tiles than edit A
        model.set_masks(downsample_mask(mask_b.to(DEV), min_res=8))
        out_b = model(x_b.to(DEV).half(), t)
        assert model.fused_step is step
        model.set_fused(False)
        want = model(x_b.to(DEV).half(), t)
    assert float((out_b - want).abs().max() / want.abs().max()) <= TOL_MAX


def test_next_edit_without_a_host_sync():
    """SURVEY section 8f-4: `set_masks_async` reduces the new mask pyramid ON THE DEVICE straight into the fixed-capacity tile lists of
    the compiled step (counts never reach the host), so installing the next edit only enqueues work.  Same result as the
    synchronous path; a mask that does NOT fit is reported by `masks_async_ok()` (device status word), and a following
    synchronous `set_masks` recovers."""
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model, x_a, t = _prepared(cfg, 0.04, torch.float16)
    model.set_fused(True, headroom=0.6)
    with torch.no_grad():
        model(x_a, t)
        step = model.fused_step
        _, x_b, mask_b, _ = synthetic_inputs(cfg, 0.055, seed=0, edit_seed=2)       # more tiles than edit A, within the headroom
        pyr_b = downsample_mask(mask_b.to(DEV), min_res=8)
        x_b = x_b.to(DEV).half()
        torch.cuda.synchronize()
        # the proof of "no host sync": with sync debugging on, any .item() / .cpu() / nonzero in the call would raise
        torch.cuda.set_sync_debug_mode("error")
        try:
            assert model.set_masks_async(pyr_b) is True
            out_b = model(x_b, t)
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert model.fused_step is step and model.masks_async_ok()
        # reference: the synchronous path on a fresh build
        model.set_masks(pyr_b)
        want_fused = model(x_b, t)
        model.set_fused(False)
        want = model(x_b, t)
        model.set_fused(True, headroom=0.6)
        assert torch.equal(out_b, want_fused), "device-installed lists == host-installed lists"
        assert float((out_b - want).abs().max() / want.abs().max()) <= TOL_MAX
        # a much larger edit does not fit: flagged on the device, and the synchronous call rebuilds
        model(x_a, t)
        _, x_c, mask_c, _ = synthetic_inputs(cfg, 0.30, seed=0, edit_seed=4)
        pyr_c = downsample_mask(mask_c.to(DEV), min_res=8)
        if model.set_masks_async(pyr_c):
            assert not model.masks_async_ok()
        model.set_masks(pyr_c)
        out_c = model(x_c.to(DEV).half(), t)
        model.set_fused(False)
        want_c = model(x_c.to(DEV).half(), t)
    assert float((out_c - want_c).abs().max() / want_c.abs().max()) <= 6e-2

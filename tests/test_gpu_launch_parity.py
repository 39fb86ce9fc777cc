"""Every launch of the real fused step against a float64 reference of that one launch.

The step tests (test_gpu_fused.py) compare the network OUTPUT, after ~90 dependent launches, with bounds that a random-init
U-Net forces up to 6e-2; a layer-local error of a few 1e-3 on a handful of tiles can hide under them.  Here the step is built
as the product builds it (``FusedStep``, ``CudaExecutor``) and then walked launch by launch: each launch's inputs and outputs
are snapshotted, the launch runs, and what it wrote is compared with the launch contract of include/sige_b200.h evaluated in
float64 on the snapshot (tests/sim_executor.py: the same functions the CPU simulator runs in fp32).  Later launches see the real
activations, so there is no amplification and the per-layer bar of test_gpu_conv.py applies to every launch:

  * max-normalised error <= 1e-3 (fp16) / 8e-3 (bf16) over everything the launch wrote (destination and every aux view);
  * every element outside the output rectangles of the real tiles (SIGE_TILE_NONE padding is not real) is bit-identical to
    what was there before the launch.

A failure names the launch, its plan (sige_tile_conv_plan) and the worst element as (image, tile, channel, pixel).
"""
import copy
import os
import sys
import types
import warnings
from collections import Counter

import pytest
import torch

from conftest import REPO

sys.path.insert(0, os.path.join(REPO, "tests"))
import sim_executor as contract  # noqa: E402

from sige_b200.fused import CudaExecutor, FusedStep  # noqa: E402
from sim_executor import SimExecutor  # noqa: E402

DEV = "cuda:0"
BOUND = {torch.float16: 1e-3, torch.bfloat16: 8e-3, torch.float32: 1e-5}
_MANT = {torch.float16: 10, torch.bfloat16: 7, torch.float32: 23}
_EMIN = {torch.float16: -14, torch.bfloat16: -126, torch.float32: -126}
_INT = {2: torch.int16, 4: torch.int32, 8: torch.int64}


# ---------------------------------------------------------------------------------------------------------------------
# recording executors: the product executor (or the CPU simulator), plus a note of what each prepared closure was built from
# ---------------------------------------------------------------------------------------------------------------------
class _Recording:
    def _note(self, kind, fn, args):
        self.__dict__.setdefault("records", {})[fn] = (kind, args)
        return fn

    def prepare_conv_in(self, rec):
        return self._note("conv_in", super().prepare_conv_in(rec), rec)

    def prepare_tail(self, *args):
        return self._note("tail", super().prepare_tail(*args), args)

    def prepare_attention(self, qkv_tokens, out_tokens, pdl):
        return self._note("attention", super().prepare_attention(qkv_tokens, out_tokens, pdl), (qkv_tokens, out_tokens))

    def prepare_sparse_attention(self, q, k, v, scale, out):
        return self._note("sparse_attention", super().prepare_sparse_attention(q, k, v, scale, out), (q, k, v, scale, out))

    def prepare_spade(self, x, gamma, beta, slope, out):
        return self._note("spade", super().prepare_spade(x, gamma, beta, slope, out), (x, gamma, beta, slope, out))


class RecordingCudaExecutor(_Recording, CudaExecutor):
    pass


class RecordingSimExecutor(_Recording, SimExecutor):
    pass


# ---------------------------------------------------------------------------------------------------------------------
# snapshots and comparison
# ---------------------------------------------------------------------------------------------------------------------
def _cpu(t):
    return None if t is None else t.detach().to("cpu", copy=True)


def _f64(t):
    return None if t is None else t.to(torch.float64)


def _ulp(a, dtype):
    """1 ulp of `dtype` at |a| (float64 tensor)."""
    e = torch.floor(torch.log2(a.abs().clamp_min(2.0 ** _EMIN[dtype])))
    return torch.exp2(e - _MANT[dtype])


class Result:
    def __init__(self, kind, name, plan=""):
        self.kind, self.name, self.plan = kind, name, plan
        self.err, self.ulps, self.where, self.untouched = 0.0, 0.0, "", True
        self.problems = []

    @property
    def ok(self):
        return not self.problems

    def __repr__(self):
        return "%s %s%s: max-normalised %.3g (%.1f ulp where |ref| >= 5 %% of max) at %s%s" % (
            self.kind, self.name, self.plan, self.err, self.ulps, self.where, "" if self.ok else " -- " + "; ".join(self.problems))


def _compare(res, label, got, before, want, written, dtype, bound, locate):
    """got: the launch's output (device), before: its snapshot, want: float64 reference, written: bool [B, H, W] of written
    pixels or None (all).  Updates `res` with the error and any violation."""
    g = got.detach().cpu()
    m = torch.ones(g.shape, dtype=torch.bool) if written is None else written.view(g.shape[0], 1, *g.shape[2:]).expand(g.shape)
    d = torch.nan_to_num((g.double() - want).abs(), nan=float("inf"))
    d = torch.where(m, d, torch.zeros_like(d))
    if bool(m.any()):
        scale = max(float(want.abs()[m].max()), 1e-30)
        err = float(d.max()) / scale
        big = m & (want.abs() >= 0.05 * scale)          # (near zero one ulp is meaningless: cancellation)
        ulps = float((d / _ulp(want, dtype))[big].max()) if bool(big.any()) else 0.0
        worst = locate(tuple(int(i) for i in torch.unravel_index(d.argmax(), d.shape)))
        if err >= res.err:
            res.err, res.ulps, res.where = err, ulps, "%s %s" % (label, worst)
        if not err <= bound:
            res.problems.append("%s: max-normalised error %.3g > %.3g at %s" % (label, err, bound, worst))
    if written is not None:
        gb, bb = g.view(_INT[g.element_size()]), before.view(_INT[before.element_size()])
        changed = (gb != bb) & ~m
        if bool(changed.any()):
            res.untouched = False
            first = tuple(int(i) for i in changed.nonzero()[0])
            res.problems.append("%s: %d elements outside the real tiles changed, first at (image, channel, y, x) = %s" % (label, int(changed.sum()), first))


def _plan(fc):
    if fc.desc is None:
        return ""
    from ctypes import byref

    from sige_b200 import _cabi

    pl = _cabi.TileConvPlan()
    if _cabi.lib().sige_tile_conv_plan(byref(fc.desc), byref(pl)) != 0:
        return " [plan: error]"
    return " [path %s bn %d ksplit %d deep_ring %d]" % ("tcgen05" if pl.path else "mma.sync", pl.bn, pl.ksplit, pl.deep_ring)


def _check_conv(fc, launch, dtype, stage, bound, perturb=None):
    s = fc.spec
    snap = copy.copy(s)
    snap.srcs = [(_cpu(t), up) for t, up in s.srcs]
    snap.idx, snap.tile_img, snap.scale, snap.shift = _cpu(s.idx), _cpu(s.tile_img), _cpu(s.scale), _cpu(s.shift)
    snap.weight, snap.bias, snap.residual = _cpu(s.weight), _cpu(s.bias), _cpu(s.residual)
    if s.shortcut is not None:
        t_, w_, b_, f_ = s.shortcut
        snap.shortcut = ([_cpu(t) for t in t_], _cpu(w_), _cpu(b_), _cpu(f_))
    outs = []                                # (label, device tensor, snapshot before the launch)
    if s.dst_stack is not None:
        outs.append(("dst", s.dst_stack, _cpu(s.dst_stack)))
    elif s.dst.has_raw:
        outs.append(("dst", s.dst.raw, _cpu(s.dst.raw)))
    outs += [("aux%d" % i, v, _cpu(v)) for i, (v, _, _, _) in enumerate(s.aux)]
    launch()
    wants = {label: _f64(before) for label, _, before in outs}
    if s.dst_stack is not None:
        snap.dst_stack = wants["dst"]
    else:
        snap.dst = types.SimpleNamespace(raw=wants.get("dst"), has_raw=s.dst.has_raw, shape=s.dst.shape)
    snap.aux = [(wants["aux%d" % i], _cpu(sc), _cpu(sh), act) for i, (_, sc, sh, act) in enumerate(s.aux)]
    if perturb is not None:
        perturb(snap, outs)
    tile_map = contract.tile_conv(snap, torch.float64, stage)
    idx = None if snap.idx is None else snap.idx.tolist()

    def locate(i):
        b, c, y, x = i
        if tile_map is None:
            return "(stack row %d, channel %d, pixel %d,%d)" % (b, c, y, x)
        m = int(tile_map[b, y, x])
        origin = idx[m % len(idx)] if (idx and m >= 0) else None
        return "(image %d, tile %d origin %s, channel %d, pixel %d,%d)" % (b, m, origin, c, y, x)

    res = Result("conv", s.name, _plan(fc))
    written = None if tile_map is None else tile_map >= 0
    for label, dev_t, before in outs:
        _compare(res, label, dev_t, before, wants[label], written, dtype, bound, locate)
    return res


def _pixel(i):
    return "(image %d, channel %d, pixel %d,%d)" % i if len(i) == 4 else "(index %s)" % (i,)


def _check_other(kind, args, fn, stream, sync, dtype, stage, bound):
    """conv_in / tail / attention / sparse_attention / spade: snapshot, launch, float64 reference."""
    if kind == "conv_in":
        rec = args
        outs = ([("dst", rec.out.raw, _cpu(rec.out.raw))] if rec.out.has_raw else []) + [("aux%d" % i, v, _cpu(v)) for i, (v, _, _, _) in enumerate(rec.aux)]
        snap = types.SimpleNamespace(x=_cpu(rec.x), weight=_cpu(rec.weight), bias=_cpu(rec.bias), tiles=_cpu(rec.tiles), tile_img=_cpu(rec.tile_img),
                                     tile_size=rec.tile_size)
        aux_vecs = [(_cpu(sc), _cpu(sh), act) for (_, sc, sh, act) in rec.aux]
        fn(stream)
        sync()
        wants = {label: _f64(before) for label, _, before in outs}
        snap.out = types.SimpleNamespace(raw=wants.get("dst"), has_raw=rec.out.has_raw)
        snap.aux = [(wants["aux%d" % i],) + aux_vecs[i] for i in range(len(rec.aux))]
        written = contract.conv_in(snap, torch.float64, stage)
        res = Result(kind, "conv_in" + ("" if rec.tiles is None else " (%d tiles%s)" % (rec.tiles.shape[0], ", per image" if rec.tile_img is not None else "")))
        for label, dev_t, before in outs:
            _compare(res, label, dev_t, before, wants[label], written, dtype, bound, _pixel)
        return res
    if kind == "tail":
        x, groups, eps, gamma, beta, act, weight, bias, out = args
        ins = [_cpu(t) if isinstance(t, torch.Tensor) else t for t in (x, groups, eps, gamma, beta, act, weight, bias)]
        before = _cpu(out)
        fn(stream)
        sync()
        want = _f64(before)
        contract.tail(*ins, want, torch.float64, stage)
    elif kind == "attention":
        qkv, out = args
        q_, before = _cpu(qkv), _cpu(out)
        fn(stream)
        sync()
        want = _f64(before)
        contract.attention(q_, want, torch.float64)
    elif kind == "sparse_attention":
        q, k, v, scale, out = args
        ins, before = [_cpu(q), _cpu(k), _cpu(v)], _cpu(out)
        fn(stream)
        sync()
        want = _f64(before)
        contract.sparse_attention(*ins, scale, want, torch.float64)
    elif kind == "spade":
        x, gamma, beta, slope, out = args
        ins, before = [_cpu(x), _cpu(gamma), _cpu(beta)], _cpu(out)
        fn(stream)
        sync()
        want = _f64(before)
        contract.spade(*ins, slope, want, torch.float64)
    else:
        raise AssertionError("unknown launch kind %r" % kind)
    res = Result(kind, "%s %s" % (kind, tuple(out.shape)))
    _compare(res, "out", out, before, want, None, dtype, bound, _pixel)
    return res


def walk(step, ex, dtype, stage, perturb=None):
    """Run `step` launch by launch, checking each non-eager launch against the float64 contract.  `perturb`: {launch name:
    f(reference snapshot, outputs)} deliberately changes the REFERENCE of that launch (the check must then reject it)."""
    cuda = step.dev.type == "cuda"
    stream = torch.cuda.current_stream(step.dev).cuda_stream if cuda else 0

    def sync():
        if cuda:
            torch.cuda.synchronize(step.dev)

    bound = BOUND[dtype]
    results = []
    with torch.no_grad():
        for b in step.low.cached_bufs:           # every tile-written buffer back to the cached activations: launches write fresh tiles
            b.restore()
        sync()
        for kind, fn in step.steps:
            if kind == "eager":
                fn(stream)
                continue
            if kind == "conv":
                fc = fn.__self__
                results.append(_check_conv(fc, lambda: (fn(stream), sync()), dtype, stage, bound, (perturb or {}).get(fc.name)))
            else:
                k2, args = ex.records[fn]
                assert k2 == kind, (k2, kind)
                results.append(_check_other(kind, args, fn, stream, sync, dtype, stage, bound))
    return results


def summarize(tag, results):
    counts = Counter(r.kind for r in results)
    worst = max(results, key=lambda r: r.err)
    print("%s: %d launches checked (%s); worst %r" % (tag, len(results), ", ".join("%s %d" % kv for kv in sorted(counts.items())), worst))
    bad = [r for r in results if not r.ok]
    return counts, worst, bad


def assert_all_ok(tag, results):
    counts, worst, bad = summarize(tag, results)
    assert not bad, "%s: %d of %d launches out of contract:\n  %s" % (tag, len(bad), len(results), "\n  ".join(repr(r) for r in bad[:12]))
    return counts


# ---------------------------------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------------------------------
def _model(cfg, dtype, dev):
    from sige_b200.workloads.ddpm import SIGEDDPMUNet, init_deterministic

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = init_deterministic(SIGEDDPMUNet(cfg), seed=0).eval()
    m = m.to(dev).to(dtype)
    return m.to(memory_format=torch.channels_last) if dev != "cpu" else m


def _prepared(cfg, ratio, dtype, dev=DEV):
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import synthetic_inputs

    model = _model(cfg, dtype, dev)
    x0, x1, mask, t = synthetic_inputs(cfg, ratio, seed=0)
    with torch.no_grad():
        model.set_mode("full")
        model(x0.to(dev).to(dtype), t.to(dev))
        model.set_masks(downsample_mask(mask.to(dev), min_res=8))
        model.set_mode("sparse")
    return model, x1.to(dev).to(dtype), t.to(dev)


def _cuda_step(model, x, t, **opts):
    ex = RecordingCudaExecutor(torch.device(DEV), x.dtype)
    with torch.no_grad():
        step = FusedStep(model, x, t, use_graph=False, executor=ex, **opts)
    if opts.get("fused_attention", True):
        assert step.eager_nodes == [], step.eager_nodes      # (with fused_attention=False the attention core runs as torch calls)
    return step, ex


def _stage(dtype):
    return None if dtype == torch.float32 else dtype


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the walker itself, on the simulator (fp32 sim vs the float64 contract)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rebind", [False, True])
def test_walker_on_the_cpu_simulator(rebind):
    """The snapshot / region logic without a GPU: DDPMConfig.small() through the simulator, every launch checked against
    float64 (including the untouched-outside check).  rebind: built with capacity headroom, then a smaller mask installed in
    place, so the lists carry SIGE_TILE_NONE tails."""
    from sige.utils import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model, x1, t = _prepared(cfg, 0.05, torch.float32, dev="cpu")
    ex = RecordingSimExecutor()
    with torch.no_grad():
        step = FusedStep(model, x1, t, executor=ex, **({"headroom": 0.6} if rebind else {}))
    if rebind:
        _, x_b, mask_b, _ = synthetic_inputs(cfg, 0.03, seed=0, edit_seed=2)
        model.set_masks(downsample_mask(mask_b, min_res=8))
        assert step.rebind()
        assert any(sl.cap > sl.n for sl in step.low.slots.values())
        step.static_inputs[0].copy_(x_b)
    results = walk(step, ex, torch.float32, None)
    counts = assert_all_ok("ddpm_small sim%s" % (" rebind" if rebind else ""), results)
    assert counts["conv"] == len(step.fused) and counts["conv_in"] == 1 and counts["tail"] == 1 and counts["attention"] == 4
    assert max(r.err for r in results) > 0, "the fp32 simulator and the float64 reference are different computations"


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every launch of the real step
# ---------------------------------------------------------------------------------------------------------------------
OPTS = [
    {"tc5": False, "producer_preop": False, "pdl": False, "fused_attention": False, "sparse_stem": False},
    {"tc5": False, "producer_preop": True, "pdl": False},
    {"tc5": True, "producer_preop": True, "pdl": False, "fuse_shortcut": False},
    {"tc5": True, "producer_preop": True, "pdl": True},
    {"tc5": True, "producer_preop": False, "pdl": True},
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("opts", OPTS)
def test_every_launch_ddpm_small(opts, dtype):
    """DDPMConfig.small() (5 % edit) under the option sets of test_fused_step_options_vs_modules_and_reference: mma.sync vs
    tcgen05, gather-side vs producer-side pre-op, PDL, fused vs unfused shortcut; fp16 and bf16."""
    from sige_b200.workloads.ddpm import DDPMConfig

    model, x1, t = _prepared(DDPMConfig.small(), 0.05, dtype)
    step, ex = _cuda_step(model, x1, t, **opts)
    counts = assert_all_ok("ddpm_small %s %s" % (str(dtype)[6:], opts), walk(step, ex, dtype, _stage(dtype)))
    assert counts["conv"] == len(step.fused)


@pytest.mark.gpu
@pytest.mark.parametrize("ratio", [0.012, 0.30])
def test_every_launch_ddpm256(ratio):
    """The flagship DDPM-256 step at 1.2 % and at 30 % (1296 tiles at 256x256: BN = 128, no split-K), fp16."""
    from sige_b200.workloads.ddpm import DDPMConfig

    model, x1, t = _prepared(DDPMConfig(), ratio, torch.float16)
    step, ex = _cuda_step(model, x1, t)
    counts = assert_all_ok("ddpm256 %.1f %%" % (100 * ratio), walk(step, ex, torch.float16, torch.float16))
    assert counts["conv"] == len(step.fused) == 86


@pytest.mark.gpu
def test_every_launch_batch_of_edits():
    """A batch of 4 independent edits (different masks) in one step, built as in test_batch_of_independent_edits_on_gpu:
    per-image tile lists padded with SIGE_TILE_NONE, CTAs spanning two images, the stem on per-image tiles."""
    from sige.utils import downsample_mask
    from sige_b200.masks import stack_mask_pyramids
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig()
    model, _, t = _prepared(cfg, 0.012, torch.float16)
    xs, masks = [], []
    for e, (ratio, shift) in enumerate([(0.012, (0, 0)), (0.012, (-70, 45)), (0.03, (60, -80)), (0.006, (-100, -100))]):
        x0, x1, mask, _ = synthetic_inputs(cfg, ratio, seed=0, edit_seed=e)
        masks.append(downsample_mask(torch.roll(mask, shift, (0, 1)).to(DEV), min_res=8))
        xs.append((x0 + torch.roll(x1 - x0, shift, (2, 3))).to(DEV).half())
    model.set_masks(stack_mask_pyramids(masks))
    step, ex = _cuda_step(model, torch.cat(xs, 0), t)
    per_image = [f for f in step.fused if f.spec.tile_img is not None]
    assert len(per_image) >= 30
    counts = assert_all_ok("ddpm256 batch of 4 edits", walk(step, ex, torch.float16, torch.float16))
    assert counts["conv"] == len(step.fused)


@pytest.mark.gpu
def test_every_launch_after_rebind_and_device_rebind():
    """set_fused(headroom=0.6): tile lists with capacity headroom (whole CTAs of padding, SIGE_CONV_PADDED); then a smaller
    mask installed in place by `rebind` (set_masks), then another by `rebind_device` (set_masks_async, lists written on the
    device).  Every launch is checked after each install."""
    from sige.utils import downsample_mask
    from sige_b200 import _cabi
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    cfg = DDPMConfig.small()
    model, x_a, t = _prepared(cfg, 0.04, torch.float16)
    step, ex = _cuda_step(model, x_a, t, headroom=0.6)
    assert any(f.desc.flags & _cabi.CONV_PADDED for f in step.fused)
    assert_all_ok("headroom 0.6, first mask", walk(step, ex, torch.float16, torch.float16))
    _, x_b, mask_b, _ = synthetic_inputs(cfg, 0.02, seed=0, edit_seed=2)
    model.set_masks(downsample_mask(mask_b.to(DEV), min_res=8))
    assert step.rebind()
    step.static_inputs[0].copy_(x_b.to(DEV).half())
    assert_all_ok("headroom 0.6, rebind", walk(step, ex, torch.float16, torch.float16))
    _, x_c, mask_c, _ = synthetic_inputs(cfg, 0.03, seed=0, edit_seed=3)
    assert step.rebind_device(downsample_mask(mask_c.to(DEV), min_res=8))
    step.static_inputs[0].copy_(x_c.to(DEV).half())
    assert_all_ok("headroom 0.6, rebind_device", walk(step, ex, torch.float16, torch.float16))
    assert step.async_ok()


@pytest.mark.gpu
def test_the_check_rejects_a_small_difference():
    """The check has teeth: the reference of one real launch gets one tile's halo shifted by one pixel, and the reference of
    another gets one output channel's bias moved by 4 fp16 ulps (at the output's magnitude).  Both launches must be rejected,
    every other launch of the step must pass.  Only the reference changes; the kernels run as always."""
    from sige_b200.workloads.ddpm import DDPMConfig

    model, x1, t = _prepared(DDPMConfig.small(), 0.05, torch.float16)
    step, ex = _cuda_step(model, x1, t)
    cands = [f for f in step.fused if f.spec.bias is not None and f.spec.dst is not None and f.spec.dst.has_raw
             and not f.spec.src_is_stack and all(up == 0 for _, up in f.spec.srcs) and f.spec.k == 3 and f.spec.stride == 1]
    assert len(cands) >= 2
    halo_launch, bias_launch = cands[0].name, cands[-1].name

    def shift_halo(snap, outs):
        src = snap.srcs[0][0].clone()
        H, W = src.shape[2], src.shape[3]
        iy, ix = next((a, b) for a, b in snap.idx.tolist() if a > -20000)
        y0, y1, x0, x1_ = max(iy, 0), min(iy + snap.block, H), max(ix, 0), min(ix + snap.block, W - 1)
        src[0, :, y0:y1, x0:x1_] = src[0, :, y0:y1, x0 + 1:x1_ + 1].clone()
        snap.srcs = [(src, snap.srcs[0][1])] + snap.srcs[1:]

    def nudge_bias(snap, outs):
        peak = float(outs[0][1].abs().max())
        snap.bias = snap.bias.clone()
        snap.bias[0] += 4 * float(_ulp(torch.tensor(peak, dtype=torch.float64), torch.float16))

    results = walk(step, ex, torch.float16, torch.float16, perturb={halo_launch: shift_halo, bias_launch: nudge_bias})
    _, _, bad = summarize("teeth", results)
    assert sorted(r.name for r in bad) == sorted([halo_launch, bias_launch]), bad
    for r in bad:
        print("rejected as it must be: %r" % r)

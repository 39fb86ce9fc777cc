"""GPU parity of the tile convolution: tensor-core fused kernel (fp16/bf16) and CUDA-core generic
kernel (fp32 exact) vs the CPU oracle.  Tolerances are the north-star's: conv outputs within
1e-3 rel (fp16) / 1e-5 rel (fp32) of the fp32 reference, max-normalised; bf16 (8-bit mantissa)
is given 8e-3."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def T(a, dtype=torch.float32, cl=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    if t.is_floating_point():
        t = t.to(dtype)
    if cl and t.dim() == 4:
        t = t.contiguous(memory_format=torch.channels_last)
    return t


def _round(a, dtype):
    return a if dtype == torch.float32 else torch.from_numpy(a).to(dtype).float().numpy()


def rel_err(got, want):
    g = got.float().cpu().numpy()
    assert g.shape == want.shape, (g.shape, want.shape)
    return float(np.abs(g - want).max() / max(np.abs(want).max(), 1e-12))


TOL = {torch.float32: 1e-5, torch.float16: 1e-3, torch.bfloat16: 8e-3}
TC5 = 2           # SIGE_CONV_TC5
PADDED = 4        # SIGE_CONV_PADDED
TILE_NONE = -30000


@pytest.mark.parametrize("cl", [False, True])
def test_generic_conv_fp32_exact(oracle, cl):
    from sige_b200 import ops

    rng = np.random.default_rng(1)
    # (groups == Cin == Cout: the depthwise kernel — GauGAN's separable convs, gaugan/models/mobile_modules.py:83-91 — in its
    #  16-byte-vector NHWC form (Cin % 4 == 0 for fp32), its scalar NHWC form (Cin = 6) and its NCHW form)
    for (M, Ci, Co, R, k, s, d, g) in [(5, 8, 12, 6, 3, 1, 1, 1), (3, 16, 16, 5, 3, 2, 1, 1), (4, 12, 12, 6, 3, 1, 1, 12), (7, 36, 70, 6, 3, 1, 1, 1),
                                       (2, 36, 20, 4, 1, 1, 1, 1), (3, 8, 8, 7, 3, 1, 2, 2), (64, 64, 64, 6, 3, 1, 1, 1), (2, 3, 5, 10, 3, 1, 1, 1),
                                       (300, 128, 128, 6, 3, 1, 1, 128), (9, 6, 6, 5, 3, 2, 1, 6), (5, 64, 64, 8, 3, 1, 2, 64)]:
        x = rng.standard_normal((M, Ci, R, R)).astype(np.float32)
        w = rng.standard_normal((Co, Ci // g, k, k)).astype(np.float32) / np.sqrt(Ci // g * k * k)
        b = rng.standard_normal((Co,)).astype(np.float32)
        want = oracle.conv2d_tiles(x, w, b, (s, s), (d, d), g)
        got = ops.tile_conv_generic(T(x, cl=cl), T(w), T(b), (s, s), (d, d), g)
        assert rel_err(got, want) <= 1e-5
        got = ops.tile_conv_generic(T(x, cl=cl), T(w), None, (s, s), (d, d), g)
        assert rel_err(got, oracle.conv2d_tiles(x, w, None, (s, s), (d, d), g)) <= 1e-5


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_generic_conv_half(oracle, dtype):
    from sige_b200 import ops

    rng = np.random.default_rng(2)
    x = _round(rng.standard_normal((6, 36, 6, 6)).astype(np.float32), dtype)
    w = _round(rng.standard_normal((48, 36, 3, 3)).astype(np.float32) / 18, dtype)
    b = _round(rng.standard_normal((48,)).astype(np.float32), dtype)
    want = oracle.conv2d_tiles(x, w, b)
    assert rel_err(ops.tile_conv_generic(T(x, dtype), T(w, dtype), T(b, dtype), (1, 1), (1, 1), 1), want) <= TOL[dtype]
    for cl in (False, True):            # depthwise
        xd = _round(rng.standard_normal((40, 96, 6, 6)).astype(np.float32), dtype)
        wd = _round(rng.standard_normal((96, 1, 3, 3)).astype(np.float32) / 3, dtype)
        bd = _round(rng.standard_normal((96,)).astype(np.float32), dtype)
        got = ops.tile_conv_generic(T(xd, dtype, cl=cl), T(wd, dtype), T(bd, dtype), (1, 1), (1, 1), 96)
        assert rel_err(got, oracle.conv2d_tiles(xd, wd, bd, (1, 1), (1, 1), 96)) <= TOL[dtype]


STACK_CASES = [  # M, Cin, Cout, R, k, stride  — DDPM shape classes (SURVEY.md Appendix B) + edge sizes
    (64, 128, 128, 6, 3, 1), (64, 256, 128, 6, 3, 1), (32, 384, 128, 6, 3, 1), (16, 512, 256, 6, 3, 1), (4, 512, 512, 6, 3, 1),
    (64, 256, 128, 4, 1, 1), (12, 384, 256, 4, 1, 1), (64, 128, 128, 5, 3, 2), (13, 256, 256, 5, 3, 2),
    (1, 64, 8, 6, 3, 1), (3, 64, 72, 6, 3, 1), (700, 128, 128, 6, 3, 1), (1300, 64, 64, 6, 3, 1), (33, 128, 136, 4, 1, 1),
]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_tensor_core_conv_on_stacks(oracle, dtype):
    from sige_b200 import ops

    rng = np.random.default_rng(3)
    for (M, Ci, Co, R, k, s) in STACK_CASES:
        x = _round(rng.standard_normal((M, Ci, R, R)).astype(np.float32), dtype)
        w = _round(rng.standard_normal((Co, Ci, k, k)).astype(np.float32) / np.sqrt(Ci * k * k), dtype)
        b = rng.standard_normal((Co,)).astype(np.float32)
        want = oracle.conv2d_tiles(x, w, b, (s, s))
        wp = ops.pack_conv_weight(T(w, dtype), dtype)
        assert tuple(wp.shape) == (k * k, Co, Ci)
        got = ops.tile_conv_stack(T(x, dtype, cl=True), wp, T(b), (k, k), s)
        assert got.is_contiguous(memory_format=torch.channels_last) or got.is_contiguous()
        e = rel_err(got, want)
        assert e <= TOL[dtype], "case %s: rel err %g" % ((M, Ci, Co, R, k, s), e)


def _fused_desc(ops, x, wp, bias, idx, out, *, R, k, stride, off, scale=None, shift=None, act=0, residual=None, x2=None, up=0):
    d = ops.tile_conv_descriptor()
    B, C, H, W = x.shape
    d.dtype = ops._dt(x)
    d.n_src = 1 if x2 is None else 2
    d.src[0].ptr, d.src[0].C, d.src[0].up = x.data_ptr(), C, up
    cin = C
    if x2 is not None:
        d.src[1].ptr, d.src[1].C, d.src[1].up = x2.data_ptr(), x2.shape[1], 0
        cin += x2.shape[1]
    d.B, d.H, d.W = B, H << up, W << up
    d.src_is_stack = 0
    d.idx, d.N = idx.data_ptr(), idx.shape[0]
    d.R = d.S = R
    d.scale = None if scale is None else scale.data_ptr()
    d.shift = None if shift is None else shift.data_ptr()
    d.affine_bstride = 0 if (scale is None or scale.shape[0] == 1) else cin
    d.act = act
    d.w_packed, d.bias = wp.data_ptr(), (None if bias is None else bias.data_ptr())
    d.Cin, d.Cout, d.kH, d.kW, d.stride = cin, wp.shape[1], k, k, stride
    d.dst, d.dst_is_stack = out.data_ptr(), 0
    d.dH, d.dW, d.dC, d.dst_c0 = out.shape[2], out.shape[3], out.shape[1], 0
    d.offH = d.offW = off
    d.residual = None if residual is None else residual.data_ptr()
    d.rC, d.res_c0 = (0 if residual is None else residual.shape[1]), 0
    d._keep = (x, wp, bias, idx, out, scale, shift, residual, x2)   # descriptors hold raw pointers: keep the tensors alive
    return d


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_fused_gather_conv_scatter_vs_oracle(oracle, dtype):
    """One launch == oracle gather(affine+swish) -> conv -> scatter(+residual) composite.  Measured on a B200 (1000 W) over the
    cases, split-K factors and PDL: max-normalised 3.0e-4 (fp16) / 2.4e-3 (bf16), within TOL with 3x margin."""
    from sige_b200 import ops

    rng = np.random.default_rng(4)
    for (B, C, Co, H, W, bs, ts, k, s, off, p) in [(1, 128, 128, 64, 64, 6, 4, 3, 1, 1, 0.02), (2, 64, 192, 24, 40, 6, 4, 3, 1, 1, 0.1),
                                                   (1, 256, 128, 32, 32, 4, 4, 1, 1, 0, 0.05), (1, 128, 128, 33, 33, 5, 4, 3, 2, 0, 0.05),
                                                   (1, 64, 64, 16, 16, 6, 4, 3, 1, 1, 1.0)]:
        mask = rng.random((H, W)) < p
        mask[0, 0] = mask[H - 1, W - 1] = True
        idx = oracle.reduce_mask(mask, bs, ts, off)
        x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
        w = _round(rng.standard_normal((Co, C, k, k)).astype(np.float32) / np.sqrt(C * k * k), dtype)
        b = rng.standard_normal((Co,)).astype(np.float32)
        sc = (1 + 0.2 * rng.standard_normal((B, C, 1, 1))).astype(np.float32)
        sh = (0.2 * rng.standard_normal((B, C, 1, 1))).astype(np.float32)
        Ho = H if s == 1 else (H + 1 - k) // 2 + 1
        Wo = W if s == 1 else (W + 1 - k) // 2 + 1
        y = _round(rng.standard_normal((B, Co, Ho, Wo)).astype(np.float32), dtype)
        res = _round(rng.standard_normal((B, Co, Ho, Wo)).astype(np.float32), dtype)
        g = oracle.gather(x, bs, bs, idx, sc, sh, "swish", False)
        g = _round(g, dtype)                     # the kernel stages the pre-op result in fp16/bf16
        c = oracle.conv2d_tiles(g, w, b, (s, s))
        want = oracle.scatter(c, y, off, off, s, s, idx, res)
        out = T(y, dtype, cl=True).clone(memory_format=torch.channels_last)
        tx, tres = T(x, dtype, cl=True), T(res, dtype, cl=True)
        d = _fused_desc(ops, tx, ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(idx), out, R=bs, k=k, stride=s, off=off,
                        scale=T(sc).reshape(B, C).contiguous(), shift=T(sh).reshape(B, C).contiguous(), act=1, residual=tres)
        first = None
        for ks in (0, 1, 2, 4, 8):     # split-K over a thread-block cluster must not change the result beyond fp32 reassociation
            out.copy_(T(y, dtype, cl=True))
            d.ksplit = ks
            ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            e = rel_err(out, want)
            print("fused case %s %s ksplit %d: rel err %.3g" % ((B, C, Co, H, W, bs, k, s), dtype, ks, e))
            assert e <= TOL[dtype], "fused case %s ksplit %d: rel err %g" % ((B, C, Co, H, W, bs, k, s), ks, e)
            if first is None:
                first = out.clone()
            else:
                assert float((out.float() - first.float()).abs().max()) <= 2e-2 * float(first.float().abs().max())
        d.ksplit, d.flags = 0, 1       # programmatic dependent launch path
        out.copy_(T(y, dtype, cl=True))
        ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        e = rel_err(out, want)
        print("fused case %s %s PDL: rel err %.3g" % ((B, C, Co, H, W, bs, k, s), dtype, e))
        assert e <= TOL[dtype]


def test_fused_concat_and_upsample_sources(oracle):
    """Two channel-concatenated sources (torch.cat dim=1, the DDPM up path's 128 + 64 split) and a nearest-x2-upsampled
    source are read in place by the gather stage, on both kernels and over the split-K sweep: results equal the oracle on
    the materialised tensors."""
    from ctypes import byref

    from sige_b200 import _cabi, ops

    dtype = torch.float16
    rng = np.random.default_rng(6)
    B, C1, C2, Co, H, W = 1, 128, 64, 128, 32, 32
    mask = rng.random((H, W)) < 0.05
    mask[0, 0] = mask[H - 1, W - 1] = True
    idx = oracle.reduce_mask(mask, 6, 4, 1)
    x1 = _round(rng.standard_normal((B, C1, H, W)).astype(np.float32), dtype)
    x2 = _round(rng.standard_normal((B, C2, H, W)).astype(np.float32), dtype)
    w = _round(rng.standard_normal((Co, C1 + C2, 3, 3)).astype(np.float32) / np.sqrt((C1 + C2) * 9), dtype)
    y = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
    want_cat = oracle.gather_conv_scatter(np.concatenate([x1, x2], 1), w, None, y, idx, (6, 6), (1, 1), (1, 1))
    # upsample: source at half resolution, logical extent HxW
    xs = _round(rng.standard_normal((B, C1, H // 2, W // 2)).astype(np.float32), dtype)
    xu = xs.repeat(2, axis=2).repeat(2, axis=3)
    wu = _round(rng.standard_normal((Co, C1, 3, 3)).astype(np.float32) / np.sqrt(C1 * 9), dtype)
    want_up = oracle.gather_conv_scatter(xu, wu, None, y, idx, (6, 6), (1, 1), (1, 1))
    ty = T(y, dtype, cl=True)
    out = ty.clone(memory_format=torch.channels_last)
    d_cat = _fused_desc(ops, T(x1, dtype, cl=True), ops.pack_conv_weight(T(w, dtype), dtype), None, T(idx), out, R=6, k=3, stride=1, off=1,
                        x2=T(x2, dtype, cl=True))
    d_up = _fused_desc(ops, T(xs, dtype, cl=True), ops.pack_conv_weight(T(wu, dtype), dtype), None, T(idx), out, R=6, k=3, stride=1, off=1, up=1)
    for flags in (0, TC5, TC5 | 1):                  # mma.sync, tcgen05, tcgen05 + PDL
        for what, d, want in (("concat", d_cat, want_cat), ("upsample", d_up, want_up)):
            for ks in (0, 1, 2, 4, 8):
                d.flags, d.ksplit = flags, ks
                plan = _cabi.TileConvPlan()
                assert _cabi.lib().sige_tile_conv_plan(byref(d), byref(plan)) == 0 and plan.path == (1 if flags & TC5 else 0)
                out.copy_(ty)
                ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                e = rel_err(out, want)
                print("%s flags %d ksplit %d: rel err %.3g" % (what, flags, ks, e))
                assert e <= TOL[dtype], "%s flags %d ksplit %d: rel err %g" % (what, flags, ks, e)


def test_linearity_and_dense_equals_sparse_at_full_size(oracle):
    """Size-independent properties at the benchmark's layer size (no oracle run needed):
    (1) with every tile active the fused sparse layer equals the dense convolution (example.py:95's
    identity), (2) conv is linear: f(a x1 + x2) = a f(x1) + f(x2) (bias-free)."""
    from sige_b200 import ops

    dtype = torch.float16
    torch.manual_seed(0)
    B, C, H, W = 1, 128, 256, 256
    x = torch.randn(B, C, H, W, device=DEV, dtype=dtype).contiguous(memory_format=torch.channels_last)
    w = (torch.randn(C, C, 3, 3, device=DEV) / (C * 9) ** 0.5).to(dtype)
    bias = torch.randn(C, device=DEV)
    ii, jj = torch.meshgrid(torch.arange(0, H, 4), torch.arange(0, W, 4), indexing="ij")
    idx = (torch.stack([ii.reshape(-1), jj.reshape(-1)], 1) - 1).to(torch.int32).to(DEV).contiguous()
    out = torch.zeros(B, C, H, W, device=DEV, dtype=dtype).contiguous(memory_format=torch.channels_last)
    wp = ops.pack_conv_weight(w, dtype)
    d = _fused_desc(ops, x, wp, bias, idx, out, R=6, k=3, stride=1, off=1)
    ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
    dense = torch.nn.functional.conv2d(x.float(), w.float(), bias, 1, 1)
    assert float((out.float() - dense).abs().max() / dense.abs().max()) <= 1e-3
    x2 = torch.randn_like(x)
    o1, o2, o3 = (torch.zeros_like(out) for _ in range(3))
    for src, dst in ((x, o1), (x2, o2), ((0.5 * x + x2).contiguous(memory_format=torch.channels_last), o3)):
        d = _fused_desc(ops, src, wp, None, idx, dst, R=6, k=3, stride=1, off=1)
        ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
    lin = 0.5 * o1.float() + o2.float()
    assert float((o3.float() - lin).abs().max() / lin.abs().max()) <= 3e-3


# ---------------------------------------------------------------------------------------------------
# Blackwell-native kernel (tcgen05.mma + TMEM + TMA weights), flags = SIGE_CONV_TC5
# ---------------------------------------------------------------------------------------------------
TC5_STACK_CASES = [(64, 128, 128, 6, 3), (8, 64, 64, 6, 3), (1, 64, 64, 6, 3), (13, 128, 192, 6, 3), (32, 384, 128, 6, 3), (16, 512, 256, 6, 3),
                   (700, 128, 128, 6, 3), (1300, 64, 256, 6, 3), (64, 256, 128, 4, 1), (12, 384, 256, 4, 1), (5, 64, 64, 4, 1), (300, 128, 512, 4, 1)]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_tc5_conv_on_stacks(oracle, dtype):
    from sige_b200 import ops

    rng = np.random.default_rng(13)
    for (M, Ci, Co, R, k) in TC5_STACK_CASES:
        x = _round(rng.standard_normal((M, Ci, R, R)).astype(np.float32), dtype)
        w = _round(rng.standard_normal((Co, Ci, k, k)).astype(np.float32) / np.sqrt(Ci * k * k), dtype)
        b = rng.standard_normal((Co,)).astype(np.float32)
        want = oracle.conv2d_tiles(x, w, b, (1, 1))
        wp = ops.pack_conv_weight(T(w, dtype), dtype)
        tx, tb = T(x, dtype, cl=True), T(b)
        for ks in (1, 0, 2, 4, 8):
            got = ops.tile_conv_stack(tx, wp, tb, (k, k), 1, flags=TC5, ksplit=ks)
            torch.cuda.synchronize()
            e = rel_err(got, want)
            assert e <= TOL[dtype], "tc5 stack case %s ksplit %d: rel err %g" % ((M, Ci, Co, R, k), ks, e)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_tc5_fused_gather_conv_scatter_vs_oracle(oracle, dtype):
    """tcgen05 kernel, same composite.  Measured on a B200 (1000 W): max-normalised 3.1e-4 (fp16) / 2.5e-3 (bf16)."""
    from sige_b200 import ops

    rng = np.random.default_rng(14)
    for (B, C, Co, H, W, bs, ts, k, off, p) in [(1, 128, 128, 64, 64, 6, 4, 3, 1, 0.02), (2, 64, 192, 24, 40, 6, 4, 3, 1, 0.1),
                                                (1, 256, 128, 32, 32, 4, 4, 1, 0, 0.05), (1, 64, 64, 16, 16, 6, 4, 3, 1, 1.0)]:
        mask = rng.random((H, W)) < p
        mask[0, 0] = mask[H - 1, W - 1] = True
        idx = oracle.reduce_mask(mask, bs, ts, off)
        x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
        w = _round(rng.standard_normal((Co, C, k, k)).astype(np.float32) / np.sqrt(C * k * k), dtype)
        b = rng.standard_normal((Co,)).astype(np.float32)
        sc = (1 + 0.2 * rng.standard_normal((B, C, 1, 1))).astype(np.float32)
        sh = (0.2 * rng.standard_normal((B, C, 1, 1))).astype(np.float32)
        y = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
        res = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
        g = _round(oracle.gather(x, bs, bs, idx, sc, sh, "swish", False), dtype)
        want = oracle.scatter(oracle.conv2d_tiles(g, w, b, (1, 1)), y, off, off, 1, 1, idx, res)
        out = T(y, dtype, cl=True).clone(memory_format=torch.channels_last)
        d = _fused_desc(ops, T(x, dtype, cl=True), ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(idx), out, R=bs, k=k, stride=1, off=off,
                        scale=T(sc).reshape(B, C).contiguous(), shift=T(sh).reshape(B, C).contiguous(), act=1, residual=T(res, dtype, cl=True))
        for ks, flags in ((1, TC5), (0, TC5), (4, TC5), (0, TC5 | 1)):
            out.copy_(T(y, dtype, cl=True))
            d.ksplit, d.flags = ks, flags
            ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            e = rel_err(out, want)
            print("tc5 fused case %s %s ksplit %d flags %d: rel err %.3g" % ((B, C, Co, H, W, bs, k), dtype, ks, flags, e))
            assert e <= TOL[dtype], "tc5 fused case %s ksplit %d flags %d: rel err %g" % ((B, C, Co, H, W, bs, k), ks, flags, e)


@pytest.mark.parametrize("flags", [0, TC5])
def test_aux_destinations_apply_the_consumers_preop(oracle, flags):
    """Extra epilogue outputs: aux = act(out*scale+shift), primary destination optional."""
    from sige_b200 import _cabi, ops

    dtype = torch.float16
    rng = np.random.default_rng(21)
    B, C, Co, H, W = 1, 128, 128, 32, 32
    mask = rng.random((H, W)) < 0.1
    mask[0, 0] = True
    idx = oracle.reduce_mask(mask, 6, 4, 1)
    x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
    w = _round(rng.standard_normal((Co, C, 3, 3)).astype(np.float32) / np.sqrt(C * 9), dtype)
    b = rng.standard_normal((Co,)).astype(np.float32)
    y = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
    res = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
    sc = (1 + 0.2 * rng.standard_normal((1, Co, 1, 1))).astype(np.float32)
    sh = (0.2 * rng.standard_normal((1, Co, 1, 1))).astype(np.float32)
    tiles = oracle.conv2d_tiles(oracle.gather(x, 6, 6, idx), w, b, (1, 1))
    want_raw = oracle.scatter(tiles, y, 1, 1, 1, 1, idx, res)
    z = want_raw * sc + sh
    want_aux = z / (1 + np.exp(-z))
    fresh = want_raw != y                      # only active tiles are rewritten
    out = T(y, dtype, cl=True).clone(memory_format=torch.channels_last)
    aux0 = torch.zeros_like(out)
    aux1 = torch.zeros_like(out)
    tsc, tsh = T(sc).reshape(-1).contiguous(), T(sh).reshape(-1).contiguous()
    d = _fused_desc(ops, T(x, dtype, cl=True), ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(idx), out, R=6, k=3, stride=1, off=1,
                    residual=T(res, dtype, cl=True))
    d.flags, d.n_aux = flags, 2
    d.aux[0].ptr, d.aux[0].C, d.aux[0].c0, d.aux[0].scale, d.aux[0].shift, d.aux[0].act = aux0.data_ptr(), Co, 0, tsc.data_ptr(), tsh.data_ptr(), 1
    d.aux[1].ptr, d.aux[1].C, d.aux[1].c0, d.aux[1].scale, d.aux[1].shift, d.aux[1].act = aux1.data_ptr(), Co, 0, None, None, 0
    ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rel_err(out, want_raw) <= 2e-3
    g0, g1 = aux0.float().cpu().numpy(), aux1.float().cpu().numpy()
    assert np.abs(g0 - want_aux)[fresh].max() / np.abs(want_aux).max() <= 2e-3 and (g0[~fresh] == 0).all()
    assert np.abs(g1 - want_raw)[fresh].max() / np.abs(want_raw).max() <= 2e-3
    d.dst = None                               # aux-only launch
    aux0.zero_()
    ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.abs(aux0.float().cpu().numpy() - want_aux)[fresh].max() / np.abs(want_aux).max() <= 2e-3


def test_tc5_fused_shortcut_matches_block_residual_semantics(oracle):
    """conv2 + fused 1x1 shortcut in one launch == reference ScatterWithBlockResidual: fresh shortcut where the
    shortcut's own tile is active, cached shortcut elsewhere (sige/cuda/scatter_kernel.cu:46-74,119-146)."""
    from sige_b200 import ops

    dtype = torch.float16
    rng = np.random.default_rng(31)
    for (B, Cm, Cx2, Co, H, W, p) in [(1, 128, (128, 64), 128, 32, 32, 0.04), (1, 64, (64,), 64, 16, 16, 1.0)]:
        mask = rng.random((H, W)) < p
        mask[0, 0] = True
        idx0 = oracle.reduce_mask(mask, 6, 4, 1)          # main 3x3 tiles
        idx1 = oracle.reduce_mask(mask, 4, 4, 0)          # shortcut 1x1 tiles (subset, shifted frame)
        assert idx1.shape[0] <= idx0.shape[0]
        t1 = _round(rng.standard_normal((B, Cm, H, W)).astype(np.float32), dtype)            # conv2 input (already transformed)
        xs = [_round(rng.standard_normal((B, c, H, W)).astype(np.float32), dtype) for c in Cx2]  # raw block input(s), concatenated
        xcat = np.concatenate(xs, 1)
        Cx = xcat.shape[1]
        w2 = _round(rng.standard_normal((Co, Cm, 3, 3)).astype(np.float32) / np.sqrt(Cm * 9), dtype)
        b2 = rng.standard_normal((Co,)).astype(np.float32)
        wsc = _round(rng.standard_normal((Co, Cx, 1, 1)).astype(np.float32) / np.sqrt(Cx), dtype)
        bsc = rng.standard_normal((Co,)).astype(np.float32)
        y0 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)            # cached block output
        y1 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)            # cached shortcut output
        # reference composite through the oracle
        main_tiles = oracle.conv2d_tiles(oracle.gather(t1, 6, 6, idx0), w2, b2, (1, 1))
        sc_tiles = oracle.conv2d_tiles(oracle.gather(xcat, 4, 4, idx1), wsc, bsc, (1, 1))
        want = oracle.scatter_with_block_residual(main_tiles, y0, sc_tiles, y1, 1, 1, 1, 1, idx0, idx1)
        keys1 = {(int(a), int(b)) for a, b in idx1}
        flags = np.array([1 if (int(a) + 1, int(b) + 1) in keys1 else 0 for a, b in idx0], dtype=np.uint8)
        assert flags.sum() == idx1.shape[0]
        out = T(y0, dtype, cl=True).clone(memory_format=torch.channels_last)
        txs = [T(v, dtype, cl=True) for v in xs]
        d = _fused_desc(ops, T(t1, dtype, cl=True), ops.pack_conv_weight(T(w2, dtype), dtype), T(b2), T(idx0), out, R=6, k=3, stride=1, off=1,
                        residual=T(y1, dtype, cl=True))
        wscp, tb, tf = ops.pack_conv_weight(T(wsc, dtype), dtype), T(bsc), torch.from_numpy(flags).to(DEV)
        d.n_src2 = len(txs)
        for i, t in enumerate(txs):
            d.src2[i].ptr, d.src2[i].C, d.src2[i].up = t.data_ptr(), t.shape[1], 0
        d.Cin2, d.w2_packed, d.bias2, d.sc_flags = Cx, wscp.data_ptr(), tb.data_ptr(), tf.data_ptr()
        for ks in (1, 2, 0, 8):
            out.copy_(T(y0, dtype, cl=True))
            d.flags, d.ksplit = TC5, ks
            ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            e = rel_err(out, want)
            assert e <= 2e-3, "fused shortcut (%s) ksplit %d: rel err %g" % ((Cm, Cx2, Co, H), ks, e)
        d.flags = 0                                   # the mma.sync kernel does not implement it: loud error, not a wrong result
        with pytest.raises(Exception, match="tcgen05"):
            ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("cl", [False, True])
def test_few_channel_stacks_take_the_tensor_cores(oracle, dtype, cl):
    """SIGEConv2d on a stack whose channel count is not a multiple of 64 (GauGAN's 36-channel label maps,
    reference gaugan/models/sige_normalization.py): zero channels are appended to stack and weights — exact."""
    from sige_b200 import ops
    from sige_b200.nn import SIGEConv2d

    rng = np.random.default_rng(11)
    for (M, Ci, Co, R, k) in [(37, 36, 128, 6, 3), (16, 8, 64, 4, 1), (9, 100, 72, 6, 3)]:
        conv = SIGEConv2d(Ci, Co, k, padding=k // 2).to(DEV).to(dtype)
        conv.set_mode("sparse")
        x = _round(rng.standard_normal((M, Ci, R, R)).astype(np.float32), dtype)
        w = conv.weight.detach().float().cpu().numpy()
        b = conv.bias.detach().float().cpu().numpy()
        want = oracle.conv2d_tiles(x, w, b, (1, 1))
        before = ops.launch_count
        got = conv(T(x, dtype, cl=cl))
        assert got.shape == want.shape
        e = rel_err(got, want)
        assert e <= TOL[dtype], "case %s: rel err %g" % ((M, Ci, Co, R, k), e)
        assert ops.launch_count - before <= 2, "one weight pack + one tensor-core launch"


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_tc5_stride2_downsample_vs_oracle(oracle, dtype):
    """The DDPM Downsample (3x3 stride 2 on 5x5 tiles -> 2x2 outputs, reference sige_fused_unet.py:212-221) on the tcgen05 kernel:
    32 tiles per CTA, halo rows as even / odd planes.  Pure-copy gather (this geometry has no pre-op in the model), ragged image
    edges (odd extents: tiles overhang), more and fewer tiles than one CTA holds, batch 2, a channel-concatenated source, residual,
    every split-K factor; and the plan really is the tcgen05 path.  Measured on a B200 (1000 W): max-normalised 3.2e-4 (fp16) /
    2.9e-3 (bf16)."""
    from ctypes import byref

    from sige_b200 import _cabi, ops

    rng = np.random.default_rng(21)
    for (B, C, Co, H, W, p, two) in [(1, 128, 128, 64, 64, 0.03, False), (1, 256, 256, 32, 32, 1.0, False), (2, 64, 192, 33, 41, 0.1, False),
                                     (1, 512, 512, 16, 16, 1.0, False), (1, 128, 64, 40, 24, 0.3, True), (1, 64, 64, 8, 8, 0.02, False)]:
        bs, ts, k, s, off = 5, 4, 3, 2, 0
        mask = rng.random((H, W)) < p
        mask[0, 0] = mask[H - 1, W - 1] = True
        idx = oracle.reduce_mask(mask, bs, ts, off)
        x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
        w = _round(rng.standard_normal((Co, C, k, k)).astype(np.float32) / np.sqrt(C * k * k), dtype)
        b = rng.standard_normal((Co,)).astype(np.float32)
        Ho, Wo = (H + 1 - k) // 2 + 1, (W + 1 - k) // 2 + 1
        y = _round(rng.standard_normal((B, Co, Ho, Wo)).astype(np.float32), dtype)
        res = _round(rng.standard_normal((B, Co, Ho, Wo)).astype(np.float32), dtype)
        g = oracle.gather(x, bs, bs, idx, None, None, "identity", False)
        want = oracle.scatter(oracle.conv2d_tiles(g, w, b, (s, s)), y, off, off, s, s, idx, res)
        out = T(y, dtype, cl=True).clone(memory_format=torch.channels_last)
        tx = T(x, dtype, cl=True)
        if two:        # torch.cat([a, b], 1) as two sources
            xa, xb = tx[:, :C // 2].contiguous(memory_format=torch.channels_last), tx[:, C // 2:].contiguous(memory_format=torch.channels_last)
            d = _fused_desc(ops, xa, ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(idx), out, R=bs, k=k, stride=s, off=off,
                            residual=T(res, dtype, cl=True), x2=xb)
        else:
            d = _fused_desc(ops, tx, ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(idx), out, R=bs, k=k, stride=s, off=off,
                            residual=T(res, dtype, cl=True))
        d.flags, d.ksplit = TC5, 0
        plan = _cabi.TileConvPlan()
        assert _cabi.lib().sige_tile_conv_plan(byref(d), byref(plan)) == 0 and plan.path == 1 and plan.grid_x == -(-B * idx.shape[0] // 32)
        for ks, flags in ((0, TC5), (1, TC5), (2, TC5), (4, TC5), (8, TC5), (0, TC5 | 1), (0, 0)):
            out.copy_(T(y, dtype, cl=True))
            d.ksplit, d.flags = ks, flags
            ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            e = rel_err(out, want)
            print("stride-2 case %s %s ksplit %d flags %d: rel err %.3g" % ((B, C, Co, H, W), dtype, ks, flags, e))
            assert e <= TOL[dtype], "stride-2 case %s ksplit %d flags %d: rel err %g" % ((B, C, Co, H, W), ks, flags, e)


# ---------------------------------------------------------------------------------------------------
# tile lists with SIGE_TILE_NONE entries, channel windows, sige_resblock
# ---------------------------------------------------------------------------------------------------
GEOMS = [(128, 128, 6, 3, 1, 1), (256, 128, 4, 1, 1, 0), (128, 128, 5, 3, 2, 0)]     # Cin, Cout, R, k, stride, off: 3x3, 1x1, 3x3-s2


def _padded_lists(lists, n):
    """Per-image layout of the C-ABI: row b*n + i = tile i of image b, SIGE_TILE_NONE behind each list."""
    out = np.full((len(lists) * n, 2), TILE_NONE, np.int32)
    for b, l in enumerate(lists):
        out[b * n:b * n + len(l)] = l
    return out


def _written(shape, lists, off, s, ro):
    """bool [B, 1, Ho, Wo]: the output pixels of the real tiles of each image's list."""
    m = np.zeros((shape[0], 1, shape[2], shape[3]), bool)
    for b, l in enumerate(lists):
        for iy, ix in np.asarray(l).reshape(-1, 2):
            oy, ox = (off + int(iy)) // s, (off + int(ix)) // s
            m[b, :, oy:oy + ro, ox:ox + ro] = True
    return m


def _changed_outside(got, before, written):
    """Number of elements outside `written` (broadcast over channels) whose bits differ from `before`."""
    bits = {2: torch.int16, 4: torch.int32}[got.element_size()]
    diff = (got.cpu().view(bits) != before.cpu().view(bits)).numpy()
    return int((diff & ~np.broadcast_to(written, diff.shape)).sum())


def _lists(oracle, rng, R, off, H, W, sizes):
    full = oracle.reduce_mask(rng.random((H, W)) < 0.4, R, 4, off)
    return [full[np.sort(rng.choice(len(full), n, replace=False))] for n in sizes]


def _geom_case(oracle, rng, geom, B, H, W, dtype):
    C, Co, R, k, s, off = geom
    Ho, Wo = (H, W) if s == 1 else ((H + 1 - k) // 2 + 1, (W + 1 - k) // 2 + 1)
    x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
    w = _round(rng.standard_normal((Co, C, k, k)).astype(np.float32) / np.sqrt(C * k * k), dtype)
    b = rng.standard_normal((Co,)).astype(np.float32)
    sc = (1 + 0.2 * rng.standard_normal((B, C, 1, 1))).astype(np.float32)
    sh = (0.2 * rng.standard_normal((B, C, 1, 1))).astype(np.float32)
    y = _round(rng.standard_normal((B, Co, Ho, Wo)).astype(np.float32), dtype)
    res = _round(rng.standard_normal((B, Co, Ho, Wo)).astype(np.float32), dtype)
    return x, w, b, sc, sh, y, res


def _oracle_per_image(oracle, lists, x, w, b, sc, sh, y, res, R, s, off, dtype):
    """oracle gather (affine + swish, staged in dtype) -> conv -> scatter (+residual), image by image with its own list."""
    want = y.copy()
    for bi, l in enumerate(lists):
        if len(l):
            g = _round(oracle.gather(x[bi:bi + 1], R, R, l, sc[bi:bi + 1], sh[bi:bi + 1], "swish", False), dtype)
            want[bi:bi + 1] = oracle.scatter(oracle.conv2d_tiles(g, w, b, (s, s)), y[bi:bi + 1], off, off, s, s, l, res[bi:bi + 1])
    return want


@pytest.mark.parametrize("geom", GEOMS)
def test_per_image_tile_lists_vs_oracle(oracle, geom):
    """idx_per_image = 1, B = 3 with lists of 5, 13 and 0 tiles (the last image is all padding): lengths that are not
    multiples of the tiles per CTA, so CTAs straddle images and padding rows.  Both kernels, the split-K sweep, per-image
    affine; everything outside the real tiles stays bitwise untouched."""
    from sige_b200 import ops

    dtype = torch.float16
    C, Co, R, k, s, off = geom
    rng = np.random.default_rng(41)
    B, H, W, n = 3, 32, 32, 13
    x, w, b, sc, sh, y, res = _geom_case(oracle, rng, geom, B, H, W, dtype)
    lists = _lists(oracle, rng, R, off, H, W, (5, 13, 0))
    want = _oracle_per_image(oracle, lists, x, w, b, sc, sh, y, res, R, s, off, dtype)
    written = _written(y.shape, lists, off, s, (R - k) // s + 1)
    ty = T(y, dtype, cl=True)
    out = ty.clone(memory_format=torch.channels_last)
    d = _fused_desc(ops, T(x, dtype, cl=True), ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(_padded_lists(lists, n)), out, R=R, k=k, stride=s,
                    off=off, scale=T(sc).reshape(B, C).contiguous(), shift=T(sh).reshape(B, C).contiguous(), act=1, residual=T(res, dtype, cl=True))
    d.idx_per_image, d.N = 1, n
    for flags in (0, TC5):
        for ks in (0, 1, 2, 4, 8):
            out.copy_(ty)
            d.flags, d.ksplit = flags, ks
            ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            e = rel_err(out, want)
            print("per-image lists %s flags %d ksplit %d: rel err %.3g" % (geom, flags, ks, e))
            assert e <= TOL[dtype], "per-image lists %s flags %d ksplit %d: rel err %g" % (geom, flags, ks, e)
            assert _changed_outside(out, ty, written) == 0, "per-image lists %s flags %d ksplit %d: writes outside the real tiles" % (geom, flags, ks)


def test_tc5_fused_shortcut_with_per_image_lists(oracle):
    """The 3x3 conv2 + fused 1x1 shortcut with per-image lists (5, 13, 0 tiles) and per-image sc_flags: image by image, the
    reference's ScatterWithBlockResidual composite."""
    from sige_b200 import ops

    dtype = torch.float16
    rng = np.random.default_rng(43)
    B, Cm, Cx, Co, H, W, n = 3, 128, 128, 128, 32, 32, 13
    lists = _lists(oracle, rng, 6, 1, H, W, (5, 13, 0))
    flags = [np.arange(len(l)) % 2 == 0 for l in lists]                 # every other main tile has its shortcut tile active
    t1 = _round(rng.standard_normal((B, Cm, H, W)).astype(np.float32), dtype)
    xs = _round(rng.standard_normal((B, Cx, H, W)).astype(np.float32), dtype)
    w2 = _round(rng.standard_normal((Co, Cm, 3, 3)).astype(np.float32) / np.sqrt(Cm * 9), dtype)
    b2 = rng.standard_normal((Co,)).astype(np.float32)
    wsc = _round(rng.standard_normal((Co, Cx, 1, 1)).astype(np.float32) / np.sqrt(Cx), dtype)
    bsc = rng.standard_normal((Co,)).astype(np.float32)
    y0 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
    y1 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)
    want = y0.copy()
    for bi, (l, f) in enumerate(zip(lists, flags)):
        if len(l):
            idx1 = (l[f] + 1).astype(np.int32)
            main = oracle.conv2d_tiles(oracle.gather(t1[bi:bi + 1], 6, 6, l), w2, b2, (1, 1))
            sct = oracle.conv2d_tiles(oracle.gather(xs[bi:bi + 1], 4, 4, idx1), wsc, bsc, (1, 1))
            want[bi:bi + 1] = oracle.scatter_with_block_residual(main, y0[bi:bi + 1], sct, y1[bi:bi + 1], 1, 1, 1, 1, l, idx1)
    pflags = np.zeros((B * n,), np.uint8)
    for bi, f in enumerate(flags):
        pflags[bi * n:bi * n + len(f)] = f
    written = _written(y0.shape, lists, 1, 1, 4)
    ty = T(y0, dtype, cl=True)
    out = ty.clone(memory_format=torch.channels_last)
    d = _fused_desc(ops, T(t1, dtype, cl=True), ops.pack_conv_weight(T(w2, dtype), dtype), T(b2), T(_padded_lists(lists, n)), out, R=6, k=3, stride=1,
                    off=1, residual=T(y1, dtype, cl=True))
    txs, wscp, tb, tf = T(xs, dtype, cl=True), ops.pack_conv_weight(T(wsc, dtype), dtype), T(bsc), torch.from_numpy(pflags).to(DEV)
    d.n_src2, d.src2[0].ptr, d.src2[0].C, d.src2[0].up = 1, txs.data_ptr(), Cx, 0
    d.Cin2, d.w2_packed, d.bias2, d.sc_flags = Cx, wscp.data_ptr(), tb.data_ptr(), tf.data_ptr()
    d.idx_per_image, d.N = 1, n
    for ks in (1, 2, 0, 8):
        out.copy_(ty)
        d.flags, d.ksplit = TC5, ks
        ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        e = rel_err(out, want)
        print("per-image fused shortcut ksplit %d: rel err %.3g" % (ks, e))
        assert e <= TOL[dtype], "per-image fused shortcut ksplit %d: rel err %g" % (ks, e)
        assert _changed_outside(out, ty, written) == 0


@pytest.mark.parametrize("geom", GEOMS)
def test_padded_lists_equal_the_unpadded_launch(oracle, geom):
    """A fixed-capacity list (B = 1): 13 real tiles, then SIGE_TILE_NONE entries — three whole 32-tile CTAs' worth with
    SIGE_CONV_PADDED, or padding that only fills the last CTA without the flag.  Where sige_tile_conv_plan picks the same
    (path, bn, ksplit, deep_ring) as for the 13-tile list the result is bitwise that launch's; always within TOL of the
    oracle, nothing written outside the real tiles."""
    from ctypes import byref

    from sige_b200 import _cabi, ops

    dtype = torch.float16
    C, Co, R, k, s, off = geom
    rng = np.random.default_rng(47)
    H, W, n = 32, 32, 13
    x, w, b, sc, sh, y, res = _geom_case(oracle, rng, geom, 1, H, W, dtype)
    real = _lists(oracle, rng, R, off, H, W, (n,))
    want = _oracle_per_image(oracle, real, x, w, b, sc, sh, y, res, R, s, off, dtype)
    written = _written(y.shape, real, off, s, (R - k) // s + 1)
    ty, wp = T(y, dtype, cl=True), ops.pack_conv_weight(T(w, dtype), dtype)
    args = dict(R=R, k=k, stride=s, off=off, scale=T(sc).reshape(1, C).contiguous(), shift=T(sh).reshape(1, C).contiguous(), act=1,
                residual=T(res, dtype, cl=True))
    tx = T(x, dtype, cl=True)
    out_u, out_p = ty.clone(memory_format=torch.channels_last), ty.clone(memory_format=torch.channels_last)
    d_u = _fused_desc(ops, tx, wp, T(b), T(real[0]), out_u, **args)
    for cap, pad_flag in ((n + 96, PADDED), (16, 0)):
        d_p = _fused_desc(ops, tx, wp, T(b), T(_padded_lists(real, cap)), out_p, **args)
        for kern in (0, TC5):
            for ks in (1, 2, 4, 8):
                d_u.flags, d_u.ksplit = kern, ks
                d_p.flags, d_p.ksplit = kern | pad_flag, ks
                plans = []
                for d, o in ((d_u, out_u), (d_p, out_p)):
                    pl = _cabi.TileConvPlan()
                    assert _cabi.lib().sige_tile_conv_plan(byref(d), byref(pl)) == 0
                    plans.append((pl.path, pl.bn, pl.ksplit, pl.deep_ring))
                    o.copy_(ty)
                    ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                e = rel_err(out_p, want)
                tag = "%s cap %d flags %d ksplit %d plans %s" % (geom, cap, kern | pad_flag, ks, plans)
                print("padded list %s: rel err %.3g, bitwise %s" % (tag, e, torch.equal(out_p, out_u)))
                assert e <= TOL[dtype], "padded list %s: rel err %g" % (tag, e)
                assert _changed_outside(out_p, ty, written) == 0, "padded list %s: writes outside the real tiles" % tag
                if plans[0] == plans[1]:
                    assert torch.equal(out_p, out_u), "padded list %s: same plan, different result" % tag


@pytest.mark.parametrize("flags", [0, TC5])
def test_channel_windows(oracle, flags):
    """dst_c0 > 0 in a wider destination (dC > Cout), res_c0 > 0 in a wider residual, aux.c0 > 0: exactly channels
    [c0, c0 + Cout) of the real tiles are written, every other channel stays bitwise untouched."""
    from sige_b200 import ops

    dtype = torch.float16
    rng = np.random.default_rng(53)
    B, C, Co, H, W = 1, 128, 128, 32, 32
    dC, dc0, rC, rc0, aC, ac0 = Co + 128, 64, Co + 64, 32, Co + 16, 8
    mask = rng.random((H, W)) < 0.1
    mask[0, 0] = mask[H - 1, W - 1] = True
    idx = oracle.reduce_mask(mask, 6, 4, 1)
    x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
    w = _round(rng.standard_normal((Co, C, 3, 3)).astype(np.float32) / np.sqrt(C * 9), dtype)
    b = rng.standard_normal((Co,)).astype(np.float32)
    y = _round(rng.standard_normal((B, dC, H, W)).astype(np.float32), dtype)
    res = _round(rng.standard_normal((B, rC, H, W)).astype(np.float32), dtype)
    a0 = _round(rng.standard_normal((B, aC, H, W)).astype(np.float32), dtype)
    asc = (1 + 0.2 * rng.standard_normal((Co,))).astype(np.float32)
    ash = (0.2 * rng.standard_normal((Co,))).astype(np.float32)
    tiles = oracle.conv2d_tiles(oracle.gather(x, 6, 6, idx), w, b, (1, 1))
    want = oracle.scatter(tiles, y[:, dc0:dc0 + Co], 1, 1, 1, 1, idx, res[:, rc0:rc0 + Co])
    z = want * asc.reshape(1, -1, 1, 1) + ash.reshape(1, -1, 1, 1)
    want_aux = z / (1 + np.exp(-z))
    written = _written((B, Co, H, W), [idx], 1, 1, 4)
    ty, ta0 = T(y, dtype, cl=True), T(a0, dtype, cl=True)
    out, aux = ty.clone(memory_format=torch.channels_last), ta0.clone(memory_format=torch.channels_last)
    tsc, tsh = T(asc), T(ash)
    d = _fused_desc(ops, T(x, dtype, cl=True), ops.pack_conv_weight(T(w, dtype), dtype), T(b), T(idx), out, R=6, k=3, stride=1, off=1,
                    residual=T(res, dtype, cl=True))
    d.dst_c0, d.res_c0 = dc0, rc0
    d.n_aux = 1
    d.aux[0].ptr, d.aux[0].C, d.aux[0].c0, d.aux[0].scale, d.aux[0].shift, d.aux[0].act = aux.data_ptr(), aC, ac0, tsc.data_ptr(), tsh.data_ptr(), 1
    d.flags = flags
    ops.launch_tile_conv(d, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    e = rel_err(out[:, dc0:dc0 + Co], want)
    g = aux[:, ac0:ac0 + Co].float().cpu().numpy()
    wm = np.broadcast_to(written, g.shape)
    ea = float(np.abs(g - want_aux)[wm].max() / np.abs(want_aux[wm]).max())
    print("channel windows flags %d: dst rel err %.3g, aux rel err %.3g" % (flags, e, ea))
    assert e <= TOL[dtype] and ea <= TOL[dtype]
    in_dst = np.zeros((1, dC, 1, 1), bool)
    in_dst[:, dc0:dc0 + Co] = True
    in_aux = np.zeros((1, aC, 1, 1), bool)
    in_aux[:, ac0:ac0 + Co] = True
    assert _changed_outside(out, ty, written & in_dst) == 0, "channels outside [dst_c0, dst_c0 + Cout) or pixels outside the tiles changed"
    assert _changed_outside(aux, ta0, written & in_aux) == 0, "aux channels outside [c0, c0 + Cout) or pixels outside the tiles changed"


def test_resblock_vs_oracle(oracle):
    """sige_resblock (C-ABI) against the oracle composite, every tile: conv1 (GroupNorm affine + SiLU gather) -> its aux view
    act(h*scale2+shift2) -> conv2 from that view + fused 1x1 shortcut on flagged tiles / cached shortcut output elsewhere.
    conv2's reference is evaluated on the aux view as conv1 left it, so the check is per launch (no amplification) and also
    proves conv2 read conv1's tiles."""
    import ctypes

    from sige_b200 import _cabi, ops

    dtype = torch.float16
    rng = np.random.default_rng(59)
    B, C, Co, H, W = 1, 128, 128, 32, 32
    mask = rng.random((H, W)) < 0.1
    mask[0, 0] = mask[H - 1, W - 1] = True
    idx = oracle.reduce_mask(mask, 6, 4, 1)
    flags = (np.arange(len(idx)) % 3 != 1).astype(np.uint8)
    idx1 = (idx[flags == 1] + 1).astype(np.int32)
    x = _round(rng.standard_normal((B, C, H, W)).astype(np.float32), dtype)
    w1 = _round(rng.standard_normal((Co, C, 3, 3)).astype(np.float32) / np.sqrt(C * 9), dtype)
    b1 = rng.standard_normal((Co,)).astype(np.float32)
    w2 = _round(rng.standard_normal((Co, Co, 3, 3)).astype(np.float32) / np.sqrt(Co * 9), dtype)
    b2 = rng.standard_normal((Co,)).astype(np.float32)
    wsc = _round(rng.standard_normal((Co, C, 1, 1)).astype(np.float32) / np.sqrt(C), dtype)
    bsc = rng.standard_normal((Co,)).astype(np.float32)
    sc1 = (1 + 0.2 * rng.standard_normal((1, C, 1, 1))).astype(np.float32)
    sh1 = (0.2 * rng.standard_normal((1, C, 1, 1))).astype(np.float32)
    sc2 = (1 + 0.2 * rng.standard_normal((Co,))).astype(np.float32)
    sh2 = (0.2 * rng.standard_normal((Co,))).astype(np.float32)
    h0 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)          # cached conv1 output
    v0 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)          # its transformed view (cached)
    y0 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)          # cached block output
    y1 = _round(rng.standard_normal((B, Co, H, W)).astype(np.float32), dtype)          # cached shortcut output
    th0, tv0, ty0 = T(h0, dtype, cl=True), T(v0, dtype, cl=True), T(y0, dtype, cl=True)
    h, v, out = (t.clone(memory_format=torch.channels_last) for t in (th0, tv0, ty0))
    tx, tidx = T(x, dtype, cl=True), T(idx)
    d1 = _fused_desc(ops, tx, ops.pack_conv_weight(T(w1, dtype), dtype), T(b1), tidx, h, R=6, k=3, stride=1, off=1,
                     scale=T(sc1).reshape(1, C).contiguous(), shift=T(sh1).reshape(1, C).contiguous(), act=1)
    tsc2, tsh2 = T(sc2), T(sh2)
    d1.n_aux = 1
    d1.aux[0].ptr, d1.aux[0].C, d1.aux[0].c0, d1.aux[0].scale, d1.aux[0].shift, d1.aux[0].act = v.data_ptr(), Co, 0, tsc2.data_ptr(), tsh2.data_ptr(), 1
    d2 = _fused_desc(ops, v, ops.pack_conv_weight(T(w2, dtype), dtype), T(b2), tidx, out, R=6, k=3, stride=1, off=1, residual=T(y1, dtype, cl=True))
    wscp, tbsc, tf = ops.pack_conv_weight(T(wsc, dtype), dtype), T(bsc), torch.from_numpy(flags).to(DEV)
    d2.n_src2, d2.src2[0].ptr, d2.src2[0].C, d2.src2[0].up = 1, tx.data_ptr(), C, 0
    d2.Cin2, d2.w2_packed, d2.bias2, d2.sc_flags = C, wscp.data_ptr(), tbsc.data_ptr(), tf.data_ptr()
    d1.flags = d2.flags = TC5
    rc = _cabi.lib().sige_resblock(ctypes.byref(d1), ctypes.byref(d2), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, _cabi.last_error()
    torch.cuda.synchronize()
    written = _written(h0.shape, [idx], 1, 1, 4)
    # conv1 and its view
    want_h = oracle.scatter(oracle.conv2d_tiles(_round(oracle.gather(x, 6, 6, idx, sc1, sh1, "swish", False), dtype), w1, b1, (1, 1)), h0, 1, 1, 1, 1, idx)
    z = want_h * sc2.reshape(1, -1, 1, 1) + sh2.reshape(1, -1, 1, 1)
    want_v = np.where(written, z / (1 + np.exp(-z)), v0)
    e_h, e_v = rel_err(h, want_h), rel_err(v, want_v)
    # conv2 + shortcut, from the view as conv1 left it
    v_now = v.float().cpu().numpy()
    main = oracle.conv2d_tiles(oracle.gather(v_now, 6, 6, idx), w2, b2, (1, 1))
    sct = oracle.conv2d_tiles(oracle.gather(x, 4, 4, idx1), wsc, bsc, (1, 1))
    want_out = oracle.scatter_with_block_residual(main, y0, sct, y1, 1, 1, 1, 1, idx, idx1)
    e_o = rel_err(out, want_out)
    print("sige_resblock, %d tiles: conv1 %.3g, its view %.3g, conv2 + shortcut %.3g" % (len(idx), e_h, e_v, e_o))
    assert e_h <= TOL[dtype] and e_v <= TOL[dtype] and e_o <= TOL[dtype]
    for got, before in ((h, th0), (v, tv0), (out, ty0)):
        assert _changed_outside(got, before, written) == 0, "sige_resblock wrote outside the active tiles"

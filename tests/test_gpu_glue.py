"""Dense glue kernels (conv_in, GroupNorm fold, conv_out) vs a plain PyTorch fp32 reference of the same
op (these are floating-point kernels with no counterpart in the reference's native code: the reference
calls ATen/cuDNN for them, sige_fused_unet.py:395,431-433)."""
import pytest
import torch
from torch.nn import functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 1e-3), (torch.bfloat16, 8e-3)])
def test_conv_in(dtype, tol):
    from sige_b200 import ops

    torch.manual_seed(0)
    for (B, Cin, Cout, H, W) in [(1, 3, 128, 256, 256), (2, 3, 64, 37, 52), (1, 4, 8, 8, 8), (1, 1, 16, 5, 12)]:
        x = torch.randn(B, Cin, H, W, device=DEV).to(dtype)
        w = (torch.randn(Cout, Cin, 3, 3, device=DEV) / (Cin * 9) ** 0.5).to(dtype)
        b = torch.randn(Cout, device=DEV).to(dtype)
        want = F.conv2d(x.float(), w.float(), b.float(), 1, 1)
        got = ops.conv_in_nhwc(x.contiguous(memory_format=torch.channels_last), w, b)
        assert got.shape == want.shape and got.is_contiguous(memory_format=torch.channels_last)
        assert float((got.float() - want).abs().max() / want.abs().max()) <= tol


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 2e-3), (torch.bfloat16, 1.6e-2)])
def test_group_norm_fold_and_conv_out(dtype, tol):
    from sige_b200 import ops

    torch.manual_seed(1)
    for (B, C, G, H, W, Cout) in [(1, 128, 32, 256, 256, 3), (2, 64, 32, 24, 40, 3), (1, 256, 32, 16, 16, 4), (1, 32, 32, 7, 9, 1), (1, 64, 32, 40, 70, 8)]:
        x = (torch.randn(B, C, H, W, device=DEV) * 1.5 + 0.3).to(dtype).contiguous(memory_format=torch.channels_last)
        gamma = (1 + 0.1 * torch.randn(C, device=DEV)).to(dtype)
        beta = (0.1 * torch.randn(C, device=DEV)).to(dtype)
        w = (torch.randn(Cout, C, 3, 3, device=DEV) / (C * 9) ** 0.5).to(dtype)
        b = torch.randn(Cout, device=DEV).to(dtype)
        scale, shift = ops.group_norm_fold(x, G, 1e-6, gamma, beta)
        gn = F.group_norm(x.float(), G, gamma.float(), beta.float(), 1e-6)
        folded = x.float() * scale.view(B, C, 1, 1) + shift.view(B, C, 1, 1)
        assert float((folded - gn).abs().max() / gn.abs().max()) <= 1e-4      # fp32 statistics
        s1, h1 = ops.group_norm_fold(x, G, 1e-6, gamma, beta)
        assert torch.equal(s1, scale) and torch.equal(h1, shift), "deterministic reduction"
        want = F.conv2d(F.silu(gn), w.float(), b.float(), 1, 1)
        got = ops.conv_out_nhwc(x, scale, shift, "swish", w, b)
        assert got.shape == want.shape and got.is_contiguous()
        assert float((got.float() - want).abs().max() / want.abs().max()) <= tol
        plain = ops.conv_out_nhwc(x, None, None, "identity", w, None)
        want2 = F.conv2d(x.float(), w.float(), None, 1, 1)
        assert float((plain.float() - want2).abs().max() / want2.abs().max()) <= tol


@pytest.mark.parametrize("N,C", [(256, 512), (64, 512), (128, 512), (128, 256), (256, 256), (64, 256)])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_attention_tokens_matches_fp32_softmax(N, C, dtype):
    """The fused attention core (reference sige_fused_unet.py:185-199: bmm, softmax, bmm) vs plain fp32 torch on the same
    16-bit inputs.  Logit scale ~ N(0, 2) gives a peaked softmax, so the cluster's flash-style combine is exercised."""
    from sige_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(N * 7 + C)
    qkv = torch.randn(2, N, 3 * C, generator=g)
    qkv[:, :, :C] *= 2.0 * C ** -0.5           # q carries the c^-0.5 attention scale
    qkv = qkv.to(DEV, dtype)
    out = ops.attention_tokens(qkv)
    q, k, v = (t.float() for t in qkv.split(C, dim=2))
    ref = torch.softmax(q @ k.transpose(1, 2), dim=-1) @ v
    err = float((out.float() - ref).abs().max()) / float(ref.abs().max())
    assert err <= (4e-3 if dtype == torch.float16 else 2e-2), err
    # programmatic-dependent-launch flavour of the same launch, back to back on one stream
    out2 = torch.empty_like(out)
    for _ in range(3):
        ops.attention_tokens(qkv, out=out2, flags=1)
    assert torch.equal(out, out2)


def test_attention_tokens_rejects_unsupported_shapes():
    from sige_b200 import ops

    assert not ops.attention_tokens_supported(100, 512, torch.float16)
    assert not ops.attention_tokens_supported(256, 192, torch.float16)
    assert not ops.attention_tokens_supported(256, 512, torch.float32)
    with pytest.raises(RuntimeError):
        ops.attention_tokens(torch.zeros(1, 96, 3 * 512, device=DEV, dtype=torch.float16))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_conv_in_tiles_matches_dense_inside_the_tiles(dtype):
    """Stem restricted to a tile list (sige_conv_in_nhwc_tiles): bit-identical to the dense stem inside the tiles,
    untouched outside; tiles may overlap and may stick out of the image."""
    from sige_b200 import ops

    torch.manual_seed(3)
    B, Cin, Cout, H, W = 1, 3, 128, 64, 48
    x = torch.randn(B, Cin, H, W, device=DEV).to(dtype).contiguous(memory_format=torch.channels_last)
    w = (torch.randn(Cout, Cin, 3, 3, device=DEV) / (Cin * 9) ** 0.5).to(dtype)
    b = torch.randn(Cout, device=DEV).to(dtype)
    sc, sh = torch.rand(Cout, device=DEV) + 0.5, torch.randn(Cout, device=DEV)
    dense_aux = torch.empty(B, Cout, H, W, device=DEV, dtype=dtype).contiguous(memory_format=torch.channels_last)
    dense = ops.conv_in_nhwc(x, w, b, aux=[ops.conv_aux(dense_aux, sc, sh, "swish")])
    tiles = torch.tensor([[-1, -1], [3, 7], [7, 7], [59, 43], [30, 44]], dtype=torch.int32, device=DEV)
    out = torch.full_like(dense, 7.0)
    aux = torch.full_like(dense, 7.0)
    ops.conv_in_nhwc(x, w, b, out=out, aux=[ops.conv_aux(aux, sc, sh, "swish")], tiles=tiles, tile_size=6)
    inside = torch.zeros(H, W, dtype=torch.bool, device=DEV)
    for (y0, x0) in tiles.tolist():
        inside[max(y0, 0):max(min(y0 + 6, H), 0), max(x0, 0):max(min(x0 + 6, W), 0)] = True
    assert torch.equal(out[:, :, inside], dense[:, :, inside]) and torch.equal(aux[:, :, inside], dense_aux[:, :, inside])
    assert bool((out[:, :, ~inside] == 7.0).all()) and bool((aux[:, :, ~inside] == 7.0).all())


@pytest.mark.parametrize("dtype,tol", [(torch.float16, 1e-3), (torch.bfloat16, 8e-3)])
def test_conv_in_per_image_tiles_vs_float64(dtype, tol):
    """sige_conv_in_nhwc_tiles with idx_per_image = 1 (a batch of edits): B = 2, each image with its own list padded with
    SIGE_TILE_NONE rows; inside each image's own tiles the float64 conv, nothing written anywhere else (not in the other
    image's tiles either)."""
    from sige_b200 import ops

    torch.manual_seed(5)
    B, Cin, Cout, H, W, n, NONE = 2, 3, 128, 40, 36, 6, -30000
    x = torch.randn(B, Cin, H, W, device=DEV).to(dtype).contiguous(memory_format=torch.channels_last)
    w = (torch.randn(Cout, Cin, 3, 3, device=DEV) / (Cin * 9) ** 0.5).to(dtype)
    b = torch.randn(Cout, device=DEV).to(dtype)
    lists = [[[-1, -1], [3, 7], [35, 31]], [[7, 7], [19, -1], [-1, 27], [11, 15], [23, 3], [35, 11]]]
    tiles = torch.full((B * n, 2), NONE, dtype=torch.int32)
    for bi, l in enumerate(lists):
        tiles[bi * n:bi * n + len(l)] = torch.tensor(l, dtype=torch.int32)
    out = torch.full((B, Cout, H, W), 7.0, device=DEV, dtype=dtype).contiguous(memory_format=torch.channels_last)
    ops.conv_in_nhwc(x, w, b, out=out, tiles=tiles.to(DEV), tile_size=6, tiles_per_image=True)
    want = F.conv2d(x.double().cpu(), w.double().cpu(), b.double().cpu(), 1, 1)
    inside = torch.zeros(B, 1, H, W, dtype=torch.bool)
    for bi, l in enumerate(lists):
        for (y0, x0) in l:
            inside[bi, :, max(y0, 0):min(y0 + 6, H), max(x0, 0):min(x0 + 6, W)] = True
    inside = inside.expand(B, Cout, H, W)
    got = out.double().cpu()
    err = float((got - want)[inside].abs().max() / want[inside].abs().max())
    print("conv_in per-image tiles %s: %.3g" % (dtype, err))
    assert err <= tol
    assert bool((got[~inside] == 7.0).all()), "written outside the image's own tiles"


# Stable Diffusion v1 shapes at a 15 % edit (8 heads x batch 2; head dims 40 / 80 / 160; self-attention against all 4096 / 1024 /
# 256 / 64 tokens, cross-attention against the 77 text tokens) plus ragged ones (one query, one key, tails that are not a
# multiple of the 64-row blocks).
_SATTN_SHAPES = [(16, 1000, 4096, 40), (16, 250, 1024, 80), (16, 70, 256, 160), (16, 16, 64, 160), (16, 1000, 77, 40), (16, 250, 77, 80),
                 (3, 1, 1, 64), (2, 65, 130, 128), (1, 129, 63, 40), (2, 64, 64, 64), (4, 200, 6, 32)]


@pytest.mark.parametrize("BH,Nq,Nk,D", _SATTN_SHAPES)
@pytest.mark.parametrize("dtype,tol", [(torch.float16, 1e-3), (torch.bfloat16, 8e-3)])
def test_sparse_attention_matches_fp32_softmax(BH, Nq, Nk, D, dtype, tol):
    """sige_sparse_attention (the reference's bmm -> * scale -> softmax -> bmm for sparse queries, stable-diffusion/ldm/modules/
    attention.py:81-93, sige_attention.py:44-58) vs plain fp32 torch on the same 16-bit operands.  Logits ~ N(0, 4): a peaked
    softmax, so the online rescaling across key blocks is exercised."""
    from sige_b200 import ops

    g = torch.Generator(device="cpu").manual_seed(BH * 131 + Nq * 7 + Nk + D)
    q = (torch.randn(BH, Nq, D, generator=g) * 2.0).to(DEV).to(dtype)
    k = torch.randn(BH, Nk, D, generator=g).to(DEV).to(dtype)
    v = torch.randn(BH, Nk, D, generator=g).to(DEV).to(dtype)
    scale = D ** -0.5
    want = torch.bmm(torch.softmax(torch.bmm(q.float(), k.float().transpose(1, 2)) * scale, dim=-1), v.float())
    got = ops.sparse_attention(q, k, v, scale)
    assert got.shape == q.shape and got.dtype == dtype
    err = float((got.float() - want).abs().max() / want.abs().max())
    assert err <= tol, err
    again = ops.sparse_attention(q, k, v, scale)
    assert torch.equal(got, again), "deterministic"


def test_sparse_attention_strided_heads_and_empty():
    """Operands addressed in place in the 'b n (h d)' layout the Linear layers produce (no rearrange copy), and the no-tile case."""
    from sige_b200 import ops

    torch.manual_seed(5)
    b, h, nq, nk, d = 2, 8, 150, 300, 40
    q = torch.randn(b, nq, h * d, device=DEV).half()
    k = torch.randn(b, nk, h * d, device=DEV).half()
    v = torch.randn(b, nk, h * d, device=DEV).half()
    out = torch.zeros(b, nq, h * d, device=DEV).half()
    view = lambda t: t.view(t.shape[0], t.shape[1], h, d).permute(0, 2, 1, 3)          # [b, h, n, d], strided
    ops.sparse_attention(view(q), view(k), view(v), d ** -0.5, out=view(out))
    q3, k3, v3 = (view(t).reshape(b * h, -1, d).float() for t in (q, k, v))
    want = torch.bmm(torch.softmax(torch.bmm(q3, k3.transpose(1, 2)) * d ** -0.5, dim=-1), v3)
    got = view(out).reshape(b * h, nq, d).float()
    assert float((got - want).abs().max() / want.abs().max()) <= 1e-3
    empty = ops.sparse_attention(q3[:, :0].half().contiguous(), k3.half(), v3.half(), d ** -0.5)
    assert empty.shape == (b * h, 0, d)
    with pytest.raises(Exception):
        ops.sparse_attention(q3.half(), k3.half()[:, :, :32].contiguous(), v3.half(), d ** -0.5)      # head dims differ


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-6), (torch.float16, 1e-3), (torch.bfloat16, 8e-3)])
def test_spade_modulate_matches_torch(dtype, tol):
    """sige_spade_modulate = act(x * (1 + gamma) + beta) (reference gaugan/models/sige_normalization.py:84-86 + the block's
    leaky_relu) vs plain fp32 torch on the same operands: NHWC tile stacks, gamma / beta as the channel halves of one stack
    (torch.split views, pixel stride 2C), with and without the activation, an NHWC full tensor, and the refusal of NCHW operands."""
    from sige_b200 import ops

    torch.manual_seed(3)
    for (N, C, R) in [(300, 128, 6), (7, 64, 4), (1, 256, 6), (33, 32, 5)]:
        x = torch.randn(N, C, R, R, device=DEV).to(dtype).contiguous(memory_format=torch.channels_last)
        gb = (0.5 * torch.randn(N, 2 * C, R, R, device=DEV)).to(dtype).contiguous(memory_format=torch.channels_last)
        gamma, beta = torch.split(gb, C, dim=1)
        for slope in (1.0, 0.2):
            want = x.float() * (1 + gamma.float()) + beta.float()
            want = torch.where(want > 0, want, want * slope)
            got = ops.spade_modulate(x, gamma, beta, slope)
            assert got.shape == x.shape and got.dtype == dtype and got.is_contiguous(memory_format=torch.channels_last)
            assert float((got.float() - want).abs().max() / want.abs().max()) <= tol
    full = torch.randn(2, 64, 16, 24, device=DEV).to(dtype).contiguous(memory_format=torch.channels_last)
    got = ops.spade_modulate(full, full, full, 1.0)
    want = full.float() * (1 + full.float()) + full.float()
    assert float((got.float() - want).abs().max() / want.abs().max()) <= tol
    nchw = torch.randn(4, 64, 6, 6, device=DEV).to(dtype)
    assert not ops.spade_modulate_supported(nchw, nchw, nchw)
    with pytest.raises(ValueError):
        ops.spade_modulate(nchw, nchw, nchw)

"""CPU simulator of the launch descriptors of sige_b200.fused — TEST INFRASTRUCTURE.

``sige_b200.fused.Lowering`` turns a traced forward into ``ConvSpec`` / conv_in / tail / attention records and
hands them to an executor.  The product executor (``CudaExecutor``) builds C-ABI descriptors for
libsige_b200.so.  This one interprets the SAME records with plain fp32 torch ops on the CPU, following the
launch contract of include/sige_b200.h (``sige_tile_conv_t``): gather halo tiles from the (virtually
concatenated / upsampled) sources, pre-op, zero outside the image AFTER the pre-op, conv, + bias, fused 1x1
shortcut on flagged tiles / cached residual elsewhere, in-place scatter, extra transformed destinations.

It lets the CPU suite check the tracing + lowering (which launches, which buffers, which folds) against the
reference's golden outputs without a GPU; the kernels themselves are checked on the GPU against the oracle.  The contract
itself lives in plain functions (`tile_conv`, `conv_in`, `tail`, `attention`, `sparse_attention`, `spade`) that
tests/test_gpu_launch_parity.py also evaluates in float64 on snapshots of every launch of the real step.
"""
from __future__ import annotations

import torch
from torch.nn import functional as F


def _act(z, name):
    return z * torch.sigmoid(z) if name == "swish" else z


def _stage(z, stage):
    """Round to the storage type the kernels stage an operand in (fp16 / bf16), back in z's dtype; None: no rounding."""
    return z if stage is None else z.to(stage).to(z.dtype)


def _vec(t, dtype, stage=None):
    return None if t is None else _stage(t.to(dtype), stage)


# =====================================================================================================================
# The launch contract as plain functions.  Each one reads the tensors of its record, computes in `dtype` and writes its
# outputs IN PLACE.  `stage` (torch.float16 / torch.bfloat16 or None) rounds what the kernels stage in that type: the
# gather-side pre-op act(x*scale+shift) and the weights; aux outputs come from the unrounded accumulator.  SimExecutor
# runs them in fp32 without staging; tests/test_gpu_launch_parity.py runs them in float64 on snapshots of GPU launches.
# =====================================================================================================================
def tile_conv(s, dtype=torch.float32, stage=None):
    """One ``sige_tile_conv`` launch of ConvSpec `s` (include/sige_b200.h, sige_tile_conv_t): gather halo tiles from the
    (virtually concatenated / upsampled) sources, pre-op, zero outside the image AFTER the pre-op, conv, + bias, fused 1x1
    shortcut on flagged tiles / cached residual elsewhere, in-place scatter, extra transformed destinations.

    Returns the tile map of the destination: int64 [B, dH, dW], the list position of the tile that wrote each pixel and
    -1 where nothing was written (None for a tile-stack destination, which is written whole)."""
    w = s.weight.to(dtype)
    b = None if s.bias is None else s.bias.to(dtype)
    if s.out_row_scale is not None:
        rows, f = s.out_row_scale
        w = w.clone()
        w[:rows] *= f
        if b is not None:
            b = b.clone()
            b[:rows] *= f
    w = _stage(w, stage)
    k, st, R = s.k, s.stride, s.block
    ro = (R - k) // st + 1
    if s.src_is_stack:
        X = s.srcs[0][0].to(dtype)
        M = X.shape[0]
        coords = None if s.idx is None else [(bi, iy, ix) for bi in range(s.B) for (iy, ix) in s.idx.tolist()]
    else:
        parts = [F.interpolate(t.to(dtype), scale_factor=2.0, mode="nearest") if up else t.to(dtype) for (t, up) in s.srcs]
        full = parts[0] if len(parts) == 1 else torch.cat(parts, 1)
        B, C, H, W = full.shape
        assert (H, W) == (s.H, s.W) and B == s.B, (s.name, full.shape, s.B, s.H, s.W)
        if s.scale is not None:
            sc = s.scale.to(dtype)
            full = full * (sc.view(1, -1, 1, 1) if sc.dim() == 1 else sc.view(B, -1, 1, 1))
        if s.shift is not None:
            sh = s.shift.to(dtype)
            full = full + (sh.view(1, -1, 1, 1) if sh.dim() == 1 else sh.view(B, -1, 1, 1))
        full = _stage(_act(full, s.act), stage)
        P = R + 4
        padded = F.pad(full, (P, P, P, P))                  # zero AFTER the pre-op
        idx = s.idx.tolist()
        tiles, coords = [], []
        if s.tile_img is not None:          # batch of independent edits: tile i belongs to image tile_img[i]
            assert len(idx) == s.N == s.tile_img.numel()
            for bi, (iy, ix) in zip(s.tile_img.tolist(), idx):
                assert 0 <= bi < B
                tiles.append(padded[bi, :, iy + P:iy + P + R, ix + P:ix + P + R])
                coords.append((bi, iy, ix))
        else:
            for bi in range(B):
                for (iy, ix) in idx:
                    if iy <= -20000:          # SIGE_TILE_NONE padding of a fixed-capacity list: reads zeros, writes nothing
                        tiles.append(torch.zeros_like(padded[0, :, :R, :R]))
                        coords.append(None)
                        continue
                    tiles.append(padded[bi, :, iy + P:iy + P + R, ix + P:ix + P + R])
                    coords.append((bi, iy, ix))
        X = torch.stack(tiles)
        M = X.shape[0]
    out = F.conv2d(X, w, b, stride=st)
    assert out.shape[2] == ro
    fresh = torch.zeros(M, dtype=torch.bool)
    if s.shortcut is not None:
        sc_tensors, sc_w, sc_b, sc_flags = s.shortcut
        raw = torch.cat([t.to(dtype) for t in sc_tensors], 1)
        sw = _stage(sc_w.to(dtype), stage)
        sb = None if sc_b is None else sc_b.to(dtype)
        flags = [1] * s.N if sc_flags is None else sc_flags.tolist()
        assert k == 3 and R == 6 and st == 1
        Pp = 8
        rp = F.pad(raw, (Pp, Pp, Pp, Pp))
        for m, co_ in enumerate(coords):
            if co_ is None:
                continue
            bi, iy, ix = co_
            if flags[m % s.N]:
                fresh[m] = True
                centre = rp[bi:bi + 1, :, iy + 1 + Pp:iy + 5 + Pp, ix + 1 + Pp:ix + 5 + Pp]
                out[m] += F.conv2d(centre, sw, sb)[0]
    if s.dst_stack is not None:
        assert s.residual is None and not s.aux
        s.dst_stack.copy_(out)
        return None
    dst = s.dst
    Bd, Cd, Hd, Wd = dst.shape
    # scatter: output pixel (r, c) of tile m lands at ((off + iy) / stride + r, (off + ix) / stride + c) of image bi
    if coords is None:
        coords = [(0, 0, 0)] * M
    real = [m for m in range(M) if coords[m] is not None]
    tile_map = torch.full((Bd, Hd, Wd), -1, dtype=torch.int64)
    if not real:
        return tile_map
    cm = torch.tensor([coords[m] for m in real], dtype=torch.int64).view(-1, 3)
    assert bool(((s.off + cm[:, 1:]) >= 0).all()), s.name
    r = torch.arange(ro)
    bi = cm[:, 0].view(-1, 1, 1).expand(-1, ro, ro)
    hh = ((s.off + cm[:, 1]) // st).view(-1, 1, 1) + r.view(1, -1, 1)
    ww = ((s.off + cm[:, 2]) // st).view(-1, 1, 1) + r.view(1, 1, -1)
    hh, ww = hh.expand(-1, ro, ro), ww.expand(-1, ro, ro)
    inside = (hh < Hd) & (ww < Wd)
    m_of = torch.tensor(real, dtype=torch.int64).view(-1, 1, 1).expand(-1, ro, ro)
    bi, hh, ww, m_of = bi[inside], hh[inside], ww[inside], m_of[inside]
    v = out.permute(0, 2, 3, 1)[torch.tensor(real)][inside]             # [pixels, Cout]
    if s.residual is not None:
        res = s.residual.to(dtype).permute(0, 2, 3, 1)[bi, hh, ww]
        v = torch.where(fresh[m_of].view(-1, 1), v, v + res)
    if dst.has_raw:
        dst.raw.permute(0, 2, 3, 1)[bi, hh, ww] = v.to(dst.raw.dtype)
    for (view, sc, sh, act) in s.aux:
        z = v
        if sc is not None:
            z = z * sc.to(dtype)
        if sh is not None:
            z = z + sh.to(dtype)
        view.permute(0, 2, 3, 1)[bi, hh, ww] = _act(z, act).to(view.dtype)
    tile_map[bi, hh, ww] = m_of
    return tile_map


def conv_in(rec, dtype=torch.float32, stage=None):
    """``sige_conv_in_nhwc`` / ``sige_conv_in_nhwc_tiles`` of ConvInRec `rec`: 3x3 pad-1 conv of the <=4-channel input,
    written (with its aux views) only inside the tiles when `rec.tiles` is set.  Returns the written-pixel mask [B, H, W]."""
    y = F.conv2d(rec.x.to(dtype), _vec(rec.weight, dtype, stage), _vec(rec.bias, dtype, stage), padding=1)
    B, C, H, W = y.shape
    sel = torch.zeros((B, H, W), dtype=torch.bool)
    if rec.tiles is None:
        sel[:] = True
    else:
        imgs = [None] * rec.tiles.shape[0] if rec.tile_img is None else rec.tile_img.tolist()
        for bi, (iy, ix) in zip(imgs, rec.tiles.tolist()):
            if iy <= -20000:
                continue
            sel[slice(None) if bi is None else bi, max(iy, 0):max(iy + rec.tile_size, 0), max(ix, 0):max(ix + rec.tile_size, 0)] = True
    sel4 = sel[:, None].expand_as(y)
    if rec.out.has_raw:
        rec.out.raw[sel4] = y[sel4].to(rec.out.raw.dtype)
    for (view, sc, sh, act) in rec.aux:
        z = y
        if sc is not None:
            z = z * sc.to(dtype).view(1, -1, 1, 1)
        if sh is not None:
            z = z + sh.to(dtype).view(1, -1, 1, 1)
        view[sel4] = _act(z, act)[sel4].to(view.dtype)
    return sel


def tail(x, groups, eps, gamma, beta, act, weight, bias, out, dtype=torch.float32, stage=None):
    """GroupNorm -> act -> 3x3 pad-1 conv to few channels (``sige_group_norm_fold`` + ``sige_conv_out_nhwc``)."""
    z = F.group_norm(x.to(dtype), groups, _vec(gamma, dtype, stage), _vec(beta, dtype, stage), eps)
    out.copy_(F.conv2d(_stage(_act(z, act), stage), _vec(weight, dtype, stage), _vec(bias, dtype, stage), padding=1))


def attention(qkv_tokens, out_tokens, dtype=torch.float32):
    """``sige_attention_tokens``: softmax(q k^T) v per image, tokens [B, N, 3C] = [q | k | v], q pre-scaled."""
    C = qkv_tokens.shape[2] // 3
    q, k, v = (qkv_tokens[..., i * C:(i + 1) * C].to(dtype) for i in range(3))
    out_tokens.copy_(torch.softmax(q @ k.transpose(1, 2), dim=-1) @ v)


def sparse_attention(q, k, v, scale, out, dtype=torch.float32):
    """``sige_sparse_attention``: softmax(scale q k^T) v of [bh, n, d] or strided [b, h, n, d] operands."""
    att = torch.softmax(torch.matmul(q.to(dtype), k.to(dtype).transpose(-1, -2)) * scale, dim=-1)
    out.copy_(torch.matmul(att, v.to(dtype)))


def spade(x, gamma, beta, slope, out, dtype=torch.float32):
    """``sige_spade_modulate``: leaky_relu(x * (1 + gamma) + beta, slope)."""
    z = x.to(dtype) * (1 + gamma.to(dtype)) + beta.to(dtype)
    out.copy_(torch.where(z > 0, z, z * slope))


class SimExecutor:
    name = "sim"

    def __init__(self):
        self.launches = 0
        self.device = torch.device("cpu")
        self.dtype = torch.float32

    # ------------------------------------------------------------------ fused tile conv
    def prepare_conv(self, fc) -> None:
        def run(_stream):
            self.launches += 1
            tile_conv(fc.spec)

        fc.launch_fn = run

    # ------------------------------------------------------------------ stem / tail / attention / gather
    def prepare_conv_in(self, rec):
        def run(_stream):
            self.launches += 1
            conv_in(rec)

        return run

    def prepare_tail(self, x, groups, eps, gamma, beta, act, weight, bias, out):
        def run(_stream):
            self.launches += 3
            tail(x, groups, eps, gamma, beta, act, weight, bias, out)

        return run

    def attention_supported(self, n_tokens, channels):
        return True

    def tail_supported(self, channels, cout):
        return True

    def prepare_attention(self, qkv_tokens, out_tokens, pdl):
        def run(_stream):
            self.launches += 1
            attention(qkv_tokens, out_tokens)

        return run

    def spade_supported(self, x, gamma, beta):
        return True

    def prepare_spade(self, x, gamma, beta, slope, out):
        def run(_stream):
            self.launches += 1
            spade(x, gamma, beta, slope, out)

        return run

    def sparse_attention_supported(self, head_dim):
        return True

    def prepare_sparse_attention(self, q, k, v, scale, out):
        def run(_stream):
            self.launches += 1
            sparse_attention(q, k, v, scale, out)

        return run

    def gather(self, x, block, idx, scale, shift, act, act_first, up=0):
        if up:
            x = F.interpolate(x.float(), scale_factor=2.0, mode="nearest")
        B, C, H, W = x.shape
        z = x.float()
        if not act_first:
            if scale is not None:
                z = z * scale
            if shift is not None:
                z = z + shift
        z = _act(z, act)
        if act_first:
            if scale is not None:
                z = z * scale
            if shift is not None:
                z = z + shift
        P = max(block) + 4
        padded = F.pad(z, (P, P, P, P))
        tiles = [padded[b, :, iy + P:iy + P + block[0], ix + P:ix + P + block[1]] for b in range(B) for (iy, ix) in idx.tolist()]
        if not tiles:
            return x.new_zeros((0, C, block[0], block[1]))
        return torch.stack(tiles)

    def launch_counter(self):
        return self.launches

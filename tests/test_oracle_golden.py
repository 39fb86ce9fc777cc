"""Pins the CPU oracle (oracle/sige_oracle.c) against
  (a) the known-answer vectors probed on the compiled reference (SURVEY.md Appendix A),
  (b) golden fixtures produced by running the reference itself (tests/golden/make_golden.py),
  (c) the reference's compiled CPU backend (oracle/_ref): live when present, and always through the stored digests of
      its outputs (tests/golden/make_golden_compiled_reference.py).
"""
import hashlib

import numpy as np
import pytest
import torch

from conftest import golden


def _mask(h, w, *pts):
    m = np.zeros((h, w), dtype=bool)
    for p in pts:
        m[p] = True
    return m


KATS = [  # (mask, block, stride, pad, expected)   SURVEY.md Appendix A KAT 1-6
    (_mask(8, 8, (3, 3)), 6, 4, 1, [[-1, -1], [-1, 3], [3, -1], [3, 3]]),
    (_mask(8, 8, (3, 3)), 4, 4, 0, [[0, 0]]),
    (_mask(8, 8, (3, 3)), 5, 4, 0, [[0, 0]]),
    (_mask(8, 8, (0, 0)), 6, 4, 1, [[-1, -1]]),
    (_mask(8, 8, (7, 7)), 6, 4, 1, [[3, 3], [3, 7], [7, 3], [7, 7]]),
    (_mask(8, 8, (7, 7)), 4, 4, 0, [[4, 4]]),
    (_mask(8, 8, (7, 7)), 5, 4, 0, [[4, 4]]),
    (_mask(8, 8, (4, 4)), 6, 4, 1, [[-1, -1], [-1, 3], [3, -1], [3, 3]]),
    (_mask(6, 10, (5, 9)), 6, 4, 1, [[3, 7]]),
]


@pytest.mark.parametrize("mask,bs,st,pad,expected", KATS)
def test_reduce_mask_kats(oracle, mask, bs, st, pad, expected):
    got = oracle.reduce_mask(mask, bs, st, pad)
    assert got.dtype == np.int32
    assert got.tolist() == expected


def test_empty_mask_kat6(oracle):
    idx = oracle.reduce_mask(np.zeros((8, 8), bool), 6, 4, 1)
    assert idx.shape == (0, 2) and idx.dtype == np.int32
    x = np.random.default_rng(0).standard_normal((1, 3, 8, 8)).astype(np.float32)
    assert oracle.gather(x, 6, 6, idx).shape == (0, 3, 6, 6)
    y = np.random.default_rng(1).standard_normal((1, 3, 8, 8)).astype(np.float32)
    assert np.array_equal(oracle.scatter(np.zeros((0, 3, 4, 4), np.float32), y, 1, 1, 1, 1, idx), y)


def test_scatter_map_and_gather_kats(oracle):
    idx = oracle.reduce_mask(_mask(8, 8, (3, 3)), 6, 4, 1)
    smap = oracle.get_scatter_map(8, 8, 6, 6, 3, 3, 1, 1, 1, 1, idx)          # KAT 7
    assert smap[4, 5].tolist() == [3, 0, 1] and smap[3, 3].tolist() == [0, 3, 3]
    for q, (r0, c0) in enumerate([(0, 0), (0, 4), (4, 0), (4, 4)]):
        assert (smap[r0:r0 + 4, c0:c0 + 4, 0] == q).all()
    x = np.arange(64, dtype=np.float32).reshape(1, 1, 8, 8)                     # KAT 8
    g = oracle.gather(x, 6, 6, idx)[0, 0]
    assert (g[0] == 0).all() and (g[:, 0] == 0).all()
    assert g[1].tolist() == [0, 0, 1, 2, 3, 4] and g[5].tolist() == [0, 32, 33, 34, 35, 36]
    sc, sh = np.full((1, 1, 1, 1), 2, np.float32), np.full((1, 1, 1, 1), 1, np.float32)
    g = oracle.gather(x, 6, 6, idx, sc, sh)[0, 0]                               # KAT 9: halo stays 0
    assert (g[0] == 0).all() and g[1].tolist() == [0, 1, 3, 5, 7, 9]
    one = np.ones((1, 1, 1, 1), np.float32)                                     # KAT 11
    v = oracle.gather(one, 1, 1, np.zeros((1, 2), np.int32), None, None, "swish")[0, 0, 0, 0]
    assert v == np.float32(0.7310585975646973)


def test_ops_against_reference_golden(oracle):
    """Outputs of the reference's CPU backend on seeded inputs; the inputs are regenerated here
    from the recorded seed in the exact order make_golden.py drew them."""
    G = golden("ops_golden.npz")
    rng = np.random.default_rng(int(G["seed"][0]))
    for ci, (B, C, H, W, bs, ts, k, cs, off) in enumerate(G["cases"].tolist()):
        mask = rng.random((H, W)) < 0.06
        mask[0, 0] = True
        mask[H - 1, W - 1] = True
        assert np.array_equal(mask, G[f"c{ci}_mask"])
        idx = oracle.reduce_mask(mask, bs, ts, off)
        assert np.array_equal(idx, G[f"c{ci}_idx"]), "reduce_mask must be bit-exact"
        N = idx.shape[0]
        x = rng.standard_normal((B, C, H, W)).astype(np.float32) * 2
        scale = rng.standard_normal((1, C, 1, 1)).astype(np.float32)
        shift = rng.standard_normal((B, C, 1, 1)).astype(np.float32)
        assert np.array_equal(oracle.gather(x, bs, bs, idx), G[f"c{ci}_gather_id"])
        assert np.array_equal(oracle.gather(x, bs, bs, idx, scale, shift, "swish", False), G[f"c{ci}_gather_sw"])
        assert np.array_equal(oracle.gather(x, bs, bs, idx, scale, shift, "swish", True), G[f"c{ci}_gather_af"])
        ro = (bs - k) // cs + 1
        ys = G[f"c{ci}_scatter"].shape
        xs = rng.standard_normal((B * N, C, ro, ro)).astype(np.float32)
        y = rng.standard_normal(ys).astype(np.float32)
        res = rng.standard_normal(ys).astype(np.float32)
        assert np.array_equal(oracle.scatter(xs, y, off, off, cs, cs, idx), G[f"c{ci}_scatter"])
        assert np.array_equal(oracle.scatter(xs, y, off, off, cs, cs, idx, res), G[f"c{ci}_scatter_res"])
        if cs == 1:
            smap = oracle.get_scatter_map(H, W, bs, bs, k, k, off, off, cs, cs, idx)
            assert np.array_equal(smap, G[f"c{ci}_map"])
            xprev = rng.standard_normal((B * N, C, ro, ro)).astype(np.float32)
            sg = oracle.scatter_gather(xprev, x, bs, bs, idx, smap, scale, shift, "swish", False)
            assert np.array_equal(sg, G[f"c{ci}_sg"])
    B, C, H, W = 2, 6, 20, 24
    mask = rng.random((H, W)) < 0.05
    idx0, idx1 = oracle.reduce_mask(mask, 6, 4, 1), oracle.reduce_mask(mask, 4, 4, 0)
    assert np.array_equal(idx0, G["br_idx0"]) and np.array_equal(idx1, G["br_idx1"])
    x0 = rng.standard_normal((B * idx0.shape[0], C, 4, 4)).astype(np.float32)
    x1 = rng.standard_normal((B * idx1.shape[0], C, 4, 4)).astype(np.float32)
    y0 = rng.standard_normal((B, C, H, W)).astype(np.float32)
    y1 = rng.standard_normal((B, C, H, W)).astype(np.float32)
    assert np.array_equal(oracle.scatter_with_block_residual(x0, y0, x1, y1, 1, 1, 1, 1, idx0, idx1), G["br_out"])


def test_example_indices_golden(oracle):
    G = golden("example_golden.npz")
    idx = oracle.reduce_mask(G["mask"], 6, 4, 1)
    assert idx.shape[0] == 783 and idx[0].tolist() == [-1, 107]     # SURVEY.md Appendix A 'ex'
    assert np.array_equal(idx, G["idx"])


def test_conv_oracle_against_torch(oracle):
    """The conv arithmetic lives in the pinned torch wheel (reference sige/nn/base.py:89 ->
    F.conv2d); the restatement must agree with it to fp32 rounding."""
    rng = np.random.default_rng(5)
    for (M, Ci, Co, R, k, s, g) in [(5, 8, 12, 6, 3, 1, 1), (3, 16, 16, 5, 3, 2, 1), (4, 12, 12, 6, 3, 1, 12), (2, 36, 20, 4, 1, 1, 1)]:
        x = rng.standard_normal((M, Ci, R, R)).astype(np.float32)
        w = rng.standard_normal((Co, Ci // g, k, k)).astype(np.float32)
        b = rng.standard_normal((Co,)).astype(np.float32)
        a = oracle.conv2d_tiles(x, w, b, (s, s), (1, 1), g)
        ref = torch.nn.functional.conv2d(torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b), s, 0, 1, g).numpy()
        assert np.abs(a - ref).max() <= 1e-5 * np.abs(ref).max()


def _digest(a):
    """SHA-256 of an array's shape and values (-0.0 counted as 0.0): for NaN-free arrays of one dtype, equal digests
    mean np.array_equal."""
    a = np.ascontiguousarray(np.asarray(a) + 0)
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()


def _against_compiled_reference(key, pairs, ref_cpu):
    """`pairs` yields (oracle output, thunk -> the reference's compiled CPU backend's output on the same inputs).  Every
    oracle output must equal the reference's: live when oracle/_ref is present, and always through the digests of the
    reference's outputs stored in tests/golden/compiled_reference_digests.npz (tests/golden/make_golden_compiled_reference.py).
    The digests pin bit-exact values, so they also assume the libm (swish calls expf) and the compiler flags of the machine
    that made them: where the live comparison passes and only the digests differ, the math library differs, not the oracle.
    Each thunk is called before the sweep advances (its lambda reads the loop variables of the current step)."""
    want = list(golden("compiled_reference_digests.npz")[key])
    got = []
    for a, ref_out in pairs:
        if ref_cpu is not None:
            assert np.array_equal(a, ref_out().numpy())
        got.append(_digest(a))
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, ("output %d of the sweep differs from the stored digest of the reference's output (%s; a different libm "
                        "or compiler changes the last bits of swish)" % (i, "the live comparison passed" if ref_cpu is not None else "oracle/_ref absent"))


def sweep_ops(oracle, ref_cpu):
    t = torch.from_numpy
    rng = np.random.default_rng(11)
    for trial in range(25):
        B, C = int(rng.integers(1, 3)), int(rng.integers(1, 9))
        H, W = int(rng.integers(5, 30)), int(rng.integers(5, 30))
        bs, ts, k, off = [(6, 4, 3, 1), (4, 4, 1, 0), (5, 4, 3, 0)][trial % 3]
        cs = 2 if bs == 5 else 1
        mask = rng.random((H, W)) < 0.08
        idx = oracle.reduce_mask(mask, bs, ts, off)
        N = idx.shape[0]
        x = rng.standard_normal((B, C, H, W)).astype(np.float32) * 3
        dims = [(1, C, 1, 1), (B, C, 1, 1), (1, 1, 1, 1), (B, C, H, W), (1, C, H, W), (1, 1, H, 1)][trial % 6]
        sc = rng.standard_normal(dims).astype(np.float32)
        sh = rng.standard_normal(dims).astype(np.float32)
        for af in (False, True):
            yield oracle.gather(x, bs, bs, idx, sc, sh, "swish", af), lambda: ref_cpu.gather(t(x), bs, bs, t(idx), t(sc), t(sh), "swish", af)
        if N == 0:
            continue
        ro = (bs - k) // cs + 1
        Ho, Wo = (H if cs == 1 else (H + 1 - k) // 2 + 1), (W if cs == 1 else (W + 1 - k) // 2 + 1)
        xs = rng.standard_normal((B * N, C, ro, ro)).astype(np.float32)
        y = rng.standard_normal((B, C, Ho, Wo)).astype(np.float32)
        rd = [(B, C, Ho, Wo), (1, C, 1, 1), (1, 1, Ho, Wo)][trial % 3]
        res = rng.standard_normal(rd).astype(np.float32)
        yield oracle.scatter(xs, y, off, off, cs, cs, idx, res), lambda: ref_cpu.scatter(t(xs), t(y), off, off, cs, cs, t(idx), t(res))
        if cs == 1:
            m1 = oracle.get_scatter_map(H, W, bs, bs, k, k, off, off, 1, 1, idx)
            yield m1, lambda: ref_cpu.get_scatter_map(H, W, bs, bs, k, k, off, off, 1, 1, t(idx))
            yield oracle.scatter_gather(xs, x, bs, bs, idx, m1, sc, sh, "swish", False), \
                lambda: ref_cpu.scatter_gather(t(xs), t(x), bs, bs, t(idx), t(m1), t(sc), t(sh), "swish", False)


def test_oracle_against_compiled_reference(oracle, ref_cpu):
    """Differential test vs the reference's own compiled CPU backend over randomised shapes."""
    _against_compiled_reference("ops", sweep_ops(oracle, ref_cpu), ref_cpu)


def sweep_block_residual(oracle, ref_cpu):
    t = torch.from_numpy
    rng = np.random.default_rng(23)
    for trial in range(16):
        B, C = int(rng.integers(1, 3)), [3, 36, 64, 128][trial % 4]
        H, W = int(rng.integers(8, 26)), int(rng.integers(8, 26))
        # main 3x3 tiles and the 1x1 shortcut's own tiles on the same mask (a ResBlock with Cin != Cout)
        mask = rng.random((H, W)) < (0.0 if trial == 5 else 0.06)
        idx0 = oracle.reduce_mask(mask, 6, 4, 1)
        idx1 = oracle.reduce_mask(mask, 4, 4, 0)
        N0, N1 = idx0.shape[0], idx1.shape[0]
        x0 = rng.standard_normal((B * N0, C, 4, 4)).astype(np.float32)
        x1 = rng.standard_normal((B * N1, C, 4, 4)).astype(np.float32)
        y0 = rng.standard_normal((B, C, H, W)).astype(np.float32)
        y1 = rng.standard_normal((B, C, H, W)).astype(np.float32)
        yield oracle.scatter_with_block_residual(x0, y0, x1, y1, 1, 1, 1, 1, idx0, idx1), \
            lambda: ref_cpu.scatter_with_block_residual(t(x0), t(y0), t(x1), t(y1), 1, 1, 1, 1, t(idx0), t(idx1))
        # identity activation, no affine / scale only / shift only
        x = rng.standard_normal((B, C, H, W)).astype(np.float32)
        sc = rng.standard_normal((1, C, 1, 1)).astype(np.float32)
        for (s_, h_) in ((None, None), (sc, None), (None, sc)):
            yield oracle.gather(x, 6, 6, idx0, s_, h_, "identity", False), \
                lambda: ref_cpu.gather(t(x), 6, 6, t(idx0), None if s_ is None else t(s_), None if h_ is None else t(h_), "identity", False)
        # SD down-sampling geometry: k3 s2 p1 -> 5x5 tiles, tile stride 4, offset 1, 2x2 outputs
        idx2 = oracle.reduce_mask(mask, 5, 4, 1)
        N2 = idx2.shape[0]
        Ho, Wo = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
        xs = rng.standard_normal((B * N2, C, 2, 2)).astype(np.float32)
        y = rng.standard_normal((B, C, Ho, Wo)).astype(np.float32)
        yield oracle.scatter(xs, y, 1, 1, 2, 2, idx2, None), lambda: ref_cpu.scatter(t(xs), t(y), 1, 1, 2, 2, t(idx2), None)


def test_block_residual_and_remaining_geometries_against_compiled_reference(oracle, ref_cpu):
    """Second differential sweep vs the reference's compiled CPU backend: scatter_with_block_residual (reference
    sige/cpu/scatter.cpp:41-68,111-135), the identity activation, wider channel counts, the SD down-sampling geometry
    (k3 s2 p1: 5x5 tiles, offset 1) and empty index lists."""
    _against_compiled_reference("block_residual", sweep_block_residual(oracle, ref_cpu), ref_cpu)

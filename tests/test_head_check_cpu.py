"""CPU tests of the DPT-head checks in tools/gpu_check.py (transposed convs, bilinear upsample, patch gather) and of the
output tails' geometry: the upsample reference is pinned to ATen, emulations of the kernels' arithmetic pass the bounds,
simulated kernel bugs fail them, and no geometry the tail launchers accept reaches a trap of tail_mma_kernel or
tail_gather_kernel. The tails' arithmetic (fp16 interpolation, HFMA2 accumulation) has no error model here yet: only their
index math is checked. No kernel is launched."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gpu_check as G  # noqa: E402

F = torch.nn.functional


# ---------------------------------------------------------------------------------------------------- upsample
def test_upsample_reference_weights_match_aten():
    """One-hot rows / columns through F.interpolate (fp32, align_corners=True) give up_matrix's weights: the reference's
    source rows and lambdas are ATen's, not the kernel's."""
    for n_in, n_out in ((1, 1), (1, 2), (2, 4), (3, 5), (5, 10), (19, 37), (37, 74), (40, 70), (148, 296), (7, 14), (36, 72)):
        eye = torch.eye(n_in, dtype=torch.float32).view(1, n_in, n_in, 1)
        aten = F.interpolate(eye, (n_out, 1), mode="bilinear", align_corners=True)[0, :, :, 0].t().double()
        A = G.up_matrix(n_in, n_out)
        assert (A - aten).abs().max().item() <= 2.0 ** -22, (n_in, n_out)
        assert torch.equal(A != 0, aten != 0), (n_in, n_out)
    # and in 2-D, on a non-square map
    x = torch.randn(2, 9, 7, 8).bfloat16()
    ref, _ = G.up_ref64(x, 18, 14)
    aten = F.interpolate(x.float().permute(0, 3, 1, 2), (18, 14), mode="bilinear", align_corners=True).permute(0, 2, 3, 1)
    assert (ref - aten.double()).abs().max().item() <= 1e-5


def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).bfloat16()


def emulate_upsample(x, Ho, Wo, bug=None):
    """upsample_bilinear_kernel in numpy fp32: 16-row strips, each keeping the horizontally interpolated source rows in
    top / bot while it walks down, then one bf16 store. x: NHWC bf16. bug: a simulated kernel bug."""
    xf = x.float().numpy()
    B, Hi, Wi, C = xf.shape
    f32 = np.float32
    if bug == "i1_unclamped":  # i1 = i0 + 1 at the last row: reads the next image / the NaN guard
        xf = np.concatenate([xf, np.full((B, 1, Wi, C), np.nan, np.float32)], 1)

    def coords(n_in, n_out, rows):
        if bug == "align_corners_false":
            s = f32(n_in) / f32(n_out)
            src = np.maximum((np.arange(n_out, dtype=np.float32) + f32(0.5)) * s - f32(0.5), f32(0)).astype(np.float32)
        else:
            s = f32(n_in - 1) / f32(n_out - 1) if n_out > 1 else f32(0)
            src = (s * np.arange(n_out, dtype=np.float32)).astype(np.float32)
        i0 = src.astype(np.int64)
        i1 = i0 + 1 if bug == "i1_unclamped" and rows else i0 + (i0 < n_in - 1)
        lam = (src - i0.astype(np.float32)).astype(np.float32)
        return i0, i1, lam, (f32(1) - lam).astype(np.float32)

    x0, x1, lx, hx = coords(Wi, Wo, False)
    if bug == "hx_lx_swapped":
        lx, hx = hx, lx
    if bug == "weights_bf16":
        lx, hx = _bf16(lx).float().numpy(), _bf16(hx).float().numpy()
    y0s, y1s, lys, hys = coords(Hi, Ho, True)

    def hlerp(row):  # [B, Wi, C] -> [B, Wo, C]
        return (hx[None, :, None] * row[:, x0] + lx[None, :, None] * row[:, x1]).astype(np.float32)

    out = np.empty((B, Ho, Wo, C), np.float32)
    top = bot = None
    cy0 = cy1 = -1
    for yo in range(Ho):
        if yo % 16 == 0 and bug != "stale_top_at_strip":  # a new strip (thread block) starts with nothing cached
            cy0 = cy1 = -1
        y0, y1, ly, hy = y0s[yo], y1s[yo], lys[yo], hys[yo]
        if y0 != cy0:
            if bug == "stale_top_at_strip" and yo % 16 == 0 and cy0 >= 0:
                pass  # the strip boundary: top keeps the previous strip's row
            else:
                top = bot if y0 == cy1 else hlerp(xf[:, y0])
            cy0, cy1 = y0, -1
        if y1 != cy1:
            bot = top if y1 == y0 else hlerp(xf[:, y1])
            cy1 = y1
        out[:, yo] = (hy * top + ly * bot).astype(np.float32)
    return _bf16(out)


UP_CASES = [(1, 1, 1, 1), (1, 1, 2, 2), (3, 3, 5, 5), (5, 5, 10, 10), (10, 10, 20, 20), (20, 20, 40, 40), (5, 4, 9, 7),
            (9, 7, 18, 14), (36, 28, 72, 56), (19, 19, 37, 37), (40, 40, 70, 70)]


def _up_verdict(x, got, Ho, Wo):
    ref, bound = G.up_ref64(x, Ho, Wo)
    return G.head_verdict(got, ref, bound)


def test_upsample_emulation_passes_bound():
    worst = 0.0
    for i, (Hi, Wi, Ho, Wo) in enumerate(UP_CASES):
        for mode in ("rand", "ramp"):
            for C in (8, 24):
                x = G.up_operands(2, Hi, Wi, C, mode, i)
                r = _up_verdict(x, emulate_upsample(x, Ho, Wo), Ho, Wo)
                assert r["ok"], (Hi, Wi, Ho, Wo, mode, r)
                worst = max(worst, r["err_bound"])
    print(f"upsample emulation: largest err/bound {worst:.3f}")


@pytest.mark.parametrize("bug", ["align_corners_false", "i1_unclamped", "hx_lx_swapped", "stale_top_at_strip"])
def test_upsample_simulated_bug_fails(bug):
    # a stale top only shows where a strip boundary is also a source-row change: the down2(g) -> g maps (19 -> 37) and
    # 40 -> 70 have such boundaries, the near-2x maps g -> 2g do not
    maps =[(19, 19, 37, 37), (40, 40, 70, 70)] if bug == "stale_top_at_strip" else [(19, 19, 37, 37), (5, 4, 9, 7)]
    for i, (Hi, Wi, Ho, Wo) in enumerate(maps):
        x = G.up_operands(2, Hi, Wi, 8, "ramp", 100 + i)
        r = _up_verdict(x, emulate_upsample(x, Ho, Wo, bug), Ho, Wo)
        assert not r["ok"] and r["err_bound"] > 10.0, (bug, Hi, Ho, r)


def test_old_upsample_tolerance_misses_bf16_weights():
    """Interpolation weights rounded to bf16 stay inside the old _cmp(2e-2, 1e-2) on its random inputs, but miss the fp64
    bound wherever corners of opposite sign cancel."""
    x = G.up_operands(2, 37, 37, 64, "rand", 7)
    bad = emulate_upsample(x, 74, 74, "weights_bf16")
    old = F.interpolate(x.float().permute(0, 3, 1, 2), (74, 74), mode="bilinear", align_corners=True).permute(0, 2, 3, 1)
    assert G._cmp("up", bad, old, 2e-2, 1e-2)["ok"]
    assert not _up_verdict(x, bad, 74, 74)["ok"]


def test_up_maps_are_the_four_launched_maps():
    assert G.up_maps(37, 37) == [(19, 19, 37, 37), (37, 37, 74, 74), (74, 74, 148, 148), (148, 148, 296, 296)]
    assert G.up_maps(1, 1)[0] == (1, 1, 1, 1) and G.up_maps(9, 7)[0] == (5, 4, 9, 7)
    assert 384 in G.UP_WIDTHS and (384 // 8) & (384 // 8 - 1)  # 48 channel groups: not a power of two
    for c in G.UP_WIDTHS:
        for gh, gw in G.UP_GRIDS:
            assert f"upsample_geo_c{c}_{gh}x{gw}" in G.CHECKS


# ---------------------------------------------------------------------------------------------------- transposed conv
CONVT_CASES = [(4, 48, 2, 7, 5), (2, 96, 3, 5, 3), (4, 64, 2, 3, 4)]


def _convT_verdict(op, ks, got):
    ref, bound = G.convT_ref64(op, ks)
    return G.head_verdict(got, ref, bound)


@pytest.mark.parametrize("mode", ["rand", "onehot"])
def test_convT_correctly_rounded_output_passes(mode):
    for i, (ks, Ci, B, H, W) in enumerate(CONVT_CASES):
        op = G.convT_operands(B, H, W, Ci, Ci, ks, mode, i)
        ref, _ = G.convT_ref64(op, ks)
        r = _convT_verdict(op, ks, ref.bfloat16())
        assert r["ok"], (ks, Ci, mode, r)


@pytest.mark.parametrize("mode", ["rand", "onehot"])
@pytest.mark.parametrize("bug", ["ky_kx_swapped", "last_column_dropped", "neighbouring_image"])
def test_convT_simulated_bug_fails(mode, bug):
    """Each bug is a permutation (or loss) of where EPI_CONVT's outputs land, applied to the correctly rounded result
    rather than to an emulation of the epilogue: this shows that the bound and the one-hot inputs tell such misplaced
    stores apart from rounding, not that the epilogue's index math is right (the GPU rows check that)."""
    for i, (ks, Ci, B, H, W) in enumerate(CONVT_CASES):
        op = G.convT_operands(B, H, W, Ci, Ci, ks, mode, i)
        ref, _ = G.convT_ref64(op, ks)
        out = ref.clone()
        if bug == "ky_kx_swapped":  # the pixel shuffle with ky and kx exchanged inside each ks x ks block
            out = out.view(B, H, ks, W, ks, Ci).transpose(2, 4).reshape(out.shape)
        elif bug == "last_column_dropped":  # the last input column never reaches the output: bias only there
            out[:, :, (W - 1) * ks:] = op["b"].double()
        else:  # the rows of image b + 1 stored into image b
            out = out[[min(b + 1, B - 1) for b in range(B)]]
        r = _convT_verdict(op, ks, out.bfloat16())
        assert not r["ok"] and r["err_bound"] > 10.0, (bug, ks, Ci, r)


def test_convT_rows_name_every_launched_width():
    rows = G.CONVT_GEO_ROWS
    assert {r[1] for r in rows if r[0] == 4} >= {48, 96, 256, 1536}
    assert {r[1] for r in rows if r[0] == 2} >= {96, 192, 512, 1536}
    assert {r[4] for r in rows} >= {37, 49, 7, 5, 32, 1}
    assert any(r[5] == 2 and r[3:5] == (32, 32) for r in rows) and any(r[5] == 2 and r[3:5] == (37, 37) for r in rows)
    assert (4, 256, 4, 32, 32, 0, None) in rows and (4, 256, 32, 37, 37, 0, (0, 16, 31)) in rows


# ---------------------------------------------------------------------------------------------------- patch gather
def test_patch_gather_wrong_channel_statistics_fail():
    g = torch.Generator().manual_seed(3)
    rgb = torch.rand(2, 3, 28, 70, generator=g)
    guides = [torch.rand(2, 1, 28, 70, generator=g) * 2 - 1 for _ in range(2)]
    exp = G.patch_gather_expected(rgb, guides)
    assert exp.shape == (2 * 2 * 5, 5 * 196)
    # patch (b 1, py 1, px 3), channel 1 (green), ky 2, kx 5
    assert exp[1 * 10 + 1 * 5 + 3, 196 + 2 * 14 + 5].item() == torch.tensor(
        (rgb[1, 1, 16, 47].item() - np.float32(0.456)) / np.float32(0.224)).bfloat16().item()
    for mean, std in (((0.456, 0.485, 0.406), G.PG_STD), (G.PG_MEAN, (0.229, 0.225, 0.224))):
        bad = G.patch_gather_expected(rgb, guides, mean, std)
        assert not torch.equal(bad.view(torch.int16), exp.view(torch.int16))


def test_patch_gather_rows_cover_chunking():
    pw = {r[2] // 14 for r in G.PG_ROWS}
    assert pw >= {1, 5, 32, 33, 37, 74}
    assert {sum(r[3]) for r in G.PG_ROWS} >= {0, 2, 4, 5}
    assert all(len(r[3]) <= 3 and 3 + sum(r[3]) <= 8 for r in G.PG_ROWS)
    assert max(r[0] for r in G.PG_ROWS if r[1:3] == (518, 518)) == 32


# ---------------------------------------------------------------------------------------------------- tail geometry
# The trap conditions of tail_mma_kernel (0x7A21 / 0x7A22) and tail_gather_kernel (0x7A11), evaluated in fp32 exactly as
# the kernels compute them, for every geometry the launchers accept: Hl 14 == H 8 and Wl 14 == W 8 (tail_mma also needs
# W % 14 == 0), H, W up to 4200.
f32 = np.float32
KMAX = 600  # H = 7 k


def _scale(n_lo, n_hi):
    return f32(n_lo - 1) / f32(n_hi - 1) if n_hi > 1 else f32(0)


def tm_rows(H, Hl):
    """tail_mma_kernel's TMA warp for every row tile: (trap 0x7A22 anywhere, interior tiles, interior tiles off the fast
    row table)."""
    sh = _scale(Hl, H)
    Y0 = np.arange(0, H, 8)
    r0 = (sh * np.maximum(Y0 - 1, 0).astype(np.float32)).astype(np.int64)
    Y = Y0[:, None] - 1 + np.arange(10)[None, :]
    inside = (Y >= 0) & (Y < H)
    fy = (sh * np.clip(Y, 0, None).astype(np.float32)).astype(np.float32)
    y0 = fy.astype(np.int64)
    jrow = y0 - r0[:, None]
    trap = inside & ((jrow < 0) | (jrow > 7) | ((jrow == 7) & (y0 < Hl - 1)))
    d = (np.arange(10) * 57) // 100
    in_table = ~inside | (jrow == d) | (jrow == d + 1)
    interior = inside.all(1)
    return bool(trap.any()), int(interior.sum()), int((interior & ~in_table.all(1)).sum())


def tm_cols(W, Wl):
    """tail_mma_kernel's interpolation warps for every column tile: trap 0x7A21 anywhere."""
    sw = _scale(Wl, W)
    X0 = np.arange(0, W, 14)
    c0 = (sw * np.maximum(X0 - 1, 0).astype(np.float32)).astype(np.int64)
    X = X0[:, None] - 1 + np.arange(16)[None, :]
    xok = (X >= 0) & (X < W)
    fx = (sw * np.clip(X, 0, W - 1).astype(np.float32)).astype(np.float32)
    x0 = fx.astype(np.int64)
    xo0, xo1 = x0 - c0[:, None], x0 + (x0 < Wl - 1) - c0[:, None]
    return bool((xok & ((xo0 < 0) | (xo1 >= 12))).any())


def tg_axis(H, Hl):
    """tail_gather_kernel along one axis for every 16-pixel tile: (patch extent > 12 anywhere = trap 0x7A11, a tap's
    source row outside the staged patch anywhere)."""
    sh = _scale(Hl, H)
    Y0 = np.arange(0, H, 16)
    r0 = (sh * np.maximum(Y0 - 1, 0).astype(np.float32)).astype(np.int64)
    r1 = np.minimum((sh * np.minimum(Y0 + 16, H - 1).astype(np.float32)).astype(np.int64) + 1, Hl - 1)
    n = r1 - r0 + 1
    py = Y0[:, None] - 1 + np.arange(18)[None, :]  # the tap rows of the tile's rows Y0 .. min(Y0 + 16, H) - 1
    ok = (py >= 0) & (py < H) & (py <= np.minimum(Y0 + 16, H)[:, None])
    y0 = (sh * np.clip(py, 0, None).astype(np.float32)).astype(np.float32).astype(np.int64)
    yr0, yr1 = y0 - r0[:, None], y0 + (y0 < Hl - 1) - r0[:, None]
    outside = ok & ((yr0 < 0) | (yr1 > (n - 1)[:, None]))
    return bool((n > 12).any()), bool(outside.any())


def test_no_accepted_tail_geometry_traps():
    """Every H = 7 k (Hl = 4 k) and W = 14 k (Wl = 8 k) up to 4200 for tail_mma_kernel, every H, W = 7 k for
    tail_gather_kernel: no trap condition holds and every tap reads inside the staged patch. Interior row tiles whose halo
    rows miss tm_row_d's d / d + 1 table take the general path; their count is reported, not judged."""
    misses, interior = 0, 0
    for k in range(1, KMAX + 1):
        H, Hl = 7 * k, 4 * k
        trap, n_int, n_miss = tm_rows(H, Hl)
        assert not trap, ("0x7A22", H)
        interior += n_int
        misses += n_miss
        ext, outside = tg_axis(H, Hl)
        assert not ext and not outside, ("0x7A11", H, ext, outside)
        if k % 2 == 0:
            assert not tm_cols(H, Hl), ("0x7A21", H)
    print(f"tail_mma: {misses} of {interior} interior row tiles off the fast-path table (H = 7k, k <= {KMAX})")


def test_trap_emulation_sees_other_geometries():
    """The emulated conditions are live: a 1:1 map (not 8h -> 14h) trips them, which is why the launchers refuse it."""
    assert tm_rows(64, 64)[0] and tm_cols(64, 64)
    assert tg_axis(64, 64)[0]

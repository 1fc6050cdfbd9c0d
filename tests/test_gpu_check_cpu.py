"""CPU tests of the kernel checks in tools/gpu_check.py: the conv tile-shape table reaches every geometry the picker can
choose, and the fp64 reference, its error bound and the exact checks reject simulated kernel bugs while a correctly
rounded result passes. No kernel is launched (ada_conv_tile_shape runs on the host)."""
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gpu_check as G  # noqa: E402

ALL_GEOS = {(lw, lh, 7 - lw - lh, pair) for lw in range(1, 6) for lh in range(0, 8 - lw) for pair in (1, 2)}


def _row(geo):
    return next(r for r in G.CONV_GEO_ROWS if r[:4] == geo)


# small rows: 32 images per tile (residual neighbours), a ragged 96-channel input, two 64-column groups of N
ROW_MULTI = _row((1, 1, 5, 1))     # B 25, 5 x 5, Cin 64, N 96
ROW_CIN96 = _row((1, 5, 1, 1))     # B 5, 25 x 5, Cin 96, N 96
ROW_N128 = _row((2, 3, 2, 1))      # B 7, 21 x 11, Cin 48, N 128


def _operands(row, seed=0):
    B, H, W, Cin, N = row[4:]
    return G.conv_geo_operands(B, H, W, Cin, N, seed)


def _rounded(ref, variant):
    return ref.to(torch.float16 if G.CONV_VARIANTS[variant].get("epi") == "f16" else torch.bfloat16)


def _kernel_like(op, variant):
    """What a correct kernel stores: the fp64 result rounded once, and its ReLU copy."""
    ref, _, relu_copy = G.conv_ref64(op, variant)
    out = _rounded(ref, variant)
    return out, (G.relu_copy_of(out) if relu_copy else None)


def _verdict(op, variant, got, got_relu):
    ref, bound, relu_copy = G.conv_ref64(op, variant)
    return G.conv_verdict(got, got_relu, ref, bound, relu_copy)


def test_table_covers_every_tile_shape():
    assert len(ALL_GEOS) == 50
    rows = G.CONV_GEO_ROWS
    assert sorted(r[:4] for r in rows) == sorted(ALL_GEOS)
    for lw, lh, lb, pair, B, H, W, Cin, N in rows:
        assert G.conv_tile_shape(B, H, W, pair) == (lw, lh, lb), (lw, lh, lb, pair)
        tw, th, nb = (1 << lw) * pair, 1 << lh, 1 << lb
        assert W % tw and (th == 1 or H % th) and (nb == 1 or B % nb), ("not ragged", lw, lh, lb, pair)
        assert Cin in (48, 64, 96, 256) and N in (48, 96, 128, 256)
        assert pair == 1 or N == 256  # force_cg=2 pairs only BN = 256 tiles of these epilogues
        assert B <= 40 and (H >= 3 and W >= 3 or (lw, lh, lb) == (1, 0, 6))
        assert f"conv_geo_{lw}{lh}{lb}_{pair}" in G.CHECKS
    assert {r[7] for r in rows} == {48, 64, 96, 256} and {r[8] for r in rows} == {48, 96, 128, 256}


def test_gemm_tiles_list_every_built_instantiation():
    """GEMM_TILES names exactly the (BN, CG) pairs ada_api.cu instantiates for each linear epilogue."""
    src = open(os.path.join(ROOT, "amodal-depth-anything_b200", "csrc", "ada_api.cu")).read()
    built = {}
    for bn, cg, epi in re.findall(r"^\s*ADA_GEMM_CASE\((\d+), (\d+), (\w+)\)", src, re.M):
        built.setdefault(epi, []).append((int(bn), int(cg)))
    epi_of = {"bf16": "EPI_BF16", "gelu": "EPI_BF16_GELU", "gamma": "EPI_BF16", "resid_f32": "EPI_RESID_F32",
              "swiglu": "EPI_SWIGLU", "f16": "EPI_F16", "embed": "EPI_EMBED"}
    assert set(G.GEMM_TILES) == set(epi_of)
    for kind, tiles in G.GEMM_TILES.items():
        assert sorted(tiles) == sorted(built[epi_of[kind]]), kind
        assert f"gemm_tiles_{kind}" in G.CHECKS


@pytest.mark.parametrize("row", [ROW_MULTI, ROW_CIN96, ROW_N128, _row((1, 0, 6, 2))])
def test_correctly_rounded_output_passes(row):
    op = _operands(row)
    for v in G.CONV_VARIANTS:
        out, relu = _kernel_like(op, v)
        r = _verdict(op, v, out, relu)
        assert r["ok"] and r["err_bound"] <= 1.0, (v, r)


def test_residual_of_the_neighbouring_image_fails():
    op = _operands(ROW_MULTI)
    B = op["r1"].shape[0]
    bug = dict(op, r1=op["r1"][[i ^ 1 if i ^ 1 < B else i for i in range(B)]])
    for v in ("d_resid2_relu_copy", "e_resid1"):
        out, relu = _kernel_like(bug, v)
        assert not _verdict(op, v, out, relu)["ok"], v


def test_missing_top_taps_on_the_first_row_of_each_tile_fails():
    op = _operands(ROW_MULTI)
    th = 1 << ROW_MULTI[1]
    w = op["w"].clone()
    w[:, :, 0, :] = 0
    bad, _ = _kernel_like(dict(op, w=w), "a_bias")
    out, _ = _kernel_like(op, "a_bias")
    ys = list(range(0, out.shape[1], th))
    out[:, ys] = bad[:, ys]
    assert not _verdict(op, "a_bias", out, None)["ok"]


def test_missing_bias_on_the_second_column_group_fails():
    op = _operands(ROW_N128)
    b = op["b"].clone()
    b[64:128] = 0
    for v in ("a_bias", "c_relu", "g_f16", "h_s2_bias"):
        out, relu = _kernel_like(dict(op, b=b), v)
        assert not _verdict(op, v, out, relu)["ok"], v


def test_relu_copy_taken_before_the_residual_add_fails():
    op = _operands(ROW_MULTI)
    out, _ = _kernel_like(op, "d_resid2_relu_copy")
    pre, _ = _kernel_like(op, "a_bias")
    r = _verdict(op, "d_resid2_relu_copy", out, G.relu_copy_of(pre))
    assert not r["ok"] and not r["relu_copy_exact"]


def test_chln_statistics_over_the_first_64_channels_fails():
    for row in (ROW_MULTI, ROW_N128):
        op = _operands(row)
        acc, _, _ = G.conv_ref64(op, "a_bias")
        part = acc[..., :64]
        mean = part.mean(-1, keepdim=True)
        rstd = 1.0 / torch.sqrt((part - mean).pow(2).mean(-1, keepdim=True) + 1e-6)
        out = torch.relu((acc - mean) * rstd * op["lnw"].double() + op["lnb"].double()).bfloat16()
        assert not _verdict(op, "f_chln", out, None)["ok"]


def test_dropped_ragged_input_channel_chunk_fails():
    op = _operands(ROW_CIN96)
    x, xs = op["x"].clone(), op["xs"].clone()
    x[..., 64:] = 0
    xs[..., 64:] = 0
    bug = dict(op, x=x, xs=xs)
    for v in G.CONV_VARIANTS:
        out, relu = _kernel_like(bug, v)
        assert not _verdict(op, v, out, relu)["ok"], v


def test_unwritten_tile_fails():
    lw, lh, lb = ROW_MULTI[:3]
    op = _operands(ROW_MULTI)
    for v in ("a_bias", "b_relu_copy", "f_chln"):
        out, relu = _kernel_like(op, v)
        out[:1 << lb, 1 << lh:2 << lh, :1 << lw] = float("nan")  # the second tile row: never stored
        r = _verdict(op, v, out, relu)
        assert not r["ok"] and r["nan"] > 0, v
    # an output buffer nothing was stored to
    B, H, W, _, N = ROW_MULTI[4:]
    empty = G.Guarded((B, H, W, N), torch.bfloat16, "cpu", 64)
    assert not _verdict(op, "a_bias", empty.t, None)["ok"]


def test_overwritten_canary_fails():
    B, H, W, _, N = ROW_MULTI[4:]
    op = _operands(ROW_MULTI)
    out, _ = _kernel_like(op, "a_bias")
    for where in ("before", "after"):
        g = G.Guarded((B, H, W, N), torch.bfloat16, "cpu", G._guard_for(H * W * N))
        g.t.copy_(out)
        assert g.canaries_intact() and _verdict(op, "a_bias", g.t, None)["ok"]
        i = g.guard - 1 if where == "before" else g.guard + g.n + H * W * N - 1  # last element of the image past the end
        g.buf[i] = -g.buf[i] if g.buf[i] != 0 else 1.0
        assert not g.canaries_intact(), where


def test_nan_guard_inputs_and_tensor_alignment():
    g = G.Guarded((3, 5, 7, 96), torch.bfloat16, "cpu", G._guard_for(5 * 7 * 96), fill=float("nan"))
    assert torch.isnan(g.buf[:g.guard]).all() and torch.isnan(g.buf[g.guard + g.n:]).all()
    assert g.guard % 64 == 0 and g.guard >= 5 * 7 * 96  # 16-byte aligned for TMA; a whole image of guard
    assert G.err_over_bound(torch.tensor([float("nan")]), torch.tensor([1.0], dtype=torch.float64),
                            torch.tensor([1.0], dtype=torch.float64)) == float("inf")

"""CPU tests of the encoder checks in tools/gpu_check.py (attention, token LayerNorm, channel LayerNorm): the exponential
the attention kernels evaluate on the FMA pipe is measured against the EXP_EPS the bound assumes, kernel-faithful
emulations and correctly rounded results pass the fp64 bounds, simulated kernel bugs fail them, and the shape tables
reach every residue, tile count, head count, width and launch kind they claim to. No kernel is launched."""
import math
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gpu_check as G  # noqa: E402

CSRC = os.path.join(ROOT, "amodal-depth-anything_b200", "csrc")
F32 = np.float32


# ---------------------------------------------------------------------------------------------------- exp2_fma2 (ptx.cuh)
def _exp2_fma2_constants():
    """Clamp, magic number and the four polynomial coefficients, read from exp2_fma2 itself, so that a change to the
    kernel's polynomial is re-measured here."""
    src = open(os.path.join(CSRC, "ptx.cuh")).read()
    body = src[src.index("void exp2_fma2("):]
    body = body[:body.index("\n}")]
    clamp = float(re.search(r"fmaxf\(x0, (-?[\d.]+)f\)", body).group(1))
    magic = float(re.search(r"f2_add\(xc, f2_pack\(([\d.]+)f", body).group(1))
    coef = [float(c) for c in re.findall(r"f2_pack\((0\.\d+)f, \1f\)", body)]
    assert len(coef) == 4 and "<< 23" in body, body
    return F32(clamp), F32(magic), [F32(c) for c in coef]


def _fma32(a, b, c):
    """fp32 fma: a * b is exact in fp64 (24 + 24 bits); the sum is rounded to fp64, then to fp32."""
    return (a.astype(np.float64) * np.float64(b) + np.float64(c) if np.isscalar(c) else
            a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


def exp2_fma2_emulated(x):
    """exp2_fma2 step by step in fp32: clamp at -125, round to an integer with the 1.5 * 2^23 magic number, the degree-3
    polynomial on the fraction as three FMAs, and the integer added to the exponent field as (bits(t) << 23)."""
    clamp, magic, (c3, c2, c1, c0) = _exp2_fma2_constants()
    x = np.asarray(x, dtype=F32)
    xc = np.maximum(x, clamp).astype(F32)
    with np.errstate(over="ignore"):
        t = (xc + magic).astype(F32)
        n = (t - magic).astype(F32)
    f = _fma32(n, F32(-1.0), xc)
    p = _fma32(f, c3, c2)
    p = _fma32(p, f, c1)
    p = _fma32(p, f, c0)
    tb = t.view(np.int32).astype(np.int64)
    bits = (p.view(np.int32).astype(np.int64) + (tb << 23)) & 0xFFFFFFFF
    return bits.astype(np.uint32).view(F32)


def test_exp2_polynomial_error_is_below_the_bound_constant():
    """The largest relative error of the FMA-pipe exponential over every argument a score row produces ([-125, 8]: p
    reaches 2^8 under the stale maximum) stays below EXP_EPS, the constant the attention bound uses."""
    grid = np.linspace(-125.0, 8.0, 1 << 22, dtype=np.float64).astype(F32)
    # and every fp32 value of one unit interval (the polynomial only sees the fraction, so one interval covers its shape)
    lo, hi = np.array([-1.0, 0.0], dtype=F32).view(np.int32)
    unit = np.concatenate([np.arange(0, hi.item() + 1, 7, dtype=np.int32).view(F32),
                           -np.arange(0, 0x3F800000 + 1, 7, dtype=np.int32).view(F32)])
    x = np.concatenate([grid, unit, np.array([-125.0, -124.5, -0.5, 0.5, 7.5, 8.0], dtype=F32)])
    got = exp2_fma2_emulated(x).astype(np.float64)
    exact = np.exp2(x.astype(np.float64))
    rel = np.abs(got / exact - 1.0)
    worst = rel.max()
    assert 2.0 ** -15 < worst < G.EXP_EPS, worst      # measured 7.5e-5 = 2^-13.7
    assert worst < 0.62 * G.EXP_EPS                   # the slack that covers the fp32 rounding of the argument


def test_masked_key_on_an_fma_column_gets_2_to_the_minus_125():
    """A key past N carries a score of -inf; on the FMA-pipe columns the clamp turns it into 2^-125 times the polynomial's
    value at 0, not 0 (MUFU ex2 gives exactly 0). Such a p is harmless only because the key's V row is zero-filled by
    the tensor map, so it adds 2^-125 to the row sum and nothing to P V."""
    _, _, (c3, c2, c1, c0) = _exp2_fma2_constants()
    got = exp2_fma2_emulated(np.array([-np.inf, -1e30, -125.0, -200.0], dtype=F32))
    assert (got == F32(np.ldexp(np.float64(c0), -125))).all(), got
    assert got[0] > 0 and np.isfinite(got).all()
    # representable in bf16 (8-bit exponent, normal): P = 2^-125 enters P V as a nonzero weight
    assert torch.tensor(got[:1]).bfloat16().float().item() > 0


# ------------------------------------------------------------------------------------ attention.cuh, emulated on the host
EMU_PAIRS = 0x9249  # kEmuMask: exponential pairs (of the 16 in a 32-column half) evaluated on the FMA pipe


def _exp2_mufu(x):
    """ex2.approx.ftz.f32: 2^x rounded to fp32, subnormal results flushed to 0."""
    y = torch.exp2(x.double())
    return torch.where(y < 2.0 ** -126, torch.zeros_like(y), y).float()


def emulate_attention(qkv, bug=None, scale_log2e=None):
    """attention.cuh on the host, one (image, head, 128-query tile) at a time, in the kernel's arithmetic: fp32 scores of
    the bf16 operands, keys past N zero-filled and their scores set to -inf, a stale row maximum per 128-key tile that is
    raised only when some row of the 32-row warp grows by more than 2^8 (then O and l are rescaled by ex2 of the
    difference), x = fma(s, c, -m c) in fp32, p from the FMA-pipe polynomial on the 0x9249 column pairs and MUFU ex2
    elsewhere, an fp32 row sum of the unrounded p, P rounded to bf16 for P V in fp32, and out = O * (1 / l) in bf16.
    bug: "phantom" (one key past N escapes the mask), "mask_last" (the last real key is masked too), "no_o_rescale"
    (l is rescaled, O is not)."""
    B, N, _, H, _ = qkv.shape
    c = F32(scale_log2e if scale_log2e is not None else F32(0.125) * F32(1.4426950408889634))
    T = (N + 127) // 128
    R = T * 128
    col = torch.arange(128)
    emu_col = ((EMU_PAIRS >> ((col % 32) // 2)) & 1).bool()
    x = qkv.float()
    q = torch.zeros(B, H, R, 64)
    k = torch.zeros(B, H, R, 64)
    v = torch.zeros(B, H, R, 64)
    q[:, :, :N] = x[:, :, 0].permute(0, 2, 1, 3)
    k[:, :, :N] = x[:, :, 1].permute(0, 2, 1, 3)
    v[:, :, :N] = x[:, :, 2].permute(0, 2, 1, 3)
    O = torch.zeros(B, H, R, 64)
    l = torch.zeros(B, H, R)
    m = None
    for j in range(T):
        kj, vj = k[:, :, j * 128:(j + 1) * 128], v[:, :, j * 128:(j + 1) * 128]
        s = q @ kj.transpose(-1, -2)  # [B, H, R, 128] fp32
        valid = min(128, N - j * 128)
        if bug == "phantom":
            valid = min(128, valid + 1)
        if bug == "mask_last" and j == T - 1:
            valid -= 1
        s[..., valid:] = -math.inf
        tmax = s.max(-1).values
        if m is None:
            m = tmax
        else:
            grow = (tmax - m) * torch.tensor(c) > 8.0
            anyg = grow.view(B, H, R // 32, 32).any(-1, keepdim=True).expand(B, H, R // 32, 32).reshape(B, H, R)
            m_new = torch.where(anyg, torch.maximum(m, tmax), m)
            sc = torch.where(anyg, _exp2_mufu((m - m_new) * torch.tensor(c)), torch.ones_like(m))
            l = l * sc
            if bug != "no_o_rescale":
                O = O * sc.unsqueeze(-1)
            m = m_new
        mc = (m * torch.tensor(c)).double()
        xx = (s.double() * float(c) - mc.unsqueeze(-1)).float()
        p_fma = torch.from_numpy(exp2_fma2_emulated(xx.numpy()))
        p = torch.where(emu_col, p_fma, _exp2_mufu(xx))
        l = l + p.sum(-1)
        O = O + p.bfloat16().float() @ vj
    inv = 1.0 / l
    out = (O * inv.unsqueeze(-1))[:, :, :N].bfloat16()
    return out.permute(0, 2, 1, 3).reshape(B * N, H * 64)


def _att(qkv, got):
    B, N, _, H, _ = qkv.shape
    pairs = [(b, h) for b in range(B) for h in range(H)]
    ref, bound = G.att_ref64(qkv)
    return G.att_verdict(G.att_select(got, B, N, H, pairs), ref, bound)


def _rounded_ref(qkv):
    B, N, _, H, _ = qkv.shape
    ref, _ = G.att_ref64(qkv)
    return ref.view(B, H, N, 64).permute(0, 2, 1, 3).reshape(B * N, H * 64).bfloat16()


# small rows of every kind of last tile: a single key, r = 1 / 2 / 33 / 63 / 64 / 65 / 127, 2 and 3 KV tiles
EMU_ROWS = [(2, 2, 2), (1, 17, 2), (1, 64, 1), (1, 65, 2), (1, 129, 2), (1, 130, 1), (1, 161, 1), (1, 191, 1),
            (1, 255, 1), (1, 289, 1), (1, 320, 1)]
RAGGED = [r for r in EMU_ROWS if r[1] % 128]


@pytest.mark.parametrize("row", EMU_ROWS)
def test_kernel_emulation_and_rounded_reference_pass(row):
    B, N, H = row
    modes = G.ATT_MODES if N > 256 else G._ATT_BASE + ("wide",)
    for mi, mode in enumerate(modes):
        qkv = G.att_operands(B, N, H, mode, seed=100 + mi)
        r = _att(qkv, emulate_attention(qkv))
        assert r["ok"], (mode, r)
        r = _att(qkv, _rounded_ref(qkv))
        assert r["ok"] and r["err_bound"] <= 0.6, (mode, r)


def test_grow_modes_exercise_the_rescale_rule():
    """grow forces O rescales after the first tile (some later tile's maximum is more than 2^8 above the running one in
    most rows); grow8 lifts every tile's maximum by just under 2^8, so p reaches ~2^7.5 between rescales."""
    c = 0.125 * math.log2(math.e)
    for mode in ("grow", "grow8"):
        qkv = G.att_operands(1, 1370, 2, mode, seed=3).float()
        s = qkv[0, :, 0].transpose(0, 1) @ qkv[0, :, 1].permute(1, 2, 0)  # [H, N, N]
        tile_max = torch.stack([s[..., t * 128:(t + 1) * 128].amax(-1) for t in range(11)], -1) * c
        if mode == "grow":
            running = torch.cummax(tile_max, -1).values
            jumps = tile_max[..., 2:] - running[..., 1:-1]
            assert (jumps > 8.0).any(-1).float().mean() > 0.5
        else:
            steps = tile_max[..., 1:10] - tile_max[..., :9]
            assert (steps > 7.0).all() and (steps < 8.0).all(), (steps.min(), steps.max())


def test_bf16_p_rounding_needs_the_full_2_to_the_minus_8_term():
    """Why the P term is 2^-8 R rather than 2^-9 (R + |ref|): with two keys of equal weight whose p round to bf16 in
    opposite directions while their v have opposite signs, the output moves by 2^-8 R while ref is ~0."""
    p = torch.tensor([1.0 + 2 ** -8 - 2 ** -20, 1.0 + 3 * 2 ** -8 + 2 ** -20])  # round down / up by ~2^-8 relative
    v = torch.tensor([-1.0, 1.0])
    a = p.double() / p.double().sum()
    ref, R = (a * v).sum(), (a * v.abs()).sum()
    got = (p.bfloat16().double() * v).sum() / p.double().sum()
    assert abs(got - ref) > 2 ** -9 * (R + abs(ref)) + 2 ** -8 * abs(ref)
    assert abs(got - ref) <= 2 ** -8 * R + 2 ** -8 * abs(ref)


def test_phantom_key_passes_the_old_tolerance():
    """The gap the neg inputs close: on the random inputs of the former check, a key past N that escapes the mask moves
    the output by a fraction of a percent -- inside the former atol = rtol = 2e-2 torch comparison and inside the fp64
    bound alike. With every real score negative the same bug takes most of the weight and fails both."""
    for N in (200, 1370):
        qkv = G.att_operands(1, N, 2, "rand", seed=5)
        bad = emulate_attention(qkv, bug="phantom")
        ref = _rounded_ref(qkv).float()
        assert ((bad.float() - ref).abs() <= 2e-2 + 2e-2 * ref.abs()).all(), N
        qkv = G.att_operands(1, N, 2, "neg", seed=5)
        bad = emulate_attention(qkv, bug="phantom")
        ref = _rounded_ref(qkv).float()
        assert not ((bad.float() - ref).abs() <= 2e-2 + 2e-2 * ref.abs()).all(), N
        assert not _att(qkv, bad)["ok"], N


@pytest.mark.parametrize("row", RAGGED)
def test_key_past_n_in_neg_mode_fails(row):
    qkv = G.att_operands(*row, "neg", seed=7)
    assert not _att(qkv, emulate_attention(qkv, bug="phantom"))["ok"], row


@pytest.mark.parametrize("row", RAGGED + [(1, 128, 1), (1, 256, 1)])
def test_last_real_key_masked_in_peak_last_mode_fails(row):
    qkv = G.att_operands(*row, "peak_last", seed=8)
    assert not _att(qkv, emulate_attention(qkv, bug="mask_last"))["ok"], row


def test_kv_of_the_neighbouring_image_or_head_fails():
    for mode in ("rand", "peak_first", "peak_last"):
        qkv = G.att_operands(2, 65, 2, mode, seed=9)
        for swap in ("image", "head"):
            bug = qkv.clone()
            if swap == "image":
                bug[:, :, 1:] = qkv[[1, 0], :, 1:]
            else:
                bug[:, :, 1:] = qkv[:, :, 1:][:, :, :, [1, 0]]
            assert not _att(qkv, _rounded_ref(bug))["ok"], (mode, swap)


def test_o_not_rescaled_in_grow_mode_fails():
    for row in ((1, 289, 1), (1, 320, 1)):
        for mode in ("grow", "peak_last"):
            qkv = G.att_operands(*row, mode, seed=10)
            assert not _att(qkv, emulate_attention(qkv, bug="no_o_rescale"))["ok"], (row, mode)


def test_missing_log2e_in_the_scale_fails():
    for row in ((2, 17, 2), (1, 200, 1)):
        qkv = G.att_operands(*row, "rand", seed=11)
        assert not _att(qkv, emulate_attention(qkv, scale_log2e=0.125))["ok"], row


def test_unwritten_query_rows_fail():
    qkv = G.att_operands(1, 200, 2, "rand", seed=12)
    out = _rounded_ref(qkv)
    out[128:129] = float("nan")
    r = _att(qkv, out)
    assert not r["ok"] and r["nan"] == 128


# --------------------------------------------------------------------------------------------------------- LayerNorm
def _ln_two_pass_fp32(x, w, b, relu=False, stats=None):
    """The kernels' arithmetic: fp32 mean, fp32 mean of squared deviations, rsqrt(var + eps), fp32 affine, bf16 store.
    stats = (mean, var) overrides the statistics (simulated bugs)."""
    x = x.float()
    mean, var = stats if stats is not None else (None, None)
    if mean is None:
        mean = x.mean(-1, keepdim=True)
        var = (x - mean).pow(2).mean(-1, keepdim=True)
    y = (x - mean) * torch.rsqrt(var + G.LN_EPS) * w + b
    return (torch.relu(y) if relu else y).bfloat16()


def _ln_verdict(x, w, b, got, relu=False):
    ref, bound = G.ln_ref64(x, w, b, relu=relu)
    return G.ln_verdict(got, ref, bound)


def _kind_rows(op, kind):
    return op["kind"] == G.LN_ROW_KINDS.index(kind)


@pytest.mark.parametrize("D", [48, 384, 768, 1536])
def test_ln_two_pass_and_rounded_reference_pass(D):
    op = G.ln_operands(53, D, seed=D)
    for relu in (False, True):
        for x in (op["x"], op["x"].bfloat16()):
            ref, _ = G.ln_ref64(x, op["w"], op["b"], relu=relu)
            assert _ln_verdict(x, op["w"], op["b"], ref.bfloat16(), relu)["ok"]
            r = _ln_verdict(x, op["w"], op["b"], _ln_two_pass_fp32(x, op["w"], op["b"], relu), relu)
            assert r["ok"], (relu, x.dtype, r)


@pytest.mark.parametrize("D", [384, 1536])
def test_ln_one_pass_variance_fails_on_the_offset_rows(D):
    op = G.ln_operands(50, D, seed=1)
    x = op["x"]
    mean = x.mean(-1, keepdim=True)
    var = ((x * x).mean(-1, keepdim=True) - mean * mean).clamp_min(0)
    got = _ln_two_pass_fp32(x, op["w"], op["b"], stats=(mean, var))
    off = _kind_rows(op, "offset")
    assert not _ln_verdict(x[off], op["w"], op["b"], got[off])["ok"]
    rest = _kind_rows(op, "normal") | _kind_rows(op, "massive")
    assert _ln_verdict(x[rest], op["w"], op["b"], got[rest])["ok"]  # the other rows cannot tell


def test_ln_statistics_over_the_first_half_fail():
    for D in (384, 768, 1024):
        op = G.ln_operands(20, D, seed=2)
        x = op["x"]
        h = x[:, :D // 2]
        mean = h.mean(-1, keepdim=True)
        got = _ln_two_pass_fp32(x, op["w"], op["b"], stats=(mean, (h - mean).pow(2).mean(-1, keepdim=True)))
        assert not _ln_verdict(x, op["w"], op["b"], got)["ok"], D


def test_ln_eps_outside_the_square_root_fails_on_near_constant_rows():
    op = G.ln_operands(50, 768, seed=3)
    x = op["x"]
    mean = x.mean(-1, keepdim=True)
    sd = (x - mean).pow(2).mean(-1, keepdim=True).sqrt()
    got = ((x - mean) / (sd + G.LN_EPS) * op["w"] + op["b"]).bfloat16()
    nc = _kind_rows(op, "near_const")
    assert not _ln_verdict(x[nc], op["w"], op["b"], got[nc])["ok"]


def test_ln_delta2_dropped_fails():
    op = G.ln_operands(34, 1024, seed=4, deltas=True)
    xs = (op["x"] + op["d"].float()) + op["d2"].float()
    got = _ln_two_pass_fp32(op["x"] + op["d"].float(), op["w"], op["b"])
    assert not _ln_verdict(xs, op["w"], op["b"], got)["ok"]
    assert _ln_verdict(xs, op["w"], op["b"], _ln_two_pass_fp32(xs, op["w"], op["b"]))["ok"]


def test_ln_tap_that_keeps_the_cls_row_fails():
    n_tok = 17
    op = G.ln_operands(3 * n_tok, 384, seed=5)
    x = op["x"]
    full = _ln_two_pass_fp32(x, op["w2"], op["b2"])
    kept = full[:3 * (n_tok - 1)]  # the first B (n_tok - 1) rows, cls rows included
    patch = G.drop_cls_rows(x, n_tok)
    assert _ln_verdict(patch, op["w2"], op["b2"], G.drop_cls_rows(full, n_tok))["ok"]
    assert not _ln_verdict(patch, op["w2"], op["b2"], kept)["ok"]


def test_ln_row_kinds():
    op = G.ln_operands(25, 768, seed=6, deltas=True)
    x = op["x"]
    for i, kind in enumerate(G.LN_ROW_KINDS):
        rows = x[i::5]
        sd = rows.std(-1)
        if kind == "offset":
            assert (rows.mean(-1) - G.LN_OFFSET).abs().max() < 1 and (sd > 0.8).all()
        elif kind == "massive":
            assert ((rows.abs() == 500).sum(-1) >= 1).all()
        elif kind == "near_const":
            assert (sd < 2e-3).all() and (sd > 5e-4).all()
        elif kind == "const":
            xs = (rows + op["d"][i::5].float()) + op["d2"][i::5].float()
            assert (sd == 0).all() and (xs.std(-1) == 0).all()


# ------------------------------------------------------------------------------------------------------- the tables
def test_attention_table_covers_every_edge():
    rows = G.ATT_ROWS
    shapes = {(B, N, H) for B, N, H, _, _ in rows}
    assert len(shapes) == len(rows)
    residues = {N % 128 for _, N, _, _, _ in rows}
    assert {0, 1, 2, 22, 32, 33, 63, 64, 65, 90, 101, 127} <= residues
    assert any(N < 128 for _, N, _, _, _ in rows)
    tiles = {(N + 127) // 128 for _, N, _, _, _ in rows}
    assert {1, 2, 3} <= tiles and max(tiles) >= 10
    assert {6, 12, 16, 24} <= {H for _, _, H, _, _ in rows}
    # attention2.cuh query tiles that hold a single row: the second tile of a full unit, and a short unit
    def one_row_tiles(N):
        T = (N + 127) // 128
        last_rows = N - (T - 1) * 128
        return last_rows == 1, ("full" if T % 2 == 0 else "short")
    kinds = {one_row_tiles(N)[1] for _, N, _, _, _ in rows if one_row_tiles(N)[0]}
    assert kinds == {"full", "short"}
    # every shape the former attention checks launched
    former = {(1, 128, 1), (1, 200, 2), (2, 1370, 6), (1, 1370, 2), (1, 5477, 2), (4, 1370, 16), (8, 300, 16),
              (10, 128, 16), (3, 700, 16), (32, 1370, 16), (3, 1370, 16), (2, 700, 16), (1, 5477, 4)}
    assert former <= shapes
    for B, N, H, modes, pairs in rows:
        assert set(modes) <= set(G.ATT_MODES) and "rand" in modes
        if N % 128:
            assert {"neg", "peak_last", "peak_first"} <= set(modes), (B, N, H)
        if (N + 127) // 128 >= 3:
            assert {"grow", "grow8"} <= set(modes), (B, N, H)
        if B >= 32:
            assert pairs and len(pairs) >= 3
        if pairs:
            assert all(0 <= b < B and 0 <= h < H for b, h in pairs)
        assert f"attention_geo_{B}x{N}x{H}" in G.CHECKS
    assert sum("wide" in r[3] for r in rows) >= 3
    assert (1, 5477, 6) in shapes and (32, 1370, 6) in shapes
    # the former checks keep their names, now on the fp64 bound at their own shapes and inputs
    for name in ("small", "ragged", "1370", "rescale", "5477", "multiunit_1370", "multiunit_300", "multiunit_128",
                 "multiunit_rescale"):
        assert all(f"attention{i}_{name}" in G.CHECKS for i in (0, 1, 2)), name
    assert {"attention_auto_b32", "attention_impls_agree_1370", "attention_impls_agree_rescale",
            "attention_impls_agree_5477"} <= set(G.CHECKS)
    assert {(B, N, H) for B, N, H, _ in list(G.ATT_IMPL_ROWS.values()) + list(G.ATT_AGREE_ROWS.values())} <= shapes


def test_layernorm_tables_cover_every_width_and_kind():
    combos = {(D, kind) for D, _, _, kind in G.LN_ROWS}
    assert combos == {(D, k) for D in (384, 768, 1024, 1536) for k in G.LN_KINDS}
    assert len(G.LN_ROWS) == len(combos)
    assert {n for _, _, n, _ in G.LN_ROWS} == {2, 17, 1370}
    for D, B, n_tok, kind in G.LN_ROWS:
        assert (B * n_tok) % 8 and f"ln_geo_{D}_{kind}" in G.CHECKS
    assert G.LN_KINDS["tap"] == dict(delta=True, delta2=True, write_x=True, tap=True)
    assert G.LN_KINDS["last"].get("drop_cls") and not G.LN_KINDS["last"].get("write_x")
    assert set(G.CHLN_WIDTHS) == {48, 256, 384, 512, 768, 1024, 1536}
    assert {"layernorm_384", "layernorm_1024_drop", "layernorm_1536", "layernorm_delta", "layernorm_tap_fused"} <= set(G.CHECKS)
    assert {f"channel_ln_{C}" for C in (48, 256, 512, 1024, 1536)} <= set(G.CHECKS)
    for C in G.CHLN_WIDTHS:
        assert f"ln_geo_channel_{C}" in G.CHECKS
        for sms in (148, 132, 160):
            pix = 4 if C <= 256 else 2 if C <= 512 else 1
            stride = sms * 64 * pix
            P = G.chln_pixels(C, sms)
            assert P > 2 * stride and P % stride and (pix == 1 or P % pix)

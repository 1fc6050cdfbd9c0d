"""Bring-up harness: runs each kernel check in its own subprocess (a trapped kernel poisons its CUDA context) and writes
gpurun_out/gpu_check.json. `python tools/gpu_check.py` runs all; `--one NAME` runs a single check in-process."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _imports():
    import torch
    import amodal_depth_anything_b200  # noqa: F401
    from amodal_depth_anything_b200 import _lib as L, ops
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch, L, ops


def _cmp(name, got, ref, atol, rtol):
    import torch
    got, ref = got.float(), ref.float()
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = (err > tol).sum().item()
    res = {"max_abs": err.max().item(), "max_ref": ref.abs().max().item(), "bad": bad, "n": ref.numel(),
           "nan": int(torch.isnan(got).sum().item())}
    res["ok"] = bad == 0 and res["nan"] == 0
    return res


def chk_gemm(M, N, K, bn, epi_name, cg=0):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(1)
    A = (torch.randn(M, K, generator=g, device="cuda") * 0.5).bfloat16()
    Wt = (torch.randn(N, K, generator=g, device="cuda") * 0.05).bfloat16()
    bias = torch.randn(N, generator=g, device="cuda") * 0.1
    ref = A.float() @ Wt.float().t() + bias
    if epi_name == "bias":
        out = torch.zeros(M, N, dtype=torch.bfloat16, device="cuda")
        ops.gemm(A, Wt, bias=bias, out_bf16=out, ldo=N, force_bn=bn, force_cg=cg)
    elif epi_name == "gelu":
        out = torch.zeros(M, N, dtype=torch.bfloat16, device="cuda")
        ops.gemm(A, Wt, bias=bias, out_bf16=out, ldo=N, act=L.ACT_GELU, force_bn=bn, force_cg=cg)
        ref = torch.nn.functional.gelu(ref)
    elif epi_name == "resid":  # LayerScale'd branch output (bf16); the residual add itself is fused into the next LN
        gamma = torch.randn(N, generator=g, device="cuda")
        ref = gamma * ref
        out = torch.zeros(M, N, dtype=torch.bfloat16, device="cuda")
        ops.gemm(A, Wt, bias=bias, gamma=gamma, out_bf16=out, ldo=N, force_bn=bn, force_cg=cg)
    elif epi_name == "swiglu":
        Hd = N // 2
        # interleave rows in 32-chunks exactly like ada_finalize does
        idx = torch.arange(N, device="cuda")
        chunk, within = idx // 64, idx % 64
        src = torch.where(within < 32, chunk * 32 + within, Hd + chunk * 32 + within - 32)
        out = torch.zeros(M, Hd, dtype=torch.bfloat16, device="cuda")
        ops.gemm(A, Wt[src].contiguous(), epi=L.EPI_SWIGLU, bias=bias[src].contiguous(), out_bf16=out, ldo=Hd, force_bn=bn, force_cg=cg)
        x1, x2 = ref[:, :Hd], ref[:, Hd:]
        ref = torch.nn.functional.silu(x1) * x2
    torch.cuda.synchronize()
    return _cmp("gemm", out, ref, 2e-2, 1e-2)


def chk_embed():
    torch, L, ops = _imports()
    B, P, D, K = 2, 1369, 384, 1024
    g = torch.Generator(device="cuda").manual_seed(2)
    A = (torch.randn(B * P, K, generator=g, device="cuda") * 0.5).bfloat16()
    Wt = (torch.randn(D, K, generator=g, device="cuda") * 0.05).bfloat16()
    posb = torch.randn(P, D, generator=g, device="cuda")
    x = torch.full((B * (P + 1), D), 7.0, device="cuda")
    ops.gemm(A, Wt, epi=L.EPI_EMBED, aux=posb, out_f32=x, ldo=D, P=P)
    torch.cuda.synchronize()
    ref = (A.float() @ Wt.float().t()).view(B, P, D) + posb
    got = x.view(B, P + 1, D)
    r = _cmp("embed", got[:, 1:], ref, 1e-2, 1e-3)
    r["cls_untouched"] = bool((got[:, 0] == 7.0).all().item())
    r["ok"] = r["ok"] and r["cls_untouched"]
    return r


def chk_conv(B, H, W, Cin, Cout, mode, cg=0):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(3)
    x = (torch.randn(B, Cin, H, W, generator=g, device="cuda")).bfloat16()
    w = torch.randn(Cout, Cin, 3, 3, generator=g, device="cuda") * (1.0 / (3 * Cin ** 0.5))
    bias = torch.randn(Cout, generator=g, device="cuda") * 0.1
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    wp = ops.pack_conv3x3(w)
    wq = w.bfloat16().float()
    ref = torch.nn.functional.conv2d(x.float(), wq, bias, padding=1)
    if mode == "plain":
        out = torch.zeros(B, H, W, Cout, dtype=torch.bfloat16, device="cuda")
        ops.gemm(x_nhwc, wp, conv=(B, H, W, Cin), N=Cout, bias=bias, out_bf16=out, ldo=Cout, force_cg=cg)
        torch.cuda.synchronize()
        return _cmp("conv", out.permute(0, 3, 1, 2), ref, 3e-2, 1e-2)
    if mode == "rcu":  # relu act + two residuals + relu copy
        r1 = torch.randn(B, H, W, Cout, generator=g, device="cuda").bfloat16()
        r2 = torch.randn(B, H, W, Cout, generator=g, device="cuda").bfloat16()
        out = torch.zeros(B, H, W, Cout, dtype=torch.bfloat16, device="cuda")
        outr = torch.zeros_like(out)
        ops.gemm(x_nhwc, wp, conv=(B, H, W, Cin), N=Cout, bias=bias, act=L.ACT_RELU, resid1=r1, resid2=r2, out_bf16=out,
                 out_relu=outr, ldo=Cout, force_cg=cg)
        torch.cuda.synchronize()
        ref2 = torch.relu(ref).permute(0, 2, 3, 1) + r1.float() + r2.float()
        a = _cmp("conv", out, ref2, 3e-2, 1e-2)
        b = _cmp("conv", outr, torch.relu(ref2), 3e-2, 1e-2)
        a["relu_copy_ok"] = b["ok"]
        a["ok"] = a["ok"] and b["ok"]
        return a
    if mode == "chln":  # conv + channel LayerNorm + ReLU in the epilogue (dpt.py:153-159)
        lw = 1.0 + 0.2 * torch.randn(Cout, generator=g, device="cuda")
        lb = 0.3 * torch.randn(Cout, generator=g, device="cuda")
        out = torch.zeros(B, H, W, Cout, dtype=torch.bfloat16, device="cuda")
        ops.gemm(x_nhwc, wp, conv=(B, H, W, Cin), N=Cout, epi=L.EPI_BF16_CHLN, bias=bias, gamma=lw, aux=lb, out_bf16=out,
                 ldo=Cout, force_cg=cg)
        torch.cuda.synchronize()
        u = ref.mean(1, keepdim=True)
        sv = (ref - u).pow(2).mean(1, keepdim=True)
        ref2 = torch.relu((ref - u) / torch.sqrt(sv + 1e-6) * lw.view(1, -1, 1, 1) + lb.view(1, -1, 1, 1))
        return _cmp("conv_chln", out.permute(0, 3, 1, 2), ref2, 3e-2, 1e-2)
    if mode == "tail":
        assert Cout == 32
        w2 = torch.randn(32, generator=g, device="cuda") * 0.3
        b2 = torch.randn(1, generator=g, device="cuda") * 0.1
        aux = torch.cat([w2, b2]).contiguous()
        out = torch.zeros(B, H, W, dtype=torch.float32, device="cuda")
        ops.gemm(x_nhwc, wp, conv=(B, H, W, Cin), N=32, epi=L.EPI_TAIL, bias=bias, aux=aux, out_f32=out, sigmoid=1)
        torch.cuda.synchronize()
        z = (torch.relu(ref) * w2.view(1, 32, 1, 1)).sum(1) + b2
        return _cmp("tail", out, torch.sigmoid(z), 5e-3, 0)


def chk_convT(ks, Cin=96, Cout=96, B=2, H=37, W=37, pix=False):
    """pix: A operand on 8x16 pixel tiles, pixel shuffle stored through 5-D TMA boxes (Cin, Cout % 64 == 0). Held to the fp64
    bound of convT_run."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(B, Cin, H, W, generator=g, device="cuda").bfloat16()
    w = torch.randn(Cin, Cout, ks, ks, generator=g, device="cuda") * 0.1
    bias = torch.randn(Cout, generator=g, device="cuda") * 0.1
    return convT_run({"x": x.permute(0, 2, 3, 1).contiguous(), "w": w.bfloat16().float(), "b": bias}, ks, pix)


def chk_upsample(Hi, Ho, C=64):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.randn(2, Hi, Hi, C, generator=g, device="cuda").bfloat16()
    return upsample_run(x, Ho, Ho)


def chk_fused_tail(gh, gw):
    """tap GEMM at low res + gather == conv2(interp(y)) chain of dpt.py:194-195."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(17)
    B, Cm = 2, 64
    Hl, Wl, H, W = 8 * gh, 8 * gw, 14 * gh, 14 * gw
    y = torch.randn(B, Cm, Hl, Wl, generator=g, device="cuda").bfloat16()
    w2 = torch.randn(32, Cm, 3, 3, generator=g, device="cuda") * (1.0 / (3 * Cm ** 0.5))
    b2 = torch.randn(32, generator=g, device="cuda") * 0.1
    w3 = torch.randn(32, generator=g, device="cuda") * 0.3
    b3 = torch.randn(1, generator=g, device="cuda") * 0.1
    up = torch.nn.functional.interpolate(y.float(), (H, W), mode="bilinear", align_corners=True)
    z = torch.relu(torch.nn.functional.conv2d(up, w2.bfloat16().float(), b2, padding=1))
    ref = torch.sigmoid((z * w3.view(1, 32, 1, 1)).sum(1) + b3)
    wt = ops.pack_tail_taps(w2)
    ya = y.permute(0, 2, 3, 1).reshape(B * Hl * Wl, Cm).contiguous()
    V = torch.zeros(B, Hl, Wl, 288, dtype=torch.float16, device="cuda")
    ops.gemm(ya, wt, epi=L.EPI_F16, out_bf16=V, ldo=288)
    out = ops.tail_gather(V, b2, torch.cat([w3, b3]).contiguous(), H, W, True)
    torch.cuda.synchronize()
    return _cmp("fused_tail", out, ref, 5e-3, 0)


def chk_tail_mma(gh, gw, Cm=64, B=2, sigmoid=1):
    """upsample + output_conv2 on tensor cores (tail_mma_kernel) == conv2(interp(y)) chain of dpt.py:194-195."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(19)
    Hl, Wl, H, W = 8 * gh, 8 * gw, 14 * gh, 14 * gw
    y = (torch.randn(B, Cm, Hl, Wl, generator=g, device="cuda") * 1.5).half()
    w2 = torch.randn(32, Cm, 3, 3, generator=g, device="cuda") * (1.0 / (3 * Cm ** 0.5))
    b2 = torch.randn(32, generator=g, device="cuda") * 0.1
    w3 = torch.randn(32, generator=g, device="cuda") * 0.3
    b3 = torch.randn(1, generator=g, device="cuda") * 0.1
    up = torch.nn.functional.interpolate(y.float(), (H, W), mode="bilinear", align_corners=True)
    z = torch.relu(torch.nn.functional.conv2d(up, w2.half().float(), b2, padding=1))
    ref = (z * w3.view(1, 32, 1, 1)).sum(1) + b3
    ref = torch.sigmoid(ref) if sigmoid == 1 else torch.relu(ref) if sigmoid == 2 else ref
    wpk = ops.pack_tail_mma(w2)
    ya = y.permute(0, 2, 3, 1).contiguous()
    out = ops.tail_mma(ya, wpk, b2, torch.cat([w3, b3]).contiguous(), H, W, sigmoid)
    torch.cuda.synchronize()
    return _cmp("tail_mma", out, ref, 5e-3, 0)


def chk_patch_gather():
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(9)
    B, H, W = 2, 70, 98
    rgb = torch.rand(B, 3, H, W, generator=g, device="cuda")
    m = torch.rand(B, 1, H, W, generator=g, device="cuda") * 2 - 1
    o = torch.rand(B, 1, H, W, generator=g, device="cuda") * 2 - 1
    return patch_gather_run(rgb, [m, o], 1024)


def chk_conv_s2(B, H, W, Cin, Cout):
    """3x3, stride 2, pad 1 (resize_layers[3], dpt.py:102-107) as an implicit GEMM: the tensor map walks the input with
    element stride 2; odd and even input sizes, ragged output tiles."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(10)
    x = torch.randn(B, Cin, H, W, generator=g, device="cuda").bfloat16()
    w = torch.randn(Cout, Cin, 3, 3, generator=g, device="cuda") * (1.0 / (3 * Cin ** 0.5))
    bias = torch.randn(Cout, generator=g, device="cuda") * 0.1
    ref = torch.nn.functional.conv2d(x.float(), w.bfloat16().float(), bias, stride=2, padding=1)
    Ho, Wo = ref.shape[2:]
    out = torch.zeros(B, Ho, Wo, Cout, dtype=torch.bfloat16, device="cuda")
    ops.gemm(x.permute(0, 2, 3, 1).contiguous(), ops.pack_conv3x3(w), conv=(B, H, W, Cin), N=Cout, bias=bias, out_bf16=out,
             ldo=Cout, conv_stride=2)
    torch.cuda.synchronize()
    return _cmp("conv_s2", out.permute(0, 3, 1, 2), ref, 3e-2, 1e-2)


def chk_gemm_resid_f32(M, N, K, gamma=True, cg=0):
    """EPI_RESID_F32: x (fp32, in place) += gamma * (A W^T + b) -- the residual update of block.py:105-106."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(23)
    A = (torch.randn(M, K, generator=g, device="cuda") * 0.5).bfloat16()
    Wt = (torch.randn(N, K, generator=g, device="cuda") * 0.05).bfloat16()
    bias = torch.randn(N, generator=g, device="cuda") * 0.1
    gam = (1.0 + 0.1 * torch.randn(N, generator=g, device="cuda")) if gamma else None
    x = torch.randn(M, N, generator=g, device="cuda") * 2
    ref = A.float() @ Wt.float().t() + bias
    if gamma:
        ref = ref * gam
    ref = x + ref
    out = x.clone()
    ops.gemm(A, Wt, epi=L.EPI_RESID_F32, bias=bias, gamma=gam, out_f32=out, ldo=N, force_cg=cg)
    torch.cuda.synchronize()
    return _cmp("resid_f32", out, ref, 2e-3, 2e-3)


# ---- implicit-GEMM conv: every pixel-tile shape and every epilogue the model launches, against an fp64 reference
#
# Error model. The kernels multiply bf16 operands exactly and accumulate in fp32, so an output before its final rounding is
# off the fp64 result by less than 2^-16 * S, S = conv(|x|, |w|) + |b| (+ |r1| + |r2|): fp32 accumulation over K <= 9 * 1536
# terms with room to spare. The output rounding adds at most one unit roundoff of the stored type: 2^-8 |ref| for bf16,
# 2^-11 for fp16 (held to 2^-10), 2^-24 for fp32 (held to 2^-22: the epilogue rounds twice). The channel-LayerNorm
# epilogue scales a pre-normalisation error by |LN weight| * rstd; its mean carries the channel average of the errors.
REL_BF16, REL_F16, REL_F32, REL_ACC = 2.0 ** -8, 2.0 ** -10, 2.0 ** -22, 2.0 ** -16

# One row per pixel-tile geometry (lw, lh, lb, pair) = 2^lw x 2^lh pixels of 2^lb images, CTA pairs side by side in x: all
# 25 shapes with lw + lh + lb = 7, 1 <= lw <= 5, single and paired. (B, H, W) is a small map for which pick_tile_geo
# (ada_conv_tile_shape) picks that shape, ragged in x, y and the batch wherever the shape has more than one pixel / image in
# that direction; for the stride-2 variant it is the OUTPUT size. Cin 48 / 96 leave a ragged 64-channel chunk that the
# packed weights zero-pad; N 48 / 96 are ragged N tiles whose stores are clipped. ada_op_gemm pairs CTAs on force_cg=2 only
# for BN = 256 (or BN = 128 with the plain bf16 epilogue), so every paired row has N = 256, for which pick_bn picks 256.
#   (lw, lh, lb, pair,  B,  H,  W, Cin,   N)
CONV_GEO_ROWS = [
    (1, 0, 6, 1, 33,  1,  1,  48,  48),
    (1, 1, 5, 1, 25,  5,  5,  64,  96),
    (1, 2, 4, 1, 25, 11,  5,  96, 128),
    (1, 3, 3, 1, 13, 21,  5, 256, 256),
    (1, 4, 2, 1,  7, 41,  5,  64,  48),
    (1, 5, 1, 1,  5, 25,  5,  96,  96),
    (1, 6, 0, 1,  3, 41,  9, 256, 128),
    (2, 0, 5, 1, 25,  3,  9,  48, 256),
    (2, 1, 4, 1, 37,  5,  3,  96,  48),
    (2, 2, 3, 1, 13, 11, 11, 256,  96),
    (2, 3, 2, 1,  7, 21, 11,  48, 128),
    (2, 4, 1, 1,  5, 41, 11,  64, 256),
    (2, 5, 0, 1,  3, 41,  3, 256,  48),
    (3, 0, 4, 1, 25,  3, 21,  48,  96),
    (3, 1, 3, 1, 21,  5, 21,  64, 128),
    (3, 2, 2, 1,  7, 11, 21,  96, 256),
    (3, 3, 1, 1,  5, 21, 21,  48,  48),
    (3, 4, 0, 1,  2, 25, 23,  64,  96),
    (4, 0, 3, 1, 13,  3, 41,  96, 128),
    (4, 1, 2, 1, 10,  5, 41, 256, 256),
    (4, 2, 1, 1,  5,  9, 41,  64,  48),
    (4, 3, 0, 1,  2, 15, 29,  96,  96),
    (5, 0, 2, 1,  7,  3, 49, 256, 128),
    (5, 1, 1, 1,  5,  5, 49,  48, 256),
    (5, 2, 0, 1,  2, 11, 49,  96,  48),
    (1, 0, 6, 2, 33,  1,  1,  48, 256),
    (1, 1, 5, 2, 25,  5,  9,  64, 256),
    (1, 2, 4, 2, 25, 11,  9,  96, 256),
    (1, 3, 3, 2, 13, 21,  9, 256, 256),
    (1, 4, 2, 2,  7, 41,  9,  48, 256),
    (1, 5, 1, 2,  5, 25,  9,  64, 256),
    (1, 6, 0, 2,  3, 41, 17,  96, 256),
    (2, 0, 5, 2, 25,  3, 17, 256, 256),
    (2, 1, 4, 2, 37,  5,  5,  48, 256),
    (2, 2, 3, 2, 13, 11,  5,  64, 256),
    (2, 3, 2, 2,  7, 21,  5,  96, 256),
    (2, 4, 1, 2,  5, 33,  5, 256, 256),
    (2, 5, 0, 2,  3, 41,  5,  48, 256),
    (3, 0, 4, 2, 25,  3,  9,  64, 256),
    (3, 1, 3, 2, 19,  5,  9,  96, 256),
    (3, 2, 2, 2,  7, 11,  9, 256, 256),
    (3, 3, 1, 2,  5, 17,  9,  48, 256),
    (3, 4, 0, 2,  2, 25, 45,  64, 256),
    (4, 0, 3, 2, 13,  3, 21,  96, 256),
    (4, 1, 2, 2, 10,  5, 17, 256, 256),
    (4, 2, 1, 2,  5,  9, 17,  48, 256),
    (4, 3, 0, 2,  2, 15, 57,  64, 256),
    (5, 0, 2, 2,  7,  3, 41,  96, 256),
    (5, 1, 1, 2,  5,  5, 33, 256, 256),
    (5, 2, 0, 2,  3,  9, 33,  48, 256),
]

# The conv epilogues of the model's forward (csrc/ada_api.cu), each checked at every row:
CONV_VARIANTS = {
    "a_bias": dict(bias=True),                                # input_projection conv with C > 256; stride-1 plain conv
    "b_relu_copy": dict(bias=False, relu_copy=True),          # layer_rn: no bias, keeps x and relu(x)
    "c_relu": dict(bias=True, act="relu"),                    # RCU conv1
    "d_resid2_relu_copy": dict(bias=True, resid=2, relu_copy=True),  # RCU1 conv2: + layer_rn + path, and its ReLU
    "e_resid1": dict(bias=True, resid=1),                     # RCU2 conv2
    "f_chln": dict(bias=True, epi="chln"),                    # input_projection with C <= 256: conv + channel LN + ReLU
    "g_f16": dict(bias=True, epi="f16"),                      # output_conv1, stored as fp16 for the tail
    "h_s2_bias": dict(bias=True, stride=2),                   # resize_layers[3]: stride 2
}


def conv_geo_operands(B, H, W, Cin, N, seed, s2_odd=True, device="cpu", variants=tuple(CONV_VARIANTS)):
    """Operands of one table row: x NHWC [B, H, W, Cin] and xs (input of the stride-2 variant, (2H - 1) x (2W - 1) if
    s2_odd else 2H x 2W) in bf16, weights [N, Cin, 3, 3] rounded to bf16 (held as fp32, so packing is exact), fp32 bias,
    bf16 residuals [B, H, W, N], fp32 LayerNorm weight / bias. Maps no listed variant reads are left out."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    Hs, Ws = (2 * H - 1, 2 * W - 1) if s2_odd else (2 * H, 2 * W)
    vs = [CONV_VARIANTS[v] for v in variants]
    rnd = lambda *s: torch.randn(*s, generator=g, device=device)  # noqa: E731
    op = {
        "w": (rnd(N, Cin, 3, 3) / (3 * Cin ** 0.5)).bfloat16().float(),
        "b": rnd(N) * 0.1,
        "lnw": 1.0 + 0.2 * rnd(N),
        "lnb": 0.3 * rnd(N),
    }
    if any(v.get("stride", 1) == 1 for v in vs):
        op["x"] = rnd(B, H, W, Cin).bfloat16()
    if any(v.get("stride", 1) == 2 for v in vs):
        op["xs"] = rnd(B, Hs, Ws, Cin).bfloat16()
    for k in range(max(v.get("resid", 0) for v in vs)):
        op[("r1", "r2")[k]] = rnd(B, H, W, N).bfloat16()
    return op


def conv_ref64(op, variant, imgs=None):
    """fp64 reference of one epilogue variant on the operands of conv_geo_operands (any device): (ref, bound, relu_copy)
    as [b, H, W, N] fp64 over the images `imgs` (all if None); bound is the per-element error bound of the error model
    above, relu_copy whether the variant also stores relu(out)."""
    import torch
    F = torch.nn.functional
    v = CONV_VARIANTS[variant]
    stride = v.get("stride", 1)
    x = op["xs"] if stride == 2 else op["x"]
    sel = (lambda t: t) if imgs is None else (lambda t: t[list(imgs)])
    xd = sel(x).double().permute(0, 3, 1, 2)
    wd = op["w"].double()
    acc = F.conv2d(xd, wd, stride=stride, padding=1).permute(0, 2, 3, 1)
    S = F.conv2d(xd.abs(), wd.abs(), stride=stride, padding=1).permute(0, 2, 3, 1)
    if v.get("bias"):
        acc = acc + op["b"].double()
        S = S + op["b"].double().abs()
    if v.get("act") == "relu":
        acc = torch.relu(acc)
    for k in range(v.get("resid", 0)):
        r = sel(op[("r1", "r2")[k]]).double()
        acc = acc + r
        S = S + r.abs()
    if v.get("epi") == "chln":
        mean = acc.mean(-1, keepdim=True)
        rstd = 1.0 / torch.sqrt((acc - mean).pow(2).mean(-1, keepdim=True) + 1e-6)
        lnw = op["lnw"].double()
        ref = torch.relu((acc - mean) * rstd * lnw + op["lnb"].double())
        bound = REL_BF16 * ref.abs() + REL_ACC * (S + S.mean(-1, keepdim=True)) * lnw.abs() * rstd
        return ref, bound, False
    rel = REL_F16 if v.get("epi") == "f16" else REL_BF16
    return acc, rel * acc.abs() + REL_ACC * S, bool(v.get("relu_copy"))


def relu_copy_of(out):
    """What the ReLU copy must hold, bit for bit: clamp_min(out, 0), with -0 stored as +0."""
    return (out.float().clamp_min(0) + 0.0).to(out.dtype)


def err_over_bound(got, ref, bound):
    """Largest |got - ref| / bound (inf if got has a NaN or an infinity)."""
    import torch
    err = (got.to(ref.device).double() - ref).abs()
    q = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(q.nan_to_num(float("inf")).max().item())


def conv_verdict(got, got_relu, ref, bound, relu_copy):
    """Judges one variant's output(s) (already restricted to the reference's images): within the bound everywhere, no NaN
    (an unwritten pixel of the NaN-filled buffer), and the ReLU copy exactly relu_copy_of(out)."""
    import torch
    r = {"err_bound": err_over_bound(got, ref, bound), "nan": int(torch.isnan(got.float()).sum().item())}
    r["ok"] = r["err_bound"] <= 1.0 and r["nan"] == 0
    if relu_copy:
        r["relu_copy_exact"] = bool(torch.equal(got_relu.view(torch.int16), relu_copy_of(got).view(torch.int16)))
        r["ok"] = r["ok"] and r["relu_copy_exact"]
    return r


class Guarded:
    """A tensor inside a larger 1-D buffer: `guard` elements (a multiple of 64, so the tensor keeps TMA's 16-byte alignment)
    before and after it. fill=None writes a fixed canary pattern into the guards (outputs: a store past the tensor changes
    it); a float fill fills the guards with it (inputs: NaN, so a read past the tensor reaches the output)."""

    def __init__(self, shape, dtype, device, guard, fill=None, body=float("nan")):
        import torch
        n = 1
        for s in shape:
            n *= s
        self.guard, self.n = guard, n
        self.buf = torch.empty(n + 2 * guard, dtype=dtype, device=device)
        if fill is None:
            g = torch.Generator(device=device).manual_seed(1234)
            self.canary = torch.randn(2 * guard, generator=g, device=device).to(dtype)
            self.buf[:guard] = self.canary[:guard]
            self.buf[guard + n:] = self.canary[guard:]
        else:
            self.canary = None
            self.buf.fill_(fill)
        self.t = self.buf[guard:guard + n].view(shape)
        self.t.fill_(body)

    def canaries_intact(self):
        import torch
        if self.canary is None:
            return True
        got = torch.cat([self.buf[:self.guard], self.buf[self.guard + self.n:]])
        return bool(torch.equal(got.view(torch.int16), self.canary.view(torch.int16)))


def _guard_for(per_image):
    return (per_image + 64 + 63) // 64 * 64  # one whole image (a store / load one image off) and then some


def _conv_launch(L, ops, v, x, wp, op, out, out_relu, B, Hin, Win, Cin, N, cg, r1=None, r2=None):
    vv = CONV_VARIANTS[v]
    epi = {"chln": L.EPI_BF16_CHLN, "f16": L.EPI_F16}.get(vv.get("epi"), L.EPI_BF16)
    ops.gemm(x, wp, conv=(B, Hin, Win, Cin), N=N, epi=epi, act=L.ACT_RELU if vv.get("act") == "relu" else L.ACT_NONE,
             bias=op["b"] if vv.get("bias") else None,
             gamma=op["lnw"] if vv.get("epi") == "chln" else None, aux=op["lnb"] if vv.get("epi") == "chln" else None,
             resid1=r1 if vv.get("resid", 0) >= 1 else None, resid2=r2 if vv.get("resid", 0) >= 2 else None,
             out_bf16=out, out_relu=out_relu, ldo=N, force_cg=cg, conv_stride=vv.get("stride", 1))


def conv_tile_shape(B, H, W, pair):
    import ctypes
    sys.path.insert(0, ROOT)
    from amodal_depth_anything_b200 import _lib as L
    out = (ctypes.c_int64 * 4)()
    L.check(L.load().ada_conv_tile_shape(B, H, W, pair, out))
    return tuple(int(v) for v in out[:3])


def chk_conv_geo(lw, lh, lb, pair, B, H, W, Cin, N, seed=0):
    """One row of CONV_GEO_ROWS: the picker chooses the row's tile shape, and every epilogue variant passes
    conv_geo_run with the row's pairing forced."""
    res = conv_geo_run(B, H, W, Cin, N, pair, seed=seed)
    res["shape"] = list(conv_tile_shape(B, H, W, pair))
    res["ok"] = res["ok"] and res["shape"] == [lw, lh, lb]
    return res


def chk_conv_geo_bench(B, H, W, variants, ref_imgs):
    """A batch-32 map of the ViT-L head (F = 256) with the launcher's own pairing, as the model runs it: more tiles than
    SMs, so the persistent loop and both accumulator stages are exercised; fp64 on a few images, bit-equality with
    one-image launches on all of them."""
    res = conv_geo_run(B, H, W, 256, 256, 0, variants=variants, ref_imgs=ref_imgs, seed=8)  # even: odd stride-2 input
    res["shapes"] = [list(conv_tile_shape(B, H, W, p)) for p in (1, 2)]
    return res


def conv_geo_run(B, H, W, Cin, N, cg, variants=tuple(CONV_VARIANTS), ref_imgs=None, seed=0):
    """Every listed epilogue variant at one (B, H, W, Cin, N), force_cg=cg (0: the launcher's choice). Per variant: the
    fp64 bound on the images `ref_imgs` (all if None), no unwritten pixel (outputs start as NaN), canaries around every
    output intact, inputs and residuals inside NaN guards (conv padding must come from TMA's out-of-bounds zero fill), the
    ReLU copy exact; every image bit-equal to a one-image launch (another tile shape); with cg=2 bit-equal to single-CTA
    tiles."""
    torch, L, ops = _imports()
    dev = "cuda"
    res = {"err_bound": 0.0, "variants": {}}
    ok = True
    t0 = time.time()
    op = conv_geo_operands(B, H, W, Cin, N, seed, s2_odd=(seed % 2 == 0), device=dev, variants=variants)
    imgs = list(range(B)) if ref_imgs is None else list(ref_imgs)
    # fp64 reference on the host for the small rows, on the device for the large ones
    ref_dev = dev if 18 * len(imgs) * H * W * Cin * N > 3e8 else "cpu"
    ref_op = {k: (t[imgs] if k in ("x", "xs", "r1", "r2") else t).to(ref_dev) for k, t in op.items()}
    wp = ops.pack_conv3x3(op["w"])
    # inputs and residuals inside NaN guards, one image on either side
    gin = {}
    for k in ("x", "xs", "r1", "r2"):
        if k in op:
            t = op[k]
            gin[k] = Guarded(tuple(t.shape), torch.bfloat16, dev, _guard_for(t[0].numel()), fill=float("nan"))
            gin[k].t.copy_(t)
    res_t = lambda k, i=None: None if k not in gin else gin[k].t if i is None else gin[k].t[i:i + 1]  # noqa: E731
    for v in variants:
        vv = CONV_VARIANTS[v]
        s2 = vv.get("stride", 1) == 2
        x = gin["xs" if s2 else "x"].t
        Hin, Win = x.shape[1:3]
        dt = torch.float16 if vv.get("epi") == "f16" else torch.bfloat16
        guard = _guard_for(H * W * N)

        def launch(xin, nb, r1, r2, c):
            o = Guarded((nb, H, W, N), dt, dev, guard)
            orl = Guarded((nb, H, W, N), dt, dev, guard) if vv.get("relu_copy") else None
            _conv_launch(L, ops, v, xin, wp, op, o.t, orl.t if orl else None, nb, Hin, Win, Cin, N, c, r1, r2)
            return o, orl

        out, outr = launch(x, B, res_t("r1"), res_t("r2"), cg)
        torch.cuda.synchronize()
        ref, bound, relu_copy = conv_ref64(ref_op, v)
        sel = torch.tensor(imgs, device=dev)
        r = conv_verdict(out.t[sel], outr.t[sel] if outr else None, ref, bound, relu_copy)
        if relu_copy:  # the ReLU copy of the images without an fp64 comparison too
            r["relu_copy_exact"] = r["relu_copy_exact"] and bool(
                torch.equal(outr.t.view(torch.int16), relu_copy_of(out.t).view(torch.int16)))
        r["canaries_ok"] = out.canaries_intact() and (outr is None or outr.canaries_intact())
        r["nan_all"] = int(torch.isnan(out.t.float()).sum().item())
        # batch invariance: each image alone (B = 1 picks another tile shape) gives the same bits
        same = True
        for i in range(B):
            o1, o1r = launch(x[i:i + 1], 1, res_t("r1", i), res_t("r2", i), 0)
            same = same and torch.equal(o1.t.view(torch.int16), out.t[i:i + 1].view(torch.int16)) and o1.canaries_intact()
            if o1r is not None:
                same = same and torch.equal(o1r.t.view(torch.int16), outr.t[i:i + 1].view(torch.int16))
        r["batch_invariant"] = bool(same)
        if cg == 2:  # the same launch on single-CTA tiles
            o2, o2r = launch(x, B, res_t("r1"), res_t("r2"), 1)
            r["pair_invariant"] = bool(torch.equal(o2.t.view(torch.int16), out.t.view(torch.int16)) and
                                       (o2r is None or torch.equal(o2r.t.view(torch.int16), outr.t.view(torch.int16))))
        else:
            r["pair_invariant"] = True
        torch.cuda.synchronize()
        r["ok"] = r["ok"] and r["canaries_ok"] and r["nan_all"] == 0 and r["batch_invariant"] and r["pair_invariant"]
        res["variants"][v] = r
        res["err_bound"] = max(res["err_bound"], r["err_bound"])
        ok = ok and r["ok"]
    res["inputs_untouched"] = all(bool(torch.equal(gin[k].t.view(torch.int16), op[k].view(torch.int16))) for k in gin)
    res["ok"] = bool(ok and res["inputs_untouched"])
    res["run_sec"] = round(time.time() - t0, 2)
    return res


# linear GEMM: the built (BN, CG) instantiations of each epilogue (ADA_GEMM_CASE in csrc/ada_api.cu)
GEMM_TILES = {
    "bf16": [(64, 1), (128, 1), (128, 2), (256, 1), (256, 2)],
    "gelu": [(64, 1), (128, 1), (128, 2), (256, 1), (256, 2)],
    "gamma": [(64, 1), (128, 1), (128, 2), (256, 1), (256, 2)],
    "resid_f32": [(64, 1), (128, 1), (256, 1), (256, 2)],
    "swiglu": [(128, 1), (256, 1), (256, 2)],
    "f16": [(64, 1), (128, 1), (256, 1), (256, 2)],
    "embed": [(64, 1), (128, 1), (256, 1), (256, 2)],
}


def chk_gemm_tiles(kind, M=1110, N=384, K=520, P=370):
    """The tile of a linear GEMM (BN, CG; the small-launch cost model in launch_gemm picks among them) never changes a
    bit: every built instantiation of the epilogue, and the launcher's own choice, give the same output. M is ragged
    against 128 / 256 rows, N against 256 columns, K against 64. bf16 / gamma / fp32-residual / fp16 / embed outputs are
    held to the fp64 bound; GELU and SwiGLU (tanh.approx) keep the tolerance of chk_gemm."""
    torch, L, ops = _imports()
    g = torch.Generator().manual_seed(31)
    A = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    Wt = (torch.randn(N, K, generator=g) * 0.05).bfloat16()
    bias = torch.randn(N, generator=g) * 0.1
    gam = 1.0 + 0.1 * torch.randn(N, generator=g)
    x0 = torch.randn(M, N, generator=g) * 2
    posb = torch.randn(P, N, generator=g)
    acc = A.double() @ Wt.double().t()
    S = A.double().abs() @ Wt.double().abs().t()
    Ad, Wd = A.cuda(), Wt.cuda()
    bd, gd, pd = bias.cuda(), gam.cuda(), posb.cuda()
    rel, ref, tol = REL_BF16, acc + bias.double(), None
    S = S + bias.double().abs()
    if kind == "gamma":
        ref, S = ref * gam.double(), S * gam.double().abs()
    elif kind == "resid_f32":
        ref, S, rel = ref * gam.double() + x0.double(), S * gam.double().abs() + x0.double().abs(), REL_F32
    elif kind == "f16":
        rel = REL_F16
    elif kind == "embed":
        ref = (acc.view(M // P, P, N) + posb.double()).view(M, N)
        S, rel = (A.double().abs() @ Wt.double().abs().t()).view(M // P, P, N).add(posb.double().abs()).view(M, N), REL_F32
    elif kind == "gelu":
        ref, tol = torch.nn.functional.gelu(ref), (2e-2, 1e-2)
    elif kind == "swiglu":
        ref, tol = torch.nn.functional.silu(ref[:, :N // 2]) * ref[:, N // 2:], (2e-2, 1e-2)
    idx = torch.arange(N)
    src = torch.where(idx % 64 < 32, idx // 64 * 32 + idx % 64, N // 2 + idx // 64 * 32 + idx % 64 - 32)  # as ada_finalize

    def run(bn, cg):
        if kind == "resid_f32":
            out = x0.clone().cuda()
            ops.gemm(Ad, Wd, epi=L.EPI_RESID_F32, bias=bd, gamma=gd, out_f32=out, ldo=N, force_bn=bn, force_cg=cg)
        elif kind == "embed":
            out = torch.full((M // P, P + 1, N), 7.0, device="cuda")
            ops.gemm(Ad, Wd, epi=L.EPI_EMBED, aux=pd, out_f32=out, ldo=N, P=P, force_bn=bn, force_cg=cg)
        elif kind == "swiglu":
            out = torch.full((M, N // 2), float("nan"), dtype=torch.bfloat16, device="cuda")
            ops.gemm(Ad, Wd[src.cuda()].contiguous(), epi=L.EPI_SWIGLU, bias=bd[src.cuda()].contiguous(), out_bf16=out,
                     ldo=N // 2, force_bn=bn, force_cg=cg)
        else:
            dt = torch.float16 if kind == "f16" else torch.bfloat16
            out = torch.full((M, N), float("nan"), dtype=dt, device="cuda")
            ops.gemm(Ad, Wd, epi=L.EPI_F16 if kind == "f16" else L.EPI_BF16, act=L.ACT_GELU if kind == "gelu" else L.ACT_NONE,
                     bias=bd, gamma=gd if kind == "gamma" else None, out_bf16=out, ldo=N, force_bn=bn, force_cg=cg)
        torch.cuda.synchronize()
        return out

    first = run(*GEMM_TILES[kind][0])
    same = {}
    for bn, cg in GEMM_TILES[kind][1:] + [(0, 0)]:
        o = run(bn, cg)
        same[f"{bn}x{cg}" if bn else "auto"] = bool(torch.equal(o.view(torch.int32 if o.dtype == torch.float32 else torch.int16),
                                                               first.view(torch.int32 if o.dtype == torch.float32 else torch.int16)))
    got = first.cpu()
    r = {"same_bits": same}
    if kind == "embed":
        r["cls_untouched"] = bool((got[:, 0] == 7.0).all().item())
        got = got[:, 1:].reshape(M, N)
    if tol is None:
        r["err_bound"] = err_over_bound(got, ref, REL_ACC * S + rel * ref.abs())
        r["ok"] = r["err_bound"] <= 1.0
    else:
        c = _cmp(kind, got, ref.float(), *tol)
        r.update(max_abs=c["max_abs"], bad=c["bad"])
        r["ok"] = c["ok"]
    r["nan"] = int(torch.isnan(got.float()).sum().item())
    r["ok"] = bool(r["ok"] and r["nan"] == 0 and all(same.values()) and r.get("cls_untouched", True))
    return r


# ---- attention: every ragged sequence length and head count the model can launch, against an fp64 reference
#
# Error model, per query row i of one (image, head), with a_ij = softmax_j(s_ij / 8), ref_i = sum_j a_ij v_j and
# R_i = sum_j a_ij |v_j| (fp64 from the bf16 inputs):
#   2^-8 |ref_i|                     the bf16 output rounding;
#   2^-8 R_i                         P is stored as bf16 (relative error <= 2^-8 per key) while the row sum adds the
#                                    unrounded fp32 p, so the output is sum_j a_ij (1 + d_j) v_j with |d_j| <= 2^-8;
#   2 EXP_EPS (R_i + |ref_i|)        the exponential (FMA-pipe polynomial or MUFU ex2) moves every weight by a relative
#                                    error <= EXP_EPS; normalising by the row sum of the same p doubles it, and a common
#                                    weight change cancels against ref_i, hence |v_j - ref_i| <= |v_j| + |ref_i|;
#   N 2^-24 (R_i + |ref_i|)          the fp32 row sum and the fp32 P V accumulation over N keys;
#   2 sum_j a_ij e_ij (|v_j| + |ref_i|), e_ij = 2^-16 (|q_i| . |k_j|) / 8
#                                    the fp32 score accumulation (64 exact bf16 products) moves p_j by a relative e_ij;
#                                    the factor 2 covers exp(e) - 1 <= 2 e for e <= 1.
# The fp32 rounding of x = s c - m c (c = 0.125 log2 e) adds at most 2^-23 |x| ln 2 per weight; weighted by a_ij that
# is below 2^-18 for any row, inside the slack EXP_EPS keeps over the measured polynomial error.
# EXP_EPS: the FMA-pipe exp2 polynomial (ptx.cuh exp2_fma2) has a measured maximum relative error of 7.5e-5 (2^-13.7) over
# [-125, 8]; MUFU ex2.approx is good to ~2^-22. tests/test_encoder_check_cpu.py re-measures it and the P-rounding term.
EXP_EPS = 2.0 ** -13
ATT_MODES = ("rand", "neg", "peak_last", "peak_first", "grow", "grow8", "wide")
_ATT_BASE = ("rand", "neg", "peak_last", "peak_first")
_ATT_GROW = _ATT_BASE + ("grow", "grow8")

# (B, N, heads, modes, ref_pairs). Any N is a real launch (a 14 x 14 (N - 1) image has N tokens), so the table walks the
# residues N mod 128 at the edges of both kernels: N < 128 (a single ragged tile; 64 = the boundary of the two 64-column
# halves of a score row in attention.cuh), r = 1 (the second-half thread of every row has no key), 32 / 33 and 64 / 65
# (attention2.cuh skips 32-key chunks entirely past N), 127. N = 129 / 257 / 1409 put a single row in a query tile of
# attention2.cuh (the second tile of a full unit / a short unit). Heads 6 / 12 / 16 / 24 = ViT-S / B / L / G.
# ref_pairs: (image, head) pairs held to the fp64 bound on the largest rows; bit-equality with the one-image launches
# and across the kernels covers the others.
ATT_ROWS = [
    (3, 2, 6, _ATT_BASE, None),
    (2, 17, 24, _ATT_BASE, None),           # ViT-G at 56 x 56
    (2, 33, 12, _ATT_BASE, None),
    (2, 64, 6, _ATT_BASE + ("wide",), None),  # the 126 x 98 golden
    (2, 65, 16, _ATT_BASE, None),
    (1, 128, 1, _ATT_BASE, None),
    (2, 128, 12, _ATT_BASE, None),
    (10, 128, 16, _ATT_BASE, None),         # several work units per persistent CTA
    (2, 129, 6, _ATT_BASE, None),
    (1, 160, 24, _ATT_BASE, None),
    (2, 191, 16, _ATT_BASE, None),
    (1, 200, 2, _ATT_BASE, None),
    (1, 257, 12, _ATT_GROW, None),
    (1, 289, 6, _ATT_GROW, None),
    (8, 300, 16, _ATT_GROW, None),          # full and short units interleaved
    (2, 320, 16, _ATT_GROW + ("wide",), None),
    (1, 383, 24, _ATT_GROW, None),
    (2, 700, 16, _ATT_GROW, None),
    (3, 700, 16, _ATT_GROW, None),
    (1, 1370, 2, _ATT_GROW, None),
    (2, 1370, 6, _ATT_GROW + ("wide",), None),  # ViT-S at 518 x 518
    (3, 1370, 16, _ATT_GROW, None),
    (4, 1370, 16, _ATT_GROW, None),
    (1, 1409, 12, _ATT_GROW, None),
    (1, 1814, 6, _ATT_GROW + ("wide",), None),  # 518 x 686
    (1, 5477, 2, _ATT_GROW, None),
    (1, 5477, 4, _ATT_GROW, ((0, 0), (0, 3))),
    (1, 5477, 6, _ATT_GROW, ((0, 0), (0, 5))),
    (32, 1370, 6, _ATT_GROW, ((0, 0), (13, 2), (31, 5))),
    (32, 1370, 16, _ATT_GROW, ((0, 0), (16, 7), (31, 15))),  # the benchmark's ViT-L launch
]


def att_operands(B, N, heads, mode, seed, device="cpu"):
    """qkv [B, N, 3, heads, 64] bf16 of one input mode (v is 1.5 N(0, 1) throughout):
    rand        q, k ~ 1.5 N(0, 1);
    neg         q >= 0, k <= 0 elementwise: every real score is clearly negative, so a key past N that escapes the mask
                (score 0, v 0) takes most of the weight;
    peak_last / peak_first   one key (N - 1, inside the ragged tile / 0) leads every row by ~24 logits (q[0] = 4,
                k[0] = 48 there and 0 elsewhere): masking a real key, or mixing up keys, changes the output completely;
    grow        key norms ramp 1 -> 8 over the KV tiles: row maxima jump by more than 2^8 between tiles (O rescale);
    grow8       the keys of KV tile t carry k[0] = 10.375 t with q[0] = 4: every tile's maximum is ~7.5 (log2 units)
                above the previous one, just under the 2^8 rescale threshold, so p reaches ~2^7.5 without a rescale
                on every other tile;
    wide        q, k ~ 7.5 N(0, 1): scores span about +-200 logits, most p underflow, and the score error dominates."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    qkv = torch.randn(B, N, 3, heads, 64, generator=g, device=device) * 1.5
    q, k = qkv[:, :, 0], qkv[:, :, 1]
    if mode == "neg":
        q.abs_()
        k.abs_().neg_()
    elif mode in ("peak_last", "peak_first"):
        q[..., 1:] *= 0.5
        q[..., 0] = 4.0
        k[..., 0] = 0.0
        k[:, N - 1 if mode == "peak_last" else 0, :, 0] = 48.0
    elif mode == "grow":
        ramp = 1.0 + 7.0 * (torch.arange(N, device=device) // 128).float() / max((N - 1) // 128, 1)
        k *= ramp.view(1, N, 1, 1)
    elif mode == "grow8":
        q[..., 1:] *= 0.02
        q[..., 0] = 4.0
        k[..., 0] = 10.375 * (torch.arange(N, device=device) // 128).float().view(1, N, 1)
    elif mode == "wide":
        q *= 5.0
        k *= 5.0
    else:
        assert mode == "rand", mode
    return qkv.bfloat16()


def att_ref64(qkv, pairs=None, device="cpu", chunk=1024):
    """fp64 reference and per-element bound (error model above) of attention on qkv [B, N, 3, heads, 64] for the
    (image, head) pairs `pairs` (all if None): (ref, bound), each [len(pairs), N, 64] fp64 on `device`."""
    import torch
    B, N, _, H, _ = qkv.shape
    pairs = [(b, h) for b in range(B) for h in range(H)] if pairs is None else list(pairs)
    refs, bounds = [], []
    for b, h in pairs:
        q, k, v = (qkv[b, :, i, h].to(device).double() for i in range(3))
        ka, va = k.abs(), v.abs()
        ref = torch.empty(N, 64, dtype=torch.float64, device=device)
        bound = torch.empty_like(ref)
        for i0 in range(0, N, chunk):
            qc = q[i0:i0 + chunk]
            a = torch.softmax((qc @ k.t()) * 0.125, dim=-1)
            r = a @ v
            R = a @ va
            ae = a * (qc.abs() @ ka.t()) * (REL_ACC / 8)
            ra = r.abs()
            ref[i0:i0 + chunk] = r
            bound[i0:i0 + chunk] = (REL_BF16 * (ra + R) + (2 * EXP_EPS + N * 2.0 ** -24) * (R + ra) +
                                    2 * (ae @ va + ae.sum(-1, keepdim=True) * ra))
        refs.append(ref)
        bounds.append(bound)
    return torch.stack(refs), torch.stack(bounds)


def att_select(out, B, N, heads, pairs):
    """The (image, head) pairs of an attention output [B * N, heads * 64] as [len(pairs), N, 64]."""
    import torch
    o = out.view(B, N, heads, 64)
    return torch.stack([o[b, :, h] for b, h in pairs])


def att_verdict(got, ref, bound):
    """got / ref / bound [pairs, N, 64]: within the bound everywhere, no NaN."""
    import torch
    r = {"err_bound": err_over_bound(got, ref, bound), "nan": int(torch.isnan(got.float()).sum().item())}
    r["ok"] = r["err_bound"] <= 1.0 and r["nan"] == 0
    return r


def chk_attention_geo(B, N, heads, modes, ref_pairs=None, seed=0, impls=(0, 1, 2, -1)):
    """One row of ATT_ROWS, every listed input mode: qkv inside a NaN-filled buffer with one image of guard on either side
    (keys past N must come from the tensor map's zero fill), every output in a canary-guarded buffer that starts as NaN
    (unwritten rows, stores of the ragged query tile past N). Per mode: the listed impls (0 / 1 / 2, -1 = the default)
    bit-identical, every image launched alone (with the last listed impl) bit-equal to the same image in the batch, qkv
    unchanged, no NaN, canaries intact, and err_over_bound <= 1 on every (image, head) or on ref_pairs."""
    torch, L, ops = _imports()
    dev = "cuda"
    D = heads * 64
    pairs = [(b, h) for b in range(B) for h in range(heads)] if ref_pairs is None else list(ref_pairs)
    ref_dev = dev if 4 * len(pairs) * N * N * 64 > 2e9 else "cpu"
    res = {"err_bound": 0.0, "modes": {}}
    ok = True
    t0 = time.time()
    i16 = torch.int16
    for mi, mode in enumerate(modes):
        qkv = att_operands(B, N, heads, mode, seed * 16 + mi, device=dev)
        gq = Guarded(tuple(qkv.shape), torch.bfloat16, dev, _guard_for(N * 3 * D), fill=float("nan"))
        gq.t.copy_(qkv)

        def launch(x, nb, impl):
            o = Guarded((nb * N, D), torch.bfloat16, dev, _guard_for(N * D))
            ops.attention(x, nb, N, heads, impl, out=o.t)
            return o

        outs = {impl: launch(gq.t, B, impl) for impl in impls}
        torch.cuda.synchronize()
        base = outs[impls[0]].t
        r = att_verdict(att_select(base, B, N, heads, pairs).to(ref_dev), *att_ref64(qkv, pairs, ref_dev))
        r["impls_same_bits"] = all(bool(torch.equal(outs[i].t.view(i16), base.view(i16))) for i in impls[1:])
        r["canaries_ok"] = all(o.canaries_intact() for o in outs.values())
        r["nan_all"] = sum(int(torch.isnan(o.t.float()).sum().item()) for o in outs.values())
        same = True
        if B > 1:  # each image alone: another grid, another unit list
            for i in range(B):
                o1 = launch(gq.t[i:i + 1], 1, impls[-1])
                same = same and bool(torch.equal(o1.t.view(i16), base[i * N:(i + 1) * N].view(i16))) and o1.canaries_intact()
        r["batch_invariant"] = same
        r["qkv_untouched"] = bool(torch.equal(gq.t.view(i16), qkv.view(i16)))
        torch.cuda.synchronize()
        r["ok"] = bool(r["ok"] and r["impls_same_bits"] and r["canaries_ok"] and r["nan_all"] == 0 and r["batch_invariant"]
                       and r["qkv_untouched"])
        res["modes"][mode] = r
        res["err_bound"] = max(res["err_bound"], r["err_bound"])
        ok = ok and r["ok"]
        del qkv, gq, outs
    res["ok"] = bool(ok)
    res["run_sec"] = round(time.time() - t0, 2)
    return res


# ---- token LayerNorm and channel LayerNorm: one fp64 reference and bound for both kernels
#
# Error model: the kernels compute fp32 two-pass statistics (mean, then the mean of squared deviations) of the row they
# normalise. The mean is off by well under 2^-16 mean|x| (D <= 1536 terms, per-lane partial sums and a warp tree), which
# moves every output by |w| rstd times that; the variance (and hence rstd) is good to a few 2^-24, far under 2^-16
# relative, which moves an output by 2^-16 |w| rstd |x - mean|. The affine (x - mean) * rstd * w + b in fp32 adds
# 2^-22 |b| where the two terms cancel, and the bf16 store 2^-8 |ref|. ReLU (channel LN) is 1-Lipschitz.
LN_EPS = 1e-6
LN_ROW_KINDS = ("normal", "offset", "massive", "near_const", "const")
# Common offset of the "offset" rows (sigma 1): a one-pass variance E[x^2] - E[x]^2 in fp32 loses all of its digits there
# (tests/test_encoder_check_cpu.py shows it fails the bound); the two-pass statistics pass with a wide margin.
LN_OFFSET = 3000.0


def ln_operands(rows, D, seed, device="cpu", deltas=False):
    """x [rows, D] fp32 mixing the row kinds (row r is LN_ROW_KINDS[r % 5]): N(0, s) with s in [0.5, 4]; LN_OFFSET +
    N(0, 1); N(0, 1) with four +-500 "massive activation" columns; c + 1e-3 N(0, 1) (eps is as large as the variance);
    exactly constant. w, b, w2, b2: fp32 affines. deltas: also d, d2 (bf16 [rows, D], the pending residual branches)
    that keep each row's kind: N(0, 1) on the first three kinds, 1e-3 N(0, 1) on the near-constant rows, one constant per
    row on the constant rows."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g, device=device)  # noqa: E731
    kind = torch.arange(rows, device=device) % len(LN_ROW_KINDS)
    z = rnd(rows, D)
    c = rnd(rows, 1)
    s = 0.5 + 3.5 * torch.rand(rows, 1, generator=g, device=device)
    massive = z.clone()
    cols = torch.randint(0, D, (rows, 4), generator=g, device=device)
    massive.scatter_(1, cols, 500.0 * torch.sign(rnd(rows, 4)))
    cases = [z * s + 0.3 * c, LN_OFFSET + z, massive, c + 1e-3 * z, c.expand(rows, D)]
    x = torch.zeros(rows, D, device=device)
    for i, t in enumerate(cases):
        x = torch.where((kind == i).view(rows, 1), t, x)
    op = {"x": x.contiguous(), "kind": kind}
    for nm in ("w", "b", "w2", "b2"):
        op[nm] = rnd(D)
    if deltas:
        for nm in ("d", "d2"):
            zd, cd = rnd(rows, D), rnd(rows, 1)
            t = torch.where((kind == 3).view(rows, 1), 1e-3 * zd, zd)
            op[nm] = torch.where((kind == 4).view(rows, 1), cd.expand(rows, D), t).bfloat16()
    return op


def ln_ref64(x, w, b, relu=False, eps=LN_EPS):
    """fp64 LayerNorm (x - mean) * rstd * w + b over the last dim (ReLU'd for the channel LN) of fp32 / bf16 rows x, and
    the per-element bound of the error model above: (ref, bound), fp64 on x's device."""
    import torch
    xd = x.double()
    mean = xd.mean(-1, keepdim=True)
    xc = xd - mean
    rstd = 1.0 / torch.sqrt(xc.pow(2).mean(-1, keepdim=True) + eps)
    wd, bd = w.double().to(x.device), b.double().to(x.device)
    ref = xc * rstd * wd + bd
    if relu:
        ref = torch.relu(ref)
    bound = REL_BF16 * ref.abs() + REL_ACC * wd.abs() * rstd * (xc.abs() + xd.abs().mean(-1, keepdim=True)) + REL_F32 * bd.abs()
    return ref, bound


def ln_verdict(got, ref, bound):
    import torch
    r = {"err_bound": err_over_bound(got, ref, bound), "nan": int(torch.isnan(got.float()).sum().item())}
    r["ok"] = r["err_bound"] <= 1.0 and r["nan"] == 0
    return r


def drop_cls_rows(t, n_tok):
    """[B * n_tok, D] -> the [B * (n_tok - 1), D] patch rows (token 0 of every image dropped)."""
    return t.view(-1, n_tok, t.shape[-1])[:, 1:].reshape(-1, t.shape[-1])


# The four token-LayerNorm launches of forward_body (csrc/ada_api.cu):
LN_KINDS = {
    "plain": dict(),                                             # norm1 of block 0
    "norm2": dict(delta=True),                                   # norm2: x + attention branch, x not stored
    "tap": dict(delta=True, delta2=True, write_x=True, tap=True),  # norm1 after a tapped block + the fused tap
    "last": dict(delta=True, delta2=True, drop_cls=True),        # the last tap: patch rows only
}
# (D, B, n_tok, kind): every width (ViT-S / B / L / G) x every launch kind; B * n_tok is never a multiple of 8 (the
# kernel walks rows from the last one, eight per block); n_tok 2 / 17 / 1370 = one patch, ViT-G at 56^2, ViT-S at 518^2.
LN_ROWS = [
    (384, 5, 2, "plain"), (384, 3, 17, "norm2"), (384, 2, 1370, "tap"), (384, 5, 2, "last"),
    (768, 3, 17, "plain"), (768, 2, 1370, "norm2"), (768, 5, 2, "tap"), (768, 3, 17, "last"),
    (1024, 2, 1370, "plain"), (1024, 5, 2, "norm2"), (1024, 3, 17, "tap"), (1024, 2, 1370, "last"),
    (1536, 5, 2, "plain"), (1536, 3, 17, "norm2"), (1536, 2, 1370, "tap"), (1536, 3, 17, "last"),
]


def chk_layernorm_geo(D, B, n_tok, kind, seed=0):
    """One token-LayerNorm launch (kind: a key of LN_KINDS, or such a dict of launch options): out (and the fused tap
    out2) held to the fp64 bound of the fp32 stream (x + d) + d2 the kernel normalises; x afterwards bit-equal to that
    stream when write_x is set and unchanged otherwise; the fused tap bit-equal to the separate tap pass; canaries around
    out, out2 and x intact; d / d2 inside NaN guards; no unwritten (NaN) output row."""
    torch, L, ops = _imports()
    dev = "cuda"
    t0 = time.time()
    k = LN_KINDS[kind] if isinstance(kind, str) else kind
    rows = B * n_tok
    op = ln_operands(rows, D, seed, dev, deltas=k.get("delta", False))
    x0 = op["x"]
    guard = _guard_for(D)
    gx = Guarded((rows, D), torch.float32, dev, guard)
    gx.t.copy_(x0)
    gd = {}
    for nm in ("d", "d2"):
        if k.get("delta" if nm == "d" else "delta2"):
            gd[nm] = Guarded((rows, D), torch.bfloat16, dev, guard, fill=float("nan"))
            gd[nm].t.copy_(op[nm])
    xs = x0
    if "d" in gd:
        xs = xs + op["d"].float()
    if "d2" in gd:
        xs = xs + op["d2"].float()
    patch_rows = B * (n_tok - 1)
    go = Guarded((patch_rows if k.get("drop_cls") else rows, D), torch.bfloat16, dev, guard)
    go2 = Guarded((patch_rows, D), torch.bfloat16, dev, guard) if k.get("tap") else None
    ops.layernorm(gx.t, op["w"], op["b"], LN_EPS, n_tok, bool(k.get("drop_cls")), delta=gd["d"].t if "d" in gd else None,
                  write_x=bool(k.get("write_x")), delta2=gd["d2"].t if "d2" in gd else None,
                  tap_w=op["w2"] if go2 else None, tap_b=op["b2"] if go2 else None, out=go.t, out2=go2.t if go2 else None)
    torch.cuda.synchronize()
    i32 = torch.int32
    res = {}
    ref, bound = ln_ref64(drop_cls_rows(xs, n_tok) if k.get("drop_cls") else xs, op["w"], op["b"])
    res["out"] = ln_verdict(go.t, ref, bound)
    ok = res["out"]["ok"]
    res["err_bound"] = res["out"]["err_bound"]
    res["x_as_expected"] = bool(torch.equal(gx.t.view(i32), (xs if k.get("write_x") else x0).view(i32)))
    canaries = go.canaries_intact() and gx.canaries_intact()
    if go2 is not None:
        ref2, bound2 = ln_ref64(drop_cls_rows(xs, n_tok), op["w2"], op["b2"])
        res["tap"] = ln_verdict(go2.t, ref2, bound2)
        res["err_bound"] = max(res["err_bound"], res["tap"]["err_bound"])
        canaries = canaries and go2.canaries_intact()
        sep = Guarded((patch_rows, D), torch.bfloat16, dev, guard)  # the separate tap pass (what the last block uses)
        ops.layernorm(x0.clone(), op["w2"], op["b2"], LN_EPS, n_tok, True, delta=gd["d"].t, write_x=False,
                      delta2=gd["d2"].t, out=sep.t)
        torch.cuda.synchronize()
        res["tap_same_bits_as_separate_pass"] = bool(torch.equal(sep.t.view(torch.int16), go2.t.view(torch.int16)))
        ok = ok and res["tap"]["ok"] and res["tap_same_bits_as_separate_pass"] and sep.canaries_intact()
    res["canaries_ok"] = bool(canaries)
    res["deltas_untouched"] = all(bool(torch.equal(gd[nm].t.view(torch.int16), op[nm].view(torch.int16))) for nm in gd)
    res["ok"] = bool(ok and res["x_as_expected"] and res["canaries_ok"] and res["deltas_untouched"])
    res["run_sec"] = round(time.time() - t0, 2)
    return res


# Channel LayerNorm + ReLU: 48 / 256 (the conv-epilogue widths, run stand-alone here) and every width the model runs
# through channel_ln_relu_kernel (C > 256: 384 ViT-S, 512, 768 ViT-B, 1024, 1536); 384 and 768 leave the last 32-lane
# round of a multi-group instantiation (<2, true, 2>, <4, false, 1>) partly / wholly idle.
CHLN_WIDTHS = (48, 256, 384, 512, 768, 1024, 1536)


def chln_pixels(C, sms):
    """A pixel count for which the persistent warps of launch_channel_ln_relu walk more than two grid strides and the last
    stride is ragged: stride = sms * 8 blocks * 8 warps * pixels per warp."""
    pix = 4 if C <= 256 else 2 if C <= 512 else 1
    return 2 * sms * 64 * pix + 8 * pix * 37 + 5


def chk_channel_ln_geo(C, seed=0, pixels=None):
    """Channel LayerNorm + ReLU on NHWC bf16 pixels of every row kind: fp64 bound, input (in a NaN-guarded buffer)
    unchanged, output canaries intact and no unwritten pixel; in place gives the same bits."""
    torch, L, ops = _imports()
    dev = "cuda"
    t0 = time.time()
    P = pixels or chln_pixels(C, torch.cuda.get_device_properties(0).multi_processor_count)
    op = ln_operands(P, C, seed, dev)
    x = op["x"].bfloat16()
    guard = _guard_for(C)
    gx = Guarded((P, C), torch.bfloat16, dev, guard, fill=float("nan"))
    gx.t.copy_(x)
    go = Guarded((P, C), torch.bfloat16, dev, guard)
    ops.channel_ln_relu(gx.t, op["w"], op["b"], out=go.t)
    torch.cuda.synchronize()
    ref, bound = ln_ref64(x, op["w"], op["b"], relu=True)
    res = ln_verdict(go.t, ref, bound)
    res["pixels"] = P
    res["canaries_ok"] = go.canaries_intact()
    res["input_untouched"] = bool(torch.equal(gx.t.view(torch.int16), x.view(torch.int16)))
    ops.channel_ln_relu(gx.t, op["w"], op["b"], out=gx.t)  # in place, as the model runs it
    torch.cuda.synchronize()
    res["in_place_same_bits"] = bool(torch.equal(gx.t.view(torch.int16), go.t.view(torch.int16)))
    res["ok"] = bool(res["ok"] and res["canaries_ok"] and res["input_untouched"] and res["in_place_same_bits"])
    res["run_sec"] = round(time.time() - t0, 2)
    return res


# ---- DPT head bandwidth kernels: k = s transposed convs, bilinear upsample, patch gather
#
# Transposed convs (EPI_CONVT): every output is one bias plus a Ci-term dot product of bf16 operands accumulated in fp32 and
# stored as bf16, so the conv error model above holds with S = conv_transpose2d(|x|, |w|) + |b|.
def convT_operands(B, H, W, Ci, Co, ks, mode, seed, device="cpu"):
    """x [B, H, W, Ci] bf16, w [Ci, Co, ks, ks] rounded to bf16 (held as fp32), b [Co] fp32. mode "rand": N(0, 1) inputs;
    "onehot": pixel (b, y, x) is one-hot at channel (5 b + 3 y + x) mod Ci, so every output is a single weight
    w[c, co, ky, kx] + b[co], and a pixel shuffle that swaps ky and kx, or picks the wrong image or channel slab, moves it by
    O(1) instead of by rounding."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    w = (torch.randn(Ci, Co, ks, ks, generator=g, device=device) / Ci ** 0.5).bfloat16().float()
    b = torch.randn(Co, generator=g, device=device) * 0.1
    if mode == "rand":
        x = torch.randn(B, H, W, Ci, generator=g, device=device).bfloat16()
    else:
        assert mode == "onehot", mode
        bi, yi, xi = torch.meshgrid(*(torch.arange(n, device=device) for n in (B, H, W)), indexing="ij")
        x = torch.nn.functional.one_hot((5 * bi + 3 * yi + xi) % Ci, Ci).bfloat16()
    return {"x": x, "w": w, "b": b}


def convT_ref64(op, ks, imgs=None):
    """fp64 reference of the k = s transposed conv on convT_operands-style op (any device) and its per-element bound:
    (ref, bound) as [b, H ks, W ks, Co] over the images `imgs` (all if None)."""
    import torch
    F = torch.nn.functional
    x = op["x"] if imgs is None else op["x"][list(imgs)]
    xd, wd, bd = x.double().permute(0, 3, 1, 2), op["w"].double().to(x.device), op["b"].double().to(x.device)
    ref = F.conv_transpose2d(xd, wd, bd, stride=ks).permute(0, 2, 3, 1)
    S = F.conv_transpose2d(xd.abs(), wd.abs(), bd.abs(), stride=ks).permute(0, 2, 3, 1)
    return ref, REL_BF16 * ref.abs() + REL_ACC * S


def head_verdict(got, ref, bound):
    """got / ref / bound of one head kernel: within the bound everywhere, no NaN."""
    import torch
    r = {"err_bound": err_over_bound(got, ref, bound), "nan": int(torch.isnan(got.float()).sum().item())}
    r["ok"] = r["err_bound"] <= 1.0 and r["nan"] == 0
    return r


def _ref_device(work):
    """Large fp64 references (work: their multiply-adds) run on the device, as conv_geo_bench_* does; small ones on the host."""
    return "cuda" if work > 3e8 else "cpu"


def convT_run(op, ks, pix, cg=0, ref_imgs=None):
    """One transposed conv as forward_body launches it (pix: pixel-tile A operand and 5-D TMA stores, else linear A rows and
    per-thread scatter), force_cg=cg: x inside a NaN guard of one image on either side, the output canary-guarded and
    NaN-filled; fp64 bound on `ref_imgs` (all if None), no unwritten pixel, x unchanged, every image launched alone
    bit-equal to the batch, and with cg = 2 bit-equal to single-CTA tiles."""
    torch, L, ops = _imports()
    dev = "cuda"
    t0 = time.time()
    x = op["x"]
    B, H, W, Ci = x.shape
    Co = op["w"].shape[1]
    imgs = list(range(B)) if ref_imgs is None else list(ref_imgs)
    gx = Guarded(tuple(x.shape), torch.bfloat16, dev, _guard_for(H * W * Ci), fill=float("nan"))
    gx.t.copy_(x)
    wp = ops.pack_convT(op["w"], ks)
    b = op["b"].to(dev)

    def launch(xin, c):
        nb = xin.shape[0]
        o = Guarded((nb, H * ks, W * ks, Co), torch.bfloat16, dev, _guard_for(H * W * ks * ks * Co))
        if pix:
            ops.gemm(xin, wp, conv=(nb, H, W, Ci), conv_taps=1, N=ks * ks * Co, epi=L.EPI_CONVT, bias=b, out_bf16=o.t, ks=ks,
                     cout=Co, force_cg=c)
        else:
            ops.gemm(xin.reshape(nb * H * W, Ci), wp, epi=L.EPI_CONVT, bias=b, out_bf16=o.t, ks=ks, cout=Co, H=H, W=W,
                     force_cg=c)
        return o

    out = launch(gx.t, cg)
    torch.cuda.synchronize()
    rd = _ref_device(2.0 * len(imgs) * H * W * Ci * Co * ks * ks)
    ref, bound = convT_ref64({"x": x.to(rd), "w": op["w"].to(rd), "b": op["b"].to(rd)}, ks, imgs)
    r = head_verdict(out.t[imgs].to(rd), ref, bound)
    del ref, bound
    r["nan_all"] = int(torch.isnan(out.t.float()).sum().item())
    i16 = torch.int16
    same = True
    for i in range(B):
        o1 = launch(gx.t[i:i + 1], 0)
        same = same and bool(torch.equal(o1.t.view(i16), out.t[i:i + 1].view(i16))) and o1.canaries_intact()
    r["batch_invariant"] = same
    if cg == 2:
        o2 = launch(gx.t, 1)
        r["pair_invariant"] = bool(torch.equal(o2.t.view(i16), out.t.view(i16)))
    else:
        r["pair_invariant"] = True
    torch.cuda.synchronize()
    r["canaries_ok"] = out.canaries_intact()
    r["input_untouched"] = bool(torch.equal(gx.t.view(i16), x.view(i16)))
    r["ok"] = bool(r["ok"] and r["nan_all"] == 0 and r["batch_invariant"] and r["pair_invariant"] and r["canaries_ok"]
                   and r["input_untouched"])
    r["run_sec"] = round(time.time() - t0, 2)
    return r


# (ks, Ci, B, H, W, force_cg, ref_imgs): resize_layers[0] (k 4) and [1] (k 2) of every encoder, Co = Ci, on the path
# forward_body takes (pixel tiles when Ci % 64 == 0, linear A rows otherwise). Widths ragged against the 16-pixel tile
# (37, 49, 7, 5), exact (32) and 1 x 1. force_cg = 2 pairs CTAs where pick_bn gives 256-wide tiles (N = ks^2 Ci >= 768).
# At 32 x 32, B = 4, Ci 256, k 4 the launcher pairs on its own: 4096 padded pixels either way, 16 x 16 = 256 pairs >= 148.
CONVT_GEO_ROWS = [
    (4, 48, 3, 37, 37, 0, None),      # ViT-S level 0 at 518^2 (linear)
    (4, 48, 2, 7, 5, 0, None),        # ViT-S level 0 at 98 x 70
    (4, 96, 2, 37, 49, 0, None),      # ViT-B level 0 at 518 x 686 (linear)
    (4, 96, 5, 1, 1, 0, None),        # ViT-B level 0 at 14^2
    (4, 256, 2, 37, 49, 0, None),     # ViT-L level 0 (pixel tiles)
    (4, 256, 3, 1, 1, 0, None),       # ViT-L level 0 at 14^2
    (4, 1536, 2, 5, 7, 0, None),      # ViT-G level 0 (guided, and the un-guided ViT-G of infer.py)
    (4, 1536, 1, 4, 4, 0, None),      # ViT-G level 0 at 56^2
    (2, 96, 2, 37, 37, 0, None),      # ViT-S level 1 (linear)
    (2, 96, 3, 1, 1, 0, None),        # ViT-S level 1 at 14^2
    (2, 192, 2, 37, 49, 0, None),     # ViT-B level 1 (pixel tiles)
    (2, 192, 3, 7, 5, 0, None),       # ViT-B level 1 at 98 x 70
    (2, 512, 2, 32, 32, 0, None),     # ViT-L level 1 at 448^2: whole 16-pixel tiles
    (2, 1536, 2, 7, 5, 0, None),      # ViT-G level 1
    (2, 1536, 2, 1, 1, 0, None),      # ViT-G level 1 at 14^2
    (4, 256, 2, 32, 32, 2, None),     # CTA pairs, pixel tiles: bit-equal to single CTAs
    (4, 256, 2, 37, 37, 2, None),
    (2, 512, 1, 37, 37, 2, None),
    (4, 48, 2, 37, 37, 2, None),      # CTA pairs, linear A rows
    (4, 256, 4, 32, 32, 0, None),     # the launcher's own pairing (ViT-L at 448^2, batch 4)
    (4, 256, 32, 37, 37, 0, (0, 16, 31)),  # the benchmark's ViT-L launches: 518^2, batch 32
    (2, 512, 32, 37, 37, 0, (0, 16, 31)),
]


def chk_convT_geo(ks, Ci, B, H, W, cg=0, ref_imgs=None, seed=0, modes=("rand", "onehot")):
    torch, L, ops = _imports()
    parts = {}
    for mi, mode in enumerate(modes):
        op = convT_operands(B, H, W, Ci, Ci, ks, mode, seed * 8 + mi, device="cuda")
        parts[mode] = convT_run(op, ks, Ci % 64 == 0, cg, ref_imgs)
        del op
    return {"ok": all(p["ok"] for p in parts.values()), "err_bound": max(p["err_bound"] for p in parts.values()),
            "modes": parts, "run_sec": round(sum(p["run_sec"] for p in parts.values()), 2)}


# Bilinear upsample (align_corners=True). The source coordinates are ATen's, in fp32 as upsample_bilinear_kernel computes
# them: scale = (in - 1) / (out - 1), src = scale * dst, i0 = (int) src, i1 = i0 + (i0 < in - 1), l = src - i0 (exact); the
# reference interpolates with weights l and 1 - l in fp64 (tests/test_head_check_cpu.py pins these weights to
# F.interpolate). Error model: the kernel forms 1 - l in fp32 (relative error <= 2^-24: exact for l >= 1/2), then per pass
# two products and a sum in fp32 (three roundings), horizontally and then vertically: at most 6 units of 2^-24 relative to
# sum w |corner| to first order, held to UP_C = 8. The bf16 store adds 2^-8 |ref|.
UP_C = 8


def up_coords(n_in, n_out):
    """(i0, i1, l) per output index: ATen's align_corners=True source coordinates in fp32 (numpy int64 / fp64 arrays)."""
    import numpy as np
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0.0)
    src = (scale * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < n_in - 1)
    return i0, i1, (src - i0.astype(np.float32)).astype(np.float64)


def up_matrix(n_in, n_out, device="cpu"):
    """[n_out, n_in] fp64 interpolation weights of up_coords."""
    import torch
    i0, i1, lam = up_coords(n_in, n_out)
    A = torch.zeros(n_out, n_in, dtype=torch.float64)
    r = torch.arange(n_out)
    lam = torch.from_numpy(lam)
    A.index_put_((r, torch.from_numpy(i0)), 1.0 - lam, accumulate=True)
    A.index_put_((r, torch.from_numpy(i1)), lam, accumulate=True)
    return A.to(device)


def up_ref64(x, Ho, Wo):
    """fp64 bilinear of NHWC x (any device) to (Ho, Wo) and the per-element bound of the model above: (ref, bound)."""
    import torch
    Ah, Aw = up_matrix(x.shape[1], Ho, x.device), up_matrix(x.shape[2], Wo, x.device)
    xd = x.double()
    ref = torch.einsum("pw,bowc->bopc", Aw, torch.einsum("oh,bhwc->bowc", Ah, xd))
    S = torch.einsum("pw,bowc->bopc", Aw, torch.einsum("oh,bhwc->bowc", Ah, xd.abs()))
    return ref, REL_BF16 * ref.abs() + UP_C * 2.0 ** -24 * S


def up_operands(B, Hi, Wi, C, mode, seed, device="cpu"):
    """NHWC bf16 input. "rand": N(0, 1); "ramp": source row y of image b is offset by 100 ((3 y + 2 b) mod 5 - 2) on top of
    N(0, 1), so neighbouring rows differ by at least 100x the spread inside a row: reading the wrong source row, or a stale
    row across a strip boundary, misses the bound by orders of magnitude."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(B, Hi, Wi, C, generator=g, device=device)
    if mode == "ramp":
        y, b = torch.arange(Hi, device=device).view(1, Hi, 1, 1), torch.arange(B, device=device).view(B, 1, 1, 1)
        x = x + 100.0 * ((3 * y + 2 * b) % 5 - 2).float()
    else:
        assert mode == "rand", mode
    return x.bfloat16()


def upsample_run(x, Ho, Wo, ref_imgs=None):
    """One upsample launch: x inside a NaN guard of one image on either side, output canary-guarded and NaN-filled; fp64
    bound on `ref_imgs` (all if None), no unwritten pixel, x unchanged, every image launched alone bit-equal to the batch."""
    torch, L, ops = _imports()
    dev = "cuda"
    t0 = time.time()
    B, Hi, Wi, C = x.shape
    imgs = list(range(B)) if ref_imgs is None else list(ref_imgs)
    gx = Guarded(tuple(x.shape), torch.bfloat16, dev, _guard_for(Hi * Wi * C), fill=float("nan"))
    gx.t.copy_(x)

    def launch(xin):
        o = Guarded((xin.shape[0], Ho, Wo, C), torch.bfloat16, dev, _guard_for(Ho * Wo * C))
        ops.upsample(xin, Ho, Wo, out=o.t)
        return o

    out = launch(gx.t)
    torch.cuda.synchronize()
    rd = _ref_device(2.0 * len(imgs) * Ho * C * (Hi * Wi + Wo * Wi))
    ref, bound = up_ref64(x[imgs].to(rd), Ho, Wo)
    r = head_verdict(out.t[imgs].to(rd), ref, bound)
    del ref, bound
    r["nan_all"] = int(torch.isnan(out.t.float()).sum().item())
    i16 = torch.int16
    same = True
    for i in range(B):
        o1 = launch(gx.t[i:i + 1])
        same = same and bool(torch.equal(o1.t.view(i16), out.t[i:i + 1].view(i16))) and o1.canaries_intact()
    torch.cuda.synchronize()
    r["batch_invariant"] = same
    r["canaries_ok"] = out.canaries_intact()
    r["input_untouched"] = bool(torch.equal(gx.t.view(i16), x.view(i16)))
    r["ok"] = bool(r["ok"] and r["nan_all"] == 0 and r["batch_invariant"] and r["canaries_ok"] and r["input_untouched"])
    r["run_sec"] = round(time.time() - t0, 2)
    return r


def up_maps(gh, gw):
    """The four maps forward_body upsamples at patch grid gh x gw (refinenet4..1): down2(g) -> g, g -> 2g, 2g -> 4g,
    4g -> 8g, as (Hi, Wi, Ho, Wo)."""
    d2 = lambda n: (n - 1) // 2 + 1  # noqa: E731
    return [(d2(gh), d2(gw), gh, gw)] + [(gh << k, gw << k, gh << (k + 1), gw << (k + 1)) for k in range(3)]


# (gh, gw) per width F (ViT-S / B / L / G): gh = 1 gives Ho = 1 and Wo = 1 (scale 0); 5 gives maps of fewer than 16 rows and
# heights that are not multiples of 16 (the last strip ragged); 9 x 7 non-square maps; 37 the 518^2 maps. F = 384 has 48
# channel groups, not a power of two (the division path of the kernel's index math).
UP_GRIDS = ((1, 1), (4, 4), (5, 5), (9, 7), (37, 37))
UP_WIDTHS = (64, 128, 256, 384)


def chk_upsample_geo(C, maps, B, ref_imgs=None, seed=0, modes=("rand", "ramp")):
    parts = {}
    for mi, (Hi, Wi, Ho, Wo) in enumerate(maps):
        for mj, mode in enumerate(modes):
            x = up_operands(B, Hi, Wi, C, mode, seed * 64 + mi * 8 + mj, device="cuda")
            parts[f"{Hi}x{Wi}->{Ho}x{Wo}_{mode}"] = upsample_run(x, Ho, Wo, ref_imgs)
            del x
    return {"ok": all(p["ok"] for p in parts.values()), "err_bound": max(p["err_bound"] for p in parts.values()),
            "maps": parts, "run_sec": round(sum(p["run_sec"] for p in parts.values()), 2)}


# Patch gather: exactly specified, so checked bit for bit: ((x - mean) / std) in fp32 (RGB planes; guide planes pass
# through as (x - 0) / 1), rounded to bf16, in the K order c * 196 + ky * 14 + kx of the patch-embed weight.
PG_MEAN, PG_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def patch_gather_expected(rgb, guides, mean=PG_MEAN, std=PG_STD):
    """[B * ph * pw, C * 196] bf16 on the CPU: what patch_gather_kernel must store, bit for bit."""
    import torch
    m = torch.tensor(mean, dtype=torch.float32).view(1, 3, 1, 1)
    s = torch.tensor(std, dtype=torch.float32).view(1, 3, 1, 1)
    x = torch.cat([(rgb.cpu() - m) / s] + [g.cpu() for g in guides], 1)
    B, C, H, W = x.shape
    ph, pw = H // 14, W // 14
    x = x[:, :, :ph * 14, :pw * 14].reshape(B, C, ph, 14, pw, 14).permute(0, 2, 4, 1, 3, 5)
    return x.reshape(B * ph * pw, C * 196).bfloat16()


PG_SENTINEL = -3.0  # K-padding columns start as this and must keep it


def patch_gather_run(rgb, guides, Kpad=None):
    """One patch gather (normalize = 1, the path ada_op_patch_gather runs): image and guides inside NaN guards of one image
    on either side, output canary-guarded with its patch columns NaN and its K padding PG_SENTINEL; the patch columns
    bit-equal to patch_gather_expected, the padding and the inputs unchanged."""
    torch, L, ops = _imports()
    dev = "cuda"
    t0 = time.time()
    B, _, H, W = rgb.shape
    K = (3 + sum(g.shape[1] for g in guides)) * 196
    Kpad = Kpad or (K + 63) // 64 * 64
    rows = B * (H // 14) * (W // 14)
    gin = []
    for t in [rgb] + list(guides):
        gt = Guarded(tuple(t.shape), torch.float32, dev, _guard_for(t[0].numel()), fill=float("nan"))
        gt.t.copy_(t)
        gin.append(gt)
    go = Guarded((rows, Kpad), torch.bfloat16, dev, _guard_for(Kpad), body=PG_SENTINEL)
    go.t[:, :K] = float("nan")
    ops.patch_gather(gin[0].t, [g.t for g in gin[1:]], Kpad, out=go.t)
    torch.cuda.synchronize()
    i16 = torch.int16
    got = go.t.cpu()
    exp = patch_gather_expected(rgb, guides)
    r = {"bit_exact": bool(torch.equal(got[:, :K].view(i16), exp.view(i16)))}
    r["mismatches"] = int((got[:, :K].view(i16) != exp.view(i16)).sum().item())
    r["padding_untouched"] = bool((got[:, K:] == PG_SENTINEL).all().item())
    r["canaries_ok"] = go.canaries_intact()
    r["inputs_untouched"] = all(bool(torch.equal(g.t.view(torch.int32), t.view(torch.int32)))
                                for g, t in zip(gin, [rgb] + list(guides)))
    r["ok"] = bool(r["bit_exact"] and r["padding_untouched"] and r["canaries_ok"] and r["inputs_untouched"])
    r["err_bound"] = 0.0
    r["run_sec"] = round(time.time() - t0, 2)
    return r


# (B, H, W, guide channels per guide tensor): guide channels 0 (un-guided), 2 (mask + observation), 4 and 5; patches per
# row 1, 5, 32, 33 (32 + 1), 37 (518: 32 + 5 in two blocks of 19 / 18) and 74 (1036: 25 + 25 + 24); the benchmark's batch.
PG_ROWS = [
    (3, 28, 14, ()),
    (2, 42, 70, (1, 1)),
    (2, 28, 448, (1, 3)),
    (2, 14, 462, (3, 1, 1)),
    (3, 28, 518, ()),
    (2, 28, 518, (1, 1)),
    (1, 28, 1036, (1, 1)),
    (1, 14, 1036, (2, 3)),
    (32, 518, 518, (1, 1)),
]


def chk_patch_gather_geo(B, H, W, guide_ch, seed=0):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    rgb = torch.rand(B, 3, H, W, generator=g, device="cuda")
    guides = [torch.rand(B, c, H, W, generator=g, device="cuda") * 2 - 1 for c in guide_ch]
    return patch_gather_run(rgb, guides)


def _all_ok(*results):
    """Several checks under one name: ok when all are."""
    return {"ok": all(r["ok"] for r in results), "err_bound": max(r.get("err_bound", 0.0) for r in results),
            "parts": list(results)}


# The attention / LayerNorm checks of the first bring-up, by their original names: each shape and input of theirs, now held
# to the fp64 bounds above (one kernel per attention row; bit-identity of the kernels for the impls_agree rows).
#   name: (B, N, heads, input mode of att_operands)
ATT_IMPL_ROWS = {
    "small": (1, 128, 1, "rand"), "ragged": (1, 200, 2, "rand"), "1370": (2, 1370, 6, "rand"),
    "rescale": (1, 1370, 2, "grow"), "5477": (1, 5477, 2, "rand"),
    # persistent kernel: several work units per CTA, full (two query tiles) and short (one tile) units interleaved
    "multiunit_1370": (4, 1370, 16, "rand"), "multiunit_300": (8, 300, 16, "rand"), "multiunit_128": (10, 128, 16, "rand"),
    "multiunit_rescale": (3, 700, 16, "grow"),
}
ATT_AGREE_ROWS = {"1370": (3, 1370, 16, "rand"), "rescale": (2, 700, 16, "grow"), "5477": (1, 5477, 4, "rand")}

CHECKS = {
    "gemm_resid_f32": lambda: chk_gemm_resid_f32(1370 * 3, 1024, 1024),
    "gemm_resid_f32_cg2": lambda: chk_gemm_resid_f32(1370 * 3, 1024, 4096, cg=2),
    "gemm_resid_f32_ragged": lambda: chk_gemm_resid_f32(777, 384, 1536, gamma=False),
    "gemm_resid_f32_small": lambda: chk_gemm_resid_f32(100, 96, 64),
    "gemm_small_bn128": lambda: chk_gemm(300, 256, 128, 128, "bias"),
    "gemm_small_bn256": lambda: chk_gemm(300, 256, 128, 256, "bias"),
    "gemm_small_bn64": lambda: chk_gemm(300, 256, 192, 64, "bias"),
    "gemm_qkv_shape": lambda: chk_gemm(1370 * 2, 3072, 1024, 0, "bias"),
    "gemm_fc1_gelu": lambda: chk_gemm(1370, 4096, 1024, 0, "gelu"),
    "gemm_fc2_resid": lambda: chk_gemm(1370, 1024, 4096, 0, "resid"),
    "gemm_ragged_n": lambda: chk_gemm(500, 48, 384, 0, "bias"),
    "gemm_swiglu": lambda: chk_gemm(700, 1024, 256, 0, "swiglu"),
    "gemm_embed": chk_embed,
    "gemm_cg2_small": lambda: chk_gemm(300, 256, 128, 256, "bias", cg=2),
    "gemm_cg2_bn128": lambda: chk_gemm(700, 384, 192, 128, "bias", cg=2),
    "gemm_cg2_qkv": lambda: chk_gemm(1370 * 2, 3072, 1024, 0, "bias", cg=2),
    "gemm_cg2_gelu": lambda: chk_gemm(1370, 4096, 1024, 0, "gelu", cg=2),
    "gemm_cg2_gamma": lambda: chk_gemm(1370, 1024, 4096, 0, "resid", cg=2),
    "gemm_cg2_swiglu": lambda: chk_gemm(700, 1024, 256, 0, "swiglu", cg=2),
    "conv_cg2_plain": lambda: chk_conv(2, 37, 45, 128, 256, "plain", cg=2),
    "conv_cg2_rcu": lambda: chk_conv(2, 19, 33, 64, 128, "rcu", cg=2),
    "conv_plain_37": lambda: chk_conv(2, 37, 37, 128, 64, "plain"),
    "conv_c48": lambda: chk_conv(1, 20, 33, 48, 48, "plain"),
    "conv_rcu": lambda: chk_conv(2, 19, 19, 64, 64, "rcu"),
    "conv_tail": lambda: chk_conv(1, 70, 84, 64, 32, "tail"),
    "convT_k4": lambda: chk_convT(4),
    "convT_k2": lambda: chk_convT(2),
    # Cout % 64 == 0: pixel shuffle through the 5-D TMA store (warps whose 32 pixels span 1, 2 and up to 7 image rows)
    "convT_k4_c256_tma": lambda: chk_convT(4, 256, 256, pix=True),
    "convT_k2_c512_tma": lambda: chk_convT(2, 128, 512, pix=True),
    "convT_k4_c64_w5_tma": lambda: chk_convT(4, 64, 64, B=3, H=7, W=5, pix=True),
    "convT_k2_c128_w49_tma": lambda: chk_convT(2, 192, 128, B=1, H=37, W=49, pix=True),
    "convT_k2_c256_linear": lambda: chk_convT(2, 256, 256),
    "upsample_19_37": lambda: chk_upsample(19, 37),
    "upsample_37_74": lambda: chk_upsample(37, 74),
    "upsample_148_296_c256": lambda: chk_upsample(148, 296, 256),
    "upsample_40_70_c128": lambda: chk_upsample(40, 70, 128),   # not a 2x map: strips cross source rows irregularly
    "fused_tail_5x7": lambda: chk_fused_tail(5, 7),
    "fused_tail_9x9": lambda: chk_fused_tail(9, 9),
    "tail_mma_5x7_c64": lambda: chk_tail_mma(5, 7, 64),
    "tail_mma_9x9_c128": lambda: chk_tail_mma(9, 9, 128),
    "tail_mma_3x11_c32_logit": lambda: chk_tail_mma(3, 11, 32, B=3, sigmoid=0),
    "tail_mma_37x37_c128": lambda: chk_tail_mma(37, 37, 128, B=2),
    "tail_mma_1x1_c64_relu": lambda: chk_tail_mma(1, 1, 64, B=5, sigmoid=2),
    "patch_gather": chk_patch_gather,
    "conv_chln_256": lambda: chk_conv(2, 37, 45, 256, 256, "chln"),
    "conv_chln_256_cg2": lambda: chk_conv(2, 40, 70, 256, 256, "chln", cg=2),
    "conv_chln_48": lambda: chk_conv(2, 20, 33, 48, 48, "chln"),
    "conv_chln_192": lambda: chk_conv(1, 37, 37, 192, 192, "chln"),
    "conv_s2_37": lambda: chk_conv_s2(2, 37, 37, 128, 192),
    "conv_s2_74x50": lambda: chk_conv_s2(1, 74, 50, 64, 64),
    "conv_s2_1024": lambda: chk_conv_s2(2, 37, 37, 1024, 1024),
    # every pixel-tile shape x every conv epilogue against fp64 (seeded by row; odd seeds give the stride-2 input an even size)
    **{f"conv_geo_{r[0]}{r[1]}{r[2]}_{r[3]}": (lambda r=r, i=i: chk_conv_geo(*r, seed=i)) for i, r in enumerate(CONV_GEO_ROWS)},
    # batch-32 maps of the ViT-L head: layer_rn, RCU1 conv2, plain conv; resize_layers[3] 37 -> 19
    **{f"conv_geo_bench_{h}": (lambda h=h: chk_conv_geo_bench(32, h, h, ("a_bias", "b_relu_copy", "d_resid2_relu_copy"),
                                                              (0, 16, 31))) for h in (148, 74, 37, 19)},
    "conv_geo_bench_s2_37": lambda: chk_conv_geo_bench(32, 19, 19, ("h_s2_bias",), (0, 16, 31)),
    **{f"gemm_tiles_{k}": (lambda k=k: chk_gemm_tiles(k)) for k in GEMM_TILES},
    # both attention kernels (impl 0 = attention.cuh, 1 / 2 = attention2.cuh one / two threads per row), then the default
    **{f"attention{i}_{n}": (lambda i=i, r=r: chk_attention_geo(*r[:3], (r[3],), impls=(i,)))
       for n, r in ATT_IMPL_ROWS.items() for i in (0, 1, 2)},
    "attention_auto_b32": lambda: chk_attention_geo(32, 1370, 16, ("rand",), ((0, 0), (16, 7), (31, 15)), impls=(-1,)),
    **{f"attention_impls_agree_{n}": (lambda r=r: chk_attention_geo(*r[:3], (r[3],), seed=15)) for n, r in ATT_AGREE_ROWS.items()},
    "layernorm_384": lambda: chk_layernorm_geo(384, 3, 50, "plain", seed=6),
    "layernorm_1024_drop": lambda: chk_layernorm_geo(1024, 3, 50, dict(drop_cls=True), seed=6),
    "layernorm_1536": lambda: chk_layernorm_geo(1536, 3, 50, "plain", seed=6),
    "layernorm_delta": lambda: _all_ok(chk_layernorm_geo(1024, 300, 1, dict(delta=True, write_x=True), seed=16),
                                       chk_layernorm_geo(1024, 300, 1, "norm2", seed=16),
                                       chk_layernorm_geo(1024, 300, 1, dict(delta=True, delta2=True, write_x=True), seed=16)),
    "layernorm_tap_fused": lambda: chk_layernorm_geo(1024, 3, 50, "tap", seed=26),
    **{f"channel_ln_{c}": (lambda c=c: chk_channel_ln_geo(c, seed=7, pixels=2 * 9 * 11)) for c in (48, 256, 512, 1024, 1536)},
    # attention at every ragged residue, tile count and head count against fp64, all kernels bit-identical
    **{f"attention_geo_{r[0]}x{r[1]}x{r[2]}": (lambda r=r, i=i: chk_attention_geo(*r, seed=i)) for i, r in enumerate(ATT_ROWS)},
    # token LayerNorm: every width x every launch kind of the encoder; channel LayerNorm + ReLU at every width
    **{f"ln_geo_{r[0]}_{r[3]}": (lambda r=r, i=i: chk_layernorm_geo(*r, seed=i)) for i, r in enumerate(LN_ROWS)},
    **{f"ln_geo_channel_{c}": (lambda c=c, i=i: chk_channel_ln_geo(c, seed=i)) for i, c in enumerate(CHLN_WIDTHS)},
    # DPT head: transposed convs, the four upsample maps at every width, patch gather, against fp64 / exact references
    **{f"convT_geo_k{r[0]}_c{r[1]}_{r[3]}x{r[4]}_b{r[2]}" + (f"_cg{r[5]}" if r[5] else ""): (lambda r=r, i=i: chk_convT_geo(*r, seed=i))
       for i, r in enumerate(CONVT_GEO_ROWS)},
    **{f"upsample_geo_c{c}_{gh}x{gw}": (lambda c=c, gh=gh, gw=gw, i=i: chk_upsample_geo(c, up_maps(gh, gw), 2 if gh > 9 else 3, seed=i))
       for i, (c, (gh, gw)) in enumerate((c, g) for c in UP_WIDTHS for g in UP_GRIDS)},
    "upsample_geo_bench_19_37": lambda: chk_upsample_geo(256, [(19, 19, 37, 37)], 32, seed=90),
    "upsample_geo_bench_148_296": lambda: chk_upsample_geo(256, [(148, 148, 296, 296)], 32, (0, 16, 31), seed=91),
    **{f"patch_gather_geo_{r[0]}x{r[1]}x{r[2]}_g{sum(r[3])}": (lambda r=r, i=i: chk_patch_gather_geo(*r, seed=i))
       for i, r in enumerate(PG_ROWS)},
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--one")
    ap.add_argument("--only", default="")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "gpu_check.json"))
    a = ap.parse_args()
    if a.one:
        try:
            r = CHECKS[a.one]()
        except Exception as e:  # noqa: BLE001
            r = {"ok": False, "exception": repr(e)[:500]}
            try:
                _, L, _ = _imports()
                r["device_error"] = [hex(v) for v in L.device_error()]
            except Exception:  # noqa: BLE001
                pass
        print("RESULT " + json.dumps(r))
        return
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    results = {}
    names = [n for n in CHECKS if a.only in n]
    for n in names:
        t0 = time.time()
        try:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", n], capture_output=True, text=True,
                               timeout=180)
            line = [l for l in p.stdout.splitlines() if l.startswith("RESULT ")]
            r = json.loads(line[-1][7:]) if line else {"ok": False, "rc": p.returncode, "stderr": p.stderr[-800:]}
        except subprocess.TimeoutExpired:
            r = {"ok": False, "timeout": True}
        r["sec"] = round(time.time() - t0, 1)
        results[n] = r
        print(n, json.dumps(r), flush=True)
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)
    nok = sum(1 for r in results.values() if r.get("ok"))
    print(f"SUMMARY {nok}/{len(results)} ok")


if __name__ == "__main__":
    main()

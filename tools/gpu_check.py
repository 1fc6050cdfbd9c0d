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
    """pix: A operand on 8x16 pixel tiles, pixel shuffle stored through 5-D TMA boxes (Cin, Cout % 64 == 0)."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(B, Cin, H, W, generator=g, device="cuda").bfloat16()
    w = torch.randn(Cin, Cout, ks, ks, generator=g, device="cuda") * 0.1
    bias = torch.randn(Cout, generator=g, device="cuda") * 0.1
    ref = torch.nn.functional.conv_transpose2d(x.float(), w.bfloat16().float(), bias, stride=ks)
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    wp = ops.pack_convT(w, ks)
    out = torch.zeros(B, H * ks, W * ks, Cout, dtype=torch.bfloat16, device="cuda")
    if pix:
        ops.gemm(x_nhwc, wp, conv=(B, H, W, Cin), conv_taps=1, N=ks * ks * Cout, epi=L.EPI_CONVT, bias=bias, out_bf16=out, ks=ks,
                 cout=Cout)
    else:
        ops.gemm(x_nhwc.reshape(B * H * W, Cin), wp, epi=L.EPI_CONVT, bias=bias, out_bf16=out, ks=ks, cout=Cout, H=H, W=W)
    torch.cuda.synchronize()
    return _cmp("convT", out.permute(0, 3, 1, 2), ref, 3e-2, 1e-2)


def chk_attention(B, N, heads, grow=False, impl=-1):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(5)
    D = heads * 64
    qkv = torch.randn(B, N, 3, heads, 64, generator=g, device="cuda") * 1.5
    if grow:  # key norms grow along the sequence -> row maxima jump by > 2^8 between KV tiles (exercises the O rescale)
        ramp = 1.0 + 7.0 * (torch.arange(N, device="cuda") // 128).float() / max((N - 1) // 128, 1)
        qkv[:, :, 1] *= ramp.view(1, N, 1, 1)
    qkv = qkv.bfloat16()
    out = ops.attention(qkv, B, N, heads, impl)
    torch.cuda.synchronize()
    q, k, v = [t.float().permute(0, 2, 1, 3) for t in qkv.unbind(2)]  # [B,h,N,64]
    att = torch.softmax((q * 0.125) @ k.transpose(-1, -2), dim=-1)
    ref = (att @ v).permute(0, 2, 1, 3).reshape(B * N, D)
    return _cmp("attention", out, ref, 2e-2, 2e-2)


def chk_attention_impls_agree(B, N, heads, grow=False):
    """The two attention kernels are selected by grid size; an image must not change with the batch it is processed in, so
    they have to agree bit for bit (same exponential evaluation per column, same summation order of the row sums)."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(15)
    qkv = torch.randn(B, N, 3, heads, 64, generator=g, device="cuda") * 1.5
    if grow:
        ramp = 1.0 + 7.0 * (torch.arange(N, device="cuda") // 128).float() / max((N - 1) // 128, 1)
        qkv[:, :, 1] *= ramp.view(1, N, 1, 1)
    qkv = qkv.bfloat16()
    a = ops.attention(qkv, B, N, heads, 0)
    worst, n_diff, ok = 0.0, 0, True
    for impl in (1, 2):
        b = ops.attention(qkv, B, N, heads, impl)
        torch.cuda.synchronize()
        diff = (a.float() - b.float()).abs()
        ok = ok and bool(torch.equal(a, b))
        worst = max(worst, diff.max().item())
        n_diff += int((diff > 0).sum().item())
    return {"ok": ok, "max_abs": worst, "n_diff": n_diff, "n": a.numel()}


def chk_layernorm(D, drop):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(6)
    B, n_tok = 3, 50
    x = torch.randn(B * n_tok, D, generator=g, device="cuda") * 2 + 0.5
    w = torch.randn(D, generator=g, device="cuda")
    b = torch.randn(D, generator=g, device="cuda")
    out = ops.layernorm(x, w, b, 1e-6, n_tok, drop)
    torch.cuda.synchronize()
    ref = torch.nn.functional.layer_norm(x, (D,), w, b, 1e-6)
    if drop:
        ref = ref.view(B, n_tok, D)[:, 1:].reshape(-1, D)
    return _cmp("ln", out, ref, 2e-2, 1e-2)


def chk_layernorm_delta():
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(16)
    rows, D = 300, 1024
    x = torch.randn(rows, D, generator=g, device="cuda") * 2
    d = torch.randn(rows, D, generator=g, device="cuda").bfloat16()
    w = torch.randn(D, generator=g, device="cuda")
    b = torch.randn(D, generator=g, device="cuda")
    x1 = x.clone()
    out = ops.layernorm(x1, w, b, 1e-6, 1, False, delta=d, write_x=True)
    x2 = x.clone()
    out2 = ops.layernorm(x2, w, b, 1e-6, 1, False, delta=d, write_x=False)
    torch.cuda.synchronize()
    xs = x + d.float()
    ref = torch.nn.functional.layer_norm(xs, (D,), w, b, 1e-6)
    r = _cmp("ln", out, ref, 2e-2, 1e-2)
    r["x_written"] = bool(torch.equal(x1, xs))
    r["x_untouched"] = bool(torch.equal(x2, x))
    r["ok"] = r["ok"] and r["x_written"] and r["x_untouched"] and bool(torch.equal(out, out2))
    # two pending branches: (x + d) + d2, the order the encoder relies on (norm2 sees x + d, the next norm1 adds d2)
    d2 = torch.randn(rows, D, generator=g, device="cuda").bfloat16()
    x3 = x.clone()
    out3 = ops.layernorm(x3, w, b, 1e-6, 1, False, delta=d, write_x=True, delta2=d2)
    torch.cuda.synchronize()
    xs2 = (x + d.float()) + d2.float()
    r2 = _cmp("ln2", out3, torch.nn.functional.layer_norm(xs2, (D,), w, b, 1e-6), 2e-2, 1e-2)
    r["x_written_2"] = bool(torch.equal(x3, xs2))
    r["ok"] = r["ok"] and r2["ok"] and r["x_written_2"]
    return r


def chk_layernorm_tap():
    """norm1 of the next block and the tap of the previous one in one pass: same statistics, two affines, the second written
    without the cls rows (dinov2.py:337-340)."""
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(26)
    B, n_tok, D = 3, 50, 1024
    x = torch.randn(B * n_tok, D, generator=g, device="cuda") * 2 + 0.3
    d1 = torch.randn(B * n_tok, D, generator=g, device="cuda").bfloat16()
    d2 = torch.randn(B * n_tok, D, generator=g, device="cuda").bfloat16()
    w, b, w2, b2 = (torch.randn(D, generator=g, device="cuda") for _ in range(4))
    x1 = x.clone()
    out, tap = ops.layernorm(x1, w, b, 1e-6, n_tok, False, delta=d1, write_x=True, delta2=d2, tap_w=w2, tap_b=b2)
    torch.cuda.synchronize()
    xs = (x + d1.float()) + d2.float()
    r = _cmp("ln", out, torch.nn.functional.layer_norm(xs, (D,), w, b, 1e-6), 2e-2, 1e-2)
    ref2 = torch.nn.functional.layer_norm(xs, (D,), w2, b2, 1e-6).view(B, n_tok, D)[:, 1:].reshape(-1, D)
    r2 = _cmp("tap", tap, ref2, 2e-2, 1e-2)
    # the separate tap pass (what the last block still uses) must give the same bits
    x2 = x.clone()
    tap_alone = ops.layernorm(x2, w2, b2, 1e-6, n_tok, True, delta=d1, write_x=False, delta2=d2)
    torch.cuda.synchronize()
    r["tap_ok"] = r2["ok"]
    r["tap_same_bits_as_separate_pass"] = bool(torch.equal(tap, tap_alone))
    r["x_written"] = bool(torch.equal(x1, xs))
    r["ok"] = r["ok"] and r2["ok"] and r["tap_same_bits_as_separate_pass"] and r["x_written"]
    return r


def chk_channel_ln(C):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(7)
    x = (torch.randn(2, 9, 11, C, generator=g, device="cuda") * 2 + 0.3).bfloat16()
    w = torch.randn(C, generator=g, device="cuda")
    b = torch.randn(C, generator=g, device="cuda")
    out = ops.channel_ln_relu(x, w, b)
    torch.cuda.synchronize()
    xf = x.float()
    u = xf.mean(-1, keepdim=True)
    s = (xf - u).pow(2).mean(-1, keepdim=True)
    ref = torch.relu((xf - u) / torch.sqrt(s + 1e-6) * w + b)
    return _cmp("cln", out, ref, 2e-2, 1e-2)


def chk_upsample(Hi, Ho, C=64):
    torch, L, ops = _imports()
    g = torch.Generator(device="cuda").manual_seed(8)
    x = torch.randn(2, Hi, Hi, C, generator=g, device="cuda").bfloat16()
    out = ops.upsample(x, Ho, Ho)
    torch.cuda.synchronize()
    ref = torch.nn.functional.interpolate(x.float().permute(0, 3, 1, 2), (Ho, Ho), mode="bilinear", align_corners=True)
    return _cmp("up", out.permute(0, 3, 1, 2), ref, 2e-2, 1e-2)


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
    out = ops.patch_gather(rgb, [m, o], 1024)
    torch.cuda.synchronize()
    mean = torch.tensor([0.485, 0.456, 0.406], device="cuda").view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225], device="cuda").view(1, 3, 1, 1)
    x = torch.cat([(rgb - mean) / std, m, o], 1)
    ref = torch.nn.functional.unfold(x, 14, stride=14).transpose(1, 2).reshape(B * (H // 14) * (W // 14), 5 * 196)
    r = _cmp("gather", out[:, :980], ref, 1e-6, 2 ** -8)
    r["pad_zero"] = bool((out[:, 980:] == 0).all().item())
    r["ok"] = r["ok"] and r["pad_zero"]
    return r


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
    # both attention kernels on every shape (impl 0 = attention.cuh, 1 / 2 = attention2.cuh one / two threads per row), then the auto-selected one
    **{f"attention{i}_small": (lambda i=i: chk_attention(1, 128, 1, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_ragged": (lambda i=i: chk_attention(1, 200, 2, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_1370": (lambda i=i: chk_attention(2, 1370, 6, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_rescale": (lambda i=i: chk_attention(1, 1370, 2, grow=True, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_5477": (lambda i=i: chk_attention(1, 5477, 2, impl=i)) for i in (0, 1, 2)},
    # persistent kernel: several work units per CTA, full (two query tiles) and short (one tile) units interleaved
    **{f"attention{i}_multiunit_1370": (lambda i=i: chk_attention(4, 1370, 16, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_multiunit_300": (lambda i=i: chk_attention(8, 300, 16, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_multiunit_128": (lambda i=i: chk_attention(10, 128, 16, impl=i)) for i in (0, 1, 2)},
    **{f"attention{i}_multiunit_rescale": (lambda i=i: chk_attention(3, 700, 16, grow=True, impl=i)) for i in (0, 1, 2)},
    "attention_auto_b32": lambda: chk_attention(32, 1370, 16),
    "attention_impls_agree_1370": lambda: chk_attention_impls_agree(3, 1370, 16),
    "attention_impls_agree_rescale": lambda: chk_attention_impls_agree(2, 700, 16, grow=True),
    "attention_impls_agree_5477": lambda: chk_attention_impls_agree(1, 5477, 4),
    "layernorm_384": lambda: chk_layernorm(384, False),
    "layernorm_1024_drop": lambda: chk_layernorm(1024, True),
    "layernorm_1536": lambda: chk_layernorm(1536, False),
    "layernorm_delta": chk_layernorm_delta,
    "layernorm_tap_fused": chk_layernorm_tap,
    "channel_ln_48": lambda: chk_channel_ln(48),
    "channel_ln_1024": lambda: chk_channel_ln(1024),
    "upsample_19_37": lambda: chk_upsample(19, 37),
    "upsample_37_74": lambda: chk_upsample(37, 74),
    "upsample_148_296_c256": lambda: chk_upsample(148, 296, 256),
    "upsample_40_70_c128": lambda: chk_upsample(40, 70, 128),   # not a 2x map: strips cross source rows irregularly
    "channel_ln_256": lambda: chk_channel_ln(256),
    "channel_ln_512": lambda: chk_channel_ln(512),
    "channel_ln_1536": lambda: chk_channel_ln(1536),
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

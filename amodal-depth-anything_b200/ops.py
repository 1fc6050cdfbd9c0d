"""Operator-level wrappers over the C ABI, taking torch CUDA tensors. Used by tests/ and tools/ to check each kernel
against the matching torch op, and by the pre/post-processing around the forward (infer.py, DepthAnythingV2.infer_images);
the forward itself (model.py) calls ada_forward directly and does not go through here."""
from __future__ import annotations

import ctypes
import math

import torch

from . import _lib as L


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(t=None):
    """Current stream of the device the operands live on (not of whatever device happens to be current)."""
    dev = t.device if t is not None else None
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _call(t, fn, *args):
    """Runs one C-ABI entry point with `t`'s device current (the library launches on the current device, so an operand on
    cuda:1 while cuda:0 is current must switch first) on that device's current stream."""
    with torch.cuda.device(t.device):
        L.check(fn(*args, _stream(t)))


def gemm(A, Wt, *, epi=L.EPI_BF16, act=L.ACT_NONE, bias=None, gamma=None, resid_f32=None, out_f32=None, out_bf16=None,
         out_relu=None, resid1=None, resid2=None, aux=None, ldo=0, P=0, ks=0, cout=0, sigmoid=0, force_bn=0,
         force_cg=0, conv=None, N=None, K=None, M=None, H=0, W=0, conv_stride=1, conv_taps=9):
    """A: bf16 [M,K] (linear) or NHWC bf16 [B,H,W,Cin] (conv=(B,H,W,Cin)); Wt: bf16 [N,Kw]."""
    lib = L.load()
    d = L.GemmDesc()
    d.A, d.Bw = A.data_ptr(), Wt.data_ptr()
    if conv is not None:
        B_, H_, W_, Cin = conv
        d.a_mode, d.batch, d.H, d.W, d.Cin = L.A_CONV3X3, B_, H_, W_, Cin
        d.M, d.K, d.lda = B_ * H_ * W_, 0, 0
    else:
        d.a_mode = L.A_LINEAR
        d.M = M if M is not None else A.shape[0]
        d.K = K if K is not None else A.shape[1]
        d.lda = A.stride(0)
        d.H, d.W = H, W
    d.N = N if N is not None else Wt.shape[0]
    d.ldb = Wt.stride(0)
    d.epi, d.act = epi, act
    for name, t in (("bias", bias), ("gamma", gamma), ("resid_f32", resid_f32), ("out_f32", out_f32),
                    ("out_bf16", out_bf16), ("out_relu", out_relu), ("resid1", resid1), ("resid2", resid2), ("aux", aux)):
        setattr(d, name, t.data_ptr() if t is not None else None)
    d.ldo, d.P, d.ks, d.cout, d.sigmoid, d.force_bn = ldo, P, ks, cout, sigmoid, force_bn
    d.force_cg = force_cg
    d.conv_stride = conv_stride
    d.conv_taps = conv_taps
    _call(A, lib.ada_op_gemm, ctypes.byref(d))


def layernorm(x, w, b, eps=1e-6, n_tok=0, drop_cls=False, delta=None, write_x=False, delta2=None, tap_w=None, tap_b=None,
              out=None, out2=None):
    """tap_w / tap_b: also return a second affine of the same normalised rows as the cls-less patch map (needs n_tok).
    out / out2: bf16 outputs to store into (allocated when None)."""
    rows, D = x.shape
    out_rows = (rows // n_tok) * (n_tok - 1) if drop_cls else rows
    if out is None:
        out = torch.empty(out_rows, D, dtype=torch.bfloat16, device=x.device)
    assert out.shape == (out_rows, D) and out.dtype == torch.bfloat16 and out.is_contiguous()
    if tap_w is None:
        out2 = None
    else:
        if out2 is None:
            out2 = torch.empty((rows // n_tok) * (n_tok - 1), D, dtype=torch.bfloat16, device=x.device)
        assert out2.shape == ((rows // n_tok) * (n_tok - 1), D) and out2.dtype == torch.bfloat16 and out2.is_contiguous()
    _call(x, L.load().ada_op_layernorm, _p(x), _p(delta), _p(delta2), _p(w), _p(b), _p(out), rows, D, eps, n_tok, int(drop_cls),
          int(write_x), _p(tap_w), _p(tap_b), _p(out2))
    return out if out2 is None else (out, out2)


def attention(qkv, B, N, heads, impl=-1, out=None):
    """impl: -1 = the kernel the model would use at this shape, 0 / 1 / 2 = force attention.cuh / attention2.cuh (one thread per row) / attention2.cuh (two threads per row).
    out: bf16 [B * N, heads * 64] to store into (allocated when None)."""
    if out is None:
        out = torch.empty(B * N, heads * 64, dtype=torch.bfloat16, device=qkv.device)
    assert out.shape == (B * N, heads * 64) and out.dtype == torch.bfloat16 and out.is_contiguous()
    _call(qkv, L.load().ada_op_attention, _p(qkv), _p(out), B, N, heads, impl)
    return out


def channel_ln_relu(x_nhwc, w, b, eps=1e-6, out=None):
    """out: bf16 tensor of x_nhwc's shape to store into (allocated when None; x_nhwc itself is allowed)."""
    C = x_nhwc.shape[-1]
    if out is None:
        out = torch.empty_like(x_nhwc)
    assert out.shape == x_nhwc.shape and out.dtype == torch.bfloat16 and out.is_contiguous()
    _call(x_nhwc, L.load().ada_op_channel_ln_relu, _p(x_nhwc), _p(w), _p(b), _p(out), x_nhwc.numel() // C, C, eps)
    return out


def upsample(x_nhwc, Ho, Wo, out=None):
    """out: bf16 [B, Ho, Wo, C] to store into (allocated when None)."""
    B, Hi, Wi, C = x_nhwc.shape
    if out is None:
        out = torch.empty(B, Ho, Wo, C, dtype=torch.bfloat16, device=x_nhwc.device)
    assert out.shape == (B, Ho, Wo, C) and out.dtype == torch.bfloat16 and out.is_contiguous()
    _call(x_nhwc, L.load().ada_op_upsample, _p(x_nhwc), _p(out), B, Hi, Wi, Ho, Wo, C)
    return out


def patch_gather(rgb, guides, Kpad, out=None):
    """out: bf16 [B * (H // 14) * (W // 14), Kpad] to store into (allocated and zeroed when None); the kernel leaves the
    columns past the patch rows' C * 196 elements as they were."""
    B, _, H, W = rgb.shape
    if out is None:
        out = torch.zeros(B * (H // 14) * (W // 14), Kpad, dtype=torch.bfloat16, device=rgb.device)
    assert out.shape == (B * (H // 14) * (W // 14), Kpad) and out.dtype == torch.bfloat16 and out.is_contiguous()
    n = len(guides)
    ptrs = (ctypes.c_void_p * max(n, 1))(*[g.data_ptr() for g in guides])
    chs = (ctypes.c_int32 * max(n, 1))(*[g.shape[1] for g in guides])
    _call(rgb, L.load().ada_op_patch_gather, _p(rgb), ptrs, chs, n, _p(out), B, H, W, Kpad)
    return out


def pack_conv3x3(w):
    """torch conv weight [Cout,Cin,3,3] fp32 (any device) -> packed bf16 [Cout, 9*round_up(Cin,64)] on cuda."""
    Cout, Cin = w.shape[:2]
    Cpad = (Cin + 63) // 64 * 64
    wh = w.detach().float().cpu().contiguous()
    out = torch.empty(Cout, 9 * Cpad, dtype=torch.bfloat16, device="cuda")
    L.check(L.load().ada_pack_conv3x3(_p(wh), Cout, Cin, _p(out)))
    return out


def pack_convT(w, ks):
    """torch ConvTranspose2d weight [Cin,Cout,ks,ks] -> packed bf16 [ks*ks*Cout, Cin] on cuda."""
    Cin, Cout = w.shape[:2]
    wh = w.detach().float().cpu().contiguous()
    out = torch.empty(ks * ks * Cout, Cin, dtype=torch.bfloat16, device="cuda")
    L.check(L.load().ada_pack_convT(_p(wh), Cin, Cout, ks, _p(out)))
    return out


def pack_tail_taps(w):
    """output_conv2.0 weight [32,Cm,3,3] -> per-tap 1x1 contractions, bf16 [288, Cm] on cuda."""
    Cm = w.shape[1]
    wh = w.detach().float().cpu().contiguous()
    out = torch.empty(288, Cm, dtype=torch.bfloat16, device="cuda")
    L.check(L.load().ada_pack_tail_taps(_p(wh), Cm, _p(out)))
    return out


def tail_gather(V, bias2, aux, H, W, sigmoid=True, out=None):
    """V: NHWC fp16 [B,Hl,Wl,288] -> fp32 [B,H,W] (out: stored into when given)."""
    B, Hl, Wl, _ = V.shape
    if out is None:
        out = torch.empty(B, H, W, dtype=torch.float32, device=V.device)
    assert out.shape == (B, H, W) and out.dtype == torch.float32 and out.is_contiguous()
    _call(V, L.load().ada_op_tail_gather, _p(V), _p(bias2), _p(aux), _p(out), B, Hl, Wl, H, W, int(sigmoid))
    return out


def pack_tail_mma(w):
    """output_conv2.0 weight [32,C,3,3] -> fp16 [3, C/8, 96, 8] on cuda (the B operand of tail_mma_kernel)."""
    C = w.shape[1]
    wh = w.detach().float().cpu().contiguous()
    out = torch.empty(3, C // 8, 96, 8, dtype=torch.float16, device="cuda")
    L.check(L.load().ada_pack_tail_mma(_p(wh), C, _p(out)))
    return out


def tail_mma(Lmap, wpk, bias2, aux, H, W, sigmoid=1, out=None):
    """Lmap: NHWC fp16 [B,Hl,Wl,C] (output_conv1 map) -> fp32 [B,H,W]: upsample + output_conv2 in one kernel (out: stored
    into when given)."""
    B, Hl, Wl, C = Lmap.shape
    if out is None:
        out = torch.empty(B, H, W, dtype=torch.float32, device=Lmap.device)
    assert out.shape == (B, H, W) and out.dtype == torch.float32 and out.is_contiguous()
    _call(Lmap, L.load().ada_op_tail_mma, _p(Lmap), _p(wpk), _p(bias2), _p(aux), _p(out), B, Hl, Wl, H, W, C, int(sigmoid))
    return out


# ---- single-image pre/post-processing of infer.py (include/amodal_b200.h, "row f2")
def image_nearest(img_u8_hwc, H=518, W=518, normalize=False):
    """uint8 [H0,W0,3] (device) -> fp32 [1,3,H,W]; infer.py:84-86 (normalize=True: infer.py:18)."""
    H0, W0, C = img_u8_hwc.shape
    assert C == 3 and img_u8_hwc.dtype == torch.uint8 and img_u8_hwc.is_contiguous()
    out = torch.empty(1, 3, H, W, dtype=torch.float32, device=img_u8_hwc.device)
    _call(img_u8_hwc, L.load().ada_pre_image_nearest, _p(img_u8_hwc), H0, W0, _p(out), H, W, int(normalize))
    return out


def mask_nearest(mask_u8, H=518, W=518):
    """uint8 [H0,W0] (device, non-zero = inside) -> (mask01 [1,1,H,W], guide = mask01*2-1); infer.py:80-87,91,100-101."""
    H0, W0 = mask_u8.shape
    assert mask_u8.dtype == torch.uint8 and mask_u8.is_contiguous()
    m01 = torch.empty(1, 1, H, W, dtype=torch.float32, device=mask_u8.device)
    guide = torch.empty_like(m01)
    _call(mask_u8, L.load().ada_pre_mask_nearest, _p(mask_u8), H0, W0, _p(m01), _p(guide), H, W)
    return m01, guide


def minmax_normalize(depth):
    """fp32 map -> (base01 = (d-min)/(max-min), observation = base01*2-1), same shape; infer.py:22,92."""
    d = depth.contiguous()
    base, obs = torch.empty_like(d), torch.empty_like(d)
    scratch = torch.empty(2, dtype=torch.int32, device=d.device)
    _call(d, L.load().ada_post_minmax_normalize, _p(d), d.numel(), _p(base), _p(obs), _p(scratch))
    return base, obs


def blend_seam(raw01, amodal, mask01):
    """infer.py:30-44 median_filter_blend(amodal, raw, mask, 3) on [H,W] fp32 device maps."""
    H, W = raw01.shape[-2:]
    out = torch.empty(H, W, dtype=torch.float32, device=raw01.device)
    _call(raw01, L.load().ada_post_blend_seam, _p(raw01.contiguous()), _p(amodal.contiguous()), _p(mask01.contiguous()), _p(out), H, W)
    return out


# ---- the same pre/post-processing over a batch (include/amodal_b200.h, ada_*_batch): images of any size packed into one
#      uint8 device buffer, located by a descriptor table, int64 [B, 3] rows of {byte offset, H0, W0} (ada_img_desc)
def pack_layout(shapes, start=0):
    """Descriptor rows placing uint8 arrays of the given shapes ([H0, W0] or [H0, W0, C]) one after another from byte
    `start`, each at a 16-byte boundary. Returns (rows, end byte)."""
    rows, off = [], start
    for shp in shapes:
        off = (off + 15) // 16 * 16
        rows.append((off, shp[0], shp[1]))
        off += math.prod(shp)
    return rows, off


class Staging:
    """Reused pinned host buffers for one packed uint8 upload and its int64 [n, 3] descriptor table. A stage waits only
    for the previous upload from the buffers (its copies may still be reading them), then makes one H2D copy of each on
    the current stream."""

    def __init__(self, device):
        self.device = device
        self._data = None
        self._desc = None
        self._uploaded = None    # event after the last upload from the buffers (they are rewritten after it)

    def upload(self, end, rows, fill):
        """fill(host) writes the packed bytes into `host`, a uint8 numpy array of `end` bytes; rows are the descriptor
        rows. Returns (data uint8 [end], desc int64 [len(rows), 3]) on the device."""
        if self._uploaded is not None:
            self._uploaded.synchronize()
        if self._data is None or self._data.numel() < end:
            self._data = torch.empty(end, dtype=torch.uint8, pin_memory=True)
        if self._desc is None or self._desc.shape[0] < len(rows):
            self._desc = torch.empty(len(rows), 3, dtype=torch.int64, pin_memory=True)
        fill(self._data.numpy()[:end])
        self._desc.numpy()[:len(rows)] = rows
        data = torch.empty(end, dtype=torch.uint8, device=self.device)
        desc = torch.empty(len(rows), 3, dtype=torch.int64, device=self.device)
        data.copy_(self._data[:end], non_blocking=True)
        desc.copy_(self._desc[:len(rows)], non_blocking=True)
        self._uploaded = torch.cuda.Event()
        self._uploaded.record()
        return data, desc


def _desc(src, desc):
    assert src.dtype == torch.uint8 and src.is_contiguous()
    assert desc.dtype == torch.int64 and desc.dim() == 2 and desc.shape[1] == 3 and desc.is_contiguous()
    assert desc.device == src.device
    return desc.shape[0]


def _out(out, shape, dtype, device):
    if out is None:
        return torch.empty(shape, dtype=dtype, device=device)
    assert tuple(out.shape) == tuple(shape) and out.dtype == dtype and out.is_contiguous()
    return out


def resize_linear_batch(src_u8, desc, H=518, W=518, out=None):
    """cv2.resize(img, (W, H)) (INTER_LINEAR, infer.py:17) of each 3-channel image of the packed buffer, bit-exact ->
    uint8 [B,H,W,3]."""
    B = _desc(src_u8, desc)
    out = _out(out, (B, H, W, 3), torch.uint8, src_u8.device)
    _call(src_u8, L.load().ada_pre_resize_linear_batch, _p(src_u8), _p(desc), B, _p(out), H, W)
    return out


def image_nearest_batch(src_u8, desc, H=518, W=518, normalize=False, out=None):
    """image_nearest of each 3-channel image of the packed buffer -> fp32 [B,3,H,W]."""
    B = _desc(src_u8, desc)
    out = _out(out, (B, 3, H, W), torch.float32, src_u8.device)
    _call(src_u8, L.load().ada_pre_image_nearest_batch, _p(src_u8), _p(desc), B, _p(out), H, W, int(normalize))
    return out


def mask_nearest_batch(src_u8, desc, H=518, W=518, mask01=None, guide=None):
    """mask_nearest of each mask of the packed buffer -> (mask01 [B,1,H,W], guide [B,1,H,W])."""
    B = _desc(src_u8, desc)
    mask01 = _out(mask01, (B, 1, H, W), torch.float32, src_u8.device)
    guide = _out(guide, (B, 1, H, W), torch.float32, src_u8.device)
    _call(src_u8, L.load().ada_pre_mask_nearest_batch, _p(src_u8), _p(desc), B, _p(mask01), _p(guide), H, W)
    return mask01, guide


def minmax_normalize_batch(depth):
    """minmax_normalize of each depth[b] (min and max per map) -> (base01, observation), depth's shape."""
    d = depth.contiguous()
    B = d.shape[0]
    base, obs = torch.empty_like(d), torch.empty_like(d)
    scratch = torch.empty(2 * B, dtype=torch.int32, device=d.device)
    _call(d, L.load().ada_post_minmax_normalize_batch, _p(d), B, d.numel() // B, _p(base), _p(obs), _p(scratch))
    return base, obs


def blend_seam_batch(raw01, amodal, mask01):
    """blend_seam of each map: raw01 / amodal / mask01 [B,H,W] (or [B,1,H,W]) -> [B,H,W]."""
    B = raw01.shape[0]
    H, W = raw01.shape[-2:]
    raw01, amodal, mask01 = raw01.contiguous(), amodal.contiguous(), mask01.contiguous()
    assert raw01.numel() == amodal.numel() == mask01.numel() == B * H * W
    out = torch.empty(B, H, W, dtype=torch.float32, device=raw01.device)
    _call(raw01, L.load().ada_post_blend_seam_batch, _p(raw01), _p(amodal), _p(mask01), _p(out), B, H, W)
    return out


def resize_cubic_normalize_batch(src_u8, desc, H, W, out=None):
    """DepthAnythingV2.image2tensor of each 3-channel BGR image of the packed buffer at (H, W), bit-exact (cv2's float64
    INTER_CUBIC, then the ImageNet normalise in float64) -> fp32 [B,3,H,W]."""
    B = _desc(src_u8, desc)
    out = _out(out, (B, 3, H, W), torch.float32, src_u8.device)
    _call(src_u8, L.load().ada_pre_resize_cubic_normalize_batch, _p(src_u8), _p(desc), B, _p(out), H, W)
    return out


def upsample_restore_batch(depth, out_desc, out):
    """Bilinear (align_corners=True) of each map of depth [B,H,W] fp32 to its own size, into the fp32 buffer `out`: row b
    of out_desc (int64 [B, 3] device rows of ada_img_desc) holds map b's byte offset into `out` and its (h, w)."""
    assert depth.dtype == torch.float32 and depth.dim() == 3 and depth.is_contiguous()
    assert out.dtype == torch.float32 and out.is_contiguous() and out.device == depth.device
    assert out_desc.dtype == torch.int64 and out_desc.shape == (depth.shape[0], 3) and out_desc.is_contiguous()
    assert out_desc.device == depth.device
    B, H, W = depth.shape
    _call(depth, L.load().ada_post_upsample_restore_batch, _p(depth), B, H, W, _p(out_desc), _p(out))
    return out


# ---- per-sample evaluation post-ops of the validation loop (include/amodal_b200.h, "row f3")
EVAL_METRICS = ("abs_relative_difference", "squared_relative_difference", "rmse_linear", "rmse_log", "log10", "delta1_acc",
                "delta2_acc", "delta3_acc", "i_rmse", "silog_rmse")  # config eval.eval_metrics order


def eval_sample(pred, depth_gt, depth_obs, visible_mask, object_mask):
    """pred [.., h, w] fp32 (network output), depth_gt / depth_obs [H, W] fp32, masks [H, W] bool/uint8, all on the device.
    Returns a [24] float64 device tensor (layout in include/amodal_b200.h); no host synchronisation."""
    h, w = pred.shape[-2:]
    H, W = depth_gt.shape[-2:]
    out = torch.empty(24, dtype=torch.float64, device=pred.device)
    scratch = torch.empty(26, dtype=torch.float64, device=pred.device)
    vis = visible_mask.to(torch.uint8).contiguous()
    obj = object_mask.to(torch.uint8).contiguous()
    _call(pred, L.load().ada_eval_sample, _p(pred.contiguous()), h, w, _p(depth_gt.contiguous()), _p(depth_obs.contiguous()), _p(vis),
                                     _p(obj), H, W, _p(out), _p(scratch))
    return out


def eval_batch(pred, src_u8, desc, out=None):
    """ada_eval_batch: the eval_sample post-ops of B samples of any sizes in one launch. pred: fp32 device tensor holding
    every sample's [h, w] prediction; src_u8: uint8 device buffer holding their ground-truth maps; desc: int64 [B, 9]
    device rows of ada_eval_desc (element offset into pred, byte offsets of depth_gt, depth_obs, visible, object into src,
    then h, w, H, W). Returns [B, 24] float64 (row b bit-equal to eval_sample on sample b); no host synchronisation."""
    assert pred.dtype == torch.float32 and pred.is_contiguous() and src_u8.dtype == torch.uint8 and src_u8.is_contiguous()
    assert desc.dtype == torch.int64 and desc.dim() == 2 and desc.shape[1] == 9 and desc.is_contiguous()
    assert pred.device == src_u8.device == desc.device
    B = desc.shape[0]
    out = _out(out, (B, 24), torch.float64, pred.device)
    _call(pred, L.load().ada_eval_batch, _p(pred), _p(src_u8), _p(desc), B, _p(out))
    return out


def eval_accumulate(rows, bucket, n_buckets, acc):
    """ada_eval_accumulate: acc [(n_buckets + 1), 22] float64 (row 0 overall, 1 + k bucket k: n_used, n_skipped, 20 metric
    sums) += the [B, 24] rows, in row order; bucket: int32 [B] device labels or None (overall only)."""
    assert rows.dtype == torch.float64 and rows.dim() == 2 and rows.shape[1] == 24 and rows.is_contiguous()
    assert acc.dtype == torch.float64 and acc.numel() == (n_buckets + 1) * 22 and acc.is_contiguous()
    if bucket is not None:
        assert bucket.dtype == torch.int32 and bucket.numel() == rows.shape[0] and bucket.is_contiguous()
    _call(rows, L.load().ada_eval_accumulate, _p(rows), rows.shape[0], _p(bucket), n_buckets, _p(acc))
    return acc


def eval_sample_dict(out24):
    """One host read of the 24 numbers -> {'scale', 'shift', 'pred': {metric: value}, 'aligned': {...}}."""
    v = out24.cpu().tolist()
    return {"scale": v[0], "shift": v[1], "pred": dict(zip(EVAL_METRICS, v[2:12])), "aligned": dict(zip(EVAL_METRICS, v[12:22])),
            "n_visible": int(v[22]), "n_object": int(v[23])}

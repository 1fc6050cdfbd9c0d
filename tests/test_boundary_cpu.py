"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol of include/amodal_b200.h,
and the Python model class keeps the reference's construction / state-dict / error contract (SURVEY.md section 8b).
No kernel is launched here."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import amodal_depth_anything_b200 as pkg
from amodal_depth_anything_b200 import _lib as L
from oracle import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    hdr = open(os.path.join(ROOT, "include", "amodal_b200.h")).read()
    declared = set(re.findall(r"\b(ada_[A-Za-z0-9_]+)\s*\(", hdr))
    declared -= {"ada_model"}
    assert declared, "no declarations parsed"
    lib = L.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(L.SIGNATURES), (declared ^ set(L.SIGNATURES))


def test_no_cpu_fallback_in_c_abi():
    """On a box without a GPU every compute entry point must fail loudly (ADA_ENODEVICE), never compute on the host. Runs
    in a child process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), so it holds on GPU machines too."""
    code = f"""
import sys
sys.path.insert(0, {ROOT!r})
from amodal_depth_anything_b200 import _lib as L
lib = L.load()
rc = lib.ada_op_layernorm(None, None, None, None, None, None, 1, 384, 1e-6, 1, 0, 0, None, None, None, None)
assert rc == L.ADA_ENODEVICE, rc
assert b"CUDA" in lib.ada_last_error() or b"device" in lib.ada_last_error(), lib.ada_last_error()
"""
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]


@pytest.mark.parametrize("enc,gt", [("vits", "mask+observation"), ("vitb", "image+mask+observation"), ("vits", "none")])
def test_state_dict_keys_match_reference_template(enc, gt):
    m = pkg.AmodalDAv2(guide_type=gt, encoder=enc, pretrained=False)
    want = synth.state_dict_shapes(enc, gt)
    got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert got == dict(want)
    assert "pixel_mean" not in got  # non-persistent buffers (dav2.py:50-51)
    m.load_state_dict(synth.make_state_dict(enc, gt, 0), strict=True)


def test_guidance_conv_zero_init_and_vitg_supported():
    m = pkg.AmodalDAv2(guide_type="mask+observation", encoder="vits", pretrained=False)
    sd = m.state_dict()
    assert sd["encoder.pretrained.patch_embed_guidance.proj.weight"].abs().max() == 0  # dav2.py:55-61
    assert sd["encoder.pretrained.blocks.0.ls1.gamma"].min() == 1.0
    assert len(synth.state_dict_shapes("vitg", "mask+observation")) == 649
    assert pkg.MODEL_CONFIGS["vitg"]["features"] == 384


def test_error_conventions():
    with pytest.raises(KeyError):
        pkg.AmodalDAv2(encoder="vitx")
    with pytest.raises(NotImplementedError):
        pkg.AmodalDAv2(encoder="vits", guide_type="bogus")
    m = pkg.get_model("AmodalDAv2", guide_type="mask+observation", encoder="vits", pretrained=False)
    x = torch.rand(1, 3, 28, 28)
    with pytest.raises(RuntimeError, match="inference-only"):
        m.train()(x, guide_mask=x[:, :1], observation=x[:, :1])
    m.eval()
    with pytest.raises(TypeError):
        m(x, guide_mask=None, observation=x[:, :1])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(x, guide_mask=x[:, :1], observation=x[:, :1])
    with pytest.raises(KeyError):
        pkg.get_model("ADDeepLab")


def test_save_and_from_pretrained_roundtrip(tmp_path):
    m = pkg.AmodalDAv2(guide_type="mask", loss_stategy="ssi", encoder="vits", pretrained=False)
    m.load_state_dict(synth.make_state_dict("vits", "mask", 3), strict=True)
    m.save_pretrained(tmp_path)
    assert (tmp_path / "model.safetensors").exists() and (tmp_path / "config.json").exists()
    m2 = pkg.AmodalDAv2.from_pretrained(str(tmp_path), strict=True)
    assert m2.guide_type == "mask" and m2.loss_stategy == "ssi" and m2.encoder_name == "vits"
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_pos_embed_interpolation_host_matches_reference_formula():
    """ada_interp_pos_embed_host runs on the CPU inside the .so; compare with the oracle's interpolate_pos_encoding
    (dinov2.py:199-230: bicubic with scale_factor=(h+0.1)/37, NOT size=) incl. a non-square grid."""
    from oracle.amodal_oracle import interpolate_pos_encoding
    lib = L.load()
    D = 16
    g = torch.Generator().manual_seed(0)
    pos = torch.randn(1, 1 + 37 * 37, D, generator=g)
    for gh, gw in [(74, 74), (9, 7), (5, 5), (40, 37)]:
        ref = interpolate_pos_encoding(pos, gh * gw, gh * 14, gw * 14)[0, 1:]
        src = pos[0, 1:].contiguous()
        out = torch.empty(gh * gw, D)
        rc = lib.ada_interp_pos_embed_host(ctypes.c_void_p(src.data_ptr()), 37, D, gh, gw, 0.1, ctypes.c_void_p(out.data_ptr()))
        assert rc == 0
        assert (out - ref).abs().max().item() < 1e-4, (gh, gw)  # N(0,1) table; size= variant would differ by ~0.4


def test_conv_pixel_tile_shapes_minimise_padding():
    """ada_conv_tile_shape (host only): the M tile of an implicit-GEMM conv is 2^lw x 2^lh pixels x 2^lb images. For every
    map size of the BASELINE configurations and a sweep of odd sizes / batches: 128 rows per tile, a width an epilogue
    warp's 32 rows divide into whole tile rows, never more padded pixels than the fixed 16 x 8 x 1 tile, and the padded
    count it reports is the one its shape implies. Known answers for the batch-32 ViT-L maps (DESIGN.md section 3.1)."""
    lib = L.load()

    def shape(B, H, W, pair=1):
        out = (ctypes.c_int64 * 4)()
        assert lib.ada_conv_tile_shape(B, H, W, pair, out) == 0
        return tuple(int(v) for v in out)

    def padded(B, H, W, pair, lw, lh, lb):
        tw, th, nb = (1 << lw) * pair, 1 << lh, 1 << lb
        return -(-W // tw) * tw * (-(-H // th) * th) * (-(-B // nb) * nb)

    sizes = [296, 148, 74, 37, 19, 592, 10, 11, 22, 44, 5, 1, 76, 38, 49, 98, 100]
    for B in (1, 2, 3, 4, 5, 7, 8, 32, 33):
        for H in sizes:
            for W in (H, max(1, H - 3), H + 12):
                for pair in (1, 2):
                    lw, lh, lb, pad = shape(B, H, W, pair)
                    assert lw + lh + lb == 7 and 1 <= lw <= 5 and lh >= 0 and lb >= 0, (B, H, W, pair)
                    assert pad == padded(B, H, W, pair, lw, lh, lb), (B, H, W, pair)
                    assert pad <= padded(B, H, W, pair, 4, 3, 0), (B, H, W, pair)
                    assert pad >= B * H * W
    assert shape(32, 148, 148)[3] == 32 * 148 * 148 and shape(32, 74, 74)[3] == 32 * 74 * 74
    assert shape(32, 296, 296)[3] == 32 * 296 * 296
    assert shape(32, 37, 37)[3] == 32 * 38 * 38 and shape(32, 19, 19)[3] == 32 * 20 * 19
    assert shape(1, 37, 37)[2] == 0 or shape(1, 37, 37)[3] < padded(1, 37, 37, 1, 4, 3, 0)  # one image: no batch padding wins
    assert lib.ada_conv_tile_shape(0, 1, 1, 1, (ctypes.c_int64 * 4)()) != 0                  # ADA_EINVAL, not a crash


def test_unguided_model_mirrors_reference_class():
    """pkg.DepthAnythingV2 = depth_anything_v2_raw/dpt.py:154-187 (the observation model of infer.py:59-61): state-dict
    template without `encoder.` prefix, guidance or input_projection; same error conventions as AmodalDAv2."""
    m = pkg.DepthAnythingV2(encoder="vits", features=64, out_channels=[48, 96, 192, 384])
    want = {k[len("encoder."):]: v for k, v in
            synth.state_dict_shapes("vits", "none", 64, [48, 96, 192, 384], input_projection=False).items()}
    got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    assert got == want and not any("input_projection" in k or "guidance" in k for k in got)
    m.load_state_dict(synth.make_state_dict_raw("vits", 64, [48, 96, 192, 384], 1), strict=True)
    big = synth.state_dict_shapes("vitg", "none", 384, [1536] * 4, input_projection=False)   # infer.py:59
    assert big["encoder.depth_head.scratch.layer1_rn.weight"] == (384, 1536, 3, 3)
    with pytest.raises(KeyError):
        pkg.DepthAnythingV2(encoder="vitx")
    with pytest.raises(NotImplementedError):
        pkg.DepthAnythingV2(encoder="vits", use_clstoken=True)
    x = torch.rand(1, 3, 28, 28)
    with pytest.raises(RuntimeError, match="inference-only"):
        m.train()(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.eval()(x)
    # Resize(keep_aspect_ratio, lower_bound, multiple of 14) of util/transform.py:52-102, values from the reference class
    for hw, want_hw in (((480, 640), (518, 686)), ((1000, 518), (994, 518)), ((300, 900), (518, 1554)),
                        ((777, 333), (1204, 518)), ((1080, 1920), (518, 924))):
        assert pkg.DepthAnythingV2._input_size(*hw) == want_hw


def _tiny_cfg():
    cfg = L.AdaConfig()
    cfg.embed_dim, cfg.depth, cfg.num_heads, cfg.ffn_kind, cfg.ffn_hidden = 384, 12, 6, 0, 1536
    cfg.taps = (ctypes.c_int32 * 4)(2, 5, 8, 11)
    cfg.features = 64
    cfg.out_channels = (ctypes.c_int32 * 4)(48, 96, 192, 384)
    cfg.guide_channels, cfg.sigmoid, cfg.pos_grid, cfg.interpolate_offset = 2, 1, 37, 0.1
    cfg.input_projection, cfg.normalize_input = 1, 1
    return cfg


def test_set_weight_is_strict_and_finalize_lists_missing_keys():
    """ABI contract of include/amodal_b200.h (== load_state_dict(strict=True)): unknown keys and wrong shapes are rejected
    with ADA_EINVAL, an incomplete state dict fails ada_finalize with ADA_ESTATE naming the missing tensors. Host-only:
    no kernel is launched, so this runs on the build box."""
    lib = L.load()
    h = ctypes.c_void_p()
    assert lib.ada_create(ctypes.byref(_tiny_cfg()), ctypes.byref(h)) == 0
    try:
        w = torch.zeros(384)
        shp = (ctypes.c_int64 * 1)(384)
        assert lib.ada_set_weight(h, b"pretrained.norm.weight", ctypes.c_void_p(w.data_ptr()), shp, 1) == 0
        rc = lib.ada_set_weight(h, b"pretrained.norm.wieght", ctypes.c_void_p(w.data_ptr()), shp, 1)
        assert rc == L.ADA_EINVAL and b"unknown weight key" in lib.ada_last_error()
        rc = lib.ada_set_weight(h, b"pretrained.blocks.12.norm1.weight", ctypes.c_void_p(w.data_ptr()), shp, 1)  # depth is 12
        assert rc == L.ADA_EINVAL
        bad = (ctypes.c_int64 * 1)(383)
        rc = lib.ada_set_weight(h, b"pretrained.norm.bias", ctypes.c_void_p(w.data_ptr()), bad, 1)
        assert rc == L.ADA_EINVAL and b"shape mismatch" in lib.ada_last_error()
        rc = lib.ada_finalize(h)
        assert rc == L.ADA_ESTATE
        msg = lib.ada_last_error().decode()
        n_expected = len(synth.state_dict_shapes("vits", "mask+observation"))
        assert f"{n_expected - 1} of {n_expected} tensors were never set" in msg, msg
        assert "depth_head.projects.0.bias" in msg and "pretrained.norm.weight" not in msg
    finally:
        lib.ada_destroy(h)


def _cfg_for(enc, gt, ip):
    c = pkg.MODEL_CONFIGS[enc]
    cfg = L.AdaConfig()
    cfg.embed_dim, cfg.depth, cfg.num_heads = c["embed_dim"], c["depth"], c["num_heads"]
    cfg.ffn_kind, cfg.ffn_hidden = (0 if c["ffn"] == "mlp" else 1), c["hidden"]
    cfg.taps = (ctypes.c_int32 * 4)(*c["taps"])
    cfg.features = c["features"]
    cfg.out_channels = (ctypes.c_int32 * 4)(*c["out_channels"])
    cfg.guide_channels, cfg.sigmoid, cfg.pos_grid, cfg.interpolate_offset = pkg.GUIDE_CHANNELS[gt], 1, 37, 0.1
    cfg.input_projection, cfg.normalize_input = int(ip), 1
    return cfg


@pytest.mark.parametrize("enc,gt,ip", [("vits", "mask+observation", True), ("vitb", "none", False),
                                       ("vitg", "image+mask+observation", True)])
def test_expected_weight_table_equals_reference_state_dict(enc, gt, ip):
    """The library's own table of expected tensors (csrc/ada_api.cu expected_weights) equals the reference state dict for
    guided / un-guided heads and the Mlp / SwiGLU encoders: every reference key is known with the reference shape, and a
    complete state dict leaves nothing missing (finalize then only fails for want of a device on the build box)."""
    lib = L.load()
    h = ctypes.c_void_p()
    assert lib.ada_create(ctypes.byref(_cfg_for(enc, gt, ip)), ctypes.byref(h)) == 0
    full = enc != "vitg"  # ViT-G: 5.4 GB of fp32 -- probe keys and shapes without staging the data
    try:
        dummy = torch.zeros(4)
        for k, shp in synth.state_dict_shapes(enc, gt, input_projection=ip).items():
            key = k[len("encoder."):].encode()
            if full:
                t = torch.zeros(shp)
                arr = (ctypes.c_int64 * len(shp))(*shp)
                assert lib.ada_set_weight(h, key, ctypes.c_void_p(t.data_ptr()), arr, len(shp)) == 0, (k, lib.ada_last_error())
            else:  # a wrong shape is refused before any byte is read; the message carries the expected shape
                arr = (ctypes.c_int64 * 1)(3)
                assert lib.ada_set_weight(h, key, ctypes.c_void_p(dummy.data_ptr()), arr, 1) == L.ADA_EINVAL
                msg = lib.ada_last_error().decode()
                assert "shape mismatch" in msg and "expected [" + "".join(f"{v}," for v in shp) + "]" in msg, (k, msg)
        if full:
            assert lib.ada_finalize(h) in (0, L.ADA_ENODEVICE), lib.ada_last_error()
    finally:
        lib.ada_destroy(h)


def test_model_copies_do_not_share_the_native_handle():
    """copy / deepcopy / pickle of the module (EMA copies, torch.save(model)) carry parameters only; the ctypes handle is
    dropped and rebuilt lazily by the copy (ADVICE r1: a shared handle would be destroyed twice)."""
    import copy
    import io
    m = pkg.AmodalDAv2(guide_type="mask", encoder="vits", pretrained=False)
    m._handle, m._handle_device, m._dirty = ctypes.c_void_p(1234), torch.device("cpu"), False  # stand-in for a live handle
    try:
        for c in (copy.copy(m), copy.deepcopy(m)):
            assert c._handle is None and c._dirty and c._handle_device is None
            assert torch.equal(c.state_dict()["encoder.pretrained.pos_embed"], m.state_dict()["encoder.pretrained.pos_embed"])
        buf = io.BytesIO()
        torch.save(m, buf)
        buf.seek(0)
        m2 = torch.load(buf, weights_only=False)
        assert m2._handle is None and m2._dirty
    finally:
        m._handle = None

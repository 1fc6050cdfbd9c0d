"""Drop-in for the reference model class `AmodalDAv2` (src/models/amodalsynthdrive/dav2.py:21-90) whose forward runs
entirely in libamodal_b200.so (hand-written sm_100a kernels) through the C ABI of include/amodal_b200.h.

Kept from the reference (SURVEY.md section 8b): constructor kwargs, `forward(x, guide_rgb, guide_mask, observation)`,
nn.Module + PyTorchModelHubMixin behaviour (`from_pretrained`, `save_pretrained` -> model.safetensors + config.json),
state-dict keys/shapes (strict loading), error conventions. Differences, all deliberate:
  * inference only: calling the model in .train() mode raises (the trainer toggles modes; training is out of scope);
  * CUDA only: non-CUDA inputs raise -- there is no CPU fallback;
  * `encoder='vitg'` works (the reference's table lacks it and raises KeyError, dav2.py:31-34; head sizes from infer.py:60).
torch is used for parameter storage, device memory and the current stream only.
"""
from __future__ import annotations

import ctypes
import math

import numpy as np
import torch
import torch.nn as nn
from huggingface_hub import PyTorchModelHubMixin
from huggingface_hub.constants import SAFETENSORS_SINGLE_FILE

from . import _lib as L
from . import ops

# dav2.py:31-34 (+ vitg), dpt.py:213-218, dinov2.py:366-427, swiglu_ffn.py:57
MODEL_CONFIGS = {
    "vits": dict(embed_dim=384, depth=12, num_heads=6, ffn="mlp", hidden=1536, taps=[2, 5, 8, 11], features=64,
                 out_channels=[48, 96, 192, 384]),
    "vitb": dict(embed_dim=768, depth=12, num_heads=12, ffn="mlp", hidden=3072, taps=[2, 5, 8, 11], features=128,
                 out_channels=[96, 192, 384, 768]),
    "vitl": dict(embed_dim=1024, depth=24, num_heads=16, ffn="mlp", hidden=4096, taps=[4, 11, 17, 23], features=256,
                 out_channels=[256, 512, 1024, 1024]),
    "vitg": dict(embed_dim=1536, depth=40, num_heads=24, ffn="swiglu", hidden=4096, taps=[9, 19, 29, 39], features=384,
                 out_channels=[1536, 1536, 1536, 1536]),
}
GUIDE_CHANNELS = {"image+mask+observation": 5, "image+mask": 4, "image+observation": 4, "mask+observation": 2,
                  "mask": 1, "observation": 1, "none": 0}  # dinov2.py:110-125
POS_GRID = 37


class _Tree(nn.Module):
    """A bare parameter container; sub-trees and parameters are attached by dotted name so that state_dict() keys are
    exactly the reference's (e.g. pretrained.blocks.3.attn.qkv.weight)."""

    def put(self, dotted: str, tensor: torch.Tensor):
        head, _, rest = dotted.partition(".")
        if not rest:
            self.register_parameter(head, nn.Parameter(tensor))
            return
        if head not in self._modules:
            self.add_module(head, _Tree())
        self._modules[head].put(rest, tensor)


def _param_table(cfg, guide_type, input_projection=True):
    """(name, shape, init-kind) for every tensor under `encoder.` in reference order of construction.
    input_projection=False gives the un-guided DepthAnythingV2 of depth_anything_v2_raw/dpt.py (no guidance embed, no
    input_projection levels)."""
    D, F, C = cfg["embed_dim"], cfg["features"], cfg["out_channels"]
    t = []
    p = "pretrained."
    t += [(p + "cls_token", (1, 1, D), "cls"), (p + "pos_embed", (1, 1 + POS_GRID * POS_GRID, D), "trunc"),
          (p + "mask_token", (1, D), "zeros"),
          (p + "patch_embed.proj.weight", (D, 3, 14, 14), "conv"), (p + "patch_embed.proj.bias", (D,), "convb:588")]
    cg = GUIDE_CHANNELS[guide_type]
    if cg:  # zero-initialised by the wrapper, dav2.py:55-61
        t += [(p + "patch_embed_guidance.proj.weight", (D, cg, 14, 14), "zeros"),
              (p + "patch_embed_guidance.proj.bias", (D,), "zeros")]
    for i in range(cfg["depth"]):
        b = p + f"blocks.{i}."
        t += [(b + "norm1.weight", (D,), "ones"), (b + "norm1.bias", (D,), "zeros"),
              (b + "attn.qkv.weight", (3 * D, D), "trunc"), (b + "attn.qkv.bias", (3 * D,), "zeros"),
              (b + "attn.proj.weight", (D, D), "trunc"), (b + "attn.proj.bias", (D,), "zeros"),
              (b + "ls1.gamma", (D,), "ones"),
              (b + "norm2.weight", (D,), "ones"), (b + "norm2.bias", (D,), "zeros")]
        Hd = cfg["hidden"]
        if cfg["ffn"] == "mlp":
            t += [(b + "mlp.fc1.weight", (Hd, D), "trunc"), (b + "mlp.fc1.bias", (Hd,), "zeros"),
                  (b + "mlp.fc2.weight", (D, Hd), "trunc"), (b + "mlp.fc2.bias", (D,), "zeros")]
        else:
            t += [(b + "mlp.w12.weight", (2 * Hd, D), "trunc"), (b + "mlp.w12.bias", (2 * Hd,), "zeros"),
                  (b + "mlp.w3.weight", (D, Hd), "trunc"), (b + "mlp.w3.bias", (D,), "zeros")]
        t += [(b + "ls2.gamma", (D,), "ones")]
    t += [(p + "norm.weight", (D,), "ones"), (p + "norm.bias", (D,), "zeros")]
    h = "depth_head."

    def conv(name, cout, cin, k, bias=True):
        r = [(h + name + ".weight", (cout, cin, k, k), "conv")]
        if bias:
            r.append((h + name + ".bias", (cout,), f"convb:{cin * k * k}"))
        return r
    for i in range(4):
        t += conv(f"projects.{i}", C[i], D, 1)
    t += conv("resize_layers.0", C[0], C[0], 4) + conv("resize_layers.1", C[1], C[1], 2) + conv("resize_layers.3", C[3], C[3], 3)
    for i in range(4):
        t += conv(f"scratch.layer{i + 1}_rn", F, C[i], 3, bias=False)
    for k in range(1, 5):
        r = f"scratch.refinenet{k}."
        t += conv(r + "out_conv", F, F, 1)
        for u in (1, 2):
            for cv in (1, 2):
                t += conv(r + f"resConfUnit{u}.conv{cv}", F, F, 3)
    t += conv("scratch.output_conv1", F // 2, F, 3) + conv("scratch.output_conv2.0", 32, F // 2, 3)
    t += conv("scratch.output_conv2.2", 1, 32, 1)
    for i in range(4 if input_projection else 0):
        t += conv(f"input_projection.{i}.0", C[i], C[i], 3)
        t += [(h + f"input_projection.{i}.1.weight", (C[i],), "ones"), (h + f"input_projection.{i}.1.bias", (C[i],), "zeros")]
    return t


def _init(shape, kind):
    """Mirrors the reference's initialisation: trunc_normal(.02) Linears / pos_embed (dinov2.py:193,359-364),
    cls ~ N(0,1e-6) (dinov2.py:194), torch-default convs, LayerScale 1.0 (dinov2.py:440), LN (1, 0)."""
    if kind == "zeros":
        return torch.zeros(shape)
    if kind == "ones":
        return torch.ones(shape)
    if kind == "cls":
        return torch.randn(shape) * 1e-6
    if kind == "trunc":
        return nn.init.trunc_normal_(torch.empty(shape), std=0.02)
    if kind == "conv":
        w = torch.empty(shape)
        nn.init.kaiming_uniform_(w, a=math.sqrt(5))
        return w
    if kind.startswith("convb:"):
        bound = 1.0 / math.sqrt(int(kind.split(":")[1]))
        return torch.empty(shape).uniform_(-bound, bound)
    raise ValueError(kind)


class _NativeModel(nn.Module):
    """Weight ownership + handle management shared by the two model classes: parameters live in torch (so .cuda(),
    state_dict(), from_pretrained work as in the reference); a C-ABI handle holding the packed bf16 copies is (re)built
    lazily whenever the parameters may have changed."""

    def _native_init(self):
        self._handle = None
        self._handle_device = None
        self._dirty = True

    # ---- subclass contract
    def _native_config(self) -> dict:  # keys of L.AdaConfig
        raise NotImplementedError

    def _native_state(self) -> dict:   # reference keys relative to the inner net ("pretrained.*", "depth_head.*")
        raise NotImplementedError

    # ------------------------------------------------------------------ weight ownership / repacking
    def _apply(self, fn, *a, **k):
        self._dirty = True
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._dirty = True
        return super().load_state_dict(*a, **k)

    def repack(self):
        """Call after mutating parameters in place; .to()/.cuda()/load_state_dict() do it automatically."""
        self._dirty = True

    def _release(self):
        if self._handle is not None:
            L.load().ada_destroy(self._handle)
            self._handle = None

    # The C handle (a ctypes pointer to device-side packed weights) never travels with a copy of the module: copy.copy /
    # copy.deepcopy / pickle / torch.save(model) get the parameters only and the copy lazily builds its own handle on its
    # first forward -- as the reference nn.Module, which is freely copied for EMA or replica purposes.
    def __getstate__(self):
        state = self.__dict__.copy()
        state["_handle"] = None
        state["_handle_device"] = None
        state["_dirty"] = True
        state.pop("_staging", None)   # DepthAnythingV2.infer_images' pinned buffers and event
        return state

    def _ensure_handle(self, device):
        if self._handle is not None and not self._dirty and self._handle_device == device:
            return
        self._release()
        lib = L.load()
        c = self._native_config()
        cfg = L.AdaConfig()
        cfg.embed_dim, cfg.depth, cfg.num_heads = c["embed_dim"], c["depth"], c["num_heads"]
        cfg.ffn_kind = 0 if c["ffn"] == "mlp" else 1
        cfg.ffn_hidden = c["hidden"]
        cfg.taps = (ctypes.c_int32 * 4)(*c["taps"])
        cfg.features = c["features"]
        cfg.out_channels = (ctypes.c_int32 * 4)(*c["out_channels"])
        cfg.guide_channels = c["guide_channels"]
        cfg.sigmoid = c["final_act"]
        cfg.pos_grid = POS_GRID
        cfg.interpolate_offset = 0.1
        cfg.input_projection = c["input_projection"]
        cfg.normalize_input = c["normalize_input"]
        h = ctypes.c_void_p()
        # Weights go device -> device: ada_set_weight copies each tensor into the handle's staging memory on the legacy
        # default stream and ada_finalize packs them with kernels (csrc/pack.cuh). Any dtype conversion below therefore runs
        # on the default stream too, after whatever the caller's current stream has produced.
        torch.cuda.current_stream(device).synchronize()
        with torch.cuda.device(device), torch.cuda.stream(torch.cuda.default_stream(device)):
            L.check(lib.ada_create(ctypes.byref(cfg), ctypes.byref(h)))
            try:
                for key, p in self._native_state().items():
                    t = p.detach().to(dtype=torch.float32).contiguous()
                    shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
                    L.check(lib.ada_set_weight(h, key.encode(), ctypes.c_void_p(t.data_ptr()), shape, t.dim()))
                L.check(lib.ada_finalize(h))
            except Exception:
                lib.ada_destroy(h)
                raise
        self._handle, self._handle_device, self._dirty = h, device, False
        if getattr(self, "_capture", False):
            lib.ada_set_capture(h, 1)
        if getattr(self, "_graph", False):
            lib.ada_set_graph(h, 1)

    def _run(self, x, guides):
        """x [B,3,H,W], guides: list of [B,c,H,W]; returns [B,1,H,W] fp32 on x's device, asynchronously on the current
        stream."""
        if self.training:
            raise RuntimeError(f"{type(self).__name__} (B200 path) is inference-only: call .eval() first; training is "
                               "out of scope")
        if not x.is_cuda:
            raise RuntimeError(f"{type(self).__name__} (B200 path) needs CUDA tensors: there is no CPU fallback")
        B, C3, H, W = x.shape
        assert C3 == 3, "x must be [B,3,H,W]"
        assert H % 14 == 0, f"Input image height {H} is not a multiple of patch height 14"    # patch_embed.py:73
        assert W % 14 == 0, f"Input image width {W} is not a multiple of patch width: 14"     # patch_embed.py:74
        dev = x.device
        x = x.detach().to(torch.float32).contiguous()
        gs = []
        for g in guides:
            if g.device != dev:
                raise RuntimeError("guides must live on the same device as x")
            assert g.shape[0] == B and tuple(g.shape[2:]) == (H, W), "guide shape mismatch"
            gs.append(g.detach().to(torch.float32).contiguous())
        self._ensure_handle(dev)
        out = torch.empty((B, 1, H, W), dtype=torch.float32, device=dev)
        n = len(gs)
        ptrs = (ctypes.c_void_p * max(n, 1))(*[g.data_ptr() for g in gs])
        chs = (ctypes.c_int32 * max(n, 1))(*[g.shape[1] for g in gs])
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            L.check(L.load().ada_forward(self._handle, ctypes.c_void_p(x.data_ptr()), ptrs, chs, n,
                                         ctypes.c_void_p(out.data_ptr()), B, H, W, stream))
        return out


    # ------------------------------------------------------------------ test hooks
    def set_capture(self, on: bool):
        self._capture = bool(on)
        if self._handle is not None:
            L.load().ada_set_capture(self._handle, int(on))

    def set_graph(self, on: bool):
        """Replay the forward as a CUDA graph (captured on the second call at a given input shape). For the launch-bound
        small-batch case -- the reference's infer.py runs one image per call; results are identical to the eager path."""
        self._graph = bool(on)
        if self._handle is not None:
            L.load().ada_set_graph(self._handle, int(on))
        return self

    def read_intermediate(self, name: str, numel: int) -> torch.Tensor:
        out = torch.empty(numel, dtype=torch.float32, device=self._handle_device)
        L.check(L.load().ada_read_intermediate(self._handle, name.encode(), ctypes.c_void_p(out.data_ptr()), numel))
        return out

    def launch_count(self) -> int:
        return int(L.load().ada_launch_count(self._handle, 0, 0, 0)) if self._handle is not None else 0

    def workspace_bytes(self) -> int:
        return int(L.load().ada_workspace_bytes(self._handle)) if self._handle is not None else 0


class AmodalDAv2(_NativeModel, PyTorchModelHubMixin):
    def __init__(self, guide_type="image+mask", loss_stategy="invisible_part", encoder="vitg", pretrained=True):
        super().__init__()
        self.guide_type = guide_type
        self.loss_stategy = loss_stategy
        self.encoder_name = encoder
        self.pretrained = pretrained
        cfg = MODEL_CONFIGS[encoder]  # KeyError for unknown encoders, as the reference
        if guide_type not in GUIDE_CHANNELS:
            raise NotImplementedError  # dinov2.py:124-125
        self._cfg = cfg
        tree = _Tree()
        for name, shape, kind in _param_table(cfg, guide_type):
            tree.put(name, _init(shape, kind))
        self.encoder = tree
        self.register_buffer("pixel_mean", torch.Tensor([0.485, 0.456, 0.406]).view(-1, 1, 1), False)  # dav2.py:50
        self.register_buffer("pixel_std", torch.Tensor([0.229, 0.224, 0.225]).view(-1, 1, 1), False)   # dav2.py:51
        self._native_init()

    def _native_config(self):
        return dict(self._cfg, guide_channels=GUIDE_CHANNELS[self.guide_type],
                    final_act=0 if "ssi" in self.loss_stategy else 1,  # dpt.py:138-151
                    input_projection=1, normalize_input=1)

    def _native_state(self):
        return self.encoder.state_dict()

    # ------------------------------------------------------------------ forward
    def _guides(self, guide_rgb, guide_mask, observation):
        """dav2.py:67-82: which tensors are concatenated, in order. A required guide that is None raises TypeError
        like torch.cat does in the reference."""
        order = {"image+mask+observation": (guide_rgb, guide_mask, observation), "image+mask": (guide_rgb, guide_mask),
                 "image+observation": (guide_rgb, observation), "mask+observation": (guide_mask, observation),
                 "observation": (observation,), "mask": (guide_mask,), "none": ()}
        if self.guide_type not in order:
            raise NotImplementedError
        gs = order[self.guide_type]
        for g in gs:
            if g is None:
                raise TypeError("expected Tensor as element of the guide concatenation but got NoneType")
        return list(gs)

    def forward(self, x, guide_rgb=None, guide_mask=None, observation=None):
        if self.training:
            raise RuntimeError("AmodalDAv2 (B200 path) is inference-only: call .eval() first; training is out of scope")
        return self._run(x, self._guides(guide_rgb, guide_mask, observation))

    # ------------------------------------------------------------------ serialisation (dav2.py:87-90)
    def _save_pretrained(self, save_directory) -> None:
        from safetensors.torch import save_model as save_model_as_safetensor
        model_to_save = self.module if hasattr(self, "module") else self
        save_model_as_safetensor(model_to_save, str(save_directory / SAFETENSORS_SINGLE_FILE))


class DepthAnythingV2(_NativeModel):
    """Drop-in for the un-guided `DepthAnythingV2` of depth_anything_v2_raw/dpt.py:154-187 -- the "observation" model
    infer.py:16-28,59-61 runs before the amodal model on every image (SURVEY.md section 8 row f1). Same kernels as
    AmodalDAv2 minus the guidance embedding and the input_projection levels; the head ends in ReLU
    (depth_anything_v2_raw/dpt.py:109-116,182). Differences from the reference class: inference-only, CUDA-only,
    `use_bn` / `use_clstoken` (both False everywhere in the reference) are not implemented.

    forward(x): x [B,3,H,W] fp32, ALREADY ImageNet-normalised by the caller (infer.py:18) -> [B,H,W] fp32 >= 0."""

    def __init__(self, encoder="vitg", features=256, out_channels=(256, 512, 1024, 1024), use_bn=False,
                 use_clstoken=False):
        super().__init__()
        if use_bn or use_clstoken:
            raise NotImplementedError("use_bn / use_clstoken are not part of the B200 path")
        self.encoder = encoder
        enc = MODEL_CONFIGS[encoder]  # KeyError for unknown encoders (dpt.py:166-171 indexes intermediate_layer_idx)
        self._cfg = dict(enc, features=int(features), out_channels=[int(c) for c in out_channels])
        pre, head = _Tree(), _Tree()
        for name, shape, kind in _param_table(self._cfg, "none", input_projection=False):
            root, _, rest = name.partition(".")
            (pre if root == "pretrained" else head).put(rest, _init(shape, kind))
        self.pretrained = pre
        self.depth_head = head
        self._native_init()

    def _native_config(self):
        return dict(self._cfg, guide_channels=0, final_act=2, input_projection=0, normalize_input=0)

    def _native_state(self):
        return self.state_dict()

    def forward(self, x):
        return self._run(x, []).squeeze(1)  # depth_anything_v2_raw/dpt.py:181-184

    # ---- host-side convenience of the reference class (depth_anything_v2_raw/dpt.py:186-222); glue, not the hot path
    @staticmethod
    def _input_size(h, w, target=518, multiple=14):
        """Resize(keep_aspect_ratio, lower_bound, ensure_multiple_of=14) of util/transform.py:52-102."""
        scale = max(target / h, target / w)

        def fit(v):
            y = int(round(scale * v / multiple) * multiple)
            if y < target:
                y = int(math.ceil(scale * v / multiple) * multiple)
            return y
        return fit(h), fit(w)

    def image2tensor(self, raw_image, input_size=518):
        import cv2
        import numpy as np
        h, w = raw_image.shape[:2]
        image = cv2.cvtColor(raw_image, cv2.COLOR_BGR2RGB) / 255.0
        nh, nw = self._input_size(h, w, input_size)
        image = cv2.resize(image, (nw, nh), interpolation=cv2.INTER_CUBIC)
        image = (image - np.array([0.485, 0.456, 0.406])) / np.array([0.229, 0.224, 0.225])
        image = np.ascontiguousarray(np.transpose(image, (2, 0, 1))).astype(np.float32)
        dev = next(self.parameters()).device
        return torch.from_numpy(image).unsqueeze(0).to(dev), (h, w)

    @torch.no_grad()
    def infer_image(self, raw_image, input_size=518):
        image, (h, w) = self.image2tensor(raw_image, input_size)
        depth = self.forward(image)
        depth = torch.nn.functional.interpolate(depth[:, None], (h, w), mode="bilinear", align_corners=True)[0, 0]
        return depth.cpu().numpy()

    @staticmethod
    def _chunks(shapes, input_size, max_batch):
        """The batches infer_images runs: [(H, W, [image indices])], images grouped by the network input size
        _input_size picks for them, groups in order of first appearance, each cut into chunks of at most max_batch."""
        groups = {}
        for i, (h, w) in enumerate(shapes):
            groups.setdefault(DepthAnythingV2._input_size(h, w, input_size), []).append(i)
        return [(H, W, idx[k:k + max_batch]) for (H, W), idx in groups.items() for k in range(0, len(idx), max_batch)]

    @torch.no_grad()
    def infer_images(self, raw_images, input_size=518, max_batch=32):
        """infer_image over a list, on the device: raw_images[i] is a uint8 BGR [h_i, w_i, 3] image (as cv2.imread returns
        it); returns a list of fp32 device tensors [h_i, w_i] in input order, views into one packed buffer. Image i is
        infer_image(raw_images[i], input_size) without the host read (call .cpu() on the results you need): the resize of
        image2tensor (cv2's float64 INTER_CUBIC and the ImageNet normalise, bit-exact), the forward and the restore to
        (h_i, w_i) all run as kernels on the current stream, and each image's result is bit-equal in any batch.

        Images are grouped by the network input size _input_size picks for them; the groups run in order of first
        appearance, each in chunks of at most max_batch images. The forward re-plans its workspace whenever (B, H, W)
        changes (a drain of the stream, and a larger arena when the new shape needs one), so a call re-plans at most once
        per distinct (B, H, W) of its chunks. Each chunk is one upload of the packed images and one of its descriptors.

        Unlike infer_image, which also passes float images through cv2, only uint8 [h, w, 3] images are accepted: anything
        else raises ValueError before any upload."""
        if max_batch < 1:
            raise ValueError("max_batch must be >= 1")
        imgs = [np.asarray(a) for a in raw_images]
        for i, a in enumerate(imgs):
            if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3 or a.shape[0] < 1 or a.shape[1] < 1:
                raise ValueError(f"raw_images[{i}]: expected a uint8 [h, w, 3] BGR image, got {a.dtype} {a.shape}")
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("DepthAnythingV2 (B200 path) needs CUDA parameters: there is no CPU fallback")
        # every output in one fp32 buffer; pack_layout places [h, w, 4]-byte maps at 16-byte boundaries
        rows_out, end = ops.pack_layout([(a.shape[0], a.shape[1], 4) for a in imgs])
        out = torch.empty((end + 3) // 4, dtype=torch.float32, device=dev)
        if getattr(self, "_staging", None) is None or self._staging.device != dev:
            self._staging = ops.Staging(dev)
        with torch.cuda.device(dev):
            for H, W, idx in self._chunks([a.shape[:2] for a in imgs], input_size, max_batch):
                rows_in, n_in = ops.pack_layout([imgs[i].shape for i in idx])

                def fill(host, rows_in=rows_in, idx=idx):
                    for (o, _, _), i in zip(rows_in, idx):
                        np.copyto(host[o:o + imgs[i].size].reshape(imgs[i].shape), imgs[i])
                data, desc = self._staging.upload(n_in, rows_in + [rows_out[i] for i in idx], fill)
                x = ops.resize_cubic_normalize_batch(data, desc[:len(idx)], H, W)
                ops.upsample_restore_batch(self.forward(x), desc[len(idx):], out)
        return [out[o // 4:o // 4 + h * w].view(h, w) for o, h, w in rows_out]


def get_model(model_name, **kwargs):
    """src/models/__init__.py:24-31 for the one model this package implements."""
    if model_name != "AmodalDAv2":
        raise KeyError(f"{model_name}: only 'AmodalDAv2' is implemented by the B200 path")
    return AmodalDAv2(**kwargs)

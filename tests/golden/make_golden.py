"""Generates tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference, build container only)
on seeded synthetic weights/inputs. Re-run: `python tests/golden/make_golden.py`. The GPU box never runs this.

Import shim (SURVEY.md section 8c): the reference's src/models/__init__.py pulls in torchdiffeq/diffusers and dav2.py
imports timm (unused by AmodalDAv2); neither is installed, so stub `timm` and register `src`, `src.models` as bare
namespace packages pointing at the reference directories. No reference file is modified or copied.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def import_reference():
    sys.modules.setdefault("timm", types.ModuleType("timm"))
    for name, path in (("src", f"{REF}/src"), ("src.models", f"{REF}/src/models")):
        m = types.ModuleType(name)
        m.__path__ = [path]
        sys.modules[name] = m
    from src.models.amodalsynthdrive.dav2 import AmodalDAv2
    from src.models.amodalsynthdrive.depth_anything_v2.dpt import DepthAnythingV2
    return AmodalDAv2, DepthAnythingV2


def import_reference_raw():
    """The un-guided `DepthAnythingV2` infer.py:13,59 uses for the observation depth (SURVEY.md section 8 row f1)."""
    import_reference()
    from src.models.amodalsynthdrive.depth_anything_v2_raw.dpt import DepthAnythingV2 as RawDepthAnythingV2
    return RawDepthAnythingV2


def hook_intermediates(net, store):
    """net: DepthAnythingV2. Records the tensors named in SURVEY.md section 4 (module-level parity points)."""
    dh = net.depth_head
    hs = []
    for i in range(4):
        hs.append(dh.input_projection[i].register_forward_hook(lambda m, a, o, i=i: store.__setitem__(f"layer{i+1}", o)))
        hs.append(getattr(dh.scratch, f"layer{i+1}_rn").register_forward_hook(
            lambda m, a, o, i=i: store.__setitem__(f"layer{i+1}_rn", o)))
        hs.append(getattr(dh.scratch, f"refinenet{i+1}").register_forward_hook(
            lambda m, a, o, i=i: store.__setitem__(f"path_{i+1}", o)))
    hs.append(dh.scratch.output_conv2[2].register_forward_hook(lambda m, a, o: store.__setitem__("logits", o)))
    orig = net.pretrained.prepare_tokens_with_masks

    def wrapped(*a, **k):
        t = orig(*a, **k)
        store["tokens"] = t
        return t
    net.pretrained.prepare_tokens_with_masks = wrapped
    orig_gil = net.pretrained.get_intermediate_layers

    def wrapped_gil(*a, **k):
        r = orig_gil(*a, **k)
        for i, (f, _c) in enumerate(r):
            store[f"tap{i}"] = f
        return r
    net.pretrained.get_intermediate_layers = wrapped_gil
    return hs


def sample(t, n=4096):
    """Deterministic strided sample of a tensor (keeps fixtures small) + full-tensor moments."""
    f = t.detach().float().flatten()
    step = max(f.numel() // n, 1)
    return f[::step][:n].numpy().copy(), np.array([f.mean().item(), f.abs().mean().item(), f.std().item()], np.float64)


def byte_planes(a):
    """Lossless [4, *shape] uint8 view of a float32 array, one plane per little-endian byte: the sign / exponent planes
    compress to almost nothing, which keeps a full 518x518 output under 1 MB (tests/golden_util.py:load_golden decodes)."""
    return np.moveaxis(a.astype("<f4").view(np.uint8).reshape(a.shape + (4,)), -1, 0).copy()


CASES = [
    # name, encoder, guide_type, loss_stategy, B, H, W, seed, stress, save full output
    ("vits_518_b1", "vits", "mask+observation", "invisible_part", 1, 518, 518, 0, False),
    ("vits_126x98_b2", "vits", "mask+observation", "invisible_part", 2, 126, 98, 1, False),
    ("vits_img_mask_obs_70", "vits", "image+mask+observation", "invisible_part", 1, 70, 70, 2, False),
    ("vits_none_ssi_70", "vits", "none", "ssi", 1, 70, 70, 3, False),
    ("vits_mask_84_stress", "vits", "mask", "invisible_part", 1, 84, 84, 4, True),
    ("vitb_70_b2", "vitb", "mask+observation", "invisible_part", 2, 70, 70, 5, False),
    ("vitl_70_b1", "vitl", "mask+observation", "invisible_part", 1, 70, 70, 6, False),
    ("vitg_56_b1", "vitg", "mask+observation", "invisible_part", 1, 56, 56, 7, False),
]


RAW_CASES = [
    # name, encoder, features, out_channels, B, H, W, seed, shift of the last bias (-0.003: part of the output is clipped by ReLU)
    ("raw_vits_70x98_b2", "vits", 64, [48, 96, 192, 384], 2, 70, 98, 11, 0.25),
    ("raw_vits_84_clip", "vits", 64, [48, 96, 192, 384], 1, 84, 84, 12, -0.003),
    ("raw_vitg_56_b1", "vitg", 384, [1536, 1536, 1536, 1536], 1, 56, 56, 13, 0.25),  # infer.py:59
]


def main_raw(only):
    from oracle import synth
    from oracle.amodal_oracle import normalize_rgb
    Raw = import_reference_raw()
    os.makedirs(os.path.join(ROOT, "tests", "golden", "raw"), exist_ok=True)
    for name, enc, F_, C, B, H, W, seed, shift in RAW_CASES:
        if only and name not in only:
            continue
        sd = synth.make_state_dict_raw(enc, F_, C, seed, shift)
        net = Raw(encoder=enc, features=F_, out_channels=C).eval()
        net.load_state_dict(sd, strict=True)
        x = normalize_rgb(synth.make_inputs(B, H, W, seed)["x"])  # the caller normalises (infer.py:18)
        with torch.no_grad():
            out = net(x)
        meta = dict(encoder=enc, features=F_, out_channels=C, B=B, H=H, W=W, seed=seed, shift=shift,
                    torch=torch.__version__)
        path = os.path.join(ROOT, "tests", "golden", "raw", name + ".npz")
        np.savez_compressed(path, output=out.numpy().astype(np.float32), meta=np.array(repr(meta)))
        print(name, "out range", float(out.min()), float(out.max()), "zeros", float((out == 0).float().mean()), "->",
              os.path.getsize(path) // 1024, "KB", flush=True)


def main():
    from oracle import synth
    from oracle.amodal_oracle import CONFIGS
    AmodalDAv2, DepthAnythingV2 = import_reference()
    torch.manual_seed(0)
    only = sys.argv[1:]
    if only and not any(o in [c[0] for c in CASES] for o in only):
        return
    for name, enc, gt, ls, B, H, W, seed, stress in CASES:
        if only and name not in only:
            continue
        sd = synth.make_state_dict(enc, gt, seed, stress)
        inp = synth.make_inputs(B, H, W, seed)
        store = {}
        if enc == "vitg":
            # AmodalDAv2(encoder='vitg') raises KeyError (dav2.py:31-34); drive the inner network like the wrapper does.
            c = CONFIGS[enc]
            net = DepthAnythingV2(encoder=enc, features=c["features"], out_channels=c["out_channels"], guide_type=gt,
                                  loss_stategy=ls).eval()
            net.load_state_dict({k[len("encoder."):]: v for k, v in sd.items()}, strict=True)
            hook_intermediates(net, store)
            mean = torch.tensor([0.485, 0.456, 0.406]).view(-1, 1, 1)
            std = torch.tensor([0.229, 0.224, 0.225]).view(-1, 1, 1)
            with torch.no_grad():
                out = net((inp["x"] - mean) / std, torch.cat([inp["guide_mask"], inp["observation"]], 1))
        else:
            model = AmodalDAv2(guide_type=gt, loss_stategy=ls, encoder=enc, pretrained=False).eval()
            missing = model.load_state_dict(sd, strict=True)
            hook_intermediates(model.encoder, store)
            with torch.no_grad():
                out = model(inp["x"], guide_rgb=inp["guide_rgb"], guide_mask=inp["guide_mask"],
                            observation=inp["observation"])
        arrays = {"output_planes": byte_planes(out.numpy())}
        for k, v in store.items():
            s, mom = sample(v)
            arrays["s_" + k] = s
            arrays["m_" + k] = mom
        meta = dict(encoder=enc, guide_type=gt, loss_stategy=ls, B=B, H=H, W=W, seed=seed, stress=stress,
                    torch=torch.__version__)
        arrays["meta"] = np.array(repr(meta))
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        np.savez_compressed(path, **arrays)
        print(name, "out range", float(out.min()), float(out.max()), "->", os.path.getsize(path) // 1024, "KB", flush=True)


if __name__ == "__main__":
    main()
    main_raw(sys.argv[1:])

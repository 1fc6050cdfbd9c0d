"""End-to-end parity of the CUDA path (AmodalDAv2.forward -> C ABI -> sm_100a kernels) on a real B200.

Bars (BASELINE.json north_star / SURVEY.md section 8d), against the fp32 reference on identical seeded weights/inputs:
  per-pixel relative error  max |new - ref| / ref  <= 1e-2
  AbsRel over the mask      mean_{mask} |new - ref| / ref  <= 1e-3   (src/util/metric.py:37-47 semantics)
The reference values are (a) the committed goldens produced by the unmodified reference, (b) the CPU oracle run here.
The 'stress' golden (last conv x40, outputs spanning 0.06..0.82) is reported against a looser, stated bar."""
import numpy as np
import pytest
import torch

import amodal_depth_anything_b200 as pkg
from oracle import amodal_oracle as O
from oracle import synth
from tests.golden_util import golden_names, load_golden, sample

pytestmark = pytest.mark.gpu

REL_TOL, ABSREL_TOL = 1e-2, 1e-3
# Intermediates, max |got - ref| / max |ref| over the strided golden sample; bf16 activations, fp32 accumulation / residual
# stream. Largest values measured on a B200 over the eight goldens (round 2, gpurun_out/parity_report.json): tokens 2.6e-3,
# taps 1.55e-2 (ViT-G, 40 blocks), layerN 1.48e-2, layerN_rn 1.15e-2, path_k 1.23e-2 -- the bars sit 1.3-1.7x above them.
INTER_TOL = {"tokens": 4e-3, "tap": 2e-2, "layer": 2e-2, "layer_rn": 2e-2, "path": 2e-2}
# pre-sigmoid logits, absolute: measured <= 1.4e-3 (default init, |logit| <= 0.11) and 2.6e-2 (stress init, |logit| <= 2.7)
LOGIT_TOL, LOGIT_TOL_STRESS = 3e-3, 6e-2


def _inter_kind(k):
    if k == "tokens":
        return "tokens"
    if k.startswith("tap"):
        return "tap"
    if k.startswith("layer"):
        return "layer_rn" if k.endswith("_rn") else "layer"
    return "path"


def _record(name, report):
    """Keeps the measured errors of a GPU run (gpurun_out/ travels back from the GPU box) so the bars above can be audited."""
    import json
    import os
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    try:
        os.makedirs(d, exist_ok=True)
        path = os.path.join(d, "parity_report.json")
        allr = json.load(open(path)) if os.path.exists(path) else {}
        allr[name] = report
        json.dump(allr, open(path, "w"), indent=1, sort_keys=True)
    except OSError:
        pass


def _model(enc, gt, ls, sd):
    m = pkg.AmodalDAv2(guide_type=gt, loss_stategy=ls, encoder=enc, pretrained=False)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval()


def _run(m, inp):
    out = m(inp["x"].cuda(), guide_rgb=inp["guide_rgb"].cuda(), guide_mask=inp["guide_mask"].cuda(),
            observation=inp["observation"].cuda())
    torch.cuda.synchronize()
    return out.cpu()


def _errors(out, ref, mask):
    rel = ((out - ref).abs() / ref.abs().clamp_min(1e-6)).max().item()
    absrel = O.abs_relative_difference(out.clone(), ref, mask).item()
    return rel, absrel


@pytest.mark.parametrize("name", golden_names())
def test_forward_matches_reference_golden(name):
    meta, z = load_golden(name)
    sd = synth.make_state_dict(meta["encoder"], meta["guide_type"], meta["seed"], meta["stress"])
    inp = synth.make_inputs(meta["B"], meta["H"], meta["W"], meta["seed"])
    m = _model(meta["encoder"], meta["guide_type"], meta["loss_stategy"], sd)
    m.set_capture(True)
    out = _run(m, inp)
    ref = torch.from_numpy(z["output"])
    assert out.shape == ref.shape and out.dtype == torch.float32
    assert torch.isfinite(out).all()
    report = {}
    for key in z:  # module-level parity points (SURVEY.md section 4), strided samples
        if not key.startswith("s_"):
            continue
        k = key[2:]
        if k == "logits":
            continue  # checked below from the output (the fused tail never stores the pre-sigmoid map)
        got = m.read_intermediate(k, _numel(meta, k))   # an unreadable intermediate is a failure, not a skip
        g = sample(_to_ref_layout(meta, k, got))
        scale = float(np.abs(z[key]).max())
        report[k] = float(np.abs(g - z[key]).max() / scale)
        assert report[k] < INTER_TOL[_inter_kind(k)], (k, report)
    if "s_logits" in z and "ssi" not in meta["loss_stategy"]:
        # pre-sigmoid logits (dpt.py:195, output_conv2[2]) recovered from the fp32 output: logit = log(o / (1 - o))
        lg = sample(torch.log(out.double() / (1.0 - out.double())).float())
        report["logits_abs"] = float(np.abs(lg - z["s_logits"]).max())
        report["logits_span"] = float(np.abs(z["s_logits"]).max())
        assert report["logits_abs"] < (LOGIT_TOL_STRESS if meta["stress"] else LOGIT_TOL), report
    _record(name, report)
    if "ssi" in meta["loss_stategy"]:   # raw logits (dpt.py:138-144): absolute bar, the output crosses zero
        err = (out - ref).abs().max().item()
        print(name, "logit max abs err", err, report)
        assert err <= 5e-3
        return
    rel, absrel = _errors(out, ref, inp["mask01"])
    print(name, f"rel {rel:.3e} absrel {absrel:.3e}", report)
    _record(name, dict(report, rel=rel, absrel=absrel))
    if meta["stress"]:
        # stated looser bar for the stress init: bf16 operands cannot hold 1e-2 per pixel when logits span +-3
        # (SURVEY.md section 7: torch's own autocast-bf16 reaches 3.5e-2 there)
        assert rel <= 5e-2 and absrel <= 5e-3
    else:
        assert rel <= REL_TOL and absrel <= ABSREL_TOL


def _numel(meta, k):
    c = pkg.MODEL_CONFIGS[meta["encoder"]]
    B, gh, gw = meta["B"], meta["H"] // 14, meta["W"] // 14
    D, F = c["embed_dim"], c["features"]
    d2 = lambda v: (v - 1) // 2 + 1  # noqa: E731
    sh = [gh * 4, gh * 2, gh, d2(gh)]
    sw = [gw * 4, gw * 2, gw, d2(gw)]
    if k == "tokens":
        return B * (gh * gw + 1) * D
    if k.startswith("tap"):
        return B * gh * gw * D
    if k.endswith("_rn"):
        i = int(k[5]) - 1
        return B * sh[i] * sw[i] * F
    if k.startswith("layer"):   # input_projection output (dpt.py:178-179): C_i channels at level i
        i = int(k[5]) - 1
        return B * sh[i] * sw[i] * c["out_channels"][i]
    if k.startswith("path_"):
        i = int(k[5])
        ph = [0, sh[0] * 2, sh[0], sh[1], sh[2]]
        pw = [0, sw[0] * 2, sw[0], sw[1], sw[2]]
        return B * ph[i] * pw[i] * F
    raise KeyError(k)


def _to_ref_layout(meta, k, t):
    """CUDA path keeps feature maps NHWC; the reference tensors are NCHW. Tokens/taps are [B,N,D] in both."""
    c = pkg.MODEL_CONFIGS[meta["encoder"]]
    if k == "tokens" or k.startswith("tap"):
        return t
    B, F = meta["B"], c["features"]
    if k.startswith("layer") and not k.endswith("_rn"):
        F = c["out_channels"][int(k[5]) - 1]
    hw = t.numel() // (B * F)
    gh, gw = meta["H"] // 14, meta["W"] // 14
    # recover (h, w) from the pyramid level
    d2 = lambda v: (v - 1) // 2 + 1  # noqa: E731
    cands = [(gh * 8, gw * 8), (gh * 4, gw * 4), (gh * 2, gw * 2), (gh, gw), (d2(gh), d2(gw))]
    h, w = next((a, b) for a, b in cands if a * b == hw)
    return t.view(B, h, w, F).permute(0, 3, 1, 2).contiguous()


def test_forward_matches_oracle_vitb_518():
    """BASELINE config #2 shape (ViT-B 518x518), batch 2 so the CPU oracle finishes in seconds."""
    enc, gt = "vitb", "mask+observation"
    sd = synth.make_state_dict(enc, gt, 11)
    inp = synth.make_inputs(2, 518, 518, 11)
    ref = O.forward(sd, enc, gt, inp["x"], None, inp["guide_mask"], inp["observation"])
    out = _run(_model(enc, gt, "invisible_part", sd), inp)
    rel, absrel = _errors(out, ref, inp["mask01"])
    print(f"vitb 518 rel {rel:.3e} absrel {absrel:.3e}")
    assert rel <= REL_TOL and absrel <= ABSREL_TOL


def test_forward_matches_oracle_vitl_518():
    """The headline architecture (ViT-L, released model) at 518x518, batch 1."""
    enc, gt = "vitl", "mask+observation"
    sd = synth.make_state_dict(enc, gt, 12)
    inp = synth.make_inputs(1, 518, 518, 12)
    ref = O.forward(sd, enc, gt, inp["x"], None, inp["guide_mask"], inp["observation"])
    out = _run(_model(enc, gt, "invisible_part", sd), inp)
    rel, absrel = _errors(out, ref, inp["mask01"])
    print(f"vitl 518 rel {rel:.3e} absrel {absrel:.3e}")
    assert rel <= REL_TOL and absrel <= ABSREL_TOL


def test_forward_matches_oracle_vits_1036():
    """BASELINE config #4 resolution (1036x1036: 5477 tokens, bicubic pos-embed with the 0.1 offset, 74x74 patch grid,
    long-sequence attention, 592/1036 head maps) on the small encoder so the CPU oracle stays within seconds."""
    enc, gt = "vits", "mask+observation"
    sd = synth.make_state_dict(enc, gt, 17)
    inp = synth.make_inputs(1, 1036, 1036, 17)
    ref = O.forward(sd, enc, gt, inp["x"], None, inp["guide_mask"], inp["observation"])
    out = _run(_model(enc, gt, "invisible_part", sd), inp)
    rel, absrel = _errors(out, ref, inp["mask01"])
    print(f"vits 1036 rel {rel:.3e} absrel {absrel:.3e}")
    assert rel <= REL_TOL and absrel <= ABSREL_TOL


def test_batch_sharding_is_bit_exact_and_deterministic():
    """Images are independent end to end (no BatchNorm, per-token LN, per-image attention), so running a batch in
    shards -- what the multi-GPU path does -- must reproduce the full-batch result bit for bit (SURVEY.md section 4)."""
    enc, gt = "vits", "mask+observation"
    sd = synth.make_state_dict(enc, gt, 13)
    inp = synth.make_inputs(4, 126, 154, 13)
    m = _model(enc, gt, "invisible_part", sd)
    full = _run(m, inp)
    again = _run(m, inp)
    assert torch.equal(full, again)
    parts = []
    for lo, hi in ((0, 1), (1, 4)):
        sub = {k: v[lo:hi] for k, v in inp.items()}
        parts.append(_run(m, sub))
    assert torch.equal(torch.cat(parts), full)


def test_non_contiguous_and_guide_rgb_ignored():
    """guide_rgb is accepted but unused for 'mask+observation' (dav2.py:73-74); strided inputs are handled."""
    enc, gt = "vits", "mask+observation"
    sd = synth.make_state_dict(enc, gt, 14)
    inp = synth.make_inputs(1, 70, 84, 14)
    m = _model(enc, gt, "invisible_part", sd)
    a = _run(m, inp)
    x_nc = inp["x"].cuda().permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)  # channels-last strides
    b = m(x_nc, guide_rgb=None, guide_mask=inp["guide_mask"].cuda(), observation=inp["observation"].cuda()).cpu()
    assert torch.equal(a, b)


def test_repack_after_load_state_dict():
    enc, gt = "vits", "mask"
    inp = synth.make_inputs(1, 70, 70, 15)
    m = _model(enc, gt, "invisible_part", synth.make_state_dict(enc, gt, 15))
    a = _run(m, inp)
    m.load_state_dict(synth.make_state_dict(enc, gt, 16), strict=True)
    b = _run(m, inp)
    assert not torch.equal(a, b)
    ref = O.forward(synth.make_state_dict(enc, gt, 16), enc, gt, inp["x"], None, inp["guide_mask"], None)
    assert ((b - ref).abs() / ref).max().item() <= REL_TOL


def test_cuda_graph_replay_is_bit_identical():
    """ada_set_graph: the third and later calls at a shape replay a captured graph over staging buffers; outputs must
    equal the eager path bit for bit, also with new input values / new tensors, and after a shape change and back."""
    sd = synth.make_state_dict("vits", "mask+observation", 9)
    m = _model("vits", "mask+observation", "invisible_part", sd)
    a, b = synth.make_inputs(1, 126, 98, 1), synth.make_inputs(1, 126, 98, 2)
    c = synth.make_inputs(2, 70, 70, 3)
    eager = [_run(m, i).clone() for i in (a, b, c)]
    m.set_graph(True)
    for rep in range(2):
        for inp, ref in ((a, eager[0]), (a, eager[0]), (b, eager[1]), (a, eager[0]), (c, eager[2]), (c, eager[2]), (c, eager[2])):
            assert torch.equal(_run(m, inp), ref)
    m.set_graph(False)
    assert torch.equal(_run(m, b), eager[1])


def test_streamed_inference_matches_direct_calls():
    """pipeline.StreamedInference (what bench.py's e2e figure runs): pinned host batches in, pinned host results out, H2D /
    forward / D2H on three streams with double-buffered device inputs. Every batch must equal the direct model call."""
    from amodal_depth_anything_b200.pipeline import StreamedInference
    sd = synth.make_state_dict("vits", "mask+observation", 12)
    m = _model("vits", "mask+observation", "invisible_part", sd)
    batches = [synth.make_inputs(2, 126, 98, s) for s in (31, 32, 33, 34, 35)]
    want = [_run(m, b) for b in batches]
    host_in = [(b["x"].pin_memory(), b["guide_mask"].pin_memory(), b["observation"].pin_memory()) for b in batches]
    host_out = [torch.empty(2, 1, 126, 98).pin_memory() for _ in batches]
    runner = StreamedInference(m)
    for _ in range(2):  # second pass reuses the device slots
        for o in host_out:
            o.zero_()
        runner.run(iter(host_in), host_out)
        torch.cuda.synchronize()
        for got, ref in zip(host_out, want):
            assert torch.equal(got, ref)


def test_forward_matches_oracle_non_square_518x686():
    """The un-guided model's own resize rule (depth_anything_v2_raw/dpt.py:196-205) turns a 480x640 photo into 518x686:
    37x49 patches, pyramid 148x196 / 74x98 / 37x49 / 19x25 -- ragged conv tiles in both directions and a position table
    interpolated to a non-square grid (dinov2.py:199-230)."""
    sd = synth.make_state_dict("vits", "mask+observation", 19)
    inp = synth.make_inputs(1, 518, 686, 19)
    m = _model("vits", "mask+observation", "invisible_part", sd)
    out = _run(m, inp)
    ref = O.forward(sd, "vits", "mask+observation", inp["x"], None, inp["guide_mask"], inp["observation"])
    rel, absrel = _errors(out, ref, inp["mask01"])
    print("vits 518x686", f"rel {rel:.3e} absrel {absrel:.3e}")
    assert rel <= REL_TOL and absrel <= ABSREL_TOL

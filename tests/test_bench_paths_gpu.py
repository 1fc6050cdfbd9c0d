"""Model-level parity on the code paths bench.py actually times (VERDICT r1, "parity gap on the benchmarked path").

The BASELINE.json configurations run kernels that small test shapes never reach:
  * ViT-L 518x518, 32 images: M = 43 840 tokens -> gemm_tcgen05_kernel<256, 2, *> (CTA pairs, cta_group::2), programmatic
    dependent launch off (> 12 000 tokens), CTA-pair implicit-GEMM convs in the head;
  * ViT-L 1036x1036, 4 images: 5 477 tokens per image (43 KV tiles per query tile), 592^2 / 1036^2 head maps;
  * ViT-G 518x518, 8 images: D = 1536 (24 heads), 40 blocks, SwiGLU pair epilogue, 1536-channel reassemble convs.
Each is run through the public model call (AmodalDAv2.forward -> C ABI) and compared with the CPU oracle
(oracle/amodal_oracle.py, pinned to the unmodified reference by tests/test_oracle_golden.py) on a subset of the images --
the oracle costs ~1 s (ViT-L 518^2) to ~20 s (ViT-L 1036^2) per image on the GPU box's host cores. Bars: the north-star's
per-pixel relative error <= 1e-2 and AbsRel over the mask <= 1e-3 (src/util/metric.py:37-47 semantics)."""
import pytest
import torch

import amodal_depth_anything_b200 as pkg
from oracle import amodal_oracle as O
from oracle import synth
from tests.test_forward_gpu import ABSREL_TOL, REL_TOL, _errors, _model, _record, _run

pytestmark = pytest.mark.gpu

GT = "mask+observation"


def _oracle(sd, enc, inp, idx, loss="invisible_part"):
    sub = {k: v[idx:idx + 1] for k, v in inp.items()}
    return O.forward(sd, enc, GT, sub["x"], None, sub["guide_mask"], sub["observation"], loss_stategy=loss)


def test_vitl_518_batch32_cta_pair_path_matches_oracle_and_single_image_calls():
    """BASELINE configs[2], exactly the bench workload. Images 0, 15, 31 against the oracle; all 32 against one-image calls
    of the same model (single-CTA tiles, PDL on): the batch must not change any image (no cross-image arithmetic), and
    the CTA-pair kernels must agree with the single-CTA ones to fp32 rounding of identical accumulation orders."""
    enc = "vitl"
    sd = synth.make_state_dict(enc, GT, 21)
    inp = synth.make_inputs(32, 518, 518, 21)
    m = _model(enc, GT, "invisible_part", sd)
    out = _run(m, inp)
    assert out.shape == (32, 1, 518, 518) and torch.isfinite(out).all()
    rep = {}
    for i in (0, 15, 31):
        ref = _oracle(sd, enc, inp, i)
        rel, absrel = _errors(out[i:i + 1], ref, inp["mask01"][i:i + 1])
        rep[f"img{i}"] = dict(rel=rel, absrel=absrel)
        assert rel <= REL_TOL and absrel <= ABSREL_TOL, rep
    worst = 0.0
    for i in range(32):
        one = _run(m, {k: v[i:i + 1] for k, v in inp.items()})
        worst = max(worst, (one - out[i:i + 1]).abs().max().item())
    rep["max_abs_diff_vs_single_image_calls"] = worst
    _record("vitl_518_b32", rep)
    print("vitl 518 b32", rep)
    assert worst == 0.0, rep   # same per-element accumulation order in every tile shape: bit-identical


def test_vitl_518_stress_init_logits():
    """ViT-L 518x518 with the last conv scaled x40 (outputs span most of (0,1); SURVEY.md section 7 "tolerance regime"):
    reports the pre-sigmoid logit error -- the quantity bf16 compute actually perturbs -- through the 'ssi' (no sigmoid)
    head, and holds the sigmoid output to the stated looser stress bar."""
    enc = "vitl"
    sd = synth.make_state_dict(enc, GT, 22, stress=True)
    inp = synth.make_inputs(2, 518, 518, 22)
    ref_logit = torch.cat([_oracle(sd, enc, inp, i, loss="ssi") for i in range(2)])
    logit = _run(_model(enc, GT, "ssi", sd), inp)
    out = _run(_model(enc, GT, "invisible_part", sd), inp)
    err = (logit - ref_logit).abs().max().item()
    span = ref_logit.abs().max().item()
    rel, absrel = _errors(out, torch.sigmoid(ref_logit), inp["mask01"])
    rep = dict(logit_max_abs_err=err, logit_span=span, out_min=out.min().item(), out_max=out.max().item(), rel=rel, absrel=absrel)
    _record("vitl_518_stress", rep)
    print("vitl 518 stress", rep)
    assert torch.equal(out, torch.sigmoid(logit)) or (out - torch.sigmoid(logit)).abs().max().item() < 1e-6
    assert err <= 0.1 and rel <= 5e-2 and absrel <= 5e-3, rep


def test_vitl_1036_batch4_matches_oracle():
    """BASELINE configs[3]: ViT-L at 1036x1036, 4 images (5477 tokens, bicubic position table, 592^2 / 1036^2 head)."""
    enc = "vitl"
    sd = synth.make_state_dict(enc, GT, 23)
    inp = synth.make_inputs(4, 1036, 1036, 23)
    m = _model(enc, GT, "invisible_part", sd)
    out = _run(m, inp)
    assert torch.isfinite(out).all()
    ref = _oracle(sd, enc, inp, 2)
    rel, absrel = _errors(out[2:3], ref, inp["mask01"][2:3])
    one = _run(m, {k: v[2:3] for k, v in inp.items()})
    rep = dict(rel=rel, absrel=absrel, max_abs_diff_vs_single_image_call=(one - out[2:3]).abs().max().item())
    _record("vitl_1036_b4", rep)
    print("vitl 1036 b4", rep)
    assert rel <= REL_TOL and absrel <= ABSREL_TOL, rep
    assert rep["max_abs_diff_vs_single_image_call"] == 0.0, rep


def test_vitg_518_batch8_matches_oracle():
    """BASELINE configs[4] per-GPU share: ViT-G (train_discriminative_vitg architecture: SwiGLU FFN, 40 blocks, features 384,
    out_channels 4 x 1536) at 518x518, 8 images."""
    enc = "vitg"
    sd = synth.make_state_dict(enc, GT, 24)
    inp = synth.make_inputs(8, 518, 518, 24)
    m = _model(enc, GT, "invisible_part", sd)
    out = _run(m, inp)
    assert torch.isfinite(out).all()
    ref = _oracle(sd, enc, inp, 5)
    rel, absrel = _errors(out[5:6], ref, inp["mask01"][5:6])
    rep = dict(rel=rel, absrel=absrel)
    _record("vitg_518_b8", rep)
    print("vitg 518 b8", rep)
    assert rel <= REL_TOL and absrel <= ABSREL_TOL, rep


def test_alternating_batch_sizes_on_a_side_stream_match_default_stream_results():
    """ADVICE r1: a ragged last batch re-plans the workspace while the previous forward may still be running on a
    non-blocking stream. Alternate two batch sizes on a torch side stream without host syncs in between and compare with
    results computed one call at a time on the default stream."""
    enc = "vits"
    sd = synth.make_state_dict(enc, GT, 25)
    m = _model(enc, GT, "invisible_part", sd)
    a, b = synth.make_inputs(3, 126, 98, 41), synth.make_inputs(1, 126, 98, 42)
    want = {3: _run(m, a), 1: _run(m, b)}
    dev = {n: {k: v.cuda() for k, v in inp.items()} for n, inp in ((3, a), (1, b))}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    outs = []
    with torch.cuda.stream(side):
        for n in (3, 1, 3, 1, 1, 3, 3, 1):
            d = dev[n]
            outs.append((n, m(d["x"], guide_rgb=None, guide_mask=d["guide_mask"], observation=d["observation"])))
    side.synchronize()
    for n, o in outs:
        assert torch.equal(o.cpu(), want[n]), n


def test_bench_dump_is_the_last_timed_step_and_steps_sets_the_timed_steps(tmp_path):
    """bench.py --dump-outputs writes what the timed path returned in its last step: the same numbers as a direct call of
    the model on bench.py's own seeded weights and inputs. --steps is the number of timed steps."""
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--encoder", "vits", "--size", "126", "--batch", "2",
                        "--steps", "3", "--warmup", "1", "--no-extras", "--no-cpu-baseline", "--profile-steps", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 3 and len(d["ms_steps_rank0"]) == 3 and d["dump_outputs"]["file"] == "depth.npy"
    got = np.load(tmp_path / "depth.npy")
    sys.path.insert(0, root)
    import bench
    dev = torch.device("cuda", 0)
    m = bench.make_model(pkg, torch, "vits", dev)
    x, mask, obs = bench.make_inputs(torch, 2, 126, 126, dev, 1234)
    want = m(x, guide_rgb=None, guide_mask=mask, observation=obs).cpu().numpy()
    assert got.dtype == np.float32 and got.shape == (2, 1, 126, 126)
    assert np.array_equal(got, want)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")
def test_one_process_two_devices():
    """One process driving two GPUs, one model each (SURVEY.md section 5 "one process, N streams"): the per-kernel
    shared-memory opt-in and the SM count are per-device state inside the library."""
    enc = "vits"
    sd = synth.make_state_dict(enc, GT, 26)
    inp = synth.make_inputs(2, 126, 98, 26)
    ref = O.forward(sd, enc, GT, inp["x"], None, inp["guide_mask"], inp["observation"])
    outs = []
    for d in (0, 1):   # cuda:0 first: sets the attributes there; cuda:1 must then still work while cuda:0 stays current
        m = pkg.AmodalDAv2(guide_type=GT, encoder=enc, pretrained=False)
        m.load_state_dict(sd, strict=True)
        m = m.to(f"cuda:{d}").eval()
        o = m(inp["x"].to(f"cuda:{d}"), guide_rgb=None, guide_mask=inp["guide_mask"].to(f"cuda:{d}"),
              observation=inp["observation"].to(f"cuda:{d}"))
        outs.append(o.cpu())
    assert torch.equal(outs[0], outs[1])
    assert ((outs[1] - ref).abs() / ref).max().item() <= REL_TOL


@pytest.mark.parametrize("enc,B,size", [("vits", 7, 266), ("vitb", 5, 154)])
def test_pixel_tiles_spanning_images_with_a_ragged_batch(enc, B, size):
    """The implicit-GEMM convs pick their M tile as 2^lw x 2^lh pixels of 2^lb images for least padding (csrc/ada_api.cu
    pick_tile_geo). 266 -> maps of 76 / 38 / 19 / 10 pixels, 154 -> 44 / 22 / 11 / 6: with 7 (5) images the small maps take
    tiles spanning 8 (4 .. 8) images, so the last tile's TMA loads zero-fill and its TMA stores clip images that do not exist.
    Every image against the oracle, and bit-equal to one-image calls (tiles of one image, other shapes)."""
    sd = synth.make_state_dict(enc, GT, 33)
    inp = synth.make_inputs(B, size, size, 33)
    m = _model(enc, GT, "invisible_part", sd)
    out = _run(m, inp)
    assert out.shape == (B, 1, size, size) and torch.isfinite(out).all()
    rep = {}
    for i in range(B):
        ref = _oracle(sd, enc, inp, i)
        rel, absrel = _errors(out[i:i + 1], ref, inp["mask01"][i:i + 1])
        rep[f"img{i}"] = dict(rel=rel, absrel=absrel)
        assert rel <= REL_TOL and absrel <= ABSREL_TOL, rep
        one = _run(m, {k: v[i:i + 1] for k, v in inp.items()})
        assert torch.equal(one, out[i:i + 1]), f"image {i} changes with the batch it is processed in"
    _record(f"{enc}_{size}_b{B}_pixel_tiles", rep)

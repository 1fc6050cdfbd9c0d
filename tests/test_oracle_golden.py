"""Pins the oracle: the CPU restatement (oracle/amodal_oracle.py) must reproduce the outputs and intermediates that the
unmodified reference produced for the same seeded weights/inputs (tests/golden/*.npz, made by make_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import amodal_oracle as O
from oracle import synth
from tests.golden_util import golden_names, load_golden, raw_golden_names, sample

# big encoders are exercised at small resolution; still the weights are generated in full
HEAVY = {"vitl_70_b1", "vitg_56_b1"}


@pytest.mark.parametrize("name", golden_names())
def test_oracle_matches_reference_golden(name):
    meta, z = load_golden(name)
    sd = synth.make_state_dict(meta["encoder"], meta["guide_type"], meta["seed"], meta["stress"])
    inp = synth.make_inputs(meta["B"], meta["H"], meta["W"], meta["seed"])
    inter = {}
    out = O.forward(sd, meta["encoder"], meta["guide_type"], inp["x"], inp["guide_rgb"], inp["guide_mask"],
                    inp["observation"], loss_stategy=meta["loss_stategy"], inter=inter)
    ref = torch.from_numpy(z["output"])
    assert out.shape == ref.shape == (meta["B"], 1, meta["H"], meta["W"])
    # same ATen ops on the same CPU; only thread-count dependent summation order may differ -> 2e-5 absolute
    assert (out - ref).abs().max().item() < 2e-5
    for key in z:
        if not key.startswith("s_"):
            continue
        k = key[2:]
        assert k in inter, f"oracle does not expose intermediate {k}"
        got = sample(inter[k])
        scale = max(float(np.abs(z[key]).max()), 1e-3)
        assert np.abs(got - z[key]).max() < 1e-4 * scale + 2e-5, k


def test_state_dict_template_counts():
    # SURVEY.md section 3.4 [probed]: 425 tensors for ViT-L, 649 for ViT-G
    assert len(synth.state_dict_shapes("vitl", "mask+observation")) == 425
    assert len(synth.state_dict_shapes("vitg", "mask+observation")) == 649


def test_guide_type_errors():
    with pytest.raises(NotImplementedError):
        O.build_guide("bogus", None, None, None)
    with pytest.raises(TypeError):
        O.build_guide("mask+observation", None, None, None)  # torch.cat of None, as the reference (SURVEY 8b)


def test_patch_size_assert():
    sd = synth.make_state_dict("vits", "none", 0)
    with pytest.raises(AssertionError):
        O.forward(sd, "vits", "none", torch.rand(1, 3, 60, 70))


@pytest.mark.parametrize("name", raw_golden_names())
def test_oracle_raw_matches_reference_golden(name):
    """Un-guided DepthAnythingV2 (depth_anything_v2_raw/dpt.py, SURVEY.md section 8 row f1): oracle.forward_raw against the
    output of the unmodified reference class on the same seeded weights/inputs."""
    meta, z = load_golden(name, "raw")
    sd = synth.make_state_dict_raw(meta["encoder"], meta["features"], meta["out_channels"], meta["seed"], meta["shift"])
    x = O.normalize_rgb(synth.make_inputs(meta["B"], meta["H"], meta["W"], meta["seed"])["x"])
    out = O.forward_raw(sd, meta["encoder"], x)
    ref = torch.from_numpy(z["output"])
    assert out.shape == ref.shape == (meta["B"], meta["H"], meta["W"])
    assert (out >= 0).all()
    assert (out - ref).abs().max().item() < 2e-5

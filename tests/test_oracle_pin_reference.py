"""Pin the oracle's torch restatement and our UNet to the reference's real modules, through what those modules computed
on seeded inputs (tests/golden/reference_modules.npz, written by tests/golden/make_reference_modules.py)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from read_b200 import synth


@pytest.fixture(scope="module")
def ref(synth_sd):
    g = load_golden("reference_modules")
    assert abs(synth.state_dict_checksum(synth_sd) - float(g["sd_checksum"])) < 1e-6 * float(g["sd_checksum"]), \
        "synthetic weights differ from the ones the fixture was generated with (torch RNG changed?)"
    return g


def _ref_state_dict(g):
    """The reference UNet's state_dict layout: zero tensors of its keys, shapes and dtypes."""
    return {str(k): torch.zeros(tuple(int(d) for d in s if d >= 0), dtype=getattr(torch, str(t)))
            for k, s, t in zip(g["sd_keys"], g["sd_shapes"], g["sd_dtypes"])}


def test_state_dict_keys_identical_to_reference(synth_sd, ref):
    ref_sd = _ref_state_dict(ref)
    assert set(ref_sd) == set(synth_sd)
    for k, v in ref_sd.items():
        assert tuple(v.shape) == tuple(synth_sd[k].shape), k
    from read_b200.unet import UNet as OurUNet
    ours = OurUNet().state_dict()
    assert list(sorted(ours)) == list(sorted(ref_sd))
    for k, v in ref_sd.items():
        assert tuple(v.shape) == tuple(ours[k].shape) and v.dtype == ours[k].dtype, k
    OurUNet().load_state_dict(ref_sd, strict=True)


def test_unet_oracle_equals_reference_module(synth_sd, ref):
    from oracle import unet_ref
    g = torch.Generator().manual_seed(7)
    H, W = 32, 48
    xs = [torch.rand((2, 8, H >> l, W >> l), generator=g) for l in range(5)]
    want = torch.from_numpy(ref["unet_out"])
    with torch.no_grad():
        got = unet_ref.unet_forward(synth_sd, xs)
    assert float((want - got).abs().max()) < 2e-5


def test_gather_oracle_equals_reference_module(ref):
    from oracle import unet_ref
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(0, 500, (3, 1, 9, 7), generator=g).float()
    np.testing.assert_array_equal(ids.numpy(), ref["ids"])
    want = torch.from_numpy(ref["gather_out"])
    got = unet_ref.point_texture(torch.from_numpy(ref["texture"]), ids)
    assert torch.equal(want, got)


def test_training_forward_of_our_unet_equals_reference(synth_sd, ref):
    """The library (autograd) path of read_b200.unet.UNet must agree with the reference on CPU."""
    from read_b200.unet import UNet as OurUNet
    ours = OurUNet()
    ours.load_state_dict(synth_sd)
    ours.eval()
    g = torch.Generator().manual_seed(11)
    xs = [torch.rand((1, 8, 32 >> l, 32 >> l), generator=g) for l in range(4)]
    want = torch.from_numpy(ref["train_out"])
    got = ours(*xs)                      # grad enabled -> torch path
    assert float((want - got).abs().max()) < 2e-5
    got.sum().backward()
    assert ours.get_submodule("feat_extract.0").block["conv_f"].weight.grad is not None

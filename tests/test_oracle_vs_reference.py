"""CPU: pins the oracle and the product's parameter tree to the UNMODIFIED reference, through the vectors
oracle/make_golden_reference.py recorded from it (tests/golden/reference_checks.pt).  Weights are rebuilt from the
seed by the product's own constructors and must hash to the reference's, bit for bit."""
import os
import torch
from oracle.make_golden import TINY_UNET
from oracle.make_golden_reference import state_digests

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def assert_same_params(sd, ref):
    got = state_digests(sd)
    assert got["n"] == ref["n"] and got["keys"] == ref["keys"], "parameter names / order differ from the reference"
    bad = [k for k, a, b in zip(sd, got["tensors"].tolist(), ref["tensors"].tolist()) if a != b]
    assert not bad, f"parameters differ from the reference: {bad[:5]}"


def _check_unet(g, padding_mode="zeros"):
    import cvpr23_lfdm_b200 as P
    from oracle import lfdm_oracle as O
    torch.manual_seed(g["seed"])
    sd = P.Unet3D(**dict(TINY_UNET, **g["kw"])).eval().state_dict()
    assert_same_params(sd, g["params"])
    with torch.no_grad():
        for cs, ref in g["out"].items():
            mine = O.unet3d_forward_with_cond_scale(sd, g["x"], g["t"], g["cond"], cs, heads=2, padding_mode=padding_mode)
            assert torch.equal(ref, mine)


def test_oracle_matches_reference_tiny(golden):
    _check_unet(golden("reference_checks.pt")["unet_tiny"])


def test_oracle_matches_reference_natops_style(golden):
    """nearest-upsample + reflect-padded 3x3 conv instead of ConvTranspose, learned null condition (NATOPS options,
    video_flow_diffusion.py:156-163,395-399): oracle == unmodified reference, bit for bit"""
    g = golden("reference_checks.pt")["unet_natops"]
    assert g["kw"] == dict(use_deconv=False, padding_mode="reflect", learn_null_cond=True)
    _check_unet(g, padding_mode="reflect")


def test_state_dict_and_init_identity(golden):
    """same seed -> bit-identical parameters & key order as the reference (drop-in checkpoints, seeded goldens)"""
    import cvpr23_lfdm_b200 as P
    cfg = os.path.join(ROOT, "config", "mug128.yaml")
    cases = golden("reference_checks.pt")["init_identity"]
    assert [c["kw"] for c in cases] == [dict(), dict(learn_null_cond=True, use_deconv=False, padding_mode="reflect")]
    for c in cases:
        torch.manual_seed(1234)
        m = P.FlowDiffusion(is_train=False, sampling_timesteps=3, config_pth=cfg, pretrained_pth="", **c["kw"])
        assert_same_params(m.state_dict(), c["params"])


def test_repo_config_matches_reference_model_params(golden):
    import yaml
    ref = golden("reference_checks.pt")["model_params"]
    for name in ("mug128", "mhad128", "natops128"):
        ours = yaml.safe_load(open(os.path.join(ROOT, "config", f"{name}.yaml")))["model_params"]
        assert ref[name] == ours

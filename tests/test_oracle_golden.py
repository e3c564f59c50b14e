"""The oracle restatement (oracle/casmvs_oracle.py) against the golden vectors the
REAL reference produced (oracle/make_golden.py).  CPU only.  Same torch ops in
the same order => bit-exact; that is asserted (torch.equal), not approximated."""
import pytest
import torch

from oracle import casmvs_oracle as O

pytestmark = pytest.mark.usefixtures("golden_threads")


def test_homo_warp_bit_exact(golden):
    g = golden("homo_warp")
    out = O.plane_sweep_warp(g["feat"], g["proj"], g["depth_values"])
    assert torch.equal(out, g["warped"])
    # the behind-camera view must have produced exact zeros somewhere
    assert (g["warped"][1] == 0).any()


def test_homo_warp_direct_form_close(golden):
    """direct bilinear at (u,v) == grid_sample form up to sampling-position ulps"""
    g = golden("homo_warp")
    out = O.plane_sweep_warp_direct(g["feat"], g["proj"], g["depth_values"])
    assert (out - g["warped"]).abs().max() < 2e-4


@pytest.mark.parametrize("tag", ["var_c8", "var_c32_v5"])
def test_variance_cost_bit_exact(golden, tag):
    g = golden("cost_" + tag)
    out = O.variance_cost_volume(g["feats"], g["proj"], g["depth_values"])
    assert torch.equal(out, g["cost"])


@pytest.mark.parametrize("tag", ["gwc_c16_g8", "gwc_c32_g8", "gwc_c32_g2"])
def test_groupwise_cost_bit_exact(golden, tag):
    g = golden("cost_" + tag)
    out = O.groupwise_cost_volume(g["feats"], g["proj"], g["depth_values"], int(g["G"]))
    assert torch.equal(out, g["cost"])


@pytest.mark.parametrize("cin", [8, 32])
def test_costreg_bit_exact(golden, cin):
    g = golden(f"costreg_c{cin}")
    sd = {"net." + k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    out = O.cost_regularize(g["x"], sd, "net.")
    assert torch.equal(out, g["logits"])


@pytest.mark.parametrize("D", [8, 32, 48, 64])
def test_regress_bit_exact(golden, D):
    g = golden(f"regress_d{D}")
    depth, conf, index, prob = O.regress_depth(g["logits"], g["depth_values"])
    assert torch.equal(depth, g["depth"])
    assert torch.equal(conf, g["confidence"])
    assert torch.equal(index, g["index"])
    assert torch.equal(prob, g["prob"])


def test_hypotheses_bit_exact(golden):
    g = golden("hypotheses")
    assert torch.equal(O.depth_hypotheses(g["cur"], 8, 2.65), g["hyp_float"])
    assert torch.equal(O.depth_hypotheses(g["cur"], 32, g["interval_tensor"]), g["hyp_tensor"])
    assert torch.equal(O.upsample_depth(g["low"]), g["up"])
    assert torch.equal(O.depth_hypotheses(O.upsample_depth(g["low"]), 32, 2.65 * 2), g["hyp_up"])
    # first plane = max(d - D/2*interval, 1e-7)   (modules.py:44)
    assert g["hyp_float"][0, 0, 0, 0].item() == pytest.approx(1e-7)


def _seeded(G):
    from oracle.make_golden import sd_checksum, seeded_state_dict
    sd = seeded_state_dict((8, 32, 48), (1, 2, 4), G, seed=0)
    return sd, sd_checksum(sd)


@pytest.mark.parametrize("tag,G", [("var", 1), ("gwc8", 8)])
def test_cascade_bit_exact(golden, tag, G):
    from casmvsnet_pl_b200 import synth
    g = golden(f"cascade_{tag}_160x128")
    sd, chk = _seeded(G)
    if chk != float(g["sd_checksum"]):
        pytest.skip("torch RNG/init drifted from the fixture's build; regenerate goldens")
    imgs, pm, dmin, dint = synth.make_inputs(B=1, V=3, W=160, H=128, seed=0)
    res = O.cascade_forward(sd, imgs, pm, dmin, dint, num_groups=G)
    for l in range(3):
        assert torch.equal(res[f"depth_{l}"], g[f"depth_{l}"])
        assert torch.equal(res[f"confidence_{l}"], g[f"confidence_{l}"])
    # the fixture must be a sensitive target: depth varies, softmax is peaked
    assert g["depth_0"].std() > 1.0


def test_cascade_tensor_params_bit_exact(golden):
    from casmvsnet_pl_b200 import synth
    g = golden("cascade_var_tensorparams_96x64")
    sd, chk = _seeded(1)
    if chk != float(g["sd_checksum"]):
        pytest.skip("torch RNG/init drifted from the fixture's build; regenerate goldens")
    imgs, pm, _, _ = synth.make_inputs(B=2, V=3, W=96, H=64, seed=1)
    res = O.cascade_forward(sd, imgs, pm, g["init_depth_min"], g["depth_interval"])
    for l in range(3):
        assert torch.equal(res[f"depth_{l}"], g[f"depth_{l}"])
        assert torch.equal(res[f"confidence_{l}"], g[f"confidence_{l}"])

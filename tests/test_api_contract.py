"""Drop-in boundary (SURVEY.md §8b): constructor, attributes, state-dict keys and
the no-CPU-fallback rule.  CPU only."""
import inspect
import json
import os

import pytest
import torch

from casmvsnet_pl_b200 import ABN, InPlaceABN, _lib, synth
from casmvsnet_pl_b200.models import modules as M
from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet, CostRegNet, FeatureNet


def test_reference_import_path_resolves():
    from models.mvsnet import CascadeMVSNet as C2      # train.py:9 / eval.py:11
    from models.modules import homo_warp, get_depth_values, depth_regression  # noqa: F401
    assert C2 is CascadeMVSNet


def test_constructor_and_attributes():
    sig = inspect.signature(CascadeMVSNet.__init__)
    assert list(sig.parameters)[:5] == ["self", "n_depths", "interval_ratios", "num_groups",
                                        "norm_act"]
    assert sig.parameters["n_depths"].default == [8, 32, 48]
    assert sig.parameters["interval_ratios"].default == [1, 2, 4]
    m = CascadeMVSNet(norm_act=ABN)
    assert m.levels == 3 and m.G == 1
    assert isinstance(m.feature, FeatureNet) and isinstance(m.cost_reg_2, CostRegNet)
    assert m.cost_reg_2.conv0.conv.weight.shape == (8, 32, 3, 3, 3)
    assert m.cost_reg_2.conv7[0].weight.shape == (64, 32, 3, 3, 3)      # ConvT: (in,out)
    assert m.cost_reg_0.prob.weight.shape == (1, 8, 3, 3, 3) and m.cost_reg_0.prob.bias.shape == (1,)
    g = CascadeMVSNet(num_groups=8, norm_act=InPlaceABN)
    assert g.cost_reg_1.conv0.conv.weight.shape == (8, 8, 3, 3, 3)
    for fn, params in ((M.homo_warp, ["src_feat", "proj_mat", "depth_values"]),
                       (M.get_depth_values, ["current_depth", "n_depths", "depth_interval"]),
                       (M.depth_regression, ["p", "depth_values"])):
        assert list(inspect.signature(fn).parameters) == params


def test_state_dict_has_206_reference_keys():
    sd = CascadeMVSNet(norm_act=ABN).state_dict()
    assert len(sd) == 206
    for k, shape in (("feature.conv0.0.conv.weight", (8, 3, 3, 3)),
                     ("feature.conv0.0.bn.running_var", (8,)),
                     ("feature.toplayer.bias", (32,)),
                     ("cost_reg_2.conv0.conv.weight", (8, 32, 3, 3, 3)),
                     ("cost_reg_2.conv7.1.running_mean", (32,)),
                     ("cost_reg_2.prob.bias", (1,))):
        assert tuple(sd[k].shape) == shape


@pytest.mark.parametrize("G", [1, 8])
def test_state_dict_equals_reference(G):
    """Keys, shapes and dtypes of the reference's state dict (oracle/make_golden.py ->
    tests/golden/reference_state_dict.json), in order, and a strict load of that layout."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "tests", "golden", "reference_state_dict.json")) as f:
        layout = json.load(f)[str(G)]
    a = {k: torch.zeros(shape, dtype=getattr(torch, dtype)) for k, shape, dtype in layout}
    ours = CascadeMVSNet(num_groups=G, norm_act=ABN)
    b = ours.state_dict()
    assert list(a) == list(b)
    assert all(a[k].shape == b[k].shape and a[k].dtype == b[k].dtype for k in a)
    ours.load_state_dict(a, strict=True)


def test_load_ckpt_roundtrip(tmp_path):
    """utils/__init__.py:52-80: Lightning 'model.'-prefixed checkpoint, update + strict load."""
    m = CascadeMVSNet(norm_act=ABN)
    synth.randomize_model_(m, 3)
    ck = {"state_dict": {"model." + k: v for k, v in m.state_dict().items()}}
    path = os.path.join(tmp_path, "ck.ckpt")
    torch.save(ck, path)
    loaded = torch.load(path, map_location="cpu")["state_dict"]
    stripped = {k[6:]: v for k, v in loaded.items() if k.startswith("model.")}
    m2 = CascadeMVSNet(norm_act=ABN)
    d = m2.state_dict()
    d.update(stripped)
    m2.load_state_dict(d)
    assert all(torch.equal(m.state_dict()[k], m2.state_dict()[k]) for k in d)


def test_cpu_tensors_are_rejected_loudly():
    m = CascadeMVSNet(norm_act=ABN).eval()
    imgs, pm, dmin, dint = synth.make_inputs(B=1, V=3, W=64, H=64)
    with pytest.raises(_lib.CasMVSError, match="no CPU fallback"):
        m(imgs, pm, dmin, dint)
    with pytest.raises(_lib.CasMVSError, match="no CPU fallback"):
        M.homo_warp(torch.zeros(1, 8, 8, 8), torch.zeros(1, 3, 4), torch.ones(1, 2, 8, 8))
    with pytest.raises(_lib.CasMVSError):
        M.get_depth_values(torch.ones(1, 1, 8, 8), 8, 2.65)


def test_product_never_imports_the_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    bad = []
    for base in ("casmvsnet_pl_b200", "models"):
        for dp, _, files in os.walk(os.path.join(root, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    txt = open(os.path.join(dp, f)).read()
                    if "oracle" in txt.replace("oracle-only", "").replace("the oracle", "") \
                            and ("import oracle" in txt or "from oracle" in txt):
                        bad.append(f)
    assert not bad, bad


def test_synthetic_geometry_keeps_samples_in_bounds():
    """SURVEY §8d: 88-99 % of samples inside the source image (benchmark not zero-filled)."""
    pm = synth.projection_matrices(3, 640, 512)
    w, h = 160, 128
    ys, xs = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
    for v in range(2):
        P = pm[v, 2]
        inside = []
        for d in (425.0, 680.0, 923.0):
            q = P[:, :3] @ torch.stack([xs.flatten(), ys.flatten(), torch.ones(h * w)]) + P[:, 3:] / d
            u, vv = q[0] / q[2], q[1] / q[2]
            inside.append(((u >= 0) & (u <= w - 1) & (vv >= 0) & (vv <= h - 1)).float().mean())
        assert min(inside) > 0.7 and max(inside) > 0.95

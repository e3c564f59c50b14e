"""The oracle against outputs of the original project's own modules on seeded inputs beyond the
cascade fixtures (oracle/make_golden.py -> tests/golden/reference_*.npz): predict_depth on a
stress pose with one source view behind the camera, and the feature pyramid.  Bit-exact."""
import pytest
import torch

from oracle import casmvs_oracle as O
from oracle import make_golden as MG

pytestmark = pytest.mark.usefixtures("golden_threads")


@pytest.mark.parametrize("G", [1, 4])
def test_predict_depth_matches_reference(golden, G):
    g = golden("reference_predict_depth")
    sd = MG.seeded_state_dict((8, 32, 48), (1, 2, 4), G, seed=5)
    assert MG.sd_checksum(sd) == float(g[f"G{G}/sd_checksum"]), "torch RNG/init drifted: regenerate goldens"
    feats, pms, dv = MG.predict_depth_inputs()
    with torch.no_grad():
        d_o, c_o = O.predict_depth(feats, pms, dv, sd, "cost_reg_1.", G)
    assert torch.equal(g[f"G{G}/depth"], d_o) and torch.equal(g[f"G{G}/confidence"], c_o)


def test_feature_pyramid_matches_reference(golden):
    g = golden("reference_feature_pyramid")
    sd = MG.seeded_state_dict((8, 32, 48), (1, 2, 4), 1, seed=2)
    assert MG.sd_checksum(sd) == float(g["sd_checksum"]), "torch RNG/init drifted: regenerate goldens"
    with torch.no_grad():
        b = O.feature_pyramid(MG.feature_pyramid_input(), sd)
    assert sorted(b) == ["level_0", "level_1", "level_2"]
    for k, v in b.items():
        assert list(v.shape) == g[f"{k}/shape"].tolist()
        sample = v.flatten()[MG.sample_index(v.numel())]
        assert torch.equal(sample, g[f"{k}/sample"]), (k, (sample - g[f"{k}/sample"]).abs().max())
        # every element: the reference's level, bit for bit
        assert MG.tensor_digest(v).tobytes() == g[f"{k}/sha256"].numpy().tobytes(), k

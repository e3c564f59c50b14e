"""Generate tests/golden/*.npz from the REAL reference (/root/reference), run on
CPU in the build container.  TEST INFRASTRUCTURE.

    python oracle/make_golden.py

The reference ships no golden vectors of its own (SURVEY.md §8c), so these
outputs of the reference itself are the pins for both the oracle restatement
(bit-exact) and the CUDA kernels (tolerances in tests/).  Fixtures are kept small;
every array needed to replay a case is stored inline except model weights, which
are regenerated from a seed (a checksum guards against RNG drift).
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from casmvsnet_pl_b200 import ABN, synth                      # noqa: E402
from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet      # noqa: E402
from oracle import ref_loader                                  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
# ATen and oneDNN split CPU reductions by thread count, so the bits of a fixture depend on it;
# the bit-exact tests run with the same count
GOLDEN_THREADS = 8


def seeded_state_dict(n_depths, interval_ratios, G, seed):
    torch.manual_seed(seed)
    m = CascadeMVSNet(n_depths=list(n_depths), interval_ratios=list(interval_ratios),
                      num_groups=G, norm_act=ABN)
    synth.randomize_model_(m, seed)
    return {k: v.clone() for k, v in m.state_dict().items()}


def sd_checksum(sd):
    return float(sum(v.double().abs().sum().item() for v in sd.values()))


class _Capture(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.volume = None

    def forward(self, x):
        self.volume = x.clone()
        return torch.zeros(x.shape[0], 1, *x.shape[2:])


def save(name, **arrays):
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **{k: (v.numpy() if torch.is_tensor(v) else np.asarray(v))
                                 for k, v in arrays.items()})
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KiB")


def main():
    torch.set_num_threads(GOLDEN_THREADS)
    mvsnet, modules, abn = ref_loader.load_reference_models()

    # ---- a1 homo_warp: stress geometry + behind-camera branch ------------------
    g = torch.Generator().manual_seed(11)
    B, C, h, w, D = 2, 8, 32, 40, 6
    feat = torch.randn(B, C, h, w, generator=g)
    pm = synth.projection_matrices(3, W=4 * w, H=4 * h, stress=True, behind_view=2)[:, 2]
    dv = 425.0 + 10.6 * torch.arange(D).float().reshape(1, D, 1, 1) \
        + 3.0 * torch.rand(B, D, h, w, generator=g)
    warped = modules.homo_warp(feat, pm, dv)
    save("homo_warp", feat=feat, proj=pm, depth_values=dv, warped=warped)

    # ---- a2/a3 cost volumes through the reference's own predict_depth ---------
    for tag, C, G, V in (("var_c8", 8, 1, 3), ("var_c32_v5", 32, 1, 5), ("gwc_c16_g8", 16, 8, 3),
                         ("gwc_c32_g8", 32, 8, 4), ("gwc_c32_g2", 32, 2, 3)):
        g = torch.Generator().manual_seed(hash(tag) % 1000 if False else len(tag) * 7 + C + G)
        B, h, w, D = 1, 24, 32, 8
        feats = torch.randn(B, V, C, h, w, generator=g)
        pms = synth.projection_matrices(V, W=4 * w, H=4 * h, stress=True)[:, 2].unsqueeze(0)
        dv = 500.0 + 21.2 * torch.arange(D).float().reshape(1, D, 1, 1) \
            + 5.0 * torch.rand(B, D, h, w, generator=g)
        model = mvsnet.CascadeMVSNet(num_groups=G, norm_act=abn).eval()
        if G == 1:
            model.training = True          # out-of-place branch, see ref_loader
        cap = _Capture()
        with torch.no_grad():
            model.predict_depth(feats, pms, dv, cap)
        save("cost_" + tag, feats=feats, proj=pms, depth_values=dv, cost=cap.volume,
             G=np.int64(G))

    # ---- a5 CostRegNet ---------------------------------------------------------
    for cin in (8, 32):
        torch.manual_seed(5 + cin)
        net = mvsnet.CostRegNet(cin, abn).eval()
        holder = torch.nn.Module()
        holder.cost_reg_0 = net
        gg = torch.Generator().manual_seed(77)
        with torch.no_grad():
            for m in net.modules():
                if hasattr(m, "running_var"):
                    n = m.running_mean.numel()
                    m.weight.copy_(torch.rand(n, generator=gg) + 0.5)
                    m.bias.copy_(torch.randn(n, generator=gg) * 0.1)
                    m.running_mean.copy_(torch.randn(n, generator=gg) * 0.1)
                    m.running_var.copy_(torch.rand(n, generator=gg) + 0.5)
            x = torch.randn(1, cin, 8, 16, 24, generator=gg)
            y = net(x)
        arrays = {"sd." + k: v for k, v in net.state_dict().items()}
        save(f"costreg_c{cin}", x=x, logits=y, **arrays)

    # ---- a6/a7 regression + confidence, via predict_depth with fixed logits ---
    class _Fixed(torch.nn.Module):
        def __init__(self, lg):
            super().__init__()
            self.lg = lg

        def forward(self, x):
            return self.lg.unsqueeze(1)

    for D in (8, 32, 48, 64):
        g = torch.Generator().manual_seed(100 + D)
        B, h, w = 2, 12, 20
        logits = torch.randn(B, D, h, w, generator=g) * 4.0
        dv = 425.0 + 2.65 * torch.arange(D).float().reshape(1, D, 1, 1) \
            + torch.rand(B, 1, h, w, generator=g) * 50
        dv = dv.contiguous()
        feats = torch.randn(B, 2, 8, h, w, generator=g)
        pms = synth.projection_matrices(2, W=4 * w, H=4 * h)[:, 2].unsqueeze(0).expand(B, -1, -1, -1)
        model = mvsnet.CascadeMVSNet(norm_act=abn).eval()
        model.training = True
        with torch.no_grad():
            depth, conf = model.predict_depth(feats, pms, dv, _Fixed(logits))
            prob = torch.softmax(logits, 1)
            index = modules.depth_regression(prob, torch.arange(D).float()).long().clamp(0, D - 1)
        save(f"regress_d{D}", logits=logits, depth_values=dv, depth=depth, confidence=conf,
             index=index, prob=prob)

    # ---- a8/a9/a10 hypotheses ---------------------------------------------------
    g = torch.Generator().manual_seed(3)
    cur = 500 + 100 * torch.rand(2, 1, 16, 24, generator=g)
    cur[0, 0, 0, :4] = torch.tensor([0.5, 3.0, 10.0, 21.0])   # exercises clamp_min(.,1e-7)
    hyp_f = modules.get_depth_values(cur, 8, 2.65)
    hyp_t = modules.get_depth_values(cur, 32, torch.tensor([[5.3], [4.1]]))
    low = 500 + 100 * torch.rand(2, 8, 12, generator=g)
    up = torch.nn.functional.interpolate(low.unsqueeze(1), scale_factor=2, mode="bilinear",
                                         align_corners=True)
    hyp_up = modules.get_depth_values(up, 32, 2.65 * 2)
    save("hypotheses", cur=cur, hyp_float=hyp_f, hyp_tensor=hyp_t,
         interval_tensor=torch.tensor([[5.3], [4.1]]), low=low, up=up, hyp_up=hyp_up)

    # ---- a11 full cascade, 160x128, V=3 -----------------------------------------
    for tag, G, nd in (("var", 1, (8, 32, 48)), ("gwc8", 8, (8, 32, 48))):
        sd = seeded_state_dict(nd, (1, 2, 4), G, seed=0)
        ref = ref_loader.make_reference_model(nd, (1, 2, 4), G)
        ref.load_state_dict(sd, strict=True)         # also checks the key contract
        imgs, pm, dmin, dint = synth.make_inputs(B=1, V=3, W=160, H=128, seed=0)
        with torch.no_grad():
            res = ref(imgs, pm, dmin, dint)
        save(f"cascade_{tag}_160x128", sd_checksum=np.float64(sd_checksum(sd)),
             **{k: v for k, v in res.items()})
    # tensor-valued depth params (training-style call, train.py:63-64), B=2
    sd = seeded_state_dict((8, 32, 48), (1, 2, 4), 1, seed=0)
    ref = ref_loader.make_reference_model((8, 32, 48), (1, 2, 4), 1)
    ref.load_state_dict(sd, strict=True)
    imgs, pm, _, _ = synth.make_inputs(B=2, V=3, W=96, H=64, seed=1)
    dmin = torch.tensor([[425.0], [430.0]])
    dint = torch.tensor([[2.65], [2.5]])
    with torch.no_grad():
        res = ref(imgs, pm, dmin, dint)
    save("cascade_var_tensorparams_96x64", sd_checksum=np.float64(sd_checksum(sd)),
         init_depth_min=dmin, depth_interval=dint, **{k: v for k, v in res.items()})
    reference_checks()


def predict_depth_inputs():
    """Seeded inputs of the predict_depth fixture: stress pose, one source view behind the
    camera, per-pixel hypotheses."""
    g = torch.Generator().manual_seed(9)
    feats = torch.randn(2, 4, 16, 16, 24, generator=g)
    pms = synth.projection_matrices(4, W=96, H=64, stress=True, behind_view=3)[:, 1]
    pms = pms.unsqueeze(0).expand(2, -1, -1, -1).contiguous()
    dv = 430.0 + 5.3 * torch.arange(16).float().reshape(1, 16, 1, 1) + torch.rand(2, 16, 16, 24, generator=g)
    return feats, pms, dv


def feature_pyramid_input():
    return torch.randn(2, 3, 64, 96, generator=torch.Generator().manual_seed(2))


def sample_index(n, k=1024):
    """Fixed, seeded positions at which a fixture stores the values of a large output."""
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k]


def tensor_digest(t):
    """SHA-256 of a float32 tensor's values in logical order: equal digests <=> torch.equal."""
    return np.frombuffer(hashlib.sha256(t.contiguous().numpy().tobytes()).digest(), np.uint8)


def reference_checks():
    """Fixtures of tests/test_oracle_vs_reference.py and the state-dict layout of
    tests/test_api_contract.py: the reference's predict_depth and feature pyramid on seeded
    inputs (the pyramid as a digest of each level plus a sample of its values)."""
    feats, pms, dv = predict_depth_inputs()
    out = {}
    for G in (1, 4):
        sd = seeded_state_dict((8, 32, 48), (1, 2, 4), G, seed=5)
        ref = ref_loader.make_reference_model((8, 32, 48), (1, 2, 4), G)
        ref.load_state_dict(sd)
        with torch.no_grad():
            d, c = ref.predict_depth(feats, pms, dv, ref.cost_reg_1)
        out.update({f"G{G}/sd_checksum": np.float64(sd_checksum(sd)), f"G{G}/depth": d,
                    f"G{G}/confidence": c})
    save("reference_predict_depth", **out)

    sd = seeded_state_dict((8, 32, 48), (1, 2, 4), 1, seed=2)
    ref = ref_loader.make_reference_model((8, 32, 48), (1, 2, 4), 1)
    ref.load_state_dict(sd)
    with torch.no_grad():
        pyr = ref.feature(feature_pyramid_input())
    out = {"sd_checksum": np.float64(sd_checksum(sd))}
    for k, v in pyr.items():
        out.update({f"{k}/shape": np.array(v.shape), f"{k}/sha256": tensor_digest(v),
                    f"{k}/sample": v.flatten()[sample_index(v.numel())]})
    save("reference_feature_pyramid", **out)

    # {"<num_groups>": [[key, shape, dtype], ...]} in state-dict order, one entry per line
    groups = []
    for G in (1, 8):
        sd = ref_loader.make_reference_model((8, 32, 48), (1, 2, 4), G).state_dict()
        rows = [json.dumps([k, list(v.shape), str(v.dtype).replace("torch.", "")]) for k, v in sd.items()]
        groups.append(f'"{G}": [\n' + ",\n".join(rows) + "\n]")
    path = os.path.join(OUT, "reference_state_dict.json")
    with open(path, "w") as f:
        f.write("{\n" + ",\n".join(groups) + "\n}\n")
    print(f"reference_state_dict: {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()

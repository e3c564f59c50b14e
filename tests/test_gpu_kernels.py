"""GPU parity tests proper: every kernel, called through the C ABI (ops.py ->
libcasmvs.so), against the golden vectors of the real reference and against the
CPU oracle on seeded inputs.  Tolerances are stated next to each assert.

Sampling-position note (K1): the kernel evaluates u = q_x/q_z directly; the
reference normalises to [-1,1] and grid_sample un-normalises (modules.py:83-89).
Both are fp32, so sample positions differ by a few ulp(u) (ulp(600 px) = 6e-5)
and a warped value by that times the local feature gradient.  Tolerances below
are expressed on that basis and the fp64 test shows the kernel is at least as
close to exact arithmetic as the reference is.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from casmvsnet_pl_b200 import _lib, ops, synth           # noqa: E402
from oracle import casmvs_oracle as O                    # noqa: E402
from test_gpu_tf32_exact import rna_tf32                 # noqa: E402

DEV = "cuda:0"


def cl(feats):
    """(B,V,C,h,w) -> same logical tensor, channels-last storage."""
    return feats.permute(0, 1, 3, 4, 2).contiguous().permute(0, 1, 4, 2, 3)


def stats(name, got, ref):
    err = (got - ref).abs()
    print(f"{name}: max|err|={err.max().item():.3e} mean|err|={err.mean().item():.3e} "
          f"max|ref|={ref.abs().max().item():.3e}")
    return err


# ----------------------------------------------------------------------------- K1
def test_homo_warp_vs_reference_golden(golden):
    g = golden("homo_warp")
    out = ops.homo_warp(g["feat"].to(DEV), g["proj"].to(DEV), g["depth_values"].to(DEV)).cpu()
    err = stats("homo_warp", out, g["warped"])
    # w=40: ulp(u) <= 4e-6, |grad| of N(0,1) texels ~ few units -> 5e-5 absolute
    assert err.max() < 5e-5
    # exact zeros where the reference has them (behind camera / out of bounds)
    assert torch.equal(out == 0, g["warped"] == 0)


@pytest.mark.parametrize("tag", ["var_c8", "var_c32_v5", "gwc_c16_g8", "gwc_c32_g8", "gwc_c32_g2"])
@pytest.mark.parametrize("layout", ["nchw_in_nchw_out", "nhwc_in_nhwc_out"])
def test_cost_volume_vs_reference_golden(golden, tag, layout):
    g = golden("cost_" + tag)
    G = int(g["G"])
    feats = g["feats"].to(DEV)
    if layout.startswith("nhwc"):
        feats = cl(feats)
    out_layout = ops.NHWC if layout.endswith("nhwc_out") else ops.NCHW
    out = ops.warp_cost(feats, g["proj"].to(DEV), g["depth_values"].to(DEV), G, out_layout)
    assert out.shape == g["cost"].shape
    err = stats(f"cost_{tag}/{layout}", out.cpu(), g["cost"])
    # variance of O(1) features: values up to ~10; sampling ulps + reciprocal-multiply
    # instead of /V (1 ulp each) -> 1e-4 absolute, 2e-5 relative to max
    assert err.max() < 1e-4
    assert err.max() / g["cost"].abs().max() < 2e-5


def test_cost_volume_no_less_accurate_than_reference_fp64():
    """Both fp32 implementations against an fp64 evaluation of the same formula."""
    g = torch.Generator().manual_seed(4)
    B, V, C, h, w, D = 1, 3, 16, 64, 80, 16
    feats = torch.randn(B, V, C, h, w, generator=g)
    pm = synth.projection_matrices(V, W=4 * w, H=4 * h, stress=True)[:, 2].unsqueeze(0)
    dv = 450.0 + 10.6 * torch.arange(D).float().reshape(1, D, 1, 1) + torch.rand(B, D, h, w, generator=g)
    ref32 = O.variance_cost_volume(feats, pm, dv)
    # fp64: direct bilinear, double arithmetic
    f64 = feats.double()
    S = f64[:, 0].unsqueeze(2).expand(-1, -1, D, -1, -1).clone()
    Q = S ** 2
    for v in range(1, V):
        wv = _warp_fp64(f64[:, v], pm[:, v - 1].double(), dv.double())
        S = S + wv
        Q = Q + wv ** 2
    ref64 = Q / V - (S / V) ** 2
    got = ops.warp_cost(feats.to(DEV), pm.to(DEV), dv.to(DEV), 1, ops.NCHW).cpu()
    e_ref = (ref32.double() - ref64).abs()
    e_got = (got.double() - ref64).abs()
    print(f"vs fp64: reference-fp32 max {e_ref.max():.3e} mean {e_ref.mean():.3e}; "
          f"kernel max {e_got.max():.3e} mean {e_got.mean():.3e}")
    assert e_got.mean() <= 1.5 * e_ref.mean() + 1e-9
    assert e_got.max() <= 3.0 * e_ref.max() + 1e-7


def _warp_fp64(src, P, dv):
    B, C, h, w = src.shape
    D = dv.shape[1]
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float64),
                            torch.arange(w, dtype=torch.float64), indexing="ij")
    out = torch.zeros(B, C, D, h, w, dtype=torch.float64)
    for b in range(B):
        p = P[b]
        qx = p[0, 0] * xs + p[0, 1] * ys + p[0, 2] + p[0, 3] / dv[b]
        qy = p[1, 0] * xs + p[1, 1] * ys + p[1, 2] + p[1, 3] / dv[b]
        qz = p[2, 0] * xs + p[2, 1] * ys + p[2, 2] + p[2, 3] / dv[b]
        u, v = qx / qz, qy / qz
        bad = qz <= 1e-7
        u[bad], v[bad] = w, h
        x0, y0 = torch.floor(u), torch.floor(v)
        fx, fy = u - x0, v - y0
        for dy, dx, wt in ((0, 0, (1 - fx) * (1 - fy)), (0, 1, fx * (1 - fy)),
                           (1, 0, (1 - fx) * fy), (1, 1, fx * fy)):
            xi, yi = x0 + dx, y0 + dy
            ok = (xi >= 0) & (xi <= w - 1) & (yi >= 0) & (yi <= h - 1)
            tap = src[b][:, yi.clamp(0, h - 1).long(), xi.clamp(0, w - 1).long()]
            out[b] += tap * (wt * ok)
    return out


def test_cost_volume_known_answers():
    """SURVEY §4.2: identity homography => warp == src for every plane; identical
    views + identity => variance == 0 exactly; gwc with identical views => mean(ref^2)."""
    g = torch.Generator().manual_seed(0)
    B, V, C, h, w, D = 2, 3, 16, 40, 56, 8
    ref = torch.randn(B, 1, C, h, w, generator=g)
    feats = ref.expand(-1, V, -1, -1, -1).contiguous().to(DEV)
    eye = torch.eye(3, 4).reshape(1, 1, 3, 4).expand(B, V - 1, -1, -1).contiguous().to(DEV)
    dv = (400 + 50 * torch.rand(B, D, h, w, generator=g)).to(DEV)
    wv = ops.homo_warp(feats[:, 1], eye[:, 0], dv)
    assert torch.equal(wv, feats[:, 1].unsqueeze(2).expand(-1, -1, D, -1, -1))
    var = ops.warp_cost(feats, eye, dv, 1, ops.NHWC)
    # Q/V - (S/V)^2 cancels to rounding: a few ulp of max(ref^2) ~ 20
    assert var.abs().max().item() < 1e-5
    gwc = ops.warp_cost(feats, eye, dv, 4, ops.NCHW)
    expect = (feats[:, 0] ** 2).reshape(B, 4, 4, h, w).mean(2).unsqueeze(2).expand(-1, -1, D, -1, -1)
    assert (gwc - expect).abs().max().item() < 1e-5
    # projection that puts every sample behind the camera: only the reference contributes
    behind = eye.clone()
    behind[:, :, 2, 2] = -1.0
    var_b = ops.warp_cost(feats, behind, dv, 1, ops.NCHW)
    r = feats[:, 0].unsqueeze(2)
    assert torch.allclose(var_b, (r * r / V - (r / V) ** 2).expand(-1, -1, D, -1, -1), atol=1e-6)


def test_cost_volume_many_views_and_edges():
    """generic (runtime-V) path, ragged pixel counts, B>1."""
    g = torch.Generator().manual_seed(2)
    for V, C, h, w, D in ((2, 8, 9, 13, 3), (6, 8, 17, 31, 5), (8, 16, 16, 24, 4)):
        B = 2
        feats = torch.randn(B, V, C, h, w, generator=g)
        pm = synth.projection_matrices(V, W=4 * w, H=4 * h, stress=True, behind_view=1)[:, 2]
        pm = pm.unsqueeze(0).expand(B, -1, -1, -1).contiguous()
        dv = 430.0 + 20 * torch.arange(D).float().reshape(1, D, 1, 1) + torch.rand(B, D, h, w, generator=g)
        want = O.variance_cost_volume(feats, pm, dv)
        got = ops.warp_cost(feats.to(DEV), pm.to(DEV), dv.to(DEV), 1, ops.NHWC).cpu()
        err = stats(f"var V={V}", got, want)
        assert err.max() < 1e-4


_STAGING_SHAPES = [(3, 8, 0), (3, 16, 1), (3, 32, 2), (5, 16, 1), (7, 32, 2), (2, 8, 0)]
_STAGING_CASES = ["smooth", "discontinuity", "wide_sweep", "stress_pose"]


def _staging_inputs(V, C, level, case, smooth_feats):
    g = torch.Generator().manual_seed(11 + level)
    W, H = 640, 512
    h, w = (H >> level) - 3, (W >> level) - 5           # ragged tiles at the right/bottom edge
    D = {0: 8, 1: 16, 2: 24}[level]
    feats = torch.randn(1, V, C, h, w, generator=g)
    if smooth_feats:                                    # band-limited: insensitive to ulp-level
        k = torch.tensor([1., 4., 6., 4., 1.])          # differences of the sampling position
        k = (k[:, None] * k[None, :]) / 256.0
        ff = torch.nn.functional.conv2d(feats.reshape(V * C, 1, h, w), k.reshape(1, 1, 5, 5), padding=2)
        feats = (ff / ff.std()).reshape(1, V, C, h, w)
    stress = case == "stress_pose"
    pm = synth.projection_matrices(V, W, H, stress=stress,
                                   behind_view=1 if stress else None)[:, level].unsqueeze(0)
    step = 2.65 * 2 ** level * (12.0 if case == "wide_sweep" else 1.0)
    base = 600.0 + 3.0 * torch.rand(1, 1, h, w, generator=g)
    if case == "discontinuity":
        base[..., :, w // 3:] -= 150.0                    # foreground / background step
        base[..., h // 2:, :] += 80.0
    dv = (base + step * torch.arange(D).float().reshape(1, D, 1, 1)).contiguous()
    return feats, pm, dv


@pytest.mark.parametrize("V,C,level", _STAGING_SHAPES)
@pytest.mark.parametrize("case", _STAGING_CASES)
def test_cost_volume_smem_staging_paths(V, C, level, case):
    """The TMA-staged K1 (csrc/warp_cost_smem.cu) against the oracle on inputs that exercise each
    of its paths: windows inside the staged box (smooth), windows outside it (a depth step
    inside the tile -> per-sample gather path), footprints larger than the box (wide sweep ->
    the CTA halves the run and re-stages), non-axis-aligned epipolar lines and samples behind
    the camera (stress pose); image sizes that are not multiples of the pixel tile.  Band-limited
    features: on white noise the reference's own normalise / un-normalise round trip (a few
    ulp(u), ulp(600) = 6e-5 px) already moves a variance by ~1e-3, which says nothing about the
    kernel; white noise is covered by test_cost_volume_staged_equals_gather."""
    feats, pm, dv = _staging_inputs(V, C, level, case, smooth_feats=True)
    want = O.variance_cost_volume(feats, pm, dv)
    got = ops.warp_cost(cl(feats.to(DEV)), pm.to(DEV), dv.to(DEV), 1, ops.NHWC).cpu()
    err = stats(f"smem-K1 V={V} C={C} {case}", got, want)
    # ulp(u) at u ~ 600 is 6e-5 px; the reference's round trip costs 2-3 of them
    tol = 2e-4 * want.abs().max().item() + 2e-4
    if case == "stress_pose":
        # one view crosses the q_z = 0 plane inside the sweep: next to it u = q_x/q_z is
        # ill-conditioned in fp32 for ANY implementation (d u = u * d q_z/q_z, q_z itself the
        # result of a cancellation), so the worst samples are not comparable; the bulk must be,
        # and test_cost_volume_staged_equals_gather pins those samples against the gather kernel
        assert torch.quantile(err.flatten()[:: max(1, err.numel() // 4000000)], 0.999).item() < tol
    else:
        assert err.max() < tol
    assert err.mean() < 2e-5


def test_cost_volume_staged_equals_gather(tmp_path):
    """White-noise features, every staging case: the TMA-staged kernel and the gather kernel
    (CASMVS_K1_SMEM=0, child process) evaluate the same positions and weights with the same
    operations, so they agree to accumulation-order level -- a wrong tap, weight, swizzle or box
    offset would show as an O(1) difference."""
    import os, subprocess, sys
    code = (
        "import sys, torch\n"
        "sys.path.insert(0, %r)\n"
        "sys.path.insert(0, %r)\n"
        "from casmvsnet_pl_b200 import ops\n"
        "import test_gpu_kernels as T\n"
        "out = {}\n"
        "for V, C, level in T._STAGING_SHAPES:\n"
        "    for case in T._STAGING_CASES:\n"
        "        f, pm, dv = T._staging_inputs(V, C, level, case, False)\n"
        "        out[(V, C, level, case)] = ops.warp_cost(T.cl(f.cuda()), pm.cuda(), dv.cuda(), 1, ops.NHWC).cpu()\n"
        "torch.save(out, sys.argv[1])\n" % (ROOT, os.path.join(ROOT, "tests")))
    res = []
    for smem in ("1", "0"):
        path = str(tmp_path / f"k1_{smem}.pt")
        env = dict(os.environ, CASMVS_K1_SMEM=smem)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=600)
        res.append(torch.load(path))
    worst = 0.0
    for key in res[0]:
        a, b = res[0][key], res[1][key]
        d = (a - b).abs().max().item() / b.abs().max().item()
        worst = max(worst, d)
        assert d < 2e-6, (key, d)
    print(f"staged vs gather kernel: worst max|diff|/max = {worst:.2e}")


# ----------------------------------------------------------------------------- K2
@pytest.mark.parametrize("cin", [8, 32])
@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("tf32", 3e-3)])
def test_costreg_vs_reference_golden(golden, cin, precision, tol):
    from casmvsnet_pl_b200 import ABN
    from casmvsnet_pl_b200.models.mvsnet import CostRegNet
    g = golden(f"costreg_c{cin}")
    net = CostRegNet(cin, ABN).eval()
    net.load_state_dict({k[3:]: v for k, v in g.items() if k.startswith("sd.")})
    net = net.to(DEV)
    net.precision = precision
    y = net(g["x"].to(DEV)).cpu()
    assert y.shape == g["logits"].shape
    err = stats(f"costreg c{cin} {precision}", y, g["logits"])
    # fp32: only accumulation-order differences over K=27*Cin terms (<= 2e-5 of max);
    # tf32: operands rounded to 10-bit mantissa, 11 layers deep (<= 3e-3 of max)
    assert err.max() / g["logits"].abs().max() < tol


@pytest.mark.parametrize("kind,stride,cin,cout,dims", [
    ("conv", 1, 8, 8, (4, 6, 10)), ("conv", 1, 16, 16, (3, 5, 7)), ("conv", 1, 64, 64, (2, 4, 5)),
    ("conv", 1, 8, 1, (4, 6, 9)), ("conv", 2, 8, 16, (8, 8, 16)), ("conv", 2, 32, 64, (4, 6, 6)),
    ("convT", 2, 64, 32, (1, 3, 5)), ("convT", 2, 16, 8, (4, 5, 6))])
def test_conv3d_layer_vs_torch_cpu(kind, stride, cin, cout, dims):
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(cin * 100 + cout)
    B = 2
    x = torch.randn(B, cin, *dims, generator=g)
    scale = torch.rand(cout, generator=g) + 0.5
    shift = torch.randn(cout, generator=g) * 0.1
    if kind == "conv":
        wt = torch.randn(cout, cin, 3, 3, 3, generator=g) * 0.1
        y = F.conv3d(x, wt, None, stride, 1)
        k = ops.CONV
    else:
        wt = torch.randn(cin, cout, 3, 3, 3, generator=g) * 0.1
        y = F.conv_transpose3d(x, wt, None, stride=2, padding=1, output_padding=1)
        k = ops.CONV_TRANSPOSE
    skip = torch.randn_like(y)
    want = F.leaky_relu(y * scale.reshape(1, -1, 1, 1, 1) + shift.reshape(1, -1, 1, 1, 1), 0.01) + skip
    wp = ops.pack_conv3d_weight(wt.to(DEV), k)
    got = ops.conv3d(x.to(DEV), wp, cin, cout, scale.to(DEV), shift.to(DEV), 0.01, skip.to(DEV),
                     k, stride, ops.FP32).cpu()
    assert got.shape == want.shape
    err = stats(f"{kind} s{stride} {cin}->{cout}", got, want)
    assert err.max() < 2e-5 * max(1.0, want.abs().max().item())


# ----------------------------------------------------------------------------- K3
@pytest.mark.parametrize("D", [8, 32, 48, 64])
def test_regress_vs_reference_golden(golden, D):
    g = golden(f"regress_d{D}")
    depth, conf, index, prob = ops.regress(g["logits"].to(DEV), g["depth_values"].to(DEV),
                                           want_index=True, want_prob=True)
    e_d = stats(f"depth D={D}", depth.cpu(), g["depth"])
    e_c = stats(f"conf  D={D}", conf.cpu(), g["confidence"])
    e_p = stats(f"prob  D={D}", prob.cpu(), g["prob"])
    assert (e_d / g["depth"].abs()).max() < 1e-6       # SURVEY §8c: depth <= 1e-6 rel
    assert e_c.max() < 1e-6 and e_p.max() < 1e-6
    # index: p differs by exp() ulps, so only pixels whose Σp·d sits within 1e-4 of an
    # integer may legitimately flip; everything else must be exact
    frac = (g["prob"] * torch.arange(D).float().reshape(1, D, 1, 1)).sum(1)
    safe = (frac - frac.round()).abs() > 1e-4
    assert torch.equal(index.cpu()[safe], g["index"][safe])


@pytest.mark.parametrize("D", [8, 32, 48, 64])
def test_regress_index_exact_given_identical_prob(golden, D):
    """north_star: pixel-index regression bit-exact.  Fed the reference's own p
    (input_is_prob), the kernel's index equals the reference's at EVERY pixel.

    The float sums are not asserted bit-equal: ATen's CPU sum over a non-innermost
    dim changes its association with the pixel's position inside the SIMD blocking
    (multi_row_sum for full 4x16-lane column blocks, a 4-way interleaved row_sum for
    the tail vectors) and with the thread partition, so "torch's order" is not a
    function of the D values alone.  The kernel uses the main-path order (sequential
    16-term chunks cascaded) everywhere; depth agrees to 2 ulp."""
    g = golden(f"regress_d{D}")
    depth, conf, index, _ = ops.regress(g["prob"].to(DEV), g["depth_values"].to(DEV),
                                        input_is_prob=True, want_index=True)
    assert torch.equal(index.cpu(), g["index"])
    assert ((depth.cpu() - g["depth"]).abs() / g["depth"]).max() < 2.4e-7
    assert (conf.cpu() - g["confidence"]).abs().max() < 2.4e-7


def test_regress_register_path_bit_identical(tmp_path):
    """The D = 8/32/48 register-resident K3 path performs the generic path's operations in the
    generic path's order: a child process with CASMVS_K3_REG=0 must reproduce it bit for bit."""
    import subprocess, sys
    code = (
        "import sys, torch\n"
        "sys.path.insert(0, %r)\n"
        "from casmvsnet_pl_b200 import ops\n"
        "out = {}\n"
        "for D in (8, 32, 48):\n"
        "    g = torch.Generator().manual_seed(D)\n"
        "    lg = (torch.randn(2, D, 37, 53, generator=g) * 3).cuda()\n"
        "    dv = (torch.rand(2, D, 37, 53, generator=g) * 500 + 400).cuda()\n"
        "    d, c, i, p = ops.regress(lg, dv, want_index=True, want_prob=True)\n"
        "    out[D] = [t.cpu() for t in (d, c, i, p)]\n"
        "torch.save(out, sys.argv[1])\n" % ROOT)
    import os
    paths = []
    for reg in ("1", "0"):
        path = str(tmp_path / f"k3_{reg}.pt")
        env = dict(os.environ, CASMVS_K3_REG=reg)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=300)
        paths.append(path)
    a, b = torch.load(paths[0]), torch.load(paths[1])
    for D in (8, 32, 48):
        for ta, tb in zip(a[D], b[D]):
            assert torch.equal(ta, tb)


def test_depth_regression_api_vector_depths(golden):
    from casmvsnet_pl_b200.models.modules import depth_regression
    g = golden("regress_d32")
    steps = torch.arange(32).float()
    got = depth_regression(g["prob"].to(DEV), steps.to(DEV)).cpu()
    want = O.regress_depth(g["logits"], steps)[0]
    assert torch.allclose(got, want, rtol=3e-7, atol=1e-6)
    assert torch.equal(got.long(), want.long())


# ----------------------------------------------------------------------------- K4
def test_hypotheses_bit_exact(golden):
    from casmvsnet_pl_b200.models.modules import get_depth_values
    g = golden("hypotheses")
    cur = g["cur"].to(DEV)
    assert torch.equal(get_depth_values(cur, 8, 2.65).cpu(), g["hyp_float"])
    assert torch.equal(get_depth_values(cur, 32, g["interval_tensor"].to(DEV)).cpu(), g["hyp_tensor"])
    up = ops.depth_hypotheses(g["low"].to(DEV), 32, 2.65 * 2, upsample=True).cpu()
    err = stats("upsample+ladder", up, g["hyp_up"])
    assert (err / g["hyp_up"].abs()).max() < 1e-6     # bilinear blend may differ in the last ulp
    uni = ops.uniform_hypotheses(425.0, 2.65 * 4, 48, 2, 4, 6, DEV).cpu()
    assert torch.equal(uni, O.initial_hypotheses(425.0, 2.65 * 4, 48, 2, 4, 6).contiguous())
    uni_t = ops.uniform_hypotheses(torch.tensor([[425.0], [430.0]]), torch.tensor([[10.6], [10.0]]),
                                   48, 2, 4, 6, DEV).cpu()
    assert torch.equal(uni_t, O.initial_hypotheses(torch.tensor([[425.0], [430.0]]),
                                                   torch.tensor([[10.6], [10.0]]), 48, 2, 4, 6).contiguous())


def test_layout_helpers_roundtrip():
    x = torch.randn(3, 16, 7, 11, device=DEV)
    y = torch.empty(3, 7, 11, 16, device=DEV)
    lib = _lib.load()
    s = ops._stream()
    _lib.check(lib.casmvs_nchw_to_nhwc(ops._ptr(x), ops._ptr(y), 3, 16, 77, s))
    assert torch.equal(y, x.permute(0, 2, 3, 1))
    z = torch.empty_like(x)
    _lib.check(lib.casmvs_nhwc_to_nchw(ops._ptr(y), ops._ptr(z), 3, 16, 77, s))
    assert torch.equal(z, x)


# ----------------------------------------------------------------------------- FPN (adjacent)
@pytest.mark.parametrize("clat,cout,hw", [(16, 16, (20, 28)), (8, 8, (34, 50))])
def test_fused_fpn_level_vs_torch_cpu(clat, cout, hw):
    """csrc/fpn.cu against the reference formula (models/mvsnet.py:36-52) in fp32 on the CPU."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(clat)
    h, w = hw
    N = 2
    prev = torch.randn(N, 32, h // 2, w // 2, generator=g)
    c = torch.randn(N, clat, h, w, generator=g)
    lat_w = torch.randn(32, clat, 1, 1, generator=g) * 0.2
    lat_b = torch.randn(32, generator=g) * 0.1
    sm_w = torch.randn(cout, 32, 3, 3, generator=g) * 0.1
    sm_b = torch.randn(cout, generator=g) * 0.1
    feat = F.interpolate(prev, scale_factor=2, mode="bilinear", align_corners=True) + F.conv2d(c, lat_w, lat_b)
    want = F.conv2d(feat, sm_w, sm_b, padding=1)
    gf, got = ops.fpn_level(prev.to(DEV), c.to(DEV), lat_w.to(DEV), lat_b.to(DEV), sm_w.to(DEV),
                            sm_b.to(DEV), want_feat=True)
    e1 = stats(f"fpn feat clat={clat}", gf.cpu(), feat)
    e2 = stats(f"fpn out  cout={cout}", got.cpu(), want)
    assert e1.max() < 2e-5 and e2.max() < 5e-5     # fp32 FMA, different summation order only
    assert ops.is_channels_last_feats(got)


@pytest.mark.parametrize("clat,hw,with_prev", [(16, (20, 28), True), (8, (34, 50), True),
                                               (32, (9, 13), False)])
def test_fpn_merge_vs_torch_cpu(clat, hw, with_prev):
    """csrc/fpn.cu fpn_merge_kernel == up2(prev) + lat(c) (models/mvsnet.py:36-47), fp32."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(clat + 7)
    h, w = hw
    prev = torch.randn(2, 32, h // 2, w // 2, generator=g) if with_prev else None
    c = torch.randn(2, clat, h, w, generator=g)
    lat_w = torch.randn(32, clat, 1, 1, generator=g) * 0.2
    lat_b = torch.randn(32, generator=g) * 0.1
    want = F.conv2d(c, lat_w, lat_b)
    if with_prev:
        want = want + F.interpolate(prev, scale_factor=2, mode="bilinear", align_corners=True)
    got = ops.fpn_merge(prev.to(DEV) if with_prev else None, c.to(DEV), lat_w.to(DEV), lat_b.to(DEV))
    assert stats(f"fpn_merge clat={clat}", got.cpu(), want).max() < 2e-5
    assert ops.is_channels_last_feats(got)
    got_r = ops.fpn_merge(prev.to(DEV) if with_prev else None, c.to(DEV), lat_w.to(DEV),
                          lat_b.to(DEV), round_tf32=True)
    # the rounded store is exactly cvt.rna.tf32 of the unrounded one (a truncating or
    # round-to-even store differs in the last TF32 bit)
    assert torch.equal(got_r.view(torch.int32), rna_tf32(got).view(torch.int32))


@pytest.mark.parametrize("hw", [(37, 141), (21, 144), (9, 1280)])
def test_conv2d_rgb8_vs_torch_cpu(hw):
    """First FeatureNet block (ConvBnReLU(3,8,3,1,1) with folded ABN) from planar images
    (one-pixel-per-thread kernel for ragged widths, four-pixel kernel for W % 4 == 0)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(3)
    x = torch.randn(3, 3, *hw, generator=g)
    w = torch.randn(8, 3, 3, 3, generator=g) * 0.3
    b = torch.randn(8, generator=g) * 0.1
    want = F.leaky_relu(F.conv2d(x, w, b, padding=1), 0.01)
    got = ops.conv2d_rgb8(x.to(DEV), w.to(DEV), b.to(DEV), 0.01)
    assert stats("conv2d_rgb8", got.cpu(), want).max() < 1e-5
    assert ops.is_channels_last_feats(got)


@pytest.mark.parametrize("cin,cout,hw", [(8, 8, (37, 61)), (16, 16, (40, 24)), (32, 32, (18, 30)),
                                         (32, 16, (33, 47)), (32, 8, (64, 90))])
def test_planar_conv_tensor_core_vs_torch_cpu(cin, cout, hw):
    """The 3x3 Conv2d layers of FeatureNet as a CONV_PLANAR (1x3x3) convolution over the
    (views, H, W) volume on tcgen05, against torch fp32 on the CPU; and the CUDA-core kernel
    running the same packed weights (zero outer planes) in fp32."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(cin + cout)
    x = torch.randn(5, cin, *hw, generator=g)
    w = torch.randn(cout, cin, 3, 3, generator=g) * 0.1
    b = torch.randn(cout, generator=g) * 0.1
    want = F.leaky_relu(F.conv2d(x, w, b, padding=1), 0.01)
    wp = ops.pack_conv3d_weight(w.to(DEV), ops.CONV_PLANAR)
    xs = x.to(DEV).contiguous(memory_format=torch.channels_last)
    ref = ops.conv2d_planar(xs, wp, cin, cout, b.to(DEV), 0.01, ops.FP32)
    assert stats(f"planar fp32 {cin}->{cout}", ref.cpu(), want).max() < 5e-5
    got = ops.conv2d_planar(xs, wp, cin, cout, b.to(DEV), 0.01, ops.TF32, keep_fp32=True)
    err = stats(f"planar tf32 {cin}->{cout}", got.cpu(), want)
    assert err.max() < 1.5e-3 * want.abs().max().item()
    assert ops.is_channels_last_feats(got)
    rounded = ops.conv2d_planar(xs, wp, cin, cout, b.to(DEV), 0.01, ops.TF32)
    assert torch.equal(rounded.view(torch.int32), rna_tf32(got).view(torch.int32))


@pytest.mark.parametrize("cin,cout,hw", [(8, 16, (64, 96)), (16, 32, (36, 50)), (8, 16, (18, 34))])
def test_conv2d_5x5s2_tensor_core_vs_torch_cpu(cin, cout, hw):
    """FeatureNet's 5x5 stride-2 blocks on tcgen05 (even/odd TMA planes, 25 taps) vs torch fp32."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(cin * 7 + cout)
    x = torch.randn(3, cin, *hw, generator=g)
    w = torch.randn(cout, cin, 5, 5, generator=g) * 0.05
    b = torch.randn(cout, generator=g) * 0.1
    want = F.leaky_relu(F.conv2d(x, w, b, stride=2, padding=2), 0.01)
    wp = ops.pack_conv2d_5x5s2_weight(w.to(DEV))
    got = ops.conv2d_5x5s2(x.to(DEV).contiguous(memory_format=torch.channels_last), wp,
                           b.to(DEV), 0.01)
    assert got.shape == want.shape and ops.is_channels_last_feats(got)
    err = stats(f"5x5s2 {cin}->{cout}", got.cpu(), want)
    assert err.max() < 1.5e-3 * want.abs().max().item()


# ----------------------------------------------------------------------------- K2 on tcgen05
@pytest.mark.parametrize("kind,cin,cout,dims", [
    ("conv1", 8, 8, (5, 20, 13)), ("conv1", 16, 8, (16, 40, 24)), ("conv1", 32, 8, (8, 32, 40)),
    ("conv1", 16, 16, (6, 32, 24)), ("conv1", 32, 32, (4, 16, 16)), ("conv1", 8, 1, (8, 32, 16)),
    ("conv1", 64, 64, (3, 16, 24)),
    ("conv2", 8, 16, (8, 32, 40)), ("conv2", 16, 32, (6, 20, 24)), ("conv2", 32, 64, (4, 16, 16)),
    ("convT", 16, 8, (5, 18, 11)), ("convT", 32, 16, (3, 16, 16)), ("convT", 64, 32, (2, 16, 24))])
def test_tensor_core_conv_vs_cuda_core_fp32(kind, cin, cout, dims):
    """Every CostRegNet layer type on the tcgen05 path (tf32 operands, fp32 accumulate) against
    the fp32 CUDA-core kernel on the same inputs (ragged tiles, halos, skip, ABN epilogue).
    Operands carry 10 mantissa bits => relative error ~2^-11 per product, K = 27*Cin terms."""
    g = torch.Generator().manual_seed(cin * 131 + cout)
    x = torch.randn(2, cin, *dims, generator=g).to(DEV)
    scale = (torch.rand(cout, generator=g) + 0.5).to(DEV)
    shift = (torch.randn(cout, generator=g) * 0.1).to(DEV)
    if kind == "convT":
        wt = (torch.randn(cin, cout, 3, 3, 3, generator=g) * 0.1).to(DEV)
        k, stride = ops.CONV_TRANSPOSE, 2
        skip = torch.randn(2, cout, *[2 * d for d in dims], generator=g).to(DEV)
    else:
        wt = (torch.randn(cout, cin, 3, 3, 3, generator=g) * 0.1).to(DEV)
        k, stride = ops.CONV, (1 if kind == "conv1" else 2)
        skip = torch.randn(2, cout, *dims, generator=g).to(DEV) if kind == "conv1" and cout > 1 else None
    wp = ops.pack_conv3d_weight(wt, k)
    ref = ops.conv3d(x, wp, cin, cout, scale, shift, 0.01, skip, k, stride, ops.FP32)
    got = ops.conv3d(x, wp, cin, cout, scale, shift, 0.01, skip, k, stride, ops.TF32)
    assert got.shape == ref.shape
    err = stats(f"tc {kind} {cin}->{cout}", got.cpu(), ref.cpu())
    assert err.max() < 1.5e-3 * ref.abs().max().item()
    assert not torch.isnan(got).any()

"""The tcgen05 convolutions against an exact model of what they compute, at the layer shapes of
the benchmarked configurations.

Model of one tf32 layer: the operands are TF32 values (weights rounded to nearest by the weight-
image builders, activations already rounded by their producer), their products are exact in
float64, and the kernel sums them in fp32.  The reference is the same convolution in float64 on
the rounded operands, followed by the epilogue lrelu(acc * scale + shift) + skip in float64.  Per
output voxel the kernel may differ from it by at most

    (K/8 + 8) * 2^-22 * A  +  2^-22 * (|lrelu part| + |skip|),   A = |scale| * conv(|x|, |w|)

with K = taps * Cin: a worst-case bound for fp32 accumulation of exact products, with a factor of
2 for adders that do not round to nearest.  Truncating instead of rounding one operand moves an
all-positive result by about 2^-12 * A, which is 4x (Cin = 64) to 30x (Cin = 8) that bound, so a
wrong rounding mode, a stale halo value or a wrong tile fails at the voxel where it happens.

The stored output is checked separately: by default it is rna_tf32 of the unrounded
(CASMVS_KEEP_FP32_OUT) output, bit for bit; the prob head (Cout = 1) is never rounded.
"""
import inspect
import math
import os
import subprocess
import sys
import time
import zlib
from collections import namedtuple

import pytest
import torch
import torch.nn.functional as F

from casmvsnet_pl_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
U22 = 2.0 ** -22
SLOPE = 0.01                    # inplace_abn LeakyReLU default (casmvs_costreg_fwd)
gpu = pytest.mark.gpu


# ----------------------------------------------------------------------------- TF32 bit model
def rna_tf32(t):
    """cvt.rna.tf32.f32 on float32: round the 13 dropped mantissa bits to nearest, ties away
    from zero (the carry may run into the exponent)."""
    return ((t.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def trunc_tf32(t):
    """What an MMA that reads fp32 bits as tf32 sees: the 13 low mantissa bits dropped."""
    return (t.view(torch.int32) & ~0x1FFF).view(torch.float32)


def _bits(*words):
    return torch.tensor([w - (1 << 32) if w >= 1 << 31 else w for w in words],
                        dtype=torch.int32).view(torch.float32)


def test_tf32_bit_model_fixed_patterns():
    x = _bits(0x3F801000,     # 1 + 2^-11: a tie, rounds away from zero
              0x3F800FFF,     # just below the tie
              0x3F803000,     # 1 + 3 * 2^-11: odd tie, still away from zero (not to even)
              0xBF801000,     # -(1 + 2^-11): negative tie, away from zero
              0xC0A01FFF,     # negative, rounds up in magnitude
              0x3FFFF000,     # 2 - 2^-12: the mantissa carry runs into the exponent -> 2.0
              0x00000000,     # +0
              0x80000000,     # -0
              0x3F802000)     # already a TF32 value: unchanged
    rna = _bits(0x3F802000, 0x3F800000, 0x3F804000, 0xBF802000, 0xC0A02000, 0x40000000,
                0x00000000, 0x80000000, 0x3F802000)
    trunc = _bits(0x3F800000, 0x3F800000, 0x3F802000, 0xBF800000, 0xC0A00000, 0x3FFFE000,
                  0x00000000, 0x80000000, 0x3F802000)
    assert torch.equal(rna_tf32(x).view(torch.int32), rna.view(torch.int32))
    assert torch.equal(trunc_tf32(x).view(torch.int32), trunc.view(torch.int32))
    assert rna_tf32(x)[5].item() == 2.0 and rna_tf32(x)[3].item() == -(1 + 2.0 ** -10)
    # on random values: both land on TF32 values, within one (trunc) / half (rna) TF32 ulp
    g = torch.Generator().manual_seed(0)
    v = torch.randn(10000, generator=g) * 100
    for f, ulps in ((rna_tf32, 0.5), (trunc_tf32, 1.0)):
        r = f(v)
        assert torch.equal(r.view(torch.int32) & 0x1FFF, torch.zeros_like(r, dtype=torch.int32))
        assert ((r - v).abs() <= ulps * 2.0 ** -10 * v.abs()).all()
    assert (trunc_tf32(v).abs() <= v.abs()).all()


# ----------------------------------------------------------------------------- layer specs
# kind: "conv" (3x3x3, stride 1|2), "convT" (transposed, stride 2), "planar" (1x3x3 over the
# (views, H, W) volume, B = 1), "p5" (FeatureNet's 5x5 stride-2 Conv2d, B = 1, D = views).
# role: "bn" (scale + shift + LeakyReLU(0.01)), "prob" (bias only, scale 1, slope 1), "block"
# (FeatureNet block: shift + LeakyReLU, scale folded into w), "smooth" (bias only).
# skip: None, "rand" or the key of an earlier layer of the same sweep whose stored output it is.
Layer = namedtuple("Layer", "kind stride B cin cout D h w role skip")
_TAPS = {"conv": 27, "convT": 27, "planar": 9, "p5": 25}
_KIND_CODE = {"conv": ops.CONV, "convT": ops.CONV_TRANSPOSE, "planar": ops.CONV_PLANAR}


def _key(L):
    return (L.kind, L.stride, L.B, L.cin, L.cout, L.D, L.h, L.w, L.role, L.skip)


def _out_dims(L):
    if L.kind == "convT":
        return 2 * L.D, 2 * L.h, 2 * L.w
    if L.kind == "p5":
        return L.D, (L.h - 1) // 2 + 1, (L.w - 1) // 2 + 1
    s = L.stride
    return (L.D - 1) // s + 1, (L.h - 1) // s + 1, (L.w - 1) // s + 1


def kernel_kind(L):
    """The tcgen05 kernel the library's default dispatch picks for this layer (for reports)."""
    if L.kind == "p5":
        return "tma2-P5"
    if L.kind == "convT":
        return "tma2-T"
    if L.kind == "conv" and L.stride == 2:
        return "tma2-S2"
    pl = "-planar" if L.kind == "planar" else ""
    if L.cout <= 8 and L.cin in (8, 16, 32):
        return "n8" + pl + ("-cout1" if L.cout == 1 else "")
    return "tma" + pl + ("-deep" if L.cin == 64 else "")


def costreg_stage(B, cin, D, h, w):
    """The 11 CostRegNet layers (casmvs_costreg_layer_info) with their dims propagated and the
    skip additions of conv7 / conv9 / conv11 wired to the stored outputs of conv4 / conv2 / conv0."""
    out, keys = [], []
    skip_src = {7: 4, 8: 2, 9: 0}
    for i in range(11):
        info = ops.costreg_layer_info(cin, i)
        kind = "convT" if info["kind"] == ops.CONV_TRANSPOSE else "conv"
        skip = keys[skip_src[i]] if i in skip_src else None
        L = Layer(kind, info["stride"], B, info["cin"], info["cout"], D, h, w,
                  "prob" if i == 10 else "bn", skip)
        out.append(L)
        keys.append(_key(L))
        D, h, w = _out_dims(L)
    return out


def feature_layers(N, H, W):
    """FeatureNet's tcgen05 layers over a batch of N images of H x W (tf32 tensor path)."""
    H2, W2 = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    H4, W4 = (H2 - 1) // 2 + 1, (W2 - 1) // 2 + 1
    P = lambda ci, co, h, w, role: Layer("planar", 1, 1, ci, co, N, h, w, role, None)  # noqa: E731
    return [P(8, 8, H, W, "block"),                                         # conv0.1
            Layer("p5", 2, 1, 8, 16, N, H, W, "block", None),               # conv1.0
            P(16, 16, H2, W2, "block"), P(16, 16, H2, W2, "block"),         # conv1.1, conv1.2
            Layer("p5", 2, 1, 16, 32, N, H2, W2, "block", None),            # conv2.0
            P(32, 32, H4, W4, "block"), P(32, 32, H4, W4, "block"),         # conv2.1, conv2.2
            P(32, 16, H2, W2, "smooth"), P(32, 8, H, W, "smooth")]          # smooth1, smooth0


def _full_configs():
    from test_gpu_cascade import FULL_CONFIGS
    return FULL_CONFIGS


def config_stages(c, levels=(2, 1, 0)):
    """(B, cin, D, h, w) of the CostRegNet input at each cascade stage of a configuration."""
    return [(1, c["G"] if c["G"] > 1 else 8 * 2 ** l, c["n_depths"][l], c["H"] >> l, c["W"] >> l)
            for l in levels]


def config_layers(c, levels=(2, 1, 0)):
    layers = feature_layers(c["V"], c["H"], c["W"])
    for st in config_stages(c, levels):
        layers += costreg_stage(*st)
    return layers


def edge_layers():
    """Shapes where the persistent kernels go wrong if they do: a prime depth above every depth-
    chunk cap (tma / tma2 <= 32, n8 <= 21), so any chunk pick leaves a ragged last chunk; B = 2;
    h and w that are multiples of neither 8x16 (tma / tma2 tiles) nor 30x4 (n8 tiles)."""
    D, h, w = 37, 17, 61
    L = [Layer("conv", 1, 2, ci, 8, D, h, w, "bn", None) for ci in (8, 16, 32)]   # n8
    L += [Layer("conv", 1, 2, 8, 1, D, h, w, "prob", None),                       # n8 Cout = 1
          Layer("conv", 1, 2, 16, 16, D, h, w, "bn", "rand"),                     # tma
          Layer("conv", 1, 2, 32, 32, D, h, w, "bn", None),
          Layer("conv", 1, 2, 64, 64, D, 9, 13, "bn", None)]                      # tma deep
    # stride 2 with output depth 37 (from 73 and 74 input planes)
    L += [Layer("conv", 2, 2, ci, co, Di, 35, 47, "bn", None)
          for (ci, co), Di in zip(((8, 16), (16, 32), (32, 64)), (73, 74, 73))]
    L += [Layer("convT", 2, 2, ci, co, D, 9, 13, "bn", "rand")
          for ci, co in ((16, 8), (32, 16), (64, 32))]
    L += [Layer("planar", 1, 1, ci, co, 2, 17, 61, role, None)
          for ci, co, role in ((8, 8, "block"), (16, 16, "block"), (32, 32, "block"),
                               (32, 16, "smooth"), (32, 8, "smooth"))]
    L += [Layer("p5", 2, 1, 8, 16, 2, 35, 61, "block", None),
          Layer("p5", 2, 1, 16, 32, 2, 17, 31, "block", None)]
    return L


def dedupe(layers):
    seen, out = set(), []
    for L in layers:
        if _key(L) not in seen:
            seen.add(_key(L))
            out.append(L)
    return out


def new_layers(name):
    """The layers of a configuration that no configuration before it in FULL_CONFIGS has (the
    skip source of a new conv7 / conv9 / conv11 is always new too: its key holds the same dims)."""
    seen = set()
    for n, c in _full_configs().items():
        layers = dedupe(config_layers(c))
        if n == name:
            return [L for L in layers if _key(L) not in seen]
        seen.update(_key(L) for L in layers)
    raise KeyError(name)


def with_positive_variants(layers):
    """One all-positive copy (x, w, scale, shift > 0) of the smallest layer of each kernel kind:
    there every operand rounded the wrong way moves the result the same way."""
    best = {}
    for L in layers:
        k = kernel_kind(L)
        n = L.B * L.D * L.h * L.w * L.cin
        if k not in best or n < best[k][0]:
            best[k] = (n, L)
    pos = [L._replace(role=L.role + "+pos", skip=None if L.skip is None else "rand")
           for _, L in best.values()]
    return layers + pos


# ----------------------------------------------------------------------------- inputs / kernels
def _gen(L, what):
    g = torch.Generator(device=DEV)
    g.manual_seed(zlib.crc32(repr((_key(L), what)).encode()))
    return g


def layer_params(L):
    """Seeded weights (torch layout), scale, shift of a layer (device tensors)."""
    pos = L.role.endswith("+pos")
    role = L.role.replace("+pos", "")
    g = _gen(L, "params")
    K = _TAPS[L.kind] * L.cin
    if L.kind == "conv":
        shape = (L.cout, L.cin, 3, 3, 3)
    elif L.kind == "convT":
        shape = (L.cin, L.cout, 3, 3, 3)
    elif L.kind == "planar":
        shape = (L.cout, L.cin, 3, 3)
    else:
        shape = (L.cout, L.cin, 5, 5)
    w = torch.randn(shape, generator=g, device=DEV) / math.sqrt(K)
    scale = torch.rand(L.cout, generator=g, device=DEV) + 0.5 if role == "bn" else None
    shift = torch.randn(L.cout, generator=g, device=DEV) * 0.1
    if role == "prob":
        scale = torch.ones(L.cout, device=DEV)
    if pos:
        w, shift = w.abs(), shift.abs()
    return w, scale, shift


def layer_slope(L):
    return SLOPE if L.role.replace("+pos", "") in ("bn", "block") else 1.0


def layer_input(L, rounded=True):
    """Channels-last storage (B, D, h, w, Cin) of a random activation, TF32-rounded like every
    stored activation of the tf32 mode (rounded=False: the raw fp32 values)."""
    x = torch.randn(L.B, L.D, L.h, L.w, L.cin, generator=_gen(L, "x"), device=DEV)
    if L.role.endswith("+pos"):
        x = x.abs() + 2.0 ** -6
    return rna_tf32(x) if rounded else x


def random_skip(L):
    Do, ho, wo = _out_dims(L)
    s = torch.randn(L.B, Do, ho, wo, L.cout, generator=_gen(L, "skip"), device=DEV)
    return rna_tf32(s)


def pack(L, w):
    if L.kind == "p5":
        return ops.pack_conv2d_5x5s2_weight(w)
    return ops.pack_conv3d_weight(w, _KIND_CODE[L.kind])


def run_layer(L, xs, wp, scale, shift, skip, keep):
    """One library call: casmvs_conv3d_fwd through ctypes (CASMVS_KEEP_FP32_OUT OR-ed into the
    precision when keep) or, for p5, casmvs_conv2d_5x5s2_fwd.  Returns the output storage."""
    Do, ho, wo = _out_dims(L)
    if L.kind == "p5":
        x4 = xs[0].permute(0, 3, 1, 2)                       # (N,Cin,H,W) channels-last view
        y = ops.conv2d_5x5s2(x4, wp, shift, layer_slope(L), round_tf32=not keep)
        return y.permute(0, 2, 3, 1).unsqueeze(0)
    y = torch.empty(L.B, Do, ho, wo, L.cout, device=DEV)
    flags = ops.TF32 | (ops.KEEP_FP32_OUT if keep else 0)
    _lib.check(_lib.load().casmvs_conv3d_fwd(
        ops._ptr(xs), ops._ptr(wp), ops._ptr(scale), ops._ptr(shift), float(layer_slope(L)),
        ops._ptr(skip), ops._ptr(y), L.B, L.cin, L.cout, L.D, L.h, L.w, _KIND_CODE[L.kind],
        L.stride, flags, ops._stream()), "conv3d")
    return y


# ----------------------------------------------------------------------------- fp64 model
def _conv64(L, x, w):
    """x storage (B,D,h,w,Cin) float64, w torch layout float64 -> storage (B,Do,ho,wo,Cout)."""
    if L.kind in ("planar", "p5"):
        xi = x[0].permute(0, 3, 1, 2).contiguous()
        y = F.conv2d(xi, w, stride=L.stride, padding=1 if L.kind == "planar" else 2)
        return y.permute(0, 2, 3, 1).unsqueeze(0)
    xl = x.permute(0, 4, 1, 2, 3).contiguous()
    if L.kind == "conv":
        y = F.conv3d(xl, w, stride=L.stride, padding=1)
    else:
        y = F.conv_transpose3d(xl, w, stride=2, padding=1, output_padding=1)
    return y.permute(0, 2, 3, 4, 1)


def model_check(L, xs, w, scale, shift, skip, got, operand=rna_tf32):
    """Largest err / bound over the output (the layer passes when it is <= 1).  xs are the
    values the kernel was given; the model applies `operand` to them (identity on activations
    that are already TF32) and rna_tf32 to the weights."""
    x64 = operand(xs).double()
    w64 = rna_tf32(w.contiguous()).double()
    acc = _conv64(L, x64, w64)
    A = _conv64(L, x64.abs(), w64.abs())
    if scale is not None:
        s64 = scale.double()
        acc = acc * s64
        A = A * s64.abs()
    v = acc + (shift.double() if shift is not None else 0.0)
    del acc
    pre = torch.where(v >= 0, v, v * layer_slope(L))
    del v
    ref = pre if skip is None else pre + skip.double()
    K = _TAPS[L.kind] * L.cin
    bound = (K / 8 + 8) * U22 * A
    del A
    bound += U22 * pre.abs()
    del pre
    if skip is not None:
        bound += U22 * skip.double().abs()
    err = (got.double() - ref).abs()
    del ref
    # err > 0 where the bound is 0 counts as infinitely far out
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound).max().item()
    return ratio


def store_ok(L, keep, default):
    """Default store == rna_tf32(unrounded store), bit for bit; the prob head is never rounded."""
    if L.cout == 1:
        return torch.equal(default.view(torch.int32), keep.view(torch.int32)) and \
            bool(((keep.view(torch.int32) & 0x1FFF) != 0).any())
    return torch.equal(default.view(torch.int32), rna_tf32(keep).view(torch.int32))


# ----------------------------------------------------------------------------- sweeps
def run_sweep(layers):
    """Run every layer (unrounded and default store) on its seeded inputs.  Yields
    (L, xs, w, scale, shift, skip, keep_out, store_ok).  A layer whose skip is an earlier
    layer's output uses that layer's stored (rounded) output, as the CostRegNet driver does."""
    stored = {}
    needed = {L.skip for L in layers if L.skip not in (None, "rand")}
    for L in layers:
        w, scale, shift = layer_params(L)
        xs = layer_input(L)
        skip = None
        if L.skip == "rand":
            skip = random_skip(L)
        elif L.skip is not None:
            skip = stored[L.skip]
        wp = pack(L, w)
        keep = run_layer(L, xs, wp, scale, shift, skip, True)
        default = run_layer(L, xs, wp, scale, shift, skip, False)
        if _key(L) in needed:
            stored[_key(L)] = default
        yield L, xs, w, scale, shift, skip, keep, store_ok(L, keep, default)


def check_sweep(layers, title):
    worst, bad = {}, []
    t0 = time.time()
    for L, xs, w, scale, shift, skip, keep, rounded in run_sweep(layers):
        finite = bool(torch.isfinite(keep).all())
        r = model_check(L, xs, w, scale, shift, skip, keep)
        k = kernel_kind(L) + ("+pos" if L.role.endswith("+pos") else "")
        worst[k] = max(worst.get(k, 0.0), r)
        if not (finite and r <= 1.0 and rounded):
            bad.append(f"{k} {_key(L)}: err/bound {r:.3g} finite {finite} store-rounding {rounded}")
    torch.cuda.synchronize()
    print(f"{title}: {len(layers)} layers in {time.time() - t0:.1f} s; worst err/bound per kernel:")
    for k in sorted(worst):
        print(f"  {k:<22} {worst[k]:.4f}")
    return bad


@gpu
@pytest.mark.parametrize("name", ["cfg2", "cfg3_gwc8", "cfg4_view", "cfg5_half", "edge"])
def test_layers_match_exact_tf32_model(name):
    """Every tcgen05 layer of a benchmarked configuration (FeatureNet's planar and 5x5 stride-2
    blocks at the full image size, the 11 CostRegNet layers of each cascade stage), or the edge
    shapes, against the fp64 model within the fp32-accumulation bound, with the default store
    bit-exactly rounded; a tcgen05 kernel covers every configuration layer."""
    layers = edge_layers() if name == "edge" else new_layers(name)
    layers = with_positive_variants(layers)
    fb0 = _lib.fallback_count()
    bad = check_sweep(layers, name)
    assert _lib.fallback_count() == fb0, "a tf32 layer fell back to the CUDA-core kernel"
    assert not bad, "\n".join(bad)


# ----------------------------------------------------------------------------- driver chain
def _costreg_net(cin, seed):
    from casmvsnet_pl_b200 import ABN
    from casmvsnet_pl_b200.models.mvsnet import CostRegNet
    torch.manual_seed(seed)
    net = CostRegNet(cin, ABN)
    g = torch.Generator().manual_seed(seed + 1000)
    with torch.no_grad():
        for m in net.modules():
            if hasattr(m, "running_mean") and hasattr(m, "running_var"):
                n = m.running_mean.numel()
                m.weight.copy_(torch.rand(n, generator=g) + 0.5)
                m.bias.copy_(torch.randn(n, generator=g) * 0.1)
                m.running_mean.copy_(torch.randn(n, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(n, generator=g) + 0.5)
        net.prob.weight.mul_(50.0)
    net = net.eval().to(DEV)
    net.precision = "tf32"
    return net


def new_stages(name):
    """The stages of a configuration that no configuration before it in FULL_CONFIGS has."""
    seen = set()
    for n, c in _full_configs().items():
        if n == name:
            return [st for st in config_stages(c) if st not in seen]
        seen.update(config_stages(c))
    raise KeyError(name)


@gpu
@pytest.mark.parametrize("name", ["cfg2", "cfg3_gwc8", "cfg4_view", "cfg5_half"])
def test_costreg_driver_equals_layer_chain(name):
    """casmvs_costreg_fwd at every full-size stage equals, bit for bit, the chain of its 11
    layers called one by one with the blob's own weights, scales and shifts (located by
    casmvs_costreg_layer_info) and conv4 / conv2 / conv0 as the skips of conv7 / conv9 / conv11:
    this pins the driver's workspace offsets and skip wiring.  Each link is checked against the
    fp64 model of its actual input, so errors cannot compound unnoticed."""
    bad, worst = [], {}
    for B, cin, D, h, w in new_stages(name):
        net = _costreg_net(cin, seed=cin * 1000 + D)
        blob = net.packed_params()
        g = torch.Generator(device=DEV)
        g.manual_seed(D * 7 + h)
        x = rna_tf32(torch.randn(B, D, h, w, cin, generator=g, device=DEV))
        logits = ops.costreg(ops.as_volume_view(x), blob, cin, ops.TF32)
        layers = costreg_stage(B, cin, D, h, w)
        outs = []
        for i, L in enumerate(layers):
            info = ops.costreg_layer_info(cin, i)
            nw = 27 * L.cin * L.cout
            wp = blob[info["w_off"]:info["w_off"] + nw]
            scale = blob[info["scale_off"]:info["scale_off"] + L.cout]
            shift = blob[info["shift_off"]:info["shift_off"] + L.cout]
            xin = x if i == 0 else outs[i - 1]
            skip = {7: 4, 8: 2, 9: 0}.get(i)
            skip = outs[skip] if skip is not None else None
            keep = run_layer(L, xin, wp, scale, shift, skip, True)
            y = run_layer(L, xin, wp, scale, shift, skip, False)
            outs.append(y)
            wt = net._layer_tensors(net._ORDER[i])[0].detach()
            r = model_check(L, xin, wt, scale, shift, skip, keep)
            k = kernel_kind(L)
            worst[k] = max(worst.get(k, 0.0), r)
            if not (r <= 1.0 and store_ok(L, keep, y) and bool(torch.isfinite(keep).all())):
                bad.append(f"stage {(B, cin, D, h, w)} layer {i} ({k}): err/bound {r:.3g}")
            del keep
        same = torch.equal(outs[-1].reshape(B, D, h, w), logits)
        if not same:
            d = (outs[-1].reshape(B, D, h, w) - logits).abs().max().item()
            bad.append(f"stage {(B, cin, D, h, w)}: driver logits != layer chain (max|diff| {d:.3e})")
        del outs, logits, blob, net
    print(f"{name} chain: worst err/bound per kernel: " +
          ", ".join(f"{k} {v:.4f}" for k, v in sorted(worst.items())))
    assert not bad, "\n".join(bad)


# ----------------------------------------------------------------------------- switch variants
# The kernel variants the shipped defaults were chosen among (DESIGN.md, profiles/r2_switch_ab.txt);
# the switches are read once per process, so each setting runs in a child process.
VARIANTS = {
    "n8_sets2_none": {"CASMVS_N8_SETS2_MASK": "0"},
    "n8_sets2_all": {"CASMVS_N8_SETS2_MASK": "7"},
    "n8_slots8_6": {"CASMVS_N8_SETS2_MASK": "0", "CASMVS_N8_SLOTS8": "6"},
    "no_n8": {"CASMVS_N8": "0"},          # Cout <= 8 layers and prob on conv3d_tma
    "one_cta_per_sm": {"CASMVS_TMA_PER_SM": "1", "CASMVS_N8_PER_SM": "1",
                       "CASMVS_TMA2_PER_SM": "1"},
    "dchunk3": {"CASMVS_TMA_DCHUNK": "3", "CASMVS_N8_DCHUNK": "3"},
}


def moderate_layers():
    """The first (coarsest) cascade stage of every configuration plus the edge shapes."""
    layers = []
    for c in _full_configs().values():
        layers += [L for L in config_layers(c, levels=(2,)) if L.kind not in ("planar", "p5")]
    return dedupe(layers + edge_layers())


def child_main(path):
    """Runs in a child process with a switch set: every moderate layer, unrounded outputs saved
    for the parent, plus the store-rounding verdicts and the fallback count."""
    fb0 = _lib.fallback_count()
    outs, rounded = {}, {}
    with torch.no_grad():
        for L, xs, w, scale, shift, skip, keep, ok in run_sweep(moderate_layers()):
            outs[_key(L)] = keep.cpu()
            rounded[_key(L)] = ok
        torch.cuda.synchronize()
    torch.save({"outs": outs, "rounded": rounded, "fallbacks": _lib.fallback_count() - fb0}, path)


@gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_switch_variants_match_exact_tf32_model(variant, tmp_path):
    path = str(tmp_path / f"{variant}.pt")
    code = ("import sys\n"
            "sys.path.insert(0, %r)\n"
            "sys.path.insert(0, %r)\n"
            "import test_gpu_tf32_exact as T\n"
            "T.child_main(sys.argv[1])\n" % (ROOT, os.path.join(ROOT, "tests")))
    env = dict(os.environ, **VARIANTS[variant])
    subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=1200)
    res = torch.load(path)
    os.remove(path)
    assert res["fallbacks"] == 0, f"{variant}: {res['fallbacks']} layers fell back"
    bad, worst = [], {}
    stored = {}
    layers = moderate_layers()
    needed = {L.skip for L in layers if L.skip not in (None, "rand")}
    for L in layers:
        w, scale, shift = layer_params(L)
        xs = layer_input(L)
        skip = random_skip(L) if L.skip == "rand" else stored[L.skip] if L.skip else None
        keep = res["outs"][_key(L)].to(DEV)
        if _key(L) in needed:             # the child's stored skip: rna of its unrounded store
            stored[_key(L)] = keep if L.cout == 1 else rna_tf32(keep)
        r = model_check(L, xs, w, scale, shift, skip, keep)
        k = kernel_kind(L)
        worst[k] = max(worst.get(k, 0.0), r)
        if not (r <= 1.0 and res["rounded"][_key(L)] and bool(torch.isfinite(keep).all())):
            bad.append(f"{variant} {k} {_key(L)}: err/bound {r:.3g} "
                       f"store-rounding {res['rounded'][_key(L)]}")
    print(f"{variant}: worst err/bound per layer type: " +
          ", ".join(f"{k} {v:.4f}" for k, v in sorted(worst.items())))
    assert not bad, "\n".join(bad)


# ----------------------------------------------------------------------------- round flags
def _same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _cl(feats):
    return feats.permute(0, 1, 3, 4, 2).contiguous().permute(0, 1, 4, 2, 3)


@gpu
@pytest.mark.parametrize("V,C,G,layout", [(3, 8, 1, "cl"), (3, 32, 8, "cl"), (2, 16, 1, "cl"),
                                          (5, 16, 1, "cl"), (3, 16, 1, "nchw"), (7, 8, 1, "cl")])
def test_warp_cost_round_flag_is_rna(V, C, G, layout):
    """K1's ROUND_TF32 store (staged and gather kernels, variance and group-wise correlation)
    is exactly rna_tf32 of its unrounded store; so is the ladder entry's."""
    from casmvsnet_pl_b200 import synth
    g = torch.Generator().manual_seed(V * 100 + C)
    h, w, D = 37, 53, 8
    feats = torch.randn(1, V, C, h, w, generator=g).to(DEV)
    if layout == "cl":
        feats = _cl(feats)
    pm = synth.projection_matrices(V, W=4 * w, H=4 * h, stress=True)[:, 2].unsqueeze(0).to(DEV)
    dv = (430.0 + 20 * torch.arange(D).float().reshape(1, D, 1, 1)
          + torch.rand(1, D, h, w, generator=g)).to(DEV)
    for out_layout in (ops.NHWC, ops.NCHW):
        a = ops.warp_cost(feats, pm, dv, G, out_layout)
        b = ops.warp_cost(feats, pm, dv, G, out_layout, round_tf32=True)
        assert ((a.contiguous().view(torch.int32) & 0x1FFF) != 0).any()
        assert _same_bits(b, rna_tf32(a.contiguous()))
    if layout == "cl" and ops.ladder_supported(V, C, G):
        first = (600.0 + 3.0 * torch.rand(1, h, w, generator=g)).to(DEV)
        for f in (first, 425.0):
            lad = ops.Ladder(f, 2.65, D, 1, h, w, DEV)
            a = ops.warp_cost_ladder(feats, pm, lad, G)
            b = ops.warp_cost_ladder(feats, pm, lad, G, round_tf32=True)
            assert _same_bits(b, rna_tf32(a.contiguous()))


@gpu
@pytest.mark.parametrize("hw", [(37, 141), (21, 144)])
def test_conv2d_rgb8_round_flag_is_rna(hw):
    g = torch.Generator().manual_seed(5)
    x = torch.randn(3, 3, *hw, generator=g).to(DEV)
    w = (torch.randn(8, 3, 3, 3, generator=g) * 0.3).to(DEV)
    b = (torch.randn(8, generator=g) * 0.1).to(DEV)
    a = ops.conv2d_rgb8(x, w, b, 0.01)
    r = ops.conv2d_rgb8(x, w, b, 0.01, round_tf32=True)
    assert _same_bits(r, rna_tf32(a.contiguous()))


@gpu
def test_bias_act_round_flag_is_rna():
    g = torch.Generator().manual_seed(6)
    x = torch.randn(2, 16, 13, 21, generator=g).to(DEV).contiguous(memory_format=torch.channels_last)
    b = (torch.randn(16, generator=g) * 0.1).to(DEV)
    a = ops.bias_lrelu_(x.clone(), b, 0.01)
    r = ops.bias_lrelu_(x.clone(), b, 0.01, round_tf32=True)
    assert _same_bits(r, rna_tf32(a.contiguous()))


# ----------------------------------------------------------------------------- operand invariant
@gpu
def test_tensor_core_operands_are_rounded_along_the_model(monkeypatch):
    """Every activation a tcgen05 conv receives in the tf32 forward (FeatureNet's 5x5 stride-2
    and planar blocks, the CostRegNet input) is a TF32 value: the MMA reads its operand by
    truncation, so an unrounded operand would be biased toward zero."""
    from casmvsnet_pl_b200 import ABN, synth
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet
    from oracle.make_golden import seeded_state_dict
    sd = seeded_state_dict((8, 32, 48), (1, 2, 4), 1, seed=0)
    model = CascadeMVSNet(num_groups=1, norm_act=ABN, precision="tf32")
    model.load_state_dict(sd)
    model = model.eval().to(DEV)
    seen = []

    def spy(name, is_tf32):
        fn = getattr(ops, name)
        sig = inspect.signature(fn)

        def wrapper(*a, **k):
            args = sig.bind(*a, **k)
            args.apply_defaults()
            if is_tf32(args.arguments):
                seen.append((name, next(iter(args.arguments.values()))))
            return fn(*a, **k)
        monkeypatch.setattr(ops, name, wrapper)

    spy("conv2d_5x5s2", lambda a: True)
    spy("conv2d_planar", lambda a: a["precision"] == ops.TF32)
    spy("costreg", lambda a: a["precision"] == ops.TF32)
    imgs, pm, dmin, dint = synth.make_inputs(B=1, V=3, W=160, H=128, seed=0)
    model(imgs.to(DEV), pm.to(DEV), dmin, dint)
    torch.cuda.synchronize()
    counts = {n: sum(1 for s, _ in seen if s == n) for n in ("conv2d_5x5s2", "conv2d_planar", "costreg")}
    assert counts == {"conv2d_5x5s2": 2, "conv2d_planar": 7, "costreg": 3}, counts
    bad = [f"{n} #{i}: {int(((t.view(torch.int32) & 0x1FFF) != 0).sum())} of {t.numel()} "
           "values are not TF32" for i, (n, t) in enumerate(seen)
           if ((t.view(torch.int32) & 0x1FFF) != 0).any()]
    assert not bad, "\n".join(bad)


@gpu
@pytest.mark.parametrize("L", [Layer("conv", 1, 1, 8, 8, 8, 32, 64, "bn+pos", None),      # n8
                               Layer("conv", 1, 1, 16, 16, 8, 32, 64, "bn+pos", None),    # tma
                               Layer("conv", 2, 1, 8, 16, 8, 32, 64, "bn+pos", None)],    # tma2
                         ids=lambda L: kernel_kind(L))
def test_mma_truncates_unrounded_operands(L):
    """The hardware behaviour the rounding convention rests on (DESIGN.md, include/casmvs.h):
    fed unrounded fp32 activations, the tf32 MMA uses them truncated.  All-positive operands, so
    the truncation model fits within the bound and the round-to-nearest model does not."""
    w, scale, shift = layer_params(L)
    xs = layer_input(L, rounded=False)
    assert ((xs.view(torch.int32) & 0x1FFF) != 0).float().mean() > 0.99
    keep = run_layer(L, xs, pack(L, w), scale, shift, None, True)
    r_trunc = model_check(L, xs, w, scale, shift, None, keep, operand=trunc_tf32)
    r_rna = model_check(L, xs, w, scale, shift, None, keep, operand=rna_tf32)
    print(f"{kernel_kind(L)}: err/bound vs truncated-operand model {r_trunc:.4f}, "
          f"vs rounded-operand model {r_rna:.2f}")
    assert r_trunc <= 1.0
    assert r_rna > 2.0

"""``CascadeMVSNet`` with the reference's constructor, attributes, state-dict
keys and forward contract (reference models/mvsnet.py:107-244), running the
three-stage hot path on the B200 kernels.

Host side (this file) is glue: it owns the parameters, runs the 2D FeatureNet
with PyTorch/cuDNN in channels-last (so the fused warp kernel gets HWC features
without a transpose) and sequences K4 -> K1 -> K2 -> K3 per stage.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from ..norm_act import activation_slope, folded_scale_shift
from .modules import *  # noqa: F401,F403  (reference does the same, mvsnet.py:5)
from .modules import ConvBnReLU, ConvBnReLU3D, InPlaceABN


class FeatureNet(nn.Module):
    """3-level FPN (reference models/mvsnet.py:7-57).  Inference on the GPU runs entirely on this
    library's kernels in both precision modes (tf32: tcgen05 planar / 5x5 convs; fp32: CUDA-core
    FMA kernels); PyTorch modules are only the parameter holders and the training / CPU path."""

    def __init__(self, norm_act=InPlaceABN):
        super().__init__()
        self.conv0 = nn.Sequential(ConvBnReLU(3, 8, 3, 1, 1, norm_act=norm_act),
                                   ConvBnReLU(8, 8, 3, 1, 1, norm_act=norm_act))
        self.conv1 = nn.Sequential(ConvBnReLU(8, 16, 5, 2, 2, norm_act=norm_act),
                                   ConvBnReLU(16, 16, 3, 1, 1, norm_act=norm_act),
                                   ConvBnReLU(16, 16, 3, 1, 1, norm_act=norm_act))
        self.conv2 = nn.Sequential(ConvBnReLU(16, 32, 5, 2, 2, norm_act=norm_act),
                                   ConvBnReLU(32, 32, 3, 1, 1, norm_act=norm_act),
                                   ConvBnReLU(32, 32, 3, 1, 1, norm_act=norm_act))
        self.toplayer = nn.Conv2d(32, 32, 1)
        self.lat1 = nn.Conv2d(16, 32, 1)
        self.lat0 = nn.Conv2d(8, 32, 1)
        self.smooth1 = nn.Conv2d(32, 16, 3, padding=1)
        self.smooth0 = nn.Conv2d(32, 8, 3, padding=1)

    @staticmethod
    def _up2(x):
        return F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)

    # cuDNN would run fp32 convs as TF32 on B200 by default; the reference path is fp32
    # (opt.py:69-70), so IEEE fp32 is kept unless the model runs in its tf32 precision mode.
    allow_tf32 = False
    # tf32 precision mode, inference: the 3x3 stride-1 and 5x5 stride-2 convs run on tcgen05 as
    # planar convolutions over the (views, H, W) volume, the first block and the top-down
    # merges in this library's own kernels: no cuDNN kernel is left on this path
    tensor_path = True
    # the reference's inference script turns cuDNN autotuning on (eval.py:19); without it
    # cuDNN's heuristics pick FFT/sgemm algorithms that are several times slower here
    benchmark = True

    def forward(self, x, overlap=False):
        """overlap=True (tf32 inference path only): the two finer pyramid levels are produced on a
        side stream and the result carries "_ready" = {level: event}; the caller must make its
        stream wait for the event before touching that level (CascadeMVSNet.forward does, so the
        coarsest cascade stage -- many small, latency-bound kernels -- runs concurrently with the
        bandwidth-heavy top-down half of the pyramid)."""
        with torch.backends.cudnn.flags(enabled=True, benchmark=self.benchmark,
                                        allow_tf32=self.allow_tf32):
            if self.training or torch.is_grad_enabled():
                return self._forward_modules(x)
            if self.allow_tf32 and self.tensor_path and x.is_cuda:
                return self._forward_tensor(x, overlap)
            return self._forward_folded(x)

    # -- inference path: eval-mode ABN folded into the conv (w*alpha, beta') so each block
    #    is one cuDNN conv with bias + an in-place LeakyReLU instead of conv + BN + act
    def _folded(self):
        from ..norm_act import activation_slope, folded_scale_shift
        blocks = [m for seq in (self.conv0, self.conv1, self.conv2) for m in seq]
        key = tuple((t.data_ptr(), t._version) for b in blocks for t in
                    (b.conv.weight, b.bn.weight, b.bn.bias, b.bn.running_mean, b.bn.running_var))
        if getattr(self, "_fold_key", None) != key:
            cache = []
            for b in blocks:
                a, beta = folded_scale_shift(b.bn)
                w = (b.conv.weight.detach() * a.reshape(-1, 1, 1, 1)).contiguous(
                    memory_format=torch.channels_last)
                cache.append((w, beta.contiguous(), b.conv.stride, b.conv.padding,
                              activation_slope(b.bn)))
            self._fold_cache, self._fold_key = cache, key
        return self._fold_cache

    # -- tf32 inference path (see `tensor_path`)
    def _packed(self):
        cache = self._folded()
        key = self._fold_key
        if getattr(self, "_pack_key", None) != key:
            for old in getattr(self, "_pack_cache", {}).values():
                ops.release_weight_images(old)
            packed = {}
            for i in (1, 3, 4, 6, 7):               # the 3x3 stride-1 blocks
                w = cache[i][0]
                packed[i] = ops.pack_conv3d_weight(w.contiguous(), ops.CONV_PLANAR)
            for i in (2, 5):                        # the 5x5 stride-2 blocks: plain (O,I,5,5)
                packed[i] = ops.pack_conv2d_5x5s2_weight(cache[i][0])
            self._pack_cache, self._pack_key = packed, key
        skey = tuple((t.data_ptr(), t._version) for t in (self.smooth0.weight, self.smooth1.weight))
        if getattr(self, "_smooth_key", None) != skey:
            for old in getattr(self, "_smooth_pack", ()):
                ops.release_weight_images(old)
            self._smooth_pack = (ops.pack_conv3d_weight(self.smooth0.weight.detach(), ops.CONV_PLANAR),
                                 ops.pack_conv3d_weight(self.smooth1.weight.detach(), ops.CONV_PLANAR))
            self._smooth_key = skey
        return cache, self._pack_cache, self._smooth_pack

    def _forward_tensor(self, x, overlap=False):
        cache, packed, (sm0, sm1) = self._packed()

        def planar(t, i, keep):
            w, b, _, _, slope = cache[i]
            return ops.conv2d_planar(t, packed[i], w.shape[1], w.shape[0], b, slope, ops.TF32,
                                     keep_fp32=keep)

        def strided(t, i):
            _, b, _, _, slope = cache[i]
            return ops.conv2d_5x5s2(t, packed[i], b, slope, round_tf32=True)

        w0, b0, _, _, slope0 = cache[0]
        t = ops.conv2d_rgb8(x, w0, b0, slope0, round_tf32=True)
        # c0 and c1 feed the next 5x5 stride-2 tcgen05 conv, which reads its operand by
        # truncation: stored rounded to nearest (the fp32 lateral merges then read a value within
        # half a TF32 ulp, unbiased).  c2 is read by the fp32 toplayer merge only.
        c0 = planar(t, 1, False)
        c1 = planar(planar(strided(c0, 2), 3, False), 4, False)
        c2 = planar(planar(strided(c1, 5), 6, False), 7, True)
        f2 = ops.fpn_merge(None, c2, self.toplayer.weight, self.toplayer.bias)

        def top_down():
            m1 = ops.fpn_merge(f2, c1, self.lat1.weight, self.lat1.bias, round_tf32=True)
            l1 = ops.conv2d_planar(m1, sm1, 32, 16, self.smooth1.bias, 1.0, ops.TF32,
                                   keep_fp32=True)
            return m1, l1

        def finest(m1):
            m0 = ops.fpn_merge(m1, c0, self.lat0.weight, self.lat0.bias, round_tf32=True)
            return ops.conv2d_planar(m0, sm0, 32, 8, self.smooth0.bias, 1.0, ops.TF32,
                                     keep_fp32=True)

        if not overlap:
            m1, l1 = top_down()
            return {"level_0": finest(m1), "level_1": l1, "level_2": f2}
        main = torch.cuda.current_stream(x.device)
        side = getattr(self, "_side_stream", None)
        if side is None or side.device != x.device:
            side = self._side_stream = torch.cuda.Stream(device=x.device)
        side.wait_stream(main)                       # c0, c1, f2 are complete for the side stream
        with torch.cuda.stream(side):
            m1, l1 = top_down()
            ev1 = torch.cuda.Event()
            ev1.record(side)
            l0 = finest(m1)
            ev0 = torch.cuda.Event()
            ev0.record(side)
        for t in (l1, l0):                           # consumed on the caller's stream
            t.record_stream(main)
        for t in (c0, c1, f2):                       # produced on main, read on the side stream
            t.record_stream(side)
        return {"level_0": l0, "level_1": l1, "level_2": f2, "_ready": {1: ev1, 0: ev0}}

    def _forward_folded(self, x):
        """fp32 inference path.  On the GPU every layer runs on this library's CUDA-core fp32
        kernels (bit-faithful products, no cuDNN / cuBLAS kernel anywhere): first block
        straight from the planar image batch, 3x3 blocks as planar convolutions over the
        (views, H, W) volume, 5x5 stride-2 blocks, then the fused top-down levels."""
        cache = self._folded()
        if not x.is_cuda:                     # CPU: plain torch (never on the product's hot path)
            x = x.contiguous(memory_format=torch.channels_last)

            def run(t, lo, hi):
                for w, b, stride, pad, slope in cache[lo:hi]:
                    t = F.leaky_relu_(F.conv2d(t, w, b, stride, pad), slope)
                return t
            c0 = run(x, 0, 2)
            c1 = run(c0, 2, 5)
            c2 = run(c1, 5, 8)
            return self._head(c0, c1, c2)
        packed = self._packed_fp32()

        def planar(t, i):
            w, b, _, _, slope = cache[i]
            return ops.conv2d_planar(t, packed[i], w.shape[1], w.shape[0], b, slope, ops.FP32)

        def strided(t, i):
            _, b, _, _, slope = cache[i]
            return ops.conv2d_5x5s2_fp32(t, packed[i], b, slope)

        w0, b0, _, _, slope0 = cache[0]
        c0 = planar(ops.conv2d_rgb8(x, w0, b0, slope0), 1)
        c1 = planar(planar(strided(c0, 2), 3), 4)
        c2 = planar(planar(strided(c1, 5), 6), 7)
        return self._head(c0, c1, c2)

    def _packed_fp32(self):
        """Packed weights of the fp32 path ([27][Cin][Cout] planar 3x3 blocks, plain contiguous
        (O,I,5,5) copies of the strided ones); no tensor-core operand image is involved."""
        key = self._fold_key
        if getattr(self, "_pack32_key", None) != key:
            cache = self._fold_cache
            packed = {i: ops.pack_conv3d_weight(cache[i][0].contiguous(), ops.CONV_PLANAR)
                      for i in (1, 3, 4, 6, 7)}
            for i in (2, 5):
                packed[i] = cache[i][0].detach().contiguous(memory_format=torch.contiguous_format).clone()
            self._pack32_cache, self._pack32_key = packed, key
        return self._pack32_cache

    def _forward_modules(self, x):
        # channels-last end to end: level_l come out physically (N,h,w,C)
        x = x.contiguous(memory_format=torch.channels_last)
        c0 = self.conv0(x)
        c1 = self.conv1(c0)
        c2 = self.conv2(c1)
        return self._head(c0, c1, c2)

    def _head(self, c0, c1, c2):
        if c0.is_cuda and not (self.training or torch.is_grad_enabled()):
            f2 = ops.fpn_merge(None, c2, self.toplayer.weight, self.toplayer.bias)   # 1x1 lateral
        else:
            f2 = self.toplayer(c2)
        if c0.is_cuda and not (self.training or torch.is_grad_enabled()):
            # fused top-down path: upsample + lateral 1x1 + add + 3x3 smooth in one kernel per
            # level (csrc/fpn.cu); the 32-channel full-resolution tensor is never stored
            f1, l1 = ops.fpn_level(f2, c1, self.lat1.weight, self.lat1.bias,
                                   self.smooth1.weight, self.smooth1.bias, want_feat=True)
            _, l0 = ops.fpn_level(f1, c0, self.lat0.weight, self.lat0.bias,
                                  self.smooth0.weight, self.smooth0.bias, want_feat=False)
            return {"level_0": l0, "level_1": l1,
                    "level_2": f2.contiguous(memory_format=torch.channels_last)}
        f1 = self._up2(f2) + self.lat1(c1)
        f0 = self._up2(f1) + self.lat0(c0)
        f1 = self.smooth1(f1)
        f0 = self.smooth0(f0)
        return {"level_0": f0.contiguous(memory_format=torch.channels_last),
                "level_1": f1.contiguous(memory_format=torch.channels_last),
                "level_2": f2.contiguous(memory_format=torch.channels_last)}


class CostRegNet(nn.Module):
    """3D U-Net cost regularisation (reference models/mvsnet.py:60-104).

    Sub-module names/shapes follow the reference so checkpoints load unchanged;
    ``forward`` hands the whole 11-layer stack to ``casmvs_costreg_fwd``."""

    _ORDER = ("conv0", "conv1", "conv2", "conv3", "conv4", "conv5", "conv6",
              "conv7", "conv9", "conv11", "prob")

    def __init__(self, in_channels, norm_act=InPlaceABN):
        super().__init__()
        self.in_channels = in_channels
        self.conv0 = ConvBnReLU3D(in_channels, 8, norm_act=norm_act)
        self.conv1 = ConvBnReLU3D(8, 16, stride=2, norm_act=norm_act)
        self.conv2 = ConvBnReLU3D(16, 16, norm_act=norm_act)
        self.conv3 = ConvBnReLU3D(16, 32, stride=2, norm_act=norm_act)
        self.conv4 = ConvBnReLU3D(32, 32, norm_act=norm_act)
        self.conv5 = ConvBnReLU3D(32, 64, stride=2, norm_act=norm_act)
        self.conv6 = ConvBnReLU3D(64, 64, norm_act=norm_act)

        def up(cin, cout):
            return nn.Sequential(nn.ConvTranspose3d(cin, cout, 3, padding=1, output_padding=1,
                                                    stride=2, bias=False), norm_act(cout))
        self.conv7 = up(64, 32)
        self.conv9 = up(32, 16)
        self.conv11 = up(16, 8)
        self.prob = nn.Conv3d(8, 1, 3, stride=1, padding=1)
        self.precision = "fp32"
        self._blob = None
        self._blob_key = None

    def _layer_tensors(self, name):
        m = getattr(self, name)
        if name == "prob":
            return m.weight, None, m.bias
        if isinstance(m, ConvBnReLU3D):
            return m.conv.weight, m.bn, None
        return m[0].weight, m[1], None

    def _norm_modules(self):
        for name in self._ORDER[:-1]:
            yield self._layer_tensors(name)[1]

    def packed_params(self):
        """Device blob for casmvs_costreg_fwd (layout: casmvs_costreg_layer_info)."""
        key = tuple((t.data_ptr(), t._version) for t in
                    list(self.parameters()) + list(self.buffers()))
        if key == self._blob_key:
            return self._blob
        dev = self.prob.weight.device
        if self._blob is not None:
            ops.release_weight_images(self._blob)     # the old blob's operand images die with it
        n = ops._lib.load().casmvs_costreg_param_floats(self.in_channels)
        blob = torch.empty(n, device=dev, dtype=torch.float32)
        ops.release_weight_images(blob)     # a recycled address must not hit stale operand images
        for i, name in enumerate(self._ORDER):
            info = ops.costreg_layer_info(self.in_channels, i)
            w, bn, bias = self._layer_tensors(name)
            wp = ops.pack_conv3d_weight(w, info["kind"])
            blob[info["w_off"]:info["w_off"] + wp.numel()] = wp
            co = info["cout"]
            if bn is not None:
                a, b = folded_scale_shift(bn)
            else:
                a = torch.ones(co, device=dev)
                b = bias.detach().float()
            blob[info["scale_off"]:info["scale_off"] + co] = a
            blob[info["shift_off"]:info["shift_off"] + co] = b
        self._blob, self._blob_key = blob, key
        return blob

    def _forward_autograd(self, x):
        """Differentiable path (training, or eval-mode BN with parameters that require grad):
        raw convolutions through autograd.Conv3dFn (own forward / dgrad / wgrad kernels), the
        norm-act as the module itself (batch statistics in training mode, like InPlaceABN)."""
        from .. import autograd as AG
        prec = ops.PRECISIONS[self.precision]

        def cbr(m, t, stride=1):
            return m.bn(AG.conv3d(t, m.conv.weight, ops.CONV, stride, prec))

        def up(m, t):
            return m[1](AG.conv3d(t, m[0].weight, ops.CONV_TRANSPOSE, 2, prec))

        conv0 = cbr(self.conv0, x)
        conv2 = cbr(self.conv2, cbr(self.conv1, conv0, 2))
        conv4 = cbr(self.conv4, cbr(self.conv3, conv2, 2))
        x = cbr(self.conv6, cbr(self.conv5, conv4, 2))
        x = conv4 + up(self.conv7, x)                                  # mvsnet.py:96-102
        x = conv2 + up(self.conv9, x)
        x = conv0 + up(self.conv11, x)
        return AG.conv3d(x, self.prob.weight, ops.CONV, 1, prec) + self.prob.bias.view(1, -1, 1, 1, 1)

    def forward(self, x):
        if torch.is_grad_enabled() and (x.requires_grad or
                                        any(p.requires_grad for p in self.parameters())):
            return self._forward_autograd(x)
        for bn in self._norm_modules():
            if bn.training:
                raise ops._lib.CasMVSError("CostRegNet inference path needs .eval() (training "
                                           "runs through the autograd path: enable grad)")
            if abs(activation_slope(bn) - 0.01) > 1e-12:
                raise ops._lib.CasMVSError("casmvs_costreg_fwd assumes LeakyReLU(0.01) norm_act")
        logits = ops.costreg(x, self.packed_params(), self.in_channels,
                             ops.PRECISIONS[self.precision])
        return logits.unsqueeze(1)                                   # (B,1,D,h,w)


class CascadeMVSNet(nn.Module):
    def __init__(self, n_depths=[8, 32, 48], interval_ratios=[1, 2, 4], num_groups=1,
                 norm_act=InPlaceABN, precision="fp32"):
        super().__init__()
        self.levels = 3
        self.n_depths = n_depths
        self.interval_ratios = interval_ratios
        self.G = num_groups
        self.feature = FeatureNet(norm_act)
        # run the top-down half of the pyramid on a side stream, concurrently with the coarsest
        # cascade stage (tf32 inference path; CASMVS_OVERLAP=0 turns it off)
        import os
        self.overlap_pyramid = os.environ.get("CASMVS_OVERLAP", "1") != "0"
        # diagnostics: also return the int64 depth_index_l maps (mvsnet.py:185-190) that the
        # confidence gather uses; the reference keeps them internal
        self.return_index = False
        self._last_index = None
        # cascade-internal fusion: K4 writes only the first rung of each stage's hypothesis ladder
        # and K1 / K3 generate first + step*d themselves (bit-identical results; the (B,D,h,w)
        # hypothesis tensor is neither written nor read).  CASMVS_LADDER=0 turns it off.
        self.fuse_hypotheses = os.environ.get("CASMVS_LADDER", "1") != "0"
        for l in range(self.levels):
            cin = self.G if self.G > 1 else 8 * 2 ** l
            setattr(self, f"cost_reg_{l}", CostRegNet(cin, norm_act))
        self.set_precision(precision)

    def set_precision(self, precision):
        """'fp32' (CUDA-core FMA, bit-faithful products) or 'tf32' (tcgen05) for the convs."""
        if precision not in ops.PRECISIONS:
            raise ValueError(f"precision must be one of {list(ops.PRECISIONS)}")
        self.precision = precision
        for m in self.modules():
            if isinstance(m, (CostRegNet, ConvBnReLU3D)):
                m.precision = precision
        # in tf32 mode the 2D FeatureNet convs may use cuDNN's TF32 tensor-core kernels too
        self.feature.allow_tf32 = precision == "tf32"
        return self

    def predict_depth(self, feats, proj_mats, depth_values, cost_reg):
        """feats (B,V,C,h,w), proj_mats (B,V-1,3,4), depth_values (B,D,h,w),
        cost_reg: module (B,C,D,h,w)->(B,1,D,h,w).  Returns depth, confidence (B,h,w)
        (reference models/mvsnet.py:125-195)."""
        if torch.is_grad_enabled() and (feats.requires_grad or
                                        any(p.requires_grad for p in cost_reg.parameters())):
            from .. import autograd as AG
            cost = AG.warp_cost(feats, proj_mats, depth_values, self.G)
            logits = cost_reg(cost).squeeze(1)
            return AG.regress(logits, depth_values)
        cost = ops.warp_cost(feats, proj_mats, depth_values, self.G, ops.NHWC,
                             round_tf32=(getattr(cost_reg, "precision", "fp32") == "tf32"))
        logits = cost_reg(cost).squeeze(1)
        del cost
        depth, confidence, index, _ = ops.regress(logits, depth_values,
                                                  want_index=self.return_index)
        self._last_index = index
        return depth, confidence

    def _forward_autograd(self, imgs, proj_mats, init_depth_min, depth_interval):
        """The differentiable forward of the reference (mvsnet.py:197-244) for train.py:99-127:
        FeatureNet through its torch modules (host glue), every cascade stage through the
        autograd wrappers of K1 / K2 / K3; hypotheses are detached like mvsnet.py:231."""
        B, V, _, H, W = imgs.shape
        # The 2D FeatureNet trains through torch / cuDNN.  cuDNN's fp32 convolutions default to
        # TF32 on this GPU, and the BACKWARD convolutions run later, outside any context manager
        # around this forward: the flag has to be set process-wide.  The reference is fp32
        # (opt.py:69-70), so fp32 precision means fp32 here too.
        torch.backends.cudnn.allow_tf32 = self.precision == "tf32"
        feats = self.feature(imgs.reshape(B * V, 3, H, W))
        proj_by_level = proj_mats.permute(2, 0, 1, 3, 4).contiguous()
        results = {}
        depth_l = None
        for l in reversed(range(self.levels)):
            feats_l = feats[f"level_{l}"]
            feats_l = feats_l.view(B, V, *feats_l.shape[1:])
            depth_interval_l = depth_interval * self.interval_ratios[l]
            D = self.n_depths[l]
            h, w = feats_l.shape[-2:]
            with torch.no_grad():
                if l == self.levels - 1:
                    depth_values = ops.uniform_hypotheses(init_depth_min, depth_interval_l, D, B,
                                                          h, w, imgs.device)
                else:
                    depth_values = ops.depth_hypotheses(depth_l.detach(), D, depth_interval_l,
                                                        upsample=True)
            depth_l, confidence_l = self.predict_depth(feats_l, proj_by_level[l], depth_values,
                                                       getattr(self, f"cost_reg_{l}"))
            results[f"depth_{l}"] = depth_l
            results[f"confidence_{l}"] = confidence_l
        return results

    def packed_buffers(self):
        """The packed-weight tensors whose tensor-core operand images a captured CUDA graph of this
        model embeds (CostRegNet blobs, FeatureNet packs): GraphedCascade watches them."""
        bufs = []
        for l in range(self.levels):
            b = getattr(self, f"cost_reg_{l}")._blob
            if b is not None:
                bufs.append(b)
        f = self.feature
        bufs += list(getattr(f, "_pack_cache", {}).values()) + list(getattr(f, "_smooth_pack", ()))
        return [b for b in bufs if torch.is_tensor(b) and b.is_cuda]

    def run_stage(self, l, feats_l, proj_mats_l, depth_prev, init_depth_min, depth_interval):
        """One cascade stage of the inference path (no grad): hypotheses -> K1 -> K2 -> K3.
        feats_l (B,V,C,h,w) channels-last, proj_mats_l (B,V-1,3,4), depth_prev (B,h/2,w/2) or None
        for the coarsest stage.  Returns depth, confidence (B,h,w)."""
        B, V, C, h, w = feats_l.shape
        D = self.n_depths[l]
        depth_interval_l = depth_interval * self.interval_ratios[l]
        cost_reg = getattr(self, f"cost_reg_{l}")
        if self.fuse_hypotheses and ops.ladder_supported(V, C, self.G) and \
                ops.is_channels_last_feats(feats_l):
            first = init_depth_min if depth_prev is None else ops.depth_first(depth_prev, D, depth_interval_l)
            lad = ops.Ladder(first, depth_interval_l, D, B, h, w, feats_l.device)
            cost = ops.warp_cost_ladder(feats_l, proj_mats_l, lad, self.G,
                                        round_tf32=(cost_reg.precision == "tf32"))
            logits = cost_reg(cost).squeeze(1)
            del cost
            depth, confidence, self._last_index = ops.regress_ladder(logits, lad,
                                                                     want_index=self.return_index)
            return depth, confidence
        if depth_prev is None:
            depth_values = ops.uniform_hypotheses(init_depth_min, depth_interval_l, D, B, h, w,
                                                  feats_l.device)
        else:
            depth_values = ops.depth_hypotheses(depth_prev, D, depth_interval_l, upsample=True)
        return self.predict_depth(feats_l, proj_mats_l, depth_values, cost_reg)

    def forward(self, imgs, proj_mats, init_depth_min, depth_interval):
        """imgs (B,V,3,H,W); proj_mats (B,V-1,levels,3,4) fine->coarse;
        init_depth_min, depth_interval: float or (B,1) tensors.
        Returns {depth_l, confidence_l : (B,h_l,w_l)} (reference mvsnet.py:197-244)."""
        B, V, _, H, W = imgs.shape
        if not imgs.is_cuda:
            raise ops._lib.CasMVSError(
                "CascadeMVSNet (B200 engine) needs CUDA inputs; there is no CPU fallback")
        differentiable = torch.is_grad_enabled() and (
            imgs.requires_grad or any(p.requires_grad for p in self.parameters()))
        # (B,1) depth parameters may arrive as CPU tensors from the reference's data loader
        # (datasets/dtu.py:188-189): move them once, not once per stage
        if torch.is_tensor(init_depth_min):
            init_depth_min = init_depth_min.to(imgs.device, torch.float32)
        if torch.is_tensor(depth_interval):
            depth_interval = depth_interval.to(imgs.device, torch.float32)
        if differentiable:
            return self._forward_autograd(imgs, proj_mats, init_depth_min, depth_interval)
        results = {}
        with torch.no_grad():
            feats = self.feature(imgs.reshape(B * V, 3, H, W), overlap=self.overlap_pyramid)
            ready = feats.get("_ready", {})
            # one re-layout for all levels instead of a strided slice copy per stage
            proj_by_level = proj_mats.permute(2, 0, 1, 3, 4).contiguous()
            depth_l = None
            for l in reversed(range(self.levels)):
                if l in ready:                      # level produced on the side stream
                    torch.cuda.current_stream(imgs.device).wait_event(ready[l])
                feats_l = feats[f"level_{l}"]
                feats_l = feats_l.view(B, V, *feats_l.shape[1:])
                proj_mats_l = proj_by_level[l]
                depth_l, confidence_l = self.run_stage(l, feats_l, proj_mats_l, depth_l,
                                                       init_depth_min, depth_interval)
                results[f"depth_{l}"] = depth_l
                results[f"confidence_{l}"] = confidence_l
                if self.return_index:
                    results[f"depth_index_{l}"] = self._last_index
        return results

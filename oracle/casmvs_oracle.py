"""TEST INFRASTRUCTURE — CPU oracle for the cascade-MVS hot path.  NOT product code.

A plain-PyTorch (CPU, fp32) restatement of the reference algorithm for the path
SURVEY.md §8(a) lists, written as state-dict-driven *functions* (the reference
is nn.Module code).  Each function cites the reference file:line it follows
(paths relative to /root/reference).  It uses the same torch primitives in the
same order as the reference, so on CPU it is bit-identical to the reference
run in this container; that is pinned by ``tests/golden/*.npz`` (generated from
the REAL reference by ``oracle/make_golden.py``), which ``tests/test_oracle_golden.py``
and ``tests/test_oracle_vs_reference.py`` compare against.

Parity status: the reference ships no tests / golden vectors of its own
("parity unpinned" by the reference, SURVEY.md §8c); the pins above are outputs
of the reference itself run in the build container.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu-baseline /
``--impl reference`` legs may import this module.  The product package
``casmvsnet_pl_b200`` never does (tests/test_no_oracle_in_product.py checks).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

LEAKY_SLOPE = 0.01   # inplace_abn default activation_param (README.md:28, unpinned pkg)
BN_EPS = 1e-5        # inplace_abn / nn.BatchNorm default


# --------------------------------------------------------------------------- #
# a1  homography plane-sweep warp                       models/modules.py:52-92
# --------------------------------------------------------------------------- #
def plane_sweep_warp(src_feat, proj_mat, depth_values):
    """src_feat (B,C,h,w), proj_mat (B,3,4), depth_values (B,D,h,w) -> (B,C,D,h,w).

    q = R·(x,y,1)^T + T/depth (modules.py:63-72); q_z <= 1e-7 -> (w,h,1)
    (:76-79); perspective divide (:81); normalise to [-1,1] (:83-84);
    bilinear / zeros / align_corners=True grid_sample (:87-89).
    """
    B, C, h, w = src_feat.shape
    D = depth_values.shape[1]
    rot = proj_mat[:, :, :3]
    trans = proj_mat[:, :, 3:]
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32),
                            torch.arange(w, dtype=torch.float32), indexing="ij")
    pix = torch.stack([xs.reshape(-1), ys.reshape(-1),
                       torch.ones(h * w)], 0)                       # (3, h*w)
    pix = pix.unsqueeze(0).expand(B, -1, -1).repeat(1, 1, D)         # (B,3,D*h*w)
    q = rot @ pix + trans / depth_values.reshape(B, 1, D * h * w)
    behind = q[:, 2:] <= 1e-7
    q[:, 0:1][behind] = w
    q[:, 1:2][behind] = h
    q[:, 2:3][behind] = 1
    uv = q[:, :2] / q[:, 2:]
    uv[:, 0] = uv[:, 0] / ((w - 1) / 2) - 1
    uv[:, 1] = uv[:, 1] / ((h - 1) / 2) - 1
    grid = uv.reshape(B, 2, D, h * w).permute(0, 2, 3, 1)            # (B,D,h*w,2)
    out = F.grid_sample(src_feat, grid, mode="bilinear",
                        padding_mode="zeros", align_corners=True)    # (B,C,D,h*w)
    return out.reshape(B, C, D, h, w)


def plane_sweep_warp_direct(src_feat, proj_mat, depth_values):
    """Same as :func:`plane_sweep_warp` but with the bilinear blend written out
    (what the CUDA kernel computes: sample at (u,v) directly, skipping the
    normalise / un-normalise round trip of modules.py:83-84 + grid_sample).
    Differs from the grid_sample form by a few ulp (SURVEY §8a a1: 1.5e-6).
    Small sizes only (pure indexing)."""
    B, C, h, w = src_feat.shape
    D = depth_values.shape[1]
    ys, xs = torch.meshgrid(torch.arange(h, dtype=torch.float32),
                            torch.arange(w, dtype=torch.float32), indexing="ij")
    out = torch.zeros(B, C, D, h, w)
    for b in range(B):
        P = proj_mat[b]
        inv_d = 1.0 / depth_values[b]                                 # (D,h,w)
        qx = P[0, 0] * xs + P[0, 1] * ys + P[0, 2] + P[0, 3] * inv_d
        qy = P[1, 0] * xs + P[1, 1] * ys + P[1, 2] + P[1, 3] * inv_d
        qz = P[2, 0] * xs + P[2, 1] * ys + P[2, 2] + P[2, 3] * inv_d
        behind = qz <= 1e-7
        u = torch.where(behind, torch.full_like(qx, float(w)), qx / qz)
        v = torch.where(behind, torch.full_like(qy, float(h)), qy / qz)
        x0 = torch.floor(u)
        y0 = torch.floor(v)
        fx = u - x0
        fy = v - y0
        acc = torch.zeros(C, D, h, w)
        for dy, dx, wgt in ((0, 0, (1 - fx) * (1 - fy)), (0, 1, fx * (1 - fy)),
                            (1, 0, (1 - fx) * fy), (1, 1, fx * fy)):
            xi = x0 + dx
            yi = y0 + dy
            ok = (xi >= 0) & (xi <= w - 1) & (yi >= 0) & (yi <= h - 1)
            xi_c = xi.clamp(0, w - 1).long()
            yi_c = yi.clamp(0, h - 1).long()
            tap = src_feat[b][:, yi_c, xi_c]                          # (C,D,h,w)
            acc = acc + tap * (wgt * ok)
        out[b] = acc
    return out


# --------------------------------------------------------------------------- #
# a2 / a3  cost volume                     models/mvsnet.py:133-172
# --------------------------------------------------------------------------- #
def variance_cost_volume(feats, proj_mats, depth_values):
    """feats (B,V,C,h,w), proj_mats (B,V-1,3,4), depth_values (B,D,h,w) -> (B,C,D,h,w).
    S = ref + Σ warp, Q = ref² + Σ warp² (mvsnet.py:139-141,152-153);
    var = Q/V − (S/V)² (:166-168)."""
    B, V, C, h, w = feats.shape
    D = depth_values.shape[1]
    ref = feats[:, 0].unsqueeze(2).expand(-1, -1, D, -1, -1)
    vol_sum = ref
    vol_sq = ref ** 2
    for v in range(1, V):
        warped = plane_sweep_warp(feats[:, v], proj_mats[:, v - 1], depth_values)
        vol_sum = vol_sum + warped
        vol_sq = vol_sq + warped ** 2
    return vol_sq.div_(V).sub_(vol_sum.div(V).pow_(2))


def groupwise_cost_volume(feats, proj_mats, depth_values, num_groups):
    """-> (B,G,D,h,w): mean over the C/G channels of a group of (Σ_src warp)·ref,
    divided by V−1 (mvsnet.py:143-144,158-162,170-172)."""
    B, V, C, h, w = feats.shape
    D = depth_values.shape[1]
    G = num_groups
    ref = feats[:, 0].unsqueeze(2).expand(-1, -1, D, -1, -1).reshape(B, G, C // G, D, h, w)
    vol_sum = 0
    for v in range(1, V):
        warped = plane_sweep_warp(feats[:, v], proj_mats[:, v - 1], depth_values)
        vol_sum = vol_sum + warped.reshape(B, G, C // G, D, h, w)
    return (vol_sum * ref).mean(2).div_(V - 1)


# --------------------------------------------------------------------------- #
# a4 / a5  3D U-Net cost regularisation      models/modules.py:21-31, mvsnet.py:60-104
# --------------------------------------------------------------------------- #
def _abn(x, sd, prefix):
    """eval-mode ABN: batch norm with running stats + LeakyReLU(0.01)."""
    x = F.batch_norm(x, sd[prefix + "running_mean"], sd[prefix + "running_var"],
                     sd[prefix + "weight"], sd[prefix + "bias"], False, 0.1, BN_EPS)
    return F.leaky_relu(x, LEAKY_SLOPE)


def _conv3d_block(x, sd, prefix, stride=1):
    """ConvBnReLU3D (modules.py:21-31): Conv3d(k3,p1,no bias) -> norm_act."""
    return _abn(F.conv3d(x, sd[prefix + "conv.weight"], None, stride, 1), sd, prefix + "bn.")


def _deconv3d_block(x, sd, prefix):
    """Sequential(ConvTranspose3d(k3,s2,p1,op1,no bias), norm_act) (mvsnet.py:74-87)."""
    y = F.conv_transpose3d(x, sd[prefix + "0.weight"], None, stride=2, padding=1,
                           output_padding=1)
    return _abn(y, sd, prefix + "1.")


def cost_regularize(volume, sd, prefix):
    """CostRegNet.forward (mvsnet.py:91-104). volume (B,Cin,D,h,w) -> (B,1,D,h,w)."""
    c0 = _conv3d_block(volume, sd, prefix + "conv0.")
    c2 = _conv3d_block(_conv3d_block(c0, sd, prefix + "conv1.", 2), sd, prefix + "conv2.")
    c4 = _conv3d_block(_conv3d_block(c2, sd, prefix + "conv3.", 2), sd, prefix + "conv4.")
    x = _conv3d_block(_conv3d_block(c4, sd, prefix + "conv5.", 2), sd, prefix + "conv6.")
    x = c4 + _deconv3d_block(x, sd, prefix + "conv7.")
    x = c2 + _deconv3d_block(x, sd, prefix + "conv9.")
    x = c0 + _deconv3d_block(x, sd, prefix + "conv11.")
    return F.conv3d(x, sd[prefix + "prob.weight"], sd[prefix + "prob.bias"], 1, 1)


# --------------------------------------------------------------------------- #
# a6 / a7  softmax, depth regression, confidence   mvsnet.py:174-193, modules.py:95-104
# --------------------------------------------------------------------------- #
def regress_depth(logits, depth_values):
    """logits (B,D,h,w), depth_values (B,D,h,w) or (D,) ->
    depth (B,h,w), confidence (B,h,w), depth_index (B,h,w) int64, prob (B,D,h,w)."""
    D = logits.shape[1]
    prob = F.softmax(logits, 1)
    dv = depth_values.reshape(1, -1, 1, 1) if depth_values.dim() == 1 else depth_values
    depth = (prob * dv).sum(1).to(dv.dtype)
    # Σ of 4 neighbouring probabilities, window [d-1, d+2], zero padded (mvsnet.py:181-183)
    sum4 = 4 * F.avg_pool3d(F.pad(prob.unsqueeze(1), pad=(0, 0, 0, 0, 1, 2)),
                            (4, 1, 1), stride=1).squeeze(1)
    steps = torch.arange(D, dtype=prob.dtype).reshape(1, D, 1, 1)
    index = (prob * steps).sum(1).long().clamp(0, D - 1)             # trunc, not round (:189)
    conf = torch.gather(sum4, 1, index.unsqueeze(1)).squeeze(1)
    return depth, conf, index, prob


# --------------------------------------------------------------------------- #
# a8 / a9 / a10  depth hypotheses            modules.py:34-49, mvsnet.py:213-235
# --------------------------------------------------------------------------- #
def depth_hypotheses(current_depth, n_depths, depth_interval):
    """current_depth (B,1,h,w); depth_interval float or (B,1) -> (B,D,h,w)."""
    if not isinstance(depth_interval, float):
        depth_interval = depth_interval.reshape(-1, 1, 1, 1)
    first = torch.clamp_min(current_depth - n_depths / 2 * depth_interval, 1e-7)
    steps = torch.arange(0, n_depths, dtype=current_depth.dtype).reshape(1, -1, 1, 1)
    return first + depth_interval * steps


def initial_hypotheses(init_depth_min, depth_interval_l, n_depths, B, h, w):
    """Coarsest-level uniform planes (mvsnet.py:213-229)."""
    steps = torch.arange(0, n_depths, dtype=torch.float32)
    if isinstance(init_depth_min, float):
        vals = (init_depth_min + depth_interval_l * steps).reshape(1, -1, 1, 1)
        return vals.expand(B, -1, h, w)
    vals = init_depth_min + depth_interval_l * steps.reshape(1, -1)   # (B,D)
    return vals.reshape(B, -1, 1, 1).expand(-1, -1, h, w)


def upsample_depth(depth):
    """(B,h,w) -> (B,1,2h,2w) bilinear, align_corners=True (mvsnet.py:231-234)."""
    return F.interpolate(depth.unsqueeze(1), scale_factor=2, mode="bilinear",
                         align_corners=True)


# --------------------------------------------------------------------------- #
# FeatureNet (adjacent to the path; host side stays PyTorch)   mvsnet.py:7-57
# --------------------------------------------------------------------------- #
def _conv2d_block(x, sd, prefix, stride, pad):
    return _abn(F.conv2d(x, sd[prefix + "conv.weight"], None, stride, pad), sd, prefix + "bn.")


def feature_pyramid(imgs, sd, prefix="feature."):
    """imgs (N,3,H,W) -> dict level_0 (N,8,H,W), level_1 (N,16,H/2,W/2), level_2 (N,32,H/4,W/4)."""
    p = prefix
    c0 = _conv2d_block(_conv2d_block(imgs, sd, p + "conv0.0.", 1, 1), sd, p + "conv0.1.", 1, 1)
    c1 = _conv2d_block(c0, sd, p + "conv1.0.", 2, 2)
    c1 = _conv2d_block(_conv2d_block(c1, sd, p + "conv1.1.", 1, 1), sd, p + "conv1.2.", 1, 1)
    c2 = _conv2d_block(c1, sd, p + "conv2.0.", 2, 2)
    c2 = _conv2d_block(_conv2d_block(c2, sd, p + "conv2.1.", 1, 1), sd, p + "conv2.2.", 1, 1)
    f2 = F.conv2d(c2, sd[p + "toplayer.weight"], sd[p + "toplayer.bias"])
    up = lambda t: F.interpolate(t, scale_factor=2, mode="bilinear", align_corners=True)
    f1 = up(f2) + F.conv2d(c1, sd[p + "lat1.weight"], sd[p + "lat1.bias"])
    f0 = up(f1) + F.conv2d(c0, sd[p + "lat0.weight"], sd[p + "lat0.bias"])
    f1 = F.conv2d(f1, sd[p + "smooth1.weight"], sd[p + "smooth1.bias"], padding=1)
    f0 = F.conv2d(f0, sd[p + "smooth0.weight"], sd[p + "smooth0.bias"], padding=1)
    return {"level_0": f0, "level_1": f1, "level_2": f2}


# --------------------------------------------------------------------------- #
# a12 / a11  predict_depth and the cascade      mvsnet.py:125-195, 197-244
# --------------------------------------------------------------------------- #
def predict_depth(feats, proj_mats, depth_values, sd, prefix, num_groups=1,
                  return_intermediates=False):
    if num_groups == 1:
        cost = variance_cost_volume(feats, proj_mats, depth_values)
    else:
        cost = groupwise_cost_volume(feats, proj_mats, depth_values, num_groups)
    logits = cost_regularize(cost, sd, prefix).squeeze(1)
    depth, conf, index, prob = regress_depth(logits, depth_values)
    if return_intermediates:
        return depth, conf, dict(cost=cost, logits=logits, index=index, prob=prob)
    return depth, conf


def cascade_forward(sd, imgs, proj_mats, init_depth_min, depth_interval,
                    n_depths=(8, 32, 48), interval_ratios=(1, 2, 4), num_groups=1,
                    feats=None, want_index=False):
    """CascadeMVSNet.forward (mvsnet.py:197-244).  ``feats`` may be given as a
    dict level_l -> (B*V,C,h,w) to skip the FeatureNet (hot-path-only timing).
    want_index adds the int64 ``depth_index_l`` maps of mvsnet.py:185-190 (what the
    confidence gather uses) for the index-parity tests."""
    B, V = imgs.shape[:2] if imgs is not None else (None, None)
    results = {}
    with torch.no_grad():
        if feats is None:
            H, W = imgs.shape[-2:]
            feats = feature_pyramid(imgs.reshape(B * V, 3, H, W), sd)
        else:
            B = proj_mats.shape[0]
            V = proj_mats.shape[1] + 1
        depth_l = None
        for l in (2, 1, 0):
            f = feats[f"level_{l}"]
            f = f.reshape(B, V, *f.shape[1:])
            pm = proj_mats[:, :, l]
            interval_l = depth_interval * interval_ratios[l]
            D = n_depths[l]
            h, w = f.shape[-2:]
            if l == 2:
                dv = initial_hypotheses(init_depth_min, interval_l, D, B, h, w)
            else:
                dv = depth_hypotheses(upsample_depth(depth_l), D, interval_l)
            depth_l, conf_l, inter = predict_depth(f, pm, dv, sd, f"cost_reg_{l}.", num_groups, True)
            if want_index:
                results[f"depth_index_{l}"] = inter["index"]
            del inter
            results[f"depth_{l}"] = depth_l
            results[f"confidence_{l}"] = conf_l
    return results

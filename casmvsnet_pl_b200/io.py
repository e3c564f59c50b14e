"""Input pipeline and on-disk formats either side of the hot path (SURVEY.md §8 f-4).

Host-side Python like the reference's (it is data plumbing, not arithmetic on the path):

  read_pfm / save_pfm          reference datasets/utils.py:5-69 (PFM, bottom-up rows, scale sign
                               = endianness) -- byte-compatible both ways
  read_cam_file                reference datasets/dtu.py:77-90 (MVSNet cam.txt)
  read_pair_file               reference datasets/dtu.py:41-50 (pair.txt)
  pyramid_proj_mats            reference datasets/dtu.py:52-75 (K[R|t] per level, fine -> coarse,
                               intrinsics doubled per finer level, optional test-mode rescale)
  relative_proj_mats           reference datasets/dtu.py:181-186 (src_proj @ inv(ref_proj), rows 0..2)
  pil_bilinear_coeffs /        PIL.Image.resize(img_wh, Image.BILINEAR) of the data sets' network
  resize_images                input (datasets/dtu.py:159-162, tanks.py, blendedmvs.py:162-163),
                               bit-exact: PIL's fixed-point taps built here in float64, the
                               integer passes on the GPU by casmvs_resize_u8_fwd
  normalize_images             reference datasets/dtu.py:130-137 (ToTensor + ImageNet Normalize):
                               uint8 HWC images are uploaded AS BYTES (4x less H2D traffic than
                               fp32) and converted + normalised + re-laid-out to planar fp32 on the
                               GPU by casmvs_normalize_u8_fwd
  DepthWriter / infer_views    reference eval.py:213-229 (the per-view inference loop): views are
                               streamed through PipelinedCascade (H2D, forward and D2H of
                               neighbouring views overlap), NaNs scrubbed, depth_XXXX.pfm and
                               proba_XXXX.pfm written in the reference's layout
"""
from __future__ import annotations

import functools
import math
import os
import re
import sys

import numpy as np
import torch

IMAGENET_MEAN = (0.485, 0.456, 0.406)      # datasets/dtu.py:133-134
IMAGENET_STD = (0.229, 0.224, 0.225)


# ------------------------------------------------------------------------------ PFM
def read_pfm(filename):
    """-> (data float32 (H,W) or (H,W,3), scale).  datasets/utils.py:5-39."""
    with open(filename, "rb") as f:
        header = f.readline().decode("utf-8").rstrip()
        if header == "PF":
            color = True
        elif header == "Pf":
            color = False
        else:
            raise ValueError("Not a PFM file.")
        m = re.match(r"^(\d+)\s(\d+)\s$", f.readline().decode("utf-8"))
        if not m:
            raise ValueError("Malformed PFM header.")
        width, height = map(int, m.groups())
        scale = float(f.readline().rstrip())
        endian = "<" if scale < 0 else ">"        # negative scale = little-endian
        scale = abs(scale)
        data = np.frombuffer(f.read(), dtype=endian + "f4")
    shape = (height, width, 3) if color else (height, width)
    if data.size != int(np.prod(shape)):
        raise ValueError(f"PFM payload has {data.size} floats, header says {shape}")
    return np.flipud(data.reshape(shape)), scale


def save_pfm(filename, image, scale=1):
    """datasets/utils.py:42-69: float32 only, rows bottom-up, scale sign = byte order."""
    image = np.asarray(image)
    if image.dtype.name != "float32":
        raise TypeError("Image dtype must be float32.")
    if image.ndim == 3 and image.shape[2] == 3:
        color = True
    elif image.ndim == 2 or (image.ndim == 3 and image.shape[2] == 1):
        color = False
    else:
        raise ValueError("Image must have H x W x 3, H x W x 1 or H x W dimensions.")
    endian = image.dtype.byteorder
    if endian == "<" or (endian == "=" and sys.byteorder == "little"):
        scale = -scale
    with open(filename, "wb") as f:
        f.write(b"PF\n" if color else b"Pf\n")
        f.write(f"{image.shape[1]} {image.shape[0]}\n".encode("utf-8"))
        f.write(("%f\n" % scale).encode("utf-8"))
        np.ascontiguousarray(np.flipud(image)).tofile(f)


# ------------------------------------------------------------------------------ cameras
def read_cam_file(filename):
    """MVSNet cam.txt -> (intrinsics (3,3) f32, extrinsics (4,4) f32, depth_min float).
    datasets/dtu.py:77-90: extrinsics on lines [1,5), intrinsics on lines [7,10), depth_min first
    token of line 11."""
    with open(filename) as f:
        lines = [line.rstrip() for line in f.readlines()]
    extrinsics = np.array(" ".join(lines[1:5]).split(), dtype=np.float32).reshape(4, 4)
    intrinsics = np.array(" ".join(lines[7:10]).split(), dtype=np.float32).reshape(3, 3)
    depth_min = float(lines[11].split()[0])
    return intrinsics, extrinsics, depth_min


def read_pair_file(filename):
    """pair.txt -> [(ref_view, [src views by score])].  datasets/dtu.py:41-50 (ids are every
    second token of the score line)."""
    out = []
    with open(filename) as f:
        n = int(f.readline())
        for _ in range(n):
            ref = int(f.readline().rstrip())
            src = [int(x) for x in f.readline().rstrip().split()[1::2]]
            out.append((ref, src))
    return out


def pyramid_proj_mats(intrinsics, extrinsics, levels=3, img_wh=None, full_wh=(1600, 1200)):
    """(levels,4,4) float32 world->pixel matrices, level 0 = finest.  datasets/dtu.py:52-75:
    `intrinsics` are those of the COARSEST level (cam files hold quarter-resolution values);
    in test mode (img_wh given) they are first rescaled by img_wh / full_wh / 4.  Arithmetic in
    float32 numpy like the reference (np.eye is float64, the product is float32 @ float32 placed
    into it, then cast by torch.FloatTensor)."""
    K = np.array(intrinsics, dtype=np.float32, copy=True)
    E = np.asarray(extrinsics, dtype=np.float32)
    if img_wh is not None:
        K[0] *= img_wh[0] / full_wh[0] / 4
        K[1] *= img_wh[1] / full_wh[1] / 4
    mats = []
    for _ in range(levels):
        P = np.eye(4)
        P[:3, :4] = K @ E[:3, :4]
        K[:2] *= 2                                   # 1/4 -> 1/2 -> 1
        mats.append(torch.FloatTensor(P))
    return torch.stack(mats[::-1])


def relative_proj_mats(proj_mats_by_view, view_ids):
    """view_ids = [ref, src...] -> (V-1, levels, 3, 4): src_proj @ inv(ref_proj), rows 0..2,
    what CascadeMVSNet.forward takes (datasets/dtu.py:176-186)."""
    ref_inv = torch.inverse(proj_mats_by_view[view_ids[0]])
    return torch.stack([proj_mats_by_view[v] @ ref_inv for v in view_ids[1:]])[:, :, :3]


# ------------------------------------------------------------------------------ images
def normalize_images(images_u8, device=None, out=None):
    """uint8 (N,H,W,3) RGB images -> float32 (N,3,H,W), (x/255 - mean)/std per channel
    (ToTensor + Normalize, datasets/dtu.py:130-137) on the GPU.  `images_u8` may be a pinned
    host tensor (uploaded as bytes: 4x less H2D traffic than normalised floats) or already on
    the device.  Matches the torchvision arithmetic: x.float().div(255).sub(mean).div(std)."""
    import ctypes

    from . import _lib
    t = images_u8 if torch.is_tensor(images_u8) else torch.from_numpy(np.ascontiguousarray(images_u8))
    if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[-1] != 3:
        raise _lib.CasMVSError("normalize_images expects uint8 (N,H,W,3)")
    if not t.is_cuda:
        if device is None:
            raise _lib.CasMVSError("normalize_images: give a CUDA device for host input (no CPU path)")
        t = t.to(device, non_blocking=True)
    t = t.contiguous()
    N, H, W, _ = t.shape
    if out is None:
        out = torch.empty(N, 3, H, W, device=t.device, dtype=torch.float32)
    mean = (ctypes.c_float * 3)(*IMAGENET_MEAN)
    std = (ctypes.c_float * 3)(*IMAGENET_STD)
    with torch.cuda.device(t.device):
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.load().casmvs_normalize_u8_fwd(
            ctypes.c_void_p(t.data_ptr()), ctypes.c_void_p(out.data_ptr()), N, H, W, mean, std, st),
            "normalize_u8")
    return out


@functools.lru_cache(maxsize=64)
def pil_bilinear_coeffs(in_size, out_size):
    """PIL's fixed-point BILINEAR resampling coefficients for one axis in_size -> out_size
    (Pillow's precompute_coeffs + normalize_coeffs_8bpc, in float64 like its C code) ->
    (xmin (out_size,) int32, taps (out_size, k) int32).  Output index o reads input
    xmin[o] + j with weight taps[o, j] / 2**22; unused trailing taps are 0.  The arrays are
    shared by later calls with the same sizes: do not modify them."""
    in_size, out_size = int(in_size), int(out_size)
    if in_size <= 0 or out_size <= 0:
        raise ValueError(f"pil_bilinear_coeffs: sizes must be positive ({in_size} -> {out_size})")
    scale = in_size / out_size
    fs = max(scale, 1.0)
    support = fs                               # bilinear support 1.0, widened when downscaling
    ss = 1.0 / fs
    xmin = np.zeros(out_size, np.int32)
    taps = np.zeros((out_size, int(math.ceil(support)) * 2 + 1), np.int32)   # PIL's ksize
    k = 1
    for o in range(out_size):
        center = (o + 0.5) * scale
        lo = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), in_size) - lo
        w = [max(0.0, 1.0 - abs((j + lo - center + 0.5) * ss)) for j in range(n)]
        total = 0.0
        for v in w:                            # sequential sum, as the C loop adds them
            total += v
        xmin[o] = lo
        for j, v in enumerate(w):
            taps[o, j] = int(0.5 + (v / total if total != 0.0 else v) * (1 << 22))
        k = max(k, n)
    return xmin, np.ascontiguousarray(taps[:, :k])     # the table stride is the widest run


def resize_images(images_u8, img_wh, device=None):
    """PIL.Image.resize(img_wh, Image.BILINEAR) of every image of a uint8 (N,H,W,3) RGB batch
    (the network input of datasets/dtu.py:159-162, tanks.py, blendedmvs.py:162-163), bit-exact,
    on the GPU by casmvs_resize_u8_fwd -> uint8 (N,h,w,3) CUDA tensor, (w, h) = img_wh.
    `images_u8` may be a host tensor / ndarray (uploaded as bytes to `device`) or on the device.
    Images that already have the size are returned as they are (on the device)."""
    import ctypes

    from . import _lib
    t = images_u8 if torch.is_tensor(images_u8) else torch.from_numpy(np.ascontiguousarray(images_u8))
    if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[-1] != 3:
        raise _lib.CasMVSError("resize_images expects uint8 (N,H,W,3)")
    if not t.is_cuda:
        if device is None:
            raise _lib.CasMVSError("resize_images: give a CUDA device for host input (no CPU path)")
        t = t.to(device, non_blocking=True)
    t = t.contiguous()
    N, H, W, _ = t.shape
    w, h = int(img_wh[0]), int(img_wh[1])
    if (w, h) == (W, H):
        return t
    out = torch.empty(N, h, w, 3, device=t.device, dtype=torch.uint8)

    def tables(n_in, n_out):
        if n_in == n_out:
            return None, None, 0
        xmin, taps = pil_bilinear_coeffs(n_in, n_out)
        return (torch.from_numpy(xmin).to(t.device), torch.from_numpy(taps).to(t.device), taps.shape[1])
    xmin_x, taps_x, kx = tables(W, w)
    xmin_y, taps_y, ky = tables(H, h)

    def p(x):
        return ctypes.c_void_p(x.data_ptr()) if x is not None else None
    with torch.cuda.device(t.device):
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.load().casmvs_resize_u8_fwd(
            p(t), N, H, W, p(out), h, w, p(xmin_x), p(taps_x), kx, p(xmin_y), p(taps_y), ky, st),
            "resize_u8")
    return out


# ------------------------------------------------------------------------------ eval loop
def scrub(x):
    """np.nan_to_num of eval.py:225-227 (NaN -> 0; +-inf -> largest finite)."""
    return np.nan_to_num(x)


class DepthWriter:
    """results/<dataset>/depth/<scan>/depth_XXXX.pfm + proba_XXXX.pfm (eval.py:228-229)."""

    def __init__(self, depth_dir):
        self.depth_dir = depth_dir

    def __call__(self, scan, vid, depth, proba):
        d = os.path.join(self.depth_dir, scan)
        os.makedirs(d, exist_ok=True)
        save_pfm(os.path.join(d, f"depth_{vid:04d}.pfm"), scrub(np.asarray(depth, dtype=np.float32)))
        save_pfm(os.path.join(d, f"proba_{vid:04d}.pfm"), scrub(np.asarray(proba, dtype=np.float32)))


def infer_views(model, views, init_depth_min, depth_interval, sink, device="cuda:0"):
    """The inference loop of eval.py:213-229 for views of one shape, streamed: `views` yields
    (key, imgs (V,3,H,W) float32 host tensor, proj_mats (V-1,levels,3,4) host tensor); for each,
    `sink(key, depth_0 (H,W) ndarray, confidence_2 (H/4,W/4) ndarray)` is called in order.
    H2D copy, forward (CUDA graph) and D2H of neighbouring views overlap (PipelinedCascade).
    init_depth_min / depth_interval: floats shared by the stream (DTU: 425.0 / 2.65)."""
    from .graph import PipelinedCascade
    pipe = None
    keys = []
    n = 0
    for key, imgs, pm in views:
        imgs_h = imgs.unsqueeze(0).contiguous().pin_memory()
        pm_h = pm.unsqueeze(0).contiguous().pin_memory()
        if pipe is None:
            with torch.cuda.device(device):
                pipe = PipelinedCascade(model, imgs_h.to(device), pm_h.to(device),
                                        init_depth_min, depth_interval)
        keys.append(key)
        done = pipe.submit(imgs_h, pm_h)
        if done is not None:
            sink(keys.pop(0), done[0][0].numpy().copy(), done[1][0].numpy().copy())
        n += 1
    if pipe is not None:
        for d, c in pipe.drain():
            sink(keys.pop(0), d[0].numpy().copy(), c[0].numpy().copy())
    return n

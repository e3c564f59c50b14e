"""The reference's eval.py end to end on the B200 engine (SURVEY.md 8 f-3 / f-4 callers):

    step 1 (eval.py:198-243)  depth + confidence for every reference view of a scan
    step 2 (eval.py:245-353)  geometric filter, refinement, fusion, PLY

over the three layouts the reference reads (eval.py --dataset_name):

    dtu         DTUTestScan     <root>/Cameras/pair.txt, <root>/Cameras/{vid:08d}_cam.txt,
                                <root>/Rectified/<scan>/rect_{vid+1:03d}_3_r5000.png
    tanks       TanksScan       <root>/<split>/<scan>/pair.txt, cams/{vid:08d}_cam.txt,
                                images/{vid:08d}.jpg
    blendedmvs  BlendedMVSScan  <root>/<scan>/cams/pair.txt, cams/{vid:08d}_cam.txt,
                                blended_images/{vid:08d}.jpg, rendered_depth_maps/{vid:08d}.pfm

Each view's image is decoded once per scan on the host (PIL, a few threads), uploaded as bytes,
resized on the GPU bit-exactly like PIL's BILINEAR resize (casmvs_resize_u8_fwd) and kept there
(ViewCache); each reference view gathers its views and normalises them with
casmvs_normalize_u8_fwd.  Depth maps never pass through PFM files unless `depth_dir` is given
(then the reference's depth_XXXX.pfm / proba_XXXX.pfm are written as well).  Fusion colours are
decoded and resized with cv2 on the host like eval.py's, once per view.

    python -m casmvsnet_pl_b200.eval_pipeline --root_dir DTU --scan scan1 --ckpt ckpt.ckpt
    python -m casmvsnet_pl_b200.eval_pipeline --dataset_name tanks --root_dir TANKS \
        --split intermediate --scan Family --depth_interval DI --img_wh 1920 1056 --n_views 7

(DI: the scan's hand-tuned interval, listed in the reference's datasets/tanks.py)
"""
from __future__ import annotations

import argparse
import os
from collections import OrderedDict
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import fusion, io


def read_image_rgb_u8(path, img_wh):
    """cv2.imread + cv2.resize(INTER_LINEAR) + BGR->RGB (eval.py:76-79, 267-268) -> (H,W,3) uint8.
    (The reference's *network input* goes through PIL's BILINEAR resize, datasets/dtu.py:160-162;
    both decoders are host-side third-party code and are used as the reference uses them.)"""
    import cv2
    img = cv2.imread(path)
    if img is None:
        raise FileNotFoundError(path)
    return np.ascontiguousarray(cv2.resize(img, tuple(img_wh), interpolation=cv2.INTER_LINEAR)[:, :, ::-1])


def read_network_image_u8(path, img_wh):
    """PIL open + resize(BILINEAR) on the host (datasets/dtu.py:159-162) -> (H,W,3) uint8 RGB:
    the reference's per-view network input, which ViewCache computes on the GPU instead."""
    from PIL import Image
    img = Image.open(path).convert("RGB")
    if img.size != tuple(img_wh):
        img = img.resize(tuple(img_wh), Image.BILINEAR)
    return np.ascontiguousarray(np.asarray(img, dtype=np.uint8))


def _decode_rgb_u8(path):
    """PIL decode of one view's network input (datasets/dtu.py:159, tanks.py, blendedmvs.py:159)
    -> (H,W,3) uint8 RGB at the file's own size."""
    from PIL import Image
    with Image.open(path) as img:
        return np.array(img.convert("RGB"), dtype=np.uint8)


class ViewCache:
    """Network-input images of one scan, resident on the GPU: each view is decoded once on the
    host (PIL, `threads` at a time), uploaded as bytes and resized on the GPU (io.resize_images,
    bit-exact with the PIL BILINEAR resize the data sets apply), then kept as (h,w,3) uint8 until
    the byte budget forces the least recently used views out.  The reference decodes and resizes
    every view again for each reference view that uses it (about n_views times)."""

    def __init__(self, image_path, img_wh, device, budget_bytes=4 << 30, threads=4):
        self.image_path, self.img_wh, self.device = image_path, tuple(img_wh), device
        self.budget_bytes, self.threads = budget_bytes, threads
        self._views = OrderedDict()
        self.bytes = 0
        self.decoded = 0

    def get(self, vids):
        """-> (len(vids),h,w,3) uint8 CUDA tensor of the views `vids`, in that order."""
        missing = [v for v in dict.fromkeys(vids) if v not in self._views]
        if missing:
            paths = [self.image_path(v) for v in missing]
            if len(paths) > 1 and self.threads > 1:
                with ThreadPoolExecutor(min(self.threads, len(paths))) as pool:
                    decoded = list(pool.map(_decode_rgb_u8, paths))
            else:
                decoded = [_decode_rgb_u8(p) for p in paths]
            for v, u8 in zip(missing, decoded):
                t = io.resize_images(torch.from_numpy(u8[None]), self.img_wh, self.device)[0]
                self._views[v] = t
                self.bytes += t.numel()
            self.decoded += len(missing)
        for v in vids:
            self._views.move_to_end(v)
        keep = set(vids)
        while self.bytes > self.budget_bytes:
            v = next(iter(self._views))
            if v in keep:
                break
            self.bytes -= self._views.pop(v).numel()
        return torch.stack([self._views[v] for v in vids])


class _Scan:
    """Metas, per-view projection pyramids, per-reference-view init depth / depth interval and
    image paths of one scan.  Subclasses fill scan, img_wh, n_views, metas [(ref, [srcs])] (the
    reference views that are evaluated, pair-file order), proj_mats {vid: (levels,4,4)},
    depth_min {vid: float}, depth_interval {ref: float}, and define image_path(vid)."""

    def views(self, device, cache_bytes=4 << 30, threads=4):
        """yields (ref_vid, imgs (V,3,H,W) float32 on `device`, proj_mats (V-1,levels,3,4) host)."""
        cache = ViewCache(self.image_path, self.img_wh, device, cache_bytes, threads)
        for ref, srcs in self.metas:
            ids = [ref] + srcs[: self.n_views - 1]
            yield ref, io.normalize_images(cache.get(ids)), io.relative_proj_mats(self.proj_mats, ids)

    def _load_cams(self, vids, cam_path, levels, full_wh):
        for vid in vids:
            K, E, dmin = io.read_cam_file(cam_path(vid))
            self.proj_mats[vid] = io.pyramid_proj_mats(K, E, levels, self.img_wh, full_wh(vid))
            self.depth_min[vid] = dmin


def _img_wh(img_wh):
    """(w, h) as Python ints: a numpy integer would turn the float32 intrinsics scaling of
    io.pyramid_proj_mats into a float64 one and change the matrices' last bits."""
    w, h = int(img_wh[0]), int(img_wh[1])
    assert w % 32 == 0 and h % 32 == 0, "img_wh must both be multiples of 32!"
    return w, h


def _f32(x):
    """The value the reference hands the model: torch.FloatTensor([x]).item() (eval.py:62-63)."""
    return float(np.float32(x))


class DTUTestScan(_Scan):
    """The DTU test layout (datasets/dtu.py test mode):
        <root>/Cameras/pair.txt, <root>/Cameras/{vid:08d}_cam.txt,
        <root>/Rectified/<scan>/rect_{vid+1:03d}_3_r5000.png
    One depth interval (--depth_interval, 2.65 mm) for every reference view."""

    def __init__(self, root_dir, scan, img_wh=(1152, 864), n_views=5, levels=3, full_wh=(1600, 1200),
                 depth_interval=2.65):
        self.root_dir, self.scan, self.img_wh, self.n_views = root_dir, scan, _img_wh(img_wh), n_views
        self.metas = io.read_pair_file(os.path.join(root_dir, "Cameras", "pair.txt"))
        self.proj_mats, self.depth_min = {}, {}
        vids = sorted({r for r, _ in self.metas} | {s for _, ss in self.metas for s in ss})
        self._load_cams(vids, lambda v: os.path.join(root_dir, "Cameras", f"{v:08d}_cam.txt"),
                        levels, lambda v: full_wh)
        self.depth_interval = {r: depth_interval for r, _ in self.metas}

    def image_path(self, vid):
        return os.path.join(self.root_dir, "Rectified", self.scan, f"rect_{vid + 1:03d}_3_r5000.png")


class TanksScan(_Scan):
    """The Tanks and Temples layout of datasets/tanks.py:
        <root>/<split>/<scan>/pair.txt, cams/{vid:08d}_cam.txt, images/{vid:08d}.jpg
    init depth = depth_min of each reference view's cam file; `depth_interval` is per scan and
    hand-tuned (the reference's table is in its datasets/tanks.py).  The original image size is
    read from each image's header (the reference hard-codes the same sizes per scan).  Fusion
    colours come from the same <split>/<scan>/images directory (the reference's eval.py:89-91
    drops <split> there, which only works on a rearranged tree)."""

    def __init__(self, root_dir, split, scan, img_wh, n_views, depth_interval, levels=3):
        from PIL import Image
        self.dir = os.path.join(root_dir, split, scan)
        self.scan, self.img_wh, self.n_views = scan, _img_wh(img_wh), n_views
        self.metas = io.read_pair_file(os.path.join(self.dir, "pair.txt"))
        self.proj_mats, self.depth_min = {}, {}
        vids = list(dict.fromkeys([r for r, _ in self.metas] + [s for _, ss in self.metas for s in ss]))

        def full_wh(v):
            with Image.open(self.image_path(v)) as img:
                return img.size
        self._load_cams(vids, lambda v: os.path.join(self.dir, "cams", f"{v:08d}_cam.txt"), levels,
                        full_wh)
        self.depth_min = {v: _f32(d) for v, d in self.depth_min.items()}
        self.depth_interval = {r: _f32(depth_interval) for r, _ in self.metas}

    def image_path(self, vid):
        return os.path.join(self.dir, "images", f"{vid:08d}.jpg")


class BlendedMVSScan(_Scan):
    """The BlendedMVS layout of datasets/blendedmvs.py (test mode, img_wh given):
        <root>/<scan>/cams/pair.txt, cams/{vid:08d}_cam.txt, blended_images/{vid:08d}.jpg,
        rendered_depth_maps/{vid:08d}.pfm
    As the reference: a reference view whose pair.txt line counts fewer than n_views valid views
    is not evaluated; depths are rescaled by scale_factor = 100 / depth_min of the first cam in
    pair order (depth_min and the extrinsic translation, float32); the original size is 768x576
    under a root named dataset_low_res, else 2048x1536; per reference view
    depth_interval = (max of the scaled rendered depth, nearest-resized to img_wh,
    - depth_min) / n_depths_total.  Fusion uses the scaled projection matrices."""

    def __init__(self, root_dir, scan, img_wh, n_views, n_depths_total=192, levels=3):
        import cv2
        self.dir = os.path.join(root_dir, scan)
        self.scan, self.img_wh, self.n_views = scan, _img_wh(img_wh), n_views
        pairs = []
        with open(os.path.join(self.dir, "cams", "pair.txt")) as f:
            for _ in range(int(f.readline())):
                ref = int(f.readline().rstrip())
                line = f.readline().rstrip().split()
                pairs.append((ref, int(line[0]), [int(x) for x in line[1::2]]))
        self.metas = [(r, ss) for r, n_valid, ss in pairs if n_valid >= n_views]
        low_res = root_dir.endswith("dataset_low_res") or root_dir.endswith("dataset_low_res/")
        full_wh = (768, 576) if low_res else (2048, 1536)
        self.proj_mats, self.depth_min = {}, {}
        self.scale_factor = None
        vids = list(dict.fromkeys([r for r, _, _ in pairs] + [s for _, _, ss in pairs for s in ss]))
        for vid in vids:
            K, E, dmin = io.read_cam_file(os.path.join(self.dir, "cams", f"{vid:08d}_cam.txt"))
            if self.scale_factor is None:
                self.scale_factor = 100 / dmin            # the first cam decides
            dmin *= self.scale_factor
            E[:3, 3] *= self.scale_factor
            self.proj_mats[vid] = io.pyramid_proj_mats(K, E, levels, self.img_wh, full_wh)
            self.depth_min[vid] = dmin
        self.depth_interval = {}
        for ref, _ in self.metas:
            depth = np.array(io.read_pfm(os.path.join(self.dir, "rendered_depth_maps",
                                                      f"{ref:08d}.pfm"))[0], dtype=np.float32)
            depth *= self.scale_factor
            depth_max = cv2.resize(depth, self.img_wh, interpolation=cv2.INTER_NEAREST).max()
            self.depth_interval[ref] = _f32((depth_max - self.depth_min[ref]) / float(n_depths_total))
        self.depth_min = {v: _f32(d) for v, d in self.depth_min.items()}

    def image_path(self, vid):
        return os.path.join(self.dir, "blended_images", f"{vid:08d}.jpg")


def write_visuals(out_dir, vid, depth, proba, conf):
    """depth_visual_XXXX.jpg (JET colour map of depth normalised over its positive range) and
    proba_visual_XXXX.jpg (confidence_2 > conf, white) of eval.py:230-239."""
    import cv2
    os.makedirs(out_dir, exist_ok=True)
    pos = depth[depth > 0]
    mi = np.min(pos) if pos.size else np.float32(0)
    ma = np.max(depth)
    d = (depth - mi) / (ma - mi + 1e-8)
    d = (255 * d).astype(np.uint8)
    cv2.imwrite(os.path.join(out_dir, f"depth_visual_{vid:04d}.jpg"),
                cv2.applyColorMap(d, cv2.COLORMAP_JET))
    cv2.imwrite(os.path.join(out_dir, f"proba_visual_{vid:04d}.jpg"),
                (255 * (proba > conf)).astype(np.uint8))


@torch.no_grad()
def run_scan(model, scan, depth_interval=None, conf=0.999, min_geo_consistent=5,
             skip=1, max_ref_views=400, device="cuda:0", depth_dir=None, ply_path=None,
             save_visual=False, threads=4):
    """Step 1 and step 2 of eval.py for one scan (DTUTestScan, TanksScan or BlendedMVSScan).
    Each reference view runs with its own init depth (scan.depth_min[ref]) and depth interval
    (scan.depth_interval[ref], or `depth_interval` for all when given).
    -> (xyz (N,3) float32, rgb (N,3) uint8) CUDA tensors; optional PFM / visual / PLY outputs."""
    depths, probas = {}, {}
    writer = io.DepthWriter(depth_dir) if depth_dir else None
    if save_visual and not depth_dir:
        raise ValueError("save_visual writes next to the depth maps: give depth_dir")
    for ref, imgs, pm in scan.views(device, threads=threads):
        dint = scan.depth_interval[ref] if depth_interval is None else depth_interval
        res = model(imgs.unsqueeze(0), pm.unsqueeze(0).to(device), scan.depth_min[ref], dint)
        depths[ref] = torch.nan_to_num(res["depth_0"][0]).clone()            # eval.py:224-227
        probas[ref] = torch.nan_to_num(res["confidence_2"][0]).clone()
        if writer:
            d, p = depths[ref].cpu().numpy(), probas[ref].cpu().numpy()
            writer(scan.scan, ref, d, p)
            if save_visual:
                write_visuals(os.path.join(depth_dir, scan.scan), ref, d, p, conf)
    # fusion colours: cv2 decode + INTER_LINEAR resize like eval.py:86-94,266-268, once per view
    vids = list(depths)
    with ThreadPoolExecutor(max(1, threads)) as pool:
        rgb = list(pool.map(lambda v: read_image_rgb_u8(scan.image_path(v), scan.img_wh), vids))
    images = {v: torch.from_numpy(c).to(device).float() for v, c in zip(vids, rgb)}
    proj0 = {v: scan.proj_mats[v][0].numpy() for v in scan.proj_mats}     # finest level (eval.py:108)
    xyz, rgb = fusion.fuse_scan(scan.metas, depths, probas, images, proj0, conf, min_geo_consistent,
                                skip, max_ref_views)
    if ply_path:
        fusion.write_ply(ply_path, xyz, rgb)
    return xyz, rgb


def _scans(a):
    """--scan, else every scan of the split / list (eval.py:190-193)."""
    if a.scan:
        return [a.scan]
    if a.dataset_name == "dtu":
        d = os.path.join(a.root_dir, "Rectified")
        return sorted(x for x in os.listdir(d) if os.path.isdir(os.path.join(d, x)))
    if a.dataset_name == "tanks":
        d = os.path.join(a.root_dir, a.split)
        return sorted(x for x in os.listdir(d) if os.path.isfile(os.path.join(d, x, "pair.txt")))
    lists = {"train": "training_list.txt", "val": "validation_list.txt", "all": "all_list.txt"}
    if a.split not in lists:
        raise SystemExit(f"blendedmvs: --split must be one of {sorted(lists)} (or give --scan)")
    with open(os.path.join(a.root_dir, "..", lists[a.split])) as f:     # datasets/blendedmvs.py:37-45
        return [line.rstrip() for line in f if line.strip()]


def open_scan(a, scan):
    wh = tuple(a.img_wh)
    if a.dataset_name == "dtu":
        return DTUTestScan(a.root_dir, scan, wh, a.n_views,
                           depth_interval=2.65 if a.depth_interval is None else a.depth_interval)
    if a.dataset_name == "tanks":
        if a.depth_interval is None:
            raise SystemExit("tanks: give the scan's --depth_interval (hand-tuned per scan; see "
                             "the reference's datasets/tanks.py)")
        return TanksScan(a.root_dir, a.split, scan, wh, a.n_views, a.depth_interval)
    # eval.py hands --depth_interval to BlendedMVSDataset, which uses it as the number of depth
    # steps between depth_min and the rendered depth's maximum
    return BlendedMVSScan(a.root_dir, scan, wh, a.n_views,
                          192 if a.depth_interval is None else a.depth_interval)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root_dir", required=True)
    ap.add_argument("--dataset_name", default="dtu", choices=["dtu", "tanks", "blendedmvs"])
    ap.add_argument("--split", default="test",
                    help="tanks: intermediate | advanced; blendedmvs: train | val | all (scan list)")
    ap.add_argument("--scan", default="", help="one scan; default: every scan of the split")
    ap.add_argument("--ckpt", default="")
    ap.add_argument("--img_wh", nargs=2, type=int, default=[1152, 864])
    ap.add_argument("--n_views", type=int, default=5)
    ap.add_argument("--n_depths", nargs="+", type=int, default=[8, 32, 48])
    ap.add_argument("--interval_ratios", nargs="+", type=float, default=[1.0, 2.0, 4.0])
    ap.add_argument("--num_groups", type=int, default=1)
    ap.add_argument("--depth_interval", type=float, default=None,
                    help="dtu: default 2.65; tanks: required (per scan); blendedmvs: number of "
                         "depth steps over the rendered depth range, default 192")
    ap.add_argument("--conf", type=float, default=0.999)
    ap.add_argument("--min_geo_consistent", type=int, default=5)
    ap.add_argument("--max_ref_views", type=int, default=400)
    ap.add_argument("--skip", type=int, default=1)
    ap.add_argument("--save_visual", action="store_true")
    ap.add_argument("--precision", default="tf32", choices=["fp32", "tf32"])
    ap.add_argument("--out", default="", help="default results/<dataset_name>")
    a = ap.parse_args()
    out = a.out or os.path.join("results", a.dataset_name)
    scans = [open_scan(a, s) for s in _scans(a)]          # fail on a bad tree before loading
    from . import ABN
    from .models.mvsnet import CascadeMVSNet
    model = CascadeMVSNet(n_depths=a.n_depths, interval_ratios=a.interval_ratios,
                          num_groups=a.num_groups, norm_act=ABN, precision=a.precision)
    if a.ckpt:
        sd = torch.load(a.ckpt, map_location="cpu")
        sd = sd.get("state_dict", sd)
        sd = {k[len("model."):] if k.startswith("model.") else k: v for k, v in sd.items()}   # utils:57-59
        model.load_state_dict(sd)
    model = model.eval().cuda()
    os.makedirs(os.path.join(out, "points"), exist_ok=True)
    for scan in scans:
        xyz, _ = run_scan(model, scan, None, a.conf, a.min_geo_consistent, a.skip, a.max_ref_views,
                          depth_dir=os.path.join(out, "depth"),
                          ply_path=os.path.join(out, "points", f"{scan.scan}.ply"),
                          save_visual=a.save_visual)
        print(f"{scan.scan} contains {len(xyz) / 1e6:.2f} M points")


if __name__ == "__main__":
    main()

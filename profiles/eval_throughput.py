"""Step-1 throughput of the eval pipeline (eval.py:198-243: depth + confidence per reference
view) on a synthetic Tanks-layout scan of 1920x1080 JPEGs at the cfg5 geometry (1920x1056,
V=7, D=64/32/8), for the two image paths, in one run:

  per_ref   the reference's data path: every view of every reference view is decoded and
            PIL-resized on the host again (about V decodes per reference view), then uploaded
            as bytes and normalised on the GPU
  cached    eval_pipeline.ViewCache: each view is decoded once per scan (a few host threads),
            resized on the GPU by casmvs_resize_u8_fwd and kept there

Both paths run the same model on the same reference views; the depth maps are compared (the
resize is bit-exact, so they must be equal).  Also reported: the resize kernel time (CUDA
events over repeated launches on device-resident images), host decode time per image, and the
card's name and power limit.

    python profiles/eval_throughput.py [--views 64] [--refs 32] [--json out.json]
"""
import argparse
import ctypes
import io as pyio
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from casmvsnet_pl_b200 import ABN, _lib, eval_pipeline, io, synth   # noqa: E402
from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet         # noqa: E402

torch.set_grad_enabled(False)


def write_scan(root, n_views, src_wh, n_distinct=8, seed=0):
    """<root>/intermediate/Synth in the Tanks layout: n_views JPEGs (n_distinct different
    textured images), cam files looking at a plane ~2 units away, pair.txt with the 10 next
    views as sources."""
    from PIL import Image
    rng = np.random.default_rng(seed)
    d = os.path.join(root, "intermediate", "Synth")
    os.makedirs(os.path.join(d, "images"))
    os.makedirs(os.path.join(d, "cams"))
    w, h = src_wh
    jpgs = []
    for _ in range(n_distinct):
        coarse = rng.integers(0, 256, (h // 16 + 1, w // 16 + 1, 3), dtype=np.uint8)
        img = np.asarray(Image.fromarray(coarse).resize((w, h), Image.BICUBIC), dtype=np.int16)
        img = np.clip(img + rng.integers(-10, 11, (h, w, 3)), 0, 255).astype(np.uint8)
        buf = pyio.BytesIO()
        Image.fromarray(img).save(buf, format="JPEG", quality=90)
        jpgs.append(buf.getvalue())
    K = [[0.9 * w, 0, w / 2], [0, 0.9 * w, h / 2], [0, 0, 1]]
    for vid in range(n_views):
        with open(os.path.join(d, "images", f"{vid:08d}.jpg"), "wb") as f:
            f.write(jpgs[vid % n_distinct])
        t = np.deg2rad(0.5 * vid)
        E = np.eye(4)
        E[:3, :3] = [[np.cos(t), 0, np.sin(t)], [0, 1, 0], [-np.sin(t), 0, np.cos(t)]]
        E[:3, 3] = [-2 * np.sin(t), 0, 2 * (1 - np.cos(t))]
        rows = ["extrinsic"] + [" ".join(f"{v:.6f}" for v in r) for r in E] + ["", "intrinsic"]
        rows += [" ".join(f"{v:.6f}" for v in r) for r in K] + ["", "1.0 0.005"]
        with open(os.path.join(d, "cams", f"{vid:08d}_cam.txt"), "w") as f:
            f.write("\n".join(rows) + "\n")
    with open(os.path.join(d, "pair.txt"), "w") as f:
        f.write(f"{n_views}\n")
        for vid in range(n_views):
            srcs = [(vid + k) % n_views for k in range(1, 11)]
            f.write(f"{vid}\n10 " + " ".join(f"{s} {100 - s:.1f}" for s in srcs) + "\n")


def per_ref_views(scan, device):
    """The reference's path: decode + PIL resize of every view for every reference view."""
    for ref, srcs in scan.metas:
        ids = [ref] + srcs[: scan.n_views - 1]
        u8 = np.stack([eval_pipeline.read_network_image_u8(scan.image_path(v), scan.img_wh)
                       for v in ids])
        yield ref, io.normalize_images(torch.from_numpy(u8).pin_memory(), device), \
            io.relative_proj_mats(scan.proj_mats, ids)


def timed_step1(model, views, scan, n_refs, device):
    depths = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i, (ref, imgs, pm) in enumerate(views):
        if i == n_refs:
            break
        res = model(imgs.unsqueeze(0), pm.unsqueeze(0).to(device), scan.depth_min[ref],
                    scan.depth_interval[ref])
        depths.append(res["depth_0"][0].clone())
    torch.cuda.synchronize()
    return time.perf_counter() - t0, depths


def resize_kernel_us(src_wh, dst_wh, n_images, reps, device):
    """CUDA-event time of one casmvs_resize_u8_fwd launch over n_images device-resident images."""
    W, H = src_wh
    w, h = dst_wh
    src = torch.randint(0, 256, (n_images, H, W, 3), dtype=torch.uint8, device=device)
    dst = torch.empty(n_images, h, w, 3, dtype=torch.uint8, device=device)

    def tables(n_in, n_out):
        if n_in == n_out:
            return None, None, 0
        xmin, taps = io.pil_bilinear_coeffs(n_in, n_out)
        return torch.from_numpy(xmin).to(device), torch.from_numpy(taps).to(device), taps.shape[1]
    tx, ty = tables(W, w), tables(H, h)

    def p(t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else None
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        _lib.check(lib.casmvs_resize_u8_fwd(p(src), n_images, H, W, p(dst), h, w, p(tx[0]), p(tx[1]),
                                            tx[2], p(ty[0]), p(ty[1]), ty[2], st), "resize_u8")
    for _ in range(3):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    nbytes = n_images * (H * W + h * w) * 3
    return dict(src_wh=list(src_wh), dst_wh=list(dst_wh), images=n_images,
                us_per_launch=round(us, 2), us_per_image=round(us / n_images, 2),
                effective_GBps=round(nbytes / us / 1e3, 1))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=64)
    ap.add_argument("--refs", type=int, default=32, help="reference views timed per path")
    ap.add_argument("--n_views", type=int, default=7)
    ap.add_argument("--img_wh", nargs=2, type=int, default=[1920, 1056])
    ap.add_argument("--src_wh", nargs=2, type=int, default=[1920, 1080])
    ap.add_argument("--threads", type=int, default=4)
    ap.add_argument("--json", default="")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "eval_throughput measures the GPU pipeline: no GPU found"
    device = "cuda:0"
    out = dict(device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=card(),
               host_cpus=os.cpu_count(), views=a.views, refs_timed=a.refs, n_views=a.n_views,
               img_wh=a.img_wh, src_wh=a.src_wh, cache_threads=a.threads)
    with tempfile.TemporaryDirectory() as tmp:
        write_scan(tmp, a.views, tuple(a.src_wh))
        scan = eval_pipeline.TanksScan(tmp, "intermediate", "Synth", tuple(a.img_wh), a.n_views, 0.005)
        t0 = time.perf_counter()
        for _ in range(5):
            eval_pipeline._decode_rgb_u8(scan.image_path(0))
        out["host_decode_ms_per_image"] = round((time.perf_counter() - t0) / 5 * 1e3, 2)
        torch.manual_seed(0)
        model = CascadeMVSNet(n_depths=[8, 32, 64], norm_act=ABN, precision="tf32")
        synth.randomize_model_(model, 0)
        model = model.eval().to(device)
        # warm-up: every shape of the timed window (model, normalise, resize)
        timed_step1(model, scan.views(device, threads=a.threads), scan, 2, device)
        timed_step1(model, per_ref_views(scan, device), scan, 1, device)
        n = min(a.refs, len(scan.metas))
        t_old, d_old = timed_step1(model, per_ref_views(scan, device), scan, n, device)
        t_new, d_new = timed_step1(model, scan.views(device, threads=a.threads), scan, n, device)
        out["per_ref"] = dict(seconds=round(t_old, 3), ref_views_per_s=round(n / t_old, 2),
                              ms_per_ref_view=round(t_old / n * 1e3, 2))
        out["cached"] = dict(seconds=round(t_new, 3), ref_views_per_s=round(n / t_new, 2),
                             ms_per_ref_view=round(t_new / n * 1e3, 2))
        out["speedup"] = round(t_old / t_new, 2)
        out["depth_maps_equal"] = all(torch.equal(x, y) for x, y in zip(d_old, d_new))
    out["resize_kernel"] = [resize_kernel_us((1920, 1080), (1920, 1056), 7, 50, device),
                            resize_kernel_us((2048, 1080), (1920, 1056), 7, 50, device),
                            resize_kernel_us((1600, 1200), (1152, 864), 5, 50, device)]
    line = json.dumps(out)
    print(line)
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

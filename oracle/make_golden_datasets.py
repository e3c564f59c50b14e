"""Generate tests/golden/datasets_{tanks,blendedmvs}.npz from the REAL reference's TanksDataset
and BlendedMVSDataset (/root/reference/datasets), run in the build container.  TEST
INFRASTRUCTURE.

    python oracle/make_golden_datasets.py

Pins eval_pipeline.TanksScan / BlendedMVSScan and the GPU image path: small synthetic trees in
the two layouts (200x150 JPEGs, MVSNet cam files, pair.txt, rendered-depth PFMs; one
BlendedMVS reference view with too few valid source views, listed FIRST so that it also decides
the scale factor) are written to a temporary directory and read by the reference's own dataset
classes.  Stored per data set:
    file:<path>       every file of the scan directory, as bytes (tests rebuild the tree)
    metas             (M, 1+S) [ref, srcs...] of the evaluated reference views, padded with -1
    proj_vids, proj   (P,) / (P, levels, 4, 4) per-view projection pyramids
    rel               (M, V-1, levels, 3, 4) relative proj_mats of each sample
    init_depth_min, depth_interval   (M,) float32, as the samples carry them
    view_ids          (M, V) the views of each sample;  img_vids, imgs (K, 3, H, W) the
                      normalised network input of each view (identical in every sample)
    img_wh, n_views [, scale_factor, scan_depth_interval]
"""
import io as pyio
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("CASMVS_REFERENCE_ROOT", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")
IMG_WH, N_VIEWS, SRC_WH = (160, 128), 3, (200, 150)
TANKS_DEPTH_INTERVAL = 0.0123         # made up: the reference's hand-tuned table stays there


def cam_text(K, E, depth_min, interval):
    rows = ["extrinsic"] + [" ".join(f"{v:.6f}" for v in r) for r in E] + ["", "intrinsic"]
    rows += [" ".join(f"{v:.6f}" for v in r) for r in K] + ["", f"{depth_min} {interval}"]
    return "\n".join(rows) + "\n"


def pair_text(entries):
    """entries: [(ref, n_valid, [srcs])]"""
    rows = [str(len(entries))]
    for ref, n, srcs in entries:
        rows += [str(ref), " ".join([str(n)] + [f"{s} {100.0 - 7.5 * i:.1f}" for i, s in enumerate(srcs)])]
    return "\n".join(rows) + "\n"


def jpeg_bytes(rng):
    """A textured 200x150 RGB JPEG: blurred noise (JPEG-friendly) plus fine noise."""
    from PIL import Image
    w, h = SRC_WH
    coarse = rng.integers(0, 256, (h // 10 + 1, w // 10 + 1, 3), dtype=np.uint8)
    img = np.asarray(Image.fromarray(coarse).resize((w, h), Image.BICUBIC), dtype=np.int16)
    img = np.clip(img + rng.integers(-12, 13, (h, w, 3)), 0, 255).astype(np.uint8)
    buf = pyio.BytesIO()
    Image.fromarray(img).save(buf, format="JPEG", quality=90)
    return buf.getvalue()


def camera(vid, depth_min):
    t = np.deg2rad(4.0 * vid)
    E = np.eye(4)
    E[:3, :3] = [[np.cos(t), 0, np.sin(t)], [0, 1, 0], [-np.sin(t), 0, np.cos(t)]]
    E[:3, 3] = [-0.3 * depth_min * np.sin(t), 0.01 * vid, 0.3 * depth_min * (1 - np.cos(t))]
    K = np.array([[180.5, 0.0, 99.25], [0.0, 181.0, 74.75], [0.0, 0.0, 1.0]])
    return K, E


def write_tree(scan_dir, files):
    for rel, data in files.items():
        path = os.path.join(scan_dir, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "wb") as f:
            f.write(data)


def collect(ds, extra):
    """Run ds[i] for every meta and pack the results."""
    out = dict(extra)
    rows, rel, dmin, dint, ids, imgs = [], [], [], [], [], {}
    for i in range(len(ds)):
        sample = ds[i]
        _, _, ref, srcs = ds.metas[i]
        view_ids = [ref] + srcs[:N_VIEWS - 1]
        rows.append([ref] + srcs)
        rel.append(sample["proj_mats"].numpy())
        dmin.append(sample["init_depth_min"].item())
        dint.append(sample["depth_interval"].item())
        ids.append(view_ids)
        for v, img in zip(view_ids, sample["imgs"]):
            if v in imgs:
                assert torch.equal(imgs[v], img)
            imgs[v] = img
    width = max(len(r) for r in rows)
    out["metas"] = np.array([r + [-1] * (width - len(r)) for r in rows])
    out["rel"] = np.stack(rel)
    out["init_depth_min"] = np.array(dmin, np.float32)
    out["depth_interval"] = np.array(dint, np.float32)
    out["view_ids"] = np.array(ids)
    out["img_vids"] = np.array(sorted(imgs))
    out["imgs"] = torch.stack([imgs[v] for v in sorted(imgs)]).numpy()
    out["img_wh"], out["n_views"] = np.array(IMG_WH), np.array(N_VIEWS)
    return out


def save(name, out, files):
    for rel, data in files.items():
        out["file:" + rel] = np.frombuffer(data, np.uint8)
    path = os.path.join(OUT, f"datasets_{name}.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def tanks(tmp, rng):
    from datasets.tanks import TanksDataset
    n = 4
    files = {"pair.txt": pair_text([(0, 3, [1, 2, 3]), (1, 3, [0, 2, 3]), (2, 3, [1, 3, 0]),
                                    (3, 2, [2, 1])]).encode()}
    for vid in range(n):
        dmin = 1.5 + 0.125 * vid
        K, E = camera(vid, dmin)
        files[f"cams/{vid:08d}_cam.txt"] = cam_text(K, E, dmin, 0.01).encode()
        files[f"images/{vid:08d}.jpg"] = jpeg_bytes(rng)
    root = os.path.join(tmp, "tanks")
    # the reference's build_metas / build_proj_mats walk its fixed scan list: every scan gets
    # the same pair / cam files, the first one also the images
    ds = object.__new__(TanksDataset)
    ds.root_dir, ds.img_wh, ds.split, ds.n_views, ds.levels = root, IMG_WH, "intermediate", N_VIEWS, 3
    for scan in ("Family", "Francis", "Horse", "Lighthouse", "M60", "Panther", "Playground", "Train"):
        write_tree(os.path.join(root, "intermediate", scan),
                   files if scan == "Family" else {k: v for k, v in files.items() if not k.startswith("images/")})
    ds.build_metas()
    scan = ds.scans[0]
    ds.image_sizes[scan] = SRC_WH                 # the per-scan size table, true for these files
    ds.depth_interval = {scan: TANKS_DEPTH_INTERVAL}
    ds.metas = [m for m in ds.metas if m[0] == scan]
    ds.build_proj_mats()
    ds.define_transforms()
    vids = sorted(ds.proj_mats[scan])
    out = collect(ds, dict(
        proj_vids=np.array(vids), proj=torch.stack([ds.proj_mats[scan][v][0] for v in vids]).numpy(),
        view_depth_min=np.array([ds.proj_mats[scan][v][1] for v in vids]),
        scan_depth_interval=np.array(TANKS_DEPTH_INTERVAL)))
    save("tanks", out, files)


def blendedmvs(tmp, rng):
    from datasets.blendedmvs import BlendedMVSDataset
    from datasets.utils import save_pfm
    n = 5
    # view 3 comes first and has too few valid source views: skipped, yet its cam decides the
    # scale factor; it is also a source of view 4, whose fusion then lacks a depth map
    files = {"cams/pair.txt": pair_text([(3, 1, [2]), (0, 4, [1, 2, 4, 3]), (1, 3, [0, 2, 4]),
                                         (2, 3, [1, 0, 4]), (4, 3, [3, 2, 1])]).encode()}
    for vid in range(n):
        dmin = 480.0 + 25.0 * vid
        K, E = camera(vid, dmin)
        E[:3, 3] *= 300.0                          # BlendedMVS scenes have large extents
        files[f"cams/{vid:08d}_cam.txt"] = cam_text(K, E, dmin, 1.0).encode()
        files[f"blended_images/{vid:08d}.jpg"] = jpeg_bytes(rng)
        depth = (dmin * (1.0 + 2.0 * rng.random((30, 40)))).astype(np.float32)
        path = os.path.join(tmp, "depth.pfm")
        save_pfm(path, depth)
        with open(path, "rb") as f:
            files[f"rendered_depth_maps/{vid:08d}.pfm"] = f.read()
    scan = "5b0000000000000000000000"
    root = os.path.join(tmp, "BlendedMVS", "dataset_low_res")
    write_tree(os.path.join(root, scan), files)
    with open(os.path.join(tmp, "BlendedMVS", "validation_list.txt"), "w") as f:
        f.write(scan + "\n")
    ds = BlendedMVSDataset(root, "val", n_views=N_VIEWS, levels=3, depth_interval=192.0, img_wh=IMG_WH)
    vids = sorted(ds.proj_mats[scan])
    out = collect(ds, dict(
        proj_vids=np.array(vids), proj=torch.stack([ds.proj_mats[scan][v][0] for v in vids]).numpy(),
        view_depth_min=np.array([ds.proj_mats[scan][v][1] for v in vids]),
        scale_factor=np.array(ds.scale_factors[scan]),
        skipped=np.array([v for v in ds.ref_views_per_scan[scan]
                          if v not in [m[2] for m in ds.metas]])))
    save("blendedmvs", out, files)


def main():
    sys.path.insert(0, REF)
    rng = np.random.default_rng(0)
    with tempfile.TemporaryDirectory() as tmp:
        tanks(tmp, rng)
        blendedmvs(tmp, rng)


if __name__ == "__main__":
    main()

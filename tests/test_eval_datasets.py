"""Tanks and Temples / BlendedMVS scans of the eval pipeline and the PIL-exact image resize,
against PIL itself and against fixtures the REAL reference's TanksDataset / BlendedMVSDataset
produced on small synthetic trees (oracle/make_golden_datasets.py)."""
import os

import numpy as np
import pytest
import torch

from casmvsnet_pl_b200 import io as cio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")

# (in (W,H), out (w,h)): the data sets' pairs, upscale, identity, one axis, odd sizes, big ratios
SIZE_PAIRS = [((1920, 1080), (1920, 1056)), ((1600, 1200), (1152, 864)),
              ((2048, 1080), (1920, 1056)), ((200, 150), (160, 128)), ((100, 80), (160, 128)),
              ((37, 23), (37, 23)), ((37, 23), (37, 11)), ((37, 23), (19, 23)), ((7, 5), (3, 9)),
              ((301, 203), (17, 13)), ((1, 1), (5, 3))]


def pil_resize(u8, wh):
    from PIL import Image
    return np.asarray(Image.fromarray(u8).resize(tuple(wh), Image.BILINEAR))


def np_resize(u8, wh):
    """The integer passes of casmvs_resize_u8_fwd restated in numpy on pil_bilinear_coeffs."""
    def one_pass(a, axis, n_in, n_out):
        if n_in == n_out:
            return a
        xmin, taps = cio.pil_bilinear_coeffs(n_in, n_out)
        a = np.moveaxis(a, axis, 0)
        acc = np.full((n_out,) + a.shape[1:], 1 << 21, np.int64)
        for j in range(taps.shape[1]):
            src = np.minimum(xmin + j, n_in - 1)            # taps past the edge are 0
            acc += a[src] * taps[:, j].reshape((-1,) + (1,) * (a.ndim - 1))
        return np.moveaxis(np.clip(acc >> 22, 0, 255), 0, axis)
    H, W = u8.shape[:2]
    out = one_pass(u8.astype(np.int64), 1, W, wh[0])        # horizontal first, clipped to uint8
    return one_pass(out, 0, H, wh[1]).astype(np.uint8)


@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_integer_resample_restatement_equals_pil(src, dst):
    rng = np.random.default_rng(src[0] * 7 + dst[1])
    img = rng.integers(0, 256, (src[1], src[0], 3), dtype=np.uint8)
    assert np.array_equal(np_resize(img, dst), pil_resize(img, dst))


def test_pil_bilinear_coeffs_layout():
    xmin, taps = cio.pil_bilinear_coeffs(1080, 1056)
    assert xmin.dtype == np.int32 and taps.dtype == np.int32 and taps.shape == (1056, 3)
    assert xmin[0] == 0 and xmin[-1] + 3 >= 1080 - 1
    # each row sums to 2^22 up to the per-tap rounding; downscales up to 2x need <= 4 taps
    assert np.abs(taps.sum(1) - (1 << 22)).max() <= 2
    for n_in, n_out in ((1600, 1152), (1200, 864), (2048, 1920), (200, 160), (150, 128)):
        assert cio.pil_bilinear_coeffs(n_in, n_out)[1].shape[1] <= 4
    with pytest.raises(ValueError):
        cio.pil_bilinear_coeffs(0, 4)


def test_resize_refuses_taps_beyond_shared_memory():
    """The tap-count check runs before any launch (no GPU needed)."""
    from casmvsnet_pl_b200 import _lib
    lib = _lib.load()
    src, dst = 16, 4096                                       # never dereferenced
    rc = lib.casmvs_resize_u8_fwd(src, 1, 8, 8000, dst, 8, 10, src, src, 1601, None, None, 0, None)
    assert rc < 0 and b"shared memory" in lib.casmvs_last_error()
    rc = lib.casmvs_resize_u8_fwd(src, 1, 8, 16, dst, 8, 10, None, None, 0, None, None, 0, None)
    assert rc < 0 and b"horizontal taps" in lib.casmvs_last_error()
    rc = lib.casmvs_resize_u8_fwd(src, 1, 8, 16, src, 8, 16, None, None, 0, None, None, 0, None)
    assert rc < 0 and b"in-place" in lib.casmvs_last_error()
    assert lib.casmvs_resize_u8_fwd(src, 0, 8, 16, dst, 8, 16, None, None, 0, None, None, 0, None) == 0


# ------------------------------------------------------------------------------ data sets
def _golden(name):
    with np.load(os.path.join(G, f"datasets_{name}.npz")) as z:
        return {k: z[k] for k in z.files}


def _rebuild(g, scan_dir):
    for k, v in g.items():
        if k.startswith("file:"):
            path = os.path.join(scan_dir, k[len("file:"):])
            os.makedirs(os.path.dirname(path), exist_ok=True)
            with open(path, "wb") as f:
                f.write(v.tobytes())


def tanks_scan(tmp_path, g):
    from casmvsnet_pl_b200 import eval_pipeline
    _rebuild(g, str(tmp_path / "tanks" / "intermediate" / "Synth"))
    return eval_pipeline.TanksScan(str(tmp_path / "tanks"), "intermediate", "Synth",
                                   tuple(g["img_wh"]), int(g["n_views"]),
                                   float(g["scan_depth_interval"]))


def blendedmvs_scan(tmp_path, g):
    from casmvsnet_pl_b200 import eval_pipeline
    root = tmp_path / "BlendedMVS" / "dataset_low_res"
    _rebuild(g, str(root / "synth"))
    return eval_pipeline.BlendedMVSScan(str(root), "synth", tuple(g["img_wh"]), int(g["n_views"]))


SCANS = {"tanks": tanks_scan, "blendedmvs": blendedmvs_scan}


@pytest.mark.parametrize("name", sorted(SCANS))
def test_scan_matches_reference_dataset(tmp_path, name):
    g = _golden(name)
    scan = SCANS[name](tmp_path, g)
    metas = [[r] + s + [-1] * (g["metas"].shape[1] - 1 - len(s)) for r, s in scan.metas]
    assert np.array_equal(np.array(metas), g["metas"])
    for vid, P in zip(g["proj_vids"], g["proj"]):
        assert np.array_equal(scan.proj_mats[int(vid)].numpy(), P)
    for i, (ref, _) in enumerate(scan.metas):
        ids = [int(v) for v in g["view_ids"][i]]
        assert np.array_equal(cio.relative_proj_mats(scan.proj_mats, ids).numpy(), g["rel"][i])
        assert np.float32(scan.depth_min[ref]) == g["init_depth_min"][i]
        assert scan.depth_min[ref] == float(g["init_depth_min"][i])
        assert scan.depth_interval[ref] == float(g["depth_interval"][i])
    if name == "blendedmvs":
        assert scan.scale_factor == float(g["scale_factor"])
        assert len(g["skipped"]) == 1 and int(g["skipped"][0]) not in [r for r, _ in scan.metas]


# ------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_resize_images_bit_exact_vs_pil(src, dst):
    rng = np.random.default_rng(src[1] * 5 + dst[0])
    n = 2 if src[0] * src[1] > 1e6 else 3
    batch = rng.integers(0, 256, (n, src[1], src[0], 3), dtype=np.uint8)
    ref = np.stack([pil_resize(b, dst) for b in batch])
    got = cio.resize_images(batch, dst, device="cuda:0")
    assert got.is_cuda and got.dtype == torch.uint8 and tuple(got.shape) == ref.shape
    assert np.array_equal(got.cpu().numpy(), ref)
    # device-resident input
    dev = torch.from_numpy(batch).cuda()
    assert np.array_equal(cio.resize_images(dev, dst).cpu().numpy(), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCANS))
def test_pipeline_network_input_equals_reference(tmp_path, name):
    g = _golden(name)
    scan = SCANS[name](tmp_path, g)
    index = {int(v): i for i, v in enumerate(g["img_vids"])}
    n = 0
    for i, (ref, imgs, pm) in enumerate(scan.views("cuda:0", threads=2)):
        want = g["imgs"][[index[int(v)] for v in g["view_ids"][i]]]
        assert ref == g["metas"][i, 0]
        assert np.array_equal(imgs.cpu().numpy(), want)
        assert np.array_equal(pm.numpy(), g["rel"][i])
        n += 1
    assert n == len(g["metas"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCANS))
def test_run_scan_on_dataset_tree(tmp_path, name):
    """eval.py step 1 + 2 on the rebuilt tree: one depth / proba PFM and visual per evaluated
    reference view (none for the view the reference skips), each depth equal to an eager
    forward on the reference's inputs, and a PLY."""
    pytest.importorskip("cv2")
    from casmvsnet_pl_b200 import ABN, eval_pipeline, synth
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet
    g = _golden(name)
    scan = SCANS[name](tmp_path, g)
    torch.manual_seed(0)
    model = CascadeMVSNet(norm_act=ABN, precision="tf32")
    synth.randomize_model_(model, 0)
    model = model.eval().cuda()
    depth_dir = tmp_path / "depth"
    xyz, rgb = eval_pipeline.run_scan(model, scan, conf=0.0, min_geo_consistent=0,
                                      depth_dir=str(depth_dir), ply_path=str(tmp_path / "s.ply"),
                                      save_visual=True)
    refs = [int(r) for r in g["metas"][:, 0]]
    files = sorted(os.listdir(depth_dir / scan.scan))
    want = sorted(f"{kind}_{r:04d}.{ext}" for r in refs
                  for kind, ext in (("depth", "pfm"), ("proba", "pfm"),
                                    ("depth_visual", "jpg"), ("proba_visual", "jpg")))
    assert files == want
    index = {int(v): i for i, v in enumerate(g["img_vids"])}
    for i, ref in enumerate(refs):
        imgs = torch.from_numpy(g["imgs"][[index[int(v)] for v in g["view_ids"][i]]])
        res = model(imgs.unsqueeze(0).cuda(), torch.from_numpy(g["rel"][i]).unsqueeze(0).cuda(),
                    float(g["init_depth_min"][i]), float(g["depth_interval"][i]))
        d, _ = cio.read_pfm(depth_dir / scan.scan / f"depth_{ref:04d}.pfm")
        c, _ = cio.read_pfm(depth_dir / scan.scan / f"proba_{ref:04d}.pfm")
        assert np.array_equal(d, np.nan_to_num(res["depth_0"][0].cpu().numpy()))
        assert np.array_equal(c, np.nan_to_num(res["confidence_2"][0].cpu().numpy()))
    assert len(xyz) == len(rgb) > 0 and xyz.shape[1] == 3
    assert os.path.getsize(tmp_path / "s.ply") > 15 * len(xyz)

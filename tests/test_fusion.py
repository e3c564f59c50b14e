"""Geometric-consistency filter + fusion (SURVEY.md 8 f-3): the numpy oracle is pinned to the
REAL reference's functions (golden fixture), the GPU kernel is compared with the oracle."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import fusion_oracle as FO                       # noqa: E402


@pytest.fixture(scope="module")
def g():
    with np.load(os.path.join(ROOT, "tests", "golden", "fusion_64x48.npz")) as z:
        return {k: z[k] for k in z.files}


def test_oracle_matches_reference_golden(g):
    H, W = g["depths"][0].shape
    for s in range(1, len(g["P"])):
        r, m, i2 = FO.check_geo_consistency(g["depths"][0], g["P"][0], g["depths"][s], g["P"][s],
                                            g["images"][0], g["images"][s], (W, H))
        # numba(fastmath) vs numpy differ in the last ulp of the matrix products: masks may flip
        # only where a test sits on its threshold
        assert (m != g["mask"][s - 1]).mean() < 2e-3
        both = m & g["mask"][s - 1]
        assert np.abs(r - g["reproj"][s - 1])[both].max() < 1e-3
        assert np.abs(i2 - g["img2ref"][s - 1])[both].max() < 1e-2
    assert np.abs(FO.resize4_linear(g["proba"]) - g["proba_up"]).max() < 1e-6


def test_restated_cv2_algorithms_match_cv2(g):
    """_remap_linear / _resize4_linear restate the third-party cv2 algorithms (used only when
    cv2 is absent): check them against cv2 itself."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    img = g["depths"][1]
    H, W = img.shape
    mx = rng.uniform(-3, W + 2, (H, W)).astype(np.float32)
    my = rng.uniform(-3, H + 2, (H, W)).astype(np.float32)
    mx[0, 0], my[0, 1] = np.nan, np.inf
    want = cv2.remap(img, mx, my, interpolation=cv2.INTER_LINEAR)
    got = FO._remap_linear(img, mx, my)
    assert np.abs(got - want).max() < 1e-3 * np.abs(img).max()
    col = g["images"][1]
    assert np.abs(FO._remap_linear(col, mx, my) - cv2.remap(col, mx, my, interpolation=cv2.INTER_LINEAR)).max() < 1e-3 * 255
    assert np.abs(FO._resize4_linear(g["proba"]) - g["proba_up"]).max() < 1e-6


@pytest.mark.gpu
def test_gpu_refine_ref_view_vs_oracle(g):
    from casmvsnet_pl_b200 import fusion
    dev = "cuda:0"
    H, W = g["depths"][0].shape
    S = len(g["P"]) - 1
    want = FO.refine_ref_view(g["depths"][0], g["P"][0], g["images"][0], g["proba"],
                              list(g["depths"][1:]), list(g["P"][1:]), list(g["images"][1:]),
                              (W, H), conf=0.995, min_geo_consistent=2)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    got = fusion.refine_ref_view(t(g["depths"][0]), g["P"][0], [t(d) for d in g["depths"][1:]],
                                 list(g["P"][1:]), t(g["images"][0]), [t(i) for i in g["images"][1:]],
                                 t(g["proba"]), conf=0.995, min_geo_consistent=2, debug=True)
    mask = got["mask"].cpu().numpy()
    flips = (mask != want["masks"]).mean()
    print("mask flips", flips, "consistent fraction", want["masks"].mean())
    assert flips < 2e-3
    both = mask & want["masks"]
    assert np.abs(got["reproj"].cpu().numpy() - want["reprojs"])[both].max() < 2e-3
    same = (got["geo_count"].cpu().numpy() == want["mask_geo_sum"])
    assert same.mean() > 0.995
    d = np.abs(got["depth_refined"].cpu().numpy() - want["depth_refined"])[same]
    assert d.max() < 2e-3
    c = np.abs(got["image_refined"].cpu().numpy() - want["image_refined"])[same]
    assert c.max() < 2e-2
    mf = got["mask_final"].cpu().numpy()
    assert (mf != want["mask_final"]).mean() < 5e-3
    sel = mf & want["mask_final"] & same
    pts = got["points"].cpu().numpy()[sel]
    ref_pts = np.full((H, W, 3), np.nan, np.float64)
    ref_pts[want["mask_final"]] = want["xyz_world"]
    assert np.abs(pts - ref_pts[sel]).max() < 5e-3           # mm, depths ~600


@pytest.mark.gpu
def test_gpu_fuse_scan_and_ply(g, tmp_path):
    """Scan loop with the refined-view cache (eval.py:245-330) + PLY layout."""
    from casmvsnet_pl_b200 import fusion
    dev = "cuda:0"
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    n = len(g["P"])
    depths = {v: t(g["depths"][v]) for v in range(n)}
    images = {v: t(g["images"][v]) for v in range(n)}
    probas = {v: t(np.full_like(g["proba"], 1.0)) for v in range(n)}
    proj = {v: g["P"][v] for v in range(n)}
    metas = [(0, [1, 2, 3]), (1, [0, 2]), (2, [0, 1, 3]), (3, [7])]       # view 7 has no prediction
    xyz, rgb = fusion.fuse_scan(metas, depths, probas, images, proj, conf=0.5, min_geo_consistent=1)
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and len(xyz) == len(rgb) > 1000
    # every fused point re-projects into view 0's frustum at a plausible depth
    P0 = torch.from_numpy(g["P"][0]).to(dev)
    q = (P0[:3, :3] @ xyz.T + P0[:3, 3:]).T
    assert (q[:, 2] > 400).all() and (q[:, 2] < 900).all()
    fusion.write_ply(tmp_path / "s.ply", xyz, rgb)
    raw = open(tmp_path / "s.ply", "rb").read()
    head, body = raw.split(b"end_header\n")
    assert f"element vertex {len(xyz)}".encode() in head and len(body) == 15 * len(xyz)
    first = np.frombuffer(body[:12], "<f4")
    assert np.allclose(first, xyz[0].cpu().numpy())

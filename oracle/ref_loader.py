"""TEST INFRASTRUCTURE — loader for the REAL reference (`/root/reference/models`).

Only usable in the build container (``/root/reference`` does not exist on the
GPU box).  It is used by ``oracle/make_golden.py`` to generate the committed
golden vectors that pin the restatement in ``oracle/casmvs_oracle.py``; the
tests read only those vectors.

The reference imports two third-party packages that are neither installed nor
vendored (SURVEY.md §8c): ``inplace_abn`` (README.md:28, unpinned) and
``kornia==0.2.0`` (requirements.txt:4).  We inject minimal stand-ins with the
documented semantics:

* ``inplace_abn.ABN`` / ``InPlaceABN``: BatchNorm (eps 1e-5, momentum 0.1)
  followed by LeakyReLU(0.01) — the package defaults.
* ``kornia.utils.create_meshgrid(H, W, normalized_coordinates=False)``:
  (1, H, W, 2) float32, ``[..., 0] = x`` in [0, W-1], ``[..., 1] = y``.
"""
import importlib
import os
import sys
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

REFERENCE_ROOT = os.environ.get("CASMVS_REFERENCE_ROOT", "/root/reference")


class _ABN(nn.Module):
    """Activated batch norm stand-in: F.batch_norm + F.leaky_relu(0.01)."""

    def __init__(self, num_features, eps=1e-5, momentum=0.1,
                 activation="leaky_relu", activation_param=0.01):
        super().__init__()
        self.num_features = num_features
        self.eps = eps
        self.momentum = momentum
        self.activation = activation
        self.activation_param = activation_param
        self.weight = nn.Parameter(torch.ones(num_features))
        self.bias = nn.Parameter(torch.zeros(num_features))
        self.register_buffer("running_mean", torch.zeros(num_features))
        self.register_buffer("running_var", torch.ones(num_features))

    def forward(self, x):
        x = F.batch_norm(x, self.running_mean, self.running_var, self.weight,
                         self.bias, self.training, self.momentum, self.eps)
        return F.leaky_relu(x, self.activation_param)


def _create_meshgrid(height, width, normalized_coordinates=True, device=None):
    xs = torch.linspace(0, width - 1, width, device=device, dtype=torch.float32)
    ys = torch.linspace(0, height - 1, height, device=device, dtype=torch.float32)
    if normalized_coordinates:
        xs = (xs / (width - 1) - 0.5) * 2
        ys = (ys / (height - 1) - 0.5) * 2
    gy, gx = torch.meshgrid(ys, xs, indexing="ij")
    return torch.stack([gx, gy], dim=-1).unsqueeze(0)


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "mvsnet.py"))


def load_reference_models():
    """Import the reference's own ``models`` package; returns (mvsnet, modules, ABN)."""
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if "inplace_abn" not in sys.modules:
        m = types.ModuleType("inplace_abn")
        m.ABN = _ABN
        m.InPlaceABN = _ABN
        sys.modules["inplace_abn"] = m
    if "kornia" not in sys.modules:
        k = types.ModuleType("kornia")
        ku = types.ModuleType("kornia.utils")
        ku.create_meshgrid = _create_meshgrid
        k.utils = ku
        sys.modules["kornia"] = k
        sys.modules["kornia.utils"] = ku
    # import under a private name so it never shadows this repo's own `models`
    spec_root = os.path.join(REFERENCE_ROOT, "models")
    pkg_name = "_casmvs_reference_models"
    if pkg_name not in sys.modules:
        spec = importlib.util.spec_from_file_location(
            pkg_name, os.path.join(spec_root, "__init__.py"),
            submodule_search_locations=[spec_root])
        pkg = importlib.util.module_from_spec(spec)
        sys.modules[pkg_name] = pkg
        spec.loader.exec_module(pkg)
    modules = importlib.import_module(pkg_name + ".modules")
    mvsnet = importlib.import_module(pkg_name + ".mvsnet")
    return mvsnet, modules, _ABN


def make_reference_model(n_depths, interval_ratios, num_groups):
    """Reference CascadeMVSNet in inference mode.

    For G=1 the eval-mode branch (models/mvsnet.py:155) does an in-place add on
    an expanded stride-0 view and raises on modern torch; the arithmetic-identical
    out-of-place branch (:152-153) is selected by flipping only the top-level
    ``training`` flag (children keep eval-mode BN).  SURVEY.md §0/§8c.
    """
    mvsnet, _, abn = load_reference_models()
    model = mvsnet.CascadeMVSNet(n_depths=list(n_depths),
                                 interval_ratios=list(interval_ratios),
                                 num_groups=num_groups, norm_act=abn)
    model.eval()
    if num_groups == 1:
        model.training = True
    return model

"""Writes tests/golden/losses_ref.npz: the five terms the REFERENCE's own LossComputer (diffusionGS/utils/losses.py:239-369,
executed by path) returns on the seeded inputs of tests/test_losses_cpu.py, with the absent packages (lpips,
pytorch_msssim, skimage) stubbed by the deterministic stand-in modules below.

    DGS_REFERENCE_ROOT=<checkout of the reference> python tests/golden/make_losses_golden.py
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_import as ri  # noqa: E402

PATH = os.path.join(HERE, "losses_ref.npz")
TERMS = ("l2", "lpips", "ssim", "pointsdist", "l2_xyz")
TARGET_CHANNELS = (3, 4)


class FakeLPIPS(nn.Module):  # stand-in with LPIPS' call signature: per-image scalar [n,1,1,1]
    def __init__(self, net="vgg"):
        super().__init__()
        self.w = nn.Parameter(torch.ones(1))

    def forward(self, x, y):
        return ((x - y) ** 2).mean(dim=(1, 2, 3), keepdim=True) * self.w


class FakeSSIM(nn.Module):  # pytorch_msssim.SSIM(size_average=False) -> [n]
    def __init__(self, **kw):
        super().__init__()

    def forward(self, x, y):
        return 1.0 - (x - y).abs().mean(dim=(1, 2, 3))


def inputs(tc):
    """(rendering, target with tc channels, masks, ray_o, img_aligned_xyz, gt_img_aligned_xyz)"""
    g = torch.Generator().manual_seed(0)
    b, v, h, w = 2, 3, 16, 24
    rendering = torch.rand(b, v, 3, h, w, generator=g, requires_grad=True)
    target = torch.rand(b, v, tc, h, w, generator=g)
    masks = (torch.rand(b, v, 1, h, w, generator=g) > 0.3).float()
    ray_o = torch.randn(b, v, 3, h, w, generator=g)
    xyz = torch.randn(b, v, 3, h, w, generator=g, requires_grad=True)
    gt_xyz = torch.randn(b, v, 3, h, w, generator=g)
    return rendering, target, masks, ray_o, xyz, gt_xyz


def load_reference_losses():
    for name, attrs in (("lpips", dict(LPIPS=FakeLPIPS)), ("pytorch_msssim", dict(SSIM=FakeSSIM)),
                        ("skimage", {}), ("skimage.metrics", dict(structural_similarity=None))):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        m.__path__ = []
        sys.modules.setdefault(name, m)
    spec = importlib.util.spec_from_file_location("_ref_losses", os.path.join(ri.REF, "diffusionGS/utils/losses.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    ref = load_reference_losses().LossComputer()
    rec = {}
    for tc in TARGET_CHANNELS:
        rendering, target, masks, ray_o, xyz, gt_xyz = inputs(tc)
        out = ref(rendering, target, masks, masks, ray_o, img_aligned_xyz=xyz, gt_img_aligned_xyz=gt_xyz)
        rec.update({f"tc{tc}/{k}": v.detach().numpy() for k, v in zip(TERMS, out)})
    np.savez_compressed(PATH, **rec)
    print(PATH, os.path.getsize(PATH), "bytes")


if __name__ == "__main__":
    main()

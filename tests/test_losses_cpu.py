"""Loss stage (SURVEY 8f row 1) host logic on CPU tensors: dgs_b200.losses.LossComputer / C against what the REFERENCE's
own LossComputer (diffusionGS/utils/losses.py:239-369) returned on the same inputs (tests/golden/make_losses_golden.py,
the absent packages lpips, pytorch_msssim and skimage stubbed by deterministic stand-in modules), and schedule function C
(utils/misc.py:73-94)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

from dgs_b200 import losses

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_losses_golden as mlg  # noqa: E402


class _SsimLoss(nn.Module):  # the reference's SsimLoss (losses.py:216-236) around the SSIM stand-in
    def forward(self, x, y):
        return 1 - mlg.FakeSSIM()(x, y)


@pytest.mark.parametrize("tc", mlg.TARGET_CHANNELS)
def test_loss_computer_equals_reference(tc):
    z = np.load(mlg.PATH)
    a = [torch.from_numpy(z[f"tc{tc}/{k}"]) for k in mlg.TERMS]
    ours = losses.LossComputer(lpips_module=mlg.FakeLPIPS(), ssim_module=_SsimLoss(), compute_pointsdist=True)
    rendering, target, masks, ray_o, xyz, gt_xyz = mlg.inputs(tc)
    o = ours(rendering, target, masks, masks, ray_o, img_aligned_xyz=xyz, gt_img_aligned_xyz=gt_xyz)
    for name, x, y in zip(mlg.TERMS, o, a):
        assert x.shape == y.shape, name
        assert torch.allclose(x, y, rtol=1e-6, atol=1e-8), name
    # the l2 handed in from the fused rasterizer path is used verbatim
    o2 = ours(rendering, target, masks, masks, ray_o, img_aligned_xyz=xyz, gt_img_aligned_xyz=gt_xyz, l2_loss=a[0] * 2)
    assert torch.equal(o2[0], a[0] * 2)


def test_schedule_function_c():
    assert losses.C(0.1, 5, 500) == 0.1
    assert losses.C([150, 0.0, 1.0, 151], 0, 150) == 0.0 and losses.C([150, 0.0, 1.0, 151], 0, 151) == 1.0
    assert abs(losses.C([0.0, 1.0, 100], 0, 25) - 0.25) < 1e-12        # 3 items: start_step 0, int end -> global steps
    assert abs(losses.C([0, 0.0, 1.0, 10.0], 5, 999) - 0.5) < 1e-12     # float end_step -> epochs
    with pytest.raises(TypeError):
        losses.C([1, 2], 0, 0)


def test_combine_follows_training_step_weighting():
    lc = losses.LossComputer()
    l = (torch.tensor([1.0, 3.0]), torch.tensor(0.0), torch.zeros(2), torch.zeros(2), torch.tensor(4.0))
    out = lc.combine(l, dict(lambda_diffusion=1.0, lambda_lpips=0.0, lambda_ssim=0.0, lambda_pointsdist=0.0, lambda_xyz=0.5))
    assert float(out["loss"]) == 2.0 + 0.5 * 4.0 and float(out["loss_diffusion"]) == 2.0
    with pytest.raises(RuntimeError, match="LPIPS"):
        lc.combine(l, dict(lambda_diffusion=1.0, lambda_lpips=0.1))

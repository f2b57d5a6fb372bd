"""CPU tests of the autograd path's host logic: which (criterion, optimizer) pairs train() runs on the fused step, and
the Unet's default of the inference plan."""
import torch
import torch.nn as nn

from weatherconverter_b200.diffusion_model.train_ddpm import fused_step_supported


def _params():
    return [nn.Parameter(torch.zeros(4))]


def test_fused_step_for_the_reference_pair():
    assert fused_step_supported(nn.MSELoss(), torch.optim.Adam(_params(), lr=1e-4))
    assert fused_step_supported(nn.MSELoss(reduction="mean"), torch.optim.Adam(_params(), lr=1e-3, betas=(0.8, 0.99)))


def test_generic_step_for_everything_else():
    p = _params
    assert not fused_step_supported(nn.MSELoss(reduction="sum"), torch.optim.Adam(p()))
    assert not fused_step_supported(nn.MSELoss(reduction="none"), torch.optim.Adam(p()))
    assert not fused_step_supported(nn.L1Loss(), torch.optim.Adam(p()))
    assert not fused_step_supported(nn.SmoothL1Loss(), torch.optim.Adam(p()))
    assert not fused_step_supported(nn.MSELoss(), torch.optim.Adam(p(), weight_decay=1e-2))
    assert not fused_step_supported(nn.MSELoss(), torch.optim.Adam(p(), amsgrad=True))
    assert not fused_step_supported(nn.MSELoss(), torch.optim.Adam(p(), maximize=True))
    assert not fused_step_supported(nn.MSELoss(), torch.optim.AdamW(p()))
    assert not fused_step_supported(nn.MSELoss(), torch.optim.SGD(p(), lr=0.1))


def test_generic_step_for_subclasses():
    class WeightedMSE(nn.MSELoss):
        pass

    class MyAdam(torch.optim.Adam):
        pass

    assert not fused_step_supported(WeightedMSE(), torch.optim.Adam(_params()))
    assert not fused_step_supported(nn.MSELoss(), MyAdam(_params()))


def test_weight_decay_in_any_param_group_leaves_the_fused_step():
    opt = torch.optim.Adam([{"params": _params()}, {"params": _params(), "weight_decay": 1e-3}], lr=1e-4)
    assert not fused_step_supported(nn.MSELoss(), opt)


def test_unet_is_not_differentiable_by_default():
    from oracle.unet import DEFAULT_MODEL_CONFIG
    from weatherconverter_b200.diffusion_model.models.unet_base import Unet
    cfg = dict(DEFAULT_MODEL_CONFIG); cfg["im_size"] = 32
    assert Unet(cfg).differentiable is False

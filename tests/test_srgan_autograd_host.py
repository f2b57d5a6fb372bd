"""CPU tests of the through-SRGAN guidance's argument checks: they reject what is out of scope before any device work."""
import pytest
import torch


def _inputs():
    return torch.zeros(1, 3, 16, 32), torch.zeros(1, 64, 128, dtype=torch.long)


def test_sample_with_sgg_rejects_grad_through_srgan_with_graph_lcg_or_quirks():
    from weatherconverter_b200.translation import sample_with_sgg
    x, gt = _inputs()
    for bad in (dict(use_graph=True), dict(mode="lcg"), dict(mode="alternate"), dict(reference_quirks=True)):
        with pytest.raises(ValueError, match="grad_through_srgan"):
            sample_with_sgg(x, None, None, None, gt, None, n_steps=3, grad_through_srgan=True, **bad)


def test_sample_with_sgg_rejects_a_non_bool_grad_through_srgan():
    from weatherconverter_b200.translation import sample_with_sgg
    x, gt = _inputs()
    for bad in (1, "yes", None, torch.tensor(True)):
        with pytest.raises(TypeError, match="grad_through_srgan"):
            sample_with_sgg(x, None, None, None, gt, None, n_steps=3, grad_through_srgan=bad)


def test_apply_gsg_through_srgan_rejects_a_non_callable_criterion():
    from weatherconverter_b200.sgg.sgg import apply_gsg_through_srgan
    x, gt = _inputs()
    with pytest.raises(TypeError, match="criterion"):
        apply_gsg_through_srgan(None, None, x, x, x, gt, 60.0, criterion="cross_entropy")

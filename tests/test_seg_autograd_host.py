"""CPU tests of the custom-criterion guidance's argument checks: they reject what is out of scope before any device work."""
import pytest
import torch


def _criterion(logits, gt):
    return logits.mean((1, 2, 3))


def test_sample_with_sgg_rejects_criterion_with_graph_or_lcg():
    from weatherconverter_b200.translation import sample_with_sgg
    x = torch.zeros(1, 3, 16, 32)
    gt = torch.zeros(1, 64, 128, dtype=torch.long)
    for bad in (dict(use_graph=True), dict(mode="lcg"), dict(mode="alternate")):
        with pytest.raises(ValueError, match="criterion"):
            sample_with_sgg(x, None, None, None, gt, None, n_steps=3, criterion=_criterion, **bad)


def test_apply_gsg_batch_rejects_a_non_callable_criterion():
    from weatherconverter_b200.sgg.sgg import apply_gsg, apply_gsg_batch
    mu = torch.zeros(1, 3, 16, 32)
    sr = torch.zeros(1, 3, 64, 128)
    gt = torch.zeros(1, 64, 128, dtype=torch.long)
    with pytest.raises(TypeError, match="criterion"):
        apply_gsg_batch(None, mu, mu, sr, gt, 60.0, criterion="cross_entropy")
    with pytest.raises(TypeError, match="criterion"):
        apply_gsg(None, mu, mu, sr, gt, 60.0, criterion=3)

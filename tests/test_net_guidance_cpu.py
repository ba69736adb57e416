"""CPU: per-sample guidance of the network strategies (NetAttrFunc / ClassifierAttrFunc, ``per_sample=True``) on the
generic torch path with a user's torch parser / predictor: the loss is sum_b of the reference's loss on image b alone, so
image b's gradient is the batch-1 gradient of image b.  ``per_sample=False`` keeps the reference's batch-element-0
semantics."""
from types import SimpleNamespace

import torch

from oracle import step_math as sm


def _toy_parser(seed=0):
    torch.manual_seed(seed)
    return torch.nn.Conv2d(3, 19, 3, padding=1)


def _toy_predictor(seed=0):
    torch.manual_seed(seed)
    return torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(3 * 8 * 8, 80))


def _grad(loss_fn, x):
    x = x.detach().clone().requires_grad_(True)
    loss = loss_fn(x)
    (g,) = torch.autograd.grad(loss, x)
    return loss.detach(), g


def test_net_attr_func_per_sample_is_the_sum_of_batch_one_losses():
    from attr_functions import NetAttrFunc
    net = _toy_parser(1)
    f = NetAttrFunc(SimpleNamespace(net=lambda x: (net(x),)), idx_for_class=[17, 1], per_sample=True)
    x = torch.randn(3, 3, 16, 16, generator=torch.Generator().manual_seed(2))
    loss, g = _grad(f.loss, x)
    refs = [_grad(lambda xb: sm.segmentation_area_loss(net(xb), [17, 1]), x[b:b + 1]) for b in range(3)]
    assert torch.allclose(loss, sum(r[0] for r in refs), rtol=1e-6, atol=0)
    for b, (_, gb) in enumerate(refs):
        assert torch.allclose(g[b:b + 1], gb, rtol=1e-6, atol=1e-6 * gb.abs().max().item())


def test_net_attr_func_per_sample_with_a_single_class_id():
    from attr_functions import NetAttrFunc
    net = _toy_parser(3)
    f = NetAttrFunc(SimpleNamespace(net=lambda x: (net(x),)), idx_for_class=4, per_sample=True)
    x = torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(4))
    loss, _ = _grad(f.loss, x)
    ref = sum(sm.segmentation_area_loss(net(x[b:b + 1]), [4]) for b in range(2))
    assert torch.allclose(loss, ref.detach(), rtol=1e-6, atol=0)


def test_classifier_attr_func_per_sample_is_the_sum_of_batch_one_losses():
    from attr_functions import ClassifierAttrFunc
    pred = _toy_predictor(5)
    for reg in ((None, None, None), (3, 0, torch.tensor([0.25, -0.5]))):
        f = ClassifierAttrFunc(pred, idx_for_class=7, idx_of_interest=1, regularize_idx_idx_score=reg, per_sample=True)
        x = torch.randn(3, 3, 8, 8, generator=torch.Generator().manual_seed(6))
        loss, g = _grad(f.loss, x)
        refs = [_grad(lambda xb: sm.classifier_logit_loss(pred(xb), 7, 1, reg), x[b:b + 1]) for b in range(3)]
        assert torch.allclose(loss, sum(r[0] for r in refs), rtol=1e-6, atol=0)
        for b, (_, gb) in enumerate(refs):
            assert gb.abs().max() > 0
            assert torch.allclose(g[b:b + 1], gb, rtol=1e-6, atol=1e-6 * gb.abs().max().item())


def test_classifier_attr_func_default_still_guides_batch_element_zero_only():
    from attr_functions import ClassifierAttrFunc
    pred = _toy_predictor(7)
    f = ClassifierAttrFunc(pred, idx_for_class=7, idx_of_interest=1)
    x = torch.randn(3, 3, 8, 8, generator=torch.Generator().manual_seed(8))
    loss, g = _grad(f.loss, x)
    ref, gr = _grad(lambda xx: sm.classifier_logit_loss(pred(xx), 7, 1), x)
    assert torch.equal(loss, ref) and torch.equal(g, gr)
    assert g[0].abs().max() > 0 and g[1].abs().max().item() == 0.0 and g[2].abs().max().item() == 0.0


def test_native_path_declines_torch_networks():
    """A torch module (or any plain callable) is opaque to the native network path: it returns None and apply() falls
    back to autograd."""
    from attr_functions import ClassifierAttrFunc, NetAttrFunc
    net = _toy_parser(9)
    assert NetAttrFunc(SimpleNamespace(net=net), idx_for_class=[1], per_sample=True).native_network(64) is None
    assert ClassifierAttrFunc(_toy_predictor(9), idx_for_class=3, per_sample=True).native_network(8) is None

"""The single-workspace rule of the native networks (b200edit/engine.py): an input gradient is computed only over the
activations of the forward it belongs to.  Every call that overwrites them - another forward, a profiled forward, an
``enable_grad()`` re-bind of the workspace - makes a later ``input_grad`` / ``latent_grad`` / autograd backward raise
B2EError instead of returning the gradient at the wrong activations.  A kept forward followed by its gradient returns
the same bits as the autograd node on the same input (same launches)."""
from types import SimpleNamespace

import pytest
import torch

pytestmark = pytest.mark.gpu

B = 2


def _rand(*shape, seed):
    return (torch.rand(*shape, generator=torch.Generator().manual_seed(seed)) * 2 - 1).cuda()


def _resnet():
    from b200edit.resnet import ResNet
    net = ResNet("basic", (1, 1, 1, 1), num_classes=10, input_size=64, max_batch=B).init_random(1)
    return SimpleNamespace(net=net, x=_rand(B, 3, 64, 64, seed=2), d=_rand(B, 10, seed=3), keep=net.forward_keep,
                           grad=net.input_grad, call=net, forward=net, profile=net.profile, rebind=None)


def _bisenet():
    from b200edit.bisenet import BiSeNet
    net = BiSeNet(19, 64, max_batch=B).init_random(4).enable_grad()
    return SimpleNamespace(net=net, x=_rand(B, 3, 64, 64, seed=5), d=_rand(B, 19, 64, 64, seed=6), keep=net.forward_keep,
                           grad=net.input_grad, call=lambda x: net(x)[0], forward=net, profile=net.profile,
                           rebind=net.enable_grad)


def _vqmodel():
    from b200edit.vqmodel import VQModel
    net = VQModel(latent_channels=3, out_channels=3, block_out_channels=(32, 64), layers_per_block=1, norm_num_groups=32,
                  norm_eps=1e-6, num_vq_embeddings=64, sample_size=16, max_batch=B).init_random(7).enable_grad()
    return SimpleNamespace(net=net, x=_rand(B, 3, 16, 16, seed=8), d=_rand(B, 3, 32, 32, seed=9), keep=net.decode_keep,
                           grad=net.latent_grad, call=lambda z: net.decode(z).sample, forward=net.decode,
                           profile=net.profile, rebind=net.enable_grad)


def _lpips():
    from b200edit.lpips import LPIPS
    net = LPIPS(input_size=64, max_batch=B).init_random(10)
    ref, ref2 = _rand(1, 3, 64, 64, seed=11), _rand(1, 3, 64, 64, seed=13)
    # every LPIPS forward is kept (input_grad differentiates the last one): the other forward is a new reference's pass
    return SimpleNamespace(net=net, x=_rand(B, 3, 64, 64, seed=12), d=torch.rand(B).cuda(), keep=lambda x: net(x, ref),
                           grad=net.input_grad, call=lambda x: net(x, ref), forward=lambda x: net.set_reference(ref2),
                           profile=net.profile, rebind=net.enable_grad)


NETS = {"resnet": _resnet, "bisenet": _bisenet, "vqmodel": _vqmodel, "lpips": _lpips}
OVERWRITES = {"profile": lambda c: c.profile(c.x), "forward": lambda c: c.forward(c.x), "enable_grad": lambda c: c.rebind()}


@pytest.mark.parametrize("name,between", [(n, w) for n in NETS for w in OVERWRITES if not (n == "resnet" and w == "enable_grad")])
def test_gradient_after_an_overwriting_call_raises(name, between):
    from b200edit._C import B2EError
    c = NETS[name]()
    c.keep(c.x)
    OVERWRITES[between](c)
    with pytest.raises(B2EError):
        c.grad(c.d)
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", list(NETS))
def test_autograd_backward_after_another_forward_raises(name):
    from b200edit._C import B2EError
    c = NETS[name]()
    x = c.x.clone().requires_grad_(True)
    out = c.call(x)
    with torch.no_grad():
        c.call(c.x)
    with pytest.raises(B2EError):
        torch.autograd.grad(out, x, c.d.reshape(out.shape))
    torch.cuda.synchronize()


@pytest.mark.parametrize("name", list(NETS))
def test_kept_forward_gradient_equals_autograd_node(name):
    c = NETS[name]()
    out_k = c.keep(c.x)
    g_k = c.grad(c.d)
    x = c.x.clone().requires_grad_(True)
    out_a = c.call(x)
    g_a, = torch.autograd.grad(out_a, x, c.d.reshape(out_a.shape))
    assert torch.isfinite(g_k).all() and g_k.abs().sum() > 0
    assert torch.equal(out_k, out_a.detach()) and torch.equal(g_k, g_a)

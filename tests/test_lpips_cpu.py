"""LPIPS (vgg) without a GPU: the oracle's parameter layout against the published ``lpips.LPIPS(net='vgg').state_dict()``
names and shapes, the oracle in float64 against an independent per-layer restatement on torchvision's own VGG-16
module, and the host logic of the native wrapper, the guidance strategies and the metric."""
import pytest
import torch

tv = pytest.importorskip("torchvision")

from oracle.lpips import LPIPS as OracleLPIPS  # noqa: E402

CONVS = ((1, 0, 3, 64), (1, 2, 64, 64), (2, 5, 64, 128), (2, 7, 128, 128), (3, 10, 128, 256), (3, 12, 256, 256),
         (3, 14, 256, 256), (4, 17, 256, 512), (4, 19, 512, 512), (4, 21, 512, 512), (5, 24, 512, 512),
         (5, 26, 512, 512), (5, 28, 512, 512))
LIN = (64, 128, 256, 512, 512)


def published_shapes():
    out = {"scaling_layer.shift": (1, 3, 1, 1), "scaling_layer.scale": (1, 3, 1, 1)}
    for s, i, cin, cout in CONVS:
        out[f"net.slice{s}.{i}.weight"] = (cout, cin, 3, 3)
        out[f"net.slice{s}.{i}.bias"] = (cout,)
    for k, c in enumerate(LIN):
        out[f"lin{k}.model.1.weight"] = (1, c, 1, 1)
    return out


def test_oracle_state_dict_matches_published_layout():
    sd = OracleLPIPS().state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == published_shapes()
    assert torch.allclose(sd["scaling_layer.shift"].reshape(-1), torch.tensor([-.030, -.088, -.188]))
    assert torch.allclose(sd["scaling_layer.scale"].reshape(-1), torch.tensor([.458, .448, .450]))


def test_native_random_state_dict_has_the_published_layout():
    from b200edit.lpips import lpips_random_state_dict
    sd = lpips_random_state_dict(3)
    assert {k: tuple(v.shape) for k, v in sd.items()} == published_shapes()
    assert all(float(sd[f"lin{k}.model.1.weight"].min()) >= 0 for k in range(5))    # trained LPIPS: non-negative
    assert all(torch.equal(sd[k], v) for k, v in lpips_random_state_dict(3).items())


def per_layer_restatement(features, lins, shift, scale, x0, x1):
    """Independent statement of LPIPS on torchvision's VGG-16 ``features`` module, walked layer by layer."""
    shift, scale = shift.view(1, 3, 1, 1), scale.view(1, 3, 1, 1)
    taps = {3, 8, 15, 22, 29}

    def feats(x):
        h, out = (x - shift) / scale, []
        for i in range(30):
            h = features[i](h)
            if i in taps:
                out.append(h)
        return out

    total = torch.zeros(x0.shape[0], dtype=x0.dtype)
    for k, (f0, f1) in enumerate(zip(feats(x0), feats(x1))):
        u0 = f0 / (f0.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
        u1 = f1 / (f1.pow(2).sum(1, keepdim=True).sqrt() + 1e-10)
        d = ((u0 - u1) ** 2 * lins[k].view(1, -1, 1, 1)).sum(1)       # (B, H, W)
        total = total + d.mean(dim=(1, 2))
    return total


def test_oracle_float64_equals_per_layer_restatement():
    from b200edit.lpips import lpips_random_state_dict
    sd = lpips_random_state_dict(1)
    oracle = OracleLPIPS().double()
    oracle.load_state_dict({k: v.double() for k, v in sd.items()})
    vgg = tv.models.vgg16(weights=None).features.double().eval()
    vsd = {}
    for s, i, _, _ in CONVS:
        vsd[f"{i}.weight"] = sd[f"net.slice{s}.{i}.weight"].double()
        vsd[f"{i}.bias"] = sd[f"net.slice{s}.{i}.bias"].double()
    vgg.load_state_dict(vsd)
    lins = [sd[f"lin{k}.model.1.weight"].double().reshape(-1) for k in range(5)]
    g = torch.Generator().manual_seed(2)
    x0 = (torch.rand(2, 3, 48, 48, generator=g, dtype=torch.float64) * 2 - 1)
    x1 = (torch.rand(1, 3, 48, 48, generator=g, dtype=torch.float64) * 2 - 1)      # batch-1 reference broadcasts
    with torch.no_grad():
        got = oracle(x0, x1)
        want = per_layer_restatement(vgg, lins, sd["scaling_layer.shift"].double(), sd["scaling_layer.scale"].double(), x0, x1)
    assert got.shape == (2, 1, 1, 1)
    assert torch.allclose(got.reshape(-1), want, rtol=1e-12, atol=0)
    assert float(oracle(x0[:1], x0[:1]).abs().max()) < 1e-20                           # LPIPS(x, x) = 0


def test_use_lpips_host_logic():
    from attr_functions import AttrFunc, MultiColorAttrFunc, SingleColorAttrFunc, l2_norm
    with pytest.raises(NotImplementedError):
        SingleColorAttrFunc(target=0.1, color_idx=0, use_lpips=True)
    model = object()
    f = MultiColorAttrFunc(0.1, 0.2, 0.3, use_lpips=True, use_l2=True, lpips_model=model)
    assert f.metric is model and "lpips_model" not in f.kwargs                 # LPIPS wins over L2
    assert MultiColorAttrFunc(0.1, 0.2, 0.3, use_l2=True).metric is l2_norm
    # the generic expression, with a torch stand-in for the distance network
    calls = []

    def fake_lpips(in0, in1):
        calls.append((in0.shape, in1.shape))
        return (in0 - in1).pow(2).mean(dim=(1, 2, 3), keepdim=True)

    class Mine(AttrFunc):
        def loss(self, img, **kw):
            return img.mean()
    m = Mine(use_lpips=True, lpips_model=fake_lpips)
    pred, mask, x0 = torch.rand(1, 3, 8, 8), (torch.rand(1, 3, 8, 8) > 0.5).float(), torch.rand(1, 3, 8, 8)
    got = m.calculate_loss(pred, mask_pred_original_sample=True, use_lpips=True, lambda_=0.5, mask=mask, x_0=x0)
    want = (mask * pred).mean() + 0.5 * (1 - mask * pred - x0).pow(2).mean()
    assert torch.allclose(got.reshape(()), want) and len(calls) == 1
    with pytest.raises(NotImplementedError):     # use_lpips at call time without a model: as before
        Mine().calculate_loss(pred, mask_pred_original_sample=True, use_lpips=True, lambda_=0.5, mask=mask, x_0=x0)


def test_metric_and_wrapper_validation_without_gpu():
    import metrics
    from b200edit._C import B2EError
    from b200edit.lpips import LPIPS
    with pytest.raises(NotImplementedError):
        metrics.lpips(None, None)
    assert float(metrics.lpips(torch.ones(1), torch.zeros(1), model=lambda a, b: a - b)) == 1.0
    with pytest.raises(ValueError):
        LPIPS(net="alex")
    if not torch.cuda.is_available():
        with pytest.raises(B2EError):
            LPIPS(input_size=64)                    # no CUDA device: no CPU fallback
    # argument validation runs before any device work
    net = object.__new__(LPIPS)
    from types import SimpleNamespace
    net.config, net.max_batch = SimpleNamespace(input_size=32), 2
    x = torch.rand(1, 3, 32, 32)
    with pytest.raises(B2EError):
        net(x, x)                                   # CPU tensors
    with pytest.raises(ValueError):
        net(x, x, normalize=True)
    with pytest.raises(B2EError):
        net(x, x.clone().requires_grad_(True))      # no gradient w.r.t. in1

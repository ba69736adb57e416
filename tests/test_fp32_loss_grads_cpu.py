"""CPU: the loss networks' ``grad_precision`` is validated before anything is built - in the C ABI (``b2e_resnet_create`` /
``b2e_lpips_create`` refuse a bad combination before touching the device) and in every Python entry point (the device
lookup, replaced by a trap, is never reached)."""
import ctypes

import pytest

B2E_INVALID_ARG = -1


@pytest.mark.parametrize("precision,grad_precision", [(0, 1), (1, 2), (0, 2), (1, -1)])
@pytest.mark.parametrize("net", ["resnet", "bisenet", "lpips"])
def test_c_abi_refuses_bad_grad_precision(net, precision, grad_precision):
    from b200edit import _C
    h = ctypes.c_void_p()
    if net == "lpips":
        cfg = _C.LpipsConfig(input_size=64, precision=precision, grad_precision=grad_precision)
        rc = _C.lib.b2e_lpips_create(ctypes.byref(cfg), 1, ctypes.byref(h))
    else:
        cfg = _C.ResNetConfig(input_size=64, in_channels=3, bottleneck=0, width=64, num_classes=19 if net == "bisenet" else 16,
                              head=int(net == "bisenet"), precision=precision, grad_precision=grad_precision)
        for i in range(4):
            cfg.layers[i] = 2
        rc = _C.lib.b2e_resnet_create(ctypes.byref(cfg), 1, ctypes.byref(h))
    assert rc == B2E_INVALID_ARG and not h.value
    assert b"grad_precision" in _C.lib.b2e_last_error()


def test_config_structs_end_with_grad_precision():
    """The field is appended last, so a caller's zero-initialised config keeps the 16-bit backward."""
    from b200edit import _C
    for cls in (_C.ResNetConfig, _C.LpipsConfig):
        assert cls._fields_[-2][0] == "precision" and cls._fields_[-1][0] == "grad_precision"
        assert cls().grad_precision == 0
    assert ctypes.sizeof(_C.ResNetConfig) == 4 * 12 and ctypes.sizeof(_C.LpipsConfig) == 4 * 3


def _fast():
    from b200edit import _C
    return _C.fast_precision()


BAD = [dict(precision="fp16", grad_precision="fp32"), dict(precision="fp32", grad_precision="fp64"),
       dict(precision="fp32", grad_precision="fp16"), dict(precision="fp32", grad_precision=True)]


@pytest.fixture
def trapped(monkeypatch):
    """Replaces both device lookups (the factories' and the engines') by a trap."""
    import models
    from b200edit import _C

    def trap(*a, **k):
        raise AssertionError("something was built before grad_precision was validated")

    monkeypatch.setattr(models, "get_device", trap)
    monkeypatch.setattr(_C, "require_device", trap)


def _kw(kw):
    return dict(kw, precision=_fast()) if kw["precision"] == "fp16" else kw


@pytest.mark.parametrize("kw", BAD)
def test_engines_refuse_before_building(trapped, kw):
    from b200edit.bisenet import BiSeNet, MultiResBiSeNet
    from b200edit.lpips import LPIPS
    from b200edit.resnet import ResNet
    kw = _kw(kw)
    for make in (lambda: ResNet("basic", (2, 2, 2, 2), 16, 64, max_batch=1, **kw), lambda: BiSeNet(19, 64, **kw),
                 lambda: LPIPS(input_size=64, **kw), lambda: MultiResBiSeNet(19, **kw)):
        with pytest.raises(ValueError, match="precision"):
            make()


@pytest.mark.parametrize("kw", BAD)
def test_factories_refuse_before_building(trapped, kw):
    import models
    kw = _kw(kw)
    with pytest.raises(ValueError, match="precision"):
        models.get_pretrained_anyGAN(input_size=64, state_dict_path=None, **kw)
    with pytest.raises(ValueError, match="precision"):
        models.get_lpips(input_size=64, **kw)
    seg_kw = dict(kw, precision=None if kw["precision"] == "fp32" else "fp16")
    with pytest.raises(ValueError, match="precision"):
        models.SegmentationModel(None, **seg_kw)


def test_segmentation_model_grad_precision_is_keyword_only():
    import models
    with pytest.raises(TypeError):
        models.SegmentationModel(None, 19, (512, 512), None, 0, None, 1, "fp32")

"""CPU: ``create_diffusion_model(decoder_grad_precision=...)`` is validated on the host before anything is built."""
import pytest


@pytest.mark.parametrize("kw", [dict(precision=None, decoder_grad_precision="fp32"),
                                dict(precision="fp16", decoder_grad_precision="fp32"),
                                dict(precision="fp32", decoder_grad_precision="fp64"),
                                dict(precision="fp32", decoder_grad_precision="fp16")])
@pytest.mark.parametrize("name", ["ldm", "sd"])
def test_decoder_grad_precision_is_refused_before_building(monkeypatch, name, kw):
    """"fp32" needs precision="fp32"; any other value (unknown, or a 16-bit name) is refused as well.  The device lookup is
    the factory's first step after validation: replaced by a trap, it shows that nothing was built."""
    import models

    def trap():
        raise AssertionError("create_diffusion_model built something before validating decoder_grad_precision")

    monkeypatch.setattr(models, "get_device", trap)
    if kw["precision"] == "fp16":
        from b200edit import _C
        kw = dict(kw, precision=_C.fast_precision())
    with pytest.raises(ValueError, match="precision"):
        models.create_diffusion_model(name, **kw)

"""Evaluation harness of the editing path (drop-in for src/metrics.py:31-203): how an edit moves the predictions of the
AnyCost-GAN attribute predictor.  Everything it calls is on the engine: generation and editing through
``Diffusion.generate_image`` / ``SegDiffEditPipeline.edit_image``, the predictor through the native ResNet-50
(``models.get_pretrained_anyGAN``).  Meaningful numbers need real checkpoints; with seeded random-init weights the
harness is exercised for its contract (shapes, keys, determinism).

Deviations from the reference: ``num_inference_steps`` and ``predictor`` are parameters (the reference hard-codes 50 steps
and reloads the checkpoint inside every call), tensors follow the model's device instead of the literal "cuda", and
``lpips`` takes the distance network as ``model=`` (``models.get_lpips``: the native LPIPS-vgg; the reference's own
function shadows the ``lpips`` module it needs); without one it raises."""
from collections import defaultdict
from typing import Dict, Optional, Tuple

import torch

from constants import ANY_GAN_ATTRS_DICT
from models import get_pretrained_anyGAN
from SegDiffEditPipeline import SegDiffEditPipeline
from transforms import pil_to_tensor
from utils import generate_random_samples


def lpips(original: torch.Tensor, edited: torch.Tensor, model=None):
    """LPIPS(original, edited), (B, 1, 1, 1) (src/metrics.py: ``lpips.LPIPS(net='vgg')(original, edited)``).  ``model``:
    the distance network, e.g. ``models.get_lpips(input_size=...)``; there is no default because no VGG / lin weights
    ship offline."""
    if model is None:
        raise NotImplementedError("metrics.lpips needs model= (e.g. models.get_lpips(input_size=...)): the lpips package "
                                  "and its VGG weights are not available offline")
    with torch.no_grad():
        return model(original, edited)


def _predictor_for(img_t: torch.Tensor, predictor=None):
    if predictor is None:
        predictor = get_pretrained_anyGAN(input_size=img_t.shape[-1], max_batch=1)
    return predictor.eval()


def _original_and_edited_logits(editor: SegDiffEditPipeline, diffusion_model, attr_func, generator, predictor, steps):
    """One sample: generate (eta = 1, shared noise maps), edit with the same x_T / z maps, predict attributes of both."""
    xt = generate_random_samples(1, diffusion_model.unet, generator=generator)
    zs = generate_random_samples(steps, diffusion_model.unet, generator=generator)
    img, model_outputs, _, _ = diffusion_model.generate_image(xt=xt, eta=1, zs=zs, num_inference_steps=steps)
    img_t = pil_to_tensor(img).to(xt.device)
    predictor = _predictor_for(img_t, predictor)
    with torch.no_grad():
        o_attr = predictor(img_t).view(-1, 40, 2)
        img_edit = editor.edit_image(xt=xt, eta=1, model_outputs=model_outputs, zs=zs, attr_func=attr_func, prog_bar=False)[0]
        edit_attr = predictor(pil_to_tensor(img_edit).to(xt.device)).view(-1, 40, 2)
    return o_attr, edit_attr, predictor


def avg_increase_decrease_per_attribute(editor: SegDiffEditPipeline, diffusion_model, attr_func, n_samples, generator, *,
                                        num_inference_steps: int = 50, predictor=None) -> Tuple[Dict[str, float], Dict[str, float]]:
    """Average change of every attribute logit (edited - original), one dictionary per prediction index (0 / 1), keys
    "<attribute index> <attribute name>" (src/metrics.py:31-131)."""
    names = {v: k for k, v in ANY_GAN_ATTRS_DICT.items()}
    d_zero, d_one = defaultdict(float), defaultdict(float)
    for _ in range(n_samples):
        o_attr, edit_attr, predictor = _original_and_edited_logits(editor, diffusion_model, attr_func, generator, predictor,
                                                                   num_inference_steps)
        diff = (edit_attr - o_attr)[0].cpu()        # (40, 2)
        for i in range(40):
            d_zero[f"{i} {names[i]}"] += float(diff[i, 0])
            d_one[f"{i} {names[i]}"] += float(diff[i, 1])
    return ({k: v / n_samples for k, v in d_zero.items()}, {k: v / n_samples for k, v in d_one.items()})


def attribute_consistency(editor: SegDiffEditPipeline, diffusion_model, attr_func, n_samples, generator, *,
                          num_inference_steps: int = 50, predictor=None) -> torch.Tensor:
    """Fraction of samples whose predicted class of each attribute survives the edit: tensor (40,) (src/metrics.py:138-203)."""
    accs: Optional[torch.Tensor] = None
    for _ in range(n_samples):
        o_attr, edit_attr, predictor = _original_and_edited_logits(editor, diffusion_model, attr_func, generator, predictor,
                                                                   num_inference_steps)
        same = (torch.argmax(o_attr, dim=2) == torch.argmax(edit_attr, dim=2)).float().mean(0)
        accs = same if accs is None else accs + same
    return accs / n_samples


if __name__ == "__main__":
    # args: diffusion_model (ddpm | ldm | sd), attr_func (anygan), n_samples, seed, loss_scale, t1, t2
    import sys

    from attr_functions import AnyGANAttrFunc
    from models import SegmentationModel, create_diffusion_model
    from utils import set_seed
    name, attr_name, n, seed, loss_scale, t1, t2 = sys.argv[1:8]
    if name not in ("ddpm", "ldm", "sd"):
        raise ValueError("diffusion_model must be ddpm, ldm, or sd")
    generator = set_seed(int(seed))
    model = create_diffusion_model(name, sample_clipping=(name == "ddpm"), max_batch=1)
    size = 512 if name == "sd" else 256
    predictor = get_pretrained_anyGAN(input_size=size, max_batch=1)
    if attr_name != "anygan":
        raise ValueError("attr_func must be anygan")
    func = AnyGANAttrFunc(predictor=predictor, idx_for_class=31, loss_scale=float(loss_scale), t1=float(t1), t2=float(t2))
    editor = SegDiffEditPipeline(diffusion_wrapper=model, segmentation_model=SegmentationModel())
    print(attribute_consistency(editor, model, func, int(n), generator, predictor=predictor))
    d0, d1 = avg_increase_decrease_per_attribute(editor, model, func, int(n), generator, predictor=predictor)
    print(d0)
    print(d1)

"""Segmentation map -> binary edit mask (drop-in for src/mask_creator.py).

create_mask fuses the reference's chain - per-class equality, optional 7x7 hard-max dilation, sum
over classes, antialiased bilinear resize, threshold, 3-channel replicate - into three small CUDA
kernels with results bit-identical to the torch/torchvision path (see csrc/mask_kernels.cu)."""
import torch

from b200edit import ops
from utils import get_device


class MaskCreator:
    def __init__(self, dilate_mask: bool = True, resize_size: tuple = (256, 256), antialias: bool = True) -> None:
        self.device = get_device()
        self.dilate_mask = bool(dilate_mask)
        self.kernel_size = 7                      # Dilation2d(1, 1, 7, soft_max=False)
        self.resize_size = tuple(resize_size)     # (256,256) pixel space, (64,64) latent space
        self.antialias = antialias                # torchvision >= 0.17 default; False is not implemented

    def create_mask(self, segmentation: torch.Tensor, classes: list, channels: int = 3) -> torch.Tensor:
        """(H,W) integer parsing map -> (1,channels,d,d) float mask in {0,1} on the device; (N,H,W) maps ->
        (N,channels,d,d) in one batched call."""
        seg = segmentation.to(self.device) if not segmentation.is_cuda else segmentation
        return ops.mask_from_seg(seg, list(classes), self.dilate_mask, self.resize_size, channels=channels,
                                 ksize=self.kernel_size, antialias=self.antialias)

    # pieces of the reference's chain, kept for callers that use them individually
    def create_class_mask(self, parsing: torch.Tensor, class_label: int) -> torch.Tensor:
        H, W = parsing.shape[-2:]
        m = ops.mask_from_seg(parsing.to(self.device), [class_label], self.dilate_mask, (H, W), channels=1,
                              ksize=self.kernel_size)
        return m[0, 0]

    def resize_mask(self, mask: torch.Tensor) -> torch.Tensor:
        r = ops.resize_bilinear_aa(mask.to(self.device, torch.float32), self.resize_size)
        return (r >= 1).to(torch.float32)

    def postprocess_mask(self, mask: torch.Tensor) -> torch.Tensor:
        m = self.resize_mask(mask)
        return m.expand(3, *m.shape[-2:]).unsqueeze(0).contiguous()

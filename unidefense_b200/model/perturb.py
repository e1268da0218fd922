"""Input perturbations of the second training pass               (SURVEY.md §8a rows a13-a16).

Reference: model/modules.py:7-21 (random_noise, random_blur, downscale), :35-76
(FrequencyStyleTransfer, SpatialStyleTransfer) and utils/operation.py:15-45 (coral).  Control-flow
randomness comes from torch's CPU generator exactly as in the reference (Appendix D) so that a
shared seed reproduces the same augmentation choices.  random_noise, random_blur and downscale pass the gradient
on to the input as in the reference; the style transfers and coral run under no_grad there and here.
"""
import torch

from .. import ops


def random_noise(tensor, mean=0.0, std=1e-5):
    """modules.py:7-12."""
    white = torch.normal(mean, std, size=tensor.shape, device=tensor.device)
    return torch.clip(tensor + white, -1.0, 1.0)


def random_blur(tensor, kernel_size=(5, 5)):
    """modules.py:15-16: torchvision gaussian_blur(kernel 5x5, default sigma 1.1, reflect padding)."""
    if tuple(kernel_size) != (5, 5):
        raise ValueError("random_blur: only the reference's 5x5 kernel is implemented")
    return ops.gaussian_blur5(tensor.float())


def downscale(tensor, bottleneck_scale=0.75):
    """modules.py:19-21: nearest down by `bottleneck_scale`, nearest back up."""
    return ops.downscale_nearest(tensor.float(), bottleneck_scale)


class FrequencyStyleTransfer(object):
    """modules.py:35-55: keep the content phase, mix content/style amplitudes with lambda ~ U[0.5, 1)."""

    def __call__(self, content, style) -> torch.Tensor:
        B = content.size(0)
        lmda = (torch.rand((B, 1, 1, 1)) / 2.0 + 0.5).to(content)      # CPU generator, like the reference
        return ops.freq_style_transfer(content, style, lmda.reshape(B))


class SpatialStyleTransfer(object):
    """modules.py:58-76: exact histogram matching towards the style image, blended by lambda."""

    def __call__(self, content, style) -> torch.Tensor:
        assert content.size() == style.size()
        B = content.size(0)
        lmda = (torch.rand((B, 1, 1)) / 2.0 + 0.5).to(content)
        return ops.spatial_style_transfer(content, style, lmda.reshape(B))


def coral(source, target):
    """utils/operation.py:20-45 for one [3,H,W] pair (kept for API parity; the model uses coral_batch)."""
    return ops.coral_batch(source[None], target[None])[0]

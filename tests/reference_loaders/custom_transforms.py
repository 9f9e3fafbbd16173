"""Test double for the reference's custom_transforms module, which train.py imports from PYTHONPATH for real datasets: the
same class names and call convention (every transform maps (list of images, 3 x 3 intrinsics) to the same pair), written
for the tests of train.py's loader plumbing so that they run without the reference installed.  The arithmetic of the
reference chain itself is pinned elsewhere (oracle/augment.py against tests/golden/augment.npz)."""
import random

import numpy as np
import torch
from PIL import Image


class Compose:
    def __init__(self, transforms):
        self.transforms = transforms

    def __call__(self, images, intrinsics):
        for t in self.transforms:
            images, intrinsics = t(images, intrinsics)
        return images, intrinsics


class Normalize:
    """Per-channel (x - mean) / std on CHW tensors."""

    def __init__(self, mean, std):
        self.mean = torch.tensor(mean, dtype=torch.float32).view(-1, 1, 1)
        self.std = torch.tensor(std, dtype=torch.float32).view(-1, 1, 1)

    def __call__(self, images, intrinsics):
        return [(im - self.mean) / self.std for im in images], intrinsics


class ArrayToTensor:
    """H x W x 3 arrays in [0, 255] -> 3 x H x W float32 tensors in [0, 1]."""

    def __call__(self, images, intrinsics):
        return [torch.from_numpy(np.ascontiguousarray(np.transpose(im, (2, 0, 1)), np.float32)) / 255 for im in images], intrinsics


class RandomHorizontalFlip:
    def __call__(self, images, intrinsics):
        if random.random() < 0.5:
            intrinsics = np.copy(intrinsics)
            intrinsics[0, 2] = images[0].shape[1] - intrinsics[0, 2]
            images = [np.copy(np.fliplr(im)) for im in images]
        return images, intrinsics


class RandomScaleCrop:
    """Zoom every image by one random factor in [1, 1.15) per axis (Pillow bicubic on uint8), crop back to the input size."""

    def __call__(self, images, intrinsics):
        h, w, _ = images[0].shape
        sx, sy = np.random.uniform(1, 1.15, 2)
        big_h, big_w = int(h * sy), int(w * sx)
        oy, ox = np.random.randint(big_h - h + 1), np.random.randint(big_w - w + 1)
        out = [np.asarray(Image.fromarray(im.astype(np.uint8)).resize((big_w, big_h)), np.float32)[oy:oy + h, ox:ox + w]
               for im in images]
        k = np.copy(intrinsics)
        k[0] *= sx
        k[1] *= sy
        k[0, 2] -= ox
        k[1, 2] -= oy
        return out, k

"""Test double for the reference's datasets/sequence_folders.py (see ../custom_transforms.py): SequenceFolder over
root/<scene>/NNNNNNN.jpg + cam.txt, with the scenes listed in root/train.txt or root/val.txt.  A sample is a target frame
and its neighbours within sequence_length, as (target, [references], intrinsics, inverse intrinsics)."""
import os
import random

import numpy as np
import torch.utils.data
from PIL import Image


class SequenceFolder(torch.utils.data.Dataset):
    def __init__(self, root, seed=None, train=True, sequence_length=3, transform=None, skip_frames=1, dataset="kitti"):
        self.transform = transform
        with open(os.path.join(root, "train.txt" if train else "val.txt")) as f:
            scenes = [os.path.join(root, line.strip()) for line in f if line.strip()]
        half = (sequence_length - 1) // 2
        offsets = [d * skip_frames for d in range(-half, half + 1) if d != 0]
        self.samples = []
        for scene in scenes:
            K = np.loadtxt(os.path.join(scene, "cam.txt")).astype(np.float32).reshape(3, 3)
            frames = sorted(os.path.join(scene, n) for n in os.listdir(scene) if n.endswith(".jpg"))
            for t in range(half * skip_frames, len(frames) - half * skip_frames):
                self.samples.append((frames[t], [frames[t + d] for d in offsets], K))
        random.Random(seed).shuffle(self.samples)

    def __len__(self):
        return len(self.samples)

    def __getitem__(self, i):
        tgt, refs, K = self.samples[i]
        imgs = [np.asarray(Image.open(p), np.float32) for p in [tgt] + refs]
        K = np.copy(K)
        if self.transform is not None:
            imgs, K = self.transform(imgs, K)
        return imgs[0], imgs[1:], K, np.linalg.inv(K)

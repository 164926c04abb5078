import json
import os

import numpy as np
import torch
from PIL import Image
from scipy import sparse


def get_norm_stats(dataroot, key):
    with open(os.path.join(dataroot, "normalization_stats.json")) as f:
        rows = {r["path"]: r for r in map(json.loads, f)}
    return rows[key]["means"], rows[key]["stds"]


def find_valid_files(directory, extensions):
    return sorted(os.path.join(r, f) for r, _, fs in os.walk(directory) for f in fs if f.endswith(tuple(extensions)))


def crop_tensors(*tensors, crop_bounds):
    (x0, y0), (x1, y1) = crop_bounds
    out = [t[:, y0:y1, x0:x1] for t in tensors]
    return out[0] if len(out) == 1 else out


def decompress_cloth_segment(fname, n_labels):
    """Stored label map -> float32 one-hot [n_labels, H, W]; label 0 is the all-zero vector."""
    lab = torch.from_numpy(sparse.load_npz(fname).toarray())
    ch = torch.arange(n_labels).view(-1, 1, 1)
    return ((lab[None] == ch) & (ch > 0)).float()


def per_channel_transform(cloth, transform):
    """Each channel through `transform` as its own Pillow image."""
    planes = cloth.numpy()
    return torch.from_numpy(np.stack([np.array(transform(Image.fromarray(p))) for p in planes]))

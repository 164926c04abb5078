"""Generate tests/golden/augment_64.npz from the UNMODIFIED reference (oracle/ref_harness.py).

    SWAPNET_REFERENCE=/path/to/SwapNet python tests/tools/make_golden_augment.py

The reference's own `per_channel_transform` (datasets/data_utils.py:346-361) with its own `get_transforms(opt)`
(datasets/__init__.py:88-110; warp default --input_transforms hflip vflip affine perspective) on a seeded 19-channel
one-hot cloth tensor (64x64 and 40x56), python `random` and torch seeded per case.  Stored: the label maps, the seeds,
the transformed float32 tensors and a digest of both RNG states AFTER the call, so that
tests/test_augment_cpu.py can check the product's host draws consume the generators exactly like the reference.
"""
import hashlib
import os
import random
import sys
from argparse import Namespace

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from oracle import augment as A
from oracle import ref_harness as RH

RH.import_reference()
from datasets import get_transforms  # noqa: E402  (the reference's)
from datasets.data_utils import per_channel_transform  # noqa: E402


def rng_digest() -> str:
    h = hashlib.sha256()
    h.update(np.asarray(random.getstate()[1], dtype=np.uint64).tobytes())
    h.update(torch.get_rng_state().numpy().tobytes())
    return h.hexdigest()


def label_map(h, w, seed):
    g = np.random.default_rng(seed)
    return g.integers(0, 19, ((h + 7) // 8, (w + 7) // 8)).repeat(8, 0).repeat(8, 1)[:h, :w].astype(np.uint8)


if __name__ == "__main__":
    out = {}
    cases = [("all_64", ("hflip", "vflip", "affine", "perspective"), 64, 64, 11),
             ("all_40x56", ("hflip", "vflip", "affine", "perspective"), 40, 56, 12),
             ("affine_64", ("affine",), 64, 64, 13),
             ("flips_64", ("hflip", "vflip"), 64, 64, 14)]
    for name, names, h, w, seed in cases:
        tf = get_transforms(Namespace(input_transforms=names))
        lab = label_map(h, w, seed)
        cloth = torch.from_numpy(A.onehot(lab, 19))
        random.seed(seed)
        torch.manual_seed(seed)
        res = per_channel_transform(cloth, tf).numpy()
        out[name + "_labels"] = lab
        out[name + "_out"] = res
        out[name + "_rng"] = np.array(rng_digest())
        out[name + "_seed"] = np.array(seed)
        out[name + "_transforms"] = np.array(",".join(names))
        print(name, res.shape, "nonzero", int((res != 0).sum()), "fractional", int(((res != 0) & (res != 1)).sum()))
    path = os.path.join(ROOT, "tests", "golden", "augment_64.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
